// Host-side launchers of the CUDA kernels (internal).
#pragma once
#include <cstdlib>

#include "common.cuh"

namespace gnnb {

// ---------------------------------------------------------------- graph tables (tables.cu)
struct TableWorkspace {
    DeviceBuf keys_in, keys_out, vals_in, vals_out, cub_tmp, heavy_partial, counters;
    DeviceBuf hub_hist, hub_cnt;
    void release_all()
    {
        DeviceBuf *b[] = {&keys_in, &keys_out, &vals_in, &vals_out, &cub_tmp,
                          &heavy_partial, &counters, &hub_hist, &hub_cnt};
        for (DeviceBuf *x : b) x->release();
    }
};

// edge_list [E][2] local ids; node_ptr/edge_ptr (device int64, G+1 entries) translate them to
// ids in the batch union (pass nullptr for a single graph).  Writes in/out degree, offsets
// (n entries), neighbor_table (e entries) and, when non-null, edge_index_table (edge ids relative
// to edge_list, i.e. to edge_base).
// node_base/edge_base: values of node_ptr[0]/edge_ptr[0] when the pointers address a sub-range
// (chunk) of a larger batch whose x / edge_list pointers were advanced accordingly.
int build_tables(const int32_t *edge_list, const int64_t *node_ptr, const int64_t *edge_ptr,
                 int64_t node_base, int64_t edge_base, int n_graphs, int n, int e, int32_t *in_deg, int32_t *out_deg, int32_t *offsets,
                 int32_t *nbr, int32_t *edge_index, TableWorkspace &ws, cudaStream_t s,
                 int *launches, int *bad = nullptr);
// `bad` (device int, optional): set to 1 when an edge endpoint lies outside its graph; such edges
// are dropped from the degree counts so the tables stay memory-safe, and the caller reports
// GNNB_ERR_INVALID (the fused kernels report the same condition as status 2)
// degree tables only (lib:1051-1083)
int build_degree_tables(const int32_t *edge_list, int n, int e, int32_t *in_deg, int32_t *out_deg,
                        cudaStream_t s, int *launches, int *bad = nullptr);
// offsets + neighbor table from given in-degree (lib:1086-1166)
int build_neighbor_tables(const int32_t *edge_list, const int32_t *in_deg, int n, int e,
                          int32_t *offsets, int32_t *nbr, int32_t *edge_index, TableWorkspace &ws,
                          cudaStream_t s, int *launches, int *bad = nullptr);
// CSR slice of a 1D row partition: edge_list holds the in-edges of the owned destination rows
// [row_begin, row_begin + n_local) with GLOBAL node ids; neighbors keep their global ids
int build_partition_tables(const int32_t *edge_list, int row_begin, int n_local, int e,
                           int32_t *in_deg_local, int32_t *offsets_local, int32_t *nbr_global,
                           TableWorkspace &ws, cudaStream_t s, int *launches);
// Degree bucketing: rows longer than `threshold` ("heavy" rows; on the 2M-node power-law graph
// 0.5 % of the rows hold 49 % of the edges) are cut into chunks of kHeavyChunk neighbors, one warp
// per chunk, and a second kernel adds a row's chunk sums in order (deterministic).
constexpr int kHeavyChunk = 128;
struct HeavyList {
    DeviceBuf rows;        // [n_heavy] row ids
    DeviceBuf chunk_base;  // [n_heavy] first chunk of the row
    DeviceBuf chunk_row;   // [n_chunks] index into rows[] of the chunk's row
    int n_heavy = 0, n_chunks = 0;
    void release() { rows.release(); chunk_base.release(); chunk_row.release(); n_heavy = n_chunks = 0; }
};
// fills `hl` from the row lengths (two small kernels and one host synchronisation)
int find_heavy_rows(const int32_t *lengths, int n, int threshold, TableWorkspace &ws, HeavyList &hl,
                    cudaStream_t s, int *launches);
// degree bucketing parameters + partial-sum scratch for the heavy-row kernels
constexpr int kHeavyThreshold = 256;
// (tuning hook: GNNB_HEAVY_THRESHOLD overrides the bucket boundary)
inline int heavy_threshold()
{
    static const int v = [] {
        const char *e = getenv("GNNB_HEAVY_THRESHOLD");
        const int t = e ? atoi(e) : 0;
        return t > 0 ? t : kHeavyThreshold;
    }();
    return v;
}
// partial-sum scratch of the heavy rows: [n_chunks][F] floats (grow-only)
int heavy_setup(TableWorkspace &ws, int n_chunks, int F);
// hub sources: copy of the neighbor table with bit 31 set on the most-referenced sources whose
// feature rows fit budget_bytes (L2-resident set of the aggregation); tables.cu
int mark_hub_sources(const int32_t *nbr_in, int32_t *nbr_out, int e, const int32_t *ref_cnt,
                     int n_src, size_t row_bytes, size_t budget_bytes, TableWorkspace &ws,
                     int *n_hubs_host, cudaStream_t s, int *launches);
// L2 budget for hub rows in bytes (GNNB_HUB_L2_MB overrides; 0 disables the hints)
inline size_t hub_l2_budget()
{
    static const size_t v = [] {
        const char *e = getenv("GNNB_HUB_L2_MB");
        const long mb = e ? atol(e) : 0;   // off by default: measured, it cuts DRAM bytes by 10 %
                                           // and no time (profiles/r2_agg_c5.txt), and costs the
                                           // out-degree atomics + a marking pass per run
        return (size_t)(mb > 0 ? mb : 0) << 20;
    }();
    return v;
}
// dinv[i] = 1 / sqrt(1 + in_deg[i])
int compute_dinv(const int32_t *in_deg, float *dinv, int n, cudaStream_t s, int *launches);

// ---------------------------------------------------------------- aggregation (agg.cu)
// The heavy rows of one aggregation (degree bucketing): rows longer than `threshold` are left to the
// chunked heavy-row kernels; n == 0 (the zero-initialised block) turns the bucketing off.
struct HeavyArgs {
    const int32_t *rows;   // [n] row ids
    int n;
    int threshold;
    float *partial;        // [chunks][...] per-chunk partials, laid out by the aggregation
    const int32_t *chunk_base, *chunk_row;   // HeavyList::chunk_base / chunk_row
    int chunks;
    void set(const HeavyList &hl, float *p)
    {
        rows = hl.rows.as<int32_t>(); n = hl.n_heavy;
        chunk_base = hl.chunk_base.as<int32_t>(); chunk_row = hl.chunk_row.as<int32_t>();
        chunks = hl.n_chunks; partial = p;
    }
};

enum AggMode { AGG_GCN = 0, AGG_GIN = 1, AGG_MEAN = 2, AGG_SUM = 3, AGG_LG = 4 };

struct AggArgs {
    int mode;
    const float *x;        // [n][ldx]
    int ldx;
    int F;
    float *out;            // [n][ldo]
    int ldo;
    const int32_t *offsets, *nbr, *in_deg;
    const float *dinv;     // AGG_GCN fast mode only
    int n;
    float eps;             // AGG_GIN
    HeavyArgs heavy;       // partial: [chunks][F] chunk sums
    int row_base;          // row-partitioned graphs: global id of local row 0 (x / dinv are global,
                           // offsets / in_deg / out are local); 0 otherwise
    // ---- FAST-mode extensions (all 0 / null by default)
    const int32_t *counts; // row lengths when they differ from in_deg (one PART of a split CSR: the
                           // rows' owned-source or halo-source edges); in_deg still feeds the mean
    int accumulate;        // start every row sum from what `out` already holds (second CSR part)
    int no_finish;         // store the plain partial sum: no self term / normalisation (first part)
    int short_ctas;        // 1: one pass per CTA instead of a capped grid-stride grid, so that the CTAs
                           // of a higher-priority kernel (the halo pack on the exchange stream) are
                           // placed as these retire instead of waiting for the whole kernel
    int hub_bit;           // 1: bit 31 of a neighbor entry marks a hub source (high out-degree);
                           // its row is loaded with an L2 evict_last policy, every other row with
                           // evict_first, so the hub rows stay resident in the 126 MB L2
};
int launch_agg(const AggArgs &a, bool strict, cudaStream_t s, int *launches);

// GINE aggregation (lib:1555-1623): sum_k relu(x[nbr_k] + proj[edge_index_k]) + (1 + eps) x_v
struct GineAggArgs {
    const float *x;        // [n][ldx]
    int ldx, F;
    const float *proj;     // [E][ldp] projected edge features (edge id order)
    int ldp;
    float *out;            // [n][ldo]
    int ldo;
    const int32_t *offsets, *nbr, *edge_index, *in_deg;
    int n;
    float eps;
};
int launch_gine_agg(const GineAggArgs &a, cudaStream_t s, int *launches);

// GINE aggregation of the model path: the same sum with the edge projection computed on the fly,
// proj_e = b_e + sum_j W_e[.][j] ef[e][j], so the [E][F] projection is never materialised.  The edge
// features are read in CSR slot order (ef_sorted[k] belongs to neighbor slot k, see
// launch_permute_edge_rows).  Every operation is separately rounded in the reference's order.
constexpr int kGineMaxEdgeDim = 64;
struct GineProjAggArgs {
    const float *x;          // [n][ldx]
    int ldx, F;
    const float *ef_sorted;  // [E][lde] edge features in neighbor-slot order (lde = round_up(edge_dim, 4))
    int lde, edge_dim;
    const float *We_t;       // [edge_dim][ldw] W_e^T (ldw multiple of 4, zero padded)
    int ldw;
    const float *be;         // [F] b_e
    float *out;              // [n][ldo]
    int ldo;
    const int32_t *offsets, *nbr, *in_deg;
    int n;
    float eps;
};
int launch_gine_agg_proj(const GineProjAggArgs &a, cudaStream_t s, int *launches);
// dst[k][0..dim) = src[idx[k]][0..dim) for k < e (dst row stride ldd, src row stride dim)
int launch_permute_edge_rows(const float *src, int dim, const int32_t *idx, int e, float *dst,
                             int ldd, cudaStream_t s, int *launches);

// What the GAT, GATv2 and TransformerConv aggregations share: the layer's GEMM output, the attention
// shape, the epilogue y_v = act(sum softmax_v(e) m_u + bias (+ skip_v)) written to out, the CSR and
// the heavy rows, whose partials are [heavy.chunks][ldp]: accumulator (H*C), then max [H], sum [H].
struct AttnAggArgs {
    const float *g;        // [n][ldg]: GAT [h | a_src | a_dst], GATv2 [xl | xr], TransformerConv [k | v]
    int ldg;
    int H, C;
    float slope;           // LeakyReLU negative slope
    const float *bias;     // [H*C]
    const float *skip;     // [n][ldskip] or null
    int ldskip;
    int act;
    float *out;            // [n][ldo]
    int ldo;
    const int32_t *offsets, *nbr, *in_deg;
    int n;
    HeavyArgs heavy;
    int ldp;               // >= H*C + 2H, multiple of 4
};

// GAT attention aggregation (PyG GATConv, concat heads, inference).  g is the output of the layer's
// one GEMM: per row h (H*C columns, head-major), then a_src [H] and a_dst [H].  Per destination v and
// head: e_uv = LeakyReLU(a_src[u] + a_dst[v]) over the in-neighbours u != v plus one self term,
// y_v = act(sum softmax_v(e) h_u + bias (+ skip_v)), written to out.  One gather pass with an online
// softmax (running max, rescaled sum and accumulator).  Rows longer than heavy.threshold (when a
// heavy list is given) are cut into kHeavyChunk-neighbour chunks whose (max, sum, accumulator)
// partials are merged per row in a fixed order.
struct GatAggArgs : AttnAggArgs {
    // edge attention (GATConv with edge_dim), else null: the logits of launch_gat_edge_logits
    // advanced to this layer's H columns; the neighbor logit adds elog[slot][hd], the self term
    // self_elog[v][hd]
    const float *elog, *self_elog;   // [slots][ldl], [n][ldl]
    int ldl;
};
int launch_gat_agg(const GatAggArgs &a, cudaStream_t s, int *launches);

// Edge terms of GAT's attention logits for every layer and head at once (they do not depend on the
// layer input), once per run.  w_edge [lh][edge_dim], lh = layer * H + head, is lin_edge folded with
// att_edge.  A (sub-)warp per destination row v walks its neighbor slots: elog[slot][lh] =
// sum_j ef[edge_index[slot]][j] w_edge[lh][j] (fp32, ascending j), and self_elog[v][lh] = the mean
// of elog over the row's slots whose source is not v (0 when there is none).  Slots whose source is
// v get 0 and are left out of the mean: the aggregation never uses them.
struct GatEdgeLogitsArgs {
    const float *ef;           // [E][edge_dim], COO edge order
    int edge_dim;
    const float *w_edge;       // [LH][edge_dim]
    int LH;
    const int32_t *offsets, *nbr, *in_deg, *edge_index;
    int n;
    float *elog;               // [E][LH], neighbor-slot order
    float *self_elog;          // [n][LH]
};
int launch_gat_edge_logits(const GatEdgeLogitsArgs &a, int avg_deg, cudaStream_t s, int *launches);

// GATv2 attention aggregation (PyG GATv2Conv, concat heads, inference).  g holds the layer's two
// GEMM outputs per row: xl = x W_l^T + b_l in columns [0, H*C), xr = x W_r^T + b_r in [H*C, 2 H*C).
// Per destination v and head h, over the in-neighbours u != v plus one self term (u = v):
// z = xl_u + xr_v (+ e_uv W_e^T), e_uvh = sum_c att_hc LeakyReLU(z_hc), y_v = act(sum softmax_v(e)
// xl_u + bias (+ skip_v)).  The logit is a dot product over each head's lanes, computed per edge; the
// online softmax, the epilogue and the heavy-row scheme are GAT's (AttnAggArgs).
// a head's columns are spread over at most 32 lanes, each holding at most two VEC-column groups
constexpr int kGatv2MaxHeadWidth = 256;   // C % 4 == 0 (float4 lanes)
constexpr int kGatv2MaxHeadWidth1 = 64;   // other C (scalar lanes)
struct Gatv2AggArgs : AttnAggArgs {
    const float *att;      // [H*C]
    // xr of row v at xr + v * ldxr; null: g + H*C with stride ldg.  The row partition passes the
    // owned rows' xr separately, since only xl crosses ranks.
    const float *xr;
    int ldxr;
    // edge features (edge_dim > 0), else ef_sorted null: the edge term of slot k is
    // ef_sorted[k] W_e^T, the self term's self_attr[v] W_e^T
    const float *ef_sorted;  // [slots][lde], neighbor-slot order
    const float *self_attr;  // [n][lde]
    int lde, edge_dim;
    const float *We_t;       // [edge_dim][ldw] (ldw multiple of 4, zero padded)
    int ldw;
};
int launch_gatv2_agg(const Gatv2AggArgs &a, cudaStream_t s, int *launches);
// self_attr[v][0..lde) = the mean of ef_sorted[k] over the slots k of row v whose source is not v, in
// slot order (0 when there is none); columns past edge_dim are 0
int launch_gatv2_self_attr(const float *ef_sorted, int lde, int edge_dim, const int32_t *offsets,
                           const int32_t *nbr, const int32_t *in_deg, int n, float *self_attr,
                           cudaStream_t s, int *launches);

// TransformerConv attention aggregation (PyG TransformerConv, concat heads, root_weight, inference).
// g holds the source-side GEMM outputs per row: k = x W_k^T + b_k in columns [0, H*C), v = x W_v^T +
// b_v in [H*C, 2 H*C); q holds q = x W_q^T + b_q, already scaled by 1/sqrt(C).  Per destination v and
// head h, over every in-edge u -> v (self loops and duplicates included, no self term):
// ê = e_uv W_e^T (edge features only, else 0), e_uvh = <q_v, k_u + ê>_h, y_v = act(sum softmax_v(e)
// (v_u + ê) + bias (+ skip_v)); a row without in-edges gets act(bias (+ skip_v)).  The model handle
// passes bias = b_skip and skip = x W_skip^T (+ the model's residual).  GATv2's lane layout, head
// width limits and edge projection; GAT's online softmax, epilogue and heavy-row scheme.
struct TransformerAggArgs : AttnAggArgs {
    const float *q;          // [n][ldq]
    int ldq;
    // edge features (edge_dim > 0), else ef_sorted null: the edge term of slot k is ef_sorted[k] W_e^T
    const float *ef_sorted;  // [slots][lde], neighbor-slot order
    int lde, edge_dim;
    const float *We_t;       // [edge_dim][ldw] (ldw multiple of 4, zero padded)
    int ldw;
};
int launch_transformer_agg(const TransformerAggArgs &a, cudaStream_t s, int *launches);

struct PnaAggArgs {
    const float *ab;       // [n][2F]: cols [0,F) = x.W_nbr^T, cols [F,2F) = x.W_self^T + b_pre
    int F;
    float *cat12;          // [n][12F]: (max,min,mean,std) x (identity, amplification, attenuation)
    const int32_t *offsets, *nbr, *in_deg;
    int n;
    float delta;
    int compact;           // 1: write only the [n][4F] statistics (max,min,mean,std); the two degree
                           // scalers are applied by the consumer (gemm_tc.cu expands them on the fly)
};
int launch_pna_agg(const PnaAggArgs &a, cudaStream_t s, int *launches);

// PNA statistics of the owned rows of a row-partitioned graph whose CSR is split by source
// (owned-source part, then halo-source part; neighbor entries are ext indices, bit 31 ignored).
// The message of edge u -> v is t = A_u + B_v with A in ext space: the owned rows' A and the A rows
// the owners sent for the halo.  in_deg is the FULL in-degree of every owned row (mean, std and
// the degree scalers).  Output as PnaAggArgs::cat12 / compact.
struct PnaHaloArgs {
    const float *a_ext;    // [n_ext][F]  A = x.W_nbr^T
    const float *b;        // [n][F]      B = x.W_self^T + b_pre (owned rows)
    int F;
    float *cat12;          // [n][12F], or [n][4F] when compact
    const int32_t *own_off, *own_cnt, *own_nbr, *halo_off, *halo_cnt, *halo_nbr, *in_deg;
    int n;
    float delta;
    int compact;
};
int launch_pna_halo_stats(const PnaHaloArgs &a, cudaStream_t s, int *launches);

// ---------------------------------------------------------------- GEMM (gemm.cu)
// C[M][N] = act( A1[M][K1].W1t[K1][N] (+ A2[M][K2].W2t[K2][N]) + bias (+ skip) )
// weights are pre-transposed: Wt[k][n], row stride ldw (multiple of 4, zero padded)
struct GemmArgs {
    const float *A1; int lda1; int K1; const float *W1t; int ldw1;
    const float *A2; int lda2; int K2; const float *W2t; int ldw2;
    const float *img1, *img2;   // optional tensor-core weight images of W1 / W2 (gemm_tc.cu); when
                                // present (and FAST math) the GEMM runs on tcgen05, else on the FMA pipe
    // PNA "expand" mode (tensor-core path only): A2 holds the [M][K2/3] statistics and stands for
    // [A2 | amp_v A2 | att_v A2] (lib:1857-1875), amp_v = log(max(deg_v,1)+1)/delta, att_v = 1/amp_v
    const int32_t *expand_deg; float expand_delta;
    int second_separate;        // STRICT only: A2.W2t is a separate bias-free sum added last (SAGE)
    const float *bias;          // [N] or null
    const float *skip; int ldskip;  // added before the activation, or null
    int act;
    float *C; int ldc;
    int M; int N;
};
int launch_gemm(const GemmArgs &g, bool strict, cudaStream_t s, int *launches);
// gemm_tc.cu: tcgen05 (3xTF32) version of the same contract, for large M
size_t gemm_tc_image_floats(int K, int N);
int gemm_tc_build_image(const float *Wt, int ldw, int K, int N, float *img, cudaStream_t s);
bool gemm_tc_supported(const GemmArgs &g);
int launch_gemm_tc(const GemmArgs &g, cudaStream_t s, int *launches);
// Wt[k][n] (ld = ldw) from W[n][k] (reference layout); pads columns n..ldw with zeros.
// ld_src: row stride of W when it is a column block of a wider matrix (0: in_size)
int launch_transpose_weight(const float *W, float *Wt, int out_size, int in_size, int ldw,
                            cudaStream_t s, int *launches, int ld_src = 0);

// ---------------------------------------------------------------- pooling / misc (pool.cu)
// pooled[g][p*F + f] for pools[p] over rows node_ptr[g]..node_ptr[g+1]
int launch_pool(const float *x, int ldx, int F, const int64_t *node_ptr, int64_t node_base,
                int n_graphs, int64_t total_nodes, const int *pools, int num_pools, float *pooled,
                DeviceBuf &tmp, cudaStream_t s, int *launches, bool single_pass = false);
int launch_activation(int act, const float *x, float *y, size_t n, cudaStream_t s, int *launches);

}  // namespace gnnb
