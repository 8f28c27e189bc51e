// Layer-function entry points: the C-ABI twins of the reference's template functions
// (gnn_builder_lib.h), same argument order and array layouts, dimensions as runtime ints.
// They exist so that every function of the hot path can be parity-tested in isolation against
// the reference; each call stages host buffers, runs the same kernels the model path uses on
// the default stream, and returns when the results are back.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "kernels.h"

namespace gnnb {

bool is_device_pointer(const void *p);

namespace {

// Maps caller buffers (host or device) to device pointers for the duration of one call.
class Stage {
  public:
    ~Stage()
    {
        for (void *p : owned_) cudaFree(p);
    }
    template <typename T>
    int in(const T *p, size_t count, const T **dev)
    {
        *dev = nullptr;
        if (p == nullptr || count == 0) { *dev = p; return GNNB_OK; }
        if (is_device_pointer(p)) { *dev = p; return GNNB_OK; }
        void *d = nullptr;
        GNNB_CUDA(cudaMalloc(&d, count * sizeof(T)));
        owned_.push_back(d);
        GNNB_CUDA(cudaMemcpy(d, p, count * sizeof(T), cudaMemcpyHostToDevice));
        *dev = static_cast<const T *>(d);
        return GNNB_OK;
    }
    template <typename T>
    int out(T *p, size_t count, T **dev)
    {
        *dev = nullptr;
        if (p == nullptr || count == 0) { *dev = p; return GNNB_OK; }
        if (is_device_pointer(p)) { *dev = p; return GNNB_OK; }
        void *d = nullptr;
        GNNB_CUDA(cudaMalloc(&d, count * sizeof(T)));
        owned_.push_back(d);
        back_.push_back({p, d, count * sizeof(T)});
        *dev = static_cast<T *>(d);
        return GNNB_OK;
    }
    template <typename T>
    int scratch(size_t count, T **dev)
    {
        void *d = nullptr;
        GNNB_CUDA(cudaMalloc(&d, (count ? count : 1) * sizeof(T)));
        owned_.push_back(d);
        *dev = static_cast<T *>(d);
        return GNNB_OK;
    }
    // tensor-core weight images built by pack_weight, looked up by the packed-weight pointer
    void add_image(const float *Wt, const float *img) { images_.push_back({Wt, img}); }
    const float *image_of(const float *Wt) const
    {
        for (const auto &p : images_)
            if (p.first == Wt) return p.second;
        return nullptr;
    }
    // device int the table kernels set when an edge endpoint is outside [0, num_nodes)
    int bad_flag(int **flag)
    {
        GNNB_TRY(scratch(1, &bad_));
        GNNB_CUDA(cudaMemset(bad_, 0, sizeof(int)));
        *flag = bad_;
        return GNNB_OK;
    }
    int finish()
    {
        GNNB_CUDA(cudaDeviceSynchronize());
        if (bad_ != nullptr) {
            int bad = 0;
            GNNB_CUDA(cudaMemcpy(&bad, bad_, sizeof(int), cudaMemcpyDeviceToHost));
            GNNB_REQUIRE(bad == 0, "edge_list holds a node index outside [0, num_nodes)");
        }
        for (const Back &b : back_) GNNB_CUDA(cudaMemcpy(b.host, b.dev, b.bytes, cudaMemcpyDeviceToHost));
        return GNNB_OK;
    }

  private:
    struct Back { void *host; void *dev; size_t bytes; };
    std::vector<void *> owned_;
    std::vector<Back> back_;
    std::vector<std::pair<const float *, const float *>> images_;
    int *bad_ = nullptr;
};

struct TempWs {
    TableWorkspace ws;
    ~TempWs() { ws.release_all(); }
};

// W[out][in] (reference layout, host or device) -> packed Wt[in][ldw] on the device
int pack_weight(Stage &st, const float *W, int out, int in, const float **Wt, int *ldw)
{
    const float *dW;
    GNNB_TRY(st.in(W, (size_t)out * in, &dW));
    float *t;
    *ldw = round_up(out, 4);
    GNNB_TRY(st.scratch((size_t)in * *ldw, &t));
    GNNB_TRY(launch_transpose_weight(dW, t, out, in, *ldw, 0, nullptr));
    *Wt = t;
    float *img;   // the same weight as a tensor-core image (used by the GEMM when M is large)
    GNNB_TRY(st.scratch(gemm_tc_image_floats(in, out), &img));
    GNNB_TRY(gemm_tc_build_image(t, *ldw, in, out, img, 0));
    st.add_image(t, img);
    return GNNB_OK;
}

// launch_gemm with the tensor-core images of the staged weights attached
int stage_gemm(const Stage &st, GemmArgs g, bool strict)
{
    g.img1 = st.image_of(g.W1t);
    g.img2 = g.W2t != nullptr ? st.image_of(g.W2t) : nullptr;
    return launch_gemm(g, strict, 0, nullptr);
}

GemmArgs simple_gemm(const float *A, int lda, int K, const float *Wt, int ldw, const float *bias,
                     float *C, int ldc, int M, int N, int act)
{
    GemmArgs g{};
    g.A1 = A; g.lda1 = lda; g.K1 = K; g.W1t = Wt; g.ldw1 = ldw;
    g.ldw2 = 4;
    g.bias = bias; g.act = act; g.C = C; g.ldc = ldc; g.M = M; g.N = N;
    return g;
}

struct ConvCommon {
    const float *x; float *y; const int32_t *off, *nbr, *ind;
};

int stage_conv(Stage &st, int n, int e, const float *x_in, float *x_out, const int32_t *offsets,
               const int32_t *nbr, const int32_t *in_deg, int fi, int fo, ConvCommon *c)
{
    GNNB_REQUIRE(n >= 0 && e >= 0 && fi > 0 && fo > 0, "bad conv dimensions");
    GNNB_TRY(st.in(x_in, (size_t)n * fi, &c->x));
    GNNB_TRY(st.out(x_out, (size_t)n * fo, &c->y));
    GNNB_TRY(st.in(offsets, (size_t)n, &c->off));
    GNNB_TRY(st.in(nbr, (size_t)e, &c->nbr));
    GNNB_TRY(st.in(in_deg, (size_t)n, &c->ind));
    return GNNB_OK;
}

int pool_common(int kind, int n, const float *x, float *pooled, int emb)
{
    GNNB_REQUIRE(n >= 0 && emb > 0 && pooled != nullptr, "bad pooling arguments");
    Stage st;
    const float *dx;
    float *dp;
    GNNB_TRY(st.in(x, (size_t)n * emb, &dx));
    GNNB_TRY(st.out(pooled, (size_t)emb, &dp));
    int64_t *np;
    GNNB_TRY(st.scratch(2, &np));
    const int64_t h[2] = {0, n};
    GNNB_CUDA(cudaMemcpy(np, h, sizeof(h), cudaMemcpyHostToDevice));
    DeviceBuf tmp;
    const int pools[1] = {kind};
    int rc = launch_pool(dx, emb, emb, np, 0, 1, n, pools, 1, dp, tmp, 0, nullptr);
    if (rc == GNNB_OK) rc = st.finish();
    tmp.release();
    return rc;
}

}  // namespace
}  // namespace gnnb

using namespace gnnb;

extern "C" int gnnb_compute_degree_tables(const int32_t *edge_list, int32_t *in_degree_table,
                                          int32_t *out_degree_table, int num_nodes, int num_edges)
{
    GNNB_REQUIRE(num_nodes >= 0 && num_edges >= 0, "negative size");
    Stage st;
    const int32_t *coo;
    int32_t *ind, *outd;
    GNNB_TRY(st.in(edge_list, 2 * (size_t)num_edges, &coo));
    GNNB_TRY(st.out(in_degree_table, (size_t)num_nodes, &ind));
    GNNB_TRY(st.out(out_degree_table, (size_t)num_nodes, &outd));
    int *bad;
    GNNB_TRY(st.bad_flag(&bad));
    GNNB_TRY(build_degree_tables(coo, num_nodes, num_edges, ind, outd, 0, nullptr, bad));
    return st.finish();
}

extern "C" int gnnb_compute_neighbor_and_edge_index_tables(
    const int32_t *edge_list, const int32_t *in_degree_table, const int32_t *out_degree_table,
    int32_t *neighbor_table_offsets, int32_t *neighbor_table, int32_t *edge_index_table,
    int num_nodes, int num_edges)
{
    (void)out_degree_table;  // threaded through by the reference but never read (lib:1086-1166)
    GNNB_REQUIRE(num_nodes >= 0 && num_edges >= 0, "negative size");
    Stage st;
    TempWs t;
    const int32_t *coo, *ind;
    int32_t *off, *nbr, *eidx = nullptr;
    GNNB_TRY(st.in(edge_list, 2 * (size_t)num_edges, &coo));
    GNNB_TRY(st.in(in_degree_table, (size_t)num_nodes, &ind));
    GNNB_TRY(st.out(neighbor_table_offsets, (size_t)num_nodes, &off));
    GNNB_TRY(st.out(neighbor_table, (size_t)num_edges, &nbr));
    if (edge_index_table) GNNB_TRY(st.out(edge_index_table, (size_t)num_edges, &eidx));
    int *bad;
    GNNB_TRY(st.bad_flag(&bad));
    GNNB_TRY(build_neighbor_tables(coo, ind, num_nodes, num_edges, off, nbr, eidx, t.ws, 0, nullptr, bad));
    return st.finish();
}

extern "C" int gnnb_compute_neighbor_tables(const int32_t *edge_list, const int32_t *in_degree_table,
                                            const int32_t *out_degree_table,
                                            int32_t *neighbor_table_offsets, int32_t *neighbor_table,
                                            int num_nodes, int num_edges)
{
    return gnnb_compute_neighbor_and_edge_index_tables(edge_list, in_degree_table, out_degree_table,
                                                       neighbor_table_offsets, neighbor_table,
                                                       nullptr, num_nodes, num_edges);
}

extern "C" int gnnb_linear(const float *x, float *y, const float *weight, const float *bias,
                           int rows, int in_size, int out_size, int math)
{
    GNNB_REQUIRE(rows >= 0 && in_size > 0 && out_size > 0, "bad linear dimensions");
    Stage st;
    const float *dx, *db, *Wt;
    float *dy;
    int ldw;
    GNNB_TRY(st.in(x, (size_t)rows * in_size, &dx));
    GNNB_TRY(st.in(bias, (size_t)out_size, &db));
    GNNB_TRY(st.out(y, (size_t)rows * out_size, &dy));
    GNNB_TRY(pack_weight(st, weight, out_size, in_size, &Wt, &ldw));
    GemmArgs g = simple_gemm(dx, in_size, in_size, Wt, ldw, db, dy, out_size, rows, out_size,
                             GNNB_ACT_IDENTITY);
    GNNB_TRY(stage_gemm(st, g, math == GNNB_MATH_STRICT));
    return st.finish();
}

extern "C" int gnnb_apply_activation(int act, const float *x, float *y, size_t n)
{
    GNNB_REQUIRE(act >= 0 && act <= GNNB_ACT_COS, "unknown activation");
    Stage st;
    const float *dx;
    float *dy;
    GNNB_TRY(st.in(x, n, &dx));
    GNNB_TRY(st.out(y, n, &dy));
    GNNB_TRY(launch_activation(act, dx, dy, n, 0, nullptr));
    return st.finish();
}

extern "C" int gnnb_gcn_conv(int num_nodes, int num_edges, const float *x_in, float *x_out,
                             const int32_t *edge_list, const int32_t *neighbor_table_offsets,
                             const int32_t *neighbor_table, const int32_t *in_degree_table,
                             const int32_t *out_degree_table, const float *weight, const float *bias,
                             int emb_in, int emb_out, int math)
{
    (void)edge_list; (void)out_degree_table;  // unused by the reference body as well
    const bool strict = math == GNNB_MATH_STRICT;
    Stage st;
    ConvCommon c;
    GNNB_TRY(stage_conv(st, num_nodes, num_edges, x_in, x_out, neighbor_table_offsets,
                        neighbor_table, in_degree_table, emb_in, emb_out, &c));
    const float *Wt, *db;
    int ldw;
    GNNB_TRY(pack_weight(st, weight, emb_out, emb_in, &Wt, &ldw));
    GNNB_TRY(st.in(bias, (size_t)emb_out, &db));
    float *agg, *dinv = nullptr;
    const int lda = round_up(emb_in, 4);
    GNNB_TRY(st.scratch((size_t)num_nodes * lda, &agg));
    if (!strict) {
        GNNB_TRY(st.scratch((size_t)num_nodes, &dinv));
        GNNB_TRY(compute_dinv(c.ind, dinv, num_nodes, 0, nullptr));
    }
    AggArgs a{};
    a.mode = AGG_GCN; a.x = c.x; a.ldx = emb_in; a.F = emb_in; a.out = agg; a.ldo = lda;
    a.offsets = c.off; a.nbr = c.nbr; a.in_deg = c.ind; a.dinv = dinv; a.n = num_nodes;
    GNNB_TRY(launch_agg(a, strict, 0, nullptr));
    GemmArgs g = simple_gemm(agg, lda, emb_in, Wt, ldw, db, c.y, emb_out, num_nodes, emb_out,
                             GNNB_ACT_IDENTITY);
    GNNB_TRY(stage_gemm(st, g, strict));
    return st.finish();
}

extern "C" int gnnb_gin_conv(int num_nodes, int num_edges, const float *x_in, float *x_out,
                             const int32_t *edge_list, const int32_t *neighbor_table_offsets,
                             const int32_t *neighbor_table, const int32_t *in_degree_table,
                             const int32_t *out_degree_table, const float *mlp_0_weight,
                             const float *mlp_0_bias, const float *mlp_1_weight,
                             const float *mlp_1_bias, float gin_eps, int emb_in, int hidden,
                             int emb_out, int math)
{
    (void)edge_list; (void)out_degree_table;
    GNNB_REQUIRE(hidden > 0, "bad hidden size");
    const bool strict = math == GNNB_MATH_STRICT;
    Stage st;
    ConvCommon c;
    GNNB_TRY(stage_conv(st, num_nodes, num_edges, x_in, x_out, neighbor_table_offsets,
                        neighbor_table, in_degree_table, emb_in, emb_out, &c));
    const float *W0t, *W1t, *b0, *b1;
    int ld0, ld1;
    GNNB_TRY(pack_weight(st, mlp_0_weight, hidden, emb_in, &W0t, &ld0));
    GNNB_TRY(pack_weight(st, mlp_1_weight, emb_out, hidden, &W1t, &ld1));
    GNNB_TRY(st.in(mlp_0_bias, (size_t)hidden, &b0));
    GNNB_TRY(st.in(mlp_1_bias, (size_t)emb_out, &b1));
    float *agg, *hid;
    const int lda = round_up(emb_in, 4), ldh = round_up(hidden, 4);
    GNNB_TRY(st.scratch((size_t)num_nodes * lda, &agg));
    GNNB_TRY(st.scratch((size_t)num_nodes * ldh, &hid));
    AggArgs a{};
    a.mode = AGG_GIN; a.x = c.x; a.ldx = emb_in; a.F = emb_in; a.out = agg; a.ldo = lda;
    a.offsets = c.off; a.nbr = c.nbr; a.in_deg = c.ind; a.n = num_nodes; a.eps = gin_eps;
    GNNB_TRY(launch_agg(a, strict, 0, nullptr));
    GemmArgs g0 = simple_gemm(agg, lda, emb_in, W0t, ld0, b0, hid, ldh, num_nodes, hidden,
                              GNNB_ACT_RELU);
    GNNB_TRY(stage_gemm(st, g0, strict));
    GemmArgs g1 = simple_gemm(hid, ldh, hidden, W1t, ld1, b1, c.y, emb_out, num_nodes, emb_out,
                              GNNB_ACT_IDENTITY);
    GNNB_TRY(stage_gemm(st, g1, strict));
    return st.finish();
}

extern "C" int gnnb_sage_conv(int num_nodes, int num_edges, const float *x_in, float *x_out,
                              const int32_t *edge_list, const int32_t *neighbor_table_offsets,
                              const int32_t *neighbor_table, const int32_t *in_degree_table,
                              const int32_t *out_degree_table, const float *neighbor_lin_weight,
                              const float *neighbor_lin_bias, const float *self_lin_weight,
                              int emb_in, int emb_out, int math)
{
    (void)edge_list; (void)out_degree_table;
    const bool strict = math == GNNB_MATH_STRICT;
    Stage st;
    ConvCommon c;
    GNNB_TRY(stage_conv(st, num_nodes, num_edges, x_in, x_out, neighbor_table_offsets,
                        neighbor_table, in_degree_table, emb_in, emb_out, &c));
    const float *Wlt, *Wrt, *bl;
    int ldl, ldr;
    GNNB_TRY(pack_weight(st, neighbor_lin_weight, emb_out, emb_in, &Wlt, &ldl));
    GNNB_TRY(pack_weight(st, self_lin_weight, emb_out, emb_in, &Wrt, &ldr));
    GNNB_TRY(st.in(neighbor_lin_bias, (size_t)emb_out, &bl));
    float *agg;
    const int lda = round_up(emb_in, 4);
    GNNB_TRY(st.scratch((size_t)num_nodes * lda, &agg));
    AggArgs a{};
    a.mode = AGG_MEAN; a.x = c.x; a.ldx = emb_in; a.F = emb_in; a.out = agg; a.ldo = lda;
    a.offsets = c.off; a.nbr = c.nbr; a.in_deg = c.ind; a.n = num_nodes;
    GNNB_TRY(launch_agg(a, strict, 0, nullptr));
    GemmArgs g = simple_gemm(agg, lda, emb_in, Wlt, ldl, bl, c.y, emb_out, num_nodes, emb_out,
                             GNNB_ACT_IDENTITY);
    g.A2 = c.x; g.lda2 = emb_in; g.K2 = emb_in; g.W2t = Wrt; g.ldw2 = ldr;
    g.second_separate = 1;
    GNNB_TRY(stage_gemm(st, g, strict));
    return st.finish();
}

// lib:1627-1742 gine_conv: per-edge projection of the edge features (one GEMM over the edges),
// gather-reduce of relu(x_u + proj_e) in neighbor-table order, then the GIN MLP.
extern "C" int gnnb_gine_conv(int num_nodes, int num_edges, const float *x_in, float *x_out,
                              const float *edge_feature_table, const int32_t *edge_list,
                              const int32_t *neighbor_table_offsets, const int32_t *neighbor_table,
                              const int32_t *edge_index_table, const int32_t *in_degree_table,
                              const int32_t *out_degree_table, const float *edge_proj_weight,
                              const float *edge_proj_bias, const float *mlp_0_weight,
                              const float *mlp_0_bias, const float *mlp_1_weight,
                              const float *mlp_1_bias, float gin_eps, int emb_in, int hidden,
                              int emb_out, int edge_dim, int math)
{
    (void)edge_list; (void)out_degree_table;
    GNNB_REQUIRE(hidden > 0 && edge_dim > 0, "bad hidden / edge feature size");
    const bool strict = math == GNNB_MATH_STRICT;
    Stage st;
    ConvCommon c;
    GNNB_TRY(stage_conv(st, num_nodes, num_edges, x_in, x_out, neighbor_table_offsets,
                        neighbor_table, in_degree_table, emb_in, emb_out, &c));
    const float *ef;
    const int32_t *eidx;
    GNNB_TRY(st.in(edge_feature_table, (size_t)num_edges * edge_dim, &ef));
    GNNB_TRY(st.in(edge_index_table, (size_t)num_edges, &eidx));
    const float *Wet, *W0t, *W1t, *be, *b0, *b1;
    int lde, ld0, ld1;
    GNNB_TRY(pack_weight(st, edge_proj_weight, emb_in, edge_dim, &Wet, &lde));
    GNNB_TRY(pack_weight(st, mlp_0_weight, hidden, emb_in, &W0t, &ld0));
    GNNB_TRY(pack_weight(st, mlp_1_weight, emb_out, hidden, &W1t, &ld1));
    GNNB_TRY(st.in(edge_proj_bias, (size_t)emb_in, &be));
    GNNB_TRY(st.in(mlp_0_bias, (size_t)hidden, &b0));
    GNNB_TRY(st.in(mlp_1_bias, (size_t)emb_out, &b1));
    float *proj, *agg, *hid;
    const int lda = round_up(emb_in, 4), ldh = round_up(hidden, 4);
    GNNB_TRY(st.scratch((size_t)std::max(num_edges, 1) * lda, &proj));
    GNNB_TRY(st.scratch((size_t)num_nodes * lda, &agg));
    GNNB_TRY(st.scratch((size_t)num_nodes * ldh, &hid));
    if (num_edges > 0) {
        GemmArgs ge = simple_gemm(ef, edge_dim, edge_dim, Wet, lde, be, proj, lda, num_edges, emb_in,
                                  GNNB_ACT_IDENTITY);
        GNNB_TRY(stage_gemm(st, ge, strict));
    }
    GineAggArgs a{};
    a.x = c.x; a.ldx = emb_in; a.F = emb_in; a.proj = proj; a.ldp = lda; a.out = agg; a.ldo = lda;
    a.offsets = c.off; a.nbr = c.nbr; a.edge_index = eidx; a.in_deg = c.ind; a.n = num_nodes;
    a.eps = gin_eps;
    GNNB_TRY(launch_gine_agg(a, 0, nullptr));
    GemmArgs g0 = simple_gemm(agg, lda, emb_in, W0t, ld0, b0, hid, ldh, num_nodes, hidden,
                              GNNB_ACT_RELU);
    GNNB_TRY(stage_gemm(st, g0, strict));
    GemmArgs g1 = simple_gemm(hid, ldh, hidden, W1t, ld1, b1, c.y, emb_out, num_nodes, emb_out,
                              GNNB_ACT_IDENTITY);
    GNNB_TRY(stage_gemm(st, g1, strict));
    return st.finish();
}

// lib:2350-2499 lg_conv (LightGCN propagation, no weights) and lib:2501-2634 simple_conv (plain
// neighbor sum): the aggregation kernel alone.
static int agg_only_conv(int mode, int num_nodes, int num_edges, const float *x_in, float *x_out,
                         const int32_t *offsets, const int32_t *nbr, const int32_t *in_deg, int emb,
                         int math)
{
    Stage st;
    ConvCommon c;
    GNNB_TRY(stage_conv(st, num_nodes, num_edges, x_in, x_out, offsets, nbr, in_deg, emb, emb, &c));
    AggArgs a{};
    a.mode = mode; a.x = c.x; a.ldx = emb; a.F = emb; a.out = c.y; a.ldo = emb;
    a.offsets = c.off; a.nbr = c.nbr; a.in_deg = c.ind; a.n = num_nodes;
    GNNB_TRY(launch_agg(a, math == GNNB_MATH_STRICT, 0, nullptr));
    return st.finish();
}

extern "C" int gnnb_lg_conv(int num_nodes, int num_edges, const float *x_in, float *x_out,
                            const int32_t *edge_list, const int32_t *neighbor_table_offsets,
                            const int32_t *neighbor_table, const int32_t *in_degree_table,
                            const int32_t *out_degree_table, int emb, int math)
{
    (void)edge_list; (void)out_degree_table;
    return agg_only_conv(AGG_LG, num_nodes, num_edges, x_in, x_out, neighbor_table_offsets,
                         neighbor_table, in_degree_table, emb, math);
}

extern "C" int gnnb_simple_conv(int num_nodes, int num_edges, const float *x_in, float *x_out,
                                const int32_t *edge_list, const int32_t *neighbor_table_offsets,
                                const int32_t *neighbor_table, const int32_t *in_degree_table,
                                const int32_t *out_degree_table, int emb, int math)
{
    (void)edge_list; (void)out_degree_table;
    return agg_only_conv(AGG_SUM, num_nodes, num_edges, x_in, x_out, neighbor_table_offsets,
                         neighbor_table, in_degree_table, emb, math);
}

extern "C" int gnnb_pna_conv(int num_nodes, int num_edges, const float *x_in, float *x_out,
                             const int32_t *edge_list, const int32_t *neighbor_table_offsets,
                             const int32_t *neighbor_table, const int32_t *in_degree_table,
                             const int32_t *out_degree_table, const float *transform_lin_weight,
                             const float *transform_lin_bias, const float *apply_lin_weight,
                             const float *apply_lin_bias, const float *final_lin_weight,
                             const float *final_lin_bias, float pna_avg_degree_log, int emb_in,
                             int emb_out)
{
    (void)edge_list; (void)out_degree_table;
    Stage st;
    ConvCommon c;
    GNNB_TRY(stage_conv(st, num_nodes, num_edges, x_in, x_out, neighbor_table_offsets,
                        neighbor_table, in_degree_table, emb_in, emb_out, &c));
    const int F = emb_in, n = num_nodes;
    // host-side split of W_pre = [W_self | W_nbr] needs the weights on the host
    std::vector<float> wpre((size_t)F * 2 * F), bpre(F), wpost((size_t)emb_out * 13 * F);
    auto fetch = [](const float *src, float *dst, size_t cnt) -> int {
        GNNB_CUDA(cudaMemcpy(dst, src, cnt * sizeof(float), cudaMemcpyDefault));
        return GNNB_OK;
    };
    GNNB_TRY(fetch(transform_lin_weight, wpre.data(), wpre.size()));
    GNNB_TRY(fetch(transform_lin_bias, bpre.data(), bpre.size()));
    GNNB_TRY(fetch(apply_lin_weight, wpost.data(), wpost.size()));
    const int ld_ab = round_up(2 * F, 4), ld_o = round_up(emb_out, 4);
    std::vector<float> wab((size_t)F * ld_ab, 0.0f), bab((size_t)2 * F, 0.0f);
    std::vector<float> wself((size_t)F * ld_o, 0.0f), wagg((size_t)12 * F * ld_o, 0.0f);
    for (int k = 0; k < F; k++)
        for (int o = 0; o < F; o++) {
            wab[(size_t)k * ld_ab + o] = wpre[(size_t)o * 2 * F + F + k];      // W_nbr^T
            wab[(size_t)k * ld_ab + F + o] = wpre[(size_t)o * 2 * F + k];      // W_self^T
        }
    for (int o = 0; o < F; o++) bab[F + o] = bpre[o];
    for (int o = 0; o < emb_out; o++) {
        for (int k = 0; k < F; k++) wself[(size_t)k * ld_o + o] = wpost[(size_t)o * 13 * F + k];
        for (int k = 0; k < 12 * F; k++) wagg[(size_t)k * ld_o + o] = wpost[(size_t)o * 13 * F + F + k];
    }
    const float *d_wab, *d_bab, *d_wself, *d_wagg, *d_bpost, *d_blin, *Wlint;
    int ldlin;
    GNNB_TRY(st.in(wab.data(), wab.size(), &d_wab));
    GNNB_TRY(st.in(bab.data(), bab.size(), &d_bab));
    GNNB_TRY(st.in(wself.data(), wself.size(), &d_wself));
    GNNB_TRY(st.in(wagg.data(), wagg.size(), &d_wagg));
    GNNB_TRY(st.in(apply_lin_bias, (size_t)emb_out, &d_bpost));
    GNNB_TRY(st.in(final_lin_bias, (size_t)emb_out, &d_blin));
    GNNB_TRY(pack_weight(st, final_lin_weight, emb_out, emb_out, &Wlint, &ldlin));
    float *ab, *cat12, *hid;
    GNNB_TRY(st.scratch((size_t)n * 2 * F + 4, &ab));
    GNNB_TRY(st.scratch((size_t)n * 12 * F + 4, &cat12));
    GNNB_TRY(st.scratch((size_t)n * ld_o, &hid));
    GemmArgs g0 = simple_gemm(c.x, F, F, d_wab, ld_ab, d_bab, ab, 2 * F, n, 2 * F, GNNB_ACT_IDENTITY);
    GNNB_TRY(stage_gemm(st, g0, false));
    PnaAggArgs pa{};
    pa.ab = ab; pa.F = F; pa.cat12 = cat12; pa.offsets = c.off; pa.nbr = c.nbr; pa.in_deg = c.ind;
    pa.n = n; pa.delta = pna_avg_degree_log;
    GNNB_TRY(launch_pna_agg(pa, 0, nullptr));
    GemmArgs g1 = simple_gemm(c.x, F, F, d_wself, ld_o, d_bpost, hid, ld_o, n, emb_out,
                              GNNB_ACT_IDENTITY);
    g1.A2 = cat12; g1.lda2 = 12 * F; g1.K2 = 12 * F; g1.W2t = d_wagg; g1.ldw2 = ld_o;
    GNNB_TRY(stage_gemm(st, g1, false));
    GemmArgs g2 = simple_gemm(hid, ld_o, emb_out, Wlint, ldlin, d_blin, c.y, emb_out, n, emb_out,
                              GNNB_ACT_IDENTITY);
    GNNB_TRY(stage_gemm(st, g2, false));
    return st.finish();
}

extern "C" int gnnb_global_add_pool(int num_nodes, int num_edges, const float *x, float *pooled,
                                    int emb)
{
    (void)num_edges;
    return pool_common(GNNB_POOL_ADD, num_nodes, x, pooled, emb);
}
extern "C" int gnnb_global_mean_pool(int num_nodes, int num_edges, const float *x, float *pooled,
                                     int emb)
{
    (void)num_edges;
    return pool_common(GNNB_POOL_MEAN, num_nodes, x, pooled, emb);
}
extern "C" int gnnb_global_max_pool(int num_nodes, int num_edges, const float *x, float *pooled,
                                    int emb)
{
    (void)num_edges;
    return pool_common(GNNB_POOL_MAX, num_nodes, x, pooled, emb);
}

// ============================================================================ row partition
// One large graph split by destination rows across GPUs (SURVEY 8e; the reference has no
// counterpart: it holds one graph in static MAX_NODES arrays).  All pointers are DEVICE pointers
// and the work is enqueued on `stream` (e.g. torch's current stream) so that it orders with the
// NCCL all-gather of the feature shards issued on the same stream.
namespace {
// rows above the heavy threshold of one CSR (part), cached by the address of its row-length table
struct HeavyCache {
    const int32_t *key = nullptr;
    int n = 0;
    HeavyList list;
};
// a weight in the reference layout, transposed for the GEMM on every call (so the caller may
// change it between calls) plus its tensor-core image
struct DevWeight {
    DeviceBuf wt, img;
    int ldw = 4;
};
struct PartitionCache {
    TableWorkspace ws;
    DeviceBuf agg, hid, pna_b, pna_stats, pool_tmp, pool_ptr;
    DeviceBuf gat_w;      // GAT: [W | w_src | w_dst], folded on every call
    DeviceBuf gatv2_xr;   // GATv2: xr of the owned rows, from phase 1 to phase 2
    DevWeight w[5];       // the weights of the layer being computed
    int64_t pool_n = -1;
    HeavyCache whole;     // gnnb_gcn_conv_partition (one CSR)
    HeavyCache part[32];  // owned-source / halo-source parts of a split CSR, per row block
    int part_next = 0;
};
thread_local PartitionCache g_part;

int heavy_rows_of(HeavyCache &hc, const int32_t *lengths, int n, cudaStream_t s)
{
    if (hc.key == lengths && hc.n == n) return GNNB_OK;
    GNNB_TRY(find_heavy_rows(lengths, n, heavy_threshold(), g_part.ws, hc.list, s, nullptr));
    hc.key = lengths;
    hc.n = n;
    return GNNB_OK;
}

// W[out][in] (device, row stride ld_src, 0 = in) -> dw.wt [in][ldw] and its tensor-core image
int dev_weight(DevWeight &dw, const float *W, int out, int in, int ld_src, cudaStream_t s)
{
    dw.ldw = round_up(out, 4);
    GNNB_TRY(dw.wt.ensure(sizeof(float) * (size_t)in * dw.ldw));
    GNNB_TRY(launch_transpose_weight(W, dw.wt.as<float>(), out, in, dw.ldw, s, nullptr, ld_src));
    GNNB_TRY(dw.img.ensure(sizeof(float) * gemm_tc_image_floats(in, out)));
    GNNB_TRY(gemm_tc_build_image(dw.wt.as<float>(), dw.ldw, in, out, dw.img.as<float>(), s));
    return GNNB_OK;
}

// heavy-row list of one part of a split CSR, cached by its row-length table and row count
HeavyCache &part_cache(const int32_t *lengths, int n)
{
    for (HeavyCache &hc : g_part.part)
        if (hc.key == lengths && hc.n == n) return hc;
    HeavyCache &hc = g_part.part[g_part.part_next];
    g_part.part_next = (g_part.part_next + 1) % 32;
    hc.key = nullptr;
    return hc;
}

// One part (owned-source or halo-source edges) of a split CSR through the aggregation kernels
// for rows [row_begin, row_begin + row_count) of `a` (whose out / n / row_base address that
// block), with the heavy rows of the part bucketed.  in_deg: the full in-degree of the owned
// rows, for the modes that read it (mean); null passes the part's lengths as the degree, which
// is all GCN (full degree through dinv) and GIN read.
int halo_agg_part(const AggArgs &a, const int32_t *off, const int32_t *cnt, const int32_t *nbr,
                  const int32_t *in_deg, bool accumulate, bool finish, int row_begin, int row_count,
                  cudaStream_t s)
{
    HeavyCache &hc = part_cache(cnt + row_begin, row_count);
    GNNB_TRY(heavy_rows_of(hc, cnt + row_begin, row_count, s));
    GNNB_TRY(heavy_setup(g_part.ws, hc.list.n_chunks, a.F));
    AggArgs b = a;
    b.offsets = off + row_begin; b.nbr = nbr;
    if (in_deg != nullptr) {
        b.in_deg = in_deg + row_begin;
        b.counts = cnt + row_begin;
    } else {
        b.in_deg = cnt + row_begin;
    }
    b.heavy.set(hc.list, g_part.ws.heavy_partial.as<float>());
    b.accumulate = accumulate ? 1 : 0; b.no_finish = finish ? 0 : 1;
    return launch_agg(b, false, s, nullptr);
}

// argument checks shared by the split-CSR layer entry points (before any device work)
int check_halo_args(int n_local, int n_ext, int emb_in, int emb_out, int act, int phase)
{
    GNNB_REQUIRE(n_local >= 0 && n_ext >= n_local, "bad row counts");
    GNNB_REQUIRE(emb_in > 0 && emb_out > 0 && act >= 0 && act <= GNNB_ACT_COS, "bad dims");
    GNNB_REQUIRE(phase >= 1 && phase <= 3, "phase: 1 owned-source edges, 2 halo edges + transform, 3 both");
    return GNNB_OK;
}
}  // namespace

// ---- halo exchange kernels ---------------------------------------------------------------
namespace gnnb {
namespace halo {
constexpr int kMaxPeers = 16;
struct PackArgs {
    const float *x;
    int ldx, F, n_peers;
    const int32_t *send_idx;
    long long start[kMaxPeers], count[kMaxPeers];   // rows for peer p: send_idx[start[p] .. +count[p])
    float *dst[kMaxPeers];          // where row i of that range goes: dst[p] + i F (a local send
                                    // buffer or the peer's halo region)
};
// A warp moves PACK_ROWS rows per iteration: all their loads are issued before the first store, so
// every warp keeps PACK_ROWS x 512 bytes (F = 128) in flight and a grid of ONE CTA per SM already
// holds several MB -- enough for the ~670 GB/s one NVLink direction delivers -- while leaving the
// other seven CTA slots of every SM to the aggregation kernel that runs beside it.  16-byte
// accesses when F % 4 == 0, so a row leaves the SM as one coalesced 512-byte write (over NVLink
// when dst_p is a peer mapping).
constexpr int PACK_ROWS = 8;
// Every warp walks ALL peers, starting from a different one (rotated by its warp index), and takes
// the chunks {warp, warp + n_warps, ...} of each peer's row list: at any moment the stores of one
// GPU are spread over all its peers and every receiver hears from all senders at once.  (Walking
// the lists in peer order made all eight ranks write to the same GPU at the same time: 247 GB/s
// into each GPU at N = 8 against 670 GB/s at N = 2.)
__global__ void __launch_bounds__(256) halo_pack_kernel(const PackArgs a)
{
    const int lane = threadIdx.x & 31;
    const int n_warps = gridDim.x * (blockDim.x >> 5);
    const int wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const bool v4 = (a.F % 4 == 0) && (a.ldx % 4 == 0);
    for (int pp = 0; pp < a.n_peers; pp++) {
        const int p = (pp + wid) % a.n_peers;
        const long long base = a.start[p], n_p = a.count[p];
        float *const dst_p = a.dst[p];
        for (long long i0 = (long long)wid * PACK_ROWS; i0 < n_p; i0 += (long long)n_warps * PACK_ROWS) {
            const float *src[PACK_ROWS];
#pragma unroll
            for (int r = 0; r < PACK_ROWS; r++)
                src[r] = i0 + r < n_p ? a.x + (size_t)__ldg(a.send_idx + base + i0 + r) * a.ldx : nullptr;
            if (v4) {
                for (int c = lane * 4; c < a.F; c += 128) {
                    float4 v[PACK_ROWS];
#pragma unroll
                    for (int r = 0; r < PACK_ROWS; r++)
                        if (src[r] != nullptr) v[r] = __ldg(reinterpret_cast<const float4 *>(src[r] + c));
#pragma unroll
                    for (int r = 0; r < PACK_ROWS; r++)
                        if (src[r] != nullptr)
                            *reinterpret_cast<float4 *>(dst_p + (size_t)(i0 + r) * a.F + c) = v[r];
                }
            } else {
                for (int c = lane; c < a.F; c += 32) {
                    float v[PACK_ROWS];
#pragma unroll
                    for (int r = 0; r < PACK_ROWS; r++)
                        if (src[r] != nullptr) v[r] = __ldg(src[r] + c);
#pragma unroll
                    for (int r = 0; r < PACK_ROWS; r++)
                        if (src[r] != nullptr) dst_p[(size_t)(i0 + r) * a.F + c] = v[r];
                }
            }
        }
    }
}

struct SignalArgs {
    unsigned long long *flag[kMaxPeers];
    int n;
    unsigned long long value;
};
// The pack kernel before it on the stream has completed, so its stores are performed; a
// system-scope release store of the epoch then tells every peer that this rank's rows landed.
__global__ void halo_signal_kernel(const SignalArgs a)
{
    const int p = threadIdx.x;
    if (p < a.n && a.flag[p] != nullptr) {
        __threadfence_system();
        asm volatile("st.release.sys.global.u64 [%0], %1;\n" ::"l"(a.flag[p]), "l"(a.value) : "memory");
    }
}
// Spins (acquire, system scope) until every flag has reached `value`; gives up after ~2 s of
// SM clocks and reports through *timed_out instead of hanging the GPU.
__global__ void halo_wait_kernel(const unsigned long long *flags, int n, unsigned long long value,
                                 int *timed_out)
{
    const int p = threadIdx.x;
    if (p >= n) return;
    const long long t0 = clock64();
    for (;;) {
        unsigned long long v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];\n" : "=l"(v) : "l"(flags + p) : "memory");
        if (v >= value) break;
        if (clock64() - t0 > 4000000000ll) {
            atomicExch(timed_out, 1);
            break;
        }
        __nanosleep(200);
    }
}
}  // namespace halo
}  // namespace gnnb
using namespace gnnb::halo;

extern "C" int gnnb_partition_tables(const int32_t *edge_list_local, int row_begin, int n_local,
                                     int num_edges_local, int32_t *in_degree_local,
                                     int32_t *offsets_local, int32_t *neighbor_table_global,
                                     void *stream)
{
    GNNB_REQUIRE(n_local >= 0 && num_edges_local >= 0 && row_begin >= 0, "negative size");
    GNNB_REQUIRE(num_edges_local == 0 || is_device_pointer(edge_list_local),
                 "gnnb_partition_tables takes device pointers");
    g_part.whole.key = nullptr;
    for (HeavyCache &hc : g_part.part) hc.key = nullptr;
    return build_partition_tables(edge_list_local, row_begin, n_local, num_edges_local,
                                  in_degree_local, offsets_local, neighbor_table_global, g_part.ws,
                                  (cudaStream_t)stream, nullptr);
}

extern "C" int gnnb_degree_inv_sqrt(const int32_t *in_degree, float *dinv, int n, void *stream)
{
    GNNB_REQUIRE(n >= 0, "negative size");
    return compute_dinv(in_degree, dinv, n, (cudaStream_t)stream, nullptr);
}

extern "C" int gnnb_gcn_conv_partition(int n_local, int row_begin, int n_total, int num_edges_local,
                                       const float *x_full, float *y_local,
                                       const int32_t *offsets_local,
                                       const int32_t *neighbor_table_global,
                                       const int32_t *in_degree_local, const float *dinv_full,
                                       const float *weight, const float *bias,
                                       const float *skip_local, int emb_in, int emb_out, int act,
                                       void *stream)
{
    (void)num_edges_local;
    GNNB_REQUIRE(n_local >= 0 && row_begin >= 0 && row_begin + n_local <= n_total, "bad row range");
    GNNB_REQUIRE(emb_in > 0 && emb_out > 0 && act >= 0 && act <= GNNB_ACT_COS, "bad dims");
    if (n_local == 0) return GNNB_OK;
    GNNB_REQUIRE(is_device_pointer(x_full) && is_device_pointer(y_local),
                 "gnnb_gcn_conv_partition takes device pointers");
    cudaStream_t s = (cudaStream_t)stream;
    const int lda = round_up(emb_in, 4);
    GNNB_TRY(g_part.agg.ensure(sizeof(float) * (size_t)n_local * lda));
    // transposed weight + its tensor-core image (two tiny kernels per call; the GEMM then runs on tcgen05)
    DevWeight &dw = g_part.w[0];
    GNNB_TRY(dev_weight(dw, weight, emb_out, emb_in, 0, s));
    // the row list is cached across layers; the partial-sum scratch is sized for THIS layer's
    // emb_in on every call (ensure() only grows)
    GNNB_TRY(heavy_rows_of(g_part.whole, in_degree_local, n_local, s));
    GNNB_TRY(heavy_setup(g_part.ws, g_part.whole.list.n_chunks, emb_in));
    AggArgs a{};
    a.mode = AGG_GCN; a.x = x_full; a.ldx = emb_in; a.F = emb_in; a.out = g_part.agg.as<float>();
    a.ldo = lda; a.offsets = offsets_local; a.nbr = neighbor_table_global; a.in_deg = in_degree_local;
    a.dinv = dinv_full; a.n = n_local; a.row_base = row_begin;
    a.heavy.threshold = heavy_threshold();
    a.heavy.set(g_part.whole.list, g_part.ws.heavy_partial.as<float>());
    GNNB_TRY(launch_agg(a, false, s, nullptr));
    GemmArgs g = simple_gemm(a.out, lda, emb_in, dw.wt.as<float>(), dw.ldw, bias, y_local, emb_out,
                             n_local, emb_out, act);
    g.skip = skip_local; g.ldskip = emb_out;
    g.img1 = dw.img.as<float>();
    GNNB_TRY(launch_gemm(g, false, s, nullptr));
    return GNNB_OK;
}

// Column-wise sum and max over the n rows of x[n][F] (device pointers, asynchronous on `stream`):
// the per-rank partial of global_add/mean/max_pool (lib:2709-2803) for a row-partitioned graph;
// out[0..F) = sums, out[F..2F) = maxima (0 for n = 0).  The ranks combine them with all_reduce.
extern "C" int gnnb_pool_partial(const float *x, int64_t n, int F, float *out, void *stream)
{
    GNNB_REQUIRE(n >= 0 && F > 0 && out != nullptr, "bad arguments");
    GNNB_REQUIRE(n == 0 || (is_device_pointer(x) && is_device_pointer(out)),
                 "gnnb_pool_partial takes device pointers");
    cudaStream_t s = (cudaStream_t)stream;
    if (g_part.pool_n != n) {
        GNNB_TRY(g_part.pool_ptr.ensure(2 * sizeof(int64_t)));
        const int64_t h[2] = {0, n};
        GNNB_CUDA(cudaMemcpyAsync(g_part.pool_ptr.ptr, h, sizeof(h), cudaMemcpyHostToDevice, s));
        GNNB_CUDA(cudaStreamSynchronize(s));   // h is a stack variable
        g_part.pool_n = n;
    }
    const int pools[2] = {GNNB_POOL_ADD, GNNB_POOL_MAX};
    return launch_pool(x, F, F, g_part.pool_ptr.as<int64_t>(), 0, 1, n, pools, 2, out, g_part.pool_tmp, s,
                       nullptr);
}

// ============================================================================ halo exchange
// Row partition with a true halo (SURVEY 8e): every rank keeps its owned feature rows followed by
// ONE copy of each remote row its in-edges reference ("ext" space: [owned | halo grouped by owner
// rank]); gnn_builder_b200/distributed.py builds the index tables once.  Per layer the owners push
// the rows their peers need (gnnb_halo_pack: into an NCCL send buffer, or straight into the peer's
// halo region through a CUDA-IPC mapping, i.e. NVLink stores + gnnb_halo_signal / gnnb_halo_wait),
// while the aggregation of the owned-source edges runs (phase 1 below); the halo-source edges,
// the normalisation and the tcgen05 transform follow on arrival (phase 2).

extern "C" int gnnb_halo_pack_ranges(const float *x, int ldx, int F, const int32_t *send_idx,
                                     const int64_t *start, const int64_t *count, float *const *dst,
                                     int n_peers, int max_ctas, void *stream)
{
    GNNB_REQUIRE(n_peers >= 0 && n_peers <= kMaxPeers, "halo pack: at most 16 peers");
    GNNB_REQUIRE(F > 0 && ldx >= F && start != nullptr && count != nullptr && dst != nullptr,
                 "halo pack: bad arguments");
    PackArgs a{};
    a.x = x; a.ldx = ldx; a.F = F; a.n_peers = n_peers; a.send_idx = send_idx;
    long long total = 0, longest = 0;
    for (int p = 0; p < n_peers; p++) {
        GNNB_REQUIRE(start[p] >= 0 && count[p] >= 0, "halo pack: negative range");
        a.start[p] = start[p];
        a.count[p] = count[p];
        a.dst[p] = dst[p];
        GNNB_REQUIRE(count[p] == 0 || (dst[p] != nullptr && (reinterpret_cast<uintptr_t>(dst[p]) & 15) == 0),
                     "halo pack: destination missing or not 16-byte aligned");
        total += count[p];
        longest = count[p] > longest ? count[p] : longest;
    }
    if (total == 0) return GNNB_OK;
    long long grid = (longest + 8 * PACK_ROWS - 1) / (8 * PACK_ROWS);
    const long long cap = max_ctas > 0 ? max_ctas : kNumSMs;   // one CTA per SM: see the kernel
    if (grid > cap) grid = cap;
    halo_pack_kernel<<<(int)grid, 256, 0, (cudaStream_t)stream>>>(a);
    GNNB_CUDA(cudaGetLastError());
    return GNNB_OK;
}

extern "C" int gnnb_halo_pack(const float *x, int ldx, int F, const int32_t *send_idx,
                              const int64_t *send_off, float *const *dst, int n_peers, int max_ctas,
                              void *stream)
{
    GNNB_REQUIRE(n_peers >= 0 && n_peers <= kMaxPeers && send_off != nullptr, "halo pack: bad arguments");
    int64_t start[kMaxPeers], count[kMaxPeers];
    for (int p = 0; p < n_peers; p++) {
        GNNB_REQUIRE(send_off[p + 1] >= send_off[p], "halo pack: offsets must be non-decreasing");
        start[p] = send_off[p];
        count[p] = send_off[p + 1] - send_off[p];
    }
    return gnnb_halo_pack_ranges(x, ldx, F, send_idx, start, count, dst, n_peers, max_ctas, stream);
}

extern "C" int gnnb_halo_signal(uint64_t *const *peer_flags, int n_peers, uint64_t value, void *stream)
{
    GNNB_REQUIRE(n_peers >= 0 && n_peers <= kMaxPeers && peer_flags != nullptr, "halo signal: bad arguments");
    if (n_peers == 0) return GNNB_OK;
    SignalArgs a{};
    a.n = n_peers; a.value = value;
    for (int p = 0; p < n_peers; p++) a.flag[p] = reinterpret_cast<unsigned long long *>(peer_flags[p]);
    halo_signal_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(a);
    GNNB_CUDA(cudaGetLastError());
    return GNNB_OK;
}

extern "C" int gnnb_halo_wait(const uint64_t *flags, int n_flags, uint64_t value, int *timed_out,
                              void *stream)
{
    GNNB_REQUIRE(n_flags >= 0 && n_flags <= 32 && flags != nullptr && timed_out != nullptr,
                 "halo wait: bad arguments");
    if (n_flags == 0) return GNNB_OK;
    halo_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const unsigned long long *>(flags), n_flags, value, timed_out);
    GNNB_CUDA(cudaGetLastError());
    return GNNB_OK;
}

// CUDA-IPC plumbing for the peer mappings (one process per GPU): the library owns the allocation.
extern "C" int gnnb_ipc_alloc(size_t bytes, void **ptr, void *handle64)
{
    GNNB_REQUIRE(ptr != nullptr && handle64 != nullptr && bytes > 0, "ipc alloc: bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    void *p = nullptr;
    GNNB_CUDA(cudaMalloc(&p, bytes));
    cudaError_t e = cudaMemset(p, 0, bytes);
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        return cuda_fail(e, "cudaIpcGetMemHandle", __FILE__, __LINE__);
    }
    memcpy(handle64, &h, 64);
    *ptr = p;
    return GNNB_OK;
}
extern "C" int gnnb_ipc_open(const void *handle64, void **ptr)
{
    GNNB_REQUIRE(ptr != nullptr && handle64 != nullptr, "ipc open: bad arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    GNNB_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return GNNB_OK;
}
extern "C" int gnnb_ipc_close(void *ptr)
{
    if (ptr) GNNB_CUDA(cudaIpcCloseMemHandle(ptr));
    return GNNB_OK;
}
extern "C" int gnnb_ipc_free(void *ptr)
{
    if (ptr) GNNB_CUDA(cudaFree(ptr));
    return GNNB_OK;
}

extern "C" int gnnb_mark_hub_sources(int32_t *neighbor_table, int num_entries, int num_sources,
                                     int row_bytes, int64_t budget_bytes, int *num_hubs, void *stream)
{
    GNNB_REQUIRE(num_entries >= 0 && num_sources >= 0 && row_bytes > 0 && budget_bytes >= 0,
                 "mark hub sources: bad arguments");
    GNNB_REQUIRE(num_entries == 0 || is_device_pointer(neighbor_table), "mark hub sources takes a device pointer");
    return mark_hub_sources(neighbor_table, neighbor_table, num_entries, nullptr, num_sources,
                            (size_t)row_bytes, (size_t)budget_bytes, g_part.ws, num_hubs,
                            (cudaStream_t)stream, nullptr);
}

extern "C" int gnnb_gcn_conv_halo(int n_local, int n_ext, const float *x_ext, float *y_local,
                                  const int32_t *own_offsets, const int32_t *own_counts,
                                  const int32_t *own_nbr, const int32_t *halo_offsets,
                                  const int32_t *halo_counts, const int32_t *halo_nbr,
                                  const float *dinv_ext, const float *weight, const float *bias,
                                  const float *skip_local, int emb_in, int emb_out, int act, int phase,
                                  int hub_bit, int row_begin, int row_count, void *stream)
{
    GNNB_TRY(check_halo_args(n_local, n_ext, emb_in, emb_out, act, phase));
    if (row_count <= 0) { row_begin = 0; row_count = n_local; }
    GNNB_REQUIRE(row_begin >= 0 && row_begin + row_count <= n_local, "row block outside the owned rows");
    if (n_local == 0) return GNNB_OK;
    GNNB_REQUIRE(is_device_pointer(x_ext) && is_device_pointer(y_local), "gnnb_gcn_conv_halo takes device pointers");
    const bool has_halo = halo_counts != nullptr && n_ext > n_local;
    cudaStream_t s = (cudaStream_t)stream;
    const int lda = round_up(emb_in, 4);
    GNNB_TRY(g_part.agg.ensure(sizeof(float) * (size_t)n_local * lda));
    AggArgs a{};
    a.mode = AGG_GCN; a.x = x_ext; a.ldx = emb_in; a.F = emb_in;
    a.out = g_part.agg.as<float>() + (size_t)row_begin * lda;
    a.ldo = lda; a.dinv = dinv_ext; a.n = row_count;
    a.row_base = row_begin;      // owned row v is ext row v: self row and dinv are indexed v + row_base
    a.heavy.threshold = heavy_threshold(); a.hub_bit = hub_bit ? 1 : 0;
    // block mode (opt-in): the halo pack of the previous row block runs beside these kernels
    a.short_ctas = row_count < n_local ? 1 : 0;
    if (phase & 1)
        GNNB_TRY(halo_agg_part(a, own_offsets, own_counts, own_nbr, nullptr, false, !has_halo,
                               row_begin, row_count, s));
    if (!(phase & 2)) return GNNB_OK;
    if (has_halo)
        GNNB_TRY(halo_agg_part(a, halo_offsets, halo_counts, halo_nbr, nullptr, true, true,
                               row_begin, row_count, s));
    DevWeight &dw = g_part.w[0];
    GNNB_TRY(dev_weight(dw, weight, emb_out, emb_in, 0, s));
    GemmArgs g = simple_gemm(a.out, lda, emb_in, dw.wt.as<float>(), dw.ldw, bias,
                             y_local + (size_t)row_begin * emb_out, emb_out, row_count, emb_out, act);
    g.skip = skip_local != nullptr ? skip_local + (size_t)row_begin * emb_in : nullptr;
    g.ldskip = emb_in;
    g.img1 = dw.img.as<float>();
    GNNB_TRY(launch_gemm(g, false, s, nullptr));
    return GNNB_OK;
}

// ---- the other convs on the split CSR (same ext-space arguments as gnnb_gcn_conv_halo) -------
extern "C" int gnnb_gin_conv_halo(int n_local, int n_ext, const float *x_ext, float *y_local,
                                  const int32_t *own_offsets, const int32_t *own_counts,
                                  const int32_t *own_nbr, const int32_t *halo_offsets,
                                  const int32_t *halo_counts, const int32_t *halo_nbr,
                                  const float *mlp_0_weight, const float *mlp_0_bias,
                                  const float *mlp_1_weight, const float *mlp_1_bias, float gin_eps,
                                  const float *skip_local, int emb_in, int hidden, int emb_out, int act,
                                  int phase, int hub_bit, void *stream)
{
    GNNB_TRY(check_halo_args(n_local, n_ext, emb_in, emb_out, act, phase));
    GNNB_REQUIRE(hidden > 0, "bad hidden size");
    GNNB_REQUIRE(skip_local == nullptr || emb_in == emb_out, "a skip connection needs emb_in == emb_out");
    if (n_local == 0) return GNNB_OK;
    GNNB_REQUIRE(is_device_pointer(x_ext) && is_device_pointer(y_local), "gnnb_gin_conv_halo takes device pointers");
    const bool has_halo = halo_counts != nullptr && n_ext > n_local;
    cudaStream_t s = (cudaStream_t)stream;
    const int lda = round_up(emb_in, 4);
    GNNB_TRY(g_part.agg.ensure(sizeof(float) * (size_t)n_local * lda));
    AggArgs a{};
    a.mode = AGG_GIN; a.x = x_ext; a.ldx = emb_in; a.F = emb_in; a.out = g_part.agg.as<float>();
    a.ldo = lda; a.n = n_local; a.eps = gin_eps;   // (1 + eps) x_v with ext row v = owned row v
    a.heavy.threshold = heavy_threshold(); a.hub_bit = hub_bit ? 1 : 0;
    if (phase & 1)
        GNNB_TRY(halo_agg_part(a, own_offsets, own_counts, own_nbr, nullptr, false, !has_halo, 0,
                               n_local, s));
    if (!(phase & 2)) return GNNB_OK;
    if (has_halo)
        GNNB_TRY(halo_agg_part(a, halo_offsets, halo_counts, halo_nbr, nullptr, true, true, 0, n_local, s));
    // the MLP (lib:1537-1541): linear_0 + ReLU into the hidden scratch, linear_1 (+ skip) + act
    const int ldh = round_up(hidden, 4);
    GNNB_TRY(g_part.hid.ensure(sizeof(float) * (size_t)n_local * ldh));
    DevWeight &w0 = g_part.w[0], &w1 = g_part.w[1];
    GNNB_TRY(dev_weight(w0, mlp_0_weight, hidden, emb_in, 0, s));
    GNNB_TRY(dev_weight(w1, mlp_1_weight, emb_out, hidden, 0, s));
    float *hid = g_part.hid.as<float>();
    GemmArgs g0 = simple_gemm(a.out, lda, emb_in, w0.wt.as<float>(), w0.ldw, mlp_0_bias, hid, ldh,
                              n_local, hidden, GNNB_ACT_RELU);
    g0.img1 = w0.img.as<float>();
    GNNB_TRY(launch_gemm(g0, false, s, nullptr));
    GemmArgs g1 = simple_gemm(hid, ldh, hidden, w1.wt.as<float>(), w1.ldw, mlp_1_bias, y_local,
                              emb_out, n_local, emb_out, act);
    g1.skip = skip_local; g1.ldskip = emb_in;
    g1.img1 = w1.img.as<float>();
    GNNB_TRY(launch_gemm(g1, false, s, nullptr));
    return GNNB_OK;
}

extern "C" int gnnb_sage_conv_halo(int n_local, int n_ext, const float *x_ext, float *y_local,
                                   const int32_t *own_offsets, const int32_t *own_counts,
                                   const int32_t *own_nbr, const int32_t *halo_offsets,
                                   const int32_t *halo_counts, const int32_t *halo_nbr,
                                   const int32_t *in_degree_local, const float *neighbor_lin_weight,
                                   const float *neighbor_lin_bias, const float *self_lin_weight,
                                   const float *skip_local, int emb_in, int emb_out, int act, int phase,
                                   int hub_bit, void *stream)
{
    GNNB_TRY(check_halo_args(n_local, n_ext, emb_in, emb_out, act, phase));
    GNNB_REQUIRE(skip_local == nullptr || emb_in == emb_out, "a skip connection needs emb_in == emb_out");
    if (n_local == 0) return GNNB_OK;
    GNNB_REQUIRE(is_device_pointer(x_ext) && is_device_pointer(y_local) && is_device_pointer(in_degree_local),
                 "gnnb_sage_conv_halo takes device pointers");
    const bool has_halo = halo_counts != nullptr && n_ext > n_local;
    cudaStream_t s = (cudaStream_t)stream;
    const int lda = round_up(emb_in, 4);
    GNNB_TRY(g_part.agg.ensure(sizeof(float) * (size_t)n_local * lda));
    AggArgs a{};
    a.mode = AGG_MEAN; a.x = x_ext; a.ldx = emb_in; a.F = emb_in; a.out = g_part.agg.as<float>();
    a.ldo = lda; a.n = n_local;
    a.heavy.threshold = heavy_threshold(); a.hub_bit = hub_bit ? 1 : 0;
    // the parts' lengths walk the edges, the full in-degree divides (in-degree 0 gives 0, lib:2180-2207)
    if (phase & 1)
        GNNB_TRY(halo_agg_part(a, own_offsets, own_counts, own_nbr, in_degree_local, false, !has_halo,
                               0, n_local, s));
    if (!(phase & 2)) return GNNB_OK;
    if (has_halo)
        GNNB_TRY(halo_agg_part(a, halo_offsets, halo_counts, halo_nbr, in_degree_local, true, true, 0,
                               n_local, s));
    // mean.W_l^T + b_l + x_v.W_r^T (lib:2316-2332) (+ skip) + act: one GEMM with two operands
    DevWeight &wl = g_part.w[0], &wr = g_part.w[1];
    GNNB_TRY(dev_weight(wl, neighbor_lin_weight, emb_out, emb_in, 0, s));
    GNNB_TRY(dev_weight(wr, self_lin_weight, emb_out, emb_in, 0, s));
    GemmArgs g = simple_gemm(a.out, lda, emb_in, wl.wt.as<float>(), wl.ldw, neighbor_lin_bias, y_local,
                             emb_out, n_local, emb_out, act);
    g.A2 = x_ext; g.lda2 = emb_in; g.K2 = emb_in; g.W2t = wr.wt.as<float>(); g.ldw2 = wr.ldw;
    g.img1 = wl.img.as<float>(); g.img2 = wr.img.as<float>();
    g.second_separate = 1;
    g.skip = skip_local; g.ldskip = emb_in;
    GNNB_TRY(launch_gemm(g, false, s, nullptr));
    return GNNB_OK;
}

extern "C" int gnnb_pna_conv_halo(int n_local, int n_ext, const float *x_local, float *a_ext,
                                  float *y_local, const int32_t *own_offsets, const int32_t *own_counts,
                                  const int32_t *own_nbr, const int32_t *halo_offsets,
                                  const int32_t *halo_counts, const int32_t *halo_nbr,
                                  const int32_t *in_degree_local, const float *transform_lin_weight,
                                  const float *transform_lin_bias, const float *apply_lin_weight,
                                  const float *apply_lin_bias, const float *final_lin_weight,
                                  const float *final_lin_bias, float pna_avg_degree_log,
                                  const float *skip_local, int emb_in, int emb_out, int act, int phase,
                                  void *stream)
{
    GNNB_TRY(check_halo_args(n_local, n_ext, emb_in, emb_out, act, phase));
    GNNB_REQUIRE(skip_local == nullptr || emb_in == emb_out, "a skip connection needs emb_in == emb_out");
    if (n_local == 0) return GNNB_OK;
    GNNB_REQUIRE(is_device_pointer(x_local) && is_device_pointer(a_ext) && is_device_pointer(y_local) &&
                     is_device_pointer(in_degree_local),
                 "gnnb_pna_conv_halo takes device pointers");
    const bool has_halo = halo_counts != nullptr && n_ext > n_local;
    cudaStream_t s = (cudaStream_t)stream;
    const int F = emb_in;
    GNNB_TRY(g_part.pna_b.ensure(sizeof(float) * (size_t)n_local * F));
    float *bself = g_part.pna_b.as<float>();
    if (phase & 1) {
        // W_pre = [W_self | W_nbr] (lib:1801-1807): A = x.W_nbr^T goes to the peers, B stays
        DevWeight &wn = g_part.w[0], &ws = g_part.w[1];
        GNNB_TRY(dev_weight(wn, transform_lin_weight + F, F, F, 2 * F, s));
        GNNB_TRY(dev_weight(ws, transform_lin_weight, F, F, 2 * F, s));
        GemmArgs ga = simple_gemm(x_local, F, F, wn.wt.as<float>(), wn.ldw, nullptr, a_ext, F, n_local, F,
                                  GNNB_ACT_IDENTITY);
        ga.img1 = wn.img.as<float>();
        GNNB_TRY(launch_gemm(ga, false, s, nullptr));
        GemmArgs gb = simple_gemm(x_local, F, F, ws.wt.as<float>(), ws.ldw, transform_lin_bias, bself, F,
                                  n_local, F, GNNB_ACT_IDENTITY);
        gb.img1 = ws.img.as<float>();
        GNNB_TRY(launch_gemm(gb, false, s, nullptr));
    }
    if (!(phase & 2)) return GNNB_OK;
    // post_nn = [W_post_self | W_post_agg] over [x | 12F statistics], then the final linear
    const int ld_o = round_up(emb_out, 4);
    DevWeight &wp = g_part.w[2], &wa = g_part.w[3], &wf = g_part.w[4];
    GNNB_TRY(dev_weight(wp, apply_lin_weight, emb_out, F, 13 * F, s));
    GNNB_TRY(dev_weight(wa, apply_lin_weight + F, emb_out, 12 * F, 13 * F, s));
    GNNB_TRY(dev_weight(wf, final_lin_weight, emb_out, emb_out, 0, s));
    GNNB_TRY(g_part.hid.ensure(sizeof(float) * (size_t)n_local * ld_o));
    GNNB_TRY(g_part.pna_stats.ensure(sizeof(float) * (size_t)n_local * 12 * F));
    float *hid = g_part.hid.as<float>(), *stats = g_part.pna_stats.as<float>();
    GemmArgs g1 = simple_gemm(x_local, F, F, wp.wt.as<float>(), wp.ldw, apply_lin_bias, hid, ld_o, n_local,
                              emb_out, GNNB_ACT_IDENTITY);
    g1.img1 = wp.img.as<float>();
    g1.A2 = stats; g1.K2 = 12 * F; g1.W2t = wa.wt.as<float>(); g1.ldw2 = wa.ldw; g1.img2 = wa.img.as<float>();
    // tensor-core path: only the [n][4F] statistics are written and the GEMM expands them with the
    // degree scalers, as the layerwise path does
    g1.lda2 = 4 * F; g1.expand_deg = in_degree_local; g1.expand_delta = pna_avg_degree_log;
    const bool expand = gemm_tc_supported(g1);
    if (!expand) { g1.lda2 = 12 * F; g1.expand_deg = nullptr; }
    PnaHaloArgs pa{};
    pa.a_ext = a_ext; pa.b = bself; pa.F = F; pa.cat12 = stats;
    pa.own_off = own_offsets; pa.own_cnt = own_counts; pa.own_nbr = own_nbr;
    if (has_halo) { pa.halo_off = halo_offsets; pa.halo_cnt = halo_counts; pa.halo_nbr = halo_nbr; }
    pa.in_deg = in_degree_local; pa.n = n_local; pa.delta = pna_avg_degree_log; pa.compact = expand ? 1 : 0;
    GNNB_TRY(launch_pna_halo_stats(pa, s, nullptr));
    GNNB_TRY(launch_gemm(g1, false, s, nullptr));
    GemmArgs g2 = simple_gemm(hid, ld_o, emb_out, wf.wt.as<float>(), wf.ldw, final_lin_bias, y_local,
                              emb_out, n_local, emb_out, act);
    g2.skip = skip_local; g2.ldskip = emb_in;
    g2.img1 = wf.img.as<float>();
    GNNB_TRY(launch_gemm(g2, false, s, nullptr));
    return GNNB_OK;
}

// ---- the attention convs on the rank's CSR in ext indices ------------------------------------
// An attention layer has nothing to aggregate before the GEMM output of its halo rows arrives, so
// these take the rank's whole per-row CSR (neighbor entries = ext indices) rather than the split
// one.  Owned row v is ext row v, so the unchanged aggregation kernels read the self term at g[v]
// and skip the entries equal to v (input self loops); halo entries are >= n_local.
namespace gnnb {
// Wg [H*C + 2H][fi] = [W | w_src | w_dst], w_src,h[k] = sum_c W[h*C + c][k] att_src[h*C + c] (w_dst
// alike): summed in double in ascending c with separately rounded products and sums, rounded once,
// which is the model handle's fold (model.cu), so both give the same GEMM weights
__global__ void gat_fold_weight_kernel(const float *__restrict__ W, const float *__restrict__ att_src,
                                       const float *__restrict__ att_dst, float *__restrict__ Wg, int H,
                                       int C, int fi)
{
    const int HC = H * C;
    const int64_t total = (int64_t)(HC + 2 * H) * fi;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / fi), k = (int)(i % fi);
        if (r < HC) {
            Wg[i] = W[i];
            continue;
        }
        const int q = r - HC, h = q % H;
        const float *att = (q < H ? att_src : att_dst) + h * C;
        double acc = 0.0;
        for (int c = 0; c < C; c++)
            acc = __dadd_rn(acc, __dmul_rn((double)W[(size_t)(h * C + c) * fi + k], (double)att[c]));
        Wg[i] = __double2float_rn(acc);
    }
}
}  // namespace gnnb

namespace {

// argument checks of the attention halo layers (before any device work)
int check_attn_halo_args(const char *conv, int heads, float slope, int emb_in, int emb_out,
                         const float *skip_local, bool gatv2)
{
    const std::string name(conv);
    GNNB_REQUIRE(heads >= 1 && heads <= GNNB_GAT_MAX_HEADS,
                 name + " heads must be 1.." + std::to_string(GNNB_GAT_MAX_HEADS));
    GNNB_REQUIRE(emb_out % heads == 0, name + ": emb_out must be a multiple of heads");
    GNNB_REQUIRE(std::isfinite(slope), name + " negative_slope must be finite");
    const int C = emb_out / heads;
    GNNB_REQUIRE(!gatv2 || C <= (C % 4 == 0 ? kGatv2MaxHeadWidth : kGatv2MaxHeadWidth1),
                 "GATv2: a head's width (layer width / gat_heads) must be at most " +
                     std::to_string(kGatv2MaxHeadWidth) + " when a multiple of 4, else at most " +
                     std::to_string(kGatv2MaxHeadWidth1) + ", got " + std::to_string(C));
    GNNB_REQUIRE(skip_local == nullptr || emb_in == emb_out, "a skip connection needs emb_in == emb_out");
    return GNNB_OK;
}

// the attention arguments both convs share: the rank's CSR, the epilogue and the heavy rows (every
// row above heavy_threshold(), partials [ldp] wide)
int attn_halo_common(AttnAggArgs &at, int n_local, const int32_t *offsets_local,
                     const int32_t *in_degree_local, const int32_t *nbr_ext, int heads, float slope,
                     const float *bias, const float *skip_local, int emb_in, int emb_out, int act,
                     float *y_local, cudaStream_t s)
{
    at.H = heads; at.C = emb_out / heads; at.slope = slope;
    at.bias = bias; at.skip = skip_local; at.ldskip = emb_in; at.act = act;
    at.out = y_local; at.ldo = emb_out;
    at.offsets = offsets_local; at.nbr = nbr_ext; at.in_deg = in_degree_local; at.n = n_local;
    at.ldp = round_up(emb_out + 2 * heads, 4);
    HeavyCache &hc = part_cache(in_degree_local, n_local);
    GNNB_TRY(heavy_rows_of(hc, in_degree_local, n_local, s));
    GNNB_TRY(heavy_setup(g_part.ws, hc.list.n_chunks, at.ldp));
    at.heavy.threshold = heavy_threshold();
    at.heavy.set(hc.list, g_part.ws.heavy_partial.as<float>());
    return GNNB_OK;
}
}  // namespace

extern "C" int gnnb_gat_conv_halo(int n_local, int n_ext, const float *x_local, float *g_ext,
                                  float *y_local, const int32_t *offsets_local,
                                  const int32_t *in_degree_local, const int32_t *nbr_ext,
                                  const float *att_src, const float *att_dst, const float *bias,
                                  const float *lin_weight, int heads, float negative_slope,
                                  const float *skip_local, int emb_in, int emb_out, int act, int phase,
                                  void *stream)
{
    GNNB_TRY(check_halo_args(n_local, n_ext, emb_in, emb_out, act, phase));
    GNNB_TRY(check_attn_halo_args("GAT", heads, negative_slope, emb_in, emb_out, skip_local, false));
    if (n_local == 0) return GNNB_OK;
    GNNB_REQUIRE(is_device_pointer(x_local) && is_device_pointer(g_ext) && is_device_pointer(y_local) &&
                     is_device_pointer(offsets_local) && is_device_pointer(in_degree_local),
                 "gnnb_gat_conv_halo takes device pointers");
    cudaStream_t s = (cudaStream_t)stream;
    const int N = emb_out + 2 * heads, ldg = round_up(N, 4);
    if (phase & 1) {
        // [h | a_src | a_dst] of the owned rows = x.[W | w_src | w_dst]^T: what the peers gather
        GNNB_TRY(g_part.gat_w.ensure(sizeof(float) * (size_t)N * emb_in));
        float *Wg = g_part.gat_w.as<float>();
        const int64_t total = (int64_t)N * emb_in;
        gat_fold_weight_kernel<<<(int)std::min<int64_t>((total + 255) / 256, 4096), 256, 0, s>>>(
            lin_weight, att_src, att_dst, Wg, heads, emb_out / heads, emb_in);
        GNNB_CUDA(cudaGetLastError());
        DevWeight &dw = g_part.w[0];
        GNNB_TRY(dev_weight(dw, Wg, N, emb_in, 0, s));
        GemmArgs g = simple_gemm(x_local, emb_in, emb_in, dw.wt.as<float>(), dw.ldw, nullptr, g_ext, ldg,
                                 n_local, N, GNNB_ACT_IDENTITY);
        g.img1 = dw.img.as<float>();
        GNNB_TRY(launch_gemm(g, false, s, nullptr));
    }
    if (!(phase & 2)) return GNNB_OK;
    GatAggArgs ga{};
    GNNB_TRY(attn_halo_common(ga, n_local, offsets_local, in_degree_local, nbr_ext, heads, negative_slope,
                              bias, skip_local, emb_in, emb_out, act, y_local, s));
    ga.g = g_ext; ga.ldg = ldg;
    return launch_gat_agg(ga, s, nullptr);
}

extern "C" int gnnb_gatv2_conv_halo(int n_local, int n_ext, const float *x_local, float *xl_ext,
                                    float *y_local, const int32_t *offsets_local,
                                    const int32_t *in_degree_local, const int32_t *nbr_ext,
                                    const float *att, const float *bias, const float *lin_l_weight,
                                    const float *lin_l_bias, const float *lin_r_weight,
                                    const float *lin_r_bias, int heads, float negative_slope,
                                    const float *skip_local, int emb_in, int emb_out, int act, int phase,
                                    void *stream)
{
    GNNB_TRY(check_halo_args(n_local, n_ext, emb_in, emb_out, act, phase));
    GNNB_TRY(check_attn_halo_args("GATv2", heads, negative_slope, emb_in, emb_out, skip_local, true));
    if (n_local == 0) return GNNB_OK;
    GNNB_REQUIRE(is_device_pointer(x_local) && is_device_pointer(xl_ext) && is_device_pointer(y_local) &&
                     is_device_pointer(offsets_local) && is_device_pointer(in_degree_local),
                 "gnnb_gatv2_conv_halo takes device pointers");
    cudaStream_t s = (cudaStream_t)stream;
    const int ldl = round_up(emb_out, 4);
    GNNB_TRY(g_part.gatv2_xr.ensure(sizeof(float) * (size_t)n_local * ldl));
    float *xr = g_part.gatv2_xr.as<float>();
    if (phase & 1) {
        // xl of the owned rows goes to the peers, xr stays here
        DevWeight &wl = g_part.w[0], &wr = g_part.w[1];
        GNNB_TRY(dev_weight(wl, lin_l_weight, emb_out, emb_in, 0, s));
        GNNB_TRY(dev_weight(wr, lin_r_weight, emb_out, emb_in, 0, s));
        GemmArgs gl = simple_gemm(x_local, emb_in, emb_in, wl.wt.as<float>(), wl.ldw, lin_l_bias, xl_ext, ldl,
                                  n_local, emb_out, GNNB_ACT_IDENTITY);
        gl.img1 = wl.img.as<float>();
        GNNB_TRY(launch_gemm(gl, false, s, nullptr));
        GemmArgs gr = simple_gemm(x_local, emb_in, emb_in, wr.wt.as<float>(), wr.ldw, lin_r_bias, xr, ldl,
                                  n_local, emb_out, GNNB_ACT_IDENTITY);
        gr.img1 = wr.img.as<float>();
        GNNB_TRY(launch_gemm(gr, false, s, nullptr));
    }
    if (!(phase & 2)) return GNNB_OK;
    Gatv2AggArgs ga{};
    GNNB_TRY(attn_halo_common(ga, n_local, offsets_local, in_degree_local, nbr_ext, heads, negative_slope,
                              bias, skip_local, emb_in, emb_out, act, y_local, s));
    ga.g = xl_ext; ga.ldg = ldl; ga.xr = xr; ga.ldxr = ldl; ga.att = att;
    return launch_gatv2_agg(ga, s, nullptr);
}
