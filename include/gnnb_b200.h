/*
 * gnnb_b200.h -- C-ABI of libgnnb_b200.so, the B200 (sm_100a) backend for the hot path of
 * sharc-lab/gnn-builder: what gnnbuilder/gnn_builder_lib/gnn_builder_lib.h ("lib") and the
 * generated top function gnnbuilder/templates/model.cpp.jinja ("cpp") compute.
 *
 * Conventions
 *  - All feature/weight data are fp32.  Weights are passed in the reference's layout
 *    W[out][in] row-major (= torch.nn.Linear.weight, lib:39-41).
 *  - edge_list is COO int32 [E][2] with [i][0] = source, [i][1] = destination (lib:1060-1062).
 *  - Every pointer argument may be a HOST pointer or a DEVICE pointer (cudaMalloc / torch CUDA
 *    tensor): the library asks the CUDA runtime which it is.  Host buffers are staged through
 *    device scratch and the call returns after the results are back in the caller's buffer;
 *    with device buffers the call returns after the work is complete on the library's stream
 *    unless an *_async entry point is used.
 *  - Every function returns GNNB_OK (0) or a negative error code; gnnb_last_error() gives the
 *    message for the calling thread.  There is no CPU fallback: without a CUDA device every
 *    compute entry point fails with GNNB_ERR_CUDA.
 *  - Unlike the reference (file-scope static buffers, cpp:7-22,197-209) handles are re-entrant:
 *    one handle = one device + one stream; use one handle per host thread.
 */
#ifndef GNNB_B200_H
#define GNNB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNNB_OK 0
#define GNNB_ERR_INVALID (-1)   /* bad argument / unsupported configuration */
#define GNNB_ERR_CUDA (-2)      /* CUDA runtime error (incl. no device) */
#define GNNB_ERR_STATE (-3)     /* wrong call order (e.g. run before finalize) */
#define GNNB_ERR_PARAM (-4)     /* unknown parameter name / wrong element count */

/* activation ids: lib:308-480; cpp:164-175 maps nn.ReLU/GELU/Sigmoid/Tanh to 1/2/3/4 */
enum {
    GNNB_ACT_IDENTITY = 0, GNNB_ACT_RELU = 1, GNNB_ACT_GELU_TANH = 2, GNNB_ACT_SIGMOID = 3,
    GNNB_ACT_TANH = 4, GNNB_ACT_ELU = 5, GNNB_ACT_HARDTANH = 6, GNNB_ACT_LEAKYRELU = 7,
    GNNB_ACT_GELU_ERF = 8, GNNB_ACT_SILU = 9, GNNB_ACT_SOFTSIGN = 10, GNNB_ACT_SIN = 11,
    GNNB_ACT_COS = 12
};
/* GINE (GIN with an edge linear, PyG GINEConv with edge_dim; lib:1555-1742) runs on the layerwise
 * path only and takes its edge features through the gnnb_model_run_batch_edges* entry points */
/* GAT (PyG GATConv for inference: concat heads, self loops replaced by one per node) runs on the
 * layerwise path only.  Without edge features (edge_dim = 0) it runs through the plain run entry
 * points; with edge_dim > 0 (GATConv's edge_dim: lin_edge and att_edge add an edge term to every
 * attention logit, and the self loop's attribute is the mean of the node's other in-edge
 * attributes) through the gnnb_model_run_batch_edges* ones.  It has no reference float build:
 * GNNB_MATH_STRICT means deterministic fp32 without tensor cores for it, held to the same error
 * bound as FAST. */
/* GATv2 (PyG GATv2Conv for inference: concat heads, self loops replaced by one per node, separate
 * lin_l / lin_r with biases, share_weights=False) reads edge_dim, gat_heads and gat_negative_slope
 * as GAT does and follows GAT's entry-point, path and math rules.  Its logit
 * <att_h, LeakyReLU(xl_u + xr_v (+ e_uv W_e^T))_h> is computed per edge inside the aggregation; with
 * edge_dim > 0 the self loop's attribute is the mean of the node's other in-edge attributes.
 * Each head's width C must be at most 256 when C is a multiple of 4, else at most 64.  The value 6
 * is not assigned. */
/* TransformerConv (PyG TransformerConv for inference: concat heads, root_weight, no beta, no self
 * loops added) reads edge_dim and gat_heads as GAT does, not gat_negative_slope, and follows GAT's
 * entry-point, path and math rules.  Per head, e_uv = <q_v, k_u (+ e_uv W_e^T)> / sqrt(C) over the
 * in-edges of v (input self loops and duplicate edges count as ordinary edges),
 * y_v = sum softmax_v(e) (v_u (+ e_uv W_e^T)) + x_v W_skip^T + b_skip; a node without in-edges gets
 * x_v W_skip^T + b_skip.  Parameters in PyG's order: lin_key, lin_query, lin_value (weight and bias
 * each), lin_edge.weight (edge_dim > 0), lin_skip.  Head widths as GATv2. */
enum {
    GNNB_CONV_GCN = 0, GNNB_CONV_GIN = 1, GNNB_CONV_SAGE = 2, GNNB_CONV_PNA = 3, GNNB_CONV_GINE = 4,
    GNNB_CONV_GAT = 5, GNNB_CONV_GATV2 = 7, GNNB_CONV_TRANSFORMER = 8
};
/* edge feature widths a GINE, edge-attention GAT, GATv2 or TransformerConv model handle accepts */
#define GNNB_GINE_MAX_EDGE_DIM 64
/* attention head counts a GAT, GATv2 or TransformerConv model handle accepts */
#define GNNB_GAT_MAX_HEADS 16
enum { GNNB_POOL_ADD = 0, GNNB_POOL_MEAN = 1, GNNB_POOL_MAX = 2 };

/* execution path of gnnb_model_run_batch */
enum {
    GNNB_PATH_AUTO = 0,      /* fused when every graph fits a CTA tile, else layerwise */
    GNNB_PATH_FUSED = 1,     /* kernel (1): persistent whole-model fused kernel */
    GNNB_PATH_LAYERWISE = 2  /* kernel (2): CSR aggregation + GEMM per layer on the batch union */
};
/* arithmetic mode */
enum {
    GNNB_MATH_FAST = 0,   /* FMA contraction, factorised GCN/PNA scaling: <= 1e-4 relative */
    GNNB_MATH_STRICT = 1  /* reference operation order, no contraction (layerwise path only):
                             bit-identical to the reference float build for GCN/GIN/SAGE + ReLU */
};

/* POD description of a gnnbuilder.GNNModel (models.py:462-549) -- replaces the per-model
 * template ints of the generated top (cpp:25-148, 686-696). */
typedef struct gnnb_model_desc {
    int32_t conv_type;      /* GNNB_CONV_* (class of model.gnn_conv) */
    int32_t num_layers;     /* gnn_num_layers */
    int32_t in_dim;         /* graph_input_feature_dim */
    int32_t hidden_dim;     /* gnn_hidden_dim */
    int32_t out_dim;        /* gnn_output_dim */
    int32_t skip;           /* gnn_skip_connection */
    int32_t gnn_act;        /* gnn_activation */
    float gin_eps;          /* GINConv_GNNB.eps      (template literal, cpp:79) */
    float pna_delta;        /* PNAConv_GNNB.delta_scaler (template literal, cpp:113) */
    int32_t num_pools;      /* len(global_pooling.aggrs), 1..3 */
    int32_t pools[4];       /* GNNB_POOL_* in list order (cpp:440-448) */
    int32_t mlp_num_linear; /* mlp_head.hidden_layers + 1 */
    int32_t mlp_hidden;     /* mlp_head.hidden_dim */
    int32_t mlp_out;        /* mlp_head.out_dim */
    int32_t mlp_act;        /* mlp_head.activation */
    int32_t out_act;        /* output_activation, 0 = None */
    int32_t max_nodes;      /* capacity hints (Project.max_nodes/max_edges, code_gen.py:71-72); */
    int32_t max_edges;      /* 0 = unbounded.  A graph larger than a non-zero hint is an error. */
    int32_t edge_dim;       /* GINE: edge feature width, 1..GNNB_GINE_MAX_EDGE_DIM.  GAT: 0 for no
                               edge features, else 1..GNNB_GINE_MAX_EDGE_DIM (edge attention), so
                               C callers of GAT must set it to 0 for plain GAT (zero-initialising
                               the struct does).  GATv2 and TransformerConv: as GAT.  Read only
                               when conv_type is GNNB_CONV_GINE, GNNB_CONV_GAT, GNNB_CONV_GATV2 or
                               GNNB_CONV_TRANSFORMER, so a caller built against a header without it
                               keeps working for the other convs. */
    int32_t gat_heads;      /* GAT, GATv2 and TransformerConv only: heads H, 1..GNNB_GAT_MAX_HEADS;
                               every layer's output width must be a multiple of H (C = width / H
                               channels per head) */
    float gat_negative_slope;  /* GAT and GATv2 only: LeakyReLU slope of the attention logits (PyG:
                                  0.2).  Both fields are read only when conv_type is GNNB_CONV_GAT
                                  or GNNB_CONV_GATV2. */
} gnnb_model_desc;

typedef struct gnnb_model gnnb_model_t;

/* ---- library ---------------------------------------------------------------------------- */
const char *gnnb_last_error(void);
int gnnb_version(void);
int gnnb_device_count(int *count);

/* Page-lock / release a caller-owned HOST buffer (cudaHostRegister): the host-buffer entry points
 * below then copy it asynchronously at the full PCIe rate (45 GB/s against ~8.5 GB/s for pageable
 * memory on the bench box).  Registration costs about one pageable copy, so it pays for buffers
 * that are passed more than once. */
int gnnb_host_register(void *ptr, size_t bytes);
int gnnb_host_unregister(void *ptr);

/* ---- model handle: replaces <name>_top (model.h.jinja:67-79, cpp:686-766) ----------------- */
/* device < 0 selects the current CUDA device */
int gnnb_model_create(const gnnb_model_desc *desc, int device, gnnb_model_t **out);
int gnnb_model_destroy(gnnb_model_t *m);
/* number of parameter arrays and their names/element counts, in the reference's flat order
 * (GNNModel.layer_parameter_names_flat, models.py:607-624: mlp_head_* first, then gnn_convs_*) */
int gnnb_model_num_params(const gnnb_model_t *m);
int gnnb_model_param_info(const gnnb_model_t *m, int index, const char **name, size_t *numel);
/* replaces the trailing `<param>_fixed_in` arguments + copy_parameters_flag (cpp:724-730):
 * `name` is the reference's flat name, e.g. "gnn_convs_0_mlp_linear_0_weight" */
int gnnb_model_set_param(gnnb_model_t *m, const char *name, const float *data, size_t numel);
/* packs the weights for the kernels; must be called once after all parameters are set */
int gnnb_model_finalize(gnnb_model_t *m);
int gnnb_model_set_path(gnnb_model_t *m, int path);  /* GNNB_PATH_* */
int gnnb_model_set_math(gnnb_model_t *m, int math);  /* GNNB_MATH_* */

/* One graph, exactly the data <name>_top receives (cpp:686-692). out: [mlp_out] */
int gnnb_model_run_graph(gnnb_model_t *m, const float *node_features, const int32_t *edge_list,
                         int num_nodes, int num_edges, float *out);
/* A batch of independent graphs, concatenated: x [node_ptr[G]][in_dim], edge_list
 * [edge_ptr[G]][2] with node ids LOCAL to each graph, node_ptr/edge_ptr int64 [G+1].
 * out: [G][mlp_out].  Synchronous.  All five buffers must live in the same memory space. */
int gnnb_model_run_batch(gnnb_model_t *m, const float *x, const int32_t *edge_list,
                         const int64_t *node_ptr, const int64_t *edge_ptr, int n_graphs,
                         float *out);
/* Device buffers only; enqueues on `stream` (a cudaStream_t; NULL = the handle's stream).
 * total_nodes/total_edges = node_ptr[G]/edge_ptr[G].  The fused path returns without
 * synchronising.  The layerwise path may block: scratch buffers grow with cudaMalloc the first
 * time a batch size is seen, and a batch of large graphs (> 50 000 nodes on average) reads two
 * counters back (heavy-row and hub-row selection).  Errors the device detects (an edge endpoint
 * outside its graph, a tile over capacity) are reported by gnnb_model_synchronize.  Every entry
 * point leaves the caller's current CUDA device unchanged. */
int gnnb_model_run_batch_async(gnnb_model_t *m, const float *x, const int32_t *edge_list,
                               const int64_t *node_ptr, const int64_t *edge_ptr, int n_graphs,
                               int64_t total_nodes, int64_t total_edges, float *out, void *stream);
/* GINE models, and GAT, GATv2 and TransformerConv models with edge_dim > 0: the same contracts as
 * gnnb_model_run_batch / gnnb_model_run_batch_async, plus edge_attr float [edge_ptr[G]][edge_dim] in
 * the memory space of the other buffers, row i the features of COO edge i (one row per stored direction).  Such a handle
 * must be run through these two; a handle without edge features is rejected by them
 * (GNNB_ERR_INVALID), and so is a null edge_attr with edges present. */
int gnnb_model_run_batch_edges(gnnb_model_t *m, const float *x, const int32_t *edge_list,
                               const float *edge_attr, const int64_t *node_ptr,
                               const int64_t *edge_ptr, int n_graphs, float *out);
int gnnb_model_run_batch_edges_async(gnnb_model_t *m, const float *x, const int32_t *edge_list,
                                     const float *edge_attr, const int64_t *node_ptr,
                                     const int64_t *edge_ptr, int n_graphs, int64_t total_nodes,
                                     int64_t total_edges, float *out, void *stream);
/* node embeddings after the last conv (node_emb_out, cpp:22,349-354) of the most recent
 * LAYERWISE run: copies [total_nodes][out_dim] floats to `dst` (host or device) */
int gnnb_model_get_node_embeddings(gnnb_model_t *m, float *dst, int64_t total_nodes);
/* statistics of the most recent run: kernels launched by this library, and which path ran */
int gnnb_model_last_launches(const gnnb_model_t *m);
int gnnb_model_last_path(const gnnb_model_t *m);
/* which kernel family ran: 1 layerwise, 2 fused (fp32 FMA node transform), 3 fused (tcgen05) */
int gnnb_model_last_kernel(const gnnb_model_t *m);
/* optional per-kernel-class timing with CUDA events on the launching stream: ms[8]/counts[8]
 * indexed 0 tables, 1 aggregation, 2 GEMM, 3 pooling, 4 fused kernel, 5 GAT edge logits (the
 * once-per-run pass of GAT models with edge_dim); reading resets */
int gnnb_model_set_profile(gnnb_model_t *m, int on);
int gnnb_model_profile_read(gnnb_model_t *m, float *ms, int *counts);
void *gnnb_model_stream(gnnb_model_t *m);
int gnnb_model_synchronize(gnnb_model_t *m);

/* ---- layer functions: same arguments as the lib templates, dims as ints -------------------- */
/* lib:1051-1083 */
int gnnb_compute_degree_tables(const int32_t *edge_list, int32_t *in_degree_table,
                               int32_t *out_degree_table, int num_nodes, int num_edges);
/* lib:1086-1124 (offsets: num_nodes entries, no sentinel; neighbor order stable in COO order) */
int gnnb_compute_neighbor_tables(const int32_t *edge_list, const int32_t *in_degree_table,
                                 const int32_t *out_degree_table, int32_t *neighbor_table_offsets,
                                 int32_t *neighbor_table, int num_nodes, int num_edges);
/* lib:1126-1166 */
int gnnb_compute_neighbor_and_edge_index_tables(const int32_t *edge_list,
                                                const int32_t *in_degree_table,
                                                const int32_t *out_degree_table,
                                                int32_t *neighbor_table_offsets,
                                                int32_t *neighbor_table, int32_t *edge_index_table,
                                                int num_nodes, int num_edges);
/* lib:808-905 / 908-1003: y[rows][out] = x[rows][in] . W^T + b  (rows = 1 is the lib call) */
int gnnb_linear(const float *x, float *y, const float *weight, const float *bias, int rows,
                int in_size, int out_size, int math);
/* lib:501-509 */
int gnnb_apply_activation(int act, const float *x, float *y, size_t n);
/* lib:1291-1387 */
int gnnb_gcn_conv(int num_nodes, int num_edges, const float *x_in, float *x_out,
                  const int32_t *edge_list, const int32_t *neighbor_table_offsets,
                  const int32_t *neighbor_table, const int32_t *in_degree_table,
                  const int32_t *out_degree_table, const float *weight, const float *bias,
                  int emb_in, int emb_out, int math);
/* lib:1440-1549 */
int gnnb_gin_conv(int num_nodes, int num_edges, const float *x_in, float *x_out,
                  const int32_t *edge_list, const int32_t *neighbor_table_offsets,
                  const int32_t *neighbor_table, const int32_t *in_degree_table,
                  const int32_t *out_degree_table, const float *mlp_0_weight,
                  const float *mlp_0_bias, const float *mlp_1_weight, const float *mlp_1_bias,
                  float gin_eps, int emb_in, int hidden, int emb_out, int math);
/* lib:2211-2341 */
int gnnb_sage_conv(int num_nodes, int num_edges, const float *x_in, float *x_out,
                   const int32_t *edge_list, const int32_t *neighbor_table_offsets,
                   const int32_t *neighbor_table, const int32_t *in_degree_table,
                   const int32_t *out_degree_table, const float *neighbor_lin_weight,
                   const float *neighbor_lin_bias, const float *self_lin_weight, int emb_in,
                   int emb_out, int math);
/* lib:1627-1742 gine_conv: edge features enter through edge_index_table (lib:1126-1166);
 * edge_feature_table [num_edges][edge_dim] in COO (edge id) order, edge_proj_weight
 * [emb_in][edge_dim]; then the GIN MLP (hidden, emb_out). */
int gnnb_gine_conv(int num_nodes, int num_edges, const float *x_in, float *x_out,
                   const float *edge_feature_table, const int32_t *edge_list,
                   const int32_t *neighbor_table_offsets, const int32_t *neighbor_table,
                   const int32_t *edge_index_table, const int32_t *in_degree_table,
                   const int32_t *out_degree_table, const float *edge_proj_weight,
                   const float *edge_proj_bias, const float *mlp_0_weight, const float *mlp_0_bias,
                   const float *mlp_1_weight, const float *mlp_1_bias, float gin_eps, int emb_in,
                   int hidden, int emb_out, int edge_dim, int math);
/* lib:2398-2499 lg_conv: y_v = sum_u x_u / sqrt(deg_in(v) deg_in(u)) (no weights, emb_out = emb_in) */
int gnnb_lg_conv(int num_nodes, int num_edges, const float *x_in, float *x_out,
                 const int32_t *edge_list, const int32_t *neighbor_table_offsets,
                 const int32_t *neighbor_table, const int32_t *in_degree_table,
                 const int32_t *out_degree_table, int emb, int math);
/* lib:2564-2634 simple_conv: y_v = sum_u x_u */
int gnnb_simple_conv(int num_nodes, int num_edges, const float *x_in, float *x_out,
                     const int32_t *edge_list, const int32_t *neighbor_table_offsets,
                     const int32_t *neighbor_table, const int32_t *in_degree_table,
                     const int32_t *out_degree_table, int emb, int math);
/* lib:1891-2157 (transform 2F->F, apply 13F->emb_out, final emb_out->emb_out).  Like the reference's
 * float build, a node with in-degree 0 gets std = sqrt(0/0 + 1e-5) = NaN (lib:702), so its output row
 * is NaN (PyG clamps the degree instead; parity here is with the reference).  The model paths keep the
 * same semantics: ReLU maps such rows to 0, other activations keep the NaN. */
int gnnb_pna_conv(int num_nodes, int num_edges, const float *x_in, float *x_out,
                  const int32_t *edge_list, const int32_t *neighbor_table_offsets,
                  const int32_t *neighbor_table, const int32_t *in_degree_table,
                  const int32_t *out_degree_table, const float *transform_lin_weight,
                  const float *transform_lin_bias, const float *apply_lin_weight,
                  const float *apply_lin_bias, const float *final_lin_weight,
                  const float *final_lin_bias, float pna_avg_degree_log, int emb_in, int emb_out);
/* lib:2709-2803 */
int gnnb_global_add_pool(int num_nodes, int num_edges, const float *x, float *pooled, int emb);
int gnnb_global_mean_pool(int num_nodes, int num_edges, const float *x, float *pooled, int emb);
int gnnb_global_max_pool(int num_nodes, int num_edges, const float *x, float *pooled, int emb);

/* ---- one large graph, 1D row partition across GPUs (no reference counterpart; SURVEY 8e) ---- */
/* DEVICE pointers only; work is enqueued on `stream` (a cudaStream_t, NULL = default stream).
 * This rank owns destination rows [row_begin, row_begin + n_local); edge_list_local holds their
 * in-edges with GLOBAL node ids.  Tables: in-degree and offsets of the owned rows, neighbor table
 * with global source ids, stable in COO order like lib:1086-1124. */
int gnnb_partition_tables(const int32_t *edge_list_local, int row_begin, int n_local,
                          int num_edges_local, int32_t *in_degree_local, int32_t *offsets_local,
                          int32_t *neighbor_table_global, void *stream);
/* dinv[i] = 1 / sqrt(1 + in_degree[i]) (the factorised GCN normalisation, lib:1249-1252) */
int gnnb_degree_inv_sqrt(const int32_t *in_degree, float *dinv, int n, void *stream);
/* y_local[n_local][emb_out] = act(gcn_conv(x_full)[owned rows] (+ skip_local)); x_full holds the
 * features of ALL n_total nodes (after the halo all-gather), dinv_full their 1/sqrt(1+deg). */
int gnnb_gcn_conv_partition(int n_local, int row_begin, int n_total, int num_edges_local,
                            const float *x_full, float *y_local, const int32_t *offsets_local,
                            const int32_t *neighbor_table_global, const int32_t *in_degree_local,
                            const float *dinv_full, const float *weight, const float *bias,
                            const float *skip_local, int emb_in, int emb_out, int act, void *stream);

/* Per-rank partial of the global pools for a row-partitioned graph: out[0..F) = column sums,
 * out[F..2F) = column maxima of x[n][F] (lib:2709-2803; device pointers, asynchronous on stream).
 * The ranks combine them with all_reduce(sum) / all_reduce(max). */
int gnnb_pool_partial(const float *x, int64_t n, int F, float *out, void *stream);

/* ---- halo exchange for the row partition (no reference counterpart; SURVEY 8e) -------------
 * Every rank keeps its owned feature rows followed by ONE copy of each remote row its in-edges
 * reference: the "ext" space [owned rows | halo rows grouped by owner rank], built once by
 * gnn_builder_b200/distributed.py.  DEVICE pointers, work enqueued on `stream`. */
/* dst[p][i][0..F) = x[send_idx[send_off[p] + i]][0..F) for every peer p < n_peers (<= 16).
 * send_off (n_peers + 1 entries) and dst (n_peers pointers) are HOST arrays; dst[p] is a local
 * send buffer (NCCL transport) or the peer's halo region through a CUDA-IPC mapping (the rows
 * then leave as NVLink stores).  max_ctas <= 0: one CTA per SM, which keeps enough bytes in flight
 * for one NVLink direction and leaves the rest of every SM to the kernel running beside it. */
int gnnb_halo_pack(const float *x, int ldx, int F, const int32_t *send_idx, const int64_t *send_off,
                   float *const *dst, int n_peers, int max_ctas, void *stream);
/* the same with an explicit sub-range per peer: rows send_idx[start[p] .. start[p] + count[p]) go to
 * dst[p][0 .. count[p]) -- one block of owned rows at a time, so the sends of a finished block
 * travel while the next block is still being computed */
int gnnb_halo_pack_ranges(const float *x, int ldx, int F, const int32_t *send_idx,
                          const int64_t *start, const int64_t *count, float *const *dst, int n_peers,
                          int max_ctas, void *stream);
/* system-scope release store of `value` to peer_flags[p] (HOST array of n_peers device pointers,
 * NULL entries skipped): "this rank's rows for epoch `value` have landed" */
int gnnb_halo_signal(uint64_t *const *peer_flags, int n_peers, uint64_t value, void *stream);
/* waits on the device until flags[0..n_flags) >= value (acquire, system scope); after ~2 s of SM
 * clocks it sets *timed_out (device int) instead of hanging */
int gnnb_halo_wait(const uint64_t *flags, int n_flags, uint64_t value, int *timed_out, void *stream);
/* CUDA-IPC plumbing for the peer mappings: a zeroed device allocation + its 64-byte handle; open /
 * close a peer's handle in this process; free */
int gnnb_ipc_alloc(size_t bytes, void **ptr, void *handle64);
int gnnb_ipc_open(const void *handle64, void **ptr);
int gnnb_ipc_close(void *ptr);
int gnnb_ipc_free(void *ptr);
/* Sets bit 31 on the entries of a neighbor table whose source is among the most-referenced ones
 * whose feature rows (row_bytes each) fit budget_bytes: the aggregation keeps those rows resident
 * in L2 (evict_last) and streams the others (evict_first).  In place; *num_hubs (host) = marked
 * sources.  One host synchronisation. */
int gnnb_mark_hub_sources(int32_t *neighbor_table, int num_entries, int num_sources, int row_bytes,
                          int64_t budget_bytes, int *num_hubs, void *stream);
/* One GCN layer on the owned rows of an ext-space partition with its CSR split by source:
 * own_* = edges whose source this rank owns, halo_* = edges whose source is a halo row (offsets /
 * counts per owned row, neighbor entries = ext indices).  phase 1: aggregate the owned-source
 * edges (needs no halo: overlaps the exchange); phase 2: add the halo-source edges, normalise
 * (lib:1246-1278) and transform, y_local[n_local][emb_out] = act(agg.W^T + b (+ skip_local));
 * phase 3: both.  dinv_ext[n_ext] = 1/sqrt(1 + in-degree) of every ext row.  row_begin /
 * row_count restrict the call to one block of owned rows (row_count <= 0: all of them); every
 * pointer still addresses row 0. */
int gnnb_gcn_conv_halo(int n_local, int n_ext, const float *x_ext, float *y_local,
                       const int32_t *own_offsets, const int32_t *own_counts, const int32_t *own_nbr,
                       const int32_t *halo_offsets, const int32_t *halo_counts,
                       const int32_t *halo_nbr, const float *dinv_ext, const float *weight,
                       const float *bias, const float *skip_local, int emb_in, int emb_out, int act,
                       int phase, int hub_bit, int row_begin, int row_count, void *stream);
/* The same for the other convs, FAST math, whole layers (no row blocks).  phase 1 aggregates the
 * owned-source edges (PNA: computes the pre-transform instead, see below), phase 2 the halo-source
 * edges and the transform, phase 3 both; y_local[n_local][emb_out] = act(conv (+ skip_local)).
 * Weights in the reference layout as for gnnb_gin_conv / gnnb_sage_conv / gnnb_pna_conv.
 * hub_bit: the neighbor tables carry the marks of gnnb_mark_hub_sources.
 *
 * GIN (lib:1440-1549): sum over both parts + (1 + gin_eps) x_v, then linear_0 + ReLU and
 * linear_1. */
int gnnb_gin_conv_halo(int n_local, int n_ext, const float *x_ext, float *y_local,
                       const int32_t *own_offsets, const int32_t *own_counts, const int32_t *own_nbr,
                       const int32_t *halo_offsets, const int32_t *halo_counts,
                       const int32_t *halo_nbr, const float *mlp_0_weight, const float *mlp_0_bias,
                       const float *mlp_1_weight, const float *mlp_1_bias, float gin_eps,
                       const float *skip_local, int emb_in, int hidden, int emb_out, int act,
                       int phase, int hub_bit, void *stream);
/* SAGE, mean aggregation (lib:2211-2341): the parts' counts walk the edges and in_degree_local
 * (the FULL in-degree of every owned row) divides; in-degree 0 gives a zero mean. */
int gnnb_sage_conv_halo(int n_local, int n_ext, const float *x_ext, float *y_local,
                        const int32_t *own_offsets, const int32_t *own_counts, const int32_t *own_nbr,
                        const int32_t *halo_offsets, const int32_t *halo_counts,
                        const int32_t *halo_nbr, const int32_t *in_degree_local,
                        const float *neighbor_lin_weight, const float *neighbor_lin_bias,
                        const float *self_lin_weight, const float *skip_local, int emb_in,
                        int emb_out, int act, int phase, int hub_bit, void *stream);
/* PNA (lib:1891-2157).  What crosses ranks is A = x.W_nbr^T rather than x (W_pre = [W_self |
 * W_nbr]): phase 1 writes A of the owned rows to a_ext[0 .. n_local) and keeps B = x.W_self^T +
 * b_pre in library scratch (the caller then sends the A rows, e.g. with gnnb_halo_pack, into the
 * peers' a_ext halo regions); phase 2, once this rank's halo rows of A have arrived in
 * a_ext[n_local .. n_ext), reduces t = A_u + B_v over both parts in order (max, min, mean, std with
 * the full in_degree_local; in-degree 0 gives std = NaN as in gnnb_pna_conv) and applies the
 * apply and final linears.  x_local[n_local][emb_in] are the owned input rows; a_ext is
 * [n_ext][emb_in].  Hub marks in the neighbor tables are ignored. */
int gnnb_pna_conv_halo(int n_local, int n_ext, const float *x_local, float *a_ext, float *y_local,
                       const int32_t *own_offsets, const int32_t *own_counts, const int32_t *own_nbr,
                       const int32_t *halo_offsets, const int32_t *halo_counts,
                       const int32_t *halo_nbr, const int32_t *in_degree_local,
                       const float *transform_lin_weight, const float *transform_lin_bias,
                       const float *apply_lin_weight, const float *apply_lin_bias,
                       const float *final_lin_weight, const float *final_lin_bias,
                       float pna_avg_degree_log, const float *skip_local, int emb_in, int emb_out,
                       int act, int phase, void *stream);
/* The attention convs (PyG GATConv / GATv2Conv, concat heads, no edge features), FAST math.  An
 * attention layer gathers what its GEMM produced for each source, so what crosses ranks is that
 * GEMM output, and no GEMM runs on a halo row.  The CSR is the rank's own, whole
 * (offsets_local / in_degree_local as from gnnb_partition_tables, which are the FULL in-degrees),
 * with every neighbor entry mapped to its ext index (nbr_ext, same order).  phase 1 computes the
 * GEMM output of the owned rows into rows [0, n_local) of the ext buffer (the caller then sends
 * them, e.g. with gnnb_halo_pack at the width below, into the peers' halo regions); phase 2, once
 * rows [n_local, n_ext) have arrived, runs the attention softmax and the epilogue,
 * y_local[n_local][emb_out] = act(sum_u alpha_vu m_u + bias (+ skip_local)); phase 3 both.
 * Input self loops are replaced by one per node as PyG does; rows above the heavy-row threshold
 * are cut into chunks.  x_local[n_local][emb_in] are the owned input rows.  emb_out = heads * C,
 * heads 1..GNNB_GAT_MAX_HEADS.  Weights in PyG's layout, device pointers.
 *
 * GAT: g_ext [n_ext][ld_g], ld_g = round_up(emb_out + 2 heads, 4), rows [h | a_src | a_dst].  The
 * per-head vectors w_src,h = W_h^T att_src,h (w_dst alike) are folded into the GEMM weight on every
 * phase-1 call, in double and rounded once as the model handle does. */
int gnnb_gat_conv_halo(int n_local, int n_ext, const float *x_local, float *g_ext, float *y_local,
                       const int32_t *offsets_local, const int32_t *in_degree_local,
                       const int32_t *nbr_ext, const float *att_src, const float *att_dst,
                       const float *bias, const float *lin_weight, int heads, float negative_slope,
                       const float *skip_local, int emb_in, int emb_out, int act, int phase,
                       void *stream);
/* GATv2: xl_ext [n_ext][ld_l], ld_l = round_up(emb_out, 4), holds xl = x.W_l^T + b_l; xr = x.W_r^T +
 * b_r of the owned rows stays in library scratch from phase 1 to phase 2 (one layer in flight per
 * thread).  A head's width C must be at most 256 when a multiple of 4, else at most 64. */
int gnnb_gatv2_conv_halo(int n_local, int n_ext, const float *x_local, float *xl_ext, float *y_local,
                         const int32_t *offsets_local, const int32_t *in_degree_local,
                         const int32_t *nbr_ext, const float *att, const float *bias,
                         const float *lin_l_weight, const float *lin_l_bias,
                         const float *lin_r_weight, const float *lin_r_bias, int heads,
                         float negative_slope, const float *skip_local, int emb_in, int emb_out,
                         int act, int phase, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GNNB_B200_H */
