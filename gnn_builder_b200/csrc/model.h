// Model handle internals (not part of the public ABI).
#pragma once

#include <string>
#include <vector>

#include "kernels.h"

namespace gnnb {

struct ParamSlot {
    std::string name;
    std::vector<int> shape;   // [out] or [out][in]
    size_t numel = 0;
    std::vector<float> host;  // copy kept until finalize
    bool set = false;
};

// a Linear packed for the kernels: Wt[in][ldw] (transposed, zero padded), bias[out]
struct PackedLinear {
    const float *Wt = nullptr;
    const float *bias = nullptr;
    const float *img = nullptr;   // tensor-core weight image (gemm_tc.cu), built at finalize
    int in = 0, out = 0, ldw = 0;
};

struct LayerPack {
    int fi = 0, fo = 0;
    PackedLinear a, b, c, d;  // meaning depends on the conv type (see model.cu pack_layer)
    PackedLinear e;           // GINE: the edge linear W_e^T [edge_dim][ldw], b_e
};
// GAT: a = [W | w_src | w_dst]^T, H*C + 2H columns and no bias (one GEMM gives h and both logits
// of a row); b carries only the conv bias [H*C], which the aggregation epilogue adds.  With edge_dim,
// the edge linear folded with att_edge is one [L*H][edge_dim] table for all layers (gat_w_edge).
// GATv2: a = lin_l and b = lin_r (weights and biases, two GEMMs into one [T][round_up(2 H*C, 4)]
// buffer); c carries att [H*C] and d the conv bias [H*C] as vectors; e = lin_edge's W_e^T
// [edge_dim][ldw] without a bias (edge_dim > 0 only), applied per edge by the aggregation.
// TransformerConv: a = lin_key and b = lin_value (two GEMMs into [k | v], one [T][round_up(2 H*C, 4)]
// buffer), c = lin_query with 1/sqrt(C) folded into its weight and bias, d = lin_skip (its GEMM runs
// without the bias; the aggregation epilogue adds d.bias), e = lin_edge's W_e^T as for GATv2.

// fused-kernel plans (fused.cu, fused_tc.cu)
struct FusedPlan;
struct TcPlan;

// Optional per-kernel-class timing with CUDA events on the launching stream (bench.py uses it
// for the live roofline numbers).  Off by default: no events are recorded.
enum ProfCat { PROF_TABLES = 0, PROF_AGG = 1, PROF_GEMM = 2, PROF_POOL = 3, PROF_FUSED = 4,
               PROF_EDGE_LOGITS = 5, PROF_NCAT = 8 };
struct Profiler {
    bool on = false;
    struct Rec { int cat; cudaEvent_t a, b; };
    std::vector<Rec> recs;
    std::vector<cudaEvent_t> free_events;
    cudaEvent_t get()
    {
        cudaEvent_t e = nullptr;
        if (!free_events.empty()) { e = free_events.back(); free_events.pop_back(); }
        else cudaEventCreate(&e);
        return e;
    }
    void release()
    {
        for (Rec &r : recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
        for (cudaEvent_t e : free_events) cudaEventDestroy(e);
        recs.clear();
        free_events.clear();
    }
};
struct ProfScope {
    Profiler *p; cudaStream_t s; int idx = -1;
    ProfScope(Profiler &prof, int cat, cudaStream_t stream) : p(&prof), s(stream)
    {
        if (!p->on) return;
        Profiler::Rec r{cat, p->get(), p->get()};
        cudaEventRecord(r.a, s);
        p->recs.push_back(r);
        idx = (int)p->recs.size() - 1;
    }
    ~ProfScope()
    {
        if (idx >= 0) cudaEventRecord(p->recs[idx].b, s);
    }
};

}  // namespace gnnb

struct gnnb_model {
    gnnb_model_desc d{};
    int device = 0;
    cudaStream_t stream = nullptr;
    bool finalized = false;
    int path = GNNB_PATH_AUTO;
    int math = GNNB_MATH_FAST;

    std::vector<gnnb::ParamSlot> params;
    gnnb::DeviceBuf weights;  // all packed weights, one allocation
    gnnb::DeviceBuf weight_images;  // tensor-core images of the same linears (layerwise tcgen05 GEMM)
    std::vector<gnnb::LayerPack> layers;
    std::vector<gnnb::PackedLinear> head;
    gnnb::FusedPlan *fused = nullptr;
    gnnb::TcPlan *fused_tc = nullptr;

    // staging for host-pointer calls
    gnnb::DeviceBuf st_x, st_coo, st_ef, st_nptr, st_eptr, st_out;
    // chunked ingest pipeline (host buffers -> fused kernel): double-buffered chunk staging, a
    // copy-in and a copy-out stream beside the compute stream, events for the hand-offs
    gnnb::DeviceBuf ch_x[2], ch_coo[2], ch_nptr[2], ch_eptr[2];
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
    // layerwise workspaces
    gnnb::DeviceBuf in_deg, out_deg, offsets, nbr, nbr_hub, dinv, feat[2], agg, hid, wide, pooled,
        hbuf[2], pool_tmp, ptr_tmp;
    // GINE, GATv2, TransformerConv: edge id and edge features per neighbor slot
    gnnb::DeviceBuf edge_index, ef_sorted;
    gnnb::DeviceBuf self_attr;   // GATv2 with edge_dim: each row's self-loop attribute [n][lde]
    // GAT with edge_dim: the edge logits of every layer and head per neighbor slot and per row
    // (gat_edge_logits_kernel), and the folded edge weights [L*H][edge_dim] inside `weights`
    gnnb::DeviceBuf elog, self_elog;
    const float *gat_w_edge = nullptr;
    int last_hub_rows = 0;   // sources whose feature rows the last large-graph run kept L2-resident
    gnnb::TableWorkspace tws;
    gnnb::HeavyList heavy;       // rows above the heavy threshold of the current layerwise run
    gnnb::DeviceBuf edge_flag;   // layerwise path: set by the table kernels on an out-of-range endpoint

    gnnb::Profiler prof;
    int last_launches = 0;
    int last_path = 0;
    int last_kernel = 0;  // 1 layerwise, 2 fused fp32-FMA, 3 fused tcgen05
    const float *last_emb = nullptr;
    int last_emb_ld = 0;
    int64_t last_emb_rows = 0;

    int emb_dim() const { return d.num_layers == 0 ? d.in_dim : d.out_dim; }
    // GINE, and GAT, GATv2 and TransformerConv with edge_dim: edge features come through the *_edges
    // entry points
    bool has_edge_features() const { return d.edge_dim > 0; }
    void layer_dims(int layer, int *fi, int *fo) const
    {
        if (d.num_layers == 1) { *fi = d.in_dim; *fo = d.out_dim; return; }
        *fi = layer == 0 ? d.in_dim : d.hidden_dim;
        *fo = layer == d.num_layers - 1 ? d.out_dim : d.hidden_dim;
    }
};

namespace gnnb {

// fused.cu --------------------------------------------------------------------------------
// Builds the fused kernel's weight image for a finalized model; returns GNNB_OK and leaves
// m->fused null when the configuration is not supported by the fused kernel.
int fused_prepare(gnnb_model *m);
void fused_release(gnnb_model *m);
// true when the fused kernel can run this batch (every graph fits a CTA tile)
bool fused_supports(const gnnb_model *m, int max_nodes_in_batch, int max_edges_in_batch);
// max_nodes: upper bound on the node count of any graph in the batch (sets the tile window)
int fused_run(gnnb_model *m, const float *x, const int32_t *coo, const int64_t *node_ptr,
              const int64_t *edge_ptr, int n_graphs, int64_t total_nodes, int max_nodes, float *out,
              cudaStream_t s, int *launches);
// after the stream is synchronised: 0 ok, 1 a tile overflowed (re-run layerwise), 2 bad edge index
int fused_status(gnnb_model *m, int *status);
int fused_tile_rows(const gnnb_model *m);

// fused_tc.cu: same contract as the fused_* functions, tensor-core node transform
int fused_tc_prepare(gnnb_model *m);
void fused_tc_release(gnnb_model *m);
bool fused_tc_supports(const gnnb_model *m, int max_nodes_in_batch, int max_edges_in_batch);
// reset_status: clear the device status word first (false when a batch is run as several chunks)
int fused_tc_run(gnnb_model *m, const float *x, const int32_t *coo, const int64_t *node_ptr,
                 const int64_t *edge_ptr, int n_graphs, int64_t total_nodes, int max_nodes,
                 float *out, cudaStream_t s, int *launches, bool reset_status = true);
int fused_tc_status(gnnb_model *m, int *status);

}  // namespace gnnb
