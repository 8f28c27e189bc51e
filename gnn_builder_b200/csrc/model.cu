// Model handle: replaces the generated `<name>_top` (model.cpp.jinja:686-766) with a runtime
// description + packed device weights, and runs a batch of graphs either through the fused
// whole-model kernel (fused.cu) or layer by layer on the batch's disjoint union (this file):
//
//   tables (cpp:737-758) -> per conv layer: aggregate -> GEMM(s) with fused bias/skip/activation
//   (cpp:264-345) -> segmented global pooling (cpp:413-449) -> MLP head GEMMs (cpp:454-530).
#include "model.h"

#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstring>
#include <mutex>

namespace gnnb {

static thread_local std::string g_error;

void set_error(const std::string &msg) { g_error = msg; }

int cuda_fail(cudaError_t e, const char *what, const char *file, int line)
{
    char buf[512];
    snprintf(buf, sizeof(buf), "CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e),
             file, line, what);
    g_error = buf;
    cudaGetLastError();  // clear the sticky-less error state
    return GNNB_ERR_CUDA;
}

bool is_device_pointer(const void *p)
{
    if (p == nullptr) return false;
    cudaPointerAttributes attr;
    cudaError_t e = cudaPointerGetAttributes(&attr, p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged;
}

namespace {

// Every entry point runs on the handle's device and leaves the caller's current device as it
// found it (a host thread that drives several GPUs, or torch's notion of the current device,
// must not be switched behind its back).
struct DeviceScope {
    int prev = -1;
    explicit DeviceScope(int dev)
    {
        int cur = -1;
        if (cudaGetDevice(&cur) == cudaSuccess && cur != dev && cudaSetDevice(dev) == cudaSuccess) prev = cur;
        else if (cur != dev) cudaGetLastError();
    }
    ~DeviceScope()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
    DeviceScope(const DeviceScope &) = delete;
    DeviceScope &operator=(const DeviceScope &) = delete;
};

void add_param(gnnb_model *m, const std::string &name, std::vector<int> shape)
{
    ParamSlot p;
    p.name = name;
    p.shape = shape;
    p.numel = 1;
    for (int s : shape) p.numel *= (size_t)s;
    m->params.push_back(std::move(p));
}

// Flat parameter list in the reference's order (models.py:607-624; SURVEY appendix B).
void enumerate_params(gnnb_model *m)
{
    const gnnb_model_desc &d = m->d;
    int in = m->emb_dim() * d.num_pools;
    for (int j = 0; j < d.mlp_num_linear; j++) {
        const int out = (j == d.mlp_num_linear - 1) ? d.mlp_out : d.mlp_hidden;
        const std::string base = "mlp_head_linear_layers_" + std::to_string(j);
        add_param(m, base + "_weight", {out, in});
        add_param(m, base + "_bias", {out});
        in = out;
    }
    for (int k = 0; k < d.num_layers; k++) {
        int fi, fo;
        m->layer_dims(k, &fi, &fo);
        const std::string base = "gnn_convs_" + std::to_string(k);
        switch (d.conv_type) {
        case GNNB_CONV_GCN:
            add_param(m, base + "_conv_bias", {fo});
            add_param(m, base + "_conv_lin_weight", {fo, fi});
            break;
        case GNNB_CONV_GIN:
        case GNNB_CONV_GINE:
            add_param(m, base + "_mlp_linear_0_weight", {fo, fi});
            add_param(m, base + "_mlp_linear_0_bias", {fo});
            add_param(m, base + "_mlp_linear_1_weight", {fo, fo});
            add_param(m, base + "_mlp_linear_1_bias", {fo});
            if (d.conv_type == GNNB_CONV_GINE) {   // PyG GINEConv's edge linear: lin [F_in][edge_dim]
                add_param(m, base + "_conv_lin_weight", {fi, d.edge_dim});
                add_param(m, base + "_conv_lin_bias", {fi});
            }
            break;
        case GNNB_CONV_SAGE:
            add_param(m, base + "_conv_lin_l_weight", {fo, fi});
            add_param(m, base + "_conv_lin_l_bias", {fo});
            add_param(m, base + "_conv_lin_r_weight", {fo, fi});
            break;
        case GNNB_CONV_PNA:
            add_param(m, base + "_conv_pre_nns_0_0_weight", {fi, 2 * fi});
            add_param(m, base + "_conv_pre_nns_0_0_bias", {fi});
            add_param(m, base + "_conv_post_nns_0_0_weight", {fo, 13 * fi});
            add_param(m, base + "_conv_post_nns_0_0_bias", {fo});
            add_param(m, base + "_conv_lin_weight", {fo, fo});
            add_param(m, base + "_conv_lin_bias", {fo});
            break;
        case GNNB_CONV_GAT:   // PyG GATConv: its own parameters, then lin's (and lin_edge's)
            add_param(m, base + "_conv_att_src", {1, d.gat_heads, fo / d.gat_heads});
            add_param(m, base + "_conv_att_dst", {1, d.gat_heads, fo / d.gat_heads});
            if (m->has_edge_features())
                add_param(m, base + "_conv_att_edge", {1, d.gat_heads, fo / d.gat_heads});
            add_param(m, base + "_conv_bias", {fo});
            add_param(m, base + "_conv_lin_weight", {fo, fi});
            if (m->has_edge_features()) add_param(m, base + "_conv_lin_edge_weight", {fo, d.edge_dim});
            break;
        case GNNB_CONV_GATV2:   // PyG GATv2Conv: its own parameters, then lin_l's, lin_r's, lin_edge's
            add_param(m, base + "_conv_att", {1, d.gat_heads, fo / d.gat_heads});
            add_param(m, base + "_conv_bias", {fo});
            add_param(m, base + "_conv_lin_l_weight", {fo, fi});
            add_param(m, base + "_conv_lin_l_bias", {fo});
            add_param(m, base + "_conv_lin_r_weight", {fo, fi});
            add_param(m, base + "_conv_lin_r_bias", {fo});
            if (m->has_edge_features()) add_param(m, base + "_conv_lin_edge_weight", {fo, d.edge_dim});
            break;
        case GNNB_CONV_TRANSFORMER:   // PyG TransformerConv: lin_key, lin_query, lin_value, lin_edge, lin_skip
            for (const char *lin : {"_conv_lin_key", "_conv_lin_query", "_conv_lin_value"}) {
                add_param(m, base + lin + "_weight", {fo, fi});
                add_param(m, base + lin + "_bias", {fo});
            }
            if (m->has_edge_features()) add_param(m, base + "_conv_lin_edge_weight", {fo, d.edge_dim});
            add_param(m, base + "_conv_lin_skip_weight", {fo, fi});
            add_param(m, base + "_conv_lin_skip_bias", {fo});
            break;
        }
    }
}

// host-side packer: appends Wt[in][ldw] for W[out][ld_src] columns [col0, col0+in)
struct Packer {
    std::vector<float> data;
    size_t reserve(size_t n)
    {
        size_t off = (data.size() + 3) / 4 * 4;
        data.resize(off + (n + 3) / 4 * 4, 0.0f);
        return off;
    }
    size_t add_transposed(const float *W, int out, int ld_src, int col0, int in, int ldw,
                          int out_col0 = 0, size_t into = (size_t)-1)
    {
        size_t off = into;
        if (off == (size_t)-1) off = reserve((size_t)in * ldw);
        for (int k = 0; k < in; k++)
            for (int n = 0; n < out; n++)
                data[off + (size_t)k * ldw + out_col0 + n] = W[(size_t)n * ld_src + col0 + k];
        return off;
    }
    size_t add_vector(const float *b, int n, int pad_front = 0)
    {
        size_t off = reserve((size_t)n + pad_front);
        for (int i = 0; i < n; i++) data[off + pad_front + i] = b[i];
        return off;
    }
};

struct PendingLinear {
    size_t wt_off = 0, bias_off = 0;
    bool has_bias = false;
    int in = 0, out = 0, ldw = 0;
};

PackedLinear resolve(const PendingLinear &p, const float *base)
{
    PackedLinear l;
    l.Wt = base + p.wt_off;
    l.bias = p.has_bias ? base + p.bias_off : nullptr;
    l.in = p.in; l.out = p.out; l.ldw = p.ldw;
    return l;
}

PendingLinear pack_linear(Packer &pk, const float *W, const float *b, int out, int in,
                          int ld_src = -1, int col0 = 0)
{
    PendingLinear p;
    p.in = in; p.out = out; p.ldw = round_up(out, 4);
    p.wt_off = pk.add_transposed(W, out, ld_src < 0 ? in : ld_src, col0, in, p.ldw);
    if (b) {
        p.has_bias = true;
        p.bias_off = pk.add_vector(b, out);
    }
    return p;
}

const float *param(const gnnb_model *m, size_t idx) { return m->params[idx].host.data(); }

}  // namespace
}  // namespace gnnb

using namespace gnnb;

// ============================================================================ library
extern "C" const char *gnnb_last_error(void) { return g_error.c_str(); }
extern "C" int gnnb_version(void) { return 100; }
extern "C" int gnnb_device_count(int *count)
{
    GNNB_REQUIRE(count != nullptr, "count is null");
    *count = 0;
    GNNB_CUDA(cudaGetDeviceCount(count));
    return GNNB_OK;
}

// Page-locks a caller-owned host buffer (cudaHostRegister) so that the host-buffer entry points copy
// it at full PCIe rate and asynchronously; worth it for buffers that are passed more than once
// (registration itself costs about as much as one pageable copy).
extern "C" int gnnb_host_register(void *ptr, size_t bytes)
{
    GNNB_REQUIRE(ptr != nullptr && bytes > 0, "host register: null buffer");
    GNNB_CUDA(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable));
    return GNNB_OK;
}
extern "C" int gnnb_host_unregister(void *ptr)
{
    GNNB_REQUIRE(ptr != nullptr, "host unregister: null buffer");
    GNNB_CUDA(cudaHostUnregister(ptr));
    return GNNB_OK;
}

// ============================================================================ model handle
extern "C" int gnnb_model_create(const gnnb_model_desc *desc, int device, gnnb_model_t **out)
{
    GNNB_REQUIRE(desc != nullptr && out != nullptr, "null argument");
    // edge_dim and the GAT fields after it are only required of GINE and GAT callers: copy the
    // fields before it, then read it for GINE and GAT only (a caller built against the older,
    // shorter struct never has bytes read past its end; a GAT caller's struct always holds it)
    gnnb_model_desc d{};
    std::memcpy(&d, desc, offsetof(gnnb_model_desc, edge_dim));
    GNNB_REQUIRE((d.conv_type >= GNNB_CONV_GCN && d.conv_type <= GNNB_CONV_GAT) ||
                     d.conv_type == GNNB_CONV_GATV2 || d.conv_type == GNNB_CONV_TRANSFORMER,
                 "conv_type must be GCN, GIN, SAGE, PNA, GINE, GAT, GATv2 or TransformerConv (0..5, 7 "
                 "or 8)");
    if (d.conv_type == GNNB_CONV_GINE) {
        d.edge_dim = desc->edge_dim;
        GNNB_REQUIRE(d.edge_dim >= 1 && d.edge_dim <= kGineMaxEdgeDim,
                     "GINE edge_dim must be 1.." + std::to_string(kGineMaxEdgeDim));
    }
    GNNB_REQUIRE(d.num_layers >= 0 && d.num_layers <= 64, "num_layers out of range");
    GNNB_REQUIRE(d.in_dim > 0 && d.hidden_dim > 0 && d.out_dim > 0, "dimensions must be positive");
    const bool transformer = d.conv_type == GNNB_CONV_TRANSFORMER;
    if (d.conv_type == GNNB_CONV_GAT || d.conv_type == GNNB_CONV_GATV2 || transformer) {
        // the GAT fields follow edge_dim; only GAT, GATv2 and TransformerConv callers set them, and
        // TransformerConv has no slope to read
        const std::string conv = d.conv_type == GNNB_CONV_GAT     ? "GAT"
                                 : d.conv_type == GNNB_CONV_GATV2 ? "GATv2"
                                                                  : "TransformerConv";
        d.edge_dim = desc->edge_dim;
        GNNB_REQUIRE(d.edge_dim >= 0 && d.edge_dim <= kGineMaxEdgeDim,
                     conv + " edge_dim must be 0 (no edge features) or 1.." +
                         std::to_string(kGineMaxEdgeDim));
        d.gat_heads = desc->gat_heads;
        if (!transformer) d.gat_negative_slope = desc->gat_negative_slope;
        GNNB_REQUIRE(d.gat_heads >= 1 && d.gat_heads <= GNNB_GAT_MAX_HEADS,
                     conv + " gat_heads must be 1.." + std::to_string(GNNB_GAT_MAX_HEADS));
        GNNB_REQUIRE(std::isfinite(d.gat_negative_slope), conv + " gat_negative_slope must be finite");
        for (int k = 0; k < d.num_layers; k++) {
            const int fo = k == d.num_layers - 1 ? d.out_dim : d.hidden_dim;
            GNNB_REQUIRE(fo % d.gat_heads == 0,
                         conv + ": every layer's output width (hidden_dim, out_dim) must be a multiple "
                         "of gat_heads, got width " + std::to_string(fo) + " with " +
                             std::to_string(d.gat_heads) + " heads");
            // GATv2 and TransformerConv spread a head's columns over at most one warp (agg.cu)
            const int C = fo / d.gat_heads;
            GNNB_REQUIRE(d.conv_type == GNNB_CONV_GAT ||
                             C <= (C % 4 == 0 ? kGatv2MaxHeadWidth : kGatv2MaxHeadWidth1),
                         conv + ": a head's width (layer width / gat_heads) must be at most " +
                             std::to_string(kGatv2MaxHeadWidth) + " when a multiple of 4, else at "
                             "most " + std::to_string(kGatv2MaxHeadWidth1) + ", got " +
                             std::to_string(C));
        }
    }
    GNNB_REQUIRE(d.num_layers > 0 || d.in_dim == d.out_dim,
                 "gnn_num_layers=0 needs gnn_output_dim == graph_input_feature_dim (models.py:512)");
    GNNB_REQUIRE(d.num_pools >= 1 && d.num_pools <= 4, "1..4 global pooling aggregations");
    for (int p = 0; p < d.num_pools; p++)
        GNNB_REQUIRE(d.pools[p] >= GNNB_POOL_ADD && d.pools[p] <= GNNB_POOL_MAX,
                     "pooling must be add, mean or max (models.py:317-321)");
    GNNB_REQUIRE(d.mlp_num_linear >= 1 && d.mlp_num_linear <= 64, "mlp_num_linear out of range");
    GNNB_REQUIRE(d.mlp_out > 0 && (d.mlp_num_linear == 1 || d.mlp_hidden > 0), "bad MLP dims");
    GNNB_REQUIRE(d.gnn_act >= 0 && d.gnn_act <= GNNB_ACT_COS && d.mlp_act >= 0 &&
                     d.mlp_act <= GNNB_ACT_COS && d.out_act >= 0 && d.out_act <= GNNB_ACT_COS,
                 "unknown activation id");
    int ndev = 0;
    GNNB_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0) GNNB_CUDA(cudaGetDevice(&device));
    GNNB_REQUIRE(device < ndev, "no such CUDA device");
    DeviceScope on_device(device);
    gnnb_model *m = new gnnb_model();
    m->d = d;
    m->device = device;
    cudaError_t e = cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete m;
        return cuda_fail(e, "cudaStreamCreate", __FILE__, __LINE__);
    }
    bool ok = cudaStreamCreateWithFlags(&m->h2d_stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&m->d2h_stream, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; i < 2 && ok; i++)
        ok = cudaEventCreateWithFlags(&m->ev_h2d[i], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&m->ev_done[i], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        gnnb_model_destroy(m);
        return cuda_fail(cudaGetLastError(), "creating the ingest streams/events", __FILE__, __LINE__);
    }
    enumerate_params(m);
    *out = m;
    return GNNB_OK;
}

extern "C" int gnnb_model_destroy(gnnb_model_t *m)
{
    if (!m) return GNNB_OK;
    DeviceScope on_device(m->device);
    if (m->stream) cudaStreamSynchronize(m->stream);
    fused_release(m);
    fused_tc_release(m);
    m->prof.release();
    DeviceBuf *bufs[] = {&m->weights, &m->weight_images, &m->st_x, &m->st_coo, &m->st_ef, &m->st_nptr, &m->st_eptr, &m->st_out,
                         &m->in_deg, &m->out_deg, &m->offsets, &m->nbr, &m->nbr_hub, &m->dinv,
                         &m->edge_index, &m->ef_sorted, &m->self_attr, &m->elog, &m->self_elog,
                         &m->feat[0], &m->feat[1], &m->agg, &m->hid, &m->wide, &m->pooled,
                         &m->hbuf[0], &m->hbuf[1], &m->pool_tmp, &m->ptr_tmp, &m->edge_flag};
    for (DeviceBuf *b : bufs) b->release();
    m->tws.release_all();
    m->heavy.release();
    for (int i = 0; i < 2; i++) {
        m->ch_x[i].release(); m->ch_coo[i].release(); m->ch_nptr[i].release(); m->ch_eptr[i].release();
        if (m->ev_h2d[i]) cudaEventDestroy(m->ev_h2d[i]);
        if (m->ev_done[i]) cudaEventDestroy(m->ev_done[i]);
    }
    if (m->h2d_stream) cudaStreamDestroy(m->h2d_stream);
    if (m->d2h_stream) cudaStreamDestroy(m->d2h_stream);
    if (m->stream) cudaStreamDestroy(m->stream);
    delete m;
    return GNNB_OK;
}

extern "C" int gnnb_model_num_params(const gnnb_model_t *m) { return m ? (int)m->params.size() : 0; }

extern "C" int gnnb_model_param_info(const gnnb_model_t *m, int index, const char **name,
                                     size_t *numel)
{
    GNNB_REQUIRE(m != nullptr && index >= 0 && index < (int)m->params.size(), "bad parameter index");
    if (name) *name = m->params[index].name.c_str();
    if (numel) *numel = m->params[index].numel;
    return GNNB_OK;
}

extern "C" int gnnb_model_set_param(gnnb_model_t *m, const char *name, const float *data,
                                    size_t numel)
{
    GNNB_REQUIRE(m != nullptr && name != nullptr && data != nullptr, "null argument");
    for (ParamSlot &p : m->params) {
        if (p.name == name) {
            if (p.numel != numel) {
                set_error("parameter " + p.name + ": expected " + std::to_string(p.numel) +
                          " elements, got " + std::to_string(numel));
                return GNNB_ERR_PARAM;
            }
            p.host.resize(numel);
            if (is_device_pointer(data)) {
                GNNB_CUDA(cudaMemcpy(p.host.data(), data, numel * sizeof(float),
                                     cudaMemcpyDeviceToHost));
            } else {
                std::memcpy(p.host.data(), data, numel * sizeof(float));
            }
            p.set = true;
            m->finalized = false;
            return GNNB_OK;
        }
    }
    set_error(std::string("unknown parameter name: ") + name);
    return GNNB_ERR_PARAM;
}

extern "C" int gnnb_model_finalize(gnnb_model_t *m)
{
    GNNB_REQUIRE(m != nullptr, "null model");
    for (const ParamSlot &p : m->params)
        if (!p.set) {
            set_error("parameter not set: " + p.name);
            return GNNB_ERR_STATE;
        }
    DeviceScope on_device(m->device);
    const gnnb_model_desc &d = m->d;
    Packer pk;
    std::vector<PendingLinear> head_p;
    struct PendingLayer { int fi, fo; PendingLinear a, b, c, d, e; };
    std::vector<PendingLayer> layer_p;
    size_t idx = 0;
    std::vector<float> gat_w_edge;   // GAT with edge_dim: [L][H][edge_dim]
    if (d.conv_type == GNNB_CONV_GAT && m->has_edge_features())
        gat_w_edge.resize((size_t)d.num_layers * d.gat_heads * d.edge_dim);
    {
        int in = m->emb_dim() * d.num_pools;
        for (int j = 0; j < d.mlp_num_linear; j++) {
            const int out = (j == d.mlp_num_linear - 1) ? d.mlp_out : d.mlp_hidden;
            head_p.push_back(pack_linear(pk, param(m, idx), param(m, idx + 1), out, in));
            idx += 2;
            in = out;
        }
    }
    for (int k = 0; k < d.num_layers; k++) {
        PendingLayer L{};
        m->layer_dims(k, &L.fi, &L.fo);
        const int fi = L.fi, fo = L.fo;
        switch (d.conv_type) {
        case GNNB_CONV_GCN:  // [bias, lin_weight]
            L.a = pack_linear(pk, param(m, idx + 1), param(m, idx), fo, fi);
            idx += 2;
            break;
        case GNNB_CONV_GIN:
            L.a = pack_linear(pk, param(m, idx), param(m, idx + 1), fo, fi);
            L.b = pack_linear(pk, param(m, idx + 2), param(m, idx + 3), fo, fo);
            idx += 4;
            break;
        case GNNB_CONV_GINE:  // a, b: the GIN MLP; e: the edge linear (read by the aggregation)
            L.a = pack_linear(pk, param(m, idx), param(m, idx + 1), fo, fi);
            L.b = pack_linear(pk, param(m, idx + 2), param(m, idx + 3), fo, fo);
            L.e = pack_linear(pk, param(m, idx + 4), param(m, idx + 5), fi, d.edge_dim);
            idx += 6;
            break;
        case GNNB_CONV_SAGE:  // a = lin_l (bias), b = lin_r (no bias)
            L.a = pack_linear(pk, param(m, idx), param(m, idx + 1), fo, fi);
            L.b = pack_linear(pk, param(m, idx + 2), nullptr, fo, fi);
            idx += 3;
            break;
        case GNNB_CONV_PNA: {
            // a: X -> [A | B] = [X.W_nbr^T | X.W_self^T + b_pre]   (W_pre = [W_self | W_nbr])
            const float *Wpre = param(m, idx), *bpre = param(m, idx + 1);
            L.a.in = fi; L.a.out = 2 * fi; L.a.ldw = round_up(2 * fi, 4);
            L.a.wt_off = pk.reserve((size_t)fi * L.a.ldw);
            pk.add_transposed(Wpre, fi, 2 * fi, fi, fi, L.a.ldw, 0, L.a.wt_off);   // W_nbr
            pk.add_transposed(Wpre, fi, 2 * fi, 0, fi, L.a.ldw, fi, L.a.wt_off);   // W_self
            L.a.has_bias = true;
            L.a.bias_off = pk.add_vector(bpre, fi, fi);  // [0..0 | b_pre]
            // b: self block of post_nn (no bias), c: the 12F aggregate block (+ b_post)
            const float *Wpost = param(m, idx + 2), *bpost = param(m, idx + 3);
            L.b = pack_linear(pk, Wpost, nullptr, fo, fi, 13 * fi, 0);
            L.c = pack_linear(pk, Wpost, bpost, fo, 12 * fi, 13 * fi, fi);
            L.d = pack_linear(pk, param(m, idx + 4), param(m, idx + 5), fo, fo);
            idx += 6;
            break;
        }
        case GNNB_CONV_GAT: {
            // [att_src, att_dst, (att_edge,) bias, lin_weight (, lin_edge_weight)].  a: W with the
            // per-head logit vectors
            // w_src,h = W_h^T att_src,h and w_dst,h = W_h^T att_dst,h appended as 2H extra output
            // rows (folded in double, rounded once), so one GEMM gives h, a_src and a_dst.
            // b: the conv bias alone, added by the aggregation epilogue.
            const int H = d.gat_heads, C = fo / H;
            const bool edges = m->has_edge_features();
            const size_t ib = idx + (edges ? 3 : 2), iw = ib + 1;   // bias, lin_weight
            const float *att_src = param(m, idx), *att_dst = param(m, idx + 1);
            const float *W = param(m, iw);
            std::vector<float> Wg((size_t)(fo + 2 * H) * fi);
            std::copy(W, W + (size_t)fo * fi, Wg.begin());
            for (int h = 0; h < H; h++)
                for (int k = 0; k < fi; k++) {
                    double ss = 0.0, sd = 0.0;
                    for (int c = 0; c < C; c++) {
                        const double w = W[(size_t)(h * C + c) * fi + k];
                        ss += w * att_src[h * C + c];
                        sd += w * att_dst[h * C + c];
                    }
                    Wg[(size_t)(fo + h) * fi + k] = (float)ss;
                    Wg[(size_t)(fo + H + h) * fi + k] = (float)sd;
                }
            L.a = pack_linear(pk, Wg.data(), nullptr, fo + 2 * H, fi);
            L.b.out = fo;
            L.b.has_bias = true;
            L.b.bias_off = pk.add_vector(param(m, ib), fo);
            if (edges) {
                // w_edge,h[j] = sum_c W_e[h*C + c][j] att_edge[h*C + c], folded in double and
                // rounded once, as w_src / w_dst: lin_edge never runs as a GEMM
                const int ed = d.edge_dim;
                const float *att_edge = param(m, idx + 2), *We = param(m, iw + 1);
                for (int h = 0; h < H; h++)
                    for (int j = 0; j < ed; j++) {
                        double se = 0.0;
                        for (int c = 0; c < C; c++)
                            se += (double)We[(size_t)(h * C + c) * ed + j] * att_edge[h * C + c];
                        gat_w_edge[((size_t)k * H + h) * ed + j] = (float)se;
                    }
            }
            idx += edges ? 6 : 4;
            break;
        }
        case GNNB_CONV_GATV2: {
            // [att, bias, lin_l_weight, lin_l_bias, lin_r_weight, lin_r_bias (, lin_edge_weight)]:
            // a = lin_l, b = lin_r, c = att and d = the conv bias as vectors, e = W_e^T (no bias)
            L.a = pack_linear(pk, param(m, idx + 2), param(m, idx + 3), fo, fi);
            L.b = pack_linear(pk, param(m, idx + 4), param(m, idx + 5), fo, fi);
            L.c.out = fo;
            L.c.has_bias = true;
            L.c.bias_off = pk.add_vector(param(m, idx), fo);
            L.d.out = fo;
            L.d.has_bias = true;
            L.d.bias_off = pk.add_vector(param(m, idx + 1), fo);
            if (m->has_edge_features()) L.e = pack_linear(pk, param(m, idx + 6), nullptr, fo, d.edge_dim);
            idx += m->has_edge_features() ? 7 : 6;
            break;
        }
        case GNNB_CONV_TRANSFORMER: {
            // [key w, b, query w, b, value w, b (, lin_edge_weight), skip w, b]: a = lin_key,
            // b = lin_value, c = lin_query scaled by 1/sqrt(C) (in double, rounded once: exact when
            // C is a power of 4), d = lin_skip, e = W_e^T (no bias)
            const bool edges = m->has_edge_features();
            const double scale = 1.0 / std::sqrt((double)(fo / d.gat_heads));
            std::vector<float> Wq(param(m, idx + 2), param(m, idx + 2) + (size_t)fo * fi);
            std::vector<float> bq(param(m, idx + 3), param(m, idx + 3) + fo);
            for (float &w : Wq) w = (float)((double)w * scale);
            for (float &b : bq) b = (float)((double)b * scale);
            L.a = pack_linear(pk, param(m, idx), param(m, idx + 1), fo, fi);
            L.b = pack_linear(pk, param(m, idx + 4), param(m, idx + 5), fo, fi);
            L.c = pack_linear(pk, Wq.data(), bq.data(), fo, fi);
            const size_t is = idx + (edges ? 7 : 6);
            L.d = pack_linear(pk, param(m, is), param(m, is + 1), fo, fi);
            if (edges) L.e = pack_linear(pk, param(m, idx + 6), nullptr, fo, d.edge_dim);
            idx = is + 2;
            break;
        }
        }
        layer_p.push_back(L);
    }
    const size_t w_edge_off = gat_w_edge.empty() ? 0 : pk.add_vector(gat_w_edge.data(), (int)gat_w_edge.size());
    GNNB_TRY(m->weights.ensure(pk.data.size() * sizeof(float)));
    GNNB_CUDA(cudaMemcpyAsync(m->weights.ptr, pk.data.data(), pk.data.size() * sizeof(float),
                              cudaMemcpyHostToDevice, m->stream));
    GNNB_CUDA(cudaStreamSynchronize(m->stream));
    const float *base = m->weights.as<float>();
    m->gat_w_edge = gat_w_edge.empty() ? nullptr : base + w_edge_off;
    m->head.clear();
    for (const PendingLinear &p : head_p) m->head.push_back(resolve(p, base));
    m->layers.clear();
    for (const PendingLayer &L : layer_p) {
        LayerPack lp;
        lp.fi = L.fi; lp.fo = L.fo;
        lp.a = resolve(L.a, base); lp.b = resolve(L.b, base);
        lp.c = resolve(L.c, base); lp.d = resolve(L.d, base); lp.e = resolve(L.e, base);
        m->layers.push_back(lp);
    }
    {   // tensor-core weight images for the layerwise GEMMs (one allocation, built on the device)
        std::vector<PackedLinear *> all;
        for (PackedLinear &l : m->head) all.push_back(&l);
        for (LayerPack &lp : m->layers)
            for (PackedLinear *l : {&lp.a, &lp.b, &lp.c, &lp.d})
                if (l->Wt != nullptr && l->in > 0 && l->out > 0) all.push_back(l);
        size_t total = 0;
        for (PackedLinear *l : all) total += gemm_tc_image_floats(l->in, l->out);
        GNNB_TRY(m->weight_images.ensure(std::max<size_t>(total, 1) * sizeof(float)));
        size_t off = 0;
        for (PackedLinear *l : all) {
            float *img = m->weight_images.as<float>() + off;
            GNNB_TRY(gemm_tc_build_image(l->Wt, l->ldw, l->in, l->out, img, m->stream));
            l->img = img;
            off += gemm_tc_image_floats(l->in, l->out);
        }
        GNNB_CUDA(cudaStreamSynchronize(m->stream));
    }
    fused_release(m);
    fused_tc_release(m);
    // neither fused kernel takes GINE, GAT, GATv2 or TransformerConv (they leave m->fused /
    // m->fused_tc null): those run layerwise
    GNNB_TRY(fused_prepare(m));
    GNNB_TRY(fused_tc_prepare(m));
    m->finalized = true;
    return GNNB_OK;
}

extern "C" int gnnb_model_set_path(gnnb_model_t *m, int path)
{
    GNNB_REQUIRE(m != nullptr && path >= GNNB_PATH_AUTO && path <= GNNB_PATH_LAYERWISE, "bad path");
    m->path = path;
    return GNNB_OK;
}

extern "C" int gnnb_model_set_math(gnnb_model_t *m, int math)
{
    GNNB_REQUIRE(m != nullptr && (math == GNNB_MATH_FAST || math == GNNB_MATH_STRICT), "bad math mode");
    m->math = math;
    return GNNB_OK;
}

extern "C" int gnnb_model_last_launches(const gnnb_model_t *m) { return m ? m->last_launches : 0; }
extern "C" int gnnb_model_last_path(const gnnb_model_t *m) { return m ? m->last_path : 0; }
extern "C" int gnnb_model_last_kernel(const gnnb_model_t *m) { return m ? m->last_kernel : 0; }
extern "C" void *gnnb_model_stream(gnnb_model_t *m) { return m ? (void *)m->stream : nullptr; }
static int fused_any_status(gnnb_model_t *m, int *status);
static int edge_flag_check(gnnb_model_t *m);
extern "C" int gnnb_model_synchronize(gnnb_model_t *m)
{
    GNNB_REQUIRE(m != nullptr, "null model");
    DeviceScope on_device(m->device);
    GNNB_CUDA(cudaStreamSynchronize(m->stream));
    if (m->last_path == GNNB_PATH_LAYERWISE) GNNB_TRY(edge_flag_check(m));
    if (m->last_path == GNNB_PATH_FUSED) {
        // the async entry point cannot fall back by itself: report capacity/index problems here
        int status = 0;
        GNNB_TRY(fused_any_status(m, &status));
        if (status == 1) {
            set_error("fused kernel: a tile exceeded its node/edge capacity (raise nothing: set "
                      "accurate max_nodes/max_edges hints or use gnnb_model_run_batch, which "
                      "falls back to the layerwise path)");
            return GNNB_ERR_INVALID;
        }
        if (status == 2) {
            set_error("edge_list holds a node index outside its graph");
            return GNNB_ERR_INVALID;
        }
        if (status == 3) {
            set_error("fused kernel: non-finite activations (Inf/NaN) cannot be kept apart between "
                      "the graphs of a tile; use gnnb_model_run_batch, which re-runs such batches "
                      "on the layerwise path");
            return GNNB_ERR_INVALID;
        }
    }
    return GNNB_OK;
}

// ---------------------------------------------------------------------------- layerwise path
namespace gnnb {

static GemmArgs gemm_args(const float *A, int lda, const PackedLinear &L, float *C, int ldc, int M,
                          int act, const float *skip = nullptr, int ldskip = 0)
{
    GemmArgs g{};
    g.A1 = A; g.lda1 = lda; g.K1 = L.in; g.W1t = L.Wt; g.ldw1 = L.ldw; g.img1 = L.img;
    g.A2 = nullptr; g.lda2 = 0; g.K2 = 0; g.W2t = nullptr; g.ldw2 = 4;
    g.second_separate = 0;
    g.bias = L.bias; g.skip = skip; g.ldskip = ldskip; g.act = act;
    g.C = C; g.ldc = ldc; g.M = M; g.N = L.out;
    return g;
}

// x/coo/ef/node_ptr/edge_ptr/out are DEVICE pointers; node_ptr/edge_ptr address graph 0 of this
// chunk and hold absolute offsets (node_base/edge_base = their first values).  ef: the chunk's edge
// features [E][edge_dim] (models with edge features only).
static int run_layerwise(gnnb_model *m, const float *x, const int32_t *coo, const float *ef,
                         const int64_t *node_ptr,
                         const int64_t *edge_ptr, int64_t node_base, int64_t edge_base,
                         int n_graphs, int64_t T64, int64_t E64, float *out, cudaStream_t s,
                         int *launches)
{
    const gnnb_model_desc &d = m->d;
    GNNB_REQUIRE(T64 < (1ll << 31) && E64 < (1ll << 31), "batch chunk exceeds 2^31 nodes or edges");
    const int T = (int)T64, E = (int)E64;
    const bool strict = m->math == GNNB_MATH_STRICT;
    const int Tn = std::max(T, 1), En = std::max(E, 1);
    int maxf = std::max(std::max(d.in_dim, d.hidden_dim), d.out_dim);
    const int ldf = round_up(maxf, 4);

    GNNB_TRY(m->in_deg.ensure(sizeof(int32_t) * (size_t)Tn));
    GNNB_TRY(m->out_deg.ensure(sizeof(int32_t) * (size_t)Tn));
    GNNB_TRY(m->offsets.ensure(sizeof(int32_t) * (size_t)Tn));
    GNNB_TRY(m->nbr.ensure(sizeof(int32_t) * (size_t)En));
    int32_t *in_deg = m->in_deg.as<int32_t>(), *offsets = m->offsets.as<int32_t>();
    int32_t *nbr = m->nbr.as<int32_t>();
    const bool gine = d.conv_type == GNNB_CONV_GINE;
    const bool gat = d.conv_type == GNNB_CONV_GAT;
    const bool gat_edges = gat && m->has_edge_features();
    const bool gatv2 = d.conv_type == GNNB_CONV_GATV2;
    const bool gatv2_edges = gatv2 && m->has_edge_features();
    const bool transformer = d.conv_type == GNNB_CONV_TRANSFORMER;
    const bool transformer_edges = transformer && m->has_edge_features();
    const bool attn = gat || gatv2 || transformer;
    const int LH = gat_edges ? d.num_layers * d.gat_heads : 0;   // edge logit columns per slot / row
    // GINE has no heavy-row bucketing or hub hints, as PNA; the attention convs are bucketed but take
    // no hub hints
    const bool bucketed = d.conv_type != GNNB_CONV_PNA && !gine;
    const bool hub_hints = bucketed && !attn;
    const int lde = round_up(std::max(d.edge_dim, 1), 4);
    // GAT: the layer GEMM's output rows [h | a_src | a_dst], and the heavy-row partials, are
    // H*C + 2H floats wide
    const int ld_gat = attn ? round_up(std::max(d.hidden_dim, d.out_dim) + 2 * d.gat_heads, 4) : 0;
    // GATv2: the layer GEMMs' output rows [xl | xr], 2 H*C floats wide; TransformerConv: [k | v] and
    // [q | r] as wide
    const int ld_xlr = gatv2 || transformer ? round_up(2 * std::max(d.hidden_dim, d.out_dim), 4) : 0;
    if (d.num_layers > 0) {
        ProfScope ps(m->prof, PROF_TABLES, s);
        // the out-degree table (lib:1051-1083) is only read by the optional hub-row hints
        const bool want_out_deg = !strict && hub_l2_budget() > 0 && hub_hints && n_graphs > 0 &&
                                  T64 / n_graphs > 50000;
        int32_t *eidx = nullptr;
        if (m->has_edge_features()) {
            GNNB_TRY(m->edge_index.ensure(sizeof(int32_t) * (size_t)En));
            eidx = m->edge_index.as<int32_t>();
        }
        // with edge features the offsets are always passed: the slot -> source gather then checks
        // every endpoint
        GNNB_TRY(build_tables(coo, n_graphs > 1 || eidx ? node_ptr : nullptr, edge_ptr, node_base,
                              edge_base, n_graphs, T, E, in_deg,
                              want_out_deg ? m->out_deg.as<int32_t>() : nullptr, offsets, nbr, eidx,
                              m->tws, s, launches, m->edge_flag.as<int>()));
        // edge features in neighbor-slot order, once per run; every layer reads them in order
        if (gine || gatv2_edges || transformer_edges) {
            GNNB_TRY(m->ef_sorted.ensure(sizeof(float) * (size_t)En * lde));
            GNNB_TRY(launch_permute_edge_rows(ef, d.edge_dim, eidx, E, m->ef_sorted.as<float>(), lde, s,
                                              launches));
        }
        if (gatv2_edges) {   // each row's self-loop attribute: the mean of its other in-edge attributes
            GNNB_TRY(m->self_attr.ensure(sizeof(float) * (size_t)Tn * lde));
            GNNB_TRY(launch_gatv2_self_attr(m->ef_sorted.as<float>(), lde, d.edge_dim, offsets, nbr,
                                            in_deg, T, m->self_attr.as<float>(), s, launches));
        }
    }
    if (gat_edges && d.num_layers > 0) {   // every layer's edge logits, once per run
        ProfScope ps(m->prof, PROF_EDGE_LOGITS, s);
        GNNB_TRY(m->elog.ensure(sizeof(float) * (size_t)En * LH));
        GNNB_TRY(m->self_elog.ensure(sizeof(float) * (size_t)Tn * LH));
        GatEdgeLogitsArgs la{};
        la.ef = ef; la.edge_dim = d.edge_dim; la.w_edge = m->gat_w_edge; la.LH = LH;
        la.offsets = offsets; la.nbr = nbr; la.in_deg = in_deg; la.edge_index = m->edge_index.as<int32_t>();
        la.n = T; la.elog = m->elog.as<float>(); la.self_elog = m->self_elog.as<float>();
        GNNB_TRY(launch_gat_edge_logits(la, (int)(((int64_t)E + Tn - 1) / Tn), s, launches));
    }
    const float *dinv = nullptr;
    if (d.conv_type == GNNB_CONV_GCN && !strict && d.num_layers > 0) {
        GNNB_TRY(m->dinv.ensure(sizeof(float) * (size_t)Tn));
        GNNB_TRY(compute_dinv(in_deg, m->dinv.as<float>(), T, s, launches));
        dinv = m->dinv.as<float>();
    }
    // degree bucketing only matters for big graphs (molecular graphs have in-degree <= ~8)
    int hub_bit = 0;
    m->heavy.n_heavy = m->heavy.n_chunks = 0;
    const int heavy_thr = heavy_threshold();
    m->last_hub_rows = 0;
    if (!strict && d.num_layers > 0 && bucketed && n_graphs > 0 && T64 / n_graphs > 50000) {
        GNNB_TRY(find_heavy_rows(in_deg, T, heavy_thr, m->tws, m->heavy, s, launches));
        GNNB_TRY(heavy_setup(m->tws, m->heavy.n_chunks, attn ? ld_gat : maxf));
        // a feature matrix larger than L2: keep the rows of the most-referenced sources resident
        // (the out-degree table, lib:1051-1083, is what ranks them)
        const size_t row_bytes = sizeof(float) * (size_t)std::max(d.in_dim, d.hidden_dim);
        if (hub_hints && hub_l2_budget() > 0 && E > 0 && (size_t)T * row_bytes > (96u << 20)) {
            ProfScope ps(m->prof, PROF_TABLES, s);
            GNNB_TRY(m->nbr_hub.ensure(sizeof(int32_t) * (size_t)En));
            GNNB_TRY(mark_hub_sources(nbr, m->nbr_hub.as<int32_t>(), E, m->out_deg.as<int32_t>(), T,
                                      row_bytes, hub_l2_budget(), m->tws, &m->last_hub_rows, s,
                                      launches));
            if (m->last_hub_rows > 0) {
                nbr = m->nbr_hub.as<int32_t>();
                hub_bit = 1;
            }
        }
    }

    GNNB_TRY(m->feat[0].ensure(sizeof(float) * (size_t)Tn * ldf));
    GNNB_TRY(m->feat[1].ensure(sizeof(float) * (size_t)Tn * ldf));
    // the attention convs aggregate into dst; TransformerConv keeps [q | r] in agg
    if (!attn) GNNB_TRY(m->agg.ensure(sizeof(float) * (size_t)Tn * ldf));
    if (transformer) GNNB_TRY(m->agg.ensure(sizeof(float) * (size_t)Tn * ld_xlr));
    if (d.conv_type == GNNB_CONV_GIN || d.conv_type == GNNB_CONV_PNA || gine)
        GNNB_TRY(m->hid.ensure(sizeof(float) * (size_t)Tn * ldf));
    if (gat) GNNB_TRY(m->hid.ensure(sizeof(float) * (size_t)Tn * ld_gat));
    if (gatv2 || transformer) GNNB_TRY(m->hid.ensure(sizeof(float) * (size_t)Tn * ld_xlr));
    if (d.conv_type == GNNB_CONV_PNA)
        GNNB_TRY(m->wide.ensure(sizeof(float) * (size_t)Tn * 14 * (size_t)ldf));

    const float *cur = x;
    int cur_ld = d.in_dim;
    for (int k = 0; k < d.num_layers; k++) {
        const LayerPack &L = m->layers[k];
        const int fi = L.fi, fo = L.fo;
        const bool do_skip = d.skip && k != 0 && k != d.num_layers - 1;  // cpp:269-279
        float *dst = m->feat[k & 1].as<float>();
        const int ld_out = round_up(fo, 4);
        const float *skip = do_skip ? cur : nullptr;
        AggArgs a{};
        a.x = cur; a.ldx = cur_ld; a.F = fi; a.out = m->agg.as<float>(); a.ldo = round_up(fi, 4);
        a.offsets = offsets; a.nbr = nbr; a.in_deg = in_deg; a.dinv = dinv; a.n = T;
        a.eps = d.gin_eps;
        a.heavy.threshold = heavy_thr;
        a.heavy.set(m->heavy, m->tws.heavy_partial.as<float>());
        a.hub_bit = hub_bit;
        switch (d.conv_type) {
        case GNNB_CONV_GCN: {
            a.mode = AGG_GCN;
            { ProfScope ps(m->prof, PROF_AGG, s); GNNB_TRY(launch_agg(a, strict, s, launches)); }
            GemmArgs g = gemm_args(a.out, a.ldo, L.a, dst, ld_out, T, d.gnn_act, skip, cur_ld);
            { ProfScope ps(m->prof, PROF_GEMM, s); GNNB_TRY(launch_gemm(g, strict, s, launches)); }
            break;
        }
        case GNNB_CONV_GIN: {
            a.mode = AGG_GIN;
            { ProfScope ps(m->prof, PROF_AGG, s); GNNB_TRY(launch_agg(a, strict, s, launches)); }
            float *hid = m->hid.as<float>();
            GemmArgs g0 = gemm_args(a.out, a.ldo, L.a, hid, ld_out, T, GNNB_ACT_RELU);  // lib:1537-1541
            { ProfScope ps(m->prof, PROF_GEMM, s); GNNB_TRY(launch_gemm(g0, strict, s, launches)); }
            GemmArgs g1 = gemm_args(hid, ld_out, L.b, dst, ld_out, T, d.gnn_act, skip, cur_ld);
            { ProfScope ps(m->prof, PROF_GEMM, s); GNNB_TRY(launch_gemm(g1, strict, s, launches)); }
            break;
        }
        case GNNB_CONV_GINE: {
            GineProjAggArgs ga{};
            ga.x = cur; ga.ldx = cur_ld; ga.F = fi; ga.ef_sorted = m->ef_sorted.as<float>();
            ga.lde = lde; ga.edge_dim = d.edge_dim; ga.We_t = L.e.Wt; ga.ldw = L.e.ldw; ga.be = L.e.bias;
            ga.out = a.out; ga.ldo = a.ldo; ga.offsets = offsets; ga.nbr = nbr; ga.in_deg = in_deg;
            ga.n = T; ga.eps = d.gin_eps;
            { ProfScope ps(m->prof, PROF_AGG, s); GNNB_TRY(launch_gine_agg_proj(ga, s, launches)); }
            float *hid = m->hid.as<float>();
            GemmArgs g0 = gemm_args(a.out, a.ldo, L.a, hid, ld_out, T, GNNB_ACT_RELU);  // lib:1537-1541
            { ProfScope ps(m->prof, PROF_GEMM, s); GNNB_TRY(launch_gemm(g0, strict, s, launches)); }
            GemmArgs g1 = gemm_args(hid, ld_out, L.b, dst, ld_out, T, d.gnn_act, skip, cur_ld);
            { ProfScope ps(m->prof, PROF_GEMM, s); GNNB_TRY(launch_gemm(g1, strict, s, launches)); }
            break;
        }
        case GNNB_CONV_SAGE: {
            a.mode = AGG_MEAN;
            { ProfScope ps(m->prof, PROF_AGG, s); GNNB_TRY(launch_agg(a, strict, s, launches)); }
            GemmArgs g = gemm_args(a.out, a.ldo, L.a, dst, ld_out, T, d.gnn_act, skip, cur_ld);
            g.A2 = cur; g.lda2 = cur_ld; g.K2 = fi; g.W2t = L.b.Wt; g.ldw2 = L.b.ldw; g.img2 = L.b.img;
            g.second_separate = 1;  // lib:2316-2332
            { ProfScope ps(m->prof, PROF_GEMM, s); GNNB_TRY(launch_gemm(g, strict, s, launches)); }
            break;
        }
        case GNNB_CONV_PNA: {
            float *ab = m->wide.as<float>();                 // [T][2fi]
            float *cat12 = ab + (size_t)Tn * 2 * ldf;         // [T][12fi]
            GemmArgs g0 = gemm_args(cur, cur_ld, L.a, ab, 2 * fi, T, GNNB_ACT_IDENTITY);
            { ProfScope ps(m->prof, PROF_GEMM, s); GNNB_TRY(launch_gemm(g0, false, s, launches)); }
            float *hid = m->hid.as<float>();
            GemmArgs g1 = gemm_args(cur, cur_ld, L.b, hid, ld_out, T, GNNB_ACT_IDENTITY);
            g1.bias = L.c.bias;
            g1.A2 = cat12; g1.K2 = 12 * fi; g1.W2t = L.c.Wt; g1.ldw2 = L.c.ldw; g1.img2 = L.c.img;
            // tensor-core path: only the [T][4F] statistics are materialised; the GEMM expands them
            // to [stats | amp stats | att stats] while it feeds the MMAs (3x less HBM traffic)
            g1.lda2 = 4 * fi; g1.expand_deg = in_deg; g1.expand_delta = d.pna_delta;
            const bool expand = gemm_tc_supported(g1);
            if (!expand) { g1.lda2 = 12 * fi; g1.expand_deg = nullptr; }
            PnaAggArgs pa{};
            pa.ab = ab; pa.F = fi; pa.cat12 = cat12; pa.offsets = offsets; pa.nbr = nbr;
            pa.in_deg = in_deg; pa.n = T; pa.delta = d.pna_delta; pa.compact = expand ? 1 : 0;
            { ProfScope ps(m->prof, PROF_AGG, s); GNNB_TRY(launch_pna_agg(pa, s, launches)); }
            { ProfScope ps(m->prof, PROF_GEMM, s); GNNB_TRY(launch_gemm(g1, false, s, launches)); }   // lib:2149
            GemmArgs g2 = gemm_args(hid, ld_out, L.d, dst, ld_out, T, d.gnn_act, skip, cur_ld);
            { ProfScope ps(m->prof, PROF_GEMM, s); GNNB_TRY(launch_gemm(g2, false, s, launches)); }   // lib:2150
            break;
        }
        case GNNB_CONV_GAT:
        case GNNB_CONV_GATV2:
        case GNNB_CONV_TRANSFORMER: {
            // the attention aggregation's epilogue applies bias, skip and activation and writes the
            // layer; heavy-row partials [acc H*C | max H | sum H]
            const int H = d.gat_heads;
            AttnAggArgs at{};
            at.H = H; at.C = fo / H; at.slope = d.gat_negative_slope;
            at.skip = skip; at.ldskip = cur_ld; at.act = d.gnn_act; at.out = dst; at.ldo = ld_out;
            at.offsets = offsets; at.nbr = nbr; at.in_deg = in_deg; at.n = T;
            at.heavy.threshold = heavy_thr;
            at.heavy.set(m->heavy, m->tws.heavy_partial.as<float>());
            at.ldp = round_up(fo + 2 * H, 4);
            float *hid = m->hid.as<float>();
            at.g = hid;
            if (transformer) {
                // four GEMMs: [k | v] = x.[W_k | W_v]^T + [b_k | b_v] into hid, and [q | r] into agg:
                // q = x.W_q^T + b_q (1/sqrt(C) folded in), r = x.W_skip^T (+ the model's skip) without
                // b_skip.  The epilogue adds b_skip as its bias and r as its skip.
                const int ld2 = round_up(2 * fo, 4);
                float *qr = m->agg.as<float>();
                TransformerAggArgs ta{at};
                ta.g = hid; ta.ldg = ld2; ta.q = qr; ta.ldq = ld2;
                ta.bias = L.d.bias; ta.skip = qr + fo; ta.ldskip = ld2;
                GemmArgs gk = gemm_args(cur, cur_ld, L.a, hid, ld2, T, GNNB_ACT_IDENTITY);
                GemmArgs gv = gemm_args(cur, cur_ld, L.b, hid + fo, ld2, T, GNNB_ACT_IDENTITY);
                GemmArgs gq = gemm_args(cur, cur_ld, L.c, qr, ld2, T, GNNB_ACT_IDENTITY);
                GemmArgs gs = gemm_args(cur, cur_ld, L.d, qr + fo, ld2, T, GNNB_ACT_IDENTITY, skip, cur_ld);
                gs.bias = nullptr;
                for (const GemmArgs *g : {&gk, &gv, &gq, &gs}) {
                    ProfScope ps(m->prof, PROF_GEMM, s);
                    GNNB_TRY(launch_gemm(*g, strict, s, launches));
                }
                if (transformer_edges) {
                    ta.ef_sorted = m->ef_sorted.as<float>();
                    ta.lde = lde; ta.edge_dim = d.edge_dim; ta.We_t = L.e.Wt; ta.ldw = L.e.ldw;
                }
                { ProfScope ps(m->prof, PROF_AGG, s); GNNB_TRY(launch_transformer_agg(ta, s, launches)); }
                break;
            }
            if (gat) {
                // one GEMM: [h | a_src | a_dst] = x.[W | w_src | w_dst]^T, no bias
                GatAggArgs ga{at};
                ga.bias = L.b.bias; ga.ldg = at.ldp;
                GemmArgs g = gemm_args(cur, cur_ld, L.a, hid, ga.ldg, T, GNNB_ACT_IDENTITY);
                { ProfScope ps(m->prof, PROF_GEMM, s); GNNB_TRY(launch_gemm(g, strict, s, launches)); }
                if (gat_edges) {
                    ga.elog = m->elog.as<float>() + (size_t)k * H;
                    ga.self_elog = m->self_elog.as<float>() + (size_t)k * H;
                    ga.ldl = LH;
                }
                { ProfScope ps(m->prof, PROF_AGG, s); GNNB_TRY(launch_gat_agg(ga, s, launches)); }
                break;
            }
            // two GEMMs, xl = x.W_l^T + b_l and xr = x.W_r^T + b_r, side by side in one buffer (one
            // GEMM of N = 2 H*C would not fit the tensor-core GEMM at H*C = 128)
            Gatv2AggArgs ga{at};
            ga.bias = L.d.bias; ga.ldg = round_up(2 * fo, 4); ga.att = L.c.bias;
            GemmArgs gl = gemm_args(cur, cur_ld, L.a, hid, ga.ldg, T, GNNB_ACT_IDENTITY);
            GemmArgs gr = gemm_args(cur, cur_ld, L.b, hid + fo, ga.ldg, T, GNNB_ACT_IDENTITY);
            { ProfScope ps(m->prof, PROF_GEMM, s); GNNB_TRY(launch_gemm(gl, strict, s, launches)); }
            { ProfScope ps(m->prof, PROF_GEMM, s); GNNB_TRY(launch_gemm(gr, strict, s, launches)); }
            if (gatv2_edges) {
                ga.ef_sorted = m->ef_sorted.as<float>(); ga.self_attr = m->self_attr.as<float>();
                ga.lde = lde; ga.edge_dim = d.edge_dim; ga.We_t = L.e.Wt; ga.ldw = L.e.ldw;
            }
            { ProfScope ps(m->prof, PROF_AGG, s); GNNB_TRY(launch_gatv2_agg(ga, s, launches)); }
            break;
        }
        }
        cur = dst;
        cur_ld = ld_out;
    }
    m->last_emb = cur;
    m->last_emb_ld = cur_ld;
    m->last_emb_rows = T;

    // pooling + head
    const int emb = m->emb_dim();
    const int head_in = emb * d.num_pools;
    const int Gn = std::max(n_graphs, 1);
    int maxh = std::max(std::max(head_in, d.mlp_hidden), d.mlp_out);
    const int ldh = round_up(maxh, 4);
    GNNB_TRY(m->hbuf[0].ensure(sizeof(float) * (size_t)Gn * ldh));
    GNNB_TRY(m->hbuf[1].ensure(sizeof(float) * (size_t)Gn * ldh));
    float *h_in = m->hbuf[0].as<float>();
    int h_ld = round_up(head_in, 4);
    {
        ProfScope ps(m->prof, PROF_POOL, s);
        GNNB_TRY(launch_pool(cur, cur_ld, emb, node_ptr, node_base, n_graphs, T64, d.pools,
                             d.num_pools, h_in, m->pool_tmp, s, launches, strict));
    }
    // launch_pool writes rows of stride num_pools*emb; keep that as the leading dimension
    h_ld = head_in;
    for (int j = 0; j < d.mlp_num_linear; j++) {
        const bool last = j == d.mlp_num_linear - 1;
        float *dstp = last ? out : m->hbuf[(j + 1) & 1].as<float>();
        const int ld_out = last ? d.mlp_out : round_up(m->head[j].out, 4);
        const int act = last ? d.out_act : d.mlp_act;  // cpp:508-516, 644-650
        GemmArgs g = gemm_args(h_in, h_ld, m->head[j], dstp, ld_out, n_graphs, act);
        { ProfScope ps(m->prof, PROF_GEMM, s); GNNB_TRY(launch_gemm(g, strict, s, launches)); }
        h_in = dstp;
        h_ld = ld_out;
    }
    return GNNB_OK;
}

}  // namespace gnnb

// ---------------------------------------------------------------------------- run entry points
// layerwise path: the table kernels flag edge endpoints outside their graph (like status 2 of the
// fused kernels); cleared before a run, read once the stream has been synchronised
static int edge_flag_reset(gnnb_model_t *m, cudaStream_t s)
{
    GNNB_TRY(m->edge_flag.ensure(sizeof(int)));
    GNNB_CUDA(cudaMemsetAsync(m->edge_flag.ptr, 0, sizeof(int), s));
    return GNNB_OK;
}
static int edge_flag_check(gnnb_model_t *m)
{
    int bad = 0;
    if (m->edge_flag.ptr == nullptr) return GNNB_OK;
    GNNB_CUDA(cudaMemcpy(&bad, m->edge_flag.ptr, sizeof(int), cudaMemcpyDeviceToHost));
    if (bad) {
        set_error("edge_list holds a node index outside its graph");
        return GNNB_ERR_INVALID;
    }
    return GNNB_OK;
}

static int check_ready(gnnb_model_t *m)
{
    GNNB_REQUIRE(m != nullptr, "null model");
    if (!m->finalized) {
        set_error("gnnb_model_finalize() has not been called");
        return GNNB_ERR_STATE;
    }
    return GNNB_OK;
}

// kernel ids: 1 layerwise, 2 fused fp32-FMA (fused.cu), 3 fused tcgen05 (fused_tc.cu)
static int choose_path(gnnb_model_t *m, int max_n, int max_e, int *path, int *kernel)
{
    const bool fast = m->math == GNNB_MATH_FAST;
    const bool can_tc = fast && fused_tc_supports(m, max_n, max_e);
    const bool can_fma = fast && fused_supports(m, max_n, max_e);
    if (m->path == GNNB_PATH_FUSED) {
        if (m->d.conv_type == GNNB_CONV_GAT) {
            set_error("fused path requested but the fused kernels have no GAT attention; GAT models "
                      "run on the layerwise path");
            return GNNB_ERR_INVALID;
        }
        if (m->d.conv_type == GNNB_CONV_GATV2) {
            set_error("fused path requested but the fused kernels have no GATv2 attention; GATv2 "
                      "models run on the layerwise path");
            return GNNB_ERR_INVALID;
        }
        if (m->d.conv_type == GNNB_CONV_TRANSFORMER) {
            set_error("fused path requested but the fused kernels have no TransformerConv attention; "
                      "TransformerConv models run on the layerwise path");
            return GNNB_ERR_INVALID;
        }
        if (!can_tc && !can_fma) {
            set_error("fused path requested but unsupported for this model/batch (graph larger than "
                      "a CTA tile, strict math, or unsupported dims)");
            return GNNB_ERR_INVALID;
        }
        *path = GNNB_PATH_FUSED;
        *kernel = can_tc ? 3 : 2;
    } else if (m->path == GNNB_PATH_LAYERWISE) {
        *path = GNNB_PATH_LAYERWISE;
        *kernel = 1;
    } else {
        // AUTO: the tensor-core fused kernel when it applies, else the layerwise path (measured
        // faster than the fp32-FMA fused kernel, profiles/)
        *path = can_tc ? GNNB_PATH_FUSED : GNNB_PATH_LAYERWISE;
        *kernel = can_tc ? 3 : 1;
    }
    return GNNB_OK;
}

static int run_fused(gnnb_model_t *m, int kernel, const float *x, const int32_t *coo,
                     const int64_t *np, const int64_t *ep, int n_graphs, int64_t total_nodes,
                     int max_nodes, float *out, cudaStream_t s)
{
    ProfScope ps(m->prof, PROF_FUSED, s);
    if (kernel == 3)
        return fused_tc_run(m, x, coo, np, ep, n_graphs, total_nodes, max_nodes, out, s,
                            &m->last_launches);
    return fused_run(m, x, coo, np, ep, n_graphs, total_nodes, max_nodes, out, s,
                     &m->last_launches);
}

static int fused_any_status(gnnb_model_t *m, int *status)
{
    return m->last_kernel == 3 ? fused_tc_status(m, status) : fused_status(m, status);
}

// a handle with edge features (GINE, or GAT, GATv2 or TransformerConv with edge_dim) takes them
// through the *_edges entry points, every other handle runs through the plain ones
static int check_edges_entry(gnnb_model_t *m, bool edges_entry)
{
    GNNB_TRY(check_ready(m));
    const bool edges = m->has_edge_features();
    if (edges && !edges_entry) {
        set_error(std::string(m->d.conv_type == GNNB_CONV_GAT           ? "a GAT model with edge_dim"
                              : m->d.conv_type == GNNB_CONV_GATV2       ? "a GATv2 model with edge_dim"
                              : m->d.conv_type == GNNB_CONV_TRANSFORMER ? "a TransformerConv model with edge_dim"
                                                                        : "a GINE model") +
                  " needs its edge features: run it with gnnb_model_run_batch_edges or "
                  "gnnb_model_run_batch_edges_async");
        return GNNB_ERR_INVALID;
    }
    if (!edges && edges_entry) {
        set_error("the *_edges entry points run GINE models and GAT, GATv2 and TransformerConv models "
                  "with edge_dim only; this model has no edge features");
        return GNNB_ERR_INVALID;
    }
    return GNNB_OK;
}

static int run_batch_async(gnnb_model_t *m, const float *x, const int32_t *edge_list,
                           const float *edge_attr, const int64_t *node_ptr, const int64_t *edge_ptr,
                           int n_graphs, int64_t total_nodes, int64_t total_edges, float *out,
                           void *stream)
{
    DeviceScope on_device(m->device);
    GNNB_REQUIRE(n_graphs >= 0 && total_nodes >= 0 && total_edges >= 0, "negative size");
    GNNB_REQUIRE(node_ptr != nullptr && edge_ptr != nullptr && out != nullptr, "null argument");
    if (n_graphs == 0) return GNNB_OK;
    GNNB_REQUIRE(is_device_pointer(x) || total_nodes == 0, "run_batch_async needs device pointers");
    if (m->has_edge_features())
        GNNB_REQUIRE(total_edges == 0 || is_device_pointer(edge_attr),
                     "edge_attr must be a device pointer (null with edges present)");
    cudaStream_t s = stream ? (cudaStream_t)stream : m->stream;
    m->last_launches = 0;
    int path, kernel;
    // without host copies of the offsets the capacity hints decide whether tiles fit
    const int hint_n = m->d.max_nodes > 0 ? m->d.max_nodes : (1 << 30);
    const int hint_e = m->d.max_edges > 0 ? m->d.max_edges : (1 << 30);
    GNNB_TRY(choose_path(m, hint_n, hint_e, &path, &kernel));
    m->last_path = path;
    m->last_kernel = kernel;
    if (path == GNNB_PATH_FUSED)
        return run_fused(m, kernel, x, edge_list, node_ptr, edge_ptr, n_graphs, total_nodes, hint_n,
                         out, s);
    GNNB_TRY(edge_flag_reset(m, s));
    return run_layerwise(m, x, edge_list, edge_attr, node_ptr, edge_ptr, 0, 0, n_graphs, total_nodes,
                         total_edges, out, s, &m->last_launches);
}

extern "C" int gnnb_model_run_batch_async(gnnb_model_t *m, const float *x, const int32_t *edge_list,
                                          const int64_t *node_ptr, const int64_t *edge_ptr,
                                          int n_graphs, int64_t total_nodes, int64_t total_edges,
                                          float *out, void *stream)
{
    GNNB_TRY(check_edges_entry(m, false));
    return run_batch_async(m, x, edge_list, nullptr, node_ptr, edge_ptr, n_graphs, total_nodes,
                           total_edges, out, stream);
}

extern "C" int gnnb_model_run_batch_edges_async(gnnb_model_t *m, const float *x,
                                                const int32_t *edge_list, const float *edge_attr,
                                                const int64_t *node_ptr, const int64_t *edge_ptr,
                                                int n_graphs, int64_t total_nodes,
                                                int64_t total_edges, float *out, void *stream)
{
    GNNB_TRY(check_edges_entry(m, true));
    return run_batch_async(m, x, edge_list, edge_attr, node_ptr, edge_ptr, n_graphs, total_nodes,
                           total_edges, out, stream);
}

static int run_batch(gnnb_model_t *m, const float *x, const int32_t *edge_list,
                     const float *edge_attr, const int64_t *node_ptr, const int64_t *edge_ptr,
                     int n_graphs, float *out)
{
    DeviceScope on_device(m->device);
    GNNB_REQUIRE(n_graphs >= 0, "negative n_graphs");
    if (n_graphs == 0) return GNNB_OK;
    GNNB_REQUIRE(node_ptr && edge_ptr && out, "null argument");
    const gnnb_model_desc &d = m->d;
    cudaStream_t s = m->stream;
    const bool dev = is_device_pointer(node_ptr);
    // the offsets on the host (validation, path choice, chunking): host arrays are used in place
    std::vector<int64_t> hn_copy, he_copy;
    const int64_t *hn = node_ptr, *he = edge_ptr;
    if (dev) {
        hn_copy.resize((size_t)n_graphs + 1);
        he_copy.resize((size_t)n_graphs + 1);
        GNNB_CUDA(cudaMemcpy(hn_copy.data(), node_ptr, hn_copy.size() * 8, cudaMemcpyDeviceToHost));
        GNNB_CUDA(cudaMemcpy(he_copy.data(), edge_ptr, he_copy.size() * 8, cudaMemcpyDeviceToHost));
        hn = hn_copy.data();
        he = he_copy.data();
    }
    GNNB_REQUIRE(hn[0] == 0 && he[0] == 0, "node_ptr[0] and edge_ptr[0] must be 0");
    const int64_t T = hn[n_graphs], E = he[n_graphs];
    GNNB_REQUIRE(T >= 0 && E >= 0 && T < (1ll << 40) && E < (1ll << 40), "bad node_ptr/edge_ptr totals");
    GNNB_REQUIRE(T == 0 || x != nullptr, "x is null");
    GNNB_REQUIRE(E == 0 || edge_list != nullptr, "edge_list is null");
    const bool edges = m->has_edge_features();
    if (edges) {
        GNNB_REQUIRE(E == 0 || edge_attr != nullptr, "edge_attr is null");
        GNNB_REQUIRE(E == 0 || is_device_pointer(edge_attr) == dev,
                     "edge_attr must live in the same memory space as node_ptr");
    }
    // validation of graphs [a, b): offsets non-decreasing, capacities respected; updates the maxima
    int64_t max_n = 0, max_e = 0;
    auto scan = [&](int a, int b) -> int {
        for (int g = a; g < b; g++) {
            const int64_t n = hn[g + 1] - hn[g], e = he[g + 1] - he[g];
            GNNB_REQUIRE(n >= 0 && e >= 0, "node_ptr/edge_ptr must be non-decreasing");
            max_n = std::max(max_n, n);
            max_e = std::max(max_e, e);
        }
        if (d.max_nodes > 0) GNNB_REQUIRE(max_n <= d.max_nodes, "graph exceeds max_nodes");
        if (d.max_edges > 0) GNNB_REQUIRE(max_e <= d.max_edges, "graph exceeds max_edges");
        GNNB_REQUIRE(max_n < (1ll << 31) && max_e < (1ll << 31), "graph too large");
        return GNNB_OK;
    };

    // ---- host buffers + tensor-core fused kernel: chunked ingest pipeline.  The batch is cut into
    // chunks of graphs; chunk k+1 is validated and copied in (h2d stream) while chunk k computes
    // (compute stream) and chunk k-1's outputs are copied out (d2h stream), through double-buffered
    // chunk staging.  End to end the step then costs max(PCIe, kernel) instead of their sum, and the
    // host-side scan of the offsets hides behind the GPU as well.  The choice is optimistic (it
    // assumes every graph fits a tile); a chunk that does not, a capacity overflow or non-finite
    // activations send the whole batch to the regular path below.
    bool scanned_all = false;
    if (!dev) {
        int path0, kernel0;
        GNNB_TRY(choose_path(m, 1, 1, &path0, &kernel0));
        if (path0 == GNNB_PATH_FUSED && kernel0 == 3 && getenv("GNNB_NO_INGEST_PIPELINE") == nullptr) {
            // chunk boundaries: a short ramp (4k, 8k, 16k, 32k graphs) so that the first copy-in is
            // brief, then large chunks (fewer launches, smaller per-launch tails)
            int chunk_graphs = 65536;
            if (const char *e = getenv("GNNB_INGEST_CHUNK_GRAPHS")) chunk_graphs = std::max(1024, atoi(e));
            std::vector<int> cb{0};
            for (int sz = 4096; cb.back() < n_graphs;) {
                cb.push_back(std::min(n_graphs, cb.back() + std::min(sz, chunk_graphs)));
                if (sz < chunk_graphs) sz *= 2;
            }
            const int n_chunks = (int)cb.size() - 1;
            int64_t max_cn = 1, max_ce = 1;
            bool sane = true;
            for (int k = 0; k < n_chunks; k++) {
                const int a = cb[k], b = cb[k + 1];
                const int64_t cn = hn[b] - hn[a], ce = he[b] - he[a];
                sane = sane && cn >= 0 && ce >= 0 && cn <= T && ce <= E;
                max_cn = std::max(max_cn, cn);
                max_ce = std::max(max_ce, ce);
            }
            GNNB_REQUIRE(sane, "node_ptr/edge_ptr must be non-decreasing");
            for (int i = 0; i < 2; i++) {
                GNNB_TRY(m->ch_x[i].ensure(sizeof(float) * (size_t)max_cn * d.in_dim));
                GNNB_TRY(m->ch_coo[i].ensure(sizeof(int32_t) * 2 * (size_t)max_ce));
                GNNB_TRY(m->ch_nptr[i].ensure(8 * ((size_t)chunk_graphs + 1)));
                GNNB_TRY(m->ch_eptr[i].ensure(8 * ((size_t)chunk_graphs + 1)));
            }
            GNNB_TRY(m->st_out.ensure(sizeof(float) * (size_t)n_graphs * d.mlp_out));
            float *dout_all = m->st_out.as<float>();
            m->last_launches = 0;
            m->last_path = GNNB_PATH_FUSED;
            m->last_kernel = 3;
            int rc = GNNB_OK;
            bool too_big = false;
            {
                ProfScope ps(m->prof, PROF_FUSED, s);
                for (int k = 0; k < n_chunks && rc == GNNB_OK; k++) {
                    const int a = cb[k], b = cb[k + 1], bi = k & 1;
                    rc = scan(a, b);
                    if (rc != GNNB_OK) break;
                    if (!fused_tc_supports(m, (int)max_n, (int)max_e)) { too_big = true; break; }
                    const int64_t cn = hn[b] - hn[a], ce = he[b] - he[a];
                    auto issue = [&]() -> int {
                        if (k >= 2) GNNB_CUDA(cudaStreamWaitEvent(m->h2d_stream, m->ev_done[bi], 0));
                        if (cn > 0)
                            GNNB_CUDA(cudaMemcpyAsync(m->ch_x[bi].ptr, x + (size_t)hn[a] * d.in_dim,
                                                      sizeof(float) * (size_t)cn * d.in_dim,
                                                      cudaMemcpyHostToDevice, m->h2d_stream));
                        if (ce > 0)
                            GNNB_CUDA(cudaMemcpyAsync(m->ch_coo[bi].ptr, edge_list + 2 * (size_t)he[a],
                                                      sizeof(int32_t) * 2 * (size_t)ce, cudaMemcpyHostToDevice,
                                                      m->h2d_stream));
                        GNNB_CUDA(cudaMemcpyAsync(m->ch_nptr[bi].ptr, node_ptr + a, 8 * (size_t)(b - a + 1),
                                                  cudaMemcpyHostToDevice, m->h2d_stream));
                        GNNB_CUDA(cudaMemcpyAsync(m->ch_eptr[bi].ptr, edge_ptr + a, 8 * (size_t)(b - a + 1),
                                                  cudaMemcpyHostToDevice, m->h2d_stream));
                        GNNB_CUDA(cudaEventRecord(m->ev_h2d[bi], m->h2d_stream));
                        GNNB_CUDA(cudaStreamWaitEvent(s, m->ev_h2d[bi], 0));
                        // the offsets stay absolute (relative to the whole batch): rebase the data pointers
                        const float *xb = m->ch_x[bi].as<float>() - (size_t)hn[a] * d.in_dim;
                        const int32_t *cb = m->ch_coo[bi].as<int32_t>() - 2 * (size_t)he[a];
                        GNNB_TRY(fused_tc_run(m, xb, cb, m->ch_nptr[bi].as<int64_t>(),
                                              m->ch_eptr[bi].as<int64_t>(), b - a, cn, (int)max_n,
                                              dout_all + (size_t)a * d.mlp_out, s, &m->last_launches, k == 0));
                        GNNB_CUDA(cudaEventRecord(m->ev_done[bi], s));
                        GNNB_CUDA(cudaStreamWaitEvent(m->d2h_stream, m->ev_done[bi], 0));
                        GNNB_CUDA(cudaMemcpyAsync(out + (size_t)a * d.mlp_out, dout_all + (size_t)a * d.mlp_out,
                                                  sizeof(float) * (size_t)(b - a) * d.mlp_out,
                                                  cudaMemcpyDeviceToHost, m->d2h_stream));
                        return GNNB_OK;
                    };
                    rc = issue();
                }
            }
            // drain whatever was issued before looking at the outcome
            cudaStreamSynchronize(m->h2d_stream);
            cudaStreamSynchronize(s);
            cudaStreamSynchronize(m->d2h_stream);
            if (rc != GNNB_OK) return rc;
            int status = 0;
            if (!too_big) {
                scanned_all = true;
                GNNB_TRY(fused_any_status(m, &status));
                if (status == 2) {
                    set_error("edge_list holds a node index outside its graph");
                    return GNNB_ERR_INVALID;
                }
                if (status == 0) return GNNB_OK;
            }
            if (m->path == GNNB_PATH_FUSED) {
                set_error(too_big ? "fused path requested but a graph is larger than a CTA tile"
                          : status == 1 ? "fused path requested but a tile exceeded its capacity"
                                        : "fused path requested but the batch produced non-finite "
                                          "activations (graphs of a tile would contaminate each other)");
                return GNNB_ERR_INVALID;
            }
            if (!too_big) {
                // capacity overflow or non-finite activations: redo the batch on the layerwise path
                m->path = GNNB_PATH_LAYERWISE;
                const int rc2 = run_batch(m, x, edge_list, edge_attr, node_ptr, edge_ptr, n_graphs, out);
                m->path = GNNB_PATH_AUTO;
                return rc2;
            }
            // a graph larger than a tile: the regular path below chooses the kernel from the full scan
        }
    }
    if (!scanned_all) {
        max_n = 0;
        max_e = 0;
        GNNB_TRY(scan(0, n_graphs));
    }

    const float *dx = x, *def = edge_attr;
    const int32_t *dcoo = edge_list;
    const int64_t *dnp = node_ptr, *dep = edge_ptr;
    float *dout = out;
    if (!dev) {
        GNNB_TRY(m->st_x.ensure(sizeof(float) * (size_t)std::max<int64_t>(T, 1) * d.in_dim));
        GNNB_TRY(m->st_coo.ensure(sizeof(int32_t) * 2 * (size_t)std::max<int64_t>(E, 1)));
        GNNB_TRY(m->st_nptr.ensure(8 * ((size_t)n_graphs + 1)));
        GNNB_TRY(m->st_eptr.ensure(8 * ((size_t)n_graphs + 1)));
        GNNB_TRY(m->st_out.ensure(sizeof(float) * (size_t)n_graphs * d.mlp_out));
        if (T > 0)
            GNNB_CUDA(cudaMemcpyAsync(m->st_x.ptr, x, sizeof(float) * (size_t)T * d.in_dim,
                                      cudaMemcpyHostToDevice, s));
        if (E > 0)
            GNNB_CUDA(cudaMemcpyAsync(m->st_coo.ptr, edge_list, sizeof(int32_t) * 2 * (size_t)E,
                                      cudaMemcpyHostToDevice, s));
        if (edges) {
            GNNB_TRY(m->st_ef.ensure(sizeof(float) * (size_t)std::max<int64_t>(E, 1) * d.edge_dim));
            if (E > 0)
                GNNB_CUDA(cudaMemcpyAsync(m->st_ef.ptr, edge_attr, sizeof(float) * (size_t)E * d.edge_dim,
                                          cudaMemcpyHostToDevice, s));
            def = m->st_ef.as<float>();
        }
        GNNB_CUDA(cudaMemcpyAsync(m->st_nptr.ptr, node_ptr, 8 * ((size_t)n_graphs + 1), cudaMemcpyHostToDevice, s));
        GNNB_CUDA(cudaMemcpyAsync(m->st_eptr.ptr, edge_ptr, 8 * ((size_t)n_graphs + 1), cudaMemcpyHostToDevice, s));
        dx = m->st_x.as<float>();
        dcoo = m->st_coo.as<int32_t>();
        dnp = m->st_nptr.as<int64_t>();
        dep = m->st_eptr.as<int64_t>();
        dout = m->st_out.as<float>();
    }
    m->last_launches = 0;
    int path, kernel;
    GNNB_TRY(choose_path(m, (int)max_n, (int)max_e, &path, &kernel));
    m->last_path = path;
    m->last_kernel = kernel;
    bool ran_layerwise = false;
    auto layerwise_chunks = [&]() -> int {
        // chunk the union so that the per-layer activations stay within a fixed budget
        const int64_t kChunkNodes = 4ll << 20;
        int g0 = 0;
        ran_layerwise = true;
        GNNB_TRY(edge_flag_reset(m, s));
        while (g0 < n_graphs) {
            int g1 = g0 + 1;
            while (g1 < n_graphs && hn[g1 + 1] - hn[g0] <= kChunkNodes) g1++;
            GNNB_TRY(run_layerwise(m, dx + (size_t)hn[g0] * d.in_dim, dcoo + 2 * (size_t)he[g0],
                                   edges ? def + (size_t)he[g0] * d.edge_dim : nullptr, dnp + g0, dep + g0, hn[g0], he[g0], g1 - g0, hn[g1] - hn[g0],
                                   he[g1] - he[g0], dout + (size_t)g0 * d.mlp_out, s,
                                   &m->last_launches));
            g0 = g1;
        }
        return GNNB_OK;
    };
    if (path == GNNB_PATH_FUSED) {
        GNNB_TRY(run_fused(m, kernel, dx, dcoo, dnp, dep, n_graphs, T, (int)max_n, dout, s));
        GNNB_CUDA(cudaStreamSynchronize(s));
        int status = 0;
        GNNB_TRY(fused_any_status(m, &status));
        if (status == 2) {
            set_error("edge_list holds a node index outside its graph");
            return GNNB_ERR_INVALID;
        }
        if (status == 1 || status == 3) {  // a tile overflowed its capacity, or non-finite
                                            // activations appeared: redo the batch layerwise
            if (m->path == GNNB_PATH_FUSED) {
                set_error(status == 1 ? "fused path requested but a tile exceeded its capacity"
                                      : "fused path requested but the batch produced non-finite "
                                        "activations (graphs of a tile would contaminate each other)");
                return GNNB_ERR_INVALID;
            }
            m->last_path = GNNB_PATH_LAYERWISE;
            m->last_kernel = 1;
            GNNB_TRY(layerwise_chunks());
        }
    } else {
        GNNB_TRY(layerwise_chunks());
    }
    if (!dev)
        GNNB_CUDA(cudaMemcpyAsync(out, dout, sizeof(float) * (size_t)n_graphs * d.mlp_out,
                                  cudaMemcpyDeviceToHost, s));
    GNNB_CUDA(cudaStreamSynchronize(s));
    if (ran_layerwise) GNNB_TRY(edge_flag_check(m));
    return GNNB_OK;
}

extern "C" int gnnb_model_run_batch(gnnb_model_t *m, const float *x, const int32_t *edge_list,
                                    const int64_t *node_ptr, const int64_t *edge_ptr, int n_graphs,
                                    float *out)
{
    GNNB_TRY(check_edges_entry(m, false));
    return run_batch(m, x, edge_list, nullptr, node_ptr, edge_ptr, n_graphs, out);
}

extern "C" int gnnb_model_run_batch_edges(gnnb_model_t *m, const float *x, const int32_t *edge_list,
                                          const float *edge_attr, const int64_t *node_ptr,
                                          const int64_t *edge_ptr, int n_graphs, float *out)
{
    GNNB_TRY(check_edges_entry(m, true));
    return run_batch(m, x, edge_list, edge_attr, node_ptr, edge_ptr, n_graphs, out);
}

extern "C" int gnnb_model_run_graph(gnnb_model_t *m, const float *node_features,
                                    const int32_t *edge_list, int num_nodes, int num_edges,
                                    float *out)
{
    GNNB_REQUIRE(num_nodes >= 0 && num_edges >= 0, "negative size");
    GNNB_REQUIRE(!is_device_pointer(out) && !is_device_pointer(node_features),
                 "gnnb_model_run_graph takes host buffers (like <name>_top); use run_batch for "
                 "device buffers");
    const int64_t np[2] = {0, num_nodes}, ep[2] = {0, num_edges};
    return gnnb_model_run_batch(m, node_features, edge_list, np, ep, 1, out);
}

extern "C" int gnnb_model_get_node_embeddings(gnnb_model_t *m, float *dst, int64_t total_nodes)
{
    GNNB_TRY(check_ready(m));
    DeviceScope on_device(m->device);
    GNNB_REQUIRE(dst != nullptr, "null destination");
    if (m->last_path != GNNB_PATH_LAYERWISE || m->last_emb == nullptr ||
        total_nodes != m->last_emb_rows) {
        set_error("node embeddings are available after a single-chunk LAYERWISE run only");
        return GNNB_ERR_STATE;
    }
    const int emb = m->emb_dim();
    GNNB_CUDA(cudaMemcpy2DAsync(dst, sizeof(float) * emb, m->last_emb, sizeof(float) * m->last_emb_ld,
                                sizeof(float) * emb, (size_t)total_nodes, cudaMemcpyDefault,
                                m->stream));
    GNNB_CUDA(cudaStreamSynchronize(m->stream));
    return GNNB_OK;
}

// ---------------------------------------------------------------------------- profiling
extern "C" int gnnb_model_set_profile(gnnb_model_t *m, int on)
{
    GNNB_REQUIRE(m != nullptr, "null model");
    m->prof.on = on != 0;
    return GNNB_OK;
}

// Sum of CUDA-event durations (ms) and launch-group counts per kernel class since the last
// call: [0] tables, [1] aggregation, [2] GEMM, [3] pooling, [4] fused, [5] GAT edge logits.
// Synchronises the stream.
extern "C" int gnnb_model_profile_read(gnnb_model_t *m, float *ms, int *counts)
{
    GNNB_REQUIRE(m != nullptr && ms != nullptr && counts != nullptr, "null argument");
    DeviceScope on_device(m->device);
    GNNB_CUDA(cudaStreamSynchronize(m->stream));
    GNNB_CUDA(cudaDeviceSynchronize());
    for (int i = 0; i < PROF_NCAT; i++) { ms[i] = 0.0f; counts[i] = 0; }
    for (Profiler::Rec &r : m->prof.recs) {
        float t = 0.0f;
        if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) {
            ms[r.cat] += t;
            counts[r.cat] += 1;
        } else {
            cudaGetLastError();
        }
        m->prof.free_events.push_back(r.a);
        m->prof.free_events.push_back(r.b);
    }
    m->prof.recs.clear();
    return GNNB_OK;
}
