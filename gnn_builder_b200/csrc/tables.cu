// Degree / neighbor tables: gnn_builder_lib.h:1051-1166 on the GPU.
//
// Reference semantics: in/out degree histograms of the COO list; offsets = exclusive scan of the
// in-degree (n entries, no sentinel); neighbor_table = sources grouped by destination, STABLE in
// COO order (the serial cursor walk of lib:1113-1123).  Here: one pass of integer atomics for the
// histograms, an exclusive scan, and a stable LSD radix sort of (destination -> source) pairs --
// a stable sort by destination is exactly the cursor walk's output, so the tables are bit-exact
// for any graph size.  (The fused molecular kernel builds its tables in shared memory instead,
// see fused.cu.)  The scan and the radix sort are cub:: device primitives from the CUDA toolkit.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "kernels.h"

namespace gnnb {

namespace {

__device__ __forceinline__ int find_segment(const int64_t *__restrict__ ptr, int n_seg, int64_t i)
{
    // largest g with ptr[g] <= i   (ptr has n_seg + 1 entries, ptr[0] = 0)
    int lo = 0, hi = n_seg;
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (__ldg(ptr + mid) <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// keys = destination (union ids), vals = source (union ids) or the edge index
template <bool COUNT, bool VAL_IS_EDGE_INDEX>
__global__ void edge_prepare_kernel(const int32_t *__restrict__ edge_list,
                                    const int64_t *__restrict__ node_ptr,
                                    const int64_t *__restrict__ edge_ptr, int64_t node_base,
                                    int64_t edge_base, int n_graphs, int n, int e,
                                    uint32_t *__restrict__ keys, int32_t *__restrict__ vals,
                                    int32_t *__restrict__ in_deg, int32_t *__restrict__ out_deg,
                                    int *__restrict__ bad)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < e; i += gridDim.x * blockDim.x) {
        const int2 sd = __ldg(reinterpret_cast<const int2 *>(edge_list) + i);
        int src = sd.x, dst = sd.y;
        int limit = n;   // node ids are local to their graph: valid range [0, graph size)
        int base = 0;
        if (node_ptr != nullptr) {
            const int g = find_segment(edge_ptr, n_graphs, (int64_t)i + edge_base);
            const int64_t b0 = __ldg(node_ptr + g);
            base = (int)(b0 - node_base);
            limit = (int)(__ldg(node_ptr + g + 1) - b0);
        }
        if ((unsigned)src >= (unsigned)limit || (unsigned)dst >= (unsigned)limit) {
            // an endpoint outside its graph (the reference would index out of bounds, lib:1060-1062):
            // flag it, keep the tables memory-safe (the edge is dropped from the degree counts and
            // parked on node 0 in the sort input) -- the caller turns the flag into GNNB_ERR_INVALID
            if (bad != nullptr) atomicExch(bad, 1);
            if (keys) { keys[i] = 0u; vals[i] = 0; }
            continue;
        }
        src += base;
        dst += base;
        if (keys) {
            keys[i] = (uint32_t)dst;
            vals[i] = VAL_IS_EDGE_INDEX ? i : src;
        }
        if (COUNT) {
            if (in_deg != nullptr) atomicAdd(in_deg + dst, 1);
            if (out_deg != nullptr) atomicAdd(out_deg + src, 1);
        }
    }
}

// In-degrees from the destination keys AFTER the stable sort: a run of equal keys is one row's
// in-edges, so its length is the in-degree -- no atomics (31 M atomicAdds, 100 000 of them on one
// hub's counter, cost 0.3 ms on the 2M-node graph; this pass reads the sorted keys once).
// first / last must be zeroed: rows without in-edges keep last - first = 0.
__global__ void run_bounds_kernel(const uint32_t *__restrict__ keys_sorted, int e,
                                  int32_t *__restrict__ first, int32_t *__restrict__ last)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < e; i += gridDim.x * blockDim.x) {
        const uint32_t k = keys_sorted[i];
        if (i == 0 || keys_sorted[i - 1] != k) first[k] = i;
        if (i == e - 1 || keys_sorted[i + 1] != k) last[k] = i + 1;
    }
}
__global__ void run_length_kernel(int32_t *__restrict__ last_to_deg, const int32_t *__restrict__ first, int n)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        last_to_deg[i] -= first[i];
}

__global__ void gather_sources_kernel(const int32_t *__restrict__ edge_list,
                                      const int32_t *__restrict__ edge_index, int e,
                                      int32_t *__restrict__ nbr)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < e; i += gridDim.x * blockDim.x)
        nbr[i] = __ldg(edge_list + 2 * (size_t)__ldg(edge_index + i));
}

// the same for a batch of graphs: local source ids are translated to union ids.  A slot whose edge
// has an endpoint outside its graph (flagged by edge_prepare_kernel, parked on edge 0) reads
// source 0, so the tables stay memory-safe until the caller reports the error.
__global__ void gather_sources_batch_kernel(const int32_t *__restrict__ edge_list,
                                            const int32_t *__restrict__ edge_index,
                                            const int64_t *__restrict__ node_ptr,
                                            const int64_t *__restrict__ edge_ptr, int64_t node_base,
                                            int64_t edge_base, int n_graphs, int e,
                                            int32_t *__restrict__ nbr)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < e; i += gridDim.x * blockDim.x) {
        const int eid = __ldg(edge_index + i);
        const int g = find_segment(edge_ptr, n_graphs, (int64_t)eid + edge_base);
        const int64_t b0 = __ldg(node_ptr + g);
        const int limit = (int)(__ldg(node_ptr + g + 1) - b0);
        const int src = __ldg(edge_list + 2 * (size_t)eid);
        nbr[i] = (unsigned)src < (unsigned)limit ? src + (int)(b0 - node_base) : 0;
    }
}

// row-partitioned graph: this rank owns destination rows [row_begin, row_begin + n_local); sources
// keep their global ids
__global__ void edge_prepare_partition_kernel(const int32_t *__restrict__ edge_list, int e,
                                              int row_begin, int n_local,
                                              uint32_t *__restrict__ keys, int32_t *__restrict__ vals,
                                              int32_t *__restrict__ in_deg, int *__restrict__ bad)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < e; i += gridDim.x * blockDim.x) {
        const int2 sd = __ldg(reinterpret_cast<const int2 *>(edge_list) + i);
        const int dst = sd.y - row_begin;
        if ((unsigned)dst >= (unsigned)n_local) {
            atomicExch(bad, 1);
            keys[i] = 0;
            vals[i] = 0;
            continue;
        }
        keys[i] = (uint32_t)dst;
        vals[i] = sd.x;
        atomicAdd(in_deg + dst, 1);
    }
}

// counters: [0] heavy rows, [1] their chunks (pass 1); [2], [3] the same as running cursors (pass 2)
__global__ void heavy_count_kernel(const int32_t *__restrict__ len, int n, int threshold,
                                   int32_t *__restrict__ counters)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int l = __ldg(len + i);
        if (l > threshold) {
            atomicAdd(counters, 1);
            atomicAdd(counters + 1, (l + kHeavyChunk - 1) / kHeavyChunk);
        }
    }
}
__global__ void heavy_fill_kernel(const int32_t *__restrict__ len, int n, int threshold,
                                  int32_t *__restrict__ counters, int32_t *__restrict__ rows,
                                  int32_t *__restrict__ chunk_base, int32_t *__restrict__ chunk_row)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int l = __ldg(len + i);
        if (l > threshold) {
            const int nch = (l + kHeavyChunk - 1) / kHeavyChunk;
            const int pos = atomicAdd(counters + 2, 1);
            const int cb = atomicAdd(counters + 3, nch);
            rows[pos] = i;
            chunk_base[pos] = cb;
            for (int j = 0; j < nch; j++) chunk_row[cb + j] = pos;
        }
    }
}

__global__ void dinv_kernel(const int32_t *__restrict__ in_deg, float *__restrict__ dinv, int n)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        dinv[i] = 1.0f / sqrtf(1.0f + (float)__ldg(in_deg + i));
}

// ---- hub sources (large graphs): the sources referenced most often are marked in a copy of the
// neighbor table (bit 31) so that the aggregation keeps their feature rows in L2 (agg.cu)
__global__ void ref_count_kernel(const int32_t *__restrict__ nbr, int e, int32_t *__restrict__ cnt)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < e; i += gridDim.x * blockDim.x)
        atomicAdd(cnt + (__ldg(nbr + i) & 0x7fffffff), 1);
}
constexpr int kHubBins = 4096;
__global__ void __launch_bounds__(256) count_hist_kernel(const int32_t *__restrict__ cnt, int n,
                                                         unsigned int *__restrict__ hist)
{
    __shared__ unsigned int h[kHubBins];
    for (int i = threadIdx.x; i < kHubBins; i += blockDim.x) h[i] = 0u;
    __syncthreads();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int c = __ldg(cnt + i);
        atomicAdd(&h[c < kHubBins - 1 ? c : kHubBins - 1], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kHubBins; i += blockDim.x)
        if (h[i]) atomicAdd(hist + i, h[i]);
}
__global__ void mark_hubs_kernel(const int32_t *nbr_in, int32_t *nbr_out,   // (may alias)
                                 int e, const int32_t *__restrict__ cnt, int threshold)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < e; i += gridDim.x * blockDim.x) {
        const int u = nbr_in[i] & 0x7fffffff;
        nbr_out[i] = __ldg(cnt + u) >= threshold ? (u | (int32_t)0x80000000) : u;
    }
}

inline int grid_for(int64_t work, int block)
{
    int64_t g = ceil_div64(work, block);
    const int64_t cap = (int64_t)kNumSMs * 16;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

int bits_for(int n)
{
    int b = 1;
    while (b < 32 && (1ll << b) < (int64_t)n) ++b;
    return b;
}

int scan_offsets(const int32_t *in_deg, int32_t *offsets, int n, TableWorkspace &ws, cudaStream_t s,
                 int *launches)
{
    size_t tmp = 0;
    GNNB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp, in_deg, offsets, n, s));
    GNNB_TRY(ws.cub_tmp.ensure(tmp));
    GNNB_CUDA(cub::DeviceScan::ExclusiveSum(ws.cub_tmp.ptr, tmp, in_deg, offsets, n, s));
    if (launches) *launches += 2;
    return GNNB_OK;
}

int sort_pairs(TableWorkspace &ws, int e, int n, int32_t *vals_out, cudaStream_t s, int *launches)
{
    size_t tmp = 0;
    const int end_bit = bits_for(n);
    GNNB_TRY(ws.keys_out.ensure(sizeof(uint32_t) * (size_t)e));
    GNNB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp, ws.keys_in.as<uint32_t>(),
                                              ws.keys_out.as<uint32_t>(), ws.vals_in.as<int32_t>(),
                                              vals_out, e, 0, end_bit, s));
    GNNB_TRY(ws.cub_tmp.ensure(tmp));
    GNNB_CUDA(cub::DeviceRadixSort::SortPairs(ws.cub_tmp.ptr, tmp, ws.keys_in.as<uint32_t>(),
                                              ws.keys_out.as<uint32_t>(), ws.vals_in.as<int32_t>(),
                                              vals_out, e, 0, end_bit, s));
    if (launches) *launches += 1 + 2 * ((end_bit + 7) / 8);
    return GNNB_OK;
}

}  // namespace

int build_degree_tables(const int32_t *edge_list, int n, int e, int32_t *in_deg, int32_t *out_deg,
                        cudaStream_t s, int *launches, int *bad)
{
    if (n > 0) {
        GNNB_CUDA(cudaMemsetAsync(in_deg, 0, sizeof(int32_t) * (size_t)n, s));
        GNNB_CUDA(cudaMemsetAsync(out_deg, 0, sizeof(int32_t) * (size_t)n, s));
    }
    if (e > 0) {
        edge_prepare_kernel<true, false><<<grid_for(e, 256), 256, 0, s>>>(
            edge_list, nullptr, nullptr, 0, 0, 0, n, e, nullptr, nullptr, in_deg, out_deg, bad);
        GNNB_CUDA(cudaGetLastError());
        if (launches) ++*launches;
    }
    return GNNB_OK;
}

int build_neighbor_tables(const int32_t *edge_list, const int32_t *in_deg, int n, int e,
                          int32_t *offsets, int32_t *nbr, int32_t *edge_index, TableWorkspace &ws,
                          cudaStream_t s, int *launches, int *bad)
{
    if (n <= 0) return GNNB_OK;
    GNNB_TRY(scan_offsets(in_deg, offsets, n, ws, s, launches));
    if (e <= 0) return GNNB_OK;
    GNNB_TRY(ws.keys_in.ensure(sizeof(uint32_t) * (size_t)e));
    GNNB_TRY(ws.vals_in.ensure(sizeof(int32_t) * (size_t)e));
    if (edge_index) {
        edge_prepare_kernel<false, true><<<grid_for(e, 256), 256, 0, s>>>(
            edge_list, nullptr, nullptr, 0, 0, 0, n, e, ws.keys_in.as<uint32_t>(), ws.vals_in.as<int32_t>(),
            nullptr, nullptr, bad);
        GNNB_CUDA(cudaGetLastError());
        GNNB_TRY(sort_pairs(ws, e, n, edge_index, s, launches));
        gather_sources_kernel<<<grid_for(e, 256), 256, 0, s>>>(edge_list, edge_index, e, nbr);
        GNNB_CUDA(cudaGetLastError());
        if (launches) *launches += 2;
    } else {
        edge_prepare_kernel<false, false><<<grid_for(e, 256), 256, 0, s>>>(
            edge_list, nullptr, nullptr, 0, 0, 0, n, e, ws.keys_in.as<uint32_t>(), ws.vals_in.as<int32_t>(),
            nullptr, nullptr, bad);
        GNNB_CUDA(cudaGetLastError());
        GNNB_TRY(sort_pairs(ws, e, n, nbr, s, launches));
        if (launches) ++*launches;
    }
    return GNNB_OK;
}

// neighbor table from the sorted edge-index table (sources as union ids for a batch of graphs)
static int gather_sources(const int32_t *edge_list, const int32_t *edge_index, const int64_t *node_ptr,
                          const int64_t *edge_ptr, int64_t node_base, int64_t edge_base, int n_graphs,
                          int e, int32_t *nbr, cudaStream_t s, int *launches)
{
    if (node_ptr != nullptr)
        gather_sources_batch_kernel<<<grid_for(e, 256), 256, 0, s>>>(
            edge_list, edge_index, node_ptr, edge_ptr, node_base, edge_base, n_graphs, e, nbr);
    else
        gather_sources_kernel<<<grid_for(e, 256), 256, 0, s>>>(edge_list, edge_index, e, nbr);
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    return GNNB_OK;
}

int build_tables(const int32_t *edge_list, const int64_t *node_ptr, const int64_t *edge_ptr,
                 int64_t node_base, int64_t edge_base, int n_graphs, int n, int e, int32_t *in_deg, int32_t *out_deg, int32_t *offsets,
                 int32_t *nbr, int32_t *edge_index, TableWorkspace &ws, cudaStream_t s,
                 int *launches, int *bad)
{
    if (n <= 0) return GNNB_OK;
    // large edge lists: in-degrees as run lengths of the sorted destination keys (no atomics);
    // out_deg == nullptr: the caller does not need the out-degree table (nothing in the model path
    // reads it unless the hub-row hints are on -- the reference never reads it at all)
    const bool sorted_degrees = e >= (1 << 20);
    GNNB_CUDA(cudaMemsetAsync(in_deg, 0, sizeof(int32_t) * (size_t)n, s));
    if (out_deg != nullptr) GNNB_CUDA(cudaMemsetAsync(out_deg, 0, sizeof(int32_t) * (size_t)n, s));
    if (e > 0) {
        GNNB_TRY(ws.keys_in.ensure(sizeof(uint32_t) * (size_t)e));
        GNNB_TRY(ws.vals_in.ensure(sizeof(int32_t) * (size_t)e));
        if (edge_index) {
            edge_prepare_kernel<true, true><<<grid_for(e, 256), 256, 0, s>>>(
                edge_list, node_ptr, edge_ptr, node_base, edge_base, n_graphs, n, e,
                ws.keys_in.as<uint32_t>(), ws.vals_in.as<int32_t>(),
                sorted_degrees ? nullptr : in_deg, out_deg, bad);
        } else {
            edge_prepare_kernel<true, false><<<grid_for(e, 256), 256, 0, s>>>(
                edge_list, node_ptr, edge_ptr, node_base, edge_base, n_graphs, n, e,
                ws.keys_in.as<uint32_t>(),
                ws.vals_in.as<int32_t>(), sorted_degrees ? nullptr : in_deg, out_deg, bad);
        }
        GNNB_CUDA(cudaGetLastError());
        if (launches) ++*launches;
    }
    if (sorted_degrees) {
        GNNB_TRY(sort_pairs(ws, e, n, edge_index ? edge_index : nbr, s, launches));
        GNNB_CUDA(cudaMemsetAsync(offsets, 0, sizeof(int32_t) * (size_t)n, s));   // run starts (scratch)
        run_bounds_kernel<<<grid_for(e, 256), 256, 0, s>>>(ws.keys_out.as<uint32_t>(), e, offsets, in_deg);
        run_length_kernel<<<grid_for(n, 256), 256, 0, s>>>(in_deg, offsets, n);
        GNNB_CUDA(cudaGetLastError());
        if (launches) *launches += 2;
        GNNB_TRY(scan_offsets(in_deg, offsets, n, ws, s, launches));
        if (edge_index) GNNB_TRY(gather_sources(edge_list, edge_index, node_ptr, edge_ptr, node_base,
                                                edge_base, n_graphs, e, nbr, s, launches));
        return GNNB_OK;
    }
    GNNB_TRY(scan_offsets(in_deg, offsets, n, ws, s, launches));
    if (e > 0) {
        if (edge_index) {
            GNNB_TRY(sort_pairs(ws, e, n, edge_index, s, launches));
            GNNB_TRY(gather_sources(edge_list, edge_index, node_ptr, edge_ptr, node_base, edge_base,
                                    n_graphs, e, nbr, s, launches));
        } else {
            GNNB_TRY(sort_pairs(ws, e, n, nbr, s, launches));
        }
    }
    return GNNB_OK;
}

int build_partition_tables(const int32_t *edge_list, int row_begin, int n_local, int e,
                           int32_t *in_deg_local, int32_t *offsets_local, int32_t *nbr_global,
                           TableWorkspace &ws, cudaStream_t s, int *launches)
{
    if (n_local <= 0) return GNNB_OK;
    GNNB_CUDA(cudaMemsetAsync(in_deg_local, 0, sizeof(int32_t) * (size_t)n_local, s));
    int bad_host = 0;
    if (e > 0) {
        GNNB_TRY(ws.keys_in.ensure(sizeof(uint32_t) * (size_t)e));
        GNNB_TRY(ws.vals_in.ensure(sizeof(int32_t) * (size_t)e));
        GNNB_TRY(ws.counters.ensure(sizeof(int32_t) * 4));
        GNNB_CUDA(cudaMemsetAsync(ws.counters.ptr, 0, sizeof(int32_t) * 4, s));
        edge_prepare_partition_kernel<<<grid_for(e, 256), 256, 0, s>>>(
            edge_list, e, row_begin, n_local, ws.keys_in.as<uint32_t>(), ws.vals_in.as<int32_t>(),
            in_deg_local, ws.counters.as<int32_t>());
        GNNB_CUDA(cudaGetLastError());
        if (launches) ++*launches;
    }
    GNNB_TRY(scan_offsets(in_deg_local, offsets_local, n_local, ws, s, launches));
    if (e > 0) {
        GNNB_TRY(sort_pairs(ws, e, n_local, nbr_global, s, launches));
        GNNB_CUDA(cudaMemcpyAsync(&bad_host, ws.counters.ptr, sizeof(int), cudaMemcpyDeviceToHost, s));
        GNNB_CUDA(cudaStreamSynchronize(s));
        GNNB_REQUIRE(bad_host == 0, "partition tables: an edge's destination is outside the owned rows");
    }
    return GNNB_OK;
}

int find_heavy_rows(const int32_t *lengths, int n, int threshold, TableWorkspace &ws, HeavyList &hl,
                    cudaStream_t s, int *launches)
{
    hl.n_heavy = hl.n_chunks = 0;
    if (n <= 0) return GNNB_OK;
    GNNB_TRY(ws.counters.ensure(sizeof(int32_t) * 4));
    GNNB_CUDA(cudaMemsetAsync(ws.counters.ptr, 0, sizeof(int32_t) * 4, s));
    heavy_count_kernel<<<grid_for(n, 256), 256, 0, s>>>(lengths, n, threshold, ws.counters.as<int32_t>());
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    int32_t host[2] = {0, 0};
    GNNB_CUDA(cudaMemcpyAsync(host, ws.counters.ptr, sizeof(host), cudaMemcpyDeviceToHost, s));
    GNNB_CUDA(cudaStreamSynchronize(s));
    if (host[0] <= 0) return GNNB_OK;
    GNNB_TRY(hl.rows.ensure(sizeof(int32_t) * (size_t)host[0]));
    GNNB_TRY(hl.chunk_base.ensure(sizeof(int32_t) * (size_t)host[0]));
    GNNB_TRY(hl.chunk_row.ensure(sizeof(int32_t) * (size_t)host[1]));
    heavy_fill_kernel<<<grid_for(n, 256), 256, 0, s>>>(lengths, n, threshold, ws.counters.as<int32_t>(),
                                                      hl.rows.as<int32_t>(), hl.chunk_base.as<int32_t>(),
                                                      hl.chunk_row.as<int32_t>());
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    hl.n_heavy = host[0];
    hl.n_chunks = host[1];
    return GNNB_OK;
}

// Marks the most-referenced sources of a neighbor table: nbr_out[i] = nbr_in[i] | bit 31 when the
// source is one of the top rows by reference count whose feature rows (row_bytes each) fit
// `budget_bytes` together.  ref_cnt: per-source reference counts (the out-degree table of
// lib:1051-1083, which the reference computes and never reads), or null to count them here.
// One host synchronisation (the 16 KB histogram).  nbr_out may alias nbr_in.
int mark_hub_sources(const int32_t *nbr_in, int32_t *nbr_out, int e, const int32_t *ref_cnt,
                     int n_src, size_t row_bytes, size_t budget_bytes, TableWorkspace &ws,
                     int *n_hubs_host, cudaStream_t s, int *launches)
{
    if (n_hubs_host) *n_hubs_host = 0;
    if (e <= 0 || n_src <= 0) return GNNB_OK;
    GNNB_TRY(ws.counters.ensure(sizeof(int32_t) * 4));
    GNNB_TRY(ws.hub_hist.ensure(sizeof(unsigned int) * kHubBins));
    GNNB_CUDA(cudaMemsetAsync(ws.hub_hist.ptr, 0, sizeof(unsigned int) * kHubBins, s));
    if (ref_cnt == nullptr) {
        GNNB_TRY(ws.hub_cnt.ensure(sizeof(int32_t) * (size_t)n_src));
        GNNB_CUDA(cudaMemsetAsync(ws.hub_cnt.ptr, 0, sizeof(int32_t) * (size_t)n_src, s));
        ref_count_kernel<<<grid_for(e, 256), 256, 0, s>>>(nbr_in, e, ws.hub_cnt.as<int32_t>());
        GNNB_CUDA(cudaGetLastError());
        if (launches) ++*launches;
        ref_cnt = ws.hub_cnt.as<int32_t>();
    }
    count_hist_kernel<<<grid_for(n_src, 256), 256, 0, s>>>(ref_cnt, n_src, ws.hub_hist.as<unsigned int>());
    GNNB_CUDA(cudaGetLastError());
    static thread_local unsigned int hist[kHubBins];
    GNNB_CUDA(cudaMemcpyAsync(hist, ws.hub_hist.ptr, sizeof(hist), cudaMemcpyDeviceToHost, s));
    GNNB_CUDA(cudaStreamSynchronize(s));
    const size_t max_rows = budget_bytes / (row_bytes ? row_bytes : 1);
    size_t rows = 0;
    int threshold = kHubBins;   // nothing marked
    for (int b = kHubBins - 1; b >= 2; b--) {   // a source referenced once gains nothing
        if (rows + hist[b] > max_rows) break;
        rows += hist[b];
        threshold = b;
    }
    if (n_hubs_host) *n_hubs_host = (int)rows;
    mark_hubs_kernel<<<grid_for(e, 256), 256, 0, s>>>(nbr_in, nbr_out, e, ref_cnt, threshold);
    GNNB_CUDA(cudaGetLastError());
    if (launches) *launches += 2;
    return GNNB_OK;
}

int heavy_setup(TableWorkspace &ws, int n_chunks, int F)
{
    if (n_chunks > 0) GNNB_TRY(ws.heavy_partial.ensure(sizeof(float) * (size_t)n_chunks * (size_t)F));
    return GNNB_OK;
}

int compute_dinv(const int32_t *in_deg, float *dinv, int n, cudaStream_t s, int *launches)
{
    if (n <= 0) return GNNB_OK;
    dinv_kernel<<<grid_for(n, 256), 256, 0, s>>>(in_deg, dinv, n);
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    return GNNB_OK;
}

}  // namespace gnnb
