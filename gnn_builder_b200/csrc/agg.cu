// CSR (by destination) neighbor aggregation -- the gather/reduce half of every conv of
// gnn_builder_lib.h:  gcn_conv_agg (lib:1213-1289), gin_conv_agg (1389-1437), sage_conv_agg
// (2161-2209), pna_conv_agg (1750-1834), lg/simple (2350-2549).
//
// Kernel (2) of the design: a (sub-)warp per destination row, lanes across the feature dimension
// with float4 (16 B) gathers of each neighbor row, so one neighbor row of F=128 floats is one
// fully coalesced 512 B warp request; neighbor loop unrolled x4 so four independent gathers are
// in flight per lane.  Rows are bucketed by in-degree: rows above `heavy.threshold` are skipped
// here and handled by the chunked heavy-row kernels below (a warp per 128-neighbor chunk, chunk
// sums added in a fixed order: deterministic).
//
// HBM roofline: algorithmic bytes per layer = E*(4F + 4 [nbr idx] + 4 [dinv/deg]) +
// N*(4F self + 4F_out write + 8 [offset, degree]).  Neighbors are visited in table order, so in
// STRICT mode (no FMA contraction, reference scaling formula) sums round exactly like the
// reference's sum_incremental accumulators.
#include <type_traits>

#include "kernels.h"

namespace gnnb {

namespace {

template <int VEC>
struct Vec;
template <>
struct Vec<1> {
    float v[1];
    __device__ __forceinline__ void load(const float *p) { v[0] = __ldg(p); }
    __device__ __forceinline__ void load_rw(const float *p) { v[0] = *p; }   // data this kernel also writes
    __device__ __forceinline__ void store(float *p) const { p[0] = v[0]; }
};
template <>
struct Vec<4> {
    float v[4];
    __device__ __forceinline__ void load(const float *p)
    {
        const float4 t = __ldg(reinterpret_cast<const float4 *>(p));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    __device__ __forceinline__ void load_rw(const float *p)
    {
        const float4 t = *reinterpret_cast<const float4 *>(p);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    __device__ __forceinline__ void store(float *p) const
    {
        *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
    }
};

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// f(std::integral_constant<int, LPR>) for a row kernel's runtime lanes per row (1, 2, 4, 8, 16, else
// 32): every launcher instantiates its kernel for all six
template <typename F>
decltype(auto) with_lpr(int lpr, F &&f)
{
    switch (lpr) {
    case 1: return f(std::integral_constant<int, 1>{});
    case 2: return f(std::integral_constant<int, 2>{});
    case 4: return f(std::integral_constant<int, 4>{});
    case 8: return f(std::integral_constant<int, 8>{});
    case 16: return f(std::integral_constant<int, 16>{});
    default: return f(std::integral_constant<int, 32>{});
    }
}

// grid of a row kernel: 256-thread CTAs of 8 * (32 / lpr) rows, at most `cap` of them (the kernels
// grid-stride beyond; the default is 8 resident CTAs per SM x 4 waves)
inline int row_grid(int n, int lpr, int64_t cap = (int64_t)kNumSMs * 8 * 4)
{
    const int64_t g = ceil_div64(n, 8 * (32 / lpr));
    return (int)(g < cap ? g : cap);
}

// L2 eviction-priority policies for the gathers of a large graph (hub_bit mode): rows of hub
// sources are kept (evict_last), everything else streams through (evict_first).
__device__ __forceinline__ uint64_t l2_policy_keep()
{
    uint64_t p;
    asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;\n" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_stream()
{
    uint64_t p;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(p));
    return p;
}
template <int VEC>
__device__ __forceinline__ void load_hint(Vec<VEC> &x, const float *p, uint64_t pol);
template <>
__device__ __forceinline__ void load_hint<1>(Vec<1> &x, const float *p, uint64_t pol)
{
    asm("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;\n" : "=f"(x.v[0]) : "l"(p), "l"(pol));
}
template <>
__device__ __forceinline__ void load_hint<4>(Vec<4> &x, const float *p, uint64_t pol)
{
    asm("ld.global.nc.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;\n"
        : "=f"(x.v[0]), "=f"(x.v[1]), "=f"(x.v[2]), "=f"(x.v[3])
        : "l"(p), "l"(pol));
}

template <int MODE, bool STRICT>
__device__ __forceinline__ float neighbor_scale(const AggArgs &a, int deg_v, float dinv_v, int u)
{
    if (MODE == AGG_GCN) {
        if (STRICT) {
            const float di = __fadd_rn(1.0f, (float)deg_v);
            const float dj = __fadd_rn(1.0f, (float)__ldg(a.in_deg + u));
            return __fdiv_rn(1.0f, __fsqrt_rn(__fmul_rn(di, dj)));  // lib:1249-1252
        }
        return __ldg(a.dinv + u);  // rsqrt(1+d_u); the rsqrt(1+d_v) factor is applied once at the end
    }
    if (MODE == AGG_LG) {
        return __fdiv_rn(1.0f, __fsqrt_rn((float)(deg_v * __ldg(a.in_deg + u))));  // lib:2386
    }
    return 1.0f;
}

template <int VEC, int MODE, bool STRICT>
__device__ __forceinline__ void accumulate(Vec<VEC> &acc, const Vec<VEC> &x, float scale)
{
#pragma unroll
    for (int i = 0; i < VEC; i++) {
        if (MODE == AGG_GCN || MODE == AGG_LG)
            acc.v[i] = mac<STRICT>(acc.v[i], x.v[i], scale);
        else
            acc.v[i] = __fadd_rn(acc.v[i], x.v[i]);
    }
}

// partial sum over neighbors [k0, k1) of row v for the feature chunk starting at column c
template <int VEC, int MODE, bool STRICT>
__device__ __forceinline__ void gather_range(const AggArgs &a, int off, int k0, int k1, int deg_v,
                                             float dinv_v, int c, Vec<VEC> &acc)
{
    int k = k0;
    if (!STRICT && a.hub_bit) {
        const uint64_t keep = l2_policy_keep(), stream = l2_policy_stream();
        for (; k + 4 <= k1; k += 4) {
            int u[4];
            Vec<VEC> x[4];
            float sc[4];
#pragma unroll
            for (int j = 0; j < 4; j++) u[j] = __ldg(a.nbr + off + k + j);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint64_t pol = u[j] < 0 ? keep : stream;
                u[j] &= 0x7fffffff;
                load_hint<VEC>(x[j], a.x + (size_t)u[j] * a.ldx + c, pol);
            }
#pragma unroll
            for (int j = 0; j < 4; j++) sc[j] = neighbor_scale<MODE, STRICT>(a, deg_v, dinv_v, u[j]);
#pragma unroll
            for (int j = 0; j < 4; j++) accumulate<VEC, MODE, STRICT>(acc, x[j], sc[j]);
        }
        for (; k < k1; k++) {
            int u = __ldg(a.nbr + off + k);
            const uint64_t pol = u < 0 ? keep : stream;
            u &= 0x7fffffff;
            Vec<VEC> x;
            load_hint<VEC>(x, a.x + (size_t)u * a.ldx + c, pol);
            accumulate<VEC, MODE, STRICT>(acc, x, neighbor_scale<MODE, STRICT>(a, deg_v, dinv_v, u));
        }
        return;
    }
    for (; k + 4 <= k1; k += 4) {
        int u[4];
        Vec<VEC> x[4];
        float sc[4];
#pragma unroll
        for (int j = 0; j < 4; j++) u[j] = __ldg(a.nbr + off + k + j);
#pragma unroll
        for (int j = 0; j < 4; j++) x[j].load(a.x + (size_t)u[j] * a.ldx + c);
#pragma unroll
        for (int j = 0; j < 4; j++) sc[j] = neighbor_scale<MODE, STRICT>(a, deg_v, dinv_v, u[j]);
#pragma unroll
        for (int j = 0; j < 4; j++) accumulate<VEC, MODE, STRICT>(acc, x[j], sc[j]);
    }
    for (; k < k1; k++) {
        const int u = __ldg(a.nbr + off + k);
        Vec<VEC> x;
        x.load(a.x + (size_t)u * a.ldx + c);
        accumulate<VEC, MODE, STRICT>(acc, x, neighbor_scale<MODE, STRICT>(a, deg_v, dinv_v, u));
    }
}

// self term / normalisation and store
template <int VEC, int MODE, bool STRICT>
__device__ __forceinline__ void finish_row(const AggArgs &a, int v, int deg_v, float dinv_v, int c,
                                           Vec<VEC> &acc)
{
    if (!STRICT && a.no_finish) {   // first part of a split CSR: the plain partial sum
        acc.store(a.out + (size_t)v * a.ldo + c);
        return;
    }
    if (MODE == AGG_GCN) {
        Vec<VEC> xs;
        xs.load(a.x + (size_t)(v + a.row_base) * a.ldx + c);
        if (STRICT) {
            const float di = __fadd_rn(1.0f, (float)deg_v);
            const float ss = __fdiv_rn(1.0f, __fsqrt_rn(__fmul_rn(di, di)));  // lib:1266-1267
#pragma unroll
            for (int i = 0; i < VEC; i++)
                acc.v[i] = __fadd_rn(acc.v[i], __fmul_rn(xs.v[i], ss));
        } else {
            const float ss = dinv_v * dinv_v;
#pragma unroll
            for (int i = 0; i < VEC; i++) acc.v[i] = fmaf(xs.v[i], ss, acc.v[i] * dinv_v);
        }
    } else if (MODE == AGG_GIN) {
        Vec<VEC> xs;
        xs.load(a.x + (size_t)(v + a.row_base) * a.ldx + c);
        const float s = __fadd_rn(1.0f, a.eps);  // lib:1522
#pragma unroll
        for (int i = 0; i < VEC; i++) acc.v[i] = __fadd_rn(acc.v[i], __fmul_rn(xs.v[i], s));
    } else if (MODE == AGG_MEAN) {
        if (deg_v > 0) {
            const float d = (float)deg_v;
#pragma unroll
            for (int i = 0; i < VEC; i++) acc.v[i] = __fdiv_rn(acc.v[i], d);  // lib:661
        }
    }
    acc.store(a.out + (size_t)v * a.ldo + c);
}

// LPR lanes cooperate on one destination row; 32/LPR rows per warp.
template <int VEC, int LPR, int MODE, bool STRICT>
__global__ void __launch_bounds__(256) agg_rows_kernel(const AggArgs a)
{
    constexpr int ROWS_PER_WARP = 32 / LPR;
    const int lane = threadIdx.x & 31;
    const int lg = lane % LPR;
    const int sub = lane / LPR;
    const int warps_per_block = blockDim.x >> 5;
    const int64_t warp_global = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int64_t warp_stride = (int64_t)gridDim.x * warps_per_block;
    for (int64_t row0 = warp_global * ROWS_PER_WARP; row0 < a.n; row0 += warp_stride * ROWS_PER_WARP) {
        const int v = (int)row0 + sub;
        if (v >= a.n) continue;
        const int deg_v = __ldg(a.in_deg + v);
        const int len_v = (!STRICT && a.counts != nullptr) ? __ldg(a.counts + v) : deg_v;
        if (a.heavy.n > 0 && len_v > a.heavy.threshold) continue;  // CTA-per-row kernel does these
        const int off = __ldg(a.offsets + v);
        const float dinv_v = (MODE == AGG_GCN && !STRICT) ? __ldg(a.dinv + v + a.row_base) : 0.0f;
        for (int c = lg * VEC; c < a.F; c += LPR * VEC) {
            Vec<VEC> acc;
            if (!STRICT && a.accumulate) {
                acc.load_rw(a.out + (size_t)v * a.ldo + c);
            } else {
#pragma unroll
                for (int i = 0; i < VEC; i++) acc.v[i] = 0.0f;
            }
            gather_range<VEC, MODE, STRICT>(a, off, 0, len_v, deg_v, dinv_v, c, acc);
            finish_row<VEC, MODE, STRICT>(a, v, deg_v, dinv_v, c, acc);
        }
    }
}

// Heavy rows (longer than the threshold; on the 2M-node power-law graph 0.5 % of the rows hold
// 49 % of the edges): the neighbor list of row h is cut into chunks of kHeavyChunk neighbors and
// every chunk is one warp's work item (grid-stride over all chunks of all heavy rows, so a
// 300-neighbor row and a 100 000-neighbor hub load the machine alike); the chunk sums go to
// partial[chunk][F].  A second kernel adds a row's chunks in order and applies the self term /
// normalisation, so the result does not depend on scheduling.  (Round 1 cut every heavy row into
// a fixed number of slices x 8 warps: rows just above the threshold then gave each warp one or two
// neighbors, and the kernel reached 38 % of the DRAM rate the light-row kernel reaches.)
template <int VEC, int MODE>
__global__ void __launch_bounds__(256) agg_heavy_chunk_kernel(const AggArgs a)
{
    const int lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    const int warp_global = blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int warp_stride = gridDim.x * warps_per_block;
    for (int chunk = warp_global; chunk < a.heavy.chunks; chunk += warp_stride) {
        const int h = __ldg(a.heavy.chunk_row + chunk);
        const int v = __ldg(a.heavy.rows + h);
        const int j = chunk - __ldg(a.heavy.chunk_base + h);
        const int deg_v = __ldg(a.in_deg + v);
        const int len_v = a.counts != nullptr ? __ldg(a.counts + v) : deg_v;
        const int off = __ldg(a.offsets + v);
        const float dinv_v = (MODE == AGG_GCN) ? __ldg(a.dinv + v + a.row_base) : 0.0f;
        const int k0 = j * kHeavyChunk, k1 = min(len_v, k0 + kHeavyChunk);
        float *dst = a.heavy.partial + (size_t)chunk * a.F;
        for (int c = lane * VEC; c < a.F; c += 32 * VEC) {
            Vec<VEC> acc;
#pragma unroll
            for (int i = 0; i < VEC; i++) acc.v[i] = 0.0f;
            gather_range<VEC, MODE, false>(a, off, k0, k1, deg_v, dinv_v, c, acc);
            acc.store(dst + c);
        }
    }
}

// One CTA per heavy row: its 8 warps add contiguous ranges of the row's chunk sums (a hub with
// 100 000 neighbors has 782 of them: one warp walking them alone took ~100 us, a constant that
// did not shrink with the GPU count), the 8 range sums are then added in warp order through shared
// memory and the row is finished -- a fixed order, so the result does not depend on scheduling.
template <int VEC, int MODE>
__global__ void __launch_bounds__(256) agg_heavy_combine_kernel(const AggArgs a)
{
    extern __shared__ float ranges[];   // [8][F]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int h = blockIdx.x; h < a.heavy.n; h += gridDim.x) {
        const int v = __ldg(a.heavy.rows + h);
        const int deg_v = __ldg(a.in_deg + v);
        const int len_v = a.counts != nullptr ? __ldg(a.counts + v) : deg_v;
        const int nch = (len_v + kHeavyChunk - 1) / kHeavyChunk;
        const float *src = a.heavy.partial + (size_t)__ldg(a.heavy.chunk_base + h) * a.F;
        const float dinv_v = (MODE == AGG_GCN) ? __ldg(a.dinv + v + a.row_base) : 0.0f;
        const int per = (nch + 7) / 8;
        const int j0 = min(nch, warp * per), j1 = min(nch, j0 + per);
        for (int c = lane * VEC; c < a.F; c += 32 * VEC) {
            Vec<VEC> acc;
#pragma unroll
            for (int i = 0; i < VEC; i++) acc.v[i] = 0.0f;
            int j = j0;
            for (; j + 4 <= j1; j += 4) {     // four independent loads in flight, added in order
                Vec<VEC> t[4];
#pragma unroll
                for (int q = 0; q < 4; q++) t[q].load_rw(src + (size_t)(j + q) * a.F + c);
#pragma unroll
                for (int q = 0; q < 4; q++)
#pragma unroll
                    for (int i = 0; i < VEC; i++) acc.v[i] += t[q].v[i];
            }
            for (; j < j1; j++) {
                Vec<VEC> t;
                t.load_rw(src + (size_t)j * a.F + c);
#pragma unroll
                for (int i = 0; i < VEC; i++) acc.v[i] += t.v[i];
            }
#pragma unroll
            for (int i = 0; i < VEC; i++) ranges[warp * a.F + c + i] = acc.v[i];
        }
        __syncthreads();
        if (warp == 0) {
            for (int c = lane * VEC; c < a.F; c += 32 * VEC) {
                Vec<VEC> acc;
                if (a.accumulate) {
                    acc.load_rw(a.out + (size_t)v * a.ldo + c);
                } else {
#pragma unroll
                    for (int i = 0; i < VEC; i++) acc.v[i] = 0.0f;
                }
#pragma unroll
                for (int w = 0; w < 8; w++)
#pragma unroll
                    for (int i = 0; i < VEC; i++) acc.v[i] += ranges[w * a.F + c + i];
                finish_row<VEC, MODE, false>(a, v, deg_v, dinv_v, c, acc);
            }
        }
        __syncthreads();
    }
}

template <int VEC, int LPR, bool STRICT>
int launch_mode(const AggArgs &a, int grid, cudaStream_t s)
{
    switch (a.mode) {
    case AGG_GCN: agg_rows_kernel<VEC, LPR, AGG_GCN, STRICT><<<grid, 256, 0, s>>>(a); break;
    case AGG_GIN: agg_rows_kernel<VEC, LPR, AGG_GIN, STRICT><<<grid, 256, 0, s>>>(a); break;
    case AGG_MEAN: agg_rows_kernel<VEC, LPR, AGG_MEAN, STRICT><<<grid, 256, 0, s>>>(a); break;
    case AGG_SUM: agg_rows_kernel<VEC, LPR, AGG_SUM, STRICT><<<grid, 256, 0, s>>>(a); break;
    case AGG_LG: agg_rows_kernel<VEC, LPR, AGG_LG, STRICT><<<grid, 256, 0, s>>>(a); break;
    default: set_error("unknown aggregation mode"); return GNNB_ERR_INVALID;
    }
    return GNNB_OK;
}

template <int VEC, int MODE>
void launch_heavy_mode(const AggArgs &a, cudaStream_t s)
{
    const int cap = a.short_ctas ? (1 << 30) : kNumSMs * 8;   // 8 resident CTAs per SM, grid-stride beyond
    const int g1 = min((a.heavy.chunks + 7) / 8, cap), g2 = min(a.heavy.n, cap);
    agg_heavy_chunk_kernel<VEC, MODE><<<g1, 256, 0, s>>>(a);
    agg_heavy_combine_kernel<VEC, MODE><<<g2, 256, sizeof(float) * 8 * (size_t)a.F, s>>>(a);
}

template <int VEC>
int launch_heavy(const AggArgs &a, cudaStream_t s)
{
    switch (a.mode) {
    case AGG_GCN: launch_heavy_mode<VEC, AGG_GCN>(a, s); break;
    case AGG_GIN: launch_heavy_mode<VEC, AGG_GIN>(a, s); break;
    case AGG_MEAN: launch_heavy_mode<VEC, AGG_MEAN>(a, s); break;
    case AGG_SUM: launch_heavy_mode<VEC, AGG_SUM>(a, s); break;
    default: set_error("heavy-row path: unsupported mode"); return GNNB_ERR_INVALID;
    }
    return GNNB_OK;
}

// the heavy-row block of an aggregation whose bucketing is on (heavy.n > 0)
int check_heavy(const HeavyArgs &h)
{
    GNNB_REQUIRE(h.rows != nullptr && h.partial != nullptr && h.chunks > 0 && h.chunk_base != nullptr &&
                     h.chunk_row != nullptr,
                 "heavy row list / partial buffer missing");
    return GNNB_OK;
}

}  // namespace

int launch_agg(const AggArgs &a_in, bool strict, cudaStream_t s, int *launches)
{
    AggArgs a = a_in;
    if (a.n <= 0) return GNNB_OK;
    GNNB_REQUIRE(a.F > 0, "aggregation: feature size must be positive");
    if (strict) {
        GNNB_REQUIRE(a.counts == nullptr && !a.accumulate && !a.no_finish && !a.hub_bit,
                     "split-CSR / hub-hint aggregation is FAST-mode only");
        a.heavy.n = 0;
    }
    if (a.mode == AGG_GCN && !strict)
        GNNB_REQUIRE(a.dinv != nullptr, "gcn aggregation needs the dinv table in fast mode");
    const bool v4 = (a.F % 4 == 0) && (a.ldx % 4 == 0) && (a.ldo % 4 == 0) && aligned16(a.x) &&
                    aligned16(a.out);
    const int vec = v4 ? 4 : 1;
    int lpr = 1;
    while (lpr < 32 && lpr * vec < a.F) lpr *= 2;
    const int grid = a.short_ctas ? row_grid(a.n, lpr, (int64_t)1 << 30) : row_grid(a.n, lpr);
    GNNB_TRY(with_lpr(lpr, [&](auto L) {
        if (vec == 4)
            return strict ? launch_mode<4, L, true>(a, grid, s) : launch_mode<4, L, false>(a, grid, s);
        return strict ? launch_mode<1, L, true>(a, grid, s) : launch_mode<1, L, false>(a, grid, s);
    }));
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    if (a.heavy.n > 0) {
        GNNB_TRY(check_heavy(a.heavy));
        GNNB_TRY(vec == 4 ? launch_heavy<4>(a, s) : launch_heavy<1>(a, s));
        GNNB_CUDA(cudaGetLastError());
        if (launches) *launches += 2;
    }
    return GNNB_OK;
}

// ------------------------------------------------------------------------------------ PNA
//
// lib:1750-1834 with the legal rewrite W_pre.[x_v || x_u] + b = (W_self.x_v + b) + W_nbr.x_u
// (SURVEY section 7): `ab` holds A = X.W_nbr^T in columns [0,F) and B = X.W_self^T + b_pre in
// columns [F,2F), so the per-edge transformed message is t = A_u + B_v and the aggregation is a
// pure gather-reduce: max, min, mean and Welford variance (lib:677-705, population variance,
// std = sqrt(var + 1e-5); 0/0 = NaN for in-degree 0 exactly like the reference float build).
// The three degree scalers (lib:1973-1984, 2081-2089) are applied here and the 12F concat
// written in the reference's order (lib:1857-1875 minus the leading self block).
namespace {

template <int VEC, int LPR>
__global__ void __launch_bounds__(256) pna_agg_kernel(const PnaAggArgs a)
{
    constexpr int ROWS_PER_WARP = 32 / LPR;
    const int lane = threadIdx.x & 31;
    const int lg = lane % LPR, sub = lane / LPR;
    const int warps_per_block = blockDim.x >> 5;
    const int64_t warp_global = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int64_t warp_stride = (int64_t)gridDim.x * warps_per_block;
    const int F = a.F, ld = 2 * a.F;
    for (int64_t row0 = warp_global * ROWS_PER_WARP; row0 < a.n; row0 += warp_stride * ROWS_PER_WARP) {
        const int v = (int)row0 + sub;
        if (v >= a.n) continue;
        const int deg = __ldg(a.in_deg + v);
        const int off = __ldg(a.offsets + v);
        const int clamped = deg < 1 ? 1 : deg;
        const float lg1 = logf((float)(clamped + 1));
        const float amp = __fdiv_rn(lg1, a.delta), att = __fdiv_rn(a.delta, lg1);
        for (int c = lg * VEC; c < F; c += LPR * VEC) {
            Vec<VEC> b, vmax, vmin, vsum, wmean, wm2;
            b.load(a.ab + (size_t)v * ld + F + c);
#pragma unroll
            for (int i = 0; i < VEC; i++) {
                vmax.v[i] = 0.0f; vmin.v[i] = 0.0f; vsum.v[i] = 0.0f;
                wmean.v[i] = 0.0f; wm2.v[i] = 0.0f;
            }
            for (int k = 0; k < deg; k++) {
                const int u = __ldg(a.nbr + off + k);
                Vec<VEC> t;
                t.load(a.ab + (size_t)u * ld + c);
                const float cnt = (float)(k + 1);
#pragma unroll
                for (int i = 0; i < VEC; i++) {
                    const float tv = __fadd_rn(t.v[i], b.v[i]);
                    vmax.v[i] = (k == 0 || tv > vmax.v[i]) ? tv : vmax.v[i];  // lib:748-759
                    vmin.v[i] = (k == 0 || tv < vmin.v[i]) ? tv : vmin.v[i];  // lib:784-795
                    vsum.v[i] = __fadd_rn(vsum.v[i], tv);
                    const float d = __fsub_rn(tv, wmean.v[i]);                    // lib:693
                    wmean.v[i] = __fadd_rn(wmean.v[i], __fdiv_rn(d, cnt));        // lib:694
                    wm2.v[i] = __fadd_rn(wm2.v[i], __fmul_rn(d, __fsub_rn(tv, wmean.v[i])));
                }
            }
            Vec<VEC> o[12];
#pragma unroll
            for (int i = 0; i < VEC; i++) {
                const float mean = deg > 0 ? __fdiv_rn(vsum.v[i], (float)deg) : 0.0f;
                const float var = __fdiv_rn(wm2.v[i], (float)deg);                 // lib:702
                const float sd = __fsqrt_rn(__fadd_rn(var, 1e-5f));                // lib:703
                const float q[4] = {vmax.v[i], vmin.v[i], mean, sd};
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    o[j].v[i] = q[j];
                    o[4 + j].v[i] = __fmul_rn(amp, q[j]);
                    o[8 + j].v[i] = __fmul_rn(att, q[j]);
                }
            }
            if (a.compact) {
                float *dst = a.cat12 + (size_t)v * 4 * F + c;
#pragma unroll
                for (int j = 0; j < 4; j++) o[j].store(dst + (size_t)j * F);
            } else {
                float *dst = a.cat12 + (size_t)v * 12 * F + c;
#pragma unroll
                for (int j = 0; j < 12; j++) o[j].store(dst + (size_t)j * F);
            }
        }
    }
}

}  // namespace

int launch_pna_agg(const PnaAggArgs &a, cudaStream_t s, int *launches)
{
    if (a.n <= 0) return GNNB_OK;
    const bool v4 = (a.F % 4 == 0) && aligned16(a.ab) && aligned16(a.cat12);
    const int vec = v4 ? 4 : 1;
    int lpr = 1;
    while (lpr < 32 && lpr * vec < a.F) lpr *= 2;
    const int grid = row_grid(a.n, lpr);
    with_lpr(lpr, [&](auto L) {
        if (vec == 4) pna_agg_kernel<4, L><<<grid, 256, 0, s>>>(a);
        else pna_agg_kernel<1, L><<<grid, 256, 0, s>>>(a);
    });
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    return GNNB_OK;
}

// ------------------------------------------------------------------------------ PNA, split CSR
//
// The row-partitioned form of pna_agg_kernel: the in-edges of an owned row come in two parts, the
// owned-source edges and then the halo-source edges, and A_u is read from ext space (owned rows,
// then the A rows the owners sent).  One running sample count spans both parts, so max/min take
// the first sample of the combined order (lib:748-752, 784-788) and the Welford update (lib:693-695)
// runs over it as if the row's neighbor list were the concatenation; mean, std and the degree
// scalers use the row's full in-degree (= own + halo count), and in-degree 0 gives std = NaN like
// lib:702.
namespace {

template <int VEC>
__device__ __forceinline__ void store_scaled(const Vec<VEC> &x, float scale, float *p)
{
    Vec<VEC> o;
#pragma unroll
    for (int i = 0; i < VEC; i++) o.v[i] = __fmul_rn(scale, x.v[i]);
    o.store(p);
}

template <int VEC>
__device__ __forceinline__ void pna_halo_part(const PnaHaloArgs &a, const int32_t *nbr, int off, int len,
                                              int c, const Vec<VEC> &b, int &cnt, Vec<VEC> &vmax,
                                              Vec<VEC> &vmin, Vec<VEC> &vsum, Vec<VEC> &wmean,
                                              Vec<VEC> &wm2)
{
    for (int k = 0; k < len; k++) {
        const int u = __ldg(nbr + off + k) & 0x7fffffff;   // hub marks carry no index bits
        Vec<VEC> t;
        t.load(a.a_ext + (size_t)u * a.F + c);
        const bool first = cnt == 0;
        cnt++;
        const float fc = (float)cnt;
#pragma unroll
        for (int i = 0; i < VEC; i++) {
            const float tv = __fadd_rn(t.v[i], b.v[i]);
            vmax.v[i] = (first || tv > vmax.v[i]) ? tv : vmax.v[i];
            vmin.v[i] = (first || tv < vmin.v[i]) ? tv : vmin.v[i];
            vsum.v[i] = __fadd_rn(vsum.v[i], tv);
            const float d = __fsub_rn(tv, wmean.v[i]);
            wmean.v[i] = __fadd_rn(wmean.v[i], __fdiv_rn(d, fc));
            wm2.v[i] = __fadd_rn(wm2.v[i], __fmul_rn(d, __fsub_rn(tv, wmean.v[i])));
        }
    }
}

template <int VEC, int LPR>
__global__ void __launch_bounds__(256) pna_halo_stats_kernel(const PnaHaloArgs a)
{
    constexpr int ROWS_PER_WARP = 32 / LPR;
    const int lane = threadIdx.x & 31;
    const int lg = lane % LPR, sub = lane / LPR;
    const int warps_per_block = blockDim.x >> 5;
    const int64_t warp_global = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int64_t warp_stride = (int64_t)gridDim.x * warps_per_block;
    const int F = a.F;
    for (int64_t row0 = warp_global * ROWS_PER_WARP; row0 < a.n; row0 += warp_stride * ROWS_PER_WARP) {
        const int v = (int)row0 + sub;
        if (v >= a.n) continue;
        const int deg = __ldg(a.in_deg + v);
        const int own_off = __ldg(a.own_off + v), own_len = __ldg(a.own_cnt + v);
        const int halo_off = a.halo_cnt != nullptr ? __ldg(a.halo_off + v) : 0;
        const int halo_len = a.halo_cnt != nullptr ? __ldg(a.halo_cnt + v) : 0;
        const int clamped = deg < 1 ? 1 : deg;
        const float lg1 = logf((float)(clamped + 1));
        const float amp = __fdiv_rn(lg1, a.delta), att = __fdiv_rn(a.delta, lg1);
        for (int c = lg * VEC; c < F; c += LPR * VEC) {
            Vec<VEC> b, vmax, vmin, vsum, wmean, wm2;
            b.load(a.b + (size_t)v * F + c);
#pragma unroll
            for (int i = 0; i < VEC; i++) {
                vmax.v[i] = 0.0f; vmin.v[i] = 0.0f; vsum.v[i] = 0.0f;
                wmean.v[i] = 0.0f; wm2.v[i] = 0.0f;
            }
            int cnt = 0;
            pna_halo_part<VEC>(a, a.own_nbr, own_off, own_len, c, b, cnt, vmax, vmin, vsum, wmean, wm2);
            pna_halo_part<VEC>(a, a.halo_nbr, halo_off, halo_len, c, b, cnt, vmax, vmin, vsum, wmean, wm2);
            Vec<VEC> mean, sd;
#pragma unroll
            for (int i = 0; i < VEC; i++) {
                mean.v[i] = deg > 0 ? __fdiv_rn(vsum.v[i], (float)deg) : 0.0f;
                const float var = __fdiv_rn(wm2.v[i], (float)deg);                 // lib:702
                sd.v[i] = __fsqrt_rn(__fadd_rn(var, 1e-5f));                       // lib:703
            }
            float *dst = a.cat12 + (size_t)v * (a.compact ? 4 : 12) * F + c;
            vmax.store(dst);
            vmin.store(dst + F);
            mean.store(dst + 2 * (size_t)F);
            sd.store(dst + 3 * (size_t)F);
            if (!a.compact) {   // [stats | amp stats | att stats], lib:1857-1875
                store_scaled(vmax, amp, dst + 4 * (size_t)F);
                store_scaled(vmin, amp, dst + 5 * (size_t)F);
                store_scaled(mean, amp, dst + 6 * (size_t)F);
                store_scaled(sd, amp, dst + 7 * (size_t)F);
                store_scaled(vmax, att, dst + 8 * (size_t)F);
                store_scaled(vmin, att, dst + 9 * (size_t)F);
                store_scaled(mean, att, dst + 10 * (size_t)F);
                store_scaled(sd, att, dst + 11 * (size_t)F);
            }
        }
    }
}

}  // namespace

int launch_pna_halo_stats(const PnaHaloArgs &a, cudaStream_t s, int *launches)
{
    if (a.n <= 0) return GNNB_OK;
    GNNB_REQUIRE(a.F > 0 && a.a_ext != nullptr && a.b != nullptr && a.cat12 != nullptr,
                 "pna halo statistics: bad arguments");
    const bool v4 = (a.F % 4 == 0) && aligned16(a.a_ext) && aligned16(a.b) && aligned16(a.cat12);
    const int vec = v4 ? 4 : 1;
    int lpr = 1;
    while (lpr < 32 && lpr * vec < a.F) lpr *= 2;
    const int grid = row_grid(a.n, lpr);
    with_lpr(lpr, [&](auto L) {
        if (vec == 4) pna_halo_stats_kernel<4, L><<<grid, 256, 0, s>>>(a);
        else pna_halo_stats_kernel<1, L><<<grid, 256, 0, s>>>(a);
    });
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    return GNNB_OK;
}

// ------------------------------------------------------------------------------------ GINE
//
// lib:1555-1623 gine_conv_agg: agg_v = sum_k relu(x[u_k] + proj[eid_k]) over the in-edges of v in
// table order, where proj = edge_feat . W_e^T + b_e was computed per edge by one GEMM; then the GIN
// self term (1 + eps) x_v (lib:1519-1529).  A (sub-)warp per destination row like agg_rows_kernel;
// additions are separately rounded in reference order, so STRICT and FAST agree bit for bit.
namespace {

template <int VEC, int LPR>
__global__ void __launch_bounds__(256) gine_agg_kernel(const GineAggArgs a)
{
    constexpr int ROWS_PER_WARP = 32 / LPR;
    const int lane = threadIdx.x & 31;
    const int lg = lane % LPR, sub = lane / LPR;
    const int warps_per_block = blockDim.x >> 5;
    const int64_t warp_global = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int64_t warp_stride = (int64_t)gridDim.x * warps_per_block;
    const float self_scale = __fadd_rn(1.0f, a.eps);   // lib:1522
    for (int64_t row0 = warp_global * ROWS_PER_WARP; row0 < a.n; row0 += warp_stride * ROWS_PER_WARP) {
        const int v = (int)row0 + sub;
        if (v >= a.n) continue;
        const int deg = __ldg(a.in_deg + v);
        const int off = __ldg(a.offsets + v);
        for (int c = lg * VEC; c < a.F; c += LPR * VEC) {
            Vec<VEC> acc;
#pragma unroll
            for (int i = 0; i < VEC; i++) acc.v[i] = 0.0f;
            for (int k = 0; k < deg; k++) {
                const int u = __ldg(a.nbr + off + k);
                const int eid = __ldg(a.edge_index + off + k);
                Vec<VEC> xu, pe;
                xu.load(a.x + (size_t)u * a.ldx + c);
                pe.load(a.proj + (size_t)eid * a.ldp + c);
#pragma unroll
                for (int i = 0; i < VEC; i++) {
                    const float m = __fadd_rn(xu.v[i], pe.v[i]);                  // lib:1603
                    acc.v[i] = __fadd_rn(acc.v[i], m > 0.0f ? m : 0.0f);         // lib:1606-1610
                }
            }
            Vec<VEC> xs;
            xs.load(a.x + (size_t)v * a.ldx + c);
#pragma unroll
            for (int i = 0; i < VEC; i++) acc.v[i] = __fadd_rn(acc.v[i], __fmul_rn(xs.v[i], self_scale));
            acc.store(a.out + (size_t)v * a.ldo + c);
        }
    }
}

}  // namespace

int launch_gine_agg(const GineAggArgs &a, cudaStream_t s, int *launches)
{
    if (a.n <= 0) return GNNB_OK;
    const bool v4 = (a.F % 4 == 0) && (a.ldx % 4 == 0) && (a.ldp % 4 == 0) && (a.ldo % 4 == 0) &&
                    aligned16(a.x) && aligned16(a.proj) && aligned16(a.out);
    const int vec = v4 ? 4 : 1;
    int lpr = 1;
    while (lpr < 32 && lpr * vec < a.F) lpr *= 2;
    const int grid = row_grid(a.n, lpr);
    with_lpr(lpr, [&](auto L) {
        if (vec == 4) gine_agg_kernel<4, L><<<grid, 256, 0, s>>>(a);
        else gine_agg_kernel<1, L><<<grid, 256, 0, s>>>(a);
    });
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    return GNNB_OK;
}

// ------------------------------------------------------------------------- GINE, model path
//
// gine_agg_kernel reads a materialised projection proj[E][F] (4F bytes per edge, written by a GEMM
// and read back, every layer).  Here each edge's projection is computed where it is consumed:
// W_e^T [edge_dim][F] and b_e sit in shared memory, the edge's edge_dim features are one broadcast
// load per (sub-)warp, and the lanes of the row's (sub-)warp compute their columns of
// b_e + sum_j W_e[c][j] ef[j] (separately rounded, ascending j: the reference's linear, lib:852-903
// with BLOCK_SIZE_IN = 1), add x_u, apply ReLU and accumulate in neighbor-table order.  Per edge the
// kernel reads 4 edge_dim bytes of features instead of 4F of projection.  No heavy-row bucketing:
// a hub row is one (sub-)warp's serial work.
namespace {

template <int VEC, int LPR, bool SMEM>
__global__ void __launch_bounds__(256) gine_agg_proj_kernel(const GineProjAggArgs a)
{
    extern __shared__ float4 gine_smem4[];
    float *const smem = reinterpret_cast<float *>(gine_smem4);
    const float *Wt = a.We_t;
    const float *be = a.be;
    if (SMEM) {   // [edge_dim][ldw] W_e^T, then [F] b_e
        const int nw = a.edge_dim * a.ldw;
        for (int i = threadIdx.x; i < nw; i += blockDim.x) smem[i] = __ldg(a.We_t + i);
        for (int i = threadIdx.x; i < a.F; i += blockDim.x) smem[nw + i] = __ldg(a.be + i);
        __syncthreads();
        Wt = smem;
        be = smem + nw;
    }
    constexpr int ROWS_PER_WARP = 32 / LPR;
    const int lane = threadIdx.x & 31;
    const int lg = lane % LPR, sub = lane / LPR;
    const int warps_per_block = blockDim.x >> 5;
    const int64_t warp_global = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int64_t warp_stride = (int64_t)gridDim.x * warps_per_block;
    const float self_scale = __fadd_rn(1.0f, a.eps);   // lib:1522
    const int ed = a.edge_dim;
    for (int64_t row0 = warp_global * ROWS_PER_WARP; row0 < a.n; row0 += warp_stride * ROWS_PER_WARP) {
        const int v = (int)row0 + sub;
        if (v >= a.n) continue;
        const int deg = __ldg(a.in_deg + v);
        const int off = __ldg(a.offsets + v);
        for (int c = lg * VEC; c < a.F; c += LPR * VEC) {
            float bias[VEC];
#pragma unroll
            for (int i = 0; i < VEC; i++) bias[i] = be[c + i];
            Vec<VEC> acc;
#pragma unroll
            for (int i = 0; i < VEC; i++) acc.v[i] = 0.0f;
#pragma unroll 2
            for (int k = 0; k < deg; k++) {
                const int u = __ldg(a.nbr + off + k);
                Vec<VEC> xu;
                xu.load(a.x + (size_t)u * a.ldx + c);
                const float *ef = a.ef_sorted + (size_t)(off + k) * a.lde;
                float p[VEC];
#pragma unroll
                for (int i = 0; i < VEC; i++) p[i] = bias[i];   // lib:852-864
                for (int j0 = 0; j0 < ed; j0 += 4) {
                    const float4 e4 = __ldg(reinterpret_cast<const float4 *>(ef + j0));
#pragma unroll
                    for (int jj = 0; jj < 4; jj++) {
                        if (j0 + jj < ed) {
                            const float ej = jj == 0 ? e4.x : jj == 1 ? e4.y : jj == 2 ? e4.z : e4.w;
                            Vec<VEC> w;
                            if (SMEM) w.load_rw(Wt + (size_t)(j0 + jj) * a.ldw + c);
                            else w.load(Wt + (size_t)(j0 + jj) * a.ldw + c);
#pragma unroll
                            for (int i = 0; i < VEC; i++)
                                p[i] = __fadd_rn(p[i], __fmul_rn(w.v[i], ej));   // lib:891, 901
                        }
                    }
                }
#pragma unroll
                for (int i = 0; i < VEC; i++) {
                    const float m = __fadd_rn(xu.v[i], p[i]);                     // lib:1603
                    acc.v[i] = __fadd_rn(acc.v[i], m > 0.0f ? m : 0.0f);         // lib:1606-1610
                }
            }
            Vec<VEC> xs;
            xs.load(a.x + (size_t)v * a.ldx + c);
#pragma unroll
            for (int i = 0; i < VEC; i++) acc.v[i] = __fadd_rn(acc.v[i], __fmul_rn(xs.v[i], self_scale));
            acc.store(a.out + (size_t)v * a.ldo + c);
        }
    }
}

template <int VEC, bool SMEM>
int launch_gine_proj_lpr(const GineProjAggArgs &a, int lpr, int grid, size_t smem, cudaStream_t s)
{
    void (*k)(const GineProjAggArgs) =
        with_lpr(lpr, [](auto L) { return gine_agg_proj_kernel<VEC, L, SMEM>; });
    if (smem > 48 * 1024) GNNB_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<grid, 256, smem, s>>>(a);
    return GNNB_OK;
}

__global__ void permute_edge_rows_kernel(const float *__restrict__ src, int dim,
                                         const int32_t *__restrict__ idx, int64_t e,
                                         float *__restrict__ dst, int ldd)
{
    const int64_t total = e * ldd;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t k = t / ldd;
        const int j = (int)(t - k * ldd);
        dst[t] = j < dim ? __ldg(src + (size_t)__ldg(idx + k) * dim + j) : 0.0f;
    }
}

}  // namespace

int launch_gine_agg_proj(const GineProjAggArgs &a, cudaStream_t s, int *launches)
{
    if (a.n <= 0) return GNNB_OK;
    GNNB_REQUIRE(a.F > 0 && a.edge_dim >= 1 && a.edge_dim <= kGineMaxEdgeDim && a.lde % 4 == 0 &&
                     a.lde >= a.edge_dim && a.ldw % 4 == 0 && a.ldw >= a.F && aligned16(a.ef_sorted),
                 "gine aggregation: bad arguments");
    const bool v4 = (a.F % 4 == 0) && (a.ldx % 4 == 0) && (a.ldo % 4 == 0) && aligned16(a.x) &&
                    aligned16(a.out) && aligned16(a.We_t);
    const int vec = v4 ? 4 : 1;
    int lpr = 1;
    while (lpr < 32 && lpr * vec < a.F) lpr *= 2;
    const int grid = row_grid(a.n, lpr);
    // W_e^T + b_e in shared memory when they fit (edge_dim 64 at F = 512: 130 KB); wider layers
    // read them through the read-only cache
    const size_t smem = sizeof(float) * ((size_t)a.edge_dim * a.ldw + a.F);
    const bool in_smem = smem <= 200 * 1024;
    int rc;
    if (in_smem)
        rc = vec == 4 ? launch_gine_proj_lpr<4, true>(a, lpr, grid, smem, s)
                      : launch_gine_proj_lpr<1, true>(a, lpr, grid, smem, s);
    else
        rc = vec == 4 ? launch_gine_proj_lpr<4, false>(a, lpr, grid, 0, s)
                      : launch_gine_proj_lpr<1, false>(a, lpr, grid, 0, s);
    GNNB_TRY(rc);
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    return GNNB_OK;
}

int launch_permute_edge_rows(const float *src, int dim, const int32_t *idx, int e, float *dst,
                             int ldd, cudaStream_t s, int *launches)
{
    if (e <= 0) return GNNB_OK;
    const int64_t total = (int64_t)e * ldd;
    int64_t grid64 = ceil_div64(total, 256);
    const int64_t cap = (int64_t)kNumSMs * 16;
    permute_edge_rows_kernel<<<(int)(grid64 < cap ? grid64 : cap), 256, 0, s>>>(src, dim, idx, e,
                                                                                 dst, ldd);
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    return GNNB_OK;
}

// ------------------------------------------------------------------------------------- GAT
//
// PyG GATConv (concat heads, self loops replaced by one per node, inference).  The layer's one GEMM
// wrote [h (H*C) | a_src (H) | a_dst (H)] per row (the logit vectors are folded into the weights at
// finalize), so this is a pure gather.  A (sub-)warp per destination row with the LPR/VEC scheme of
// agg_rows_kernel; each lane owns VEC columns of one head (VEC = 4 needs C % 4 == 0).  Every lane
// runs one online softmax over the row in neighbor-table order: it starts from the self term
// (logit e_vv, weight 1, h_v), skips neighbor entries equal to v (the input's self loops are
// replaced by that one term; duplicate edges count once per entry), and for each other entry keeps
// the running max m, the sum s of exp(e - m) and the accumulator of exp(e - m) h_u, rescaling both
// when the max grows.  Every exponent is <= 0, so logits of any size neither overflow nor give NaN,
// and s >= 1.  The epilogue writes act(acc / s + bias (+ skip)): the bias, skip and activation the
// other convs apply in their GEMM epilogue.
//
// Heavy rows (the same bucketing as launch_agg): each kHeavyChunk-neighbor chunk is one warp's work
// and stores its per-head (m, s) and its accumulator (relative to its own m) in the partial scratch.
// One CTA per row then merges the chunks -- 8 warps over contiguous chunk ranges, then the self term
// and the 8 range results in warp order -- a fixed order, so the result does not depend on
// scheduling.  GATv2 shares the online softmax, the epilogue, the partial store, both combine steps
// and the heavy launch defined here (the attn_* functions, over AttnAggArgs).  Algorithmic bytes per
// layer: E (4 + 4H + 4HC) + N (8 + 4H + 4HC [+ 4HC skip]).
//
// Edge attention (GATConv with edge_dim; the EDGE instantiations): the logit of slot k adds the edge
// term elog[k][hd] and the self term self_elog[v][hd], both computed once per run by
// gat_edge_logits_kernel, so a layer reads H more floats per edge and per node: + E 4H + N 4H.
// The plain instantiations are unchanged.
namespace {

__device__ __forceinline__ float leaky_relu(float x, float slope) { return x > 0.0f ? x : x * slope; }

// One lane's online softmax over NJ groups of VEC columns of one head (GAT: NJ = 1)
template <int VEC, int NJ = 1>
struct OnlineSoftmax {
    float m, s;
    Vec<VEC> acc[NJ];
    __device__ __forceinline__ void reset()
    {
        m = -INFINITY;
        s = 0.0f;
#pragma unroll
        for (int j = 0; j < NJ; j++)
#pragma unroll
            for (int i = 0; i < VEC; i++) acc[j].v[i] = 0.0f;
    }
    // adds a part with max m2, sum s2 and accumulator acc2[NJ] (one edge: e, 1, h_u); an empty part
    // (m2 = -inf, from a chunk of self loops only) changes nothing
    __device__ __forceinline__ void merge(float m2, float s2, const Vec<VEC> *acc2)
    {
        if (m2 == -INFINITY) return;
        const float mn = fmaxf(m, m2);
        const float r = expf(m - mn), p = expf(m2 - mn);
        s = fmaf(s, r, s2 * p);
#pragma unroll
        for (int j = 0; j < NJ; j++)
#pragma unroll
            for (int i = 0; i < VEC; i++) acc[j].v[i] = fmaf(acc[j].v[i], r, acc2[j].v[i] * p);
        m = mn;
    }
};

// the columns of head hd a lane holds: col[j] .. col[j] + VEC for the groups j with valid[j]
template <int NJ>
struct AttnCols {
    int hd;
    int col[NJ];
    bool valid[NJ];
};

// the epilogue of one VEC-column group: out[v][c..] = act(acc / s + bias (+ skip))
template <int VEC>
__device__ __forceinline__ void attn_finish(const AttnAggArgs &a, int v, int c, const Vec<VEC> &acc, float s)
{
    Vec<VEC> b, sk, y;
    b.load(a.bias + c);
    if (a.skip != nullptr) sk.load(a.skip + (size_t)v * a.ldskip + c);
#pragma unroll
    for (int i = 0; i < VEC; i++) {
        float t = acc.v[i] / s + b.v[i];
        if (a.skip != nullptr) t += sk.v[i];
        y.v[i] = act_apply_compact(a.act, t);
    }
    y.store(a.out + (size_t)v * a.ldo + c);
}

// a partial [acc H*C | max H | sum H] (a chunk's in global memory, a range's in shared memory) for the
// lane's columns; head_lane: the one lane of the head that writes (max, sum)
template <int VEC, int NJ>
__device__ __forceinline__ void attn_store_partial(const AttnAggArgs &a, float *dst, const AttnCols<NJ> &cl,
                                                   bool head_lane, const OnlineSoftmax<VEC, NJ> &st)
{
    const int HC = a.H * a.C;
#pragma unroll
    for (int j = 0; j < NJ; j++)
        if (cl.valid[j]) st.acc[j].store(dst + cl.col[j]);
    if (head_lane) {
        dst[HC + cl.hd] = st.m;
        dst[HC + a.H + cl.hd] = st.s;
    }
}

// Combine step 1, one CTA per heavy row h: each of the 8 warps merges a contiguous range of the row's
// chunk partials, column by column, into ranges[warp] ([8][ldp], laid out as the partials).  Returns
// the row.
template <int VEC>
__device__ __forceinline__ int attn_combine_chunks(const AttnAggArgs &a, int h, float *ranges)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int HC = a.H * a.C;
    const int v = __ldg(a.heavy.rows + h);
    const int deg = __ldg(a.in_deg + v);
    const int nch = (deg + kHeavyChunk - 1) / kHeavyChunk;
    const float *src = a.heavy.partial + (size_t)__ldg(a.heavy.chunk_base + h) * a.ldp;
    const int per = (nch + 7) / 8;
    const int j0 = min(nch, warp * per), j1 = min(nch, j0 + per);
    float *mine = ranges + warp * a.ldp;
    for (int c = lane * VEC; c < HC; c += 32 * VEC) {
        const int hd = c / a.C;
        OnlineSoftmax<VEC> st;
        st.reset();
        for (int j = j0; j < j1; j++) {
            const float *p = src + (size_t)j * a.ldp;
            Vec<VEC> t;
            t.load_rw(p + c);
            st.merge(p[HC + hd], p[HC + a.H + hd], &t);
        }
        attn_store_partial<VEC, 1>(a, mine, {hd, {c}, {true}}, c % a.C == 0, st);
    }
    return v;
}

// Combine step 2: merges the 8 range results, in warp order, into st (which holds the self term) for
// the lane's columns; hd is the head whose (max, sum) are read (clamped for idle GATv2 groups)
template <int VEC, int NJ>
__device__ __forceinline__ void attn_merge_ranges(const AttnAggArgs &a, const float *ranges,
                                                  const AttnCols<NJ> &cl, int hd, OnlineSoftmax<VEC, NJ> &st)
{
    const int HC = a.H * a.C;
#pragma unroll 1
    for (int w = 0; w < 8; w++) {
        const float *r = ranges + w * a.ldp;
        Vec<VEC> t[NJ];
#pragma unroll
        for (int j = 0; j < NJ; j++) {
            if (cl.valid[j]) {
                t[j].load_rw(r + cl.col[j]);
            } else {
#pragma unroll
                for (int i = 0; i < VEC; i++) t[j].v[i] = 0.0f;
            }
        }
        st.merge(r[HC + hd], r[HC + a.H + hd], t);
    }
}

// the self term of row v for the lane's columns [c, c + VEC) of head hd; returns a_dst[v][hd]
template <int VEC, bool EDGE>
__device__ __forceinline__ float gat_self(const GatAggArgs &a, int v, int c, int hd, OnlineSoftmax<VEC> &st)
{
    const int HC = a.H * a.C;
    const float *row = a.g + (size_t)v * a.ldg;
    const float adst = __ldg(row + HC + a.H + hd);
    float e = __ldg(row + HC + hd) + adst;
    if (EDGE) e += __ldg(a.self_elog + (size_t)v * a.ldl + hd);
    st.m = leaky_relu(e, a.slope);
    st.s = 1.0f;
    st.acc[0].load(row + c);
    return adst;
}

// neighbor entries [k0, k1) of row v (entries equal to v skipped), four gathers in flight
template <int VEC, bool EDGE>
__device__ __forceinline__ void gat_gather(const GatAggArgs &a, int v, int off, int k0, int k1, int c,
                                           int hd, float adst, OnlineSoftmax<VEC> &st)
{
    const int HC = a.H * a.C;
    int k = k0;
    for (; k + 4 <= k1; k += 4) {
        int u[4];
        float as[4], el[4];
        Vec<VEC> x[4];
#pragma unroll
        for (int j = 0; j < 4; j++) u[j] = __ldg(a.nbr + off + k + j);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const float *row = a.g + (size_t)u[j] * a.ldg;
            as[j] = __ldg(row + HC + hd);
            if (EDGE) el[j] = __ldg(a.elog + (size_t)(off + k + j) * a.ldl + hd);
            x[j].load(row + c);
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            float e = as[j] + adst;
            if (EDGE) e += el[j];
            if (u[j] != v) st.merge(leaky_relu(e, a.slope), 1.0f, &x[j]);
        }
    }
    for (; k < k1; k++) {
        const int u = __ldg(a.nbr + off + k);
        if (u == v) continue;
        const float *row = a.g + (size_t)u * a.ldg;
        Vec<VEC> x;
        x.load(row + c);
        float e = __ldg(row + HC + hd) + adst;
        if (EDGE) e += __ldg(a.elog + (size_t)(off + k) * a.ldl + hd);
        st.merge(leaky_relu(e, a.slope), 1.0f, &x);
    }
}

template <int VEC, int LPR, bool EDGE>
__global__ void __launch_bounds__(256) gat_agg_kernel(const GatAggArgs a)
{
    constexpr int ROWS_PER_WARP = 32 / LPR;
    const int lane = threadIdx.x & 31;
    const int lg = lane % LPR, sub = lane / LPR;
    const int warps_per_block = blockDim.x >> 5;
    const int64_t warp_global = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int64_t warp_stride = (int64_t)gridDim.x * warps_per_block;
    const int HC = a.H * a.C;
    for (int64_t row0 = warp_global * ROWS_PER_WARP; row0 < a.n; row0 += warp_stride * ROWS_PER_WARP) {
        const int v = (int)row0 + sub;
        if (v >= a.n) continue;
        const int deg = __ldg(a.in_deg + v);
        if (a.heavy.n > 0 && deg > a.heavy.threshold) continue;  // the heavy-row kernels do these
        const int off = __ldg(a.offsets + v);
        for (int c = lg * VEC; c < HC; c += LPR * VEC) {
            const int hd = c / a.C;
            OnlineSoftmax<VEC> st;
            const float adst = gat_self<VEC, EDGE>(a, v, c, hd, st);
            gat_gather<VEC, EDGE>(a, v, off, 0, deg, c, hd, adst, st);
            attn_finish(a, v, c, st.acc[0], st.s);
        }
    }
}

template <int VEC, bool EDGE>
__global__ void __launch_bounds__(256) gat_heavy_chunk_kernel(const GatAggArgs a)
{
    const int lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    const int warp_global = blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int warp_stride = gridDim.x * warps_per_block;
    const int HC = a.H * a.C;
    for (int chunk = warp_global; chunk < a.heavy.chunks; chunk += warp_stride) {
        const int h = __ldg(a.heavy.chunk_row + chunk);
        const int v = __ldg(a.heavy.rows + h);
        const int j = chunk - __ldg(a.heavy.chunk_base + h);
        const int deg = __ldg(a.in_deg + v);
        const int off = __ldg(a.offsets + v);
        const int k0 = j * kHeavyChunk, k1 = min(deg, k0 + kHeavyChunk);
        const float *rowv = a.g + (size_t)v * a.ldg;
        float *dst = a.heavy.partial + (size_t)chunk * a.ldp;
        for (int c = lane * VEC; c < HC; c += 32 * VEC) {
            const int hd = c / a.C;
            OnlineSoftmax<VEC> st;
            st.reset();
            gat_gather<VEC, EDGE>(a, v, off, k0, k1, c, hd, __ldg(rowv + HC + a.H + hd), st);
            attn_store_partial<VEC, 1>(a, dst, {hd, {c}, {true}}, c % a.C == 0, st);
        }
    }
}

template <int VEC, bool EDGE>
__device__ __forceinline__ void gat_heavy_combine(const GatAggArgs &a)
{
    extern __shared__ float4 gat_smem4[];
    float *const ranges = reinterpret_cast<float *>(gat_smem4);   // [8][ldp], laid out as the partials
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int HC = a.H * a.C;
    for (int h = blockIdx.x; h < a.heavy.n; h += gridDim.x) {
        const int v = attn_combine_chunks<VEC>(a, h, ranges);
        __syncthreads();
        if (warp == 0) {
            for (int c = lane * VEC; c < HC; c += 32 * VEC) {
                const int hd = c / a.C;
                OnlineSoftmax<VEC> st;
                gat_self<VEC, EDGE>(a, v, c, hd, st);
                attn_merge_ranges<VEC, 1>(a, ranges, {hd, {c}, {true}}, hd, st);
                attn_finish(a, v, c, st.acc[0], st.s);
            }
        }
        __syncthreads();
    }
}

// plain GAT: the kernel as it always was
template <int VEC>
__global__ void __launch_bounds__(256) gat_heavy_combine_kernel(const GatAggArgs a)
{
    gat_heavy_combine<VEC, false>(a);
}
// edge attention: capped at 64 registers, where ptxas's own choice under __launch_bounds__(256)
// spilled it (one CTA per heavy row, so occupancy does not matter here)
template <int VEC>
__global__ void __maxnreg__(64) gat_heavy_combine_edge_kernel(const GatAggArgs a)
{
    gat_heavy_combine<VEC, true>(a);
}

// the heavy rows of an attention aggregation: the chunk kernel, a warp per chunk, then the combine
// kernel, a CTA per row with the [8][ldp] range table in shared memory; extra: the kernels' further
// arguments
template <typename Args, typename... Extra>
int launch_attn_heavy(void (*chunk)(Args, Extra...), void (*combine)(Args, Extra...), const Args &a,
                      cudaStream_t s, int *launches, Extra... extra)
{
    const int cap = kNumSMs * 8;   // 8 resident CTAs per SM, grid-stride beyond
    const int g1 = min((a.heavy.chunks + 7) / 8, cap), g2 = min(a.heavy.n, cap);
    chunk<<<g1, 256, 0, s>>>(a, extra...);
    const size_t smem = sizeof(float) * 8 * (size_t)a.ldp;
    if (smem > 48 * 1024)
        GNNB_CUDA(cudaFuncSetAttribute(combine, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    combine<<<g2, 256, smem, s>>>(a, extra...);
    GNNB_CUDA(cudaGetLastError());
    if (launches) *launches += 2;
    return GNNB_OK;
}

// the arguments the attention aggregations share (what = the conv's name for the messages)
int check_attn_args(const AttnAggArgs &a, const char *what)
{
    const int HC = a.H * a.C;
    GNNB_REQUIRE(a.H >= 1 && a.C >= 1 && a.ldo >= HC && a.bias != nullptr &&
                     (a.skip == nullptr || a.ldskip >= HC),
                 std::string(what) + " aggregation: bad arguments");
    if (a.heavy.n > 0) {
        GNNB_TRY(check_heavy(a.heavy));
        GNNB_REQUIRE(a.ldp >= HC + 2 * a.H && a.ldp % 4 == 0,
                     std::string(what) + " heavy rows: bad partial stride");
    }
    return GNNB_OK;
}

// float4 lanes: C % 4 == 0, and g, output, bias and skip 16-byte aligned with strides of whole float4s
bool attn_v4(const AttnAggArgs &a)
{
    return (a.C % 4 == 0) && (a.ldg % 4 == 0) && aligned16(a.g) && (a.ldo % 4 == 0) && aligned16(a.out) &&
           aligned16(a.bias) && (a.skip == nullptr || ((a.ldskip % 4 == 0) && aligned16(a.skip)));
}

template <int VEC, bool EDGE>
int launch_gat_variant(const GatAggArgs &a, int lpr, cudaStream_t s, int *launches)
{
    const int grid = row_grid(a.n, lpr);
    with_lpr(lpr, [&](auto L) { gat_agg_kernel<VEC, L, EDGE><<<grid, 256, 0, s>>>(a); });
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    if (a.heavy.n == 0) return GNNB_OK;
    auto combine = EDGE ? gat_heavy_combine_edge_kernel<VEC> : gat_heavy_combine_kernel<VEC>;
    return launch_attn_heavy(gat_heavy_chunk_kernel<VEC, EDGE>, combine, a, s, launches);
}

}  // namespace

int launch_gat_agg(const GatAggArgs &a, cudaStream_t s, int *launches)
{
    if (a.n <= 0) return GNNB_OK;
    GNNB_TRY(check_attn_args(a, "gat"));
    GNNB_REQUIRE(a.ldg >= a.H * a.C + 2 * a.H, "gat aggregation: bad arguments");
    const bool edge = a.elog != nullptr;
    if (edge) GNNB_REQUIRE(a.self_elog != nullptr && a.ldl >= a.H, "gat aggregation: bad edge logits");
    const bool v4 = attn_v4(a);
    const int vec = v4 ? 4 : 1;
    int lpr = 1;
    while (lpr < 32 && lpr * vec < a.H * a.C) lpr *= 2;
    if (vec == 4)
        return edge ? launch_gat_variant<4, true>(a, lpr, s, launches)
                    : launch_gat_variant<4, false>(a, lpr, s, launches);
    return edge ? launch_gat_variant<1, true>(a, lpr, s, launches)
                : launch_gat_variant<1, false>(a, lpr, s, launches);
}

// Edge logits of every layer and head, once per run (kernels.h).  LPR lanes per destination row; the
// row's items i = k * LH + lh (slot k, layer-head lh) are spread over them, so each lane's elog
// writes are contiguous with its neighbours'.  The LH lanes of one slot read the same edge_attr row
// (L1 hits); w_edge is staged in shared memory when it fits.  Then, after the warp barrier, each
// lane averages one lh column of the row's elog in slot order for self_elog.  Hub rows are one
// sub-warp's serial work (no bucketing: the pass runs once per run, not once per layer).
// Algorithmic bytes: E (4 + 4 + 4 edge_dim + 4 LH) + N (8 + 4 LH).
namespace {

template <int LPR>
__global__ void __launch_bounds__(256) gat_edge_logits_kernel(const GatEdgeLogitsArgs a, bool w_smem)
{
    extern __shared__ float4 elog_smem4[];
    const float *w = a.w_edge;
    if (w_smem) {
        float *sw = reinterpret_cast<float *>(elog_smem4);
        for (int i = threadIdx.x; i < a.LH * a.edge_dim; i += blockDim.x) sw[i] = __ldg(a.w_edge + i);
        __syncthreads();
        w = sw;
    }
    constexpr int ROWS_PER_WARP = 32 / LPR;
    const int lane = threadIdx.x & 31;
    const int lg = lane % LPR, sub = lane / LPR;
    const int warps_per_block = blockDim.x >> 5;
    const int64_t warp_global = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int64_t warp_stride = (int64_t)gridDim.x * warps_per_block;
    const int LH = a.LH;
    // row0 is warp-uniform, so every lane reaches the __syncwarp
    for (int64_t row0 = warp_global * ROWS_PER_WARP; row0 < a.n; row0 += warp_stride * ROWS_PER_WARP) {
        const int v = (int)row0 + sub;
        const bool valid = v < a.n;
        const int deg = valid ? __ldg(a.in_deg + v) : 0;
        const int off = valid ? __ldg(a.offsets + v) : 0;
        float *el = a.elog + (size_t)off * LH;
        // int64 items: one hub row may hold deg * LH >= 2^31 of them
        const int64_t items = (int64_t)deg * LH;
        for (int64_t i = lg; i < items; i += LPR) {
            const int k = (int)(i / LH), lh = (int)(i - (int64_t)k * LH);
            float acc = 0.0f;   // self-loop slots hold 0: never read as logits, but defined
            if (__ldg(a.nbr + off + k) != v) {
                const float *ef = a.ef + (size_t)__ldg(a.edge_index + off + k) * a.edge_dim;
                const float *wr = w + (size_t)lh * a.edge_dim;
                for (int j = 0; j < a.edge_dim; j++) acc = fmaf(__ldg(ef + j), wr[j], acc);
            }
            el[i] = acc;
        }
        __syncwarp();
        if (!valid) continue;
        for (int lh = lg; lh < LH; lh += LPR) {
            float sum = 0.0f;
            int cnt = 0;
            for (int k = 0; k < deg; k++) {
                if (__ldg(a.nbr + off + k) == v) continue;
                sum += el[(size_t)k * LH + lh];
                cnt++;
            }
            a.self_elog[(size_t)v * LH + lh] = cnt > 0 ? sum / (float)cnt : 0.0f;
        }
    }
}

}  // namespace

int launch_gat_edge_logits(const GatEdgeLogitsArgs &a, int avg_deg, cudaStream_t s, int *launches)
{
    if (a.n <= 0) return GNNB_OK;
    GNNB_REQUIRE(a.edge_dim >= 1 && a.LH >= 1 && a.w_edge != nullptr && a.elog != nullptr &&
                     a.self_elog != nullptr && a.edge_index != nullptr,
                 "gat edge logits: bad arguments");
    int lpr = 1;
    const int64_t items = (int64_t)std::max(avg_deg, 1) * a.LH;
    while (lpr < 32 && lpr < items) lpr *= 2;
    const size_t smem_w = sizeof(float) * (size_t)a.LH * a.edge_dim;
    const bool w_smem = smem_w <= 48 * 1024;
    const size_t smem = w_smem ? smem_w : 0;
    const int grid = row_grid(a.n, lpr, (int64_t)kNumSMs * 8);
    with_lpr(lpr, [&](auto L) { gat_edge_logits_kernel<L><<<grid, 256, smem, s>>>(a, w_smem); });
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    return GNNB_OK;
}

// ----------------------------------------------------------------------------------- GATv2
//
// PyG GATv2Conv (concat heads, self loops replaced by one per node, inference).  The layer's two
// GEMMs wrote [xl | xr] per row.  The logit e_uvh = <att_h, LeakyReLU(xl_u + xr_v (+ e_uv W_e^T))_h>
// has its nonlinearity inside the dot product, so it is formed per edge from the gathered row: each
// lane holds xr_v and att for its columns in registers, forms its partial dot product and the head's
// lanes add the partials with an xor butterfly.  A butterfly gives every lane of the head the same
// bits (each level adds the same two values, commutatively), so their online-softmax states stay
// identical.
//
// Lane layout: a head's columns are spread over G lanes, G the smallest power of two >= C / VEC
// (at most 32), each lane holding NJ <= 2 groups of VEC columns; the G-lane groups are aligned inside
// the row's LPR-lane sub-warp and a sub-warp covers LPR / G heads per pass.  Lanes past C, and the
// groups of a pass past the last head, contribute 0 but run the same shuffles: every shuffle's mask
// is the row's sub-warp, whose lanes all reach it (rows of one warp differ in degree).
//
// The online softmax (OnlineSoftmax with NJ groups), the self term first and the skipping of entries
// equal to v are GAT's.  With edge features each edge's projection is computed where it is consumed
// from ef_sorted[slot] and W_e^T (staged in shared memory when it fits), never materialised.  Heavy
// rows are GAT's chunk / fixed-order combine scheme (attn_store_partial, attn_combine_chunks,
// attn_merge_ranges, launch_attn_heavy).  The kernels declare one resident CTA per SM as their
// minimum: ptxas's own register choice under __launch_bounds__(256) spilled them.  Algorithmic bytes
// per layer: E (4 + 4HC [+ 4 lde]) + N (8 + 8HC + 4HC [+ 4HC skip] [+ 4 lde]).
namespace {

// one lane's share of one head: its columns (AttnCols), and xr_v and att for them
template <int VEC, int NJ>
struct Gatv2Lane : AttnCols<NJ> {
    Vec<VEC> xr[NJ], att[NJ];
};

template <int VEC, int NJ>
__device__ __forceinline__ void gatv2_load(const float *row, const AttnCols<NJ> &cl, Vec<VEC> (&x)[NJ])
{
#pragma unroll
    for (int j = 0; j < NJ; j++) {
        if (cl.valid[j]) {
            x[j].load(row + cl.col[j]);
        } else {
#pragma unroll
            for (int i = 0; i < VEC; i++) x[j].v[i] = 0.0f;
        }
    }
}

// the columns of head hd (>= H: an idle group) that lane hl of its G lanes holds
template <int VEC, int NJ>
__device__ __forceinline__ void attn_lane_cols(const AttnAggArgs &a, int hd, int hl, int G, AttnCols<NJ> &cl)
{
    cl.hd = hd;
#pragma unroll
    for (int j = 0; j < NJ; j++) {
        const int c = (hl + j * G) * VEC;
        cl.valid[j] = hd < a.H && c < a.C;
        cl.col[j] = hd * a.C + c;
    }
}

// head hd (>= H: an idle group), lane hl of its G lanes.  XR: xr has a pointer and stride of its own
// (the row partition); else it sits in columns [H*C, 2 H*C) of g (the model handle), addressed
// from g's row so that those kernels keep their register budget
template <int VEC, int NJ, bool XR>
__device__ __forceinline__ Gatv2Lane<VEC, NJ> gatv2_lane(const Gatv2AggArgs &a, int v, int hd, int hl,
                                                         int G)
{
    Gatv2Lane<VEC, NJ> ln;
    attn_lane_cols<VEC, NJ>(a, hd, hl, G, ln);
    if (XR) {
        gatv2_load<VEC, NJ>(a.xr + (size_t)v * a.ldxr, ln, ln.xr);
    } else {
        const int HC = a.H * a.C;
        AttnCols<NJ> sh = ln;   // the same columns, shifted to xr
#pragma unroll
        for (int j = 0; j < NJ; j++) sh.col[j] += HC;
        gatv2_load<VEC, NJ>(a.g + (size_t)v * a.ldg, sh, ln.xr);
    }
    gatv2_load<VEC, NJ>(a.att, ln, ln.att);
    return ln;
}

// z += ef W_e^T for the lane's columns: ef one row of lde floats (edge_dim used), We [edge_dim][ldw].
// Args: Gatv2AggArgs or TransformerAggArgs (edge_dim, ldw)
template <int VEC, int NJ, typename Args>
__device__ __forceinline__ void gatv2_edge_proj(const Args &a, const float *We, const float *ef,
                                                const AttnCols<NJ> &ln, Vec<VEC> (&z)[NJ])
{
    for (int j0 = 0; j0 < a.edge_dim; j0 += 4) {
        const float4 e4 = __ldg(reinterpret_cast<const float4 *>(ef + j0));
#pragma unroll
        for (int jj = 0; jj < 4; jj++) {
            if (j0 + jj < a.edge_dim) {
                const float ej = jj == 0 ? e4.x : jj == 1 ? e4.y : jj == 2 ? e4.z : e4.w;
                const float *wr = We + (size_t)(j0 + jj) * a.ldw;
#pragma unroll
                for (int j = 0; j < NJ; j++) {
                    if (!ln.valid[j]) continue;
#pragma unroll
                    for (int i = 0; i < VEC; i++) z[j].v[i] = fmaf(wr[ln.col[j] + i], ej, z[j].v[i]);
                }
            }
        }
    }
}

// the lane's partial dot product <att, LeakyReLU(xl + xr + ep)> (columns past C hold att = 0)
template <int VEC, int NJ>
__device__ __forceinline__ float gatv2_partial(const Gatv2AggArgs &a, const Gatv2Lane<VEC, NJ> &ln,
                                               const Vec<VEC> (&xl)[NJ], const Vec<VEC> (&ep)[NJ])
{
    float part = 0.0f;
#pragma unroll
    for (int j = 0; j < NJ; j++)
#pragma unroll
        for (int i = 0; i < VEC; i++)
            part = fmaf(ln.att[j].v[i], leaky_relu(xl[j].v[i] + ln.xr[j].v[i] + ep[j].v[i], a.slope), part);
    return part;
}

__device__ __forceinline__ float gatv2_head_sum(float part, unsigned mask, int G)
{
    for (int o = G >> 1; o > 0; o >>= 1) part += __shfl_xor_sync(mask, part, o);
    return part;
}

template <int VEC, int NJ>
__device__ __forceinline__ void gatv2_zero(Vec<VEC> (&x)[NJ])
{
#pragma unroll
    for (int j = 0; j < NJ; j++)
#pragma unroll
        for (int i = 0; i < VEC; i++) x[j].v[i] = 0.0f;
}

// the self term of row v: logit from xl_v + xr_v (+ self_attr_v W_e^T), weight 1, message xl_v
template <int VEC, int NJ, bool EDGE>
__device__ __forceinline__ void gatv2_self(const Gatv2AggArgs &a, const float *We, int v,
                                           const Gatv2Lane<VEC, NJ> &ln, unsigned mask, int G,
                                           OnlineSoftmax<VEC, NJ> &st)
{
    Vec<VEC> ep[NJ];
    gatv2_load<VEC, NJ>(a.g + (size_t)v * a.ldg, ln, st.acc);
    gatv2_zero<VEC, NJ>(ep);
    if (EDGE) gatv2_edge_proj<VEC, NJ>(a, We, a.self_attr + (size_t)v * a.lde, ln, ep);
    st.m = gatv2_head_sum(gatv2_partial<VEC, NJ>(a, ln, st.acc, ep), mask, G);
    st.s = 1.0f;
}

// neighbor slots [k0, k1) of row v (entries equal to v skipped, uniformly over the sub-warp), U
// gathers in flight
template <int VEC, int NJ, bool EDGE>
__device__ __forceinline__ void gatv2_gather(const Gatv2AggArgs &a, const float *We, int v, int off,
                                             int k0, int k1, const Gatv2Lane<VEC, NJ> &ln,
                                             unsigned mask, int G, OnlineSoftmax<VEC, NJ> &st)
{
    constexpr int U = NJ == 1 ? 4 : 2;
    int k = k0;
#pragma unroll 1
    for (; k + U <= k1; k += U) {
        int u[U];
        Vec<VEC> xl[U][NJ], ep[U][NJ];
        float e[U];
#pragma unroll
        for (int q = 0; q < U; q++) u[q] = __ldg(a.nbr + off + k + q);
#pragma unroll
        for (int q = 0; q < U; q++) gatv2_load<VEC, NJ>(a.g + (size_t)u[q] * a.ldg, ln, xl[q]);
#pragma unroll
        for (int q = 0; q < U; q++) {
            gatv2_zero<VEC, NJ>(ep[q]);
            if (EDGE) gatv2_edge_proj<VEC, NJ>(a, We, a.ef_sorted + (size_t)(off + k + q) * a.lde, ln, ep[q]);
            e[q] = gatv2_partial<VEC, NJ>(a, ln, xl[q], ep[q]);
        }
        for (int o = G >> 1; o > 0; o >>= 1)
#pragma unroll
            for (int q = 0; q < U; q++) e[q] += __shfl_xor_sync(mask, e[q], o);
#pragma unroll
        for (int q = 0; q < U; q++)
            if (u[q] != v) st.merge(e[q], 1.0f, xl[q]);
    }
#pragma unroll 1
    for (; k < k1; k++) {
        const int u = __ldg(a.nbr + off + k);
        if (u == v) continue;
        Vec<VEC> xl[NJ], ep[NJ];
        gatv2_load<VEC, NJ>(a.g + (size_t)u * a.ldg, ln, xl);
        gatv2_zero<VEC, NJ>(ep);
        if (EDGE) gatv2_edge_proj<VEC, NJ>(a, We, a.ef_sorted + (size_t)(off + k) * a.lde, ln, ep);
        st.merge(gatv2_head_sum(gatv2_partial<VEC, NJ>(a, ln, xl, ep), mask, G), 1.0f, xl);
    }
}

// the epilogue of the lane's valid column groups (none in an idle group)
template <int VEC, int NJ>
__device__ __forceinline__ void gatv2_finish(const Gatv2AggArgs &a, int v, const Gatv2Lane<VEC, NJ> &ln,
                                             const OnlineSoftmax<VEC, NJ> &st)
{
#pragma unroll
    for (int j = 0; j < NJ; j++)
        if (ln.valid[j]) attn_finish(a, v, ln.col[j], st.acc[j], st.s);
}

// W_e^T staged in shared memory (w_smem) or read in place; Args as gatv2_edge_proj
template <typename Args>
__device__ __forceinline__ const float *gatv2_stage_we(const Args &a, bool w_smem)
{
    extern __shared__ float4 gatv2_smem4[];
    if (!w_smem) return a.We_t;
    float *sw = reinterpret_cast<float *>(gatv2_smem4);
    const int nw = a.edge_dim * a.ldw;
    for (int i = threadIdx.x; i < nw; i += blockDim.x) sw[i] = __ldg(a.We_t + i);
    __syncthreads();
    return sw;
}

// lpr lanes per destination row (a power of two, a multiple of G); G lanes per head
template <int VEC, int NJ, bool EDGE, bool XR>
__global__ void __launch_bounds__(256, 1) gatv2_agg_kernel(const Gatv2AggArgs a, int lpr, int G, bool w_smem)
{
    const float *We = EDGE ? gatv2_stage_we(a, w_smem) : nullptr;
    const int rows_per_warp = 32 / lpr;
    const int lane = threadIdx.x & 31;
    const int lg = lane % lpr, sub = lane / lpr;
    const unsigned mask = lpr == 32 ? 0xffffffffu : ((1u << lpr) - 1u) << (sub * lpr);
    const int grp = lg / G, hl = lg % G, heads_per_pass = lpr / G;
    const int warps_per_block = blockDim.x >> 5;
    const int64_t warp_global = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int64_t warp_stride = (int64_t)gridDim.x * warps_per_block;
    for (int64_t row0 = warp_global * rows_per_warp; row0 < a.n; row0 += warp_stride * rows_per_warp) {
        // everything below is uniform over the row's sub-warp, so all its lanes reach every shuffle
        const int v = (int)row0 + sub;
        if (v >= a.n) continue;
        const int deg = __ldg(a.in_deg + v);
        if (a.heavy.n > 0 && deg > a.heavy.threshold) continue;  // the heavy-row kernels do these
        const int off = __ldg(a.offsets + v);
        for (int h0 = 0; h0 < a.H; h0 += heads_per_pass) {
            const Gatv2Lane<VEC, NJ> ln = gatv2_lane<VEC, NJ, XR>(a, v, h0 + grp, hl, G);
            OnlineSoftmax<VEC, NJ> st;
            gatv2_self<VEC, NJ, EDGE>(a, We, v, ln, mask, G, st);
            gatv2_gather<VEC, NJ, EDGE>(a, We, v, off, 0, deg, ln, mask, G, st);
            gatv2_finish<VEC, NJ>(a, v, ln, st);
        }
    }
}

// one warp per kHeavyChunk-neighbor chunk of a heavy row: the chunk's per-head (m, s) and its
// accumulator, as GAT's chunk kernel
template <int VEC, int NJ, bool EDGE, bool XR>
__global__ void __launch_bounds__(256, 1) gatv2_heavy_chunk_kernel(const Gatv2AggArgs a, int G)
{
    const int lane = threadIdx.x & 31;
    const int grp = lane / G, hl = lane % G, heads_per_pass = 32 / G;
    const int warps_per_block = blockDim.x >> 5;
    const int warp_global = blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int warp_stride = gridDim.x * warps_per_block;
    for (int chunk = warp_global; chunk < a.heavy.chunks; chunk += warp_stride) {
        const int h = __ldg(a.heavy.chunk_row + chunk);
        const int v = __ldg(a.heavy.rows + h);
        const int j = chunk - __ldg(a.heavy.chunk_base + h);
        const int deg = __ldg(a.in_deg + v);
        const int off = __ldg(a.offsets + v);
        const int k0 = j * kHeavyChunk, k1 = min(deg, k0 + kHeavyChunk);
        float *dst = a.heavy.partial + (size_t)chunk * a.ldp;
        for (int h0 = 0; h0 < a.H; h0 += heads_per_pass) {
            const Gatv2Lane<VEC, NJ> ln = gatv2_lane<VEC, NJ, XR>(a, v, h0 + grp, hl, G);
            OnlineSoftmax<VEC, NJ> st;
            st.reset();
            gatv2_gather<VEC, NJ, EDGE>(a, a.We_t, v, off, k0, k1, ln, 0xffffffffu, G, st);
            attn_store_partial<VEC, NJ>(a, dst, ln, hl == 0 && ln.hd < a.H, st);
        }
    }
}

// one CTA per heavy row: combine steps 1 and 2 (GAT's), warp 0 starting from the self term
template <int VEC, int NJ, bool EDGE, bool XR>
__global__ void __launch_bounds__(256, 1) gatv2_heavy_combine_kernel(const Gatv2AggArgs a, int G)
{
    extern __shared__ float4 gatv2_comb_smem4[];
    float *const ranges = reinterpret_cast<float *>(gatv2_comb_smem4);   // [8][ldp], as the partials
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int grp = lane / G, hl = lane % G, heads_per_pass = 32 / G;
    for (int h = blockIdx.x; h < a.heavy.n; h += gridDim.x) {
        const int v = attn_combine_chunks<VEC>(a, h, ranges);
        __syncthreads();
        if (warp == 0) {
            for (int h0 = 0; h0 < a.H; h0 += heads_per_pass) {
                const Gatv2Lane<VEC, NJ> ln = gatv2_lane<VEC, NJ, XR>(a, v, h0 + grp, hl, G);
                OnlineSoftmax<VEC, NJ> st;
                gatv2_self<VEC, NJ, EDGE>(a, a.We_t, v, ln, 0xffffffffu, G, st);
                attn_merge_ranges<VEC, NJ>(a, ranges, ln, ln.hd < a.H ? ln.hd : 0, st);
                gatv2_finish<VEC, NJ>(a, v, ln, st);
            }
        }
        __syncthreads();
    }
}

template <int VEC, int NJ, bool EDGE, bool XR = false>
int launch_gatv2_variant(const Gatv2AggArgs &a, int lpr, int G, size_t smem, cudaStream_t s, int *launches)
{
    auto k = gatv2_agg_kernel<VEC, NJ, EDGE, XR>;
    if (smem > 48 * 1024) GNNB_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<row_grid(a.n, lpr), 256, smem, s>>>(a, lpr, G, smem > 0);
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    if (a.heavy.n == 0) return GNNB_OK;
    return launch_attn_heavy(gatv2_heavy_chunk_kernel<VEC, NJ, EDGE, XR>,
                             gatv2_heavy_combine_kernel<VEC, NJ, EDGE, XR>, a, s, launches, G);
}

__global__ void gatv2_self_attr_kernel(const float *__restrict__ ef, int lde, int edge_dim,
                                       const int32_t *__restrict__ offsets,
                                       const int32_t *__restrict__ nbr,
                                       const int32_t *__restrict__ in_deg, int n,
                                       float *__restrict__ self_attr)
{
    const int64_t total = (int64_t)n * lde;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (int64_t)gridDim.x * blockDim.x) {
        const int v = (int)(t / lde), j = (int)(t - (int64_t)v * lde);
        float sum = 0.0f;
        int cnt = 0;
        if (j < edge_dim) {
            const int off = __ldg(offsets + v), deg = __ldg(in_deg + v);
            for (int k = 0; k < deg; k++) {
                if (__ldg(nbr + off + k) == v) continue;
                sum += __ldg(ef + (size_t)(off + k) * lde + j);
                cnt++;
            }
        }
        self_attr[t] = cnt > 0 ? sum / (float)cnt : 0.0f;
    }
}

}  // namespace

int launch_gatv2_agg(const Gatv2AggArgs &args, cudaStream_t s, int *launches)
{
    if (args.n <= 0) return GNNB_OK;
    Gatv2AggArgs a = args;
    const int HC = a.H * a.C;
    GNNB_TRY(check_attn_args(a, "gatv2"));
    const bool sep = a.xr != nullptr;   // xr through its own pointer: the XR kernels
    if (!sep) {
        GNNB_REQUIRE(a.ldg >= 2 * HC, "gatv2 aggregation: bad arguments");
        a.xr = a.g + HC;
        a.ldxr = a.ldg;
    }
    GNNB_REQUIRE(a.ldg >= HC && a.ldxr >= HC && a.att != nullptr, "gatv2 aggregation: bad arguments");
    const bool edge = a.ef_sorted != nullptr;
    if (edge)
        GNNB_REQUIRE(a.self_attr != nullptr && a.We_t != nullptr && a.edge_dim >= 1 &&
                         a.edge_dim <= kGineMaxEdgeDim && a.lde % 4 == 0 && a.lde >= a.edge_dim &&
                         a.ldw % 4 == 0 && a.ldw >= HC && aligned16(a.ef_sorted) && aligned16(a.self_attr),
                     "gatv2 aggregation: bad edge features");
    GNNB_REQUIRE(!(edge && sep), "gatv2 aggregation: a separate xr is taken without edge features only");
    const bool v4 = attn_v4(a) && aligned16(a.att) && a.ldxr % 4 == 0 && aligned16(a.xr) &&
                    (!edge || aligned16(a.We_t));
    const int vec = v4 ? 4 : 1;
    const int cg = (a.C + vec - 1) / vec;   // VEC-column groups per head
    int G = 1;
    while (G < 32 && G < cg) G *= 2;
    const int nj = (cg + G - 1) / G;
    GNNB_REQUIRE(nj <= 2, "gatv2 aggregation: head width C = " + std::to_string(a.C) +
                              " exceeds the lanes of a warp (at most " +
                              std::to_string(kGatv2MaxHeadWidth) + " with C % 4 == 0, else " +
                              std::to_string(kGatv2MaxHeadWidth1) + ")");
    int lpr = G;
    while (lpr < 32 && lpr < G * a.H) lpr *= 2;
    // W_e^T in shared memory when it fits (edge_dim 64 at H*C = 256: 64 KB), as the GINE aggregation
    const size_t w_bytes = edge ? sizeof(float) * (size_t)a.edge_dim * a.ldw : 0;
    const size_t smem = w_bytes <= 200 * 1024 ? w_bytes : 0;
    if (vec == 4) {
        if (nj == 1)
            return edge ? launch_gatv2_variant<4, 1, true>(a, lpr, G, smem, s, launches)
                        : sep ? launch_gatv2_variant<4, 1, false, true>(a, lpr, G, 0, s, launches)
              : launch_gatv2_variant<4, 1, false>(a, lpr, G, 0, s, launches);
        return edge ? launch_gatv2_variant<4, 2, true>(a, lpr, G, smem, s, launches)
                    : sep ? launch_gatv2_variant<4, 2, false, true>(a, lpr, G, 0, s, launches)
              : launch_gatv2_variant<4, 2, false>(a, lpr, G, 0, s, launches);
    }
    if (nj == 1)
        return edge ? launch_gatv2_variant<1, 1, true>(a, lpr, G, smem, s, launches)
                    : sep ? launch_gatv2_variant<1, 1, false, true>(a, lpr, G, 0, s, launches)
              : launch_gatv2_variant<1, 1, false>(a, lpr, G, 0, s, launches);
    return edge ? launch_gatv2_variant<1, 2, true>(a, lpr, G, smem, s, launches)
                : sep ? launch_gatv2_variant<1, 2, false, true>(a, lpr, G, 0, s, launches)
              : launch_gatv2_variant<1, 2, false>(a, lpr, G, 0, s, launches);
}

int launch_gatv2_self_attr(const float *ef_sorted, int lde, int edge_dim, const int32_t *offsets,
                           const int32_t *nbr, const int32_t *in_deg, int n, float *self_attr,
                           cudaStream_t s, int *launches)
{
    if (n <= 0) return GNNB_OK;
    const int64_t grid64 = ceil_div64((int64_t)n * lde, 256);
    const int64_t cap = (int64_t)kNumSMs * 16;
    gatv2_self_attr_kernel<<<(int)(grid64 < cap ? grid64 : cap), 256, 0, s>>>(
        ef_sorted, lde, edge_dim, offsets, nbr, in_deg, n, self_attr);
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    return GNNB_OK;
}

// ----------------------------------------------------------------------------- TransformerConv
//
// PyG TransformerConv (concat heads, root_weight, no beta, inference).  The layer's GEMMs wrote
// [k | v] per row into g and q (scaled by 1/sqrt(C) at finalize) into its own rows; the root term
// r = x W_skip^T (+ the model's residual) comes in as the epilogue's skip and b_skip as its bias.
// The logit e_uvh = <q_v, k_u (+ ê_uv)>_h is a dot product over the head's lanes, formed per edge as
// GATv2's: each lane holds q_v for its columns in registers and the head's lanes add their partials
// with the xor butterfly, so every lane of a head holds the same logit bits.  With edge features
// ê_uv = ef_sorted[slot] W_e^T is computed once per slot (gatv2_edge_proj) and added to both k_u and
// the message v_u.  Lane layout, masks and the W_e^T staging are GATv2's.
//
// There is no self term: every neighbor entry, the input's self loops and duplicates included, is an
// ordinary edge, and the online softmax starts from reset().  A row with no in-edges ends with s = 0
// and acc = 0; its epilogue divides by 1 instead, so y_v = act(b_skip + r_v).  Heavy rows are GAT's
// chunk / fixed-order combine scheme, warp 0 of the combine also starting from reset().  Algorithmic
// bytes per layer: E (4 + 8HC [+ 4 lde]) + N (8 + 4HC q + 4HC r + 4HC out).
namespace {

// one lane's share of one head: its columns (AttnCols) and q_v for them
template <int VEC, int NJ>
struct TransformerLane : AttnCols<NJ> {
    Vec<VEC> q[NJ];
};

template <int VEC, int NJ>
__device__ __forceinline__ TransformerLane<VEC, NJ> transformer_lane(const TransformerAggArgs &a, int v, int hd,
                                                                     int hl, int G)
{
    TransformerLane<VEC, NJ> ln;
    attn_lane_cols<VEC, NJ>(a, hd, hl, G, ln);
    gatv2_load<VEC, NJ>(a.q + (size_t)v * a.ldq, ln, ln.q);
    return ln;
}

// the lane's partial dot product <q_v, k> (columns past C hold q = 0)
template <int VEC, int NJ>
__device__ __forceinline__ float transformer_partial(const TransformerLane<VEC, NJ> &ln, const Vec<VEC> (&k)[NJ])
{
    float part = 0.0f;
#pragma unroll
    for (int j = 0; j < NJ; j++)
#pragma unroll
        for (int i = 0; i < VEC; i++) part = fmaf(ln.q[j].v[i], k[j].v[i], part);
    return part;
}

// k_u and v_u of one slot for the lane's columns, both plus ê = ef_sorted[slot] W_e^T with EDGE
template <int VEC, int NJ, bool EDGE>
__device__ __forceinline__ void transformer_load(const TransformerAggArgs &a, const float *We, int u, int slot,
                                                 const AttnCols<NJ> &cl, Vec<VEC> (&k)[NJ], Vec<VEC> (&val)[NJ])
{
    const float *row = a.g + (size_t)u * a.ldg;
    gatv2_load<VEC, NJ>(row, cl, k);
    gatv2_load<VEC, NJ>(row + a.H * a.C, cl, val);
    if (EDGE) {
        Vec<VEC> ep[NJ];
        gatv2_zero<VEC, NJ>(ep);
        gatv2_edge_proj<VEC, NJ>(a, We, a.ef_sorted + (size_t)slot * a.lde, cl, ep);
#pragma unroll
        for (int j = 0; j < NJ; j++)
#pragma unroll
            for (int i = 0; i < VEC; i++) {
                k[j].v[i] += ep[j].v[i];
                val[j].v[i] += ep[j].v[i];
            }
    }
}

// neighbor slots [k0, k1) of a row (none skipped), U gathers in flight
template <int VEC, int NJ, bool EDGE>
__device__ __forceinline__ void transformer_gather(const TransformerAggArgs &a, const float *We, int off, int k0,
                                                   int k1, const TransformerLane<VEC, NJ> &ln, unsigned mask,
                                                   int G, OnlineSoftmax<VEC, NJ> &st)
{
    constexpr int U = NJ == 1 ? 4 : 2;
    int k = k0;
#pragma unroll 1
    for (; k + U <= k1; k += U) {
        int u[U];
        Vec<VEC> kk[U][NJ], val[U][NJ];
        float e[U];
#pragma unroll
        for (int q = 0; q < U; q++) u[q] = __ldg(a.nbr + off + k + q);
#pragma unroll
        for (int q = 0; q < U; q++) {
            transformer_load<VEC, NJ, EDGE>(a, We, u[q], off + k + q, ln, kk[q], val[q]);
            e[q] = transformer_partial<VEC, NJ>(ln, kk[q]);
        }
        for (int o = G >> 1; o > 0; o >>= 1)
#pragma unroll
            for (int q = 0; q < U; q++) e[q] += __shfl_xor_sync(mask, e[q], o);
#pragma unroll
        for (int q = 0; q < U; q++) st.merge(e[q], 1.0f, val[q]);
    }
#pragma unroll 1
    for (; k < k1; k++) {
        Vec<VEC> kk[NJ], val[NJ];
        transformer_load<VEC, NJ, EDGE>(a, We, __ldg(a.nbr + off + k), off + k, ln, kk, val);
        st.merge(gatv2_head_sum(transformer_partial<VEC, NJ>(ln, kk), mask, G), 1.0f, val);
    }
}

// the epilogue of the lane's valid column groups; a row without in-edges (s = 0, acc = 0) divides by 1
template <int VEC, int NJ>
__device__ __forceinline__ void transformer_finish(const TransformerAggArgs &a, int v, const AttnCols<NJ> &cl,
                                                   const OnlineSoftmax<VEC, NJ> &st)
{
    const float s = st.s == 0.0f ? 1.0f : st.s;
#pragma unroll
    for (int j = 0; j < NJ; j++)
        if (cl.valid[j]) attn_finish(a, v, cl.col[j], st.acc[j], s);
}

// lpr lanes per destination row (a power of two, a multiple of G); G lanes per head
template <int VEC, int NJ, bool EDGE>
__global__ void __launch_bounds__(256, 1) transformer_agg_kernel(const TransformerAggArgs a, int lpr, int G,
                                                                 bool w_smem)
{
    const float *We = EDGE ? gatv2_stage_we(a, w_smem) : nullptr;
    const int rows_per_warp = 32 / lpr;
    const int lane = threadIdx.x & 31;
    const int lg = lane % lpr, sub = lane / lpr;
    const unsigned mask = lpr == 32 ? 0xffffffffu : ((1u << lpr) - 1u) << (sub * lpr);
    const int grp = lg / G, hl = lg % G, heads_per_pass = lpr / G;
    const int warps_per_block = blockDim.x >> 5;
    const int64_t warp_global = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int64_t warp_stride = (int64_t)gridDim.x * warps_per_block;
    for (int64_t row0 = warp_global * rows_per_warp; row0 < a.n; row0 += warp_stride * rows_per_warp) {
        // everything below is uniform over the row's sub-warp, so all its lanes reach every shuffle
        const int v = (int)row0 + sub;
        if (v >= a.n) continue;
        const int deg = __ldg(a.in_deg + v);
        if (a.heavy.n > 0 && deg > a.heavy.threshold) continue;  // the heavy-row kernels do these
        const int off = __ldg(a.offsets + v);
        for (int h0 = 0; h0 < a.H; h0 += heads_per_pass) {
            const TransformerLane<VEC, NJ> ln = transformer_lane<VEC, NJ>(a, v, h0 + grp, hl, G);
            OnlineSoftmax<VEC, NJ> st;
            st.reset();
            transformer_gather<VEC, NJ, EDGE>(a, We, off, 0, deg, ln, mask, G, st);
            transformer_finish<VEC, NJ>(a, v, ln, st);
        }
    }
}

// one warp per kHeavyChunk-neighbor chunk of a heavy row: the chunk's per-head (m, s) and accumulator
template <int VEC, int NJ, bool EDGE>
__global__ void __launch_bounds__(256, 1) transformer_heavy_chunk_kernel(const TransformerAggArgs a, int G)
{
    const int lane = threadIdx.x & 31;
    const int grp = lane / G, hl = lane % G, heads_per_pass = 32 / G;
    const int warps_per_block = blockDim.x >> 5;
    const int warp_global = blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int warp_stride = gridDim.x * warps_per_block;
    for (int chunk = warp_global; chunk < a.heavy.chunks; chunk += warp_stride) {
        const int h = __ldg(a.heavy.chunk_row + chunk);
        const int v = __ldg(a.heavy.rows + h);
        const int j = chunk - __ldg(a.heavy.chunk_base + h);
        const int deg = __ldg(a.in_deg + v);
        const int off = __ldg(a.offsets + v);
        const int k0 = j * kHeavyChunk, k1 = min(deg, k0 + kHeavyChunk);
        float *dst = a.heavy.partial + (size_t)chunk * a.ldp;
        for (int h0 = 0; h0 < a.H; h0 += heads_per_pass) {
            const TransformerLane<VEC, NJ> ln = transformer_lane<VEC, NJ>(a, v, h0 + grp, hl, G);
            OnlineSoftmax<VEC, NJ> st;
            st.reset();
            transformer_gather<VEC, NJ, EDGE>(a, a.We_t, off, k0, k1, ln, 0xffffffffu, G, st);
            attn_store_partial<VEC, NJ>(a, dst, ln, hl == 0 && ln.hd < a.H, st);
        }
    }
}

// one CTA per heavy row: combine steps 1 and 2, warp 0 starting from reset() (there is no self term)
template <int VEC, int NJ>
__global__ void __launch_bounds__(256, 1) transformer_heavy_combine_kernel(const TransformerAggArgs a, int G)
{
    extern __shared__ float4 transformer_comb_smem4[];
    float *const ranges = reinterpret_cast<float *>(transformer_comb_smem4);   // [8][ldp], as the partials
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int grp = lane / G, hl = lane % G, heads_per_pass = 32 / G;
    for (int h = blockIdx.x; h < a.heavy.n; h += gridDim.x) {
        const int v = attn_combine_chunks<VEC>(a, h, ranges);
        __syncthreads();
        if (warp == 0) {
            for (int h0 = 0; h0 < a.H; h0 += heads_per_pass) {
                AttnCols<NJ> cl;
                attn_lane_cols<VEC, NJ>(a, h0 + grp, hl, G, cl);
                OnlineSoftmax<VEC, NJ> st;
                st.reset();
                attn_merge_ranges<VEC, NJ>(a, ranges, cl, cl.hd < a.H ? cl.hd : 0, st);
                transformer_finish<VEC, NJ>(a, v, cl, st);
            }
        }
        __syncthreads();
    }
}

template <int VEC, int NJ, bool EDGE>
int launch_transformer_variant(const TransformerAggArgs &a, int lpr, int G, size_t smem, cudaStream_t s,
                               int *launches)
{
    auto k = transformer_agg_kernel<VEC, NJ, EDGE>;
    if (smem > 48 * 1024) GNNB_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<row_grid(a.n, lpr), 256, smem, s>>>(a, lpr, G, smem > 0);
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    if (a.heavy.n == 0) return GNNB_OK;
    return launch_attn_heavy(transformer_heavy_chunk_kernel<VEC, NJ, EDGE>,
                             transformer_heavy_combine_kernel<VEC, NJ>, a, s, launches, G);
}

template <int VEC, int NJ>
int launch_transformer_nj(const TransformerAggArgs &a, bool edge, int lpr, int G, size_t smem, cudaStream_t s,
                          int *launches)
{
    return edge ? launch_transformer_variant<VEC, NJ, true>(a, lpr, G, smem, s, launches)
                : launch_transformer_variant<VEC, NJ, false>(a, lpr, G, 0, s, launches);
}

}  // namespace

int launch_transformer_agg(const TransformerAggArgs &a, cudaStream_t s, int *launches)
{
    if (a.n <= 0) return GNNB_OK;
    const int HC = a.H * a.C;
    GNNB_TRY(check_attn_args(a, "transformer"));
    GNNB_REQUIRE(a.g != nullptr && a.ldg >= 2 * HC && a.q != nullptr && a.ldq >= HC,
                 "transformer aggregation: bad arguments");
    const bool edge = a.ef_sorted != nullptr;
    if (edge)
        GNNB_REQUIRE(a.We_t != nullptr && a.edge_dim >= 1 && a.edge_dim <= kGineMaxEdgeDim &&
                         a.lde % 4 == 0 && a.lde >= a.edge_dim && a.ldw % 4 == 0 && a.ldw >= HC &&
                         aligned16(a.ef_sorted),
                     "transformer aggregation: bad edge features");
    const bool v4 = attn_v4(a) && a.ldq % 4 == 0 && aligned16(a.q) && (!edge || aligned16(a.We_t));
    const int vec = v4 ? 4 : 1;
    const int cg = (a.C + vec - 1) / vec;   // VEC-column groups per head
    int G = 1;
    while (G < 32 && G < cg) G *= 2;
    const int nj = (cg + G - 1) / G;
    GNNB_REQUIRE(nj <= 2, "transformer aggregation: head width C = " + std::to_string(a.C) +
                              " exceeds the lanes of a warp (at most " +
                              std::to_string(kGatv2MaxHeadWidth) + " with C % 4 == 0, else " +
                              std::to_string(kGatv2MaxHeadWidth1) + ")");
    int lpr = G;
    while (lpr < 32 && lpr < G * a.H) lpr *= 2;
    // W_e^T in shared memory when it fits, as GATv2
    const size_t w_bytes = edge ? sizeof(float) * (size_t)a.edge_dim * a.ldw : 0;
    const size_t smem = w_bytes <= 200 * 1024 ? w_bytes : 0;
    if (vec == 4)
        return nj == 1 ? launch_transformer_nj<4, 1>(a, edge, lpr, G, smem, s, launches)
                       : launch_transformer_nj<4, 2>(a, edge, lpr, G, smem, s, launches);
    return nj == 1 ? launch_transformer_nj<1, 1>(a, edge, lpr, G, smem, s, launches)
                   : launch_transformer_nj<1, 2>(a, edge, lpr, G, smem, s, launches);
}

}  // namespace gnnb
