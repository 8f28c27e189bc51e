// Node transform: the `linear` of gnn_builder_lib.h:808-1003 batched over all rows (nodes or
// graphs) as one GEMM with the bias / skip-connection / activation of the generated top
// (model.cpp.jinja:304-322, 508-516) fused into the epilogue.
//
//   C[M][N] = act( A1[M][K1] . W1t[K1][N]  (+ A2[M][K2] . W2t[K2][N])  + bias  (+ skip) )
//
// FAST: register-tiled fp32 FMA kernel.  CTA tile 128 x BN (BN = 128/64/32), BK = 16, 256
// threads, 8 x (BN/16) outputs per thread, global->register prefetch of the next K tile while
// the current one is multiplied out of shared memory.  Every output element is accumulated in
// ONE thread in ascending k, starting from the bias -- the reference's order (lib:852-903) --
// so the only rounding difference is the fused multiply-add.
// STRICT: one thread per output, separately rounded multiply and add in the reference's exact
// order (bit-identical to the reference's `linear` compiled without FMA).
//
// Roofline: 2*M*N*K flops against the fp32 FMA pipe (148 SMs x 128 lanes x 2 x clk); the
// tensor-core (tcgen05, 3xTF32) variant of this node transform lives in fused.cu.
#include "kernels.h"

namespace gnnb {

namespace {

constexpr int BM = 128;
constexpr int BK = 16;
constexpr int LDAS = BM + 4;

struct TileSrc {
    const float *A; int lda; int K; const float *Wt; int ldw;
};

template <int BN>
struct Frag {
    static constexpr int TN = BN / 16;
};

// loads of one K tile into registers ------------------------------------------------------
template <int BN>
struct Prefetch {
    static constexpr int W_F4 = (BK * BN / 4) / 256 > 0 ? (BK * BN / 4) / 256 : 1;
    float a[8];
    float4 w[W_F4];
};

template <int BN>
__device__ __forceinline__ void load_tile(const TileSrc &t, int m0, int n0, int k0, int M,
                                          bool a_vec, Prefetch<BN> &p)
{
    const int tid = threadIdx.x;
    // A: thread -> rows (tid/4) and (tid/4 + 64), 4 consecutive k starting at (tid%4)*4
    const int kq = (tid & 3) * 4;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const int row = m0 + (tid >> 2) + h * 64;
        const int k = k0 + kq;
        if (row < M && a_vec && k + 3 < t.K) {
            const float4 v = __ldg(reinterpret_cast<const float4 *>(t.A + (size_t)row * t.lda + k));
            p.a[h * 4 + 0] = v.x; p.a[h * 4 + 1] = v.y; p.a[h * 4 + 2] = v.z; p.a[h * 4 + 3] = v.w;
        } else {
#pragma unroll
            for (int i = 0; i < 4; i++)
                p.a[h * 4 + i] = (row < M && k + i < t.K) ? __ldg(t.A + (size_t)row * t.lda + k + i)
                                                           : 0.0f;
        }
    }
    // W: BK x BN floats, float4 granules; granule g -> k = g / (BN/4), col = (g % (BN/4)) * 4
    constexpr int GPR = BN / 4;
#pragma unroll
    for (int j = 0; j < Prefetch<BN>::W_F4; j++) {
        const int g = tid + j * 256;
        const int k = k0 + g / GPR;
        const int col = n0 + (g % GPR) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (g < BK * GPR && k < t.K && col < t.ldw)
            v = __ldg(reinterpret_cast<const float4 *>(t.Wt + (size_t)k * t.ldw + col));
        p.w[j] = v;
    }
}

template <int BN>
__device__ __forceinline__ void store_tile(const Prefetch<BN> &p, float *As, float *Ws)
{
    const int tid = threadIdx.x;
    const int kq = (tid & 3) * 4;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const int r = (tid >> 2) + h * 64;
#pragma unroll
        for (int i = 0; i < 4; i++) As[(kq + i) * LDAS + r] = p.a[h * 4 + i];
    }
    constexpr int GPR = BN / 4;
#pragma unroll
    for (int j = 0; j < Prefetch<BN>::W_F4; j++) {
        const int g = tid + j * 256;
        if (g < BK * GPR)
            *reinterpret_cast<float4 *>(Ws + (g / GPR) * BN + (g % GPR) * 4) = p.w[j];
    }
}

// The instruction footprint matters: a first version that fully unrolled both operand loops and
// inlined the 13-way activation switch 64 times was 85 KB of SASS and spent half its issue slots
// stalled on instruction fetch (ncu: stalled_no_instructions, profiles/r1_gemm_v1.txt).  This one
// keeps a single K-tile loop (operand pointers selected per tile) whose body is 16 k-steps.
template <int BN>
__global__ void __launch_bounds__(256, BN == 128 ? 1 : 2) gemm_fma_kernel(const GemmArgs g)
{
    constexpr int TN = Frag<BN>::TN;   // 8, 4 or 2 columns per thread
    constexpr int CW = TN >= 4 ? 4 : TN;  // contiguous column group width
    constexpr int NG = TN / CW;           // number of column groups (2 for BN=128)
    __shared__ __align__(16) float As[BK * LDAS];
    __shared__ __align__(16) float Ws[BK * BN];

    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;

    float acc[8][TN];
#pragma unroll
    for (int j = 0; j < TN; j++) {
        const int col = n0 + (j / CW) * (BN / NG) + tx * CW + (j % CW);
        const float b = (g.bias != nullptr && col < g.N) ? __ldg(g.bias + col) : 0.0f;
#pragma unroll
        for (int i = 0; i < 8; i++) acc[i][j] = b;
    }

    const int nt1 = (g.K1 + BK - 1) / BK;
    const int nt2 = (g.A2 != nullptr && g.K2 > 0) ? (g.K2 + BK - 1) / BK : 0;
    const int nt = nt1 + nt2;
    const bool a1_vec = (g.lda1 % 4 == 0) && ((reinterpret_cast<uintptr_t>(g.A1) & 15) == 0);
    const bool a2_vec = nt2 > 0 && (g.lda2 % 4 == 0) && ((reinterpret_cast<uintptr_t>(g.A2) & 15) == 0);
    auto tile_src = [&](int t, TileSrc &src, int &k0, bool &vec) {
        if (t < nt1) {
            src = TileSrc{g.A1, g.lda1, g.K1, g.W1t, g.ldw1};
            k0 = t * BK;
            vec = a1_vec;
        } else {
            src = TileSrc{g.A2, g.lda2, g.K2, g.W2t, g.ldw2};
            k0 = (t - nt1) * BK;
            vec = a2_vec;
        }
    };

    Prefetch<BN> pf;
    {
        TileSrc src; int k0; bool vec;
        tile_src(0, src, k0, vec);
        load_tile<BN>(src, m0, n0, k0, g.M, vec, pf);
    }
#pragma unroll 1
    for (int t = 0; t < nt; t++) {
        __syncthreads();  // previous tile fully consumed
        store_tile<BN>(pf, As, Ws);
        __syncthreads();
        if (t + 1 < nt) {
            TileSrc src; int k0; bool vec;
            tile_src(t + 1, src, k0, vec);
            load_tile<BN>(src, m0, n0, k0, g.M, vec, pf);
        }
#pragma unroll
        for (int k = 0; k < BK; k++) {
            float a[8], b[TN];
            const float4 a0 = *reinterpret_cast<const float4 *>(As + k * LDAS + ty * 4);
            const float4 a1 = *reinterpret_cast<const float4 *>(As + k * LDAS + 64 + ty * 4);
            a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w;
            a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
#pragma unroll
            for (int q = 0; q < NG; q++) {
                const float *wp = Ws + k * BN + q * (BN / NG) + tx * CW;
                if constexpr (CW == 4) {
                    const float4 w = *reinterpret_cast<const float4 *>(wp);
                    b[q * 4 + 0] = w.x; b[q * 4 + 1] = w.y; b[q * 4 + 2] = w.z; b[q * 4 + 3] = w.w;
                } else {
                    const float2 w = *reinterpret_cast<const float2 *>(wp);
                    b[0] = w.x; b[1] = w.y;
                }
            }
#pragma unroll
            for (int i = 0; i < 8; i++)
#pragma unroll
                for (int j = 0; j < TN; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
    }

    // epilogue: (+ skip) -> activation -> store.  ReLU / identity inline, the transcendental
    // activations through one out-of-line call so the code stays small.
    const bool vec_ok = (g.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(g.C) & 15) == 0);
#pragma unroll 1
    for (int i = 0; i < 8; i++) {
        const int row = m0 + (i / 4) * 64 + ty * 4 + (i % 4);
        if (row >= g.M) continue;
#pragma unroll
        for (int q = 0; q < NG; q++) {
            const int col = n0 + q * (BN / NG) + tx * CW;
            float v[CW];
#pragma unroll
            for (int j = 0; j < CW; j++) {
                float t = 0.0f;
#pragma unroll
                for (int ii = 0; ii < 8; ii++)   // register select without dynamic indexing
                    if (ii == i) t = acc[ii][q * CW + j];
                if (g.skip != nullptr && col + j < g.N)
                    t += __ldg(g.skip + (size_t)row * g.ldskip + col + j);
                v[j] = act_apply_compact(g.act, t);
            }
            float *dst = g.C + (size_t)row * g.ldc + col;
            bool vec_store = false;
            if constexpr (CW == 4) {
                vec_store = vec_ok && col + 3 < g.N;
                if (vec_store)
                    *reinterpret_cast<float4 *>(dst) = make_float4(v[0], v[1], v[2], v[3]);
            }
            if (!vec_store) {
#pragma unroll
                for (int j = 0; j < CW; j++)
                    if (col + j < g.N) dst[j] = v[j];
            }
        }
    }
}

// STRICT: reference operation order, no contraction.  lib:852-903 with BLOCK_SIZE_IN = 1:
// y = bias; y = y + (w * x) for ascending input index.  A second operand either continues the
// same running sum (PNA's 13F concat, lib:2149) or, for SAGE, is a separate bias-free linear
// added at the end (lib:2316-2332).
__global__ void __launch_bounds__(256) gemm_strict_kernel(const GemmArgs g, int second_separate)
{
    const int64_t total = (int64_t)g.M * g.N;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int row = (int)(idx / g.N), col = (int)(idx % g.N);
        float acc = g.bias ? __ldg(g.bias + col) : 0.0f;
        const float *a = g.A1 + (size_t)row * g.lda1;
        for (int k = 0; k < g.K1; k++)
            acc = __fadd_rn(acc, __fmul_rn(__ldg(g.W1t + (size_t)k * g.ldw1 + col), __ldg(a + k)));
        if (g.A2 != nullptr && g.K2 > 0) {
            const float *a2 = g.A2 + (size_t)row * g.lda2;
            float acc2 = second_separate ? 0.0f : acc;
            for (int k = 0; k < g.K2; k++)
                acc2 = __fadd_rn(acc2,
                                 __fmul_rn(__ldg(g.W2t + (size_t)k * g.ldw2 + col), __ldg(a2 + k)));
            acc = second_separate ? __fadd_rn(acc, acc2) : acc2;
        }
        if (g.skip) acc = __fadd_rn(__ldg(g.skip + (size_t)row * g.ldskip + col), acc);
        g.C[(size_t)row * g.ldc + col] = act_apply(g.act, acc);
    }
}

__global__ void transpose_weight_kernel(const float *__restrict__ W, float *__restrict__ Wt,
                                        int out_size, int in_size, int ldw, int ld_src)
{
    const int64_t total = (int64_t)in_size * ldw;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int k = (int)(idx / ldw), n = (int)(idx % ldw);
        Wt[idx] = (n < out_size) ? __ldg(W + (size_t)n * ld_src + k) : 0.0f;
    }
}

}  // namespace

int launch_gemm(const GemmArgs &g, bool strict, cudaStream_t s, int *launches)
{
    if (g.M <= 0 || g.N <= 0) return GNNB_OK;
    GNNB_REQUIRE(g.ldw1 % 4 == 0 && (g.A2 == nullptr || g.ldw2 % 4 == 0),
                 "gemm: packed weight stride must be a multiple of 4");
    if (strict) {
        const int64_t total = (int64_t)g.M * g.N;
        int64_t grid = ceil_div64(total, 256);
        const int64_t cap = (int64_t)kNumSMs * 32;
        if (grid > cap) grid = cap;
        gemm_strict_kernel<<<(int)grid, 256, 0, s>>>(g, g.second_separate);
        GNNB_CUDA(cudaGetLastError());
        if (launches) ++*launches;
        return GNNB_OK;
    }
    if (gemm_tc_supported(g)) return launch_gemm_tc(g, s, launches);
    GNNB_REQUIRE(g.expand_deg == nullptr, "gemm: expand mode needs the tensor-core path");
    const int mb = (g.M + BM - 1) / BM;
    if (g.N > 64) {
        dim3 grid(mb, (g.N + 127) / 128);
        gemm_fma_kernel<128><<<grid, 256, 0, s>>>(g);
    } else if (g.N > 32) {
        dim3 grid(mb, 1);
        gemm_fma_kernel<64><<<grid, 256, 0, s>>>(g);
    } else {
        dim3 grid(mb, 1);
        gemm_fma_kernel<32><<<grid, 256, 0, s>>>(g);
    }
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    return GNNB_OK;
}

int launch_transpose_weight(const float *W, float *Wt, int out_size, int in_size, int ldw,
                            cudaStream_t s, int *launches, int ld_src)
{
    const int64_t total = (int64_t)in_size * ldw;
    if (total <= 0) return GNNB_OK;
    int64_t grid = ceil_div64(total, 256);
    if (grid > kNumSMs * 8) grid = kNumSMs * 8;
    transpose_weight_kernel<<<(int)grid, 256, 0, s>>>(W, Wt, out_size, in_size, ldw,
                                                  ld_src > 0 ? ld_src : in_size);
    GNNB_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    return GNNB_OK;
}

}  // namespace gnnb
