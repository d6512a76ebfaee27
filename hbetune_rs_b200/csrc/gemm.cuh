// Tiled, batched, triangular-aware GEMM for the GP hot path (sm_100a).
//
// FP64 runs on the DMMA tensor pipe (mma.sync.m8n8k4.f64 -> SASS DMMA.8x8x4; there is no tcgen05 f64
// kind), FP32 (--use-32) on plain FFMA (TF32 would break the 1e-4 parity bound).  Operand tiles are
// staged global -> shared with 16-byte cp.async (LDGSTS) through a 3-stage ring; shared rows are padded
// so that the 8x4 DMMA fragment reads are bank-conflict free.
//
// One kernel serves every dense contraction of the path (potrf panel solve + trailing SYRK, triangular
// inverse merges, W^T W, and the predictive-variance product): C = alpha * A(.,k) B(.,k)^T + beta * C
// where each operand is either k-contiguous ("KMAJOR": X[i*ld + k]) or i-contiguous (X[k*ld + i]), the
// k range of a tile may be cut by the triangular structure of an operand (KMode), only the lower tiles of
// C may be produced, and the epilogue either stores C or emits per-row sums of squares.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>

#include "launch.h"

// k depth of one pipeline stage and number of stages (probes/gemm_bench.cu: 16 x 3 and 32 x 2 are within 0.5 %)
#ifndef HBEGP_BK
#define HBEGP_BK 16
#endif
#ifndef HBEGP_STAGES
#define HBEGP_STAGES 3
#endif

namespace hbegp {

enum KMode : int {
    K_FULL = 0,
    K_LE_N = 1,  // k in [0, n0 + BN)      (B lower-triangular, indexed [n][k])
    K_GE_N = 2,  // k in [n0, K)           (B lower-triangular, indexed [k][n])
    K_LE_M = 3,  // k in [0, m0 + BM)      (A lower-triangular, indexed [m][k])
    K_GE_M = 4,  // k in [m0, K)           (A lower-triangular, indexed [k][m])
};

template <typename T>
struct GemmArgs {
    const T* A;
    const T* B;
    T* C;
    long lda, ldb, ldc;
    long sA, sB, sC;  // batch strides in elements
    int M, N, K;
    int kmode;
    int lower_only;  // produce only tiles with m0 >= n0 (BM == BN)
    T alpha, beta;
    T* rowsumsq;  // if non-null: partial[(row) * ld_rs + tile_n] = sum_j acc(row, j)^2, C untouched
    long ld_rs, s_rs;
    // K_LE_N only: rasterise in groups of `raster_group` row tiles (all column tiles of a group before the
    // next group) so that the group's A rows stay in L2 while B streams; 0 = plain column-major order.
    int raster_group;
    // Host-side hint (unused by the kernel): run on 32x32 tiles when the 64x64 grid would have at most this many CTAs
    // (see launch_gemm); 0 = never.
    long small_ctas;
};

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

template <typename T, int BM, int BN, int WM, int WN, bool A_KMAJOR, bool B_KMAJOR, int BK_ = HBEGP_BK, int STAGES_ = HBEGP_STAGES>
struct GemmCfg {
    static constexpr int BK = BK_;
    static constexpr int PAD = 4;
    static constexpr int STAGES = STAGES_;
    static constexpr int WARPS_M = BM / WM, WARPS_N = BN / WN;
    static constexpr int THREADS = WARPS_M * WARPS_N * 32;
    static constexpr int VEC = 16 / sizeof(T);
    static constexpr int A_STRIDE = A_KMAJOR ? (BK + PAD) : (BM + PAD);
    static constexpr int B_STRIDE = B_KMAJOR ? (BK + PAD) : (BN + PAD);
    static constexpr int A_ELEMS = A_KMAJOR ? BM * A_STRIDE : BK * A_STRIDE;
    static constexpr int B_ELEMS = B_KMAJOR ? BN * B_STRIDE : BK * B_STRIDE;
    static constexpr int STAGE_ELEMS = A_ELEMS + B_ELEMS;
    static constexpr size_t SMEM_BYTES = (size_t)STAGES * STAGE_ELEMS * sizeof(T);
};

// Copies one operand tile (R rows of the tile dimension x BK of k) into shared memory.
template <typename T, int R, int BK, int STRIDE, bool KMAJOR, int THREADS>
__device__ __forceinline__ void load_tile(T* __restrict__ s, const T* __restrict__ g, long ld, int r0, int k0,
                                          int tid) {
    constexpr int VEC = 16 / sizeof(T);
    if (KMAJOR) {
        constexpr int CPR = BK / VEC;  // chunks per row
        constexpr int TOTAL = R * CPR;
#pragma unroll
        for (int c = tid; c < TOTAL; c += THREADS) {
            int row = c / CPR, cc = c % CPR;
            cp_async16(s + row * STRIDE + cc * VEC, g + (long)(r0 + row) * ld + k0 + cc * VEC);
        }
    } else {
        constexpr int CPR = R / VEC;
        constexpr int TOTAL = BK * CPR;
#pragma unroll
        for (int c = tid; c < TOTAL; c += THREADS) {
            int kk = c / CPR, cc = c % CPR;
            cp_async16(s + kk * STRIDE + cc * VEC, g + (long)(k0 + kk) * ld + r0 + cc * VEC);
        }
    }
}

template <typename T, int BM, int BN, int WM, int WN, bool A_KMAJOR, bool B_KMAJOR, int BK_ = HBEGP_BK, int STAGES_ = HBEGP_STAGES>
__global__ void __launch_bounds__(GemmCfg<T, BM, BN, WM, WN, A_KMAJOR, B_KMAJOR, BK_, STAGES_>::THREADS)
    gemm_kernel(const GemmArgs<T> p) {
    using Cfg = GemmCfg<T, BM, BN, WM, WN, A_KMAJOR, B_KMAJOR, BK_, STAGES_>;
    constexpr int BK = Cfg::BK, STAGES = Cfg::STAGES, THREADS = Cfg::THREADS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* smem = reinterpret_cast<T*>(smem_raw);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp / Cfg::WARPS_N, wn = warp % Cfg::WARPS_N;
    const int tiles_m = p.M / BM, tiles_n = p.N / BN;

    // ---- tile coordinates (heavy tiles first for the triangular k ranges)
    int mt, nt;
    {
        int t = blockIdx.x;
        if (p.lower_only) {
            // enumerate mt >= nt, row by row
            int r = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
            while ((long)(r + 1) * (r + 2) / 2 <= t) ++r;
            while ((long)r * (r + 1) / 2 > t) --r;
            mt = r;
            nt = t - r * (r + 1) / 2;
            if (p.kmode != K_GE_M) {  // SYRK-like: uniform work, keep order
            }
        } else if (p.kmode == K_LE_M) {
            mt = tiles_m - 1 - t / tiles_n;
            nt = t % tiles_n;
        } else if (p.kmode == K_LE_N && p.raster_group > 0) {
            const int per_group = p.raster_group * tiles_n;
            const int g = t / per_group, base = g * p.raster_group;
            const int gsize = min(p.raster_group, tiles_m - base);
            const int r = t - g * per_group;
            nt = tiles_n - 1 - r / gsize;
            mt = base + r % gsize;
        } else if (p.kmode == K_LE_N) {
            nt = tiles_n - 1 - t / tiles_m;
            mt = t % tiles_m;
        } else {
            nt = t / tiles_m;
            mt = t % tiles_m;
        }
    }
    const int m0 = mt * BM, n0 = nt * BN;
    int kbeg = 0, kend = p.K;
    if (p.kmode == K_LE_N) kend = min(p.K, n0 + BN);
    else if (p.kmode == K_GE_N) kbeg = n0;
    else if (p.kmode == K_LE_M) kend = min(p.K, m0 + BM);
    else if (p.kmode == K_GE_M) kbeg = m0;
    const int nk = (kend - kbeg) / BK;

    const T* gA = p.A + (long)blockIdx.z * p.sA;
    const T* gB = p.B + (long)blockIdx.z * p.sB;

    auto issue = [&](int kt) {
        T* sA = smem + (kt % STAGES) * Cfg::STAGE_ELEMS;
        T* sB = sA + Cfg::A_ELEMS;
        int k0 = kbeg + kt * BK;
        load_tile<T, BM, BK, Cfg::A_STRIDE, A_KMAJOR, THREADS>(sA, gA, p.lda, m0, k0, tid);
        load_tile<T, BN, BK, Cfg::B_STRIDE, B_KMAJOR, THREADS>(sB, gB, p.ldb, n0, k0, tid);
    };

    constexpr bool F64 = std::is_same<T, double>::value;
    constexpr int FM = WM / 8;               // f64: 8-row mma tiles; f32: rows per thread
    constexpr int FN = F64 ? WN / 8 : WN / 4;  // f64: 8-col mma tiles; f32: cols per thread
    constexpr int ACC = F64 ? 2 : 1;
    T acc[FM][FN][ACC];
#pragma unroll
    for (int i = 0; i < FM; i++)
#pragma unroll
        for (int j = 0; j < FN; j++)
#pragma unroll
            for (int e = 0; e < ACC; e++) acc[i][j][e] = T(0);

#pragma unroll
    for (int s = 0; s < STAGES - 1; s++) {
        if (s < nk) issue(s);
        cp_async_commit();
    }

    const int lr = lane >> 2, lc = lane & 3;
    // warp-tile-relative row of accumulator slot i / column of slot j (see the two micro-kernels below)
    auto row_of = [&](int i) { return (F64 || A_KMAJOR) ? i * 8 + lr : FM * lr + i; };
    auto col_of = [&](int j) { return F64 ? j * 8 + 2 * lc : (B_KMAJOR ? j * 4 + lc : FN * lc + j); };
    // Early-fragment main loop (f64): the barrier of iteration kt also publishes stage kt + 1, so the operand fragments
    // of the first k4 step of the next stage are fetched during this iteration and no shared-memory latency sits
    // between the barrier and the first DMMA.  Measured +2..6 % on B200 against a loop that loads every fragment after
    // the barrier (profiles/r01_gemm_early_probe.log).
    T a_n[FM], b_n[FN];
    auto load_frag = [&](const T* sA, const T* sB, int ks, T* a, T* b) {
        const int k = ks * 4 + lc;
#pragma unroll
        for (int i = 0; i < FM; i++) {
            int row = wm * WM + i * 8 + lr;
            a[i] = A_KMAJOR ? sA[row * Cfg::A_STRIDE + k] : sA[k * Cfg::A_STRIDE + row];
        }
#pragma unroll
        for (int j = 0; j < FN; j++) {
            int col = wn * WN + j * 8 + lr;
            b[j] = B_KMAJOR ? sB[col * Cfg::B_STRIDE + k] : sB[k * Cfg::B_STRIDE + col];
        }
    };
    if constexpr (F64) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        if (nk > 0) load_frag(smem, smem + Cfg::A_ELEMS, 0, a_n, b_n);
    }
    for (int kt = 0; kt < nk; kt++) {
        if constexpr (F64) cp_async_wait<(STAGES >= 3 ? STAGES - 3 : 0)>();
        else cp_async_wait<STAGES - 2>();
        __syncthreads();
        if (kt + STAGES - 1 < nk) issue(kt + STAGES - 1);
        cp_async_commit();
        const T* sA = smem + (kt % STAGES) * Cfg::STAGE_ELEMS;
        const T* sB = sA + Cfg::A_ELEMS;
        if constexpr (F64) {
#pragma unroll
            for (int ks = 0; ks < BK / 4; ks++) {
                T a[FM], b[FN];
                if (ks == 0) {
#pragma unroll
                    for (int i = 0; i < FM; i++) a[i] = a_n[i];
#pragma unroll
                    for (int j = 0; j < FN; j++) b[j] = b_n[j];
                } else {
                    load_frag(sA, sB, ks, a, b);
                }
#pragma unroll
                for (int i = 0; i < FM; i++)
#pragma unroll
                    for (int j = 0; j < FN; j++) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
            }
            if (kt + 1 < nk) {
                const T* nA = smem + ((kt + 1) % STAGES) * Cfg::STAGE_ELEMS;
                load_frag(nA, nA + Cfg::A_ELEMS, 0, a_n, b_n);
            }
        } else {
            // FP32 (FFMA): (WM/8) x (WN/4) outputs per thread — 4 x 8 for the 64x64 tile, 8 x 8 for 128x128 —
            // operands fetched four k at a time with 16-byte shared loads.  Thread-to-row/column mapping follows
            // the contiguous direction of the staged tile: k-major tiles give rows lr + 8 i / columns lc + 4 j,
            // row-major tiles give the contiguous groups FM lr + i / FN lc + j.
            static_assert(F64 || (FM % 4 == 0 && FN % 4 == 0), "f32 micro-kernel needs FM, FN multiples of 4");
#pragma unroll
            for (int k4 = 0; k4 < BK; k4 += 4) {
                float av[FM][4], bv[FN][4];
                if (A_KMAJOR) {
#pragma unroll
                    for (int i = 0; i < FM; i++) {
                        const float4 t = *reinterpret_cast<const float4*>(&sA[(wm * WM + i * 8 + lr) * Cfg::A_STRIDE + k4]);
                        av[i][0] = t.x; av[i][1] = t.y; av[i][2] = t.z; av[i][3] = t.w;
                    }
                } else {
#pragma unroll
                    for (int kk = 0; kk < 4; kk++)
#pragma unroll
                        for (int i4 = 0; i4 < FM; i4 += 4) {
                            const float4 t = *reinterpret_cast<const float4*>(&sA[(k4 + kk) * Cfg::A_STRIDE + wm * WM + FM * lr + i4]);
                            av[i4][kk] = t.x; av[i4 + 1][kk] = t.y; av[i4 + 2][kk] = t.z; av[i4 + 3][kk] = t.w;
                        }
                }
                if (B_KMAJOR) {
#pragma unroll
                    for (int j = 0; j < FN; j++) {
                        const float4 t = *reinterpret_cast<const float4*>(&sB[(wn * WN + j * 4 + lc) * Cfg::B_STRIDE + k4]);
                        bv[j][0] = t.x; bv[j][1] = t.y; bv[j][2] = t.z; bv[j][3] = t.w;
                    }
                } else {
#pragma unroll
                    for (int kk = 0; kk < 4; kk++)
#pragma unroll
                        for (int j4 = 0; j4 < FN; j4 += 4) {
                            const float4 t = *reinterpret_cast<const float4*>(&sB[(k4 + kk) * Cfg::B_STRIDE + wn * WN + FN * lc + j4]);
                            bv[j4][kk] = t.x; bv[j4 + 1][kk] = t.y; bv[j4 + 2][kk] = t.z; bv[j4 + 3][kk] = t.w;
                        }
                }
#pragma unroll
                for (int kk = 0; kk < 4; kk++)
#pragma unroll
                    for (int i = 0; i < FM; i++)
#pragma unroll
                        for (int j = 0; j < FN; j++) acc[i][j][0] = fmaf(av[i][kk], bv[j][kk], acc[i][j][0]);
            }
        }
    }
    cp_async_wait<0>();

    // ---- epilogue
    if (p.rowsumsq != nullptr) {
        __syncthreads();  // operand ring is dead: reuse it as the cross-warp reduction buffer
        T* red = smem;    // [BM][WARPS_N]
#pragma unroll
        for (int i = 0; i < FM; i++) {
            T s = T(0);
#pragma unroll
            for (int j = 0; j < FN; j++)
#pragma unroll
                for (int e = 0; e < ACC; e++) s += acc[i][j][e] * acc[i][j][e];
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            if (lc == 0) red[(wm * WM + row_of(i)) * Cfg::WARPS_N + wn] = s;
        }
        __syncthreads();
        T* out = p.rowsumsq + (long)blockIdx.z * p.s_rs;
        for (int r = tid; r < BM; r += THREADS) {
            T s = T(0);
#pragma unroll
            for (int w = 0; w < Cfg::WARPS_N; w++) s += red[r * Cfg::WARPS_N + w];
            out[(long)(m0 + r) * p.ld_rs + nt] = s;
        }
        return;
    }

    T* gC = p.C + (long)blockIdx.z * p.sC;
    const bool use_beta = (p.beta != T(0));
#pragma unroll
    for (int i = 0; i < FM; i++) {
        const long row = m0 + wm * WM + row_of(i);
#pragma unroll
        for (int j = 0; j < FN; j++) {
            if constexpr (F64) {
                const int col = n0 + wn * WN + col_of(j);
                double2* ptr = reinterpret_cast<double2*>(gC + row * p.ldc + col);
                double2 v;
                v.x = p.alpha * acc[i][j][0];
                v.y = p.alpha * acc[i][j][1];
                if (use_beta) {
                    double2 o = *ptr;
                    v.x += p.beta * o.x;
                    v.y += p.beta * o.y;
                }
                *ptr = v;
            } else {
                const int col = n0 + wn * WN + col_of(j);
                T* ptr = gC + row * p.ldc + col;
                T v = p.alpha * acc[i][j][0];
                if (use_beta) v += p.beta * (*ptr);
                *ptr = v;
            }
        }
    }
}

template <typename T, int BM, int BN, int WM, int WN, bool AK, bool BK_>
inline cudaError_t launch_gemm_cfg(const GemmArgs<T>& a, int batch, cudaStream_t stream) {
    using Cfg = GemmCfg<T, BM, BN, WM, WN, AK, BK_>;
    auto kern = gemm_kernel<T, BM, BN, WM, WN, AK, BK_>;
    // cudaFuncAttributeMaxDynamicSharedMemorySize is set once per context (configure_gemms), never here:
    // this function also runs inside stream captures.
    long tm = a.M / BM, tn = a.N / BN;
    long tiles = a.lower_only ? tm * (tm + 1) / 2 : tm * tn;
    if (tiles <= 0 || batch <= 0) return cudaSuccess;
    dim3 grid((unsigned)tiles, 1, (unsigned)batch);
    return launch_prio(kern, grid, dim3(Cfg::THREADS), Cfg::SMEM_BYTES, stream, a);
}

// CTA tile choice.  Measured on B200 (probes/gemm_bench.cu, profiles/r01_gemm_tile_probe.log): the 64x64 tile
// (4 warps, 32x32 warp tiles, 60 KB of shared memory -> 3 CTAs per SM) sustains 33.2 TFLOP/s on 2048^3 x 4
// against 31.0 for 128x128 (8 warps, 1 CTA per SM) and 35.6 for cuBLAS, and it quantises far better on the
// small and triangular grids of the recursion.  In f32 the 128x128 configuration (8 x 8 outputs per thread) has the
// better FFMA-to-load ratio on paper but measured slower as well (north-star step 124.7 ms vs 113.8 ms, predict 455
// vs 413 ms).  So the large products run on 64x64 tiles in both precisions.
//
// Latency-bound products (the bottom levels of the recursion at small n, small batches): a 64x64 tile puts its whole k
// loop on ONE SM's FP64 pipe (0.52 us per 16-k step) while most of the 148 SMs idle.  When the caller allows it
// (GemmArgs::small_ctas) and the 64x64 grid would have at most that many CTAs, the product runs on 32x32 tiles instead
// (4 warps of 16x16; four times the CTAs, a quarter of the k-loop time each).  Same bits: every output element sees
// the same sequence of k4 steps, the tiles only differ in how many structural zeros they multiply.  FP64 only (the FFMA
// micro-kernel needs 32-wide warp tiles).  Measured (profiles/r02_small_tile.log, ms per batched evaluation, off -> 296):
// n = 500 B = 3 0.300 -> 0.257, n = 512 B = 33 0.474 -> 0.427, n = 1024 B = 9 0.875 -> 0.786, n = 1024 B = 33 1.751 ->
// 1.722; at n >= 2048 the GPU is busy with other groups' large products and the less efficient tile costs 1-1.5 %,
// so the engine only allows it up to n = 1024.
template <typename T, bool AK, bool BK_>
inline cudaError_t launch_gemm(const GemmArgs<T>& a, int batch, cudaStream_t stream) {
    const long tm = a.M / 64, tn = a.N / 64;
    const long tiles = a.lower_only ? tm * (tm + 1) / 2 : tm * tn;
    if (a.rowsumsq == nullptr && a.raster_group == 0 && tiles * batch <= a.small_ctas) {
        // f64: 4 warps of 16x16 (2 x 2 DMMA tiles); f32: 2 warps of 32x16 (4 x 4 outputs per thread, the smallest
        // warp tile of the FFMA micro-kernel)
        if constexpr (std::is_same<T, double>::value) return launch_gemm_cfg<T, 32, 32, 16, 16, AK, BK_>(a, batch, stream);
        else return launch_gemm_cfg<T, 32, 32, 32, 16, AK, BK_>(a, batch, stream);
    }
    return launch_gemm_cfg<T, 64, 64, 32, 32, AK, BK_>(a, batch, stream);
}

}  // namespace hbegp
