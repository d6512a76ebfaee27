// FP32 GEMM on the Blackwell tensor path (sm_100a): tcgen05.mma kind::tf32 with a 3xTF32 operand split, TMA-staged
// operand tiles, accumulators in TMEM.
//
// Same contract as gemm_kernel<float, ...> in gemm.cuh (C = alpha * A(.,k) B(.,k)^T + beta * C, each operand k-major or
// row-major, triangular k ranges, lower tiles only, batch in grid.z, optional row-sum-of-squares epilogue); it serves
// the --use-32 path (src/bin/hbetune/main.rs:240-244) where the plain-FFMA kernel is issue bound at ~46 TFLOP/s.
//
// One tf32 pass keeps 11 significand bits, which would break the 1e-4 parity bound, so every operand element x is
// split on the fly into hi = rn_tf32(x) and lo = rn_tf32(x - hi) (22 bits together) and three products are issued
// per k step: hi*hi into one TMEM accumulator, hi*lo and lo*hi into another one, so that the small terms are summed
// among themselves instead of being rounded away against the large running sum; the epilogue adds the two.  The
// dropped lo*lo term is below 2^-22 of the product.
//
// CTA = 10 warps, one 128 x 128 output tile:
//   warp 0   TMA producer: cp.async.bulk.tensor (boxes of 32 fp32 = 128 bytes along the contiguous direction,
//            SWIZZLE_128B for k-major operands, SWIZZLE_128B_ATOM_32B for row-major ones) into a 3-stage ring,
//            completion on an mbarrier;
//   warps 2-5 transform: read the raw tile, write hi in place and lo into a twin buffer at the same offsets (the
//            swizzle pattern is address based, so the twin inherits the layout), fence.proxy.async, arrive;
//   warp 1   MMA issuer: one elected lane issues 4 k steps x 3 tcgen05.mma (M = 128, N = 128, K = 8) per stage from
//            shared-memory descriptors (K-major SWIZZLE_128B or MN-major SWIZZLE_128B_BASE32B) and commits the stage back to the
//            producer; after the last stage it commits to the epilogue barrier;
//   warps 6-9 drain + epilogue: the tensor core's FP32 accumulation truncates (a systematic bias), so the hi*hi term is
//            not accumulated in TMEM beyond 16 k: the products land in one of three rotating 128-column buffers and are
//            added round-to-nearest into registers with tcgen05.ld (one output row per thread); at the end the small
//            terms (accumulated in TMEM: their bias is 2^-11 of that) are added, then alpha / beta and the masked
//            store (or the row sums of squares).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "gemm.cuh"
#include "tcgen05.cuh"

namespace hbegp {
namespace tf32 {

using namespace tc;

// What bounds the main loop now is shared-memory bandwidth: per 32-k block TMA writes 32 KB, the transform reads 32 KB and
// writes 64 KB, and the twelve MMAs read 96 KB of operands -- 224 KB at 128 B/cycle = 1750 cycles against ~2000 measured
// (the tensor pipe itself needs 1250).  Measured and rejected on the way: eight transform warps (145 vs 151 TFLOP/s), eight
// drain warps (107 vs 113 at the time), descriptors hoisted out of the issue loop (no change).
// Stage depth: 32 k per stage (128-byte rows, three 64 KB stages).  A finer ring -- 16 k per stage, six 32 KB stages, 64-byte
// rows with SWIZZLE_64B -- was measured as well: 120-125 TFLOP/s against 132-137 on 4096^3; the doubled number of barrier
// hand-shakes costs more than the shorter slot residence gains.
constexpr int BM = 128, BN = 128, BK = 32, STAGES = 3;
constexpr int TILE_BYTES = BM * BK * 4;  // one operand tile (hi or lo): 16 KB
constexpr int STAGE_BYTES = 4 * TILE_BYTES;  // A_hi, A_lo, B_hi, B_lo
constexpr int MN_BOX_BYTES = 32 * BK * 4;    // one TMA box of a row-major operand: BK k-rows x 32 rows (128 bytes)
constexpr int THREADS = 320;
constexpr int NBUF = 3;         // TMEM buffers the hi*hi products of successive k steps rotate through
#ifndef HBEGP_TF32_KS_PER_BUF
#define HBEGP_TF32_KS_PER_BUF 2
#endif
// k steps (of 8) whose products share a TMEM buffer before it is drained.  1 = no accumulation in TMEM at all; 2 = one
// truncating accumulation per 16 k.  Measured (profiles/r02_tf32_accumulation.md): 2 keeps the positive-definiteness margin
// and the fitted optimum of 1 while halving the MMA <-> drain hand-shakes (113 -> 135 TFLOP/s); 8 and more lose the margin.
constexpr int KS_PER_BUF = HBEGP_TF32_KS_PER_BUF;
constexpr int TMEM_COLS = 512;  // NBUF x 128 columns of per-k-step products + 128 for the small-term accumulator
constexpr size_t SMEM_BYTES = (size_t)STAGES * STAGE_BYTES + 1024 /* alignment slack */ + 256 /* barriers */;

struct Params {
    CUtensorMap mapA, mapB;  // 3-D: (contiguous dim, other dim, batch)
    float* C;
    long ldc, sC;
    int M, N, K;
    int kmode, lower_only;
    float alpha, beta;
    float* rowsumsq;
    long ld_rs, s_rs;
    int raster_group;
};

// Instruction descriptor: D fp32, A / B tf32, M = 128, N = 128; a_major / b_major: 0 = K-major, 1 = MN-major.
__host__ __device__ constexpr uint32_t make_idesc(bool a_kmajor, bool b_kmajor, int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((a_kmajor ? 0u : 1u) << 15) | ((b_kmajor ? 0u : 1u) << 16) |
           ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Round to TF32 (11 significand bits), nearest with ties away from zero -- what cvt.rna.tf32.f32 does -- as two integer
// operations.  nvcc expands cvt.rna.tf32.f32 into ~7 instructions on sm_100a (shift / add / mask plus Inf-NaN
// special-casing, see the SASS), and with 128 elements per thread and k-block the four transform warps were ISSUE
// BOUND on them: ncu put 47 % of the ALU pipe and the top stall samples of the whole kernel there while the tensor
// pipe idled at 33 %.  Finite inputs only (a value within 2^-11 of FLT_MAX would round to Inf; the GP matrices are
// nowhere near).
__device__ __forceinline__ float rn_tf32(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }

// tile coordinates, heavy tiles first (same orders as gemm_kernel)
__device__ __forceinline__ void tile_coords(const Params& p, int t, int tiles_m, int tiles_n, int& mt, int& nt) {
    if (p.lower_only) {
        int r = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
        while ((long)(r + 1) * (r + 2) / 2 <= t) ++r;
        while ((long)r * (r + 1) / 2 > t) --r;
        mt = r;
        nt = t - r * (r + 1) / 2;
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

template <bool A_KMAJOR, bool B_KMAJOR>
__global__ void __launch_bounds__(THREADS, 1) gemm_tf32x3_kernel(const __grid_constant__ Params p) {
    extern __shared__ unsigned char smem_raw[];
    // swizzle atoms (8 rows x 128 bytes) must sit on 1024-byte boundaries
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)STAGES * STAGE_BYTES);
    uint64_t* full = bars;                 // TMA landed
    uint64_t* xf = bars + STAGES;          // transform done
    uint64_t* empty = bars + 2 * STAGES;   // MMAs of the stage retired
    uint64_t* accf = bars + 3 * STAGES;    // [NBUF] the product of one k step has landed in TMEM buffer b
    uint64_t* acce = accf + NBUF;          // [NBUF] buffer b has been added into the registers
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acce + NBUF);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tiles_m = (p.M + BM - 1) / BM, tiles_n = (p.N + BN - 1) / BN;
    int mt, nt;
    tile_coords(p, blockIdx.x, tiles_m, tiles_n, mt, nt);
    const int m0 = mt * BM, n0 = nt * BN, bz = blockIdx.z;
    int kbeg = 0, kend = p.K;
    if (p.kmode == K_LE_N) kend = min(p.K, n0 + BN);
    else if (p.kmode == K_GE_N) kbeg = n0;
    else if (p.kmode == K_LE_M) kend = min(p.K, m0 + BM);
    else if (p.kmode == K_GE_M) kbeg = m0;
    const int nk = (kend - kbeg) / BK;
    constexpr int KSTEPS = BK / 8;  // tcgen05.mma kind::tf32 has K = 8

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < STAGES; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&xf[s], 4);
            mbar_init(&empty[s], 1);
        }
        for (int b = 0; b < NBUF; b++) {
            mbar_init(&accf[b], 1);
            mbar_init(&acce[b], 4);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&p.mapA)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&p.mapB)) : "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    // TMEM columns: NBUF buffers of 128 for the hi*hi product of one k step each, then 128 for the `small` accumulator
    const uint32_t d_small = tmem_base + NBUF * BN;

    if (warp == 0) {
        // ---------------------------------------------------------------- TMA producer
        if (lane == 0) {
            for (int kt = 0; kt < nk; kt++) {
                const int s = kt % STAGES;
                mbar_wait(&empty[s], ((kt / STAGES) & 1) ^ 1);
                unsigned char* st = smem + (size_t)s * STAGE_BYTES;
                mbar_expect_tx(&full[s], 2 * TILE_BYTES);
                const int k0 = kbeg + kt * BK;
                if (A_KMAJOR) {
                    tma_load_3d(&p.mapA, &full[s], st, k0, m0, bz);  // box (32 k, 128 rows)
                } else {
#pragma unroll
                    for (int j = 0; j < BM / 32; j++)  // four boxes (32 rows contiguous, 32 k)
                        tma_load_3d(&p.mapA, &full[s], st + j * MN_BOX_BYTES, m0 + 32 * j, k0, bz);
                }
                unsigned char* sb = st + 2 * TILE_BYTES;
                if (B_KMAJOR) {
                    tma_load_3d(&p.mapB, &full[s], sb, k0, n0, bz);
                } else {
#pragma unroll
                    for (int j = 0; j < BN / 32; j++) tma_load_3d(&p.mapB, &full[s], sb + j * MN_BOX_BYTES, n0 + 32 * j, k0, bz);
                }
            }
        }
    } else if (warp == 1) {
        // ---------------------------------------------------------------- MMA issuer
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc(A_KMAJOR, B_KMAJOR, BN);
            // K-major (128 rows x 128 bytes of k): 8-row groups 1024 bytes apart (SBO); one k step of 8 = 32 bytes
            // inside the swizzled row.
            // MN-major (per 32-row box: 32 k-rows x 128 bytes of rows): 32-row groups 4096 bytes apart (LBO), groups of
            // 4 k-rows 512 bytes apart (SBO); one k step of 8 = 1024 bytes.
            constexpr uint32_t k_sbo = 8 * BK * 4, k_lay = 2;  // SWIZZLE_128B
            constexpr uint32_t a_lbo = A_KMAJOR ? 16 : MN_BOX_BYTES, a_sbo = A_KMAJOR ? k_sbo : 512, a_kstep = A_KMAJOR ? 32 : 1024;
            constexpr uint32_t b_lbo = B_KMAJOR ? 16 : MN_BOX_BYTES, b_sbo = B_KMAJOR ? k_sbo : 512, b_kstep = B_KMAJOR ? 32 : 1024;
            constexpr uint32_t a_lay = A_KMAJOR ? k_lay : 1, b_lay = B_KMAJOR ? k_lay : 1;
            for (int kt = 0; kt < nk; kt++) {
                const int s = kt % STAGES;
                mbar_wait(&xf[s], (kt / STAGES) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a_hi = smem_u32(smem + (size_t)s * STAGE_BYTES), a_lo = a_hi + TILE_BYTES;
                const uint32_t b_hi = a_hi + 2 * TILE_BYTES, b_lo = a_hi + 3 * TILE_BYTES;
#pragma unroll
                for (int ks = 0; ks < KSTEPS; ks++) {
                    const int g = kt * KSTEPS + ks, grp = g / KS_PER_BUF, buf = grp % NBUF, use = grp / NBUF;
                    const bool first = (g % KS_PER_BUF) == 0, last = (g % KS_PER_BUF) == KS_PER_BUF - 1 || g == nk * KSTEPS - 1;
                    if (first) {
                        // the buffer's previous product must have been added into the registers (first NBUF uses pass at once)
                        mbar_wait(&acce[buf], (use & 1) ^ 1);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    }
                    const uint64_t dah = make_desc(a_hi + ks * a_kstep, a_lbo, a_sbo, a_lay);
                    const uint64_t dal = make_desc(a_lo + ks * a_kstep, a_lbo, a_sbo, a_lay);
                    const uint64_t dbh = make_desc(b_hi + ks * b_kstep, b_lbo, b_sbo, b_lay);
                    const uint64_t dbl = make_desc(b_lo + ks * b_kstep, b_lbo, b_sbo, b_lay);
                    mma_tf32(d_small, dal, dbh, idesc, g > 0 ? 1u : 0u);
                    mma_tf32(d_small, dah, dbl, idesc, 1u);
                    mma_tf32(tmem_base + buf * BN, dah, dbh, idesc, first ? 0u : 1u);  // fresh product per buffer use
                    if (last) mma_commit(&accf[buf]);
                }
                mma_commit(&empty[s]);  // implies tcgen05.fence::before_thread_sync
            }
        }
    } else if (warp < 6) {
        // ---------------------------------------------------------------- transform (warps 2..5)
        const int t = tid - 64;  // 0..127
        for (int kt = 0; kt < nk; kt++) {
            const int s = kt % STAGES;
            mbar_wait(&full[s], (kt / STAGES) & 1);
            float4* a_hi = reinterpret_cast<float4*>(smem + (size_t)s * STAGE_BYTES);
            float4* a_lo = a_hi + TILE_BYTES / 16;
            float4* b_hi = a_hi + 2 * TILE_BYTES / 16;
            float4* b_lo = a_hi + 3 * TILE_BYTES / 16;
#pragma unroll 4
            for (int i = t; i < TILE_BYTES / 16; i += 128) {
                const float4 va = a_hi[i], vb = b_hi[i];
                float4 h, l;
                h.x = rn_tf32(va.x); h.y = rn_tf32(va.y); h.z = rn_tf32(va.z); h.w = rn_tf32(va.w);
                l.x = rn_tf32(va.x - h.x); l.y = rn_tf32(va.y - h.y); l.z = rn_tf32(va.z - h.z); l.w = rn_tf32(va.w - h.w);
                a_hi[i] = h;
                a_lo[i] = l;
                h.x = rn_tf32(vb.x); h.y = rn_tf32(vb.y); h.z = rn_tf32(vb.z); h.w = rn_tf32(vb.w);
                l.x = rn_tf32(vb.x - h.x); l.y = rn_tf32(vb.y - h.y); l.z = rn_tf32(vb.z - h.z); l.w = rn_tf32(vb.w - h.w);
                b_hi[i] = h;
                b_lo[i] = l;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> tensor-core reads
            __syncwarp();
            if (lane == 0) mbar_arrive(&xf[s]);
        }
    } else {
        // ---------------------------------------------------------------- drain + epilogue (warps 6..9)
        // The tensor core adds into its FP32 accumulator with TRUNCATION: a bias of ~2^-24 of the running sum per
        // accumulation, always the same sign.  Accumulating k = 4096 in TMEM loses 2.7e-5 on positive data (probe), and
        // even 64-k chunks (2e-7, less than the FFMA kernel's random rounding error) cost the f32 Cholesky its
        // positive-definiteness margin, because a systematic error does not average out over the recursion
        // (a probe: K stopped factoring at 4x the noise level the FFMA path reaches).  So
        // (almost) nothing is accumulated in TMEM for the hi*hi term: every KS_PER_BUF k steps (k = 16) start a fresh product
        // in one of NBUF rotating buffers, which is added round-to-nearest into registers here while the tensor core
        // fills the next.
        // One output row per thread (a warp may touch TMEM lanes 32 * (warp % 4) .. + 31 only), 128 columns in registers.
        const int lane_base = 32 * (warp & 3);
        const int row = m0 + lane_base + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)lane_base << 16);
        float acc[BN];
#pragma unroll
        for (int j = 0; j < BN; j++) acc[j] = 0.f;
        const int nsteps = (nk * KSTEPS + KS_PER_BUF - 1) / KS_PER_BUF;
        for (int g = 0; g < nsteps; g++) {
            const int buf = g % NBUF;
            mbar_wait(&accf[buf], (g / NBUF) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int c0 = 0; c0 < BN; c0 += 32) {
                float v[32];
                tmem_ld32(lane_addr + buf * BN + c0, reinterpret_cast<uint32_t*>(v));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int j = 0; j < 32; j++) acc[c0 + j] += v[j];
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&acce[buf]);
        }
        // every MMA has retired (the last k step's commit covers the small-term products too)
        const bool row_ok = row < p.M;
        float sumsq = 0.f;
        float* crow = p.C ? p.C + (long)bz * p.sC + (long)row * p.ldc + n0 : nullptr;
        const bool use_beta = p.beta != 0.f;
#pragma unroll
        for (int c0 = 0; c0 < BN; c0 += 32) {
            float small[32];
            if (nk > 0) {
                tmem_ld32(lane_addr + NBUF * BN + c0, reinterpret_cast<uint32_t*>(small));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            } else {
#pragma unroll
                for (int j = 0; j < 32; j++) small[j] = 0.f;
            }
            // (no early exit: the tcgen05.ld above is warp-aligned, every lane must reach it in every iteration)
            const bool in_range = row_ok && n0 + c0 < p.N;  // N is a multiple of 64: a 32-column chunk is all in or all out
            if (in_range && p.rowsumsq != nullptr) {
#pragma unroll
                for (int j = 0; j < 32; j++) {
                    const float v = acc[c0 + j] + small[j];
                    sumsq = fmaf(v, v, sumsq);
                }
            } else if (in_range) {
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    float4 v;
                    v.x = p.alpha * (acc[c0 + j] + small[j]);
                    v.y = p.alpha * (acc[c0 + j + 1] + small[j + 1]);
                    v.z = p.alpha * (acc[c0 + j + 2] + small[j + 2]);
                    v.w = p.alpha * (acc[c0 + j + 3] + small[j + 3]);
                    float4* ptr = reinterpret_cast<float4*>(crow + c0 + j);
                    if (use_beta) {
                        const float4 o = *ptr;
                        v.x += p.beta * o.x; v.y += p.beta * o.y; v.z += p.beta * o.z; v.w += p.beta * o.w;
                    }
                    *ptr = v;
                }
            }
            __syncwarp();
        }
        if (p.rowsumsq != nullptr && row_ok) p.rowsumsq[(long)bz * p.s_rs + (long)row * p.ld_rs + nt] = sumsq;
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// ---- host side -------------------------------------------------------------------------------------------------
// Tensor map of one operand: `rows` x `kdim` elements of which the k-major flavour has k contiguous (X[r * ld + k]) and
// the other has rows contiguous (X[k * ld + r]); third dimension = batch.  Boxes: (BK k, 128 rows) resp. (32 rows, BK k).
inline bool make_operand_map(CUtensorMap* map, const float* base, bool kmajor, int rows, int kdim, long ld, long batch_stride, int batch) {
    EncodeTiledFn enc = encode_fn();
    if (!enc) return false;
    cuuint64_t dims[3] = {(cuuint64_t)(kmajor ? kdim : rows), (cuuint64_t)(kmajor ? rows : kdim), (cuuint64_t)batch};
    cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)(batch > 1 ? batch_stride : (long)dims[1] * ld) * 4};
    cuuint32_t box[3] = {(cuuint32_t)(kmajor ? BK : 32), (cuuint32_t)(kmajor ? BM : BK), 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE,
                     kmajor ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

template <bool AK, bool BKM>
inline cudaError_t configure() {
    return cudaFuncSetAttribute(gemm_tf32x3_kernel<AK, BKM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES);
}

// Launch with the GemmArgs<float> contract of gemm.cuh.  Returns cudaErrorNotSupported when the tensor maps cannot be
// built (misaligned operands), so that the caller can fall back to the FFMA kernel.
template <bool AK, bool BKM>
inline cudaError_t launch(const GemmArgs<float>& a, int batch, cudaStream_t stream) {
    if (batch <= 0 || a.M <= 0 || a.N <= 0) return cudaSuccess;
    Params p;
    if (batch > 1 && (a.sA == 0 || a.sB == 0)) return cudaErrorNotSupported;  // a TMA dimension needs a non-zero stride
    if (!make_operand_map(&p.mapA, a.A, AK, a.M, a.K, a.lda, a.sA, batch)) return cudaErrorNotSupported;
    if (!make_operand_map(&p.mapB, a.B, BKM, a.N, a.K, a.ldb, a.sB, batch)) return cudaErrorNotSupported;
    p.C = a.C; p.ldc = a.ldc; p.sC = a.sC;
    p.M = a.M; p.N = a.N; p.K = a.K;
    p.kmode = a.kmode; p.lower_only = a.lower_only;
    p.alpha = a.alpha; p.beta = a.beta;
    p.rowsumsq = a.rowsumsq; p.ld_rs = a.ld_rs; p.s_rs = a.s_rs;
    p.raster_group = a.raster_group;
    const long tm = (a.M + BM - 1) / BM, tn = (a.N + BN - 1) / BN;
    const long tiles = a.lower_only ? tm * (tm + 1) / 2 : tm * tn;
    dim3 grid((unsigned)tiles, 1, (unsigned)batch);
    return launch_prio(gemm_tf32x3_kernel<AK, BKM>, grid, dim3(THREADS), SMEM_BYTES, stream, p);
}

// Policy (process-wide, set by hbegp_ctx_create from HBEGP_TF32): whether f32 contractions go through the tensor path.
inline bool& enabled() {
    static bool on = true;
    return on;
}
// The smallest min(M, N) for which they do: below it one 128 x 128 tile per CTA leaves the GPU emptier than the 64 x 64
// FFMA tiles and the per-CTA pipeline start-up dominates.
constexpr int MIN_EXTENT = 256;

}  // namespace tf32

// Dispatch used by the engine: f64 -> DMMA kernel; f32 -> tcgen05 3xTF32 when the policy allows, else the FFMA kernel.
// The tensor path relies on the 128-wide-tile invariant of the recursion: every 128-wide diagonal block of a triangular
// operand has exact zeros above its diagonal (the bottom nodes write them).
template <typename T>
inline bool gemm_uses_tf32(int M, int N) {
    return std::is_same<T, float>::value && tf32::enabled() && (M < N ? M : N) >= tf32::MIN_EXTENT;
}

template <typename T, bool AK, bool BKM>
inline cudaError_t launch_gemm_auto(const GemmArgs<T>& a, int batch, cudaStream_t stream) {
    if constexpr (std::is_same<T, float>::value) {
        if (gemm_uses_tf32<T>(a.M, a.N)) return tf32::launch<AK, BKM>(a, batch, stream);
    }
    return launch_gemm<T, AK, BKM>(a, batch, stream);
}

}  // namespace hbegp
