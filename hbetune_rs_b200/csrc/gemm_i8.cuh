// K^-1 = W^T W in f64 on the integer tensor cores (sm_100a, tcgen05.mma kind::i8): Ozaki scheme II (Ozaki, Uchino,
// Imamura 2025, "Ozaki Scheme II: a GEMM-oriented emulation of floating-point matrix multiplication using an integer
// modular technique"), specialised to the symmetric product of one lower-triangular matrix with itself.
//
//   1. k_oz_colexp, k_oz_split: column j of W gets an exponent e_j such that W'[k][j] = rn(2^e_j W[k][j]) satisfies |W'| <= 2^b,
//      with b the largest value for which np 2^2b < P / 2 (P = product of the S moduli): then C' = W'^T W' is an
//      integer of magnitude below P / 2 and is fixed by its residues.  For every modulus p_m the residues
//      W' mod p_m are written as signed int8 in the symmetric range, transposed (R_m[j][k] = W'[k][j] mod p_m) so that
//      both operands of the product are K-major tiles of the same plane.
//   2. k_oz_syrk_i8: C_m = R_m R_m^T for every modulus on the lower 128 x 128 tiles, k from the tile row on (R_m is
//      upper triangular), exact in the int32 accumulator (|C_m| <= np 128^2 < 2^31 for np < 131072); the epilogue
//      reduces mod p_m and stores one byte per element.
//   3. k_oz_merge: Chinese remaindering of C' from its S residues in exact 128-bit integer arithmetic, symmetric
//      range, one rounding to double, scaling by 2^-(e_i + e_j), written into the lower 64 x 64 tiles of K^-1 (the
//      cells the DMMA product writes).
//
// The only error is the rounding of W to b bits relative to its column maximum; the result depends on the matrix
// alone (not on the batch, the stream group or a tile choice).  Why only this product and how S was chosen:
// DESIGN.md section 4 ("K6b").
//
// Workspace of one matrix (oz_slot_bytes): S planes of R_m and S planes of C_m mod p_m, each stored as the lower
// 128 x 128 tiles of the matrix, packed (tile (r, c), r >= c, at index r (r + 1) / 2 + c; R_m's tile (c, r) of the
// upper triangle is stored at the index of its transpose), one 16 KB tile = 128 rows x 128 bytes; then the np
// column exponents.  Rows and columns past np and the part of a diagonal tile of R_m below its diagonal hold zeros
// written by the split (never stale memory), so every MMA tile is full.
//
// k_oz_syrk_i8: CTA = 6 warps, one 128 x 128 output tile of one modulus and one matrix (grid: lower tiles x S x batch):
//   warp 0   TMA producer: one box of 128 rows x 128 bytes (SWIZZLE_128B) per operand and k block into a 3-stage
//            ring (the diagonal tiles load their single operand once);
//   warp 1   MMA issuer: 4 x tcgen05.mma kind::i8 (M = N = 128, K = 32) per stage, all of k accumulated in TMEM;
//   warps 2-5 epilogue: tcgen05.ld one row per thread, reduction mod p_m, 128-byte row stores.
// 2 CTAs per SM (100 KB of shared memory, 128 TMEM columns each): one CTA's epilogue overlaps the other's main loop.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.cuh"
#include "tcgen05.cuh"

namespace hbegp {
namespace oz {

using namespace tc;

// Moduli: the S largest pairwise coprime integers <= 256 (P = 2^110.2).  S = 14 measured against the truncated product
// in f64 (n = 2048, d = 16, Matern 2.5, noise 1e-2 and 1e-4): max |dK^-1| / max |K^-1| = 6e-13 / 3e-14 / 2.2e-15 /
// 6e-16 / 2e-16 at S = 12 / 13 / 14 / 15 / 16, against the 1e-9 tolerance of the factor tests.
constexpr int S = 14;
__host__ __device__ constexpr int modulus(int m) {
    return m == 0 ? 256 : m == 1 ? 255 : m == 2 ? 253 : m == 3 ? 251 : m == 4 ? 247 : m == 5 ? 241 : m == 6 ? 239
         : m == 7 ? 233 : m == 8 ? 229 : m == 9 ? 227 : m == 10 ? 223 : m == 11 ? 217 : m == 12 ? 211 : 199;
}
// P = prod p_m as two 64-bit halves, floor(P / 2), 2^58 / P, and the CRT weights c_m = (P / p_m) ((P / p_m)^-1 mod p_m)
// mod P as four 32-bit limbs, least significant first: C' = sum_m r_m c_m mod P (tests/test_kinv_emulation.py re-derives
// all of them from the moduli).
constexpr uint64_t P_LO = 0x3bdc01086e91ad00ull, P_HI = 0x0000478ff11c7ad1ull;
constexpr uint64_t HALF_LO = 0x9dee00843748d680ull, HALF_HI = 0x000023c7f88e3d68ull;
constexpr double INV_P58 = 1.9858025962649873e-16;
// (a function, not a __constant__ table: the unrolled merge folds the limbs into immediates)
__host__ __device__ constexpr uint32_t crt_limb(int m, int l) {
    constexpr uint32_t t[S][4] = {
        {0x37fb0e01u, 0x3da6cc26u, 0xcdd91dc0u, 0x00000a57u},  // 256
        {0x2d9b6200u, 0x515b4421u, 0x61efbe69u, 0x00003c0eu},  // 255
        {0x6436c700u, 0xa8c49274u, 0x2ee81407u, 0x000033c3u},  // 253
        {0x0aaff900u, 0xaff19c1cu, 0xd136bce2u, 0x00000446u},  // 251
        {0xf7471500u, 0xd3598a93u, 0xb743daa4u, 0x000032b3u},  // 247
        {0xb4ac3100u, 0x80994803u, 0x38e00b2au, 0x00003a7fu},  // 241
        {0xb50dfd00u, 0xf9cd4608u, 0xfc396104u, 0x00001c71u},  // 239
        {0x0fc58900u, 0xf5ef92cau, 0x53de92a8u, 0x00002dc3u},  // 233
        {0x2b43a200u, 0x4f7c9d74u, 0xf258b82cu, 0x0000419fu},  // 229
        {0x93d41700u, 0x4d8fc60du, 0xcd5da098u, 0x0000303bu},  // 227
        {0x1a5f8a00u, 0x9a05c78eu, 0x5ab66f28u, 0x0000421bu},  // 223
        {0x5e122800u, 0x90ded2a3u, 0x9f5e87f5u, 0x00002cd9u},  // 217
        {0xd7195400u, 0xa67b8783u, 0xca9cace9u, 0x00003a55u},  // 211
        {0x8f385a00u, 0x80e799d2u, 0x8574cdfdu, 0x00003310u},  // 199
    };
    return t[m][l];
}

constexpr int TB = 128;                 // tile edge: rows, and k bytes per TMA box / pipeline stage
constexpr int TILE_BYTES = TB * TB;     // one int8 tile: 16 KB
constexpr int STAGES = 3;
constexpr int THREADS = 192;
constexpr int TMEM_COLS = 128;
constexpr size_t SMEM_BYTES = (size_t)STAGES * 2 * TILE_BYTES + 1024 /* alignment slack */ + 256 /* barriers */;
constexpr int E_CLAMP = 400;            // |e_j| <= E_CLAMP keeps 2^(sh - e_i - e_j) a normal double in the merge
constexpr int E_BAD = -32768;           // column with a non-finite entry: its row and column of K^-1 come out NaN
constexpr int MAX_BITS = 50;            // |W'| < 2^51 for the rounding trick of the split

// Largest b with np 2^2b < P / 2 (exact, 128-bit), at most MAX_BITS.
inline int scale_bits(int np) {
    const unsigned __int128 half = ((unsigned __int128)HALF_HI << 64) | HALF_LO;
    int b = MAX_BITS;
    while (b > 0 && ((unsigned __int128)np << (2 * b)) >= half) --b;
    return b;
}

__host__ __device__ inline long ntri_of(int tiles) { return (long)tiles * (tiles + 1) / 2; }
inline long ntri(int np) { return ntri_of((np + TB - 1) / TB); }
// Bytes of one matrix's workspace: S input and S output planes of packed lower tiles, then the column exponents
// (rounded up to whole tiles, so that every slot starts on a tile boundary of the tensor map).
inline size_t slot_bytes(int np) {
    const size_t ex = ((size_t)(np + TB - 1) / TB * TB * sizeof(int) + TILE_BYTES - 1) / TILE_BYTES * TILE_BYTES;
    return 2 * (size_t)S * ntri(np) * TILE_BYTES + ex;
}

// ---- split ------------------------------------------------------------------------------------------------------
// k_oz_colexp writes the column exponents, then k_oz_split one block per tile (one block per column stripe for both
// steps left the stripes of the first columns, 32 tiles and the whole column each at n = 4096, on the critical path:
// 16 of the 28 ms of the north-star K^-1 phase).  W' is the mantissa of fma(w, 2^e, 1.5 2^52) (one rounding to
// nearest), its residues come from three pieces of the 52-bit offset value.
template <int M>
__device__ __forceinline__ uint32_t residue_byte(uint32_t lo24, uint32_t h0, uint32_t h1) {
    constexpr uint32_t p = (uint32_t)modulus(M);
    constexpr uint32_t c24 = (uint32_t)((1ull << 24) % p), c36 = (uint32_t)((1ull << 36) % p);
    constexpr uint32_t off = (uint32_t)(p - (uint32_t)((1ull << 51) % p));  // u = W' + 2^51
    const uint32_t t = lo24 + h0 * c24 + h1 * c36 + off;                      // < 2^26
    uint32_t r = t % p;
    if (r > (p - 1) / 2) r -= p;  // symmetric range, as a byte
    return r & 0xffu;
}

template <int M>
__device__ __forceinline__ void store_residues(unsigned char* dst, const uint32_t (&lo)[16], const uint32_t (&h0)[16],
                                               const uint32_t (&h1)[16]) {
    uint32_t w[4];
#pragma unroll
    for (int q = 0; q < 4; q++)
        w[q] = residue_byte<M>(lo[4 * q], h0[4 * q], h1[4 * q]) | residue_byte<M>(lo[4 * q + 1], h0[4 * q + 1], h1[4 * q + 1]) << 8 |
               residue_byte<M>(lo[4 * q + 2], h0[4 * q + 2], h1[4 * q + 2]) << 16 |
               residue_byte<M>(lo[4 * q + 3], h0[4 * q + 3], h1[4 * q + 3]) << 24;
    *reinterpret_cast<uint4*>(dst) = make_uint4(w[0], w[1], w[2], w[3]);
}

template <int M>
__device__ __forceinline__ void store_all(unsigned char* dst, size_t plane_bytes, const uint32_t (&lo)[16], const uint32_t (&h0)[16],
                                          const uint32_t (&h1)[16]) {
    store_residues<M>(dst + (size_t)M * plane_bytes, lo, h0, h1);
    if constexpr (M + 1 < S) store_all<M + 1>(dst, plane_bytes, lo, h0, h1);
}

// grid (column stripes of 128, 1, batch), 512 threads (4 rows at a time): e_j from the NaN-propagating max |W[k][j]|
// over k >= j.
__global__ void __launch_bounds__(512) k_oz_colexp(const double* __restrict__ W, long mstride, int np, int bits,
                                                   unsigned char* __restrict__ ws, size_t slot) {
    __shared__ double smax[512];
    const int c = blockIdx.x, b = blockIdx.z, tid = threadIdx.x, col = tid & (TB - 1), ph = tid >> 7;
    const int nt = (np + TB - 1) / TB;
    const double* Wb = W + (long)b * mstride;
    int* ex = reinterpret_cast<int*>(ws + (size_t)b * slot + 2 * (size_t)S * ntri_of(nt) * TILE_BYTES);
    const int j = c * TB + col;
    double m = 0.0;
    if (j < np) {
        for (int k = c * TB + ph; k < min(np, (c + 1) * TB); k += 4)
            if (k >= j) { const double a = fabs(Wb[(long)k * np + j]); m = (a > m || a != a) ? a : m; }
#pragma unroll 8
        for (int k = (c + 1) * TB + ph; k < np; k += 4) { const double a = fabs(Wb[(long)k * np + j]); m = (a > m || a != a) ? a : m; }
    }
    smax[tid] = m;
    __syncthreads();
    if (tid < TB) {
        for (int q = 1; q < 4; q++) { const double a = smax[tid + q * TB]; m = (a > m || a != a) ? a : m; }
        int e = 0;
        if (!(m <= 0x1p+440)) {  // NaN, Inf or beyond the clamp
            e = E_BAD;
        } else if (m > 0.0) {
            int E;
            frexp(m, &E);  // m < 2^E
            e = min(max(bits - E, -E_CLAMP), E_CLAMP);
        }
        ex[j] = e;  // also past np (e = 0): the split reads the exponents of whole stripes
    }
}

// grid (lower 128-tiles of W, 1, batch), 256 threads: W tile (kb, c) -> R_m tile (c, kb) of every plane; an item is 16
// consecutive k of one column.
__global__ void __launch_bounds__(256, 2) k_oz_split(const double* __restrict__ W, long mstride, int np,
                                                     unsigned char* __restrict__ ws, size_t slot) {
    int kb, c;
    lower_tile(blockIdx.x, kb, c);
    const int b = blockIdx.z, tid = threadIdx.x, col = tid & (TB - 1), j = c * TB + col;
    const long nr = ntri_of((np + TB - 1) / TB);
    const double* Wb = W + (long)b * mstride;
    unsigned char* wsb = ws + (size_t)b * slot;
    const int e = reinterpret_cast<const int*>(wsb + 2 * (size_t)S * nr * TILE_BYTES)[j];
    const double sc = e == E_BAD ? 0.0 : __longlong_as_double((long long)(1023 + e) << 52);  // 2^e, |e| <= E_CLAMP
    const size_t plane_bytes = (size_t)nr * TILE_BYTES;
    unsigned char* tile = wsb + (size_t)blockIdx.x * TILE_BYTES;
    constexpr double MAGIC = 0x1.8p+52;
    for (int it = tid; it < TB * (TB / 16); it += 256) {
        const int ch = it >> 7, k0 = kb * TB + ch * 16;  // (it & 127 == col)
        uint32_t lo[16], h0[16], h1[16];
#pragma unroll
        for (int q = 0; q < 16; q++) {
            const int k = k0 + q;
            const double w = (j < np && k < np && k >= j) ? Wb[(long)k * np + j] : 0.0;
            const uint64_t u = (uint64_t)__double_as_longlong(fma(w, sc, MAGIC)) & ((1ull << 52) - 1);  // W' + 2^51
            lo[q] = (uint32_t)u & 0xffffffu;
            h0[q] = (uint32_t)(u >> 24) & 0xfffu;
            h1[q] = (uint32_t)(u >> 36);
        }
        store_all<0>(tile + (size_t)col * TB + ch * 16, plane_bytes, lo, h0, h1);
    }
}

// ---- the per-modulus products -------------------------------------------------------------------------------------
struct SyrkParams {
    CUtensorMap map;       // all tiles of the launch's slots: (128 bytes of k, 128 rows, tiles)
    unsigned char* ws;     // first slot's workspace
    size_t slot;           // bytes per slot
    int nt;                // 128-tiles along each side
    int slot_tiles;        // slot / TILE_BYTES
};

// Instruction descriptor: D s32, A / B s8, both K-major, M = N = 128.
constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TB >> 3) << 17) | ((uint32_t)(TB >> 4) << 24);

__device__ __forceinline__ void mma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(IDESC), "r"(accumulate)
        : "memory");
}

__global__ void __launch_bounds__(THREADS, 2) k_oz_syrk_i8(const __grid_constant__ SyrkParams p) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)STAGES * 2 * TILE_BYTES);
    uint64_t* full = bars;
    uint64_t* empty = bars + STAGES;
    uint64_t* accf = bars + 2 * STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accf + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int mt, nt;
    lower_tile(blockIdx.x, mt, nt);
    const int mod = blockIdx.y, bz = blockIdx.z;
    const long nr = (long)p.nt * (p.nt + 1) / 2;
    const int nk = p.nt - mt;  // R_m is upper triangular: k blocks from the tile row on
    const bool diag = mt == nt;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < STAGES; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        mbar_init(accf, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&p.map)) : "memory");
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

    if (warp == 0) {
        if (lane == 0) {
            const int z0 = bz * p.slot_tiles + mod * (int)nr;
            for (int kt = 0; kt < nk; kt++) {
                const int s = kt % STAGES, kb = mt + kt;
                mbar_wait(&empty[s], ((kt / STAGES) & 1) ^ 1);
                unsigned char* st = smem + (size_t)s * 2 * TILE_BYTES;
                const int z = z0 + kb * (kb + 1) / 2;
                mbar_expect_tx(&full[s], diag ? TILE_BYTES : 2 * TILE_BYTES);
                tma_load_3d(&p.map, &full[s], st, 0, 0, z + mt);
                if (!diag) tma_load_3d(&p.map, &full[s], st + TILE_BYTES, 0, 0, z + nt);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // K-major SWIZZLE_128B: 8-row groups 1024 bytes apart (SBO); one k step of 32 = 32 bytes inside the row
            for (int kt = 0; kt < nk; kt++) {
                const int s = kt % STAGES;
                mbar_wait(&full[s], (kt / STAGES) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a = smem_u32(smem + (size_t)s * 2 * TILE_BYTES), bb = diag ? a : a + TILE_BYTES;
#pragma unroll
                for (int ks = 0; ks < TB / 32; ks++)
                    mma_i8(tmem_base, make_desc(a + 32 * ks, 16, 1024, 2), make_desc(bb + 32 * ks, 16, 1024, 2), (kt | ks) ? 1u : 0u);
                mma_commit(&empty[s]);
            }
            mma_commit(accf);
        }
    } else {
        const int lane_base = 32 * (warp & 3), row = lane_base + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)lane_base << 16);
        const int pm = modulus(mod);
        const float inv = 1.0f / (float)pm;
        mbar_wait(accf, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        unsigned char* dst = p.ws + (size_t)bz * p.slot + ((size_t)(S + mod) * nr + blockIdx.x) * TILE_BYTES + (size_t)row * TB;
#pragma unroll
        for (int c0 = 0; c0 < TB; c0 += 32) {
            uint32_t v[32];
            tmem_ld32(lane_addr + c0, v);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            uint32_t w[8];
#pragma unroll
            for (int q = 0; q < 8; q++) {
                uint32_t packed = 0;
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const int x = (int)v[4 * q + e];
                    int r = x - (int)floorf((float)x * inv) * pm;  // off by at most one modulus while |x| <= 46080 * 128^2
                    r += r < 0 ? pm : 0;
                    r -= r >= pm ? pm : 0;
                    packed |= (uint32_t)r << (8 * e);
                }
                w[q] = packed;
            }
            reinterpret_cast<uint4*>(dst + c0)[0] = make_uint4(w[0], w[1], w[2], w[3]);
            reinterpret_cast<uint4*>(dst + c0)[1] = make_uint4(w[4], w[5], w[6], w[7]);
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// ---- merge ---------------------------------------------------------------------------------------------------------
// C' from its residues r_m in [0, p_m) (exact), then one rounding to double of C' 2^-(e_i + e_j).
__device__ __forceinline__ double crt_value(const uint32_t (&r)[S], int e) {
    uint64_t acc0 = 0, acc1 = 0, acc2 = 0, acc3 = 0;  // each < 14 * 255 * 2^32
#pragma unroll
    for (int m = 0; m < S; m++) {
        acc0 += (uint64_t)r[m] * crt_limb(m, 0);
        acc1 += (uint64_t)r[m] * crt_limb(m, 1);
        acc2 += (uint64_t)r[m] * crt_limb(m, 2);
        acc3 += (uint64_t)r[m] * crt_limb(m, 3);
    }
    typedef unsigned __int128 u128;
    typedef __int128 i128;
    const u128 sum = (u128)acc0 + ((u128)acc1 << 32) + ((u128)acc2 << 64) + ((u128)acc3 << 96);  // < 2^122
    const u128 P = ((u128)P_HI << 64) | P_LO, half = ((u128)HALF_HI << 64) | HALF_LO;
    const uint32_t q = (uint32_t)((double)(uint64_t)(sum >> 58) * INV_P58);  // floor(sum / P) or one less
    i128 v = (i128)(sum - (u128)q * P);
    if (v < 0) v += (i128)P;
    if (v >= (i128)P) v -= (i128)P;
    if (v > (i128)half) v -= (i128)P;
    const bool neg = v < 0;
    const u128 a = neg ? (u128)(-v) : (u128)v;  // < 2^110
    const uint64_t hi = (uint64_t)(a >> 64), lo = (uint64_t)a;
    double d;
    int sh = 0;
    if (hi == 0) {
        d = __ull2double_rn(lo);
    } else {  // top 64 bits with a sticky bit: a single rounding to 53 bits
        sh = 64 - __clzll((long long)hi);
        const uint64_t mant = (uint64_t)(a >> sh) | ((lo & ((1ull << sh) - 1)) != 0 ? 1ull : 0ull);
        d = __ull2double_rn(mant);
    }
    d *= __longlong_as_double((long long)(1023 + sh - e) << 52);  // exact: |sh - e| <= 2 E_CLAMP + 64
    return neg ? -d : d;
}

// grid (lower 128-tiles, 1, batch), 256 threads; 4 consecutive columns per item
__global__ void __launch_bounds__(256) k_oz_merge(double* __restrict__ C, long mstride, int np, const unsigned char* __restrict__ ws,
                                                  size_t slot) {
    int mt, nt;
    lower_tile(blockIdx.x, mt, nt);
    const int b = blockIdx.z, tnum = (np + TB - 1) / TB;
    const long nr = (long)tnum * (tnum + 1) / 2;
    const unsigned char* wsb = ws + (size_t)b * slot;
    const unsigned char* res = wsb + ((size_t)S * nr + blockIdx.x) * TILE_BYTES;
    const int* ex = reinterpret_cast<const int*>(wsb + 2 * (size_t)S * nr * TILE_BYTES);
    double* Cb = C + (long)b * mstride;
    for (int it = threadIdx.x; it < TB * TB / 4; it += 256) {
        const int row = it >> 5, c4 = (it & 31) * 4;
        const int gi = mt * TB + row, gj = nt * TB + c4;
        if (gi >= np || gj >= np) continue;                         // np is a multiple of 64: all four in or out
        if (mt == nt && (row >> 6) < (c4 >> 6)) continue;          // upper 64 x 64 block of a diagonal tile
        uint32_t w[S];
#pragma unroll
        for (int m = 0; m < S; m++) w[m] = *reinterpret_cast<const uint32_t*>(res + (size_t)m * nr * TILE_BYTES + row * TB + c4);
        const int ei = ex[gi];
        const int4 ej = *reinterpret_cast<const int4*>(ex + gj);
        const int ejs[4] = {ej.x, ej.y, ej.z, ej.w};
        double out[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            uint32_t r[S];
#pragma unroll
            for (int m = 0; m < S; m++) r[m] = (w[m] >> (8 * q)) & 0xffu;
            out[q] = (ei == E_BAD || ejs[q] == E_BAD) ? __longlong_as_double(0x7ff8000000000000ll) : crt_value(r, ei + ejs[q]);
        }
        double2* dst = reinterpret_cast<double2*>(Cb + (long)gi * np + gj);
        dst[0] = make_double2(out[0], out[1]);
        dst[1] = make_double2(out[2], out[3]);
    }
}

// ---- host side -------------------------------------------------------------------------------------------------
inline cudaError_t configure() {
    return cudaFuncSetAttribute(k_oz_syrk_i8, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES);
}

// K^-1 = W^T W on the lower 64 x 64 tiles of C for `cnt` matrices (stride mstride, leading dimension np), with
// `ws` the workspace of the first of them (slot_bytes(np) per matrix).  Four launches.
inline cudaError_t launch_kinv(const double* W, double* C, long mstride, int np, int cnt, unsigned char* ws, cudaStream_t st) {
    if (cnt <= 0) return cudaSuccess;
    const int tn = (np + TB - 1) / TB;
    const size_t slot = slot_bytes(np);
    k_oz_colexp<<<dim3(tn, 1, cnt), 512, 0, st>>>(W, mstride, np, scale_bits(np), ws, slot);
    k_oz_split<<<dim3((unsigned)ntri(np), 1, cnt), 256, 0, st>>>(W, mstride, np, ws, slot);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    SyrkParams p;
    p.ws = ws;
    p.slot = slot;
    p.nt = tn;
    p.slot_tiles = (int)(slot / TILE_BYTES);
    EncodeTiledFn enc = encode_fn();
    if (!enc) return cudaErrorNotSupported;
    cuuint64_t dims[3] = {(cuuint64_t)TB, (cuuint64_t)TB, (cuuint64_t)p.slot_tiles * cnt};
    cuuint64_t strides[2] = {(cuuint64_t)TB, (cuuint64_t)TILE_BYTES};
    cuuint32_t box[3] = {(cuuint32_t)TB, (cuuint32_t)TB, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    if (enc(&p.map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, ws, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return cudaErrorNotSupported;
    k_oz_syrk_i8<<<dim3((unsigned)ntri(np), S, cnt), THREADS, SMEM_BYTES, st>>>(p);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    k_oz_merge<<<dim3((unsigned)ntri(np), 1, cnt), 256, 0, st>>>(C, mstride, np, ws, slot);
    return cudaGetLastError();
}

}  // namespace oz
}  // namespace hbegp
