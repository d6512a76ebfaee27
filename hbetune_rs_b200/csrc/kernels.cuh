// Non-GEMM kernels of the GP hot path (sm_100a): kernel-matrix assembly, the 64x64 Cholesky+inverse
// leaf, triangular matrix-vector products, the fused LML-gradient contraction, the reductions that
// finish an evaluation, and the prediction kernels.  All matrices are row-major with leading dimension
// Np = n rounded up to a multiple of 64; the padding block is the identity, which keeps every tile full
// (Cholesky, inverse and log-determinant of diag(K, I) are those of K).
#pragma once
#include <cuda_runtime.h>
#include <math.h>

namespace hbegp {

constexpr int TILE = 64;  // leaf / tile edge
// Feature chunk of the kernels that stage d x 64 operand tiles in shared memory (assembly, gradient contraction, k*):
// up to this many features are staged at once, more are processed in chunks of this size (same left-to-right
// accumulation order), so d is unbounded and the shared-memory footprint is not.
constexpr int kFeatChunk = 64;
__host__ __device__ inline int feat_chunk(int d) { return d < kFeatChunk ? d : kFeatChunk; }

// `ulps_eq!(std, 0.0)` of expected_improvement (src/core/acquisition.rs:148): approx 0.3 tests abs_diff_eq with
// epsilon = f64::EPSILON first, so any |std| <= 2.2e-16 takes the trivial branch (the ULP test that follows can only
// add denormals, which the first test already covers).  Shared by the host adapter and k_acquisition.
__host__ __device__ inline bool ei_std_is_zero(double sd) { return sd <= 0.0 || fabs(sd) <= 2.220446049250313e-16; }

// Per-evaluation hyper-parameters, already clamped and rounded to T on the host
// (src/gpr/fit.rs:94-96): prm[0] = noise, prm[1] = c, prm[2 + k] = l_k.
template <typename T>
__device__ __forceinline__ T dev_exp(T x);
template <>
__device__ __forceinline__ double dev_exp<double>(double x) { return exp(x); }
template <>
__device__ __forceinline__ float dev_exp<float>(float x) { return expf(x); }
template <typename T>
__device__ __forceinline__ T dev_sqrt(T x);
template <>
__device__ __forceinline__ double dev_sqrt<double>(double x) { return sqrt(x); }
template <>
__device__ __forceinline__ float dev_sqrt<float>(float x) { return sqrtf(x); }
template <typename T>
__device__ __forceinline__ T dev_log(T x);
template <>
__device__ __forceinline__ double dev_log<double>(double x) { return log(x); }
template <>
__device__ __forceinline__ float dev_log<float>(float x) { return logf(x); }

// Matern correlation from the scaled distance r (src/gpr/matern_kernel.rs:65-80).  NU2 = 2 * nu.
template <typename T, int NU2>
__device__ __forceinline__ T matern_corr(T r) {
    if (NU2 == 1) return dev_exp<T>(-r);
    if (NU2 == 3) {
        T k = r * T(1.7320508075688772935);
        return (k + T(1)) * dev_exp<T>(-k);
    }
    T k = r * T(2.2360679774997896964);
    return (T(1) + k + k * k / T(3)) * dev_exp<T>(-k);
}

// Per-entry terms of the theta gradient (src/gpr/matern_kernel.rs:83-135) from s = sum_k d_ijk,
// d_ijk = (x_ik - x_jk)^2 / l_k^2: kval = the correlation recomputed from t = sqrt(2 nu s), and dk_factor such that
// dM_ij / d ln l_k = dk_factor * d_ijk.
template <typename T, int NU2>
__device__ __forceinline__ void matern_grad_terms(T s, T& kval, T& dk_factor) {
    if (NU2 == 5) {
        const T t = dev_sqrt<T>(T(5) * s);
        const T e = dev_exp<T>(-t);
        kval = (T(1) + t + t * t / T(3)) * e;
        dk_factor = e * (t + T(1)) * T(5.0 / 3.0);  // matern_kernel.rs:120-130
    } else if (NU2 == 3) {
        const T t = dev_sqrt<T>(T(3) * s);
        const T e = dev_exp<T>(-t);
        kval = (t + T(1)) * e;
        dk_factor = T(3) * e;  // matern_kernel.rs:112-118
    } else {
        const T r = dev_sqrt<T>(s);
        kval = dev_exp<T>(-r);
        dk_factor = (r > T(0)) ? kval / r : T(0);  // matern_kernel.rs:102-111 (non-finite -> 0)
    }
}

// lower-triangle tile enumeration: t -> (mt >= nt)
__device__ __forceinline__ void lower_tile(int t, int& mt, int& nt) {
    int r = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
    while ((long)(r + 1) * (r + 2) / 2 <= t) ++r;
    while ((long)r * (r + 1) / 2 > t) --r;
    mt = r;
    nt = t - r * (r + 1) / 2;
}

// xsT[b][k][i] = x[i][k] / l_k (division first, matern_kernel.rs:51-60); rows i >= n are zero.
template <typename T>
__global__ void k_scale_x(const T* __restrict__ x, int n, int d, int np, const T* __restrict__ prm, int pstride,
                          T* __restrict__ xsT) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int k = blockIdx.y, b = blockIdx.z;
    if (i >= np) return;
    T l = prm[(long)b * pstride + 2 + k];
    T v = (i < n) ? x[(long)i * d + k] / l : T(0);
    xsT[((long)b * d + k) * np + i] = v;
}

// Number of scaled training inputs that differ between two models' X^T buffers (first `cols` points): an
// append (model_extend) is only valid when the old rows are an unchanged prefix of the new data.
template <typename T>
__global__ void k_prefix_mismatch(const T* __restrict__ a, int lda, const T* __restrict__ b, int ldb, int d, int cols,
                                  int* __restrict__ count) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int k = blockIdx.y;
    if (i >= cols) return;
    if (!(a[(long)k * lda + i] == b[(long)k * ldb + i])) atomicAdd(count, 1);
}

// K = c * matern(|xs_i - xs_j|) + noise * I on the lower tiles (diagonal tiles written in full).
template <typename T, int NU2>
__global__ void __launch_bounds__(256) k_assemble(const T* __restrict__ xsT, int n, int d, int np,
                                                  const T* __restrict__ prm, int pstride, T* __restrict__ K,
                                                  long kstride, int tile0) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int dc = feat_chunk(d);
    T* xi = reinterpret_cast<T*>(smem_raw);  // [dc][64]
    T* xj = xi + dc * TILE;
    int mt, nt;
    lower_tile(blockIdx.x + tile0, mt, nt);  // tile0 > 0: only the tile rows an append adds (model_extend)
    const int b = blockIdx.z;
    const int i0 = mt * TILE, j0 = nt * TILE;
    const T* xb = xsT + (long)b * d * np;
    const T noise = prm[(long)b * pstride + 0], c = prm[(long)b * pstride + 1];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    T acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int q = 0; q < 4; q++) acc[a][q] = T(0);
    for (int c0 = 0; c0 < d; c0 += dc) {
        const int dl = min(dc, d - c0);
        if (c0 > 0) __syncthreads();  // the previous chunk has been consumed
        for (int e = threadIdx.x; e < dl * TILE; e += 256) {
            int k = e / TILE, r = e % TILE;
            xi[e] = xb[(long)(c0 + k) * np + i0 + r];
            xj[e] = xb[(long)(c0 + k) * np + j0 + r];
        }
        __syncthreads();
        for (int k = 0; k < dl; k++) {
            T vi[4], vj[4];
#pragma unroll
            for (int a = 0; a < 4; a++) vi[a] = xi[k * TILE + ty + 16 * a];
#pragma unroll
            for (int q = 0; q < 4; q++) vj[q] = xj[k * TILE + tx + 16 * q];
#pragma unroll
            for (int a = 0; a < 4; a++)
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    T df = vi[a] - vj[q];
                    acc[a][q] += df * df;
                }
        }
    }
    T* Kb = K + (long)b * kstride;
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int q = 0; q < 4; q++) {
            int gi = i0 + ty + 16 * a, gj = j0 + tx + 16 * q;
            T v;
            if (gi >= n || gj >= n) v = (gi == gj) ? T(1) : T(0);
            else {
                v = c * matern_corr<T, NU2>(dev_sqrt<T>(acc[a][q]));
                if (gi == gj) v += noise;
            }
            Kb[(long)gi * np + gj] = v;
        }
}

// Reciprocal of a Cholesky pivot.  It sits on the 64-step critical path of the leaf, where an IEEE FP64
// division costs ~8 dependent FP64 operations plus a slow-path branch; the hardware seed (rcp.approx.ftz.f64,
// ~20 bits) plus two Newton steps (4 dependent DFMAs, relative error ~2^-52) halves that.
template <typename T>
__device__ __forceinline__ T pivot_rcp(T d);
template <>
__device__ __forceinline__ float pivot_rcp<float>(float d) { return 1.0f / d; }
template <>
__device__ __forceinline__ double pivot_rcp<double>(double d) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));  // MUFU.RCP64H: ~20 bits, full exponent range
    double e = fma(-d, r, 1.0);
    r = fma(r, e, r);
    e = fma(-d, r, 1.0);
    r = fma(r, e, r);
    return r;
}

// Leaf of the recursive factorisation: 64x64 diagonal block at (r0, r0).  In: A block (lower part).
// Out: W = L^-1 as a full tile (zeros above the diagonal) in the W buffer (L itself is not needed again: the
// parent nodes solve their panels with W), sum_i ln L_ii in ldp[b][leaf], status[b] = 1 when a pivot is not
// positive (lml.rs:47-50).
//
// The 64 pivots are inherently sequential and each step costs a barrier, a shared-memory round trip and an FP64
// reciprocal, so the kernel keeps the per-pivot work minimal (blocked with nb = 16):
//  * Cholesky on unscaled columns u_ij = L_ij L_jj (u_ik -= u_ij u_kj / u_jj): a pivot step only updates the
//    remaining columns of its 16-wide panel (<= 4 cells per thread); the rest of the matrix gets one rank-16
//    update per panel.  No square root on the pivot chain: 1 / L_jj = rsqrt(u_jj) for all j at the end.
//  * inverse: the four 16x16 diagonal blocks are inverted side by side (15 steps instead of 63), the off-diagonal
//    blocks follow by block forward substitution W_PQ = -W_PP sum_R L_PR W_RQ (three levels of small products).
// A variant with 8-wide register-resident panels (one barrier pair per panel instead of one barrier per pivot) measured
// no faster in either precision: the gain needs the DMMA products and the transposed layout of node_mma.cuh.
template <typename T>
__host__ __device__ constexpr size_t leaf_tile_bytes() { return sizeof(T) * TILE * (TILE + 1); }
template <typename T>
constexpr size_t leaf_smem_bytes() { return 2 * leaf_tile_bytes<T>() + 2 * TILE * sizeof(T); }

// The leaf on shared memory.  In: as = the 64x64 block (lower part, zeros above).  Out: ws = L^-1 (zeros above the
// diagonal), dinv[i] = 1 / L_ii; *fail = 1 when a pivot is not positive.  Ends with a barrier.  `as` is scratch after.
template <typename T>
__device__ __forceinline__ void leaf_core(T (*as)[TILE + 1], T (*ws)[TILE + 1], T* rdv, T* dinv, int* fail, int tid) {
    const int tx = tid & 15, ty = tid >> 4;
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int i = ty + 16 * a, k = tx + 16 * q;
            ws[i][k] = (i == k) ? T(1) : T(0);
        }
    // ---- blocked Cholesky (nb = 16) on unscaled columns
    const int pi = tid >> 2, pq = tid & 3;  // panel phase: row pi, panel columns pq, pq + 4, pq + 8, pq + 12
    for (int P = 0; P < 4; P++) {
        const int c0 = 16 * P;
        __syncthreads();
        T pv[4];
#pragma unroll
        for (int t = 0; t < 4; t++) pv[t] = as[pi][c0 + pq + 4 * t];
#pragma unroll
        for (int jj = 0; jj < 16; jj++) {
            const int j = c0 + jj;
            if (jj > 0) {
                // column j is final after step j - 1: its owners publish it for this step
                if (pq == (jj & 3)) as[pi][j] = pv[jj >> 2];
                __syncthreads();
            }
            T dj = as[j][j];
            const T uij = as[pi][j];
            T ukj[4];
#pragma unroll
            for (int t = jj >> 2; t < 4; t++) ukj[t] = as[c0 + pq + 4 * t][j];
            if (!(dj > T(0)) || !(dj <= T(1e300))) {
                if (tid == 0) *fail = 1;
                dj = T(1);
            }
            const T rd = pivot_rcp<T>(dj);
            if (tid == 0) rdv[j] = rd;
            const T li = uij * rd;
#pragma unroll
            for (int t = jj >> 2; t < 4; t++) {
                const int k = pq + 4 * t;  // panel-relative column
                if (k > jj && c0 + k <= pi) pv[t] = fma(-li, ukj[t], pv[t]);
            }
        }
        __syncthreads();
        // rank-16 update of everything right of the panel: u_ik -= sum_{j in panel} u_ij u_kj / u_jj
#pragma unroll
        for (int q = 1; q < 4; q++) {
            if (q > P) {
                T lk[16];
#pragma unroll
                for (int jj = 0; jj < 16; jj++) lk[jj] = as[tx + 16 * q][c0 + jj] * rdv[c0 + jj];
#pragma unroll
                for (int a = 1; a < 4; a++) {
                    if (a >= q) {
                        const int i = ty + 16 * a, k = tx + 16 * q;
                        T acc = T(0);
#pragma unroll
                        for (int jj = 0; jj < 16; jj++) acc = fma(as[i][c0 + jj], lk[jj], acc);
                        if (k <= i) as[i][k] -= acc;
                    }
                }
            }
        }
    }
    __syncthreads();
    if (tid < TILE) {
        T dj = as[tid][tid];
        if (!(dj > T(0)) || !(dj <= T(1e300))) dj = T(1);
        dinv[tid] = T(1) / dev_sqrt<T>(dj);
    }
    // ---- inverse of the four 16x16 diagonal blocks, side by side (rows unscaled: W_true = W_u * dinv_row)
    const int P = tid >> 6, r = (tid & 63) >> 2, cq = tid & 3, c0 = 16 * P;
    for (int kk = 0; kk < 15; kk++) {
        __syncthreads();
        if (r > kk) {
            const T lik = as[c0 + r][c0 + kk] * rdv[c0 + kk];  // L_ik / L_kk = u_ik / u_kk
            for (int c = cq; c <= kk; c += 4) ws[c0 + r][c0 + c] = fma(-lik, ws[c0 + kk][c0 + c], ws[c0 + r][c0 + c]);
        }
    }
    __syncthreads();
    {
        const int i = c0 + r;
        for (int c = cq; c <= r; c += 4) ws[i][c0 + c] *= dinv[i];
    }
    // ---- off-diagonal blocks by block forward substitution; S_PQ goes to the free upper part of `as`
    const int sr = tid >> 4, sc = tid & 15;
    for (int PP = 1; PP < 4; PP++) {
        __syncthreads();
        for (int Q = 0; Q < PP; Q++) {
            T acc = T(0);
            for (int k = 16 * Q; k < 16 * PP; k++) acc = fma(as[16 * PP + sr][k] * dinv[k], ws[k][16 * Q + sc], acc);
            as[16 * Q + sr][16 * PP + sc] = acc;  // S_PQ (strictly upper position: Q < PP)
        }
        __syncthreads();
        for (int Q = 0; Q < PP; Q++) {
            T acc = T(0);
            for (int k = 0; k <= sr; k++) acc = fma(ws[16 * PP + sr][16 * PP + k], as[16 * Q + k][16 * PP + sc], acc);
            ws[16 * PP + sr][16 * Q + sc] = -acc;
        }
    }
    __syncthreads();
}

// sum_i ln L_ii of a leaf (first warp), from dinv
template <typename T>
__device__ __forceinline__ void leaf_logdet(const T* dinv, int tid, T* out) {
    if (tid < 32) {
        T s = T(0);
        for (int i = tid; i < TILE; i += 32) s += -dev_log<T>(dinv[i]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (tid == 0) *out = s;
    }
}

template <typename T>
__global__ void __launch_bounds__(256) k_leaf(T* __restrict__ A, T* __restrict__ W, long mstride, int np, int r0,
                                              T* __restrict__ ldp, int ldp_stride, int* __restrict__ status) {
    extern __shared__ __align__(16) unsigned char leaf_smem_raw[];
    typedef T Row[TILE + 1];
    Row* as = reinterpret_cast<Row*>(leaf_smem_raw);                              // u (lower); scratch (upper)
    Row* ws = reinterpret_cast<Row*>(leaf_smem_raw + leaf_tile_bytes<T>());      // W = L^-1
    T* rdv = reinterpret_cast<T*>(leaf_smem_raw + 2 * leaf_tile_bytes<T>());     // 1 / u_jj
    T* dinv = rdv + TILE;                                                         // 1 / L_jj
    __shared__ int fail;
    const int b = blockIdx.z, tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    T* Ab = A + (long)b * mstride + (long)r0 * np + r0;
    T* Wb = W + (long)b * mstride + (long)r0 * np + r0;
    if (tid == 0) fail = 0;
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int i = ty + 16 * a, k = tx + 16 * q;
            as[i][k] = (k <= i) ? Ab[(long)i * np + k] : T(0);
        }
    leaf_core<T>(as, ws, rdv, dinv, &fail, tid);
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int i = ty + 16 * a, k = tx + 16 * q;
            Wb[(long)i * np + k] = (k <= i) ? ws[i][k] : T(0);
        }
    leaf_logdet<T>(dinv, tid, ldp + (long)b * ldp_stride + r0 / TILE);
    if (tid == 0 && fail) status[b] = 1;
}

// u[i] = sum_{k <= i} W[i][k] v[k]   (one warp per row)
template <typename T>
__global__ void __launch_bounds__(256) k_trmv_lower(const T* __restrict__ W, long mstride, int np,
                                                    const T* __restrict__ v, long vstride, T* __restrict__ u,
                                                    long ustride) {
    const int b = blockIdx.z;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= np) return;
    const T* wr = W + (long)b * mstride + (long)row * np;
    const T* vb = v + (long)b * vstride;
    T s = T(0);
    for (int k = lane; k <= row; k += 32) s += wr[k] * vb[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) u[(long)b * ustride + row] = s;
}

// part[b][rc][j] = sum over rows i of chunk rc (256 rows), i >= j, of W[i][j] u[i]
template <typename T>
__global__ void __launch_bounds__(256) k_trmv_lower_t_part(const T* __restrict__ W, long mstride, int np,
                                                           const T* __restrict__ u, long ustride,
                                                           T* __restrict__ part, int nchunks) {
    __shared__ T red[4][TILE];
    const int b = blockIdx.z, jb = blockIdx.x, rc = blockIdx.y;
    const int tx = threadIdx.x & 63, ph = threadIdx.x >> 6;
    const int j = jb * TILE + tx;
    const int rbeg = rc * 256, rend = min(np, rbeg + 256);
    T s = T(0);
    if (rend > jb * TILE) {
        const T* Wb = W + (long)b * mstride;
        const T* ub = u + (long)b * ustride;
        for (int i = max(rbeg, jb * TILE) + ph; i < rend; i += 4)
            if (i >= j) s += Wb[(long)i * np + j] * ub[i];
    }
    red[ph][tx] = s;
    __syncthreads();
    if (ph == 0) part[((long)b * nchunks + rc) * np + j] = ((red[0][tx] + red[1][tx]) + red[2][tx]) + red[3][tx];
}

template <typename T>
__global__ void k_sum_chunks(const T* __restrict__ part, int nchunks, int np, T* __restrict__ out, long ostride) {
    const int b = blockIdx.z;
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= np) return;
    T s = T(0);
    for (int c = j / 256; c < nchunks; c++) s += part[((long)b * nchunks + c) * np + j];
    out[(long)b * ostride + j] = s;
}

// Fused LML-gradient contraction over one lower 64x64 tile of K^-1 (never materialises the (n, n, d+1)
// tensor of src/gpr/matern_kernel.rs:83-135 / product_kernel.rs:40-70):
//   g_k = 1/2 sum_ij (alpha_i alpha_j - Kinv_ij) G_ijk,   k = noise, c, l_1..l_d   (lml.rs:61-71)
// gpart[b][tile][0..p) receives this tile's contribution (symmetry: off-diagonal cells count twice).
#ifndef HBEGP_GRAD_MINBLOCKS
#define HBEGP_GRAD_MINBLOCKS 4  // 64 registers, 4 CTAs per SM: 6.8 -> 6.0 ms at the north-star shape (probes/grad_ab.py); the FP64 pipe bounds it
#endif
template <typename T, int NU2>
__global__ void __launch_bounds__(256, HBEGP_GRAD_MINBLOCKS) k_grad_contract(const T* __restrict__ Kinv, long mstride, int n, int d,
                                                       int np, const T* __restrict__ xsT,
                                                       const T* __restrict__ alpha, long astride,
                                                       const T* __restrict__ prm, int pstride,
                                                       double* __restrict__ gpart, long gp_bstride) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int dc = feat_chunk(d);
    T* xi = reinterpret_cast<T*>(smem_raw);  // [dc][64]
    T* xj = xi + dc * TILE;                  // [dc][64]
    T* ai = xj + dc * TILE;                  // [64]
    T* aj = ai + TILE;                       // [64]
    double* wsum = reinterpret_cast<double*>(aj + TILE);  // [8][dc + 2]: per-warp partials of one feature chunk (+ noise, c)
    const int p = d + 2, ws = dc + 2;
    int mt, nt;
    lower_tile(blockIdx.x, mt, nt);
    const int b = blockIdx.z, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int i0 = mt * TILE, j0 = nt * TILE;
    const T* xb = xsT + (long)b * d * np;
    auto load_chunk = [&](int c0, int dl) {
        for (int e = tid; e < dl * TILE; e += 256) {
            int k = e / TILE, r = e % TILE;
            xi[e] = xb[(long)(c0 + k) * np + i0 + r];
            xj[e] = xb[(long)(c0 + k) * np + j0 + r];
        }
    };
    if (tid < TILE) ai[tid] = alpha[(long)b * astride + i0 + tid];
    else if (tid < 2 * TILE) aj[tid - TILE] = alpha[(long)b * astride + j0 + tid - TILE];
    const int tx = tid & 15, ty = tid >> 4;
    const T* Kb = Kinv + (long)b * mstride;
    // the 16 K^-1 entries of this thread, requested up front so that their DRAM latency hides behind the shared
    // memory fill and the distance loop (ncu: long_scoreboard was the top stall with the loads at the point of use)
    T kv[16];
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int q = 0; q < 4; q++) kv[a * 4 + q] = Kb[(long)(i0 + ty + 16 * a) * np + j0 + tx + 16 * q];
    const T noise = prm[(long)b * pstride + 0], c = prm[(long)b * pstride + 1];
    T cm[16];
    double g_noise = 0.0, g_c = 0.0;
    {
        T S[16];
#pragma unroll
        for (int e = 0; e < 16; e++) S[e] = T(0);
        for (int c0 = 0; c0 < d; c0 += dc) {  // squared scaled distances, feature chunk by feature chunk
            const int dl = min(dc, d - c0);
            if (c0 > 0) __syncthreads();
            load_chunk(c0, dl);
            __syncthreads();
            for (int k = 0; k < dl; k++) {
                T vi[4], vj[4];
#pragma unroll
                for (int a = 0; a < 4; a++) vi[a] = xi[k * TILE + ty + 16 * a];
#pragma unroll
                for (int q = 0; q < 4; q++) vj[q] = xj[k * TILE + tx + 16 * q];
#pragma unroll
                for (int a = 0; a < 4; a++)
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        T df = vi[a] - vj[q];
                        S[a * 4 + q] += df * df;
                    }
            }
        }
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int li = ty + 16 * a, lj = tx + 16 * q;
                const int gi = i0 + li, gj = j0 + lj;
                T wgt = T(2);
                if (mt == nt) wgt = (li > lj) ? T(2) : ((li == lj) ? T(1) : T(0));
                if (gi >= n || gj >= n) wgt = T(0);
                const T tij = ai[li] * aj[lj] - kv[a * 4 + q];
                const T s = S[a * 4 + q];
                T base, dk_factor, kval;
                matern_grad_terms<T, NU2>(s, kval, dk_factor);
                base = wgt * tij * c;
                cm[a * 4 + q] = base * dk_factor;
                g_c += (double)(base * kval);
                if (gi == gj) g_noise += (double)(wgt * tij * noise);
            }
    }
    // block-level deterministic reduction: warp shuffle, then warps in order
    auto warp_sum = [&](double v) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        return v;
    };
    g_noise = warp_sum(g_noise);
    g_c = warp_sum(g_c);
    if (lane == 0) {
        wsum[warp * ws + dc] = g_noise;
        wsum[warp * ws + dc + 1] = g_c;
    }
    double* gout = gpart + (long)b * gp_bstride + (long)blockIdx.x * p;
    for (int c0 = 0; c0 < d; c0 += dc) {
        const int dl = min(dc, d - c0);
        if (d > dc) {  // more than one chunk: the tiles of chunk c0 have to come back (a single chunk is still there)
            __syncthreads();
            load_chunk(c0, dl);
            __syncthreads();
        }
        for (int k = 0; k < dl; k++) {
            T vi[4], vj[4];
#pragma unroll
            for (int a = 0; a < 4; a++) vi[a] = xi[k * TILE + ty + 16 * a];
#pragma unroll
            for (int q = 0; q < 4; q++) vj[q] = xj[k * TILE + tx + 16 * q];
            T acc = T(0);
#pragma unroll
            for (int a = 0; a < 4; a++)
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    T df = vi[a] - vj[q];
                    acc += cm[a * 4 + q] * (df * df);
                }
            double v = warp_sum((double)acc);
            if (lane == 0) wsum[warp * ws + k] = v;
        }
        __syncthreads();
        if (tid < dl) {
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < 8; w++) s += wsum[w * ws + tid];
            gout[2 + c0 + tid] = 0.5 * s;
        }
        if (c0 == 0 && tid >= 64 && tid < 66) {  // noise and amplitude components, once
            const int which = tid - 64;
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < 8; w++) s += wsum[w * ws + dc + which];
            gout[which] = 0.5 * s;
        }
    }
}

// Finishes one evaluation: lml = -1/2 y.alpha - sum ln L_ii - n/2 ln 2pi (lml.rs:57-59) and the sum of the
// per-tile gradient partials in tile order.  One CTA per batch element.
template <typename T>
__global__ void __launch_bounds__(256) k_finish(const T* __restrict__ y, const T* __restrict__ alpha, long astride,
                                                int n, int np, const T* __restrict__ ldp, int ldp_stride,
                                                const double* __restrict__ gpart, long gp_bstride, int ntiles,
                                                int p, const int* __restrict__ status, double* __restrict__ lml,
                                                double* __restrict__ grad, int want_grad) {
    __shared__ double red[256];
    const int b = blockIdx.x, tid = threadIdx.x;
    const bool bad = status[b] != 0;
    double s = 0.0;
    for (int i = tid; i < n; i += 256) s += (double)(y[i] * alpha[(long)b * astride + i]);
    red[tid] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (tid < o) red[tid] += red[tid + o];
        __syncthreads();
    }
    const double ya = red[0];
    __syncthreads();
    s = 0.0;
    for (int i = tid; i < np / TILE; i += 256) s += (double)ldp[(long)b * ldp_stride + i];
    red[tid] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (tid < o) red[tid] += red[tid + o];
        __syncthreads();
    }
    if (tid == 0) {
        double v = -0.5 * ya - red[0] - 0.5 * (double)n * 1.8378770664093454836;  // ln(2 pi)
        if (bad || !(v == v)) v = -INFINITY;
        lml[b] = v;
    }
    if (!want_grad) return;
    // gradient: p columns; thread groups of (256 / p') walk the tiles with a fixed stride
    const bool isbad = bad;
    for (int k = 0; k < p; k++) {
        __syncthreads();
        double acc = 0.0;
        for (int t = tid; t < ntiles; t += 256) acc += gpart[(long)b * gp_bstride + (long)t * p + k];
        red[tid] = acc;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if (tid < o) red[tid] += red[tid + o];
            __syncthreads();
        }
        if (tid == 0) grad[(long)b * p + k] = isbad ? 0.0 : red[0];
    }
}

// ------------------------------------------------------------------------------------------- predict
// Cross-kernel tile rows: for 64 candidates per CTA, k*[r][j] = c * matern(|xs_r / l - xsT_j|) over all
// train columns, mean[r] = sum_j k*[r][j] alpha[j] (src/gpr/predict.rs:18-19).  k* is written out
// (leading dimension np, zero in the padding columns) only when kstar != nullptr.
template <typename T, int NU2>
__global__ void __launch_bounds__(256) k_kstar_mean(const T* __restrict__ xs, long m, long row0, int d,
                                                    const T* __restrict__ xsT_train, int n, int np,
                                                    const T* __restrict__ ls, T c, const T* __restrict__ alpha,
                                                    T* __restrict__ kstar, T* __restrict__ mean, int tiles_per_cta,
                                                    T* __restrict__ pmean, long pm_stride) {
    // grid.y splits the train tiles when there are too few candidate tiles to fill the GPU; the partial means of
    // split y go to pmean[y * pm_stride + chunk_row] and are summed in order by k_var_finish.
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int dc = feat_chunk(d);
    T* xc = reinterpret_cast<T*>(smem_raw);  // [dc][64] candidates (scaled)
    T* xt = xc + dc * TILE;                  // [dc][64] train tile
    T* al = xt + dc * TILE;                  // [64]
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const long r0 = (long)blockIdx.x * TILE;  // row within the chunk
    auto load_candidates = [&](int c0, int dl) {
        for (int e = tid; e < dl * TILE; e += 256) {
            int r = e / dl, k = e % dl;  // (nearly) coalesced read of the row-major candidates
            long gr = row0 + r0 + r;
            xc[k * TILE + r] = (gr < m) ? xs[gr * d + c0 + k] / ls[c0 + k] : T(0);
        }
    };
    if (d <= dc) load_candidates(0, d);  // one chunk: the candidate tile stays for all train tiles
    T macc[4] = {T(0), T(0), T(0), T(0)};
    const int jbeg = blockIdx.y * tiles_per_cta * TILE, jend = min(np, jbeg + tiles_per_cta * TILE);
    for (int j0 = jbeg; j0 < jend; j0 += TILE) {
        T acc[4][4];
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int q = 0; q < 4; q++) acc[a][q] = T(0);
        for (int c0 = 0; c0 < d; c0 += dc) {
            const int dl = min(dc, d - c0);
            __syncthreads();
            for (int e = tid; e < dl * TILE; e += 256) {
                int k = e / TILE, r = e % TILE;
                xt[e] = xsT_train[(long)(c0 + k) * np + j0 + r];
            }
            if (d > dc) load_candidates(c0, dl);
            if (c0 == 0 && tid < TILE) al[tid] = alpha[j0 + tid];
            __syncthreads();
            for (int k = 0; k < dl; k++) {
                T vi[4], vj[4];
#pragma unroll
                for (int a = 0; a < 4; a++) vi[a] = xc[k * TILE + ty + 16 * a];
#pragma unroll
                for (int q = 0; q < 4; q++) vj[q] = xt[k * TILE + tx + 16 * q];
#pragma unroll
                for (int a = 0; a < 4; a++)
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        T df = vi[a] - vj[q];
                        acc[a][q] += df * df;
                    }
            }
        }
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int gj = j0 + tx + 16 * q;
                T v = (gj < n) ? c * matern_corr<T, NU2>(dev_sqrt<T>(acc[a][q])) : T(0);
                macc[a] += v * al[tx + 16 * q];
                if (kstar != nullptr) kstar[(r0 + ty + 16 * a) * (long)np + gj] = v;
            }
    }
#pragma unroll
    for (int a = 0; a < 4; a++) {
        T v = macc[a];
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        long gr = row0 + r0 + ty + 16 * a;
        if (tx == 0) {
            if (pmean != nullptr) pmean[(long)blockIdx.y * pm_stride + r0 + ty + 16 * a] = v;
            else if (gr < m) mean[gr] = v;
        }
    }
}

// ---- small-batch prediction (m <= 64 candidates; the reference's callers predict ONE point per call,
// SURVEY F4).  The throughput path above loops one CTA over all train tiles per 64 candidates and pads the
// variance GEMM to 128 rows, which is latency bound for a handful of points (n = 4096, m = 1: 0.62 ms).  Here the
// parallelism comes from the train dimension instead: k* per train tile, then one warp per row of W = L^-1.

// k*[r][j] for train tile blockIdx.x and all m candidates; pmean[tile][r] = sum_{j in tile} k*[r][j] alpha[j].
template <typename T, int NU2>
__global__ void __launch_bounds__(256) k_kstar_small(const T* __restrict__ xs, int m, int d,
                                                     const T* __restrict__ xsT_train, int n, int np,
                                                     const T* __restrict__ ls, T c, const T* __restrict__ alpha,
                                                     T* __restrict__ kstar, T* __restrict__ pmean) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* xc = reinterpret_cast<T*>(smem_raw);  // [m][d] scaled candidates
    T* red = xc + (size_t)m * d;             // [8 warps][16 slots]
    const int tid = threadIdx.x, j = blockIdx.x * TILE + (tid & 63), g = tid >> 6, lane = tid & 31, warp = tid >> 5;
    for (int e = tid; e < m * d; e += 256) xc[e] = xs[e] / ls[e % d];
    __syncthreads();
    const T aj = alpha[j];
    for (int q = 0; q < 16; q++) {
        const int r = g + 4 * q;  // warp-uniform
        T contrib = T(0);
        if (r < m) {
            T acc = T(0);
            for (int k = 0; k < d; k++) {
                const T df = xc[r * d + k] - xsT_train[(long)k * np + j];
                acc += df * df;
            }
            const T v = (j < n) ? c * matern_corr<T, NU2>(dev_sqrt<T>(acc)) : T(0);
            if (kstar != nullptr) kstar[(long)r * np + j] = v;
            contrib = v * aj;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
        if (lane == 0) red[warp * 16 + q] = contrib;
    }
    __syncthreads();
    if (tid < 64) {
        const int r = tid;  // candidate r = g + 4 q was reduced by warps 2g and 2g + 1
        if (r < m) {
            const int gg = r & 3, q = r >> 2;
            pmean[(long)blockIdx.x * 64 + r] = red[(2 * gg) * 16 + q] + red[(2 * gg + 1) * 16 + q];
        }
    }
}

// One warp per row i of W: u_i[r] = sum_{k <= i} W[i][k] k*[r][k] for the 16 candidates of group blockIdx.y;
// psq[cta][r] = sum over the CTA's 8 rows of u_i[r]^2 (the predictive variance is c + 1e-5 - |W k*|^2).
template <typename T>
__global__ void __launch_bounds__(256) k_wmatvec_small(const T* __restrict__ W, int np, const T* __restrict__ kstar, int m,
                                                       T* __restrict__ psq) {
    __shared__ T red[8][16];
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int r0 = blockIdx.y * 16;
    const T* wr = W + (long)row * np;
    T acc[16];
#pragma unroll
    for (int q = 0; q < 16; q++) acc[q] = T(0);
    for (int k = lane; k <= row; k += 32) {
        const T wv = wr[k];
#pragma unroll
        for (int q = 0; q < 16; q++)
            if (r0 + q < m) acc[q] = fma(wv, kstar[(long)(r0 + q) * np + k], acc[q]);
    }
#pragma unroll
    for (int q = 0; q < 16; q++) {
        T v = acc[q];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[warp][q] = v * v;
    }
    __syncthreads();
    if (threadIdx.x < 16 && r0 + threadIdx.x < m) {
        T s = T(0);
#pragma unroll
        for (int w = 0; w < 8; w++) s += red[w][threadIdx.x];
        psq[(long)blockIdx.x * 64 + r0 + threadIdx.x] = s;
    }
}

// A variance below the warning level -sqrt(1e-5) (predict.rs:39-46, :104-127): counted, and the first `warn_cap`
// (row, value) pairs that arrive are kept so that the host can list them like the reference's stderr message.
template <typename T>
__device__ __forceinline__ void note_below(unsigned long long* n_below, long* warn_rows, T* warn_vals, int warn_cap, long row, T v) {
    const unsigned long long slot = atomicAdd(n_below, 1ULL);
    if (warn_rows != nullptr && slot < (unsigned long long)warn_cap) {
        warn_rows[slot] = row;
        warn_vals[slot] = v;
    }
}

// mean[r] = sum_tiles pmean[tile][r]; var[r] = c + 1e-5 - sum_ctas psq[cta][r] (counted / clamped like k_var_finish)
template <typename T>
__global__ void k_small_finish(const T* __restrict__ pmean, int ntiles, const T* __restrict__ psq, int nctas, int m, T c,
                               T* __restrict__ mean, T* __restrict__ var, unsigned long long* __restrict__ n_below,
                               long* __restrict__ warn_rows, T* __restrict__ warn_vals, int warn_cap) {
    const int r = threadIdx.x;
    if (r >= m) return;
    T s = T(0);
    for (int t = 0; t < ntiles; t++) s += pmean[(long)t * 64 + r];
    mean[r] = s;
    if (var == nullptr) return;
    T q = T(0);
    for (int t = 0; t < nctas; t++) q += psq[(long)t * 64 + r];
    const T min_noise = T(1e-5);
    T v = c + min_noise - q;
    if (v < -dev_sqrt<T>(min_noise)) note_below<T>(n_below, warn_rows, warn_vals, warn_cap, r, v);
    if (v < T(0)) v = T(0);
    var[r] = v;
}

// var[r] = c + 1e-5 - sum_t part[r][t]; counts values < -sqrt(1e-5) then clamps at 0
// (src/gpr/predict.rs:25-48, :104-127).
template <typename T>
__global__ void k_var_finish(const T* __restrict__ part, int ld, int ntiles, long rows, long m, long row0, T c,
                             T* __restrict__ var, unsigned long long* __restrict__ n_below,
                             const T* __restrict__ pmean, int nsplit, long pm_stride, T* __restrict__ mean,
                             long* __restrict__ warn_rows, T* __restrict__ warn_vals, int warn_cap) {
    long r = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows || row0 + r >= m) return;
    if (pmean != nullptr) {  // mean partials of the column-split k* kernel, summed in split order
        T mu = T(0);
        for (int y = 0; y < nsplit; y++) mu += pmean[(long)y * pm_stride + r];
        mean[row0 + r] = mu;
    }
    if (var == nullptr) return;
    T s = T(0);
    for (int t = 0; t < ntiles; t++) s += part[r * ld + t];
    const T min_noise = T(1e-5);
    T v = c + min_noise - s;
    if (v < -dev_sqrt<T>(min_noise)) note_below<T>(n_below, warn_rows, warn_vals, warn_cap, row0 + r, v);
    if (v < T(0)) v = T(0);
    var[row0 + r] = v;
}

template <typename T>
__device__ __forceinline__ T mul_rn(T a, T b);
template <>
__device__ __forceinline__ double mul_rn<double>(double a, double b) { return __dmul_rn(a, b); }
template <>
__device__ __forceinline__ float mul_rn<float>(float a, float b) { return __fmul_rn(a, b); }
template <typename T>
__device__ __forceinline__ T add_rn(T a, T b);
template <>
__device__ __forceinline__ double add_rn<double>(double a, double b) { return __dadd_rn(a, b); }
template <>
__device__ __forceinline__ float add_rn<float>(float a, float b) { return __fadd_rn(a, b); }

// Acquisition epilogues on the device (SURVEY section 8 rows f1/f2).
//   mode 0: predict_mean_ei_a (src/core/gpr.rs:179-212): out1 = de-normalised mean, out2 = EI in normalised
//           units, EI evaluated in f64 from (mean, sqrt(var)) like acquisition.rs:141-171;
//   mode 1: predict_confidence_bound (gpr.rs:94-112): out1 = location_from(mean + sqrt(var) * cb).
// proj: 0 linear, 1 logarithmic (ynormalize.rs:215-225).
template <typename T>
__global__ void k_acquisition(const T* __restrict__ mean, const T* __restrict__ var, long m, int mode, int proj,
                              T amplitude, T expected, double fmin_n, T cb, T* __restrict__ out1,
                              T* __restrict__ out2) {
    long r = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= m) return;
    const T mu = mean[r], sd = dev_sqrt<T>(var[r]);
    // un-fused multiply / add so that the result is bit-identical to the host-side YNorm<A>::location_from
    auto location_from = [&](T y) -> T {
        return proj == 0 ? add_rn<T>(mul_rn<T>(y - T(0.05), amplitude), expected)
                         : add_rn<T>(dev_exp<T>(mul_rn<T>(y, amplitude)), expected);
    };
    if (mode == 0) {
        const double mean_d = (double)mu, std_d = (double)sd;
        double ei;
        if (ei_std_is_zero(std_d)) {
            ei = mean_d < fmin_n ? -(mean_d - fmin_n) : 0.0;
        } else {
            const double z = -(mean_d - fmin_n) / std_d;
            const double cdf = 0.5 * erfc(-z * 0.70710678118654752440);
            const double pdf = exp(-0.5 * z * z) * 0.39894228040143267794;
            ei = -(mean_d - fmin_n) * cdf + std_d * pdf;
        }
        out1[r] = location_from(mu);
        out2[r] = (T)ei;
    } else {
        out1[r] = location_from(add_rn<T>(mu, mul_rn<T>(sd, cb)));
    }
}

// Arg-best over a vector in two deterministic stages.  want_max = 1: maximum, the LAST one wins ties
// (Iterator::max_by, acquisition.rs:192-200); want_max = 0: minimum, the FIRST one wins (strict `<`,
// minimize.rs:702-707).  NaNs never win.
template <typename T>
__global__ void __launch_bounds__(256) k_argbest_part(const T* __restrict__ v, long m, int want_max,
                                                      T* __restrict__ pv, long* __restrict__ pi) {
    __shared__ T sv[256];
    __shared__ long si[256];
    const long chunk = (m + gridDim.x - 1) / gridDim.x;
    const long lo = (long)blockIdx.x * chunk, hi = min(m, lo + chunk);
    T best = T(0);
    long bi = -1;
    for (long i = lo + threadIdx.x; i < hi; i += 256) {
        const T x = v[i];
        if (!(x == x)) continue;
        if (bi < 0 || (want_max ? (x >= best) : (x < best))) {
            best = x;
            bi = i;
        }
    }
    sv[threadIdx.x] = best;
    si[threadIdx.x] = bi;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            const T a = sv[threadIdx.x], b = sv[threadIdx.x + o];
            const long ia = si[threadIdx.x], ib = si[threadIdx.x + o];
            bool take_b;
            if (ib < 0) take_b = false;
            else if (ia < 0) take_b = true;
            else if (want_max) take_b = (b > a) || (b == a && ib > ia);
            else take_b = (b < a) || (b == a && ib < ia);
            if (take_b) {
                sv[threadIdx.x] = b;
                si[threadIdx.x] = ib;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        pv[blockIdx.x] = sv[0];
        pi[blockIdx.x] = si[0];
    }
}

template <typename T>
__global__ void k_argbest_final(const T* __restrict__ pv, const long* __restrict__ pi, int nparts, int want_max,
                                long* __restrict__ out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    T best = T(0);
    long bi = -1;
    for (int p = 0; p < nparts; p++) {
        if (pi[p] < 0) continue;
        if (bi < 0 || (want_max ? (pv[p] >= best) : (pv[p] < best))) {
            best = pv[p];
            bi = pi[p];
        }
    }
    *out = bi;
}

// out[i][j] = (i >= j) ? in[i][j] : in[j][i] for i, j < n  (hermitian fill of potri, lml.rs:62), packed n x n
template <typename T>
__global__ void k_sym_fill(const T* __restrict__ in, int np, int n, T* __restrict__ out, int mode) {
    int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j >= n || i >= n) return;
    T v;
    if (mode == 0) v = (i >= j) ? in[(long)i * np + j] : in[(long)j * np + i];  // symmetric
    else v = (i >= j) ? in[(long)i * np + j] : T(0);                             // lower only
    out[(long)i * n + j] = v;
}

// ---- standalone kernel evaluation (trait Kernel, src/gpr/kernel.rs:8-43) for parity checks against the reference's
// golden vectors.  The hot path never materialises the (n, n, d+1) tensor; this kernel writes it with exactly the
// per-entry terms k_grad_contract contracts (matern_grad_terms), for Product<ConstantKernel, Matern>:
//   k_out[i][j] = c * matern(|x_i / l - x_j / l|)                        (matern_kernel.rs:37-80, product_kernel.rs:36-38)
//   grad[i][j][0] = c * M_ij, grad[i][j][1 + k] = dM_ij / d ln l_k * c    (product_kernel.rs:40-70)
template <typename T, int NU2>
__global__ void k_kernel_theta_grad(const T* __restrict__ x, int n, int d, const T* __restrict__ ls, T c,
                                    T* __restrict__ k_out, T* __restrict__ grad) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j >= n || i >= n) return;
    T r2 = T(0);
    for (int k = 0; k < d; k++) {
        const T df = x[(long)i * d + k] / ls[k] - x[(long)j * d + k] / ls[k];  // division first (matern_kernel.rs:51-60)
        r2 += df * df;
    }
    const T kij = c * matern_corr<T, NU2>(dev_sqrt<T>(r2));
    if (k_out) k_out[(long)i * n + j] = kij;
    if (!grad) return;
    // like k_grad_contract, d_ijk is formed from the scaled inputs ((x_ik / l_k - x_jk / l_k)^2; the reference squares
    // the raw difference and then divides by l_k^2, matern_kernel.rs:95-98 -- equal up to rounding)
    T kval, dk_factor;
    matern_grad_terms<T, NU2>(r2, kval, dk_factor);
    T* g = grad + ((long)i * n + j) * (d + 1);
    g[0] = c * kval;  // constant_kernel.rs:31-38 times k2.kernel
    for (int k = 0; k < d; k++) {
        const T df = x[(long)i * d + k] / ls[k] - x[(long)j * d + k] / ls[k];
        g[1 + k] = dk_factor * (df * df) * c;
    }
}

// One record per evaluation for the exchange between GPUs: [lml, status, grad_0 .. grad_{p-1}] with lml and gradient
// zeroed and status = 1 when the evaluation failed (like eval_batch reports it to the host), written at record
// position pos0 + i * pos_stride of `round` (records of p + 2 doubles).
__global__ void k_pack_round(const double* __restrict__ lml, const double* __restrict__ grad, const int* __restrict__ status,
                             int cnt, int p, int pos0, int pos_stride, double* __restrict__ round) {
    const int i = blockIdx.x;
    if (i >= cnt) return;
    const double l = lml[i];
    const bool bad = status[i] != 0 || !(l - l == 0.0);
    double* rec = round + (long)(pos0 + i * pos_stride) * (p + 2);
    for (int t = threadIdx.x; t < p + 2; t += blockDim.x) {
        double v;
        if (t == 0) v = bad ? 0.0 : l;
        else if (t == 1) v = bad ? 1.0 : 0.0;
        else v = bad ? 0.0 : grad[(long)i * p + t - 2];
        rec[t] = v;
    }
}

template <typename T>
__global__ void k_fill(T* __restrict__ out, long n, T v) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = v;
}

// out[i][j] = in[i * ld + j] for j < cols (drops the column padding of a k* chunk)
template <typename T>
__global__ void k_copy_cols(const T* __restrict__ in, long ld, long rows, int cols, T* __restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const long i = blockIdx.y;
    if (j < cols && i < rows) out[i * cols + j] = in[i * ld + j];
}

}  // namespace hbegp
