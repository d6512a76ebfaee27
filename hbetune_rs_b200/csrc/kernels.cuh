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
// The reference asserts that mean, std and fmin are finite before anything else (acquisition.rs:141-171); where one is
// not, expected_improvement is NaN on the host and on the device alike, the std-zero branch included.
__host__ __device__ inline bool ei_inputs_finite(double mean, double sd, double fmin) {
    return fabs(mean) <= 1.7976931348623157e308 && fabs(sd) <= 1.7976931348623157e308 && fabs(fmin) <= 1.7976931348623157e308;
}

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

// NU2 of nu = +inf, the squared exponential (RBF) kernel; every other NU2 is 2 * nu.
constexpr int kNu2Rbf = 0;

// Matern correlation from the scaled distance r (src/gpr/matern_kernel.rs:65-80).  NU2 = 2 * nu.
template <typename T, int NU2>
__device__ __forceinline__ T matern_corr(T r) {
    static_assert(NU2 == 1 || NU2 == 3 || NU2 == 5, "matern_corr: finite nu only (corr_from_sq for the RBF)");
    if (NU2 == 1) return dev_exp<T>(-r);
    if (NU2 == 3) {
        T k = r * T(1.7320508075688772935);
        return (k + T(1)) * dev_exp<T>(-k);
    }
    T k = r * T(2.2360679774997896964);
    return (T(1) + k + k * k / T(3)) * dev_exp<T>(-k);
}

// Correlation from the squared scaled distance s = sum_k (x~_ik - x~_jk)^2.  RBF: exp(-0.5 s) (sklearn's RBF; the
// product by 0.5 is exact and no square root is taken); finite nu: exactly matern_corr(sqrt(s)).
template <typename T, int NU2>
__device__ __forceinline__ T corr_from_sq(T s) {
    if constexpr (NU2 == kNu2Rbf) return dev_exp<T>(T(-0.5) * s);
    else return matern_corr<T, NU2>(dev_sqrt<T>(s));
}

// Per-entry terms of the theta gradient (src/gpr/matern_kernel.rs:83-135) from s = sum_k d_ijk,
// d_ijk = (x_ik - x_jk)^2 / l_k^2: kval = the correlation recomputed from t = sqrt(2 nu s), and dk_factor such that
// dM_ij / d ln l_k = dk_factor * d_ijk.  RBF: kval = exp(-0.5 s) and dk_factor = -2 dM/ds = kval.
template <typename T, int NU2>
__device__ __forceinline__ void matern_grad_terms(T s, T& kval, T& dk_factor) {
    if constexpr (NU2 == kNu2Rbf) {
        kval = dev_exp<T>(T(-0.5) * s);
        dk_factor = kval;
    } else if (NU2 == 5) {
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
        static_assert(NU2 == 1 || NU2 == 3 || NU2 == 5, "matern_grad_terms: unknown NU2");
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
                v = c * corr_from_sq<T, NU2>(acc[a][q]);
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
                T v = (gj < n) ? c * corr_from_sq<T, NU2>(acc[a][q]) : T(0);
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
            const T v = (j < n) ? c * corr_from_sq<T, NU2>(acc) : T(0);
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

// ------------------------------------------------------------------------------- predict gradients
// Gradients of the predictive mean and variance in the candidate x (caller's units).  With x~_k = x_k / l_k,
// X~_jk = X_jk / l_k (division first, as everywhere), s_j = sum_k (x~_k - X~_jk)^2 and dk_factor = -2 dM/ds of
// matern_grad_terms:  d k*_j / d x_k = -c dk_factor(s_j) (x~_k - X~_jk) / l_k, so
//   dmean_k = -(c / l_k) sum_j alpha_j dk_factor_j (x~_k - X~_jk),
//   dvar_k  =  (2 c / l_k) sum_j v_j dk_factor_j (x~_k - X~_jk),   v = K^-1 k* = W^T (W k*).
// At s = 0 (a candidate on a training point) every Matern order and the RBF contribute 0 (nu = 1/2: dk_factor is 0
// there; elsewhere x~_k - X~_jk is).

// u[r][i] = sum_{k <= i} W[i][k] k*[r][k] for the 16 candidates of group blockIdx.y: k_wmatvec_small with u stored
// instead of squared (latency path of the variance gradient).
template <typename T>
__global__ void __launch_bounds__(256) k_wmatvec_small_store(const T* __restrict__ W, int np, const T* __restrict__ kstar, int m,
                                                             T* __restrict__ u) {
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
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
        if (lane == 0 && r0 + q < m) u[(long)(r0 + q) * np + row] = v;
    }
}

// v = W^T u for the 16 candidates of group blockIdx.z, the 64 columns of blockIdx.x and the rows
// [blockIdx.y * split_rows, +split_rows) of W: pv[blockIdx.y][r][col] = sum_{i in split, i >= col} W[i][col] u[r][i].
// Rows of W are read along the row (64 consecutive columns per step); the 4 row groups of a CTA are summed in order, the
// splits later by the consumer (k_kstar_grad), also in order.
template <typename T>
__global__ void __launch_bounds__(256) k_wtmatvec_small(const T* __restrict__ W, int np, const T* __restrict__ u, int m,
                                                        int split_rows, T* __restrict__ pv) {
    __shared__ T red[4][16][TILE];
    const int tid = threadIdx.x, cl = tid & 63, rg = tid >> 6;
    const int col = blockIdx.x * TILE + cl, r0 = blockIdx.z * 16;
    const int ibeg = max(blockIdx.y * split_rows, (int)blockIdx.x * TILE), iend = min(np, (int)(blockIdx.y + 1) * split_rows);
    T acc[16];
#pragma unroll
    for (int q = 0; q < 16; q++) acc[q] = T(0);
    for (int i = ibeg + rg; i < iend; i += 4) {
        const T wv = (i >= col) ? W[(long)i * np + col] : T(0);
#pragma unroll
        for (int q = 0; q < 16; q++)
            if (r0 + q < m) acc[q] = fma(wv, u[(long)(r0 + q) * np + i], acc[q]);
    }
#pragma unroll
    for (int q = 0; q < 16; q++) red[rg][q][cl] = acc[q];
    __syncthreads();
    for (int e = tid; e < 16 * TILE; e += 256) {
        const int q = e / TILE, c = e % TILE;
        if (r0 + q < m)
            pv[((long)blockIdx.y * 64 + r0 + q) * np + blockIdx.x * TILE + c] = ((red[0][q][c] + red[1][q][c]) + red[2][q][c]) + red[3][q][c];
    }
}

constexpr int kGradFeat = 16;  // features per pass of k_kstar_grad (4 per thread)

// Per 64 candidates (grid.x) and the train tiles [blockIdx.y * tiles_per_cta, +tiles_per_cta): re-forms the distances
// like k_kstar_mean, then gpart[y][0][r][k] = sum_j alpha_j dk_factor_j (x~_rk - X~_jk) and, when V != nullptr,
// gpart[y][1][r][k] = the same with v_rj = sum_{s < vsplit} V[s * vstride + r * np + j] (summed in split order) in place
// of alpha_j.  Feature passes of kGradFeat features each; a pass re-forms the distances.  Fixed tiles_per_cta makes a
// candidate's partials independent of the other rows predicted with it.
template <typename T>
__host__ __device__ inline size_t kstar_grad_smem(int d) {
    return ((size_t)2 * feat_chunk(d) * TILE + 2 * TILE * (TILE + 1) + kGradFeat * TILE) * sizeof(T);
}
template <typename T, int NU2>
__global__ void __launch_bounds__(256) k_kstar_grad(const T* __restrict__ xs, long m, long row0, int d,
                                                    const T* __restrict__ xsT_train, int n, int np,
                                                    const T* __restrict__ ls, const T* __restrict__ alpha,
                                                    const T* __restrict__ V, int vsplit, long vstride, int tiles_per_cta,
                                                    T* __restrict__ gpart, long gp_rows) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int dc = feat_chunk(d);
    T* xc = reinterpret_cast<T*>(smem_raw);  // [dc][64] candidates (scaled)
    T* xt = xc + dc * TILE;                  // [dc][64] train tile
    T* wm = xt + dc * TILE;                  // [64][65] alpha_j dk_factor
    T* wv = wm + TILE * (TILE + 1);          // [64][65] v_rj dk_factor
    T* xg = wv + TILE * (TILE + 1);          // [kGradFeat][64] the pass's features of the train tile
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int pr = tid & 63, pk = tid >> 6;  // feature pass: candidate row pr, features pk + 4 i
    const long r0 = (long)blockIdx.x * TILE;
    const bool want_v = V != nullptr;
    auto load_candidates = [&](int c0, int dl) {
        for (int e = tid; e < dl * TILE; e += 256) {
            int r = e / dl, k = e % dl;
            long gr = row0 + r0 + r;
            xc[k * TILE + r] = (gr < m) ? xs[gr * d + c0 + k] / ls[c0 + k] : T(0);
        }
    };
    const int jbeg = blockIdx.y * tiles_per_cta * TILE, jend = min(np, jbeg + tiles_per_cta * TILE);
    const long gpr = row0 + r0 + pr;
    if (d <= dc) load_candidates(0, d);  // one chunk: the candidate tile stays for every pass and train tile
    for (int f0 = 0; f0 < d; f0 += kGradFeat) {
        T xr[4], am[4], av[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int k = f0 + pk + 4 * i;
            xr[i] = (gpr < m && k < d) ? xs[gpr * d + k] / ls[k] : T(0);
            am[i] = T(0);
            av[i] = T(0);
        }
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
                    const int lr = ty + 16 * a, lj = tx + 16 * q, gj = j0 + lj;
                    T kval, dkf;
                    matern_grad_terms<T, NU2>(acc[a][q], kval, dkf);
                    wm[lr * (TILE + 1) + lj] = (gj < n) ? alpha[gj] * dkf : T(0);
                    if (want_v) {
                        T v = T(0);
                        for (int s = 0; s < vsplit; s++) v += V[s * vstride + (r0 + lr) * (long)np + gj];
                        wv[lr * (TILE + 1) + lj] = (gj < n) ? v * dkf : T(0);
                    }
                }
            for (int e = tid; e < kGradFeat * TILE; e += 256) {
                const int k = f0 + e / TILE;
                xg[e] = (k < d) ? xsT_train[(long)k * np + j0 + e % TILE] : T(0);
            }
            __syncthreads();
            for (int j = 0; j < TILE; j++) {
                const T w1 = wm[pr * (TILE + 1) + j];
                const T w2 = want_v ? wv[pr * (TILE + 1) + j] : T(0);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const T df = xr[i] - xg[(pk + 4 * i) * TILE + j];
                    am[i] += w1 * df;
                    av[i] += w2 * df;
                }
            }
        }
        T* gm = gpart + ((long)blockIdx.y * 2) * gp_rows * d;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int k = f0 + pk + 4 * i;
            if (k < d) {
                gm[(r0 + pr) * d + k] = am[i];
                if (want_v) gm[(gp_rows + r0 + pr) * d + k] = av[i];
            }
        }
    }
}

// Sums the split partials of k_kstar_grad in split order and scales them: dmean[row0 + r][k] = -c S_mean / l_k,
// dvar = 2 c S_var / l_k, and dvar = 0 where the predicted variance is 0 (clamped, or a pre-clamp value of exactly 0).  One thread per (row, feature).
template <typename T>
__global__ void k_grad_finish(const T* __restrict__ gpart, int nsplit, long gp_rows, long rows, long m, long row0, int d, T c,
                              const T* __restrict__ ls, const T* __restrict__ var, T* __restrict__ dmean, T* __restrict__ dvar) {
    const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const long r = e / d;
    const int k = (int)(e % d);
    if (r >= rows || row0 + r >= m) return;
    T sm = T(0), sv = T(0);
    for (int y = 0; y < nsplit; y++) {
        const T* g = gpart + (long)y * 2 * gp_rows * d;
        sm += g[r * d + k];
        if (dvar != nullptr) sv += g[(gp_rows + r) * d + k];
    }
    dmean[(row0 + r) * d + k] = -(c * sm) / ls[k];
    if (dvar != nullptr) dvar[(row0 + r) * d + k] = (var[row0 + r] == T(0)) ? T(0) : (T(2) * c * sv) / ls[k];
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
        if (!ei_inputs_finite(mean_d, std_d, fmin_n)) {
            ei = __longlong_as_double(0x7FF8000000000000LL);  // NaN, as the host expected_improvement
        } else if (ei_std_is_zero(std_d)) {
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

// Chain rules of k_acquisition on (mean, var, dmean, dvar) of one row per thread, in place over the gradients:
//   dsd = dvar / (2 sd) where sd > 0, else 0;  d location_from(y) = amplitude * dy (linear),
//   amplitude * exp(y * amplitude) * dy (logarithmic).
//   mode 0: dmean <- d location_from(mean); dvar <- dEI in f64: -Phi(z) dmean + phi(z) dsd, in the std-zero branch
//           -dmean where mean < fmin_n and 0 otherwise, NaN in every component where EI is NaN;
//   mode 1: dmean <- d location_from(mean + cb sd) with dy = dmean + cb dsd.
template <typename T>
__global__ void k_acquisition_grad(const T* __restrict__ mean, const T* __restrict__ var, long m, int d, int mode, int proj,
                                   T amplitude, double fmin_n, T cb, T* __restrict__ dmean, T* __restrict__ dvar) {
    long r = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= m) return;
    const T mu = mean[r], sd = dev_sqrt<T>(var[r]);
    const T y = (mode == 0) ? mu : add_rn<T>(mu, mul_rn<T>(sd, cb));
    const T lf = proj == 0 ? amplitude : amplitude * dev_exp<T>(mul_rn<T>(y, amplitude));
    T* gm = dmean + r * d;
    T* gv = dvar + r * d;
    const double mean_d = (double)mu, std_d = (double)sd;
    const bool finite = ei_inputs_finite(mean_d, std_d, fmin_n), zero = ei_std_is_zero(std_d);
    double cdf = 0.0, pdf = 0.0;
    if (mode == 0 && finite && !zero) {
        const double z = -(mean_d - fmin_n) / std_d;
        cdf = 0.5 * erfc(-z * 0.70710678118654752440);
        pdf = exp(-0.5 * z * z) * 0.39894228040143267794;
    }
    for (int k = 0; k < d; k++) {
        const T dm = gm[k];
        const T dsd = (sd > T(0)) ? gv[k] / (T(2) * sd) : T(0);
        if (mode == 0) {
            double dei;
            if (!finite) dei = __longlong_as_double(0x7FF8000000000000LL);
            else if (zero) dei = mean_d < fmin_n ? -(double)dm : 0.0;
            else dei = -cdf * (double)dm + pdf * (double)dsd;
            gm[k] = lf * dm;
            gv[k] = (T)dei;
        } else {
            gm[k] = lf * (dm + cb * dsd);
        }
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

// The arg-best plan: up to kArgbestParts parts of chunk = ceil(m / nparts) elements, one 256-thread block per part, so
// from m = 256 * 1024 + 1 on a thread sees several elements of its part and trailing parts can be empty.
constexpr int kArgbestParts = 1024, kArgbestThreads = 256;
inline int argbest_parts(long m) {
    const long p = (m + kArgbestThreads - 1) / kArgbestThreads;
    return (int)(p < kArgbestParts ? (p > 0 ? p : 1) : kArgbestParts);
}
// Workspace of launch_argbest: one index and one value per part.
inline size_t argbest_ws_bytes(long m) { return (size_t)argbest_parts(m) * (sizeof(long) + 8); }

// *out (device) = the arg-best of key[0, m) under the rules of k_argbest_part; asynchronous on `st`.
template <typename T>
inline cudaError_t launch_argbest(const T* key, long m, int want_max, void* ws, long* out, cudaStream_t st) {
    const int nparts = argbest_parts(m);
    long* pi = static_cast<long*>(ws);
    T* pv = reinterpret_cast<T*>(pi + nparts);
    k_argbest_part<T><<<nparts, kArgbestThreads, 0, st>>>(key, m, want_max, pv, pi);
    k_argbest_final<T><<<1, 32, 0, st>>>(pv, pi, nparts, want_max, out);
    return cudaGetLastError();
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
    const T kij = c * corr_from_sq<T, NU2>(r2);
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

// ---- the acquisition search (hbegp_acquire_ei / hbegp_acquire_confidence_bound): BoundedLbfgs of lbfgs.h restated for
// the device, one thread per start, so that the whole search loop stays on the device.  Every operation is the one
// lbfgs.h performs on the host (built with -ffp-contract=off), in the same order: explicit round-to-nearest double
// operations keep nvcc from contracting them into FMAs, and std::min / std::max are written as libstdc++'s ternaries
// (NaN behaviour included).  lbfgs.h's rho is never read there and is not kept here.
constexpr int kAcqMemory = 10;  // BoundedLbfgs's default memory

// Per-start scalars of the optimiser and of the capture.
struct AcqScalars {
    double f, alpha, best_f;
    long long best_eval;
    int evals, ls_iter, stall, k, head, have_x, done, steepest, rounds, pad;
};

// Device state of S starts; arrays are per start, contiguous (d or kAcqMemory * d values each).
struct AcqState {
    AcqScalars* sc;
    double *x, *g, *xt, *dir, *s, *y, *a;  // dir doubles as the two-loop recursion's q, as it is overwritten from it
    unsigned char* fr;                     // free flags
    const double *lo, *hi;
};

__device__ __forceinline__ double acq_min(double a, double b) { return (b < a) ? b : a; }  // std::min
__device__ __forceinline__ double acq_max(double a, double b) { return (a < b) ? b : a; }  // std::max

struct AcqRun {  // the view of one start: BoundedLbfgs's members
    AcqScalars& c;
    double *x, *g, *xt, *dir, *s, *y, *a;
    unsigned char* fr;
    const double *lo, *hi;
    int n, maxeval;
    double ftol, gtol;

    __device__ double* S(int j) const { return s + (size_t)((c.head + j) % kAcqMemory) * n; }  // j = 0: oldest pair
    __device__ double* Y(int j) const { return y + (size_t)((c.head + j) % kAcqMemory) * n; }
    __device__ void clear() { c.k = 0; c.head = 0; }
    __device__ bool finish() {
        c.done = 1;
        return true;
    }

    __device__ bool make_trial() {
        if (c.evals >= maxeval) return finish();
        bool moved = false;
        for (int i = 0; i < n; i++) {
            double v = __dadd_rn(x[i], __dmul_rn(c.alpha, dir[i]));
            v = acq_min(acq_max(v, lo[i]), hi[i]);
            xt[i] = v;
            if (v != x[i]) moved = true;
        }
        if (!moved) return finish();
        return false;
    }

    __device__ bool next_direction(bool force_steepest) {
        if (c.evals >= maxeval) return finish();
        double pgmax = 0.0;
        int nfree = 0;
        for (int i = 0; i < n; i++) {
            const bool at_lo = x[i] <= lo[i] && g[i] > 0.0;
            const bool at_hi = x[i] >= hi[i] && g[i] < 0.0;
            fr[i] = !(at_lo || at_hi);
            if (fr[i]) {
                nfree++;
                pgmax = acq_max(pgmax, fabs(g[i]));
            }
        }
        if (nfree == 0 || pgmax <= (gtol > 0 ? gtol : 0.0)) return finish();
        c.steepest = force_steepest || c.k == 0;
        double* q = dir;
        for (int i = 0; i < n; i++) q[i] = fr[i] ? g[i] : 0.0;
        if (!c.steepest) {
            const int k = c.k;
            for (int j = k - 1; j >= 0; j--) {
                const double *Sj = S(j), *Yj = Y(j);
                double sq = 0, sy = 0;
                for (int i = 0; i < n; i++)
                    if (fr[i]) {
                        sq = __dadd_rn(sq, __dmul_rn(Sj[i], q[i]));
                        sy = __dadd_rn(sy, __dmul_rn(Sj[i], Yj[i]));
                    }
                if (!(sy > 0)) {
                    a[j] = 0;
                    continue;
                }
                a[j] = __ddiv_rn(sq, sy);
                for (int i = 0; i < n; i++)
                    if (fr[i]) q[i] = __dsub_rn(q[i], __dmul_rn(a[j], Yj[i]));
            }
            {
                const double *Sl = S(k - 1), *Yl = Y(k - 1);
                double sy = 0, yy = 0;
                for (int i = 0; i < n; i++)
                    if (fr[i]) {
                        sy = __dadd_rn(sy, __dmul_rn(Sl[i], Yl[i]));
                        yy = __dadd_rn(yy, __dmul_rn(Yl[i], Yl[i]));
                    }
                const double gamma = (sy > 0 && yy > 0) ? __ddiv_rn(sy, yy) : 1.0;
                for (int i = 0; i < n; i++) q[i] = __dmul_rn(q[i], gamma);
            }
            for (int j = 0; j < k; j++) {
                const double *Sj = S(j), *Yj = Y(j);
                double yq = 0, sy = 0;
                for (int i = 0; i < n; i++)
                    if (fr[i]) {
                        yq = __dadd_rn(yq, __dmul_rn(Yj[i], q[i]));
                        sy = __dadd_rn(sy, __dmul_rn(Sj[i], Yj[i]));
                    }
                if (!(sy > 0)) continue;
                const double beta = __ddiv_rn(yq, sy);
                for (int i = 0; i < n; i++)
                    if (fr[i]) q[i] = __dadd_rn(q[i], __dmul_rn(__dsub_rn(a[j], beta), Sj[i]));
            }
        }
        double gd = 0, gnorm1 = 0;
        for (int i = 0; i < n; i++) {
            dir[i] = fr[i] ? -q[i] : 0.0;
            gd = __dadd_rn(gd, __dmul_rn(g[i], dir[i]));
            if (fr[i]) gnorm1 = __dadd_rn(gnorm1, fabs(g[i]));
        }
        if (!(gd < 0) || !isfinite(gd)) {
            c.steepest = 1;
            gd = 0;
            for (int i = 0; i < n; i++) {
                dir[i] = fr[i] ? -g[i] : 0.0;
                gd = __dadd_rn(gd, __dmul_rn(g[i], dir[i]));
            }
        }
        c.alpha = c.steepest ? acq_min(1.0, __ddiv_rn(1.0, gnorm1)) : 1.0;
        c.ls_iter = 0;
        return make_trial();
    }

    // BoundedLbfgs::tell; gt(i) is component i of the gradient at xt
    template <typename G>
    __device__ bool tell(double ft, const G& gt) {
        if (c.done) return true;
        c.evals++;
        const bool finite = isfinite(ft);
        if (!c.have_x) {
            for (int i = 0; i < n; i++) x[i] = xt[i];
            c.f = ft;
            c.have_x = 1;
            if (!finite) return finish();
            for (int i = 0; i < n; i++) g[i] = gt(i);
            return next_direction(true);
        }
        double dec = 0.0;
        for (int i = 0; i < n; i++) dec = __dadd_rn(dec, __dmul_rn(g[i], __dsub_rn(xt[i], x[i])));
        if (!(dec < 0.0)) {
            if (c.k > 0 || !c.steepest) {
                clear();
                return next_direction(true);
            }
            return finish();
        }
        if (finite && ft <= __dadd_rn(c.f, __dmul_rn(1e-4, dec))) {
            double sy = 0, ss = 0, yy = 0;
            for (int i = 0; i < n; i++) {
                const double si = __dsub_rn(xt[i], x[i]), yi = __dsub_rn(gt(i), g[i]);
                sy = __dadd_rn(sy, __dmul_rn(si, yi));
                ss = __dadd_rn(ss, __dmul_rn(si, si));
                yy = __dadd_rn(yy, __dmul_rn(yi, yi));
            }
            if (sy > __dmul_rn(1e-10, __dsqrt_rn(__dmul_rn(ss, yy))) && sy > 0) {
                // push_back, dropping the oldest pair when the memory is full; s and y are recomputed with the same
                // operations, so the ring keeps the bits lbfgs.h stores
                int slot;
                if (c.k == kAcqMemory) {
                    slot = c.head;
                    c.head = (c.head + 1) % kAcqMemory;
                } else {
                    slot = (c.head + c.k) % kAcqMemory;
                    c.k++;
                }
                double* Sn = s + (size_t)slot * n;
                double* Yn = y + (size_t)slot * n;
                for (int i = 0; i < n; i++) {
                    Sn[i] = __dsub_rn(xt[i], x[i]);
                    Yn[i] = __dsub_rn(gt(i), g[i]);
                }
            }
            const double fprev = c.f;
            for (int i = 0; i < n; i++) x[i] = xt[i];
            c.f = ft;
            for (int i = 0; i < n; i++) g[i] = gt(i);
            const double scale = acq_max(acq_max(fabs(fprev), fabs(c.f)), 1.0);
            if (ftol > 0 && __dsub_rn(fprev, c.f) <= __dmul_rn(ftol, scale)) c.stall++;
            else c.stall = 0;
            if (c.stall >= 2) return finish();
            return next_direction(false);
        }
        c.ls_iter++;
        double anew;
        if (finite) {
            const double denom = __dmul_rn(2.0, __dsub_rn(__dsub_rn(ft, c.f), dec));
            anew = (denom > 0) ? __ddiv_rn(__dmul_rn(-dec, c.alpha), denom) : __dmul_rn(0.5, c.alpha);
            anew = acq_min(acq_max(anew, __dmul_rn(0.1, c.alpha)), __dmul_rn(0.5, c.alpha));
        } else {
            anew = __dmul_rn(0.25, c.alpha);
        }
        c.alpha = anew;
        if (c.ls_iter > 25 || c.alpha < 1e-18) {
            if (c.k > 0 || !c.steepest) {
                clear();
                return next_direction(true);
            }
            return finish();
        }
        return make_trial();
    }
};

// One step of every start (thread i = start i) after the round evaluated the S rows of xs:
//   mode 0: f = -EI (val = ei_out), gradient -dei (grad), mean = de-normalised mean (captured with the point);
//   mode 1: f = the confidence bound (val), gradient grad; mean unused.
// A live start applies the capture rule of fit_runs_impl (first finite value, then a strictly smaller f), tells the
// optimiser, and writes its next trial point, rounded to T, back into its row; a finished start changes nothing, so its
// row keeps its last trial point.  *live counts the starts not done yet.
template <typename T>
__global__ void k_acq_step(int S, int d, int mode, int maxeval, double ftol, double gtol, const T* __restrict__ val,
                           const T* __restrict__ grad, const T* __restrict__ mean, T* __restrict__ xs, AcqState st,
                           T* __restrict__ best_x, T* __restrict__ best_mean, int* __restrict__ live) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S) return;
    AcqScalars& c = st.sc[i];
    if (c.done) return;
    const size_t o = (size_t)i * d, om = o * kAcqMemory;
    AcqRun r{c, st.x + o, st.g + o, st.xt + o, st.dir + o, st.s + om, st.y + om, st.a + (size_t)i * kAcqMemory, st.fr + o,
             st.lo, st.hi, d, maxeval, ftol, gtol};
    c.rounds++;
    const double v = (double)val[i];
    const double f = (mode == 0) ? -v : v;
    T* row = xs + o;
    if (isfinite(f) && (c.best_eval < 0 || f < c.best_f)) {
        c.best_f = f;
        c.best_eval = c.evals;
        for (int k = 0; k < d; k++) best_x[o + k] = row[k];
        if (mode == 0) best_mean[i] = mean[i];
    }
    const T* gr = grad + o;
    auto gt = [&](int k) -> double { return (mode == 0) ? -(double)gr[k] : (double)gr[k]; };
    r.tell(f, gt);
    for (int k = 0; k < d; k++) row[k] = (T)r.xt[k];
    if (c.done) atomicSub(live, 1);
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
