// The 128-wide bottom node of the factor + inverse recursion, second generation (round 2).  FP64 arithmetic; the matrices
// in global memory are double or (--use-32) float.
//
// The first-generation node (two leaf_core leaves of kernels.cuh and four 64^3 FMA-pipe products in one CTA) spent its
// 59 us on (i) two 64-pivot chains with a CTA barrier and a shared-memory round trip per pivot, (ii) 15 more barrier
// steps for the diagonal-block inverses and (iii) four 64^3 products whose operand fetches saturate the shared-memory
// pipe (one 8-byte LDS per FMA and thread).  This kernel keeps the same contract
// (W11, W21, W22 = the inverse of the Cholesky factor of the 128-wide diagonal block, sum ln L_ii per 64-wide half,
// status = 1 on a non-positive pivot) and removes all three:
//  * Cholesky in panels of 8 whose pivot chain lives in registers: every row thread holds the panel's 8x8 diagonal
//    block (broadcast loads) and eliminates it redundantly — identical bits in every thread, no communication — while
//    carrying its own row through the same eliminations.  One CTA barrier per panel (plus two among the two panel warps)
//    instead of one per pivot.
//  * every product — the rank-8 trailing updates, the recursive-doubling levels of the triangular inverse, and the
//    four 64^3 products between the halves — runs on the DMMA pipe (mma.sync.m8n8k4.f64) straight from shared
//    memory, with the k ranges cut to the triangular structure at 8x8-tile granularity.  One warp-wide LDS feeds 256
//    FMAs instead of 32, and the tiles are dealt so that the four sub-partitions carry the same number of DMMAs.
//  * the block being factored is held TRANSPOSED (at[k][i] = A[i][k], i >= k): a row thread's panel entries are then
//    consecutive words across the warp, and both DMMA operands of the trailing update come from the same panel rows.
//    Tiles have a row stride of 68 doubles (= 4 mod 16): both fragment shapes load without bank conflicts.
//  * look-ahead: after a panel the two panel warps update only the rows the next panel reads and go on to its pivot
//    chain; the other six warps apply the rest of the rank-8 update underneath it, scale the panel before to the true
//    factor (L_ik = u_ik / L_kk), take the square roots and accumulate the logarithm's argument.
// Measured on B200 (probes/leaf2_bench.cu, probes/lat_probe.cu): DFMA 8 cycles dependent / 2 per warp issue,
// MUFU.RCP64H 17, DMMA 26 dependent / ~17.5 per sub-partition in a saturated GEMM, ~24 per warp in short bursts
// (probes/dmma_warm_probe.cu), CTA barrier 15-30, shared-memory round trip 42.
#pragma once
#include <cuda_runtime.h>

#include "kernels.cuh"

namespace hbegp {

constexpr int LDT = TILE + 4;
typedef double RowT[LDT];
__host__ __device__ constexpr size_t node_v2_tile_bytes() { return sizeof(double) * TILE * LDT; }
constexpr size_t node128_v2_smem_bytes() { return 5 * node_v2_tile_bytes() + 2 * TILE * sizeof(double); }

__device__ __forceinline__ void dmma_acc(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// 1 / d for a Cholesky pivot: hardware seed (~20 bits) and one third-order step: r (1 + e + e^2), e = 1 - d r.
__device__ __forceinline__ double pivot_rcp3(double d) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    const double e = fma(-d, r, 1.0);
    const double t = fma(e, e, e);
    return fma(r, t, r);
}

// tile t of the row-by-row enumeration of a lower triangle: (tr, tc), tr >= tc
__device__ __forceinline__ void lower_tile_of(int t, int& tr, int& tc) {
    tr = 0;
    while ((tr + 1) * (tr + 2) / 2 <= t) ++tr;
    tc = t - tr * (tr + 1) / 2;
}

// PROF (probes only): thread 0 appends clock64() stamps at the phase boundaries to tp
#define HBEGP_STAMP() do { if (PROF && tid == 0) *tp++ = clock64(); } while (0)

// Cholesky + inverse of one 64x64 block held transposed in shared memory.  In: at[k][i] = A[i][k] for i >= k (the
// part below the diagonal of `at` is scratch).  Out: ws = L^-1 (zeros above the diagonal), dinv[i] = 1 / L_ii,
// *fail = 1 when a pivot is not positive, and in thread 64 + 24 j (j = 0..7) `rdprod` = the product of 1 / u_kk =
// 1 / L_kk^2 over k = j (mod 8): sum ln L_kk = -1/2 ln prod.  Begins and ends with a barrier.  `at` is scratch after.
template <bool PROF = false>
__device__ __forceinline__ void leaf_mma(RowT* at, RowT* ws, double* rdv, double* dinv, int* fail, int tid, double& rdprod,
                                         long long*& tp, long long* pp, double* pending_log = nullptr) {
    constexpr int NB = 8, NP = TILE / NB;
    const int tx = tid & 15, ty = tid >> 4, warp = tid >> 5, lane = tid & 31, lr = lane >> 2, lc = lane & 3;
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int q = 0; q < 4; q++) ws[ty + 16 * a][tx + 16 * q] = 0.0;
    // Tiles of the rank-8 trailing update after panel P, relative to its first tile (c0 + 8, c0 + 8):
    //  * column 0 — the rows the NEXT panel reads — belongs to the two panel warps (tile rows w, w + 2, ..), which update
    //    it and go straight on to the next panel's pivot chain (look-ahead);
    //  * the rest (tile rows/columns >= 1, a lower triangle again) is dealt to warps 2..7 (tile t = (warp - 2) + 6 s) and
    //    runs underneath that chain, together with the scaling of the panel before.
    int ttr[4], ttc[4];
#pragma unroll
    for (int s = 0; s < 4; s++) {
        if (warp < 2) {
            ttr[s] = warp + 2 * s;
            ttc[s] = 0;
        } else {
            lower_tile_of(warp - 2 + 6 * s, ttr[s], ttc[s]);
            ttr[s] += 1;
            ttc[s] += 1;
        }
    }
    rdprod = 1.0;
    // finishes panel P (rows c0 .. c0 + 7 of `at`): true factor L_ik = u_ik / L_kk, 1 / L_kk = sqrt(1 / u_kk)
    auto finish_panel = [&](int c0, int idx) {  // idx = 0 .. 191
        const int j = idx / 24, l24 = idx % 24, k = c0 + j;
        const double rk = rdv[k], dk = sqrt(rk);
        if (l24 == 0) {
            dinv[k] = dk;
            rdprod *= rk;
        }
        for (int i = k + 1 + l24; i < TILE; i += 24) at[k][i] *= dk;
    };
    // one panel: rows c0 .. c0 + 7 of `at`, one row of the (untransposed) panel per thread of warps 0 and 1
    auto eliminate_panel = [&](int c0) {
        const int i = tid;
        double U[NB][NB], x[NB], rd[NB];
#pragma unroll
        for (int r = 0; r < NB; r++)
#pragma unroll
            for (int k = 0; k <= r; k++) U[r][k] = at[c0 + k][c0 + r];
#pragma unroll
        for (int k = 0; k < NB; k++) x[k] = at[c0 + k][i];
        // the diagonal rows are overwritten below by their owners: every row thread must hold its copy first
        asm volatile("bar.sync 1, 64;" ::: "memory");
        if (i >= c0) {
            bool bad = false;
#pragma unroll
            for (int j = 0; j < NB; j++) {
                // A non-positive (or non-finite) pivot is recorded, not repaired: the test stays off the dependent
                // chain and whatever follows in this matrix is discarded with status = 1 (lml.rs:47-50).
                const double dj = U[j][j];
                bad |= !(dj > 0.0) || !(dj <= 1e300);
                const double r_ = pivot_rcp3(dj);
                rd[j] = r_;
#pragma unroll
                for (int r = j + 1; r < NB; r++) {
                    const double l = U[r][j] * r_;
#pragma unroll
                    for (int k = j + 1; k <= r; k++) U[r][k] = fma(-l, U[k][j], U[r][k]);
                }
                const double lx = x[j] * r_;
#pragma unroll
                for (int k = j + 1; k < NB; k++) x[k] = fma(-lx, U[k][j], x[k]);
            }
#pragma unroll
            for (int k = 0; k < NB; k++)
                if (c0 + k <= i) at[c0 + k][i] = x[k];
            if (i == c0) {
#pragma unroll
                for (int j = 0; j < NB; j++) rdv[c0 + j] = rd[j];
                if (bad) *fail = 1;
            }
        }
    };
    // this warp's share of the rank-8 update after panel c0 on the DMMA pipe: C'[k'][i] -= sum_j (u_k'j / u_jj) u_ij.
    // All operand loads are unconditional (clamped tiles) so that they issue back to back; only the DMMAs and the
    // stores of tiles outside the remaining triangle are predicated off.
    auto trailing = [&](int c0, int nt) {
        double2 c[4];
        double2* cp[4];
        double a[4][2], bq[4][2];
        bool on[4];
        const double r0 = rdv[c0 + lc], r1 = rdv[c0 + 4 + lc];
#pragma unroll
        for (int s = 0; s < 4; s++) {
            on[s] = ttr[s] < nt;
            const int row0 = c0 + NB + 8 * (on[s] ? ttr[s] : 0), col0 = c0 + NB + 8 * (on[s] ? ttc[s] : 0);
            cp[s] = reinterpret_cast<double2*>(&at[col0 + lr][row0 + 2 * lc]);
            c[s] = *cp[s];
            a[s][0] = at[c0 + lc][col0 + lr];
            a[s][1] = at[c0 + 4 + lc][col0 + lr];
            bq[s][0] = at[c0 + lc][row0 + lr];
            bq[s][1] = at[c0 + 4 + lc][row0 + lr];
        }
#pragma unroll
        for (int s = 0; s < 4; s++) {
            a[s][0] = -(a[s][0] * r0);
            a[s][1] = -(a[s][1] * r1);
        }
#pragma unroll
        for (int h = 0; h < 2; h++)
#pragma unroll
            for (int s = 0; s < 4; s++)
                if (on[s]) dmma_acc(c[s].x, c[s].y, a[s][h], bq[s][h]);
#pragma unroll
        for (int s = 0; s < 4; s++)
            if (on[s]) *cp[s] = c[s];
    };
    // ---- Cholesky on unscaled columns u_ij = L_ij L_jj:  u_ik -= u_ij u_kj / u_jj
    // Iteration P: [warps 0, 1] column 0 of the update after panel P, then panel P + 1;  [warps 2..7] the rest of that
    // update and the scaling of panel P - 1.  P = -1 is the prologue (panel 0 only; one copy of the code for both).
    for (int P = -1; P + 1 < NP; P++) {
        const int c0 = NB * P, nt = NP - 1 - P;
        __syncthreads();  // panel P is in place; the update after panel P - 1 is complete
        if (PROF && tid == 0) pp[P + 1] = clock64();
        if (tid < TILE) {
            if (P >= 0) {
                trailing(c0, nt);  // tile column 0: the next panel's rows
                asm volatile("bar.sync 1, 64;" ::: "memory");
            }
            eliminate_panel(c0 + NB);
        } else {
            if (P >= 0) trailing(c0, nt);                        // the rest, underneath the next panel's chain
            if (P > 0) finish_panel(c0 - NB, tid - TILE);        // panel P - 1 is not read any more
            if (P < 0 && pending_log != nullptr && (tid - TILE) % 24 == 0)
                *pending_log = -0.5 * log(*pending_log);  // the previous leaf's log-determinant part, off the critical path
        }
    }
    __syncthreads();
    if (PROF && tid == 0) pp[NP] = clock64();
    if (tid >= TILE) {
        finish_panel(TILE - 2 * NB, tid - TILE);
        finish_panel(TILE - NB, tid - TILE);
    }
    __syncthreads();
    HBEGP_STAMP();
    // ---- inverse, level 0: the eight 8x8 diagonal blocks, one column per thread, in registers
    if (tid < TILE) {
        const int c0 = tid & ~(NB - 1), c = tid & (NB - 1);
        double Lv[NB][NB], dv[NB], sv[NB];
#pragma unroll
        for (int i = 0; i < NB; i++) {
            dv[i] = dinv[c0 + i];
            sv[i] = (i == c) ? 1.0 : 0.0;
#pragma unroll
            for (int k = 0; k < i; k++) Lv[i][k] = at[c0 + k][c0 + i];
        }
        // column-oriented forward substitution: once x_k is known every later row takes its term (one multiply and one
        // FMA on the dependent chain per step)
#pragma unroll
        for (int k = 0; k < NB; k++) {
            const double xk = sv[k] * dv[k];
            if (k >= c) ws[c0 + k][c0 + c] = xk;
#pragma unroll
            for (int i = k + 1; i < NB; i++) sv[i] = fma(-Lv[i][k], xk, sv[i]);
        }
    }
    HBEGP_STAMP();
    // ---- levels 1..3 (half-width h = 8, 16, 32): W21 = -W22 (L21 W11); S = L21 W11 goes to the lower-left block of `at`
#pragma unroll
    for (int h = NB; h < TILE; h *= 2) {
        const int th = h / 8, per = th * th, ntiles = (TILE / (2 * h)) * per;  // 4, 8, 16 tiles: at most two per warp
        const int nmine = (ntiles + 7) / 8;
        int ti[2], tj[2], o[2];
        bool on[2];
#pragma unroll
        for (int s = 0; s < 2; s++) {
            const int t = warp + 8 * s;
            on[s] = s < nmine && t < ntiles;
            const int tt = on[s] ? t : 0;
            o[s] = 2 * h * (tt / per);
            ti[s] = (tt % per) / th;
            tj[s] = tt % th;
        }
        __syncthreads();
        {
            double2 c[2];
            double av[2][8], bv[2][8];
#pragma unroll
            for (int s = 0; s < 2; s++) {
                c[s] = make_double2(0.0, 0.0);
#pragma unroll
                for (int q = 0; q < h / 4; q++) {  // W11 is lower triangular: k >= column tile
                    const int k4 = 4 * q;
                    if (on[s] && k4 >= 8 * tj[s]) {
                        av[s][q] = at[o[s] + k4 + lc][o[s] + h + 8 * ti[s] + lr];
                        bv[s][q] = ws[o[s] + k4 + lc][o[s] + 8 * tj[s] + lr];
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < h / 4; q++)
#pragma unroll
                for (int s = 0; s < 2; s++)
                    if (on[s] && 4 * q >= 8 * tj[s]) dmma_acc(c[s].x, c[s].y, av[s][q], bv[s][q]);
#pragma unroll
            for (int s = 0; s < 2; s++)
                if (on[s]) *reinterpret_cast<double2*>(&at[o[s] + h + 8 * ti[s] + lr][o[s] + 8 * tj[s] + 2 * lc]) = c[s];
        }
        __syncthreads();
        {
            double2 c[2];
            double av[2][8], bv[2][8];
#pragma unroll
            for (int s = 0; s < 2; s++) {
                c[s] = make_double2(0.0, 0.0);
#pragma unroll
                for (int q = 0; q < h / 4; q++) {  // W22 is lower triangular: k <= row tile
                    const int k4 = 4 * q;
                    if (on[s] && k4 < 8 * ti[s] + 8) {
                        av[s][q] = -ws[o[s] + h + 8 * ti[s] + lr][o[s] + h + k4 + lc];
                        bv[s][q] = at[o[s] + h + k4 + lc][o[s] + 8 * tj[s] + lr];
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < h / 4; q++)
#pragma unroll
                for (int s = 0; s < 2; s++)
                    if (on[s] && 4 * q < 8 * ti[s] + 8) dmma_acc(c[s].x, c[s].y, av[s][q], bv[s][q]);
#pragma unroll
            for (int s = 0; s < 2; s++)
                if (on[s]) *reinterpret_cast<double2*>(&ws[o[s] + h + 8 * ti[s] + lr][o[s] + 8 * tj[s] + 2 * lc]) = c[s];
        }
    }
    __syncthreads();
    HBEGP_STAMP();
}

// The four 64^3 products between the halves.  All are bound by the FP64 pipe of the SM (a DMMA occupies a
// sub-partition for 16 cycles), so the tiles are dealt to the warps such that the four sub-partitions (warp % 4) carry
// the same number of DMMAs: a warp owns a whole tile row (or column) when the k range depends on the column (row) only.

// out[r][c] = sum_{k <= c} A[r][k] Wl[c][k]     (A times the transpose of a lower-triangular tile; warp = tile row)
__device__ __forceinline__ void prod_a_wt(const RowT* Am, const RowT* Wl, double acc[8][2], int warp, int lr, int lc) {
#pragma unroll
    for (int j = 0; j < 8; j++) acc[j][0] = acc[j][1] = 0.0;
#pragma unroll
    for (int k4 = 0; k4 < TILE; k4 += 4) {
        const double a = Am[8 * warp + lr][k4 + lc];
#pragma unroll
        for (int j = k4 / 8; j < 8; j++) dmma_acc(acc[j][0], acc[j][1], a, Wl[8 * j + lr][k4 + lc]);
    }
}

// out[r][c] = sum_{k >= c} A[r][k] Wl[k][c]     (A times a lower-triangular tile; warp = tile row)
__device__ __forceinline__ void prod_a_w(const RowT* Am, const RowT* Wl, double acc[8][2], int warp, int lr, int lc) {
#pragma unroll
    for (int j = 0; j < 8; j++) acc[j][0] = acc[j][1] = 0.0;
#pragma unroll
    for (int k4 = 0; k4 < TILE; k4 += 4) {
        const double a = Am[8 * warp + lr][k4 + lc];
#pragma unroll
        for (int j = 0; j <= k4 / 8; j++) dmma_acc(acc[j][0], acc[j][1], a, Wl[k4 + lc][8 * j + lr]);
    }
}

// out[r][c] = sum_{k <= r} Wl[r][k] B[k][c]     (a lower-triangular tile times B; warp = tile column, acc per tile row)
__device__ __forceinline__ void prod_w_b(const RowT* Wl, const RowT* Bm, double acc[8][2], int warp, int lr, int lc) {
#pragma unroll
    for (int i = 0; i < 8; i++) acc[i][0] = acc[i][1] = 0.0;
#pragma unroll
    for (int k4 = 0; k4 < TILE; k4 += 4) {
        const double b = Bm[k4 + lc][8 * warp + lr];
#pragma unroll
        for (int i = k4 / 8; i < 8; i++) dmma_acc(acc[i][0], acc[i][1], Wl[8 * i + lr][k4 + lc], b);
    }
}

//   W11 = leaf(A11); L21 = A21 W11^T; A22 -= L21 L21^T; T = L21 W11; W22 = leaf(A22); W21 = -W22 T.
// TIO is the type of the matrices in global memory.  The arithmetic inside the node is FP64 in both cases: for --use-32
// (TIO = float) the block is widened on load and rounded once on store — the node is latency bound, not FP64-rate bound,
// so this costs nothing (35 us against 52 us for the first-generation node in FP32) and the bottom of the recursion adds no FP32
// rounding of its own.
template <bool PROF = false, typename TIO = double>
__global__ void __launch_bounds__(256) k_node128_v2(TIO* __restrict__ A, TIO* __restrict__ W, long mstride, int np, int r0g,
                                                    TIO* __restrict__ ldp, int ldp_stride, int* __restrict__ status,
                                                    long long* __restrict__ prof = nullptr) {
    extern __shared__ __align__(16) unsigned char leaf_smem_raw[];
    RowT* at = reinterpret_cast<RowT*>(leaf_smem_raw);                              // the block being factored, transposed
    RowT* w1 = reinterpret_cast<RowT*>(leaf_smem_raw + 1 * node_v2_tile_bytes());
    RowT* w2 = reinterpret_cast<RowT*>(leaf_smem_raw + 2 * node_v2_tile_bytes());  // A22^T until the second leaf
    RowT* pm = reinterpret_cast<RowT*>(leaf_smem_raw + 3 * node_v2_tile_bytes());  // A21, later T
    RowT* qm = reinterpret_cast<RowT*>(leaf_smem_raw + 4 * node_v2_tile_bytes());  // L21
    double* rdv = reinterpret_cast<double*>(leaf_smem_raw + 5 * node_v2_tile_bytes());
    double* dinv = rdv + TILE;
    __shared__ int fail;
    const int b = blockIdx.z, tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int warp = tid >> 5, lane = tid & 31, lr = lane >> 2, lc = lane & 3;
    TIO* Ab = A + (long)b * mstride + (long)r0g * np + r0g;
    TIO* Wb = W + (long)b * mstride + (long)r0g * np + r0g;
    TIO* ld = ldp + (long)b * ldp_stride + r0g / TILE;
    if (tid == 0) fail = 0;
    long long* tp = PROF ? prof + (long)b * 64 : nullptr;
    HBEGP_STAMP();
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int i = ty + 16 * a, k = tx + 16 * q;
            if (k <= i) {
                at[k][i] = (double)Ab[(long)i * np + k];
                w2[k][i] = (double)Ab[(long)(i + TILE) * np + TILE + k];  // A22, transposed as well
            }
            pm[i][k] = (double)Ab[(long)(i + TILE) * np + k];  // A21
        }
    HBEGP_STAMP();
    double rdprod1, rdprod2;
    leaf_mma<PROF>(at, w1, rdv, dinv, &fail, tid, rdprod1, tp, PROF ? prof + (long)b * 64 + 16 : nullptr);
    double acc[8][2];
    // L21 = A21 W11^T -> qm
    prod_a_wt(pm, w1, acc, warp, lr, lc);
#pragma unroll
    for (int j = 0; j < 8; j++)
        *reinterpret_cast<double2*>(&qm[8 * warp + lr][8 * j + 2 * lc]) = make_double2(acc[j][0], acc[j][1]);
    __syncthreads();
    HBEGP_STAMP();
    // (A22 - L21 L21^T)^T -> at: the 36 lower tiles dealt round-robin (warp w: tiles w, w + 8, ..), as C'[c][r]
    {
        int tr[5], tc[5];
#pragma unroll
        for (int s5 = 0; s5 < 5; s5++) {
            lower_tile_of(min(warp + 8 * s5, 35), tr[s5], tc[s5]);
            acc[s5][0] = acc[s5][1] = 0.0;
        }
        const int mine = (warp + 32 < 36) ? 5 : 4;
#pragma unroll 4
        for (int k4 = 0; k4 < TILE; k4 += 4) {
#pragma unroll
            for (int s5 = 0; s5 < 5; s5++)
                if (s5 < mine) dmma_acc(acc[s5][0], acc[s5][1], qm[8 * tc[s5] + lr][k4 + lc], qm[8 * tr[s5] + lr][k4 + lc]);
        }
#pragma unroll
        for (int s5 = 0; s5 < 5; s5++)
            if (s5 < mine) {
                const int row = 8 * tc[s5] + lr, col = 8 * tr[s5] + 2 * lc;
                const double2 o = *reinterpret_cast<const double2*>(&w2[row][col]);
                *reinterpret_cast<double2*>(&at[row][col]) = make_double2(o.x - acc[s5][0], o.y - acc[s5][1]);
            }
    }
    // T = L21 W11 -> pm (A21 is dead since the barrier above)
    prod_a_w(qm, w1, acc, warp, lr, lc);
#pragma unroll
    for (int j = 0; j < 8; j++)
        *reinterpret_cast<double2*>(&pm[8 * warp + lr][8 * j + 2 * lc]) = make_double2(acc[j][0], acc[j][1]);
    __syncthreads();  // leaf_mma starts by clearing w2, which holds A22^T until here
    HBEGP_STAMP();
    leaf_mma<PROF>(at, w2, rdv, dinv, &fail, tid, rdprod2, tp, PROF ? prof + (long)b * 64 + 40 : nullptr, &rdprod1);
    // W21 = -W22 T, straight to global memory
    prod_w_b(w2, pm, acc, warp, lr, lc);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        TIO* dst = &Wb[(long)(8 * i + lr + TILE) * np + 8 * warp + 2 * lc];
        if constexpr (sizeof(TIO) == 8) *reinterpret_cast<double2*>(dst) = make_double2(-acc[i][0], -acc[i][1]);
        else *reinterpret_cast<float2*>(dst) = make_float2((float)-acc[i][0], (float)-acc[i][1]);
    }
    HBEGP_STAMP();
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int i = ty + 16 * a, k = tx + 16 * q;
            Wb[(long)i * np + k] = (TIO)w1[i][k];            // zeros above the diagonal
            Wb[(long)i * np + TILE + k] = TIO(0);            // (0,1) block: read by the 128-wide GEMM tiles' triangular k ranges
            Wb[(long)(i + TILE) * np + TILE + k] = (TIO)w2[i][k];
        }
    // sum ln L_kk = -1/2 ln prod 1 / u_kk: the eight partial products per half sit in threads 64 + 24 j
    {
        const int idx = tid - TILE;
        if (idx >= 0 && idx % 24 == 0) {
            rdv[idx / 24] = rdprod1;  // already -1/2 ln (taken during the second leaf)
            rdv[8 + idx / 24] = -0.5 * log(rdprod2);
        }
        __syncthreads();
        if (tid < 2) {
            double s = 0.0;
#pragma unroll
            for (int j = 0; j < 8; j++) s += rdv[8 * tid + j];
            ld[tid] = (TIO)s;
        }
    }
    if (tid == 0 && fail) status[b] = 1;
    HBEGP_STAMP();
}

#undef HBEGP_STAMP

}  // namespace hbegp
