// Probe: time per launch of the 128-wide bottom node k_node128_v2 (node_mma.cuh) in f64, with the per-phase clock
// stamps of its PROF build (thread 0 of matrix 0) and the failure flags of the indefinite test block.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o probes/leaf2_bench probes/leaf2_bench.cu
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "../hbetune_rs_b200/csrc/node_mma.cuh"
using namespace hbegp;
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); exit(1);} } while (0)

float run_v2(int B, const double* A0, double* A, double* W, int np, double* ldp, int* st, int reps) {
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    size_t bytes = (size_t)B * np * np * sizeof(double), smem = node128_v2_smem_bytes();
    CK(cudaFuncSetAttribute(k_node128_v2<false, double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaFuncSetAttribute(k_node128_v2<true, double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    {
        long long* prof; CK(cudaMalloc(&prof, B * 64 * 8)); CK(cudaMemset(prof, 0, B * 64 * 8));
        CK(cudaMemcpy(A, A0, bytes, cudaMemcpyDeviceToDevice));
        k_node128_v2<true, double><<<dim3(1, 1, B), 256, smem>>>(A, W, (long)np * np, np, 0, ldp, np / 64, st, prof);
        CK(cudaDeviceSynchronize());
        long long h[64]; CK(cudaMemcpy(h, prof, 64 * 8, cudaMemcpyDeviceToHost));
        const char* names[] = {"load", "chol1", "lvl0_1", "lvls1", "L21", "syrk+T", "chol2", "lvl0_2", "lvls2", "W21", "store+logdet"};
        printf("   v2 phases (cycles, matrix 0):");
        for (int i = 0; i < 11; i++) printf(" %s %lld", names[i], h[i + 1] - h[i]);
        printf(" | total %lld\n", h[11] - h[0]);
        for (int leaf = 0; leaf < 2; leaf++) {
            const long long* q = h + (leaf ? 40 : 16);
            printf("   leaf %d panel iterations (cycles):", leaf + 1);
            for (int P = 0; P < 8; P++) printf(" %lld", q[P + 1] - q[P]);  // prologue (panel 0), then iterations 0..6
            printf("\n");
        }
        cudaFree(prof);
    }
    float total = 0;
    for (int r = 0; r < reps + 1; r++) {
        CK(cudaMemcpy(A, A0, bytes, cudaMemcpyDeviceToDevice));
        CK(cudaMemset(W, 0xff, bytes));
        CK(cudaMemset(st, 0, B * sizeof(int)));
        CK(cudaDeviceSynchronize());
        cudaEventRecord(e0);
        k_node128_v2<false, double><<<dim3(1, 1, B), 256, smem>>>(A, W, (long)np * np, np, 0, ldp, np / 64, st, nullptr);
        cudaEventRecord(e1); CK(cudaEventSynchronize(e1));
        CK(cudaGetLastError());
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        if (r > 0) total += ms;
    }
    return total / reps * 1e3f;
}

int main() {
    const int np = 128;
    for (int B : {1, 33, 148}) {
        size_t elems = (size_t)B * np * np, bytes = elems * sizeof(double);
        double *A0, *A, *W, *ldp; int* st;
        CK(cudaMalloc(&A0, bytes)); CK(cudaMalloc(&A, bytes)); CK(cudaMalloc(&W, bytes));
        CK(cudaMalloc(&ldp, B * 2 * sizeof(double))); CK(cudaMalloc(&st, B * 4));
        // SPD test blocks: Matern-like kernel matrix of random 3-d points + noise (condition number ~1e3..1e5), one
        // indefinite matrix (b == 5) to check the failure flag
        std::vector<double> h(elems);
        srand(7);
        for (int b = 0; b < B; b++) {
            std::vector<double> pts(np * 3);
            for (auto& v : pts) v = rand() / (double)RAND_MAX;
            for (int i = 0; i < np; i++)
                for (int j = 0; j < np; j++) {
                    double d2 = 0;
                    for (int k = 0; k < 3; k++) { double t = (pts[i * 3 + k] - pts[j * 3 + k]) / 0.4; d2 += t * t; }
                    double r = sqrt(5.0 * d2);
                    double v = 1.7 * (1 + r + r * r / 3) * exp(-r) + (i == j ? 0.01 : 0.0);
                    if (b == 5 && i == j && i == 70) v = -1.0;
                    h[(size_t)b * np * np + (size_t)i * np + j] = v;
                }
        }
        CK(cudaMemcpy(A0, h.data(), bytes, cudaMemcpyHostToDevice));
        printf("B=%3d\n", B);
        const float us = run_v2(B, A0, A, W, np, ldp, st, 10);
        std::vector<int> s(B);
        CK(cudaMemcpy(s.data(), st, B * 4, cudaMemcpyDeviceToHost));
        int nfail = 0;
        for (int b = 0; b < B; b++) nfail += s[b];
        printf("B=%3d k_node128_v2 %.1f us per launch, failed %d (expected %d)\n", B, us, nfail, B > 5 ? 1 : 0);
        cudaFree(A0); cudaFree(A); cudaFree(W); cudaFree(ldp); cudaFree(st);
    }
    return 0;
}
