// The emulated f64 product K^-1 = W^T W of hbetune_rs_b200/csrc/gemm_i8.cuh behind a C ABI, so that tests can feed it
// arbitrary W (non-finite columns, exponent extremes, rounding ties, the edges of the CRT range) instead of the W = L^-1
// a factorisation produces.  Buffers are device pointers the caller owns; tests/test_kinv_bits.py drives it with torch.
#include "gemm_i8.cuh"

extern "C" {

// Workspace bytes of one np x np matrix (residue planes and column exponents).
size_t oz_slot_bytes(int np) { return hbegp::oz::slot_bytes(np); }

// The b of the scheme: W is scaled per column to b bits.
int oz_scale_bits(int np) { return hbegp::oz::scale_bits(np); }

// The lower 64 x 64 tiles of C_b = W_b^T W_b for cnt matrices mstride elements apart, with ws of cnt * oz_slot_bytes(np)
// bytes; asynchronous on `stream`.  Returns a cudaError_t.
int oz_kinv(const double* W, double* C, long mstride, int np, int cnt, void* ws, void* stream) {
    static const cudaError_t cfg = hbegp::oz::configure();
    if (cfg != cudaSuccess) return (int)cfg;
    return (int)hbegp::oz::launch_kinv(W, C, mstride, np, cnt, static_cast<unsigned char*>(ws), static_cast<cudaStream_t>(stream));
}

}  // extern "C"
