// The acquisition epilogue (k_acquisition) and the arg-best pick (launch_argbest) of hbetune_rs_b200/csrc/kernels.cuh
// behind a C ABI, so that tests can feed them any mean, variance and key vectors (non-finite values, the std-zero
// threshold, planted ties, more than 2^31 elements) instead of what a model predicts.  Buffers are device pointers the
// caller owns; tests/test_acquisition.py drives it with torch.  dtype: 0 f64, 1 f32.
#include "kernels.cuh"

extern "C" {

int acq_argbest_parts(long m) { return hbegp::argbest_parts(m); }
size_t acq_argbest_ws_bytes(long m) { return hbegp::argbest_ws_bytes(m); }

// out1 / out2 as in ModelT::predict_acquisition (mode 0: de-normalised mean, EI; mode 1: confidence bound, out2
// unused); amplitude, expected and cb are rounded to the data type first, as the library does.  Asynchronous on
// `stream`; returns a cudaError_t.
int acq_epilogue(int dtype, const void* mean, const void* var, long m, int mode, int proj, double amplitude,
                 double expected, double fmin_n, double cb, void* out1, void* out2, void* stream) {
    if (m <= 0) return 0;
    const unsigned blocks = (unsigned)((m + 255) / 256);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dtype == 0)
        hbegp::k_acquisition<double><<<blocks, 256, 0, st>>>((const double*)mean, (const double*)var, m, mode, proj, amplitude,
                                                             expected, fmin_n, cb, (double*)out1, (double*)out2);
    else
        hbegp::k_acquisition<float><<<blocks, 256, 0, st>>>((const float*)mean, (const float*)var, m, mode, proj,
                                                            (float)amplitude, (float)expected, fmin_n, (float)cb,
                                                            (float*)out1, (float*)out2);
    return (int)cudaGetLastError();
}

// *out (device) = the arg-best of key[0, m); ws of acq_argbest_ws_bytes(m) bytes.
int acq_argbest(int dtype, const void* key, long m, int want_max, void* ws, long* out, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dtype == 0) return (int)hbegp::launch_argbest<double>((const double*)key, m, want_max, ws, out, st);
    return (int)hbegp::launch_argbest<float>((const float*)key, m, want_max, ws, out, st);
}

}  // extern "C"
