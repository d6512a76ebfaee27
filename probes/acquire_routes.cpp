// Timed routes of a multi-start acquisition search over a model, driven from C++ so that no interpreter sits in the
// loop (probes/acquire_bench.py compiles this file against libhbegp.so and loads it):
//   time_device:         hbegp_acquire_ei;
//   time_fit_runs_with:  the route before it: hbegp_fit_runs_with as the lockstep bounded L-BFGS over the box given as
//                        exp(lo), exp(hi), one hbegp_predict_mean_ei_grad call on the live rows per round;
//   time_one_point:      `calls` one-point hbegp_predict_mean_ei calls, the shape of BOBYQA's batch-of-1 evaluations.
// Each returns the milliseconds of the whole run (host clock, every call ends in a stream synchronise).
#include <chrono>
#include <cmath>
#include <vector>

#include "hbegp.h"

static double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

extern "C" double time_device(hbegp_model* model, const hbegp_ynorm* yn, double fmin, long S, const void* starts, const double* lo,
                              const double* hi, int maxeval, long long* n_rounds) {
    const int d = hbegp_model_dim(model);
    const size_t es = yn->dtype == HBEGP_F64 ? 8 : 4;
    std::vector<char> x((size_t)S * d * es), mean((size_t)S * es);
    std::vector<hbegp_acq_result> res(S);
    long best = -1;
    const double t0 = now_ms();
    if (hbegp_acquire_ei(model, yn, fmin, S, starts, lo, hi, maxeval, x.data(), mean.data(), res.data(), &best, n_rounds)) return -1;
    return now_ms() - t0;
}

namespace {
struct EiState {
    hbegp_model* model;
    const hbegp_ynorm* yn;
    double fmin;
    long long rounds;
    std::vector<char> xs, mean, ei, dei;
};

template <typename T>
int ei_objective_t(EiState* s, int B, int p, const double* th, double* out, double* grad, int* status) {
    s->xs.resize((size_t)B * p * sizeof(T));
    s->mean.resize((size_t)B * sizeof(T));
    s->ei.resize((size_t)B * sizeof(T));
    s->dei.resize((size_t)B * p * sizeof(T));
    T* xs = (T*)s->xs.data();
    for (long t = 0; t < (long)B * p; t++) xs[t] = (T)th[t];
    if (hbegp_predict_mean_ei_grad(s->model, s->yn, B, xs, s->fmin, s->mean.data(), s->ei.data(), nullptr, s->dei.data(), nullptr))
        return 1;
    const T* ei = (const T*)s->ei.data();
    const T* dei = (const T*)s->dei.data();
    for (int b = 0; b < B; b++) {
        out[b] = (double)ei[b];  // maximised as the "LML"
        status[b] = std::isfinite(out[b]) ? HBEGP_OK : HBEGP_NOT_PD;
        for (int k = 0; k < p; k++) grad[(size_t)b * p + k] = (double)dei[(size_t)b * p + k];
    }
    s->rounds++;
    return 0;
}

int ei_objective(void* user, int B, int p, const double* th, double* out, double* grad, int* status) {
    EiState* s = (EiState*)user;
    return s->yn->dtype == HBEGP_F64 ? ei_objective_t<double>(s, B, p, th, out, grad, status)
                                     : ei_objective_t<float>(s, B, p, th, out, grad, status);
}
}  // namespace

extern "C" double time_fit_runs_with(hbegp_model* model, const hbegp_ynorm* yn, double fmin, int S, const double* starts,
                                     const double* lo, const double* hi, int maxeval, long long* n_rounds) {
    const int d = hbegp_model_dim(model);
    std::vector<double> blo(d), bhi(d), best((size_t)S * d);
    for (int k = 0; k < d; k++) {
        blo[k] = std::exp(lo[k]);
        bhi[k] = std::exp(hi[k]);
    }
    std::vector<hbegp_run_result> res(S);
    EiState s{model, yn, fmin, 0, {}, {}, {}, {}};
    const double t0 = now_ms();
    if (hbegp_fit_runs_with(ei_objective, &s, d, S, starts, blo.data(), bhi.data(), maxeval, 0, 1, nullptr, nullptr, res.data(),
                            best.data()))
        return -1;
    const double ms = now_ms() - t0;
    *n_rounds = s.rounds;
    return ms;
}

extern "C" double time_one_point(hbegp_model* model, const hbegp_ynorm* yn, double fmin, long calls, const void* points) {
    const int d = hbegp_model_dim(model);
    const size_t es = yn->dtype == HBEGP_F64 ? 8 : 4;
    double mean[1], ei[1];
    const double t0 = now_ms();
    for (long c = 0; c < calls; c++)
        if (hbegp_predict_mean_ei(model, yn, 1, (const char*)points + (size_t)c * d * es, fmin, mean, ei, nullptr, nullptr)) return -1;
    return now_ms() - t0;
}
