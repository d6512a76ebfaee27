// The acquisition search (hbegp_acquire_ei / hbegp_acquire_confidence_bound) restated on the host from lbfgs.h itself:
// one BoundedLbfgs per start and, every round, one public hbegp_predict_mean_ei_grad / hbegp_predict_confidence_bound_grad
// call on all S rows in start order (a finished start's row keeps its last trial point, its result is ignored), the
// capture rule of fit_runs_impl per start and the reference's best-index rules across starts.  Built with the library's
// host flags (-ffp-contract=off); tests/test_acquire.py loads it and requires the device search to equal it bit for bit.
#include <cmath>
#include <cstring>
#include <limits>
#include <vector>

#include "hbegp.h"
#include "lbfgs.h"

using hbegp::BoundedLbfgs;

template <typename T>
static int restate(hbegp_model* model, const hbegp_ynorm* yn, int mode, double param, long S, const T* starts, const double* lo,
                   const double* hi, int maxeval, T* x_out, T* mean_out, hbegp_acq_result* results, long* best_index,
                   long long* n_rounds) {
    const int d = hbegp_model_dim(model);
    std::vector<BoundedLbfgs> opt;
    opt.reserve(S);
    std::vector<double> x0(d);
    for (long i = 0; i < S; i++) {
        for (int k = 0; k < d; k++) x0[k] = (double)starts[i * d + k];
        opt.emplace_back(d, x0.data(), lo, hi, maxeval);
        results[i] = {std::numeric_limits<double>::quiet_NaN(), -1, 0, HBEGP_NOT_PD, 0};
        for (int k = 0; k < d; k++) x_out[i * d + k] = (T)opt[i].ask()[k];
        if (mean_out) mean_out[i] = std::numeric_limits<T>::quiet_NaN();
    }
    std::vector<double> best_f(S, 0.0), g(d);
    std::vector<T> xs((size_t)S * d), v1(S), v2(S), gr((size_t)S * d);
    long long rounds = 0;
    for (;;) {
        bool any = false;
        for (long i = 0; i < S; i++) any = any || !opt[i].done();
        if (!any) break;
        rounds++;
        for (long i = 0; i < S; i++)
            for (int k = 0; k < d; k++) xs[i * d + k] = (T)opt[i].ask()[k];
        int rc = (mode == 0) ? hbegp_predict_mean_ei_grad(model, yn, S, xs.data(), param, v1.data(), v2.data(), nullptr, gr.data(), nullptr)
                             : hbegp_predict_confidence_bound_grad(model, yn, S, xs.data(), param, v1.data(), gr.data(), nullptr);
        if (rc < 0) return rc;
        for (long i = 0; i < S; i++) {
            if (opt[i].done()) continue;
            const double f = (mode == 0) ? -(double)v2[i] : (double)v1[i];
            hbegp_acq_result& r = results[i];
            if (std::isfinite(f) && (r.best_eval < 0 || f < best_f[i])) {
                best_f[i] = f;
                r.best_eval = opt[i].evals();
                r.status = HBEGP_OK;
                r.best_value = (mode == 0) ? -f : f;
                std::memcpy(x_out + i * d, xs.data() + i * d, sizeof(T) * d);
                if (mean_out && mode == 0) mean_out[i] = v1[i];
            }
            for (int k = 0; k < d; k++) g[k] = (mode == 0) ? -(double)gr[i * d + k] : (double)gr[i * d + k];
            opt[i].tell(f, g.data());
            r.n_evals = opt[i].evals();
        }
    }
    long best = -1;
    for (long i = 0; i < S; i++) {
        if (results[i].status != HBEGP_OK) continue;
        const double v = results[i].best_value;
        if (best < 0 || (mode == 0 ? v >= results[best].best_value : v < results[best].best_value)) best = i;
    }
    *best_index = best;
    *n_rounds = rounds;
    return HBEGP_OK;
}

// The arguments of hbegp_acquire_ei (mode 0, param = fmin) / hbegp_acquire_confidence_bound (mode 1, param = cb), plus
// the stopping tolerances (the copy of lbfgs.h compiled here keeps its own).
extern "C" int acq_restatement(hbegp_model* model, const hbegp_ynorm* yn, int mode, double param, long S, const void* starts,
                               const double* lo, const double* hi, int maxeval, double ftol, double gtol, void* x_out,
                               void* mean_out, hbegp_acq_result* results, long* best_index, long long* n_rounds) {
    hbegp::lbfgs_tolerances().ftol = ftol;
    hbegp::lbfgs_tolerances().gtol = gtol;
    if (yn->dtype == HBEGP_F64)
        return restate<double>(model, yn, mode, param, S, (const double*)starts, lo, hi, maxeval, (double*)x_out, (double*)mean_out,
                               results, best_index, n_rounds);
    return restate<float>(model, yn, mode, param, S, (const float*)starts, lo, hi, maxeval, (float*)x_out, (float*)mean_out, results,
                          best_index, n_rounds);
}
