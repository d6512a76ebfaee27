// hbegp.hpp — C++ host-side mirror of the reference's GP interface on top of the C ABI (hbegp.h).
//
// Same names, argument meaning and error behaviour as the Rust reference (latk/hbetune.rs):
//   BoundedValue / BoundsError            src/util/bounded_value.rs
//   ConstantKernel, Matern, Product        src/gpr/{constant,matern,product}_kernel.rs   (parameters; evaluation is on the GPU)
//   RNG                                    src/core/random.rs
//   FittedKernel::{create, extend}, predict   src/gpr/fit.rs, src/gpr/predict.rs
//   YNormalize, EstimatorGPR, SurrogateModelGPR, SummaryStatistics   src/core/{ynormalize,gpr,surrogate_model}.rs
// It is the C++ twin of the `impl Estimator<A>` sketched in INTEGRATION.md and is what tests/cpp exercises.
// Header-only; link with -lhbegp.  Panics of the reference are std::runtime_error here.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <memory>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "hbegp.h"

namespace hbegp_cpp {

struct BoundsError : std::runtime_error {
    double value, min, max;
    BoundsError(double v, double lo, double hi)
        : std::runtime_error("value " + std::to_string(v) + " violated bounds [" + std::to_string(lo) + ", " + std::to_string(hi) + "]"),
          value(v), min(lo), max(hi) {}
};

struct GpuError : std::runtime_error {
    int code;
    GpuError(int c, const std::string& where) : std::runtime_error(where + ": " + hbegp_last_error()), code(c) {}
};
inline void check(int rc, const char* where) {
    if (rc < 0) throw GpuError(rc, where);
}

// src/util/bounded_value.rs:3-56
class BoundedValue {
public:
    BoundedValue(double value, double min, double max) : value_(value), min_(min), max_(max) {
        if (!(min <= value && value <= max)) throw BoundsError(value, min, max);
    }
    double value() const { return value_; }
    double min() const { return min_; }
    double max() const { return max_; }
    BoundedValue with_value(double v) const { return BoundedValue(v, min_, max_); }
    BoundedValue with_clamped_value(double v) const {
        if (v < min_) v = min_;
        else if (max_ < v) v = max_;
        return BoundedValue(v, min_, max_);
    }

private:
    double value_, min_, max_;
};

// src/gpr/constant_kernel.rs, matern_kernel.rs, product_kernel.rs: parameter holders with the reference's
// theta conventions (theta = ln of the natural values; Product = [constant | length scales]).
struct ConstantKernel {
    BoundedValue constant;
};
struct Matern {
    double nu;
    std::vector<BoundedValue> length_scale;
};
struct Product {
    ConstantKernel k1;
    Matern k2;
    size_t n_params() const { return 1 + k2.length_scale.size(); }
    std::vector<double> theta() const {
        std::vector<double> t{std::log(k1.constant.value())};
        for (auto& l : k2.length_scale) t.push_back(std::log(l.value()));
        return t;
    }
    std::vector<std::pair<double, double>> bounds() const {
        std::vector<std::pair<double, double>> b{{std::log(k1.constant.min()), std::log(k1.constant.max())}};
        for (auto& l : k2.length_scale) b.push_back({std::log(l.min()), std::log(l.max())});
        return b;
    }
    Product with_clamped_theta(const double* theta) const {
        Product out{{k1.constant.with_clamped_value(std::exp(theta[0]))}, {k2.nu, {}}};
        for (size_t k = 0; k < k2.length_scale.size(); k++)
            out.k2.length_scale.push_back(k2.length_scale[k].with_clamped_value(std::exp(theta[1 + k])));
        return out;
    }
};

// src/core/random.rs
class RNG {
public:
    static RNG new_with_seed(uint64_t seed) {
        RNG r;
        hbegp_rng_seed(seed, r.s_);
        return r;
    }
    RNG fork_random_state() {
        RNG c;
        hbegp_rng_fork(s_, c.s_);
        return c;
    }
    double uniform(double lo, double hi) { return hbegp_rng_uniform(s_, lo, hi); }  // lo..=hi

private:
    unsigned long long s_[4];
};

template <typename A>
constexpr int dtype_of() {
    static_assert(std::is_same<A, double>::value || std::is_same<A, float>::value, "A must be f64 or f32");
    return std::is_same<A, double>::value ? HBEGP_F64 : HBEGP_F32;
}

class Context {
public:
    Context(int device, int dtype) { check(hbegp_ctx_create(device, dtype, nullptr, &h_), "hbegp_ctx_create"); }
    ~Context() { hbegp_ctx_destroy(h_); }
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;
    hbegp_ctx* get() const { return h_; }

private:
    hbegp_ctx* h_ = nullptr;
};

struct ModelHandle {
    hbegp_model* h = nullptr;
    ~ModelHandle() { hbegp_model_destroy(h); }
};

// src/gpr/fit.rs:6-12 — alpha stays on the host like the reference's field; k_inv stays on the device
template <typename A>
struct FittedKernel {
    Product kernel;
    BoundedValue noise;
    std::vector<A> alpha;
    double lml;
    std::shared_ptr<ModelHandle> model;
    long n_evals;

    // FittedKernel::new (fit.rs:18-31, :71-176) with gradmin.rs:7-33's start-point draws
    static FittedKernel create(Context& ctx, const Product& kernel, const std::vector<A>& x, long n, int d,
                               const std::vector<A>& y, RNG& rng, size_t n_restarts_optimizer, const BoundedValue& noise) {
        if ((long)y.size() != n || (long)x.size() != n * d) throw std::runtime_error("assertion failed: y_train.dim() == n_observations");
        check(hbegp_set_data(ctx.get(), n, d, x.data(), y.data()), "hbegp_set_data");
        const size_t p = kernel.n_params() + 1;
        std::vector<double> lo{noise.min(), kernel.k1.constant.min()}, hi{noise.max(), kernel.k1.constant.max()};
        for (auto& l : kernel.k2.length_scale) {
            lo.push_back(l.min());
            hi.push_back(l.max());
        }
        std::vector<double> starts{std::log(noise.value())};
        for (double t : kernel.theta()) starts.push_back(t);
        for (size_t r = 0; r < n_restarts_optimizer; r++)
            for (size_t k = 0; k < p; k++) starts.push_back(rng.uniform(std::log(lo[k]), std::log(hi[k])));
        const int n_runs = 1 + (int)n_restarts_optimizer;
        std::vector<hbegp_run_result> res(n_runs);
        std::vector<double> best_theta((size_t)n_runs * p);
        check(hbegp_fit_runs(ctx.get(), kernel.k2.nu, n_runs, starts.data(), lo.data(), hi.data(), 150, res.data(), best_theta.data()),
              "hbegp_fit_runs");
        const int best = hbegp_pick_best_run(n_runs, res.data());
        if (best < 0) throw std::runtime_error("called `Option::unwrap()` on a `None` value");  // fit.rs:161
        const double* theta = &best_theta[(size_t)best * p];
        long evals = 0;
        for (auto& r : res) evals += r.n_evals;
        return finish(ctx, kernel.with_clamped_theta(theta + 1), noise.with_clamped_value((double)(A)std::exp(theta[0])), theta,
                      lo.data(), hi.data(), n, evals);
    }

    // FittedKernel::extend (fit.rs:33-68)
    static FittedKernel extend(Context& ctx, const Product& kernel, const std::vector<A>& x, long n, int d, const std::vector<A>& y,
                               const BoundedValue& noise) {
        check(hbegp_set_data(ctx.get(), n, d, x.data(), y.data()), "hbegp_set_data");
        std::vector<double> theta{std::log(noise.value())};
        for (double t : kernel.theta()) theta.push_back(t);
        return finish(ctx, kernel, noise, theta.data(), nullptr, nullptr, n, 1);
    }

    // FittedKernel::extend as the reference spells it -- `self` is the fitted kernel being extended.  The library
    // appends to the prior factorisation when the old rows are an unchanged prefix of x (hbegp_model_extend).
    FittedKernel extend(Context& ctx, const std::vector<A>& x, long n, int d, const std::vector<A>& y, bool* appended = nullptr) const {
        check(hbegp_set_data(ctx.get(), n, d, x.data(), y.data()), "hbegp_set_data");
        FittedKernel fk{kernel, noise, std::vector<A>(n), 0.0, std::make_shared<ModelHandle>(), 1};
        int app = 0;
        int rc = hbegp_model_extend(ctx.get(), model->h, &fk.model->h, &fk.lml, fk.alpha.data(), nullptr, &app);
        if (rc == HBEGP_NOT_PD) throw std::runtime_error("Kernel matrix must be invertible.");  // fit.rs:55
        check(rc, "hbegp_model_extend");
        if (appended) *appended = app != 0;
        return fk;
    }

private:
    static FittedKernel finish(Context& ctx, const Product& kernel, const BoundedValue& noise, const double* theta, const double* lo,
                               const double* hi, long n, long evals) {
        FittedKernel fk{kernel, noise, std::vector<A>(n), 0.0, std::make_shared<ModelHandle>(), evals};
        int rc = hbegp_model_create(ctx.get(), kernel.k2.nu, theta, lo, hi, &fk.model->h, &fk.lml, fk.alpha.data(), nullptr);
        if (rc == HBEGP_NOT_PD) throw std::runtime_error("Kernel matrix must be invertible.");  // fit.rs:55
        check(rc, "hbegp_model_create");
        return fk;
    }
};

// src/gpr/predict.rs:7-52; `variance` (may be null) is filled when wanted
template <typename A>
std::vector<A> predict(const FittedKernel<A>& fk, const std::vector<A>& x, long m, std::vector<A>* variance = nullptr) {
    std::vector<A> mean(m);
    long below = 0;
    if (variance) variance->assign(m, A(0));
    check(hbegp_predict(fk.model->h, m, x.data(), mean.data(), variance ? variance->data() : nullptr, &below), "hbegp_predict");
    if (below > 0) {  // predict.rs:39-46 lists the offending values ("{:.2e}", comma separated)
        std::vector<double> vals((size_t)std::min<long>(below, 4096));
        const int k = hbegp_predict_warn_values(fk.model->h, (int)vals.size(), vals.data(), nullptr);
        fprintf(stderr, "Variances below 0 were predicted and will be corrected: ");
        for (int i = 0; i < k; i++) fprintf(stderr, i ? ", %.2e" : "%.2e", vals[i]);
        fprintf(stderr, "\n");
    }
    return mean;
}

enum class Projection { Linear = HBEGP_PROJ_LINEAR, Logarithmic = HBEGP_PROJ_LOG };

// hbegp_predict_grad: the mean (returned), its gradient in the candidate (m x d, row-major) into *dmean and, when
// `variance` is given, the variance and its gradient into *variance / *dvar (normalised units)
template <typename A>
std::vector<A> predict_grad(const FittedKernel<A>& fk, const std::vector<A>& x, long m, int d, std::vector<A>* dmean,
                            std::vector<A>* variance = nullptr, std::vector<A>* dvar = nullptr) {
    std::vector<A> mean(m);
    dmean->assign((size_t)m * d, A(0));
    if (variance) variance->assign(m, A(0));
    if (dvar) dvar->assign((size_t)m * d, A(0));
    check(hbegp_predict_grad(fk.model->h, m, x.data(), mean.data(), variance ? variance->data() : nullptr, dmean->data(),
                             dvar ? dvar->data() : nullptr, nullptr),
          "hbegp_predict_grad");
    return mean;
}

// src/core/ynormalize.rs:158-288
template <typename A>
class YNormalize {
public:
    static std::pair<std::vector<A>, YNormalize> new_project_into_normalized(const std::vector<A>& y, Projection proj,
                                                                            const double* known_optimum) {
        YNormalize yn;
        std::vector<A> out(y.size());
        check(hbegp_ynorm_fit(dtype_of<A>(), (int)proj, (long)y.size(), y.data(), known_optimum, out.data(), &yn.raw_), "hbegp_ynorm_fit");
        return {out, yn};
    }
    std::vector<A> project_into_normalized(const std::vector<A>& y) const { return apply(0, y, nullptr); }
    std::vector<A> project_location_from_normalized(const std::vector<A>& y) const { return apply(1, y, nullptr); }
    std::vector<A> project_mean_from_normalized(const std::vector<A>& m, const std::vector<A>& v) const { return apply(2, m, &v); }
    std::vector<A> project_std_from_normalized(const std::vector<A>& m, const std::vector<A>& v) const { return apply(3, m, &v); }
    std::vector<A> project_cv_from_normalized(const std::vector<A>& m, const std::vector<A>& v) const { return apply(4, m, &v); }
    const hbegp_ynorm& raw() const { return raw_; }

private:
    std::vector<A> apply(int op, const std::vector<A>& a, const std::vector<A>* b) const {
        std::vector<A> out(a.size());
        check(hbegp_ynorm_apply(&raw_, op, (long)a.size(), a.data(), b ? b->data() : nullptr, out.data()), "hbegp_ynorm_apply");
        return out;
    }
    hbegp_ynorm raw_{};
};

// src/core/surrogate_model.rs:67-135
template <typename A>
struct SummaryStatistics {
    A mean, std, cv, q1, q2, q3;
    A median() const { return q2; }
    A iqr() const { return q3 - q1; }
};

// src/core/gpr.rs:53-213
template <typename A>
class SurrogateModelGPR {
public:
    SurrogateModelGPR(FittedKernel<A> fk, YNormalize<A> yn, int d) : fitted_(std::move(fk)), y_norm_(yn), d_(d) {}
    const Product& kernel() const { return fitted_.kernel; }
    const BoundedValue& noise() const { return fitted_.noise; }
    double lml() const { return fitted_.lml; }
    std::vector<double> length_scales() const {
        std::vector<double> out;
        for (auto& l : fitted_.kernel.k2.length_scale) out.push_back(l.value());
        return out;
    }
    std::vector<A> predict_mean_a(const std::vector<A>& x, long m) const {
        return y_norm_.project_location_from_normalized(predict(fitted_, x, m));
    }
    A predict_mean(const std::vector<A>& x) const { return predict_mean_a(x, 1)[0]; }
    // (mean, ei): gpr.rs:179-212, on the device in one pass; `best` (optional) = find_best_candidate_by_ei's index
    std::pair<std::vector<A>, std::vector<A>> predict_mean_ei_a(const std::vector<A>& x, long m, A fmin, long* best = nullptr) const {
        std::vector<A> mean(m), ei(m);
        long below = 0;
        check(hbegp_predict_mean_ei(fitted_.model->h, &y_norm_.raw(), m, x.data(), (double)fmin, mean.data(), ei.data(), best, &below),
              "hbegp_predict_mean_ei");
        for (A v : ei)
            if (!std::isfinite((double)v)) throw std::runtime_error("EI must be finite");
        return {mean, ei};
    }
    std::pair<A, A> predict_mean_ei(const std::vector<A>& x, A fmin) const {
        auto r = predict_mean_ei_a(x, 1, fmin);
        return {r.first[0], r.second[0]};
    }
    // predict_confidence_bound for m points in one pass; `best` (optional) = the index
    // find_best_individual_by_confidence_bound keeps (minimize.rs:680-714: strict `<`, first minimum)
    std::vector<A> predict_confidence_bound_a(const std::vector<A>& x, long m, A cb, long* best = nullptr) const {
        std::vector<A> out(m);
        check(hbegp_predict_confidence_bound(fitted_.model->h, &y_norm_.raw(), m, x.data(), (double)cb, out.data(), best, nullptr),
              "hbegp_predict_confidence_bound");
        return out;
    }
    // hbegp_predict_mean_ei_grad: (mean, ei) as predict_mean_ei_a, and their gradients in the candidate (m x d,
    // row-major; dmean de-normalised, dei in normalised units) into *dmean / *dei
    std::pair<std::vector<A>, std::vector<A>> predict_mean_ei_grad(const std::vector<A>& x, long m, A fmin, std::vector<A>* dmean,
                                                                   std::vector<A>* dei) const {
        std::vector<A> mean(m), ei(m);
        if (dmean) dmean->assign((size_t)m * d_, A(0));
        if (dei) dei->assign((size_t)m * d_, A(0));
        check(hbegp_predict_mean_ei_grad(fitted_.model->h, &y_norm_.raw(), m, x.data(), (double)fmin, mean.data(), ei.data(),
                                         dmean ? dmean->data() : nullptr, dei ? dei->data() : nullptr, nullptr),
              "hbegp_predict_mean_ei_grad");
        return {mean, ei};
    }
    // hbegp_predict_confidence_bound_grad: the bounds of m points, their gradients (m x d) into *dout
    std::vector<A> predict_confidence_bound_grad(const std::vector<A>& x, long m, A cb, std::vector<A>* dout) const {
        std::vector<A> out(m);
        if (dout) dout->assign((size_t)m * d_, A(0));
        check(hbegp_predict_confidence_bound_grad(fitted_.model->h, &y_norm_.raw(), m, x.data(), (double)cb, out.data(),
                                                  dout ? dout->data() : nullptr, nullptr),
              "hbegp_predict_confidence_bound_grad");
        return out;
    }
    // hbegp_acquire_ei: S bounded L-BFGS searches maximising EI from the rows of starts (S x d) over [lo, hi]; the best
    // point of each start into *x (S x d), the de-normalised mean there into *mean (may be NULL), the records into
    // *results; returns the winning start (-1 if none), the rounds into *n_rounds (may be NULL)
    long acquire_ei(const std::vector<A>& starts, long S, const std::vector<double>& lo, const std::vector<double>& hi, A fmin,
                    int maxeval, std::vector<A>* x, std::vector<A>* mean, std::vector<hbegp_acq_result>* results,
                    long long* n_rounds = nullptr) const {
        x->assign((size_t)S * d_, A(0));
        if (mean) mean->assign((size_t)S, A(0));
        results->assign((size_t)S, hbegp_acq_result{});
        long best = -1;
        long long rounds = 0;
        check(hbegp_acquire_ei(fitted_.model->h, &y_norm_.raw(), (double)fmin, S, starts.data(), lo.data(), hi.data(), maxeval,
                               x->data(), mean ? mean->data() : nullptr, results->data(), &best, &rounds),
              "hbegp_acquire_ei");
        if (n_rounds) *n_rounds = rounds;
        return best;
    }
    // hbegp_acquire_confidence_bound: the same, minimising the de-normalised confidence bound
    long acquire_confidence_bound(const std::vector<A>& starts, long S, const std::vector<double>& lo, const std::vector<double>& hi,
                                  A cb, int maxeval, std::vector<A>* x, std::vector<hbegp_acq_result>* results,
                                  long long* n_rounds = nullptr) const {
        x->assign((size_t)S * d_, A(0));
        results->assign((size_t)S, hbegp_acq_result{});
        long best = -1;
        long long rounds = 0;
        check(hbegp_acquire_confidence_bound(fitted_.model->h, &y_norm_.raw(), (double)cb, S, starts.data(), lo.data(), hi.data(),
                                             maxeval, x->data(), results->data(), &best, &rounds),
              "hbegp_acquire_confidence_bound");
        if (n_rounds) *n_rounds = rounds;
        return best;
    }
    A predict_confidence_bound(const std::vector<A>& x, A cb) const {
        A out;
        check(hbegp_predict_confidence_bound(fitted_.model->h, &y_norm_.raw(), 1, x.data(), (double)cb, &out, nullptr, nullptr),
              "hbegp_predict_confidence_bound");
        return out;
    }
    SummaryStatistics<A> predict_statistics(const std::vector<A>& x) const {
        std::vector<A> var;
        std::vector<A> mean = predict(fitted_, x, 1, &var);
        const double sd = std::sqrt((double)var[0]), mu = (double)mean[0];
        std::vector<A> q(3, (A)mu);
        if (!(std::fabs(sd) <= 2.220446049250313e-16))
            for (int i = 0; i < 3; i++) q[i] = (A)hbegp_normal_inverse_cdf(0.25 * (i + 1), mu, sd);
        q = y_norm_.project_location_from_normalized(q);
        return {y_norm_.project_mean_from_normalized(mean, var)[0], y_norm_.project_std_from_normalized(mean, var)[0],
                y_norm_.project_cv_from_normalized(mean, var)[0], q[0], q[1], q[2]};
    }
    const FittedKernel<A>& fitted() const { return fitted_; }

private:
    FittedKernel<A> fitted_;
    YNormalize<A> y_norm_;
    int d_;
};


// ---- the model's callers that predict one point per call in the reference (SURVEY 8 row f1), on already projected
//      feature rows (m x d, row major), one device pass each
struct BestCandidate {
    long index;
    double mean, ei;
};
// acquisition.rs:177-202 (max_by keeps the LAST maximum)
template <typename A>
BestCandidate find_best_candidate_by_ei(const std::vector<A>& candidate_features, long m, const SurrogateModelGPR<A>& model, A fmin) {
    if (m <= 0) throw std::runtime_error("there should be a candidate with maximal EI");
    long best = -1;
    auto r = model.predict_mean_ei_a(candidate_features, m, fmin, &best);
    return {best, (double)r.first[best], (double)r.second[best]};
}
// minimize.rs:680-714 (strict `<`: the FIRST minimum stays); returns the index and the predicted mean there
template <typename A>
std::pair<long, A> find_best_individual_by_confidence_bound(const std::vector<A>& individual_features, long m, int d,
                                                           const SurrogateModelGPR<A>& model, A confidence_bound) {
    if (m <= 0) throw std::runtime_error("should have at least one individual");
    long best = -1;
    model.predict_confidence_bound_a(individual_features, m, confidence_bound, &best);
    std::vector<A> row(individual_features.begin() + best * d, individual_features.begin() + (best + 1) * d);
    return {best, model.predict_mean(row)};
}
// src/core/gpr.rs:215-450
class EstimatorGPR {
public:
    struct Error : std::runtime_error {
        using std::runtime_error::runtime_error;
    };
    explicit EstimatorGPR(size_t n_features) : length_scale_bounds_(n_features, {1e-3, 1e3}) {}
    EstimatorGPR& noise_bounds(double lo, double hi) { noise_bounds_ = {lo, hi}; return *this; }
    EstimatorGPR& length_scale_bounds(std::vector<std::pair<double, double>> b) { length_scale_bounds_ = std::move(b); return *this; }
    EstimatorGPR& n_restarts_optimizer(size_t n) { n_restarts_ = n; return *this; }
    EstimatorGPR& matern_nu(double nu) { matern_nu_ = nu; return *this; }
    EstimatorGPR& amplitude_bounds(double lo, double hi) { has_amp_ = true; amp_[0] = lo; amp_[1] = hi; return *this; }
    EstimatorGPR& y_projection(Projection p) { y_projection_ = p; return *this; }
    EstimatorGPR& known_optimum(double v) { has_ko_ = true; ko_ = v; return *this; }

    template <typename A>
    SurrogateModelGPR<A> estimate(Context& ctx, const std::vector<A>& x, long n, const std::vector<A>& y,
                                  const SurrogateModelGPR<A>* prior, RNG& rng) const {
        const int d = (int)length_scale_bounds_.size();
        if ((long)y.size() != n) throw std::runtime_error("expected y values for " + std::to_string(n) + " observations");
        auto yn = YNormalize<A>::new_project_into_normalized(y, y_projection_, has_ko_ ? &ko_ : nullptr);  // gpr.rs:255-259
        double amp[3];
        check(hbegp_estimate_amplitude(dtype_of<A>(), n, yn.first.data(), has_amp_ ? amp_ : nullptr, amp), "hbegp_estimate_amplitude");
        auto kn = kernel_or_default(prior, BoundedValue(amp[0], amp[1], amp[2]));
        RNG fork = rng.fork_random_state();  // gpr.rs:276
        auto fk = FittedKernel<A>::create(ctx, kn.first, x, n, d, yn.first, fork, n_restarts_, kn.second);
        return SurrogateModelGPR<A>(std::move(fk), yn.second, d);
    }

    template <typename A>
    SurrogateModelGPR<A> extend(Context& ctx, const std::vector<A>& x, long n, const std::vector<A>& y,
                                const SurrogateModelGPR<A>& prior) const {
        const int d = (int)length_scale_bounds_.size();
        auto yn = YNormalize<A>::new_project_into_normalized(y, y_projection_, has_ko_ ? &ko_ : nullptr);
        auto fk = prior.fitted().extend(ctx, x, n, d, yn.first);
        return SurrogateModelGPR<A>(std::move(fk), yn.second, d);
    }

private:
    template <typename A>
    std::pair<Product, BoundedValue> kernel_or_default(const SurrogateModelGPR<A>* prior, const BoundedValue& amplitude) const {
        if (prior) return {prior->kernel(), prior->noise()};  // gpr.rs:407-409
        try {
            BoundedValue noise(1.0, noise_bounds_.first, noise_bounds_.second);
            std::vector<BoundedValue> ls;
            try {
                for (auto& b : length_scale_bounds_) ls.emplace_back(std::exp((std::log(b.first) + std::log(b.second)) / 2.0), b.first, b.second);
            } catch (const BoundsError& e) {
                throw Error("length scale " + std::to_string(e.value) + " violated bounds [" + std::to_string(e.min) + ", " +
                            std::to_string(e.max) + "] during model fitting");
            }
            return {Product{{amplitude}, {matern_nu_, ls}}, noise};
        } catch (const BoundsError& e) {
            throw Error("noise level " + std::to_string(e.value) + " violated bounds [" + std::to_string(e.min) + ", " +
                        std::to_string(e.max) + "] during model fitting");
        }
    }
    std::pair<double, double> noise_bounds_{1e-5, 1e5};
    std::vector<std::pair<double, double>> length_scale_bounds_;
    size_t n_restarts_ = 2;
    double matern_nu_ = 2.5;
    bool has_amp_ = false, has_ko_ = false;
    double amp_[2] = {0, 0}, ko_ = 0;
    Projection y_projection_ = Projection::Linear;
};

}  // namespace hbegp_cpp
