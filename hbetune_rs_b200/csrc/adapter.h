// Host-side mirror of the thin adapter the reference keeps around src/gpr (C++; no GPU work in here):
//   YNormalize              src/core/ynormalize.rs:158-320
//   estimate_amplitude      src/core/gpr.rs:429-450
//   expected_improvement    src/core/acquisition.rs:141-171
//   normal inverse CDF      statrs 0.12 Normal::inverse_cdf as used by predict_statistics (gpr.rs:140-166)
// Array arithmetic is done in the data type A (f32 under --use-32), scalars the reference keeps in f64 stay f64.
#pragma once
#include <algorithm>
#include <cmath>
#include <limits>
#include <vector>

namespace hbegp {

constexpr double FUDGE_MIN = 0.05;  // ynormalize.rs:5
enum { PROJ_LINEAR = 0, PROJ_LOG = 1 };

template <typename A>
struct YNorm {
    A amplitude = A(1), expected = A(0);
    int projection = PROJ_LINEAR;

    // ynormalize.rs:291-320
    static A guess_min(bool has_ko, A ko, const A* y, long n, A minimum) {
        A mn = y[0];
        for (long i = 1; i < n; i++) mn = std::min(mn, y[i]);
        mn = mn - minimum;
        if (has_ko && ko < mn) return ko;
        return mn;
    }
    static A guess_amplitude(const A* y, long n) {
        A acc = A(0);  // ndarray mean_axis: sequential sum / n
        for (long i = 0; i < n; i++) acc = acc + y[i];
        A amp = acc / A(n);
        return amp > A(0) ? amp : A(1);
    }
    // new_project_into_normalized (ynormalize.rs:162-195); y_out may alias y
    void fit(int proj, const A* y, long n, bool has_ko, A ko, A* y_out) {
        projection = proj;
        std::vector<A> t(n);
        if (proj == PROJ_LINEAR) {
            expected = guess_min(has_ko, ko, y, n, A(0));
            for (long i = 0; i < n; i++) t[i] = y[i] - expected;
            amplitude = guess_amplitude(t.data(), n);
            for (long i = 0; i < n; i++) y_out[i] = t[i] / amplitude + A(FUDGE_MIN);
        } else {
            expected = guess_min(has_ko, ko, y, n, A(1));
            for (long i = 0; i < n; i++) t[i] = std::log(y[i] - expected);
            amplitude = guess_amplitude(t.data(), n);
            for (long i = 0; i < n; i++) y_out[i] = t[i] / amplitude;
        }
    }
    A into(A y) const {  // project_into_normalized
        return projection == PROJ_LINEAR ? (y - expected) / amplitude + A(FUDGE_MIN) : std::log(y - expected) / amplitude;
    }
    A location_from(A y) const {  // project_location_from_normalized
        return projection == PROJ_LINEAR ? (y - A(FUDGE_MIN)) * amplitude + expected : std::exp(y * amplitude) + expected;
    }
    A mean_from(A mean, A var) const {  // project_mean_from_normalized
        if (projection == PROJ_LINEAR) return (mean - A(FUDGE_MIN)) * amplitude + expected;
        A mean_amp = mean * amplitude, var_amp = var * amplitude * amplitude;
        return std::exp(mean_amp + var_amp / A(2)) + expected;
    }
    A std_from(A mean, A var) const {  // project_std_from_normalized
        if (projection == PROJ_LINEAR) return std::sqrt(var) * amplitude;
        A mu = mean * amplitude, s2 = var * amplitude * amplitude;
        return std::sqrt(std::exp(mu * A(2) + s2) * (std::exp(s2) - A(1)));
    }
    A cv_from(A mean, A var) const {  // project_cv_from_normalized
        if (projection == PROJ_LINEAR) return std::sqrt(var) * amplitude / ((mean - A(FUDGE_MIN)) * amplitude + expected);
        return std::sqrt(std::exp(var * (amplitude * amplitude)) - A(1));
    }
};

// ndarray 0.13 `sum()` on a contiguous slice (numeric_util::unrolled_fold): eight partial sums
template <typename A>
static A nd_sum(const A* xs, long n) {
    A p[8] = {A(0), A(0), A(0), A(0), A(0), A(0), A(0), A(0)};
    long i = 0;
    for (; i + 8 <= n; i += 8)
        for (int k = 0; k < 8; k++) p[k] = p[k] + xs[i + k];
    A acc = A(0);
    acc = acc + (p[0] + p[4]);
    acc = acc + (p[1] + p[5]);
    acc = acc + (p[2] + p[6]);
    acc = acc + (p[3] + p[7]);
    for (; i < n; i++) acc = acc + xs[i];
    return acc;
}

// estimate_amplitude (gpr.rs:429-450): out = {start, lo, hi}
template <typename A>
static void estimate_amplitude(const A* y, long n, const double* bounds, double out[3]) {
    double lo, hi;
    if (bounds) {
        lo = bounds[0];
        hi = bounds[1];
    } else {
        std::vector<A> sq(n);
        for (long i = 0; i < n; i++) sq[i] = y[i] * y[i];
        hi = (double)nd_sum(sq.data(), n);
        std::vector<double> s(n);
        for (long i = 0; i < n; i++) s[i] = (double)y[i];
        std::sort(s.begin(), s.end());
        // ndarray-stats 0.3 quantile_mut(0.1, Lower): element floor((n - 1) q) of the sorted data
        double q = s[(long)std::floor((double)(n - 1) * 0.1)];
        lo = q * q * (double)n;
        lo = lo > 2e-5 ? lo : 2e-5;
        lo = lo / 2.0;
        hi = hi * 2.0;
    }
    out[0] = std::exp((std::log(lo) + std::log(hi)) / 2.0);
    out[1] = lo;
    out[2] = hi;
}

static inline double norm_cdf(double z) { return 0.5 * std::erfc(-z / std::sqrt(2.0)); }
static inline double norm_pdf(double z) { return std::exp(-0.5 * z * z) / std::sqrt(2.0 * M_PI); }

// expected_improvement (acquisition.rs:141-171); NaN signals the reference's assertion failures
static inline double expected_improvement(double mean, double std, double fmin) {
    // both predicates live in kernels.cuh, shared with k_acquisition
    if (!ei_inputs_finite(mean, std, fmin)) return std::numeric_limits<double>::quiet_NaN();
    if (ei_std_is_zero(std)) return mean < fmin ? -(mean - fmin) : 0.0;
    const double z = -(mean - fmin) / std;
    return -(mean - fmin) * norm_cdf(z) + std * norm_pdf(z);
}

// Standard normal quantile, Wichura's AS 241 (PPND16), |relative error| < 1e-16.
static inline double norm_ppf(double p) {
    const double q = p - 0.5;
    if (std::fabs(q) <= 0.425) {
        const double r = 0.180625 - q * q;
        const double num = (((((((2.5090809287301226727e3 * r + 3.3430575583588128105e4) * r + 6.7265770927008700853e4) * r +
                                4.5921953931549871457e4) * r + 1.3731693765509461125e4) * r + 1.9715909503065514427e3) * r +
                             1.3314166789178437745e2) * r + 3.3871328727963666080e0);
        const double den = (((((((5.2264952788528545610e3 * r + 2.8729085735721942674e4) * r + 3.9307895800092710610e4) * r +
                                2.1213794301586595867e4) * r + 5.3941960214247511077e3) * r + 6.8718700749205790830e2) * r +
                             4.2313330701600911252e1) * r + 1.0);
        return q * num / den;
    }
    double r = q < 0 ? p : 1.0 - p;
    r = std::sqrt(-std::log(r));
    double val;
    if (r <= 5.0) {
        r -= 1.6;
        const double num = (((((((7.74545014278341407640e-4 * r + 2.27238449892691845833e-2) * r + 2.41780725177450611770e-1) * r +
                                1.27045825245236838258e0) * r + 3.64784832476320460504e0) * r + 5.76949722146069140550e0) * r +
                             4.63033784615654529590e0) * r + 1.42343711074968357734e0);
        const double den = (((((((1.05075007164441684324e-9 * r + 5.47593808499534494600e-4) * r + 1.51986665636164571966e-2) * r +
                                1.48103976427480074590e-1) * r + 6.89767334985100004550e-1) * r + 1.67638483018380384940e0) * r +
                             2.05319162663775882187e0) * r + 1.0);
        val = num / den;
    } else {
        r -= 5.0;
        const double num = (((((((2.01033439929228813265e-7 * r + 2.71155556874348757815e-5) * r + 1.24266094738807843860e-3) * r +
                                2.65321895265761230930e-2) * r + 2.96560571828504891230e-1) * r + 1.78482653991729133580e0) * r +
                             5.46378491116411436990e0) * r + 6.65790464350110377720e0);
        const double den = (((((((2.04426310338993978564e-15 * r + 1.42151175831644588870e-7) * r + 1.84631831751005468180e-5) * r +
                                7.86869131145613259100e-4) * r + 1.48753612908506148525e-2) * r + 1.36929880922735805310e-1) * r +
                             5.99832206555887937690e-1) * r + 1.0);
        val = num / den;
    }
    return q < 0 ? -val : val;
}

}  // namespace hbegp
