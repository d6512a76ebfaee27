"""Host-side mirror of ``src/core/gpr.rs``: ``EstimatorGPR`` (builder + ``estimate`` / ``extend``) and
``SurrogateModelGPR`` (the ``SurrogateModel`` trait of ``src/core/surrogate_model.rs:34-65``).

The arithmetic lives in ``libhbegp.so``: GPU kernels for fit / predict, C++ for y-normalisation,
amplitude estimate, expected improvement and the normal quantile.  This file only wires them together in
the order the reference does.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np

from . import _lib
from ._lib import check, lib
from .gpr import BoundedValue, BoundsError, ConstantKernel, Context, FittedKernel, Matern, Product, _ptr

LINEAR, LOGARITHMIC = 0, 1  # Projection::{Linear, Logarithmic} (ynormalize.rs:14-18)


class Error(Exception):
    """``src/core/gpr.rs:452-473``."""


class NoiseBounds(Error):
    def __init__(self, e: BoundsError):
        super().__init__(f"noise level {e.value} violated bounds [{e.min}, {e.max}] during model fitting")


class LengthScaleBounds(Error):
    def __init__(self, e: BoundsError):
        super().__init__(f"length scale {e.value} violated bounds [{e.min}, {e.max}] during model fitting")


class YNormalize:
    """``src/core/ynormalize.rs:158-288`` (C++ implementation behind ``hbegp_ynorm_*``)."""

    def __init__(self, raw: _lib.YNorm, A):
        self._raw, self.A = raw, A

    amplitude = property(lambda self: self._raw.amplitude)
    expected = property(lambda self: self._raw.expected)
    projection = property(lambda self: self._raw.projection)

    @classmethod
    def new_project_into_normalized(cls, y, projection=LINEAR, known_optimum: Optional[float] = None, A=np.float64):
        y = np.ascontiguousarray(y, dtype=A)
        out = np.empty_like(y)
        raw = _lib.YNorm()
        ko = None if known_optimum is None else C.byref(C.c_double(known_optimum))
        check(lib.hbegp_ynorm_fit(_lib.F64 if A == np.float64 else _lib.F32, projection, y.shape[0], _ptr(y), ko,
                                  _ptr(out), C.byref(raw)), "hbegp_ynorm_fit")
        return out, cls(raw, A)

    def _apply(self, op, a, b=None):
        a = np.ascontiguousarray(np.atleast_1d(a), dtype=self.A)
        b = None if b is None else np.ascontiguousarray(np.atleast_1d(b), dtype=self.A)
        out = np.empty_like(a)
        check(lib.hbegp_ynorm_apply(C.byref(self._raw), op, a.shape[0], _ptr(a), _ptr(b), _ptr(out)), "hbegp_ynorm_apply")
        return out

    def project_into_normalized(self, y):
        return self._apply(0, y)

    def project_location_from_normalized(self, y):
        return self._apply(1, y)

    def project_mean_from_normalized(self, mean, variance):
        return self._apply(2, mean, variance)

    def project_std_from_normalized(self, mean, variance):
        return self._apply(3, mean, variance)

    def project_cv_from_normalized(self, mean, variance):
        return self._apply(4, mean, variance)


def estimate_amplitude(y: np.ndarray, bounds: Optional[Tuple[float, float]] = None) -> BoundedValue:
    """``src/core/gpr.rs:429-450``."""
    y = np.ascontiguousarray(y)
    out = (C.c_double * 3)()
    b = None if bounds is None else (C.c_double * 2)(*bounds)
    check(lib.hbegp_estimate_amplitude(_lib.F64 if y.dtype == np.float64 else _lib.F32, y.shape[0], _ptr(y), b, out),
          "hbegp_estimate_amplitude")
    return BoundedValue(out[0], out[1], out[2])


def expected_improvement(mean: float, std: float, fmin: float) -> float:
    """``src/core/acquisition.rs:141-171``."""
    ei = lib.hbegp_expected_improvement(mean, std, fmin)
    assert math.isfinite(ei), f"EI must be finite: {ei}"
    return ei


@dataclass
class SummaryStatistics:
    """``src/core/surrogate_model.rs:67-135``."""

    mean: float
    std: float
    cv: float
    q1: float
    q2: float
    q3: float

    def median(self):
        return self.q2

    def q13(self):
        return self.q1, self.q3

    def iqr(self):
        return self.q3 - self.q1


class SurrogateModelGPR:
    """``src/core/gpr.rs:53-213``.  ``fitted.model`` keeps X, alpha and L^-1 on the GPU."""

    def __init__(self, fitted: FittedKernel, x_train, y_train, y_norm: YNormalize, A):
        self.fitted, self.x_train, self.y_train, self.y_norm, self.A = fitted, x_train, y_train, y_norm, A
        self.kernel, self.noise, self.lml = fitted.kernel, fitted.noise, fitted.lml
        self.alpha, self.k_inv = fitted.alpha, fitted.k_inv

    def length_scales(self) -> List[float]:
        return [b.value for b in self.kernel.k2.length_scale]

    # -- normalised-space prediction (src/gpr/predict.rs)
    def _predict(self, x, want_variance):
        x = np.ascontiguousarray(x, dtype=self.A)
        return self.fitted.model.predict(x, want_variance)

    def predict_mean_a(self, x):
        mean, _ = self._predict(x, False)
        return self.y_norm.project_location_from_normalized(mean)

    def predict_mean(self, x):
        return self.predict_mean_a(np.asarray(x)[None, :])[0]

    def predict_mean_ei_a(self, x, fmin):
        mean, var = self._predict(x, True)
        fmin_n = float(self.y_norm.project_into_normalized(np.array([fmin]))[0])
        ei = np.empty_like(mean)
        check(lib.hbegp_expected_improvement_a(_lib.F64 if self.A == np.float64 else _lib.F32, mean.shape[0], _ptr(mean),
                                               _ptr(var), fmin_n, _ptr(ei)), "hbegp_expected_improvement_a")
        assert np.isfinite(ei).all(), "EI must be finite"
        return self.y_norm.project_location_from_normalized(mean), ei

    def predict_mean_ei_device(self, x, fmin, want_best: bool = True):
        """SURVEY section 8 rows f1/f2: the whole of predict_mean_ei_a plus find_best_candidate_by_ei's argmax
        (acquisition.rs:177-202, last maximum wins) in one device pass.  Returns (mean, ei, best_index)."""
        x = np.ascontiguousarray(x, dtype=self.A)
        m = x.shape[0]
        mean, ei = np.empty(m, dtype=self.A), np.empty(m, dtype=self.A)
        best, nb = C.c_long(-1), C.c_long(0)
        check(lib.hbegp_predict_mean_ei(self.fitted.model.single_handle(), C.byref(self.y_norm._raw), m, _ptr(x), float(fmin), _ptr(mean),
                                        _ptr(ei), C.byref(best) if want_best else None, C.byref(nb)), "hbegp_predict_mean_ei")
        return mean, ei, best.value

    def predict_confidence_bound_device(self, x, cb, want_best: bool = True):
        """predict_confidence_bound for many points + find_best_individual_by_confidence_bound's argmin
        (minimize.rs:680-714, first minimum wins).  Returns (bounds, best_index)."""
        x = np.ascontiguousarray(x, dtype=self.A)
        m = x.shape[0]
        out = np.empty(m, dtype=self.A)
        best, nb = C.c_long(-1), C.c_long(0)
        check(lib.hbegp_predict_confidence_bound(self.fitted.model.single_handle(), C.byref(self.y_norm._raw), m, _ptr(x), float(cb), _ptr(out),
                                                 C.byref(best) if want_best else None, C.byref(nb)),
              "hbegp_predict_confidence_bound")
        return out, best.value

    def predict_mean_ei_grad(self, x, fmin):
        """``hbegp_predict_mean_ei_grad``: (mean, ei, dmean, dei) for the rows of x, the values as
        ``predict_mean_ei_device`` and the gradients in the candidate of shape (m, d) (dmean de-normalised, dei in
        normalised units)."""
        x = np.ascontiguousarray(x, dtype=self.A)
        m, d = x.shape
        mean, ei = np.empty(m, dtype=self.A), np.empty(m, dtype=self.A)
        dmean, dei = np.empty((m, d), dtype=self.A), np.empty((m, d), dtype=self.A)
        nb = C.c_long(0)
        check(lib.hbegp_predict_mean_ei_grad(self.fitted.model.single_handle(), C.byref(self.y_norm._raw), m, _ptr(x), float(fmin),
                                             _ptr(mean), _ptr(ei), _ptr(dmean), _ptr(dei), C.byref(nb)), "hbegp_predict_mean_ei_grad")
        return mean, ei, dmean, dei

    def predict_confidence_bound_grad(self, x, cb):
        """``hbegp_predict_confidence_bound_grad``: (bounds, dbounds) for the rows of x, dbounds of shape (m, d)."""
        x = np.ascontiguousarray(x, dtype=self.A)
        m, d = x.shape
        out, dout = np.empty(m, dtype=self.A), np.empty((m, d), dtype=self.A)
        nb = C.c_long(0)
        check(lib.hbegp_predict_confidence_bound_grad(self.fitted.model.single_handle(), C.byref(self.y_norm._raw), m, _ptr(x),
                                                      float(cb), _ptr(out), _ptr(dout), C.byref(nb)),
              "hbegp_predict_confidence_bound_grad")
        return out, dout

    def _acquire_args(self, starts, lo, hi):
        starts = np.ascontiguousarray(np.atleast_2d(starts), dtype=self.A)
        d = starts.shape[1]
        lo = np.ascontiguousarray(np.broadcast_to(np.asarray(lo, dtype=np.float64), (d,)))
        hi = np.ascontiguousarray(np.broadcast_to(np.asarray(hi, dtype=np.float64), (d,)))
        return starts, lo, hi

    def acquire_ei(self, starts, lo, hi, fmin, maxeval: int = 150):
        """``hbegp_acquire_ei``: one bounded L-BFGS search maximising EI from each row of ``starts`` over the box
        [lo, hi], all on the device.  Returns (x, mean, records, best_index, n_rounds): the best point of each start
        (S x d) and the de-normalised mean there, the ``AcqResult`` records (best_value = EI in normalised units), the
        winning start (last maximum; -1 if none) and the number of rounds."""
        starts, lo, hi = self._acquire_args(starts, lo, hi)
        S, d = starts.shape
        x, mean = np.empty((S, d), dtype=self.A), np.empty(S, dtype=self.A)
        res = (_lib.AcqResult * S)()
        best, rounds = C.c_long(-1), C.c_longlong(0)
        check(lib.hbegp_acquire_ei(self.fitted.model.single_handle(), C.byref(self.y_norm._raw), float(fmin), S, _ptr(starts),
                                   _ptr(lo), _ptr(hi), maxeval, _ptr(x), _ptr(mean), res, C.byref(best), C.byref(rounds)),
              "hbegp_acquire_ei")
        return x, mean, list(res), best.value, rounds.value

    def acquire_confidence_bound(self, starts, lo, hi, cb, maxeval: int = 150):
        """``hbegp_acquire_confidence_bound``: one bounded L-BFGS search minimising the de-normalised confidence bound
        from each row of ``starts``.  Returns (x, records, best_index, n_rounds) (first minimum wins)."""
        starts, lo, hi = self._acquire_args(starts, lo, hi)
        S, d = starts.shape
        x = np.empty((S, d), dtype=self.A)
        res = (_lib.AcqResult * S)()
        best, rounds = C.c_long(-1), C.c_longlong(0)
        check(lib.hbegp_acquire_confidence_bound(self.fitted.model.single_handle(), C.byref(self.y_norm._raw), float(cb), S,
                                                 _ptr(starts), _ptr(lo), _ptr(hi), maxeval, _ptr(x), res, C.byref(best),
                                                 C.byref(rounds)), "hbegp_acquire_confidence_bound")
        return x, list(res), best.value, rounds.value

    def predict_mean_ei(self, x, fmin):
        mean, ei = self.predict_mean_ei_a(np.asarray(x)[None, :], fmin)
        return mean[0], ei[0]

    def predict_confidence_bound(self, x, cb):
        mnorm, vnorm = self._predict(np.asarray(x)[None, :], True)
        return self.y_norm.project_location_from_normalized(mnorm + np.sqrt(vnorm) * self.A(cb))[0]

    def predict_statistics(self, x) -> SummaryStatistics:
        mnorm, vnorm = self._predict(np.asarray(x)[None, :], True)
        std_n, mean_n = float(np.sqrt(vnorm[0])), float(mnorm[0])
        if abs(std_n) <= np.finfo(np.float64).eps:  # abs_diff_eq!(vnorm_scalar, 0.0)
            q = np.array([mean_n] * 3, dtype=self.A)
        else:
            q = np.array([lib.hbegp_normal_inverse_cdf(p, mean_n, std_n) for p in (0.25, 0.5, 0.75)], dtype=self.A)
        q = self.y_norm.project_location_from_normalized(q)
        return SummaryStatistics(
            mean=self.y_norm.project_mean_from_normalized(mnorm, vnorm)[0],
            std=self.y_norm.project_std_from_normalized(mnorm, vnorm)[0],
            cv=self.y_norm.project_cv_from_normalized(mnorm, vnorm)[0],
            q1=q[0], q2=q[1], q3=q[2])


# ---- the callers of the model that predict one point per call in the reference (SURVEY section 8 row f1), on
#      already projected feature rows (Space::project_into_features is outside the path), one device pass each
def find_best_candidate_by_ei(candidate_features, model: SurrogateModelGPR, fmin) -> Tuple[int, float, float]:
    """``acquisition.rs:177-202``: (index, mean, ei) of the candidate with maximal EI; ``max_by`` keeps the LAST
    maximum; a non-comparable (NaN) EI is the reference's panic."""
    x = np.ascontiguousarray(candidate_features, dtype=model.A)
    if x.shape[0] == 0:
        raise RuntimeError("there should be a candidate with maximal EI")
    mean, ei, best = model.predict_mean_ei_device(x, fmin)
    if np.isnan(ei).any():
        bad = int(np.flatnonzero(np.isnan(ei))[0])
        raise RuntimeError(f"EI should be comparable: a={ei[bad]} b={ei[bad]}")
    return best, mean[best], ei[best]


def find_best_individual_by_confidence_bound(individual_features, model: SurrogateModelGPR, confidence_bound) -> Tuple[int, float]:
    """``minimize.rs:680-714``: index of the individual with the lowest confidence bound (strict ``<``: the FIRST
    minimum stays) and the predicted mean there."""
    x = np.ascontiguousarray(individual_features, dtype=model.A)
    if x.shape[0] == 0:
        raise RuntimeError("should have at least one individual")
    _, best = model.predict_confidence_bound_device(x, confidence_bound)
    return best, model.predict_mean(x[best])


def predicted_fitness(individual_features, model: SurrogateModelGPR) -> np.ndarray:
    """``FitnessOperator::get_fitness`` with ``FitnessVia::Prediction`` (``minimize.rs:654-669``) for a whole
    population at once: the predicted means the selection compares."""
    return model.predict_mean_a(np.ascontiguousarray(individual_features, dtype=model.A))


class EstimatorGPR:
    """``src/core/gpr.rs:215-400`` (``Estimator::new`` takes the space; only its length is used)."""

    def __init__(self, n_features: int, ctx: Optional[Context] = None, dtype=np.float64):
        self.noise_bounds = (1e-5, 1e5)
        self.length_scale_bounds = [(1e-3, 1e3)] * n_features
        self._n_restarts_optimizer = 2
        self._matern_nu = 5.0 / 2.0
        self._amplitude_bounds = None
        self._y_projection = LINEAR
        self._known_optimum = None
        self.A = dtype
        self.ctx = ctx or Context(0, _lib.F64 if dtype == np.float64 else _lib.F32)
        self.shard = None  # optional multi-GPU run sharding (hbetune_rs_b200.dist.sharded_fit_runs)

    # builder methods (gpr.rs:351-400)
    def with_noise_bounds(self, lo, hi):
        self.noise_bounds = (lo, hi)
        return self

    def with_length_scale_bounds(self, bounds):
        self.length_scale_bounds = list(bounds)
        return self

    def n_restarts_optimizer(self, n):
        self._n_restarts_optimizer = n
        return self

    def matern_nu(self, nu):
        self._matern_nu = nu
        return self

    def amplitude_bounds(self, bounds):
        self._amplitude_bounds = bounds
        return self

    def y_projection(self, projection):
        self._y_projection = projection
        return self

    def known_optimum(self, value):
        self._known_optimum = value
        return self

    def _kernel_or_default(self, prior: Optional[SurrogateModelGPR], amplitude: BoundedValue):
        # gpr.rs:402-427
        if prior is not None:
            return prior.kernel, prior.noise
        try:
            noise = BoundedValue(1.0, *self.noise_bounds)
        except BoundsError as e:
            raise NoiseBounds(e)
        try:
            ls = [BoundedValue(math.exp((math.log(lo) + math.log(hi)) / 2.0), lo, hi) for lo, hi in self.length_scale_bounds]
        except BoundsError as e:
            raise LengthScaleBounds(e)
        return Product(ConstantKernel(amplitude), Matern(self._matern_nu, ls)), noise

    def estimate(self, x, y, prior: Optional[SurrogateModelGPR], rng, maxeval: int = 150, want_kinv: bool = False):
        """gpr.rs:238-291.  ``rng`` needs ``fork_random_state()`` returning an object with ``uniform_inclusive``."""
        x = np.ascontiguousarray(x, dtype=self.A)
        assert len(y) == x.shape[0], f"expected y values for {x.shape[0]} observations: {y}"
        y_train, y_norm = YNormalize.new_project_into_normalized(y, self._y_projection, self._known_optimum, self.A)
        amplitude = estimate_amplitude(y_train, self._amplitude_bounds)
        kernel, noise = self._kernel_or_default(prior, amplitude)
        fk = FittedKernel.new(self.ctx, kernel, x, y_train, rng.fork_random_state(), self._n_restarts_optimizer, noise,
                              maxeval=maxeval, want_kinv=want_kinv, shard=self.shard)
        return SurrogateModelGPR(fk, x, y_train, y_norm, self.A)

    def extend(self, x, y, prior: SurrogateModelGPR, rng=None, want_kinv: bool = False):
        """gpr.rs:293-337."""
        x = np.ascontiguousarray(x, dtype=self.A)
        assert len(y) == x.shape[0]
        y_train, y_norm = YNormalize.new_project_into_normalized(y, self._y_projection, self._known_optimum, self.A)
        fk = FittedKernel.extend(self.ctx, prior.kernel, x, y_train, prior.noise, want_kinv=want_kinv, prior=prior.fitted)
        return SurrogateModelGPR(fk, x, y_train, y_norm, self.A)
