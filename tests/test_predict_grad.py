"""Gradients in the candidate of the predictive mean, variance, EI and confidence bound (hbegp_predict_grad,
hbegp_predict_mean_ei_grad, hbegp_predict_confidence_bound_grad).

With x~_k = x_k / l_k and s_j = sum_k (x~_k - X~_jk)^2, d k*_j / d x_k = -c dk_factor(s_j) (x~_k - X~_jk) / l_k and

    dmean = sum_j alpha_j grad k*_j,     dvar = -2 sum_j v_j grad k*_j,     v = K^-1 k*.

The truth of both (`_grad_star`) is built from the accurate alpha*, W* of `Truth` (tests/test_f64_truth.py) and checked
against mpmath.diff of the posterior mean and variance at 40 digits on the CPU.  On the GPU the f64 gradients follow the
rule of the other f64 tests: |g_gpu - g*| <= R |g_LAPACK - g*| + F eps S(g), g_LAPACK the same formula in NumPy from
LAPACK's factor of the GPU's own K and S the condition sum.  The chain rules of the epilogue (EI, the confidence bound,
the de-normalisation) are checked against mpmath.diff, then the device epilogue against them applied to
hbegp_predict_grad's own outputs.  Central differences of hbegp_predict_mean_ei catch sign and l-versus-l^2 errors.
"""
import ctypes
import json
import math
import os

import numpy as np
import pytest

from tests.test_acquisition import STD_ZERO, _acq, _ei_mp
from tests.test_dispatch_sweep import _ctx, _kernel_f64, _note, _np, _predict_path, _reference, _rounded
from tests.test_f64_truth import EPS, F, R, SLACK, Truth, _candidates, _family, _gpu_k, _two_prod, dd_matmul
from tests.util import random_thetas, synth

# ------------------------------------------------------------------------------------------------ the formulas


def _dk_factor(s, nu):
    """matern_grad_terms' dk_factor = -2 dM/ds (0 at s = 0 for nu = 1/2)."""
    if nu == 0.5:
        r = np.sqrt(s)
        with np.errstate(divide="ignore", invalid="ignore"):
            return np.where(r > 0, np.exp(-r) / r, 0.0)
    if nu == 1.5:
        return 3.0 * np.exp(-np.sqrt(3.0 * s))
    t = np.sqrt(5.0 * s)
    return np.exp(-t) * (t + 1.0) * (5.0 / 3.0)


def _grad_kstar(xs, x, c, ls, nu, dtype=np.float64):
    """G[k][r, j] = d k*_rj / d xs_rk = -c dk_factor(s_rj) (x~_rk - X~_jk) / l_k, in `dtype`."""
    xs, x, ls = (np.asarray(a, dtype=dtype) for a in (xs, x, ls))
    a, b = xs / ls, x / ls
    diffs = [a[:, k, None] - b[None, :, k] for k in range(a.shape[1])]
    s = sum(df * df for df in diffs)
    f = _dk_factor(s.astype(np.float64), nu).astype(dtype)
    return [-dtype(c) * f * df / ls[k] for k, df in enumerate(diffs)]


def _dot_rows(vterms, g):
    """sum_j v_rj g_rj to about 2^-100 (TwoProduct on the leading term, exact sums), as float."""
    vh = vterms[0]
    p, e = _two_prod(vh, g)
    rest = sum(t * g for t in vterms[1:]) if len(vterms) > 1 else np.zeros_like(g)
    return np.array([math.fsum(np.concatenate([p[r], e[r], rest[r]])) for r in range(g.shape[0])])


def _grad_star(tr, theta, x, xs, nu):
    """dmean*, dvar* (m x d) from the truth's alpha* and W*, with the condition sums S(dmean), S(dvar)."""
    c, ls = math.exp(theta[1]), np.exp(np.asarray(theta[2:], dtype=np.float64))
    ks = _kernel_f64(xs, x, c, ls, nu)
    g = _grad_kstar(xs, x, c, ls, nu)
    uh, ul = dd_matmul(tuple(tr.ws), ks.T)
    vh, vl = dd_matmul(tuple(t.T for t in tr.ws), (uh, ul))  # v* = W*^T W* k*^T, n x m
    vt = [vh.T, vl.T]
    at = [np.broadcast_to(a, ks.shape) for a in tr.alpha]
    dm = np.stack([_dot_rows(at, gk) for gk in g], axis=1)
    dv = np.stack([-2.0 * _dot_rows(vt, gk) for gk in g], axis=1)
    w0 = np.abs(tr.ws[0])
    vbound = (w0.T @ (w0 @ np.abs(ks.T))).T  # |W|^T |W| |k*|: the scale of v's rounding
    s_m = np.stack([np.abs(gk) @ np.abs(tr.alpha[0]) for gk in g], axis=1)
    s_v = np.stack([2.0 * (vbound * np.abs(gk)).sum(axis=1) for gk in g], axis=1)
    return dm, dv, s_m, s_v


def _grad_numpy(w, alpha, theta, x, xs, nu, dtype=np.float64):
    """The same formulas in NumPy in `dtype` from a given factor W and alpha (LAPACK's, say)."""
    c, ls = dtype(math.exp(theta[1])), np.exp(np.asarray(theta[2:], dtype=np.float64)).astype(dtype)
    ks = _kernel_f64(np.asarray(xs, np.float64), np.asarray(x, np.float64), float(c), ls.astype(np.float64), nu).astype(dtype)
    g = _grad_kstar(xs, x, c, ls, nu, dtype)
    v = (ks @ w.T.astype(dtype)) @ w.astype(dtype)
    dm = np.stack([gk @ alpha.astype(dtype) for gk in g], axis=1)
    dv = np.stack([-2.0 * (v * gk).sum(axis=1) for gk in g], axis=1)
    return dm, dv


def _chain(mu, var, dmu, dvar, mode, proj, amplitude, fmin_n=0.0, cb=0.0):
    """The chain rules of k_acquisition_grad in f64: (d location, dEI) for mode 0, d location for mode 1."""
    mu, var = float(mu), float(var)
    sd = math.sqrt(var)
    dsd = dvar / (2.0 * sd) if sd > 0 else np.zeros_like(dvar)
    y = mu if mode == 0 else mu + sd * cb
    lf = amplitude if proj == 0 else amplitude * math.exp(y * amplitude)
    if mode == 1:
        return lf * (dmu + cb * dsd), None
    if not (math.isfinite(mu) and math.isfinite(sd) and math.isfinite(fmin_n)):
        dei = np.full_like(dmu, np.nan)
    elif sd <= STD_ZERO:
        dei = -dmu if mu < fmin_n else np.zeros_like(dmu)
    else:
        z = -(mu - fmin_n) / sd
        dei = -0.5 * math.erfc(-z / math.sqrt(2)) * dmu + math.exp(-0.5 * z * z) / math.sqrt(2 * math.pi) * dsd
    return lf * dmu, dei


def _record(key, payload):
    """Adds measured ratios to the JSON file named by HBEGP_GRAD_NOTES (profiles/r09_predict_grad.json holds one such
    record) and to the sweep notes."""
    _note(key, payload)
    path = os.environ.get("HBEGP_GRAD_NOTES")
    if not path:
        return
    data = {}
    if os.path.exists(path):
        with open(path) as f:
            data = json.load(f)
    data[key] = payload
    with open(path, "w") as f:
        json.dump(data, f, indent=1, sort_keys=True)


# ------------------------------------------------------------------------------------------------ CPU: the truth


def _mp_posterior(k, x, y, theta, nu):
    """mean(x) and var(x) as mpmath functions of the candidate, from K given exactly (at the caller's workdps)."""
    import mpmath
    n, d = x.shape
    c = mpmath.mpf(math.exp(theta[1]))
    ls = [mpmath.mpf(float(v)) for v in np.exp(np.asarray(theta[2:], dtype=np.float64))]
    K = mpmath.matrix(n, n)
    for i in range(n):
        for j in range(n):
            K[i, j] = mpmath.mpf(float(k[i, j]))
    Kinv = K ** -1
    alpha = Kinv * mpmath.matrix([mpmath.mpf(float(v)) for v in y])
    xt = [[mpmath.mpf(float(x[j, q])) / ls[q] for q in range(d)] for j in range(n)]

    def corr(s):
        if nu == 0.5:
            return mpmath.exp(-mpmath.sqrt(s))
        if nu == 1.5:
            t = mpmath.sqrt(3 * s)
            return (1 + t) * mpmath.exp(-t)
        t = mpmath.sqrt(5 * s)
        return (1 + t + t * t / 3) * mpmath.exp(-t)

    def kstar(*xv):
        return mpmath.matrix([c * corr(mpmath.fsum((xv[q] / ls[q] - xt[j][q]) ** 2 for q in range(d))) for j in range(n)])

    def mean(*xv):
        return mpmath.fsum(a * b for a, b in zip(kstar(*xv), alpha))

    def var(*xv):
        ksv = kstar(*xv)
        return c + mpmath.mpf("1e-5") - mpmath.fsum(a * b for a, b in zip(ksv, Kinv * ksv))

    return mean, var


@pytest.mark.parametrize("nu", [0.5, 1.5, 2.5])
def test_truth_is_the_derivative(nu):
    """_grad_star against mpmath.diff of the posterior mean and variance at 40 digits (K given), small n, candidates
    away from the training points.  The truth contracts the f64 grad k* (rounded like any f64 evaluation of it), so it
    agrees to a few eps of the condition sum S, the scale of the F eps S term of the GPU rule."""
    import mpmath
    n, d = 12, 2
    x, y = synth(n, d, seed=3)
    theta = random_thetas(1, d, seed=4, noise=(1e-3, 1e-3 * 1.01))[0]
    c, ls, noise = math.exp(theta[1]), np.exp(theta[2:]), math.exp(theta[0])
    k = _kernel_f64(x, x, c, ls, nu) + noise * np.eye(n)
    tr = Truth(k, y, theta, x, nu)
    xs = np.array([[0.37, 0.61], [1.2, -0.3]])
    dm, dv, s_m, s_v = _grad_star(tr, theta, x, xs, nu)
    with mpmath.workdps(40):
        mean, var = _mp_posterior(k, x, y, theta, nu)
        for r in range(xs.shape[0]):
            pt = [mpmath.mpf(float(v)) for v in xs[r]]
            for q in range(d):
                order = [0] * d
                order[q] = 1
                gm = float(mpmath.diff(mean, pt, tuple(order)))
                gv = float(mpmath.diff(var, pt, tuple(order)))
                assert abs(dm[r, q] - gm) <= 8 * EPS * s_m[r, q], (r, q, dm[r, q], gm)
                assert abs(dv[r, q] - gv) <= 8 * EPS * s_v[r, q], (r, q, dv[r, q], gv)


def _mp_loc(y, proj, amplitude):
    import mpmath
    return (y - mpmath.mpf("0.05")) * amplitude if proj == 0 else mpmath.exp(y * amplitude)


@pytest.mark.parametrize("proj", [0, 1])
def test_epilogue_chain_rules_against_mpmath(proj):
    """_chain's EI and confidence-bound derivatives against mpmath.diff of _ei_mp and location_from along a direction,
    with (mu, var) moving linearly: dmu, dvar given.  Regular branch, the std-zero branch (sigma = 0 and
    sigma <= eps), sigma = 0 for the bound, and NaN inputs."""
    import mpmath
    amplitude, fmin_n, cb = 0.7, 0.4, -1.5
    dmu, dvar = np.array([0.3, -1.1]), np.array([0.02, 0.05])
    with mpmath.workdps(40):
        for mu, var in ((0.1, 0.09), (0.9, 0.25), (0.4, 1e-3)):
            for q in range(2):
                def ei_along(t, q=q):
                    return _ei_mp(mu + t * dmu[q], mpmath.sqrt(var + t * dvar[q]), fmin_n)

                def cb_along(t, q=q):
                    return _mp_loc(mu + t * dmu[q] + cb * mpmath.sqrt(var + t * dvar[q]), proj, amplitude)

                def mean_along(t, q=q):
                    return _mp_loc(mu + t * dmu[q], proj, amplitude)

                dloc, dei = _chain(mu, var, dmu, dvar, 0, proj, amplitude, fmin_n)
                dcb, _ = _chain(mu, var, dmu, dvar, 1, proj, amplitude, cb=cb)
                for got, f in ((dei[q], ei_along), (dloc[q], mean_along), (dcb[q], cb_along)):
                    want = float(mpmath.diff(f, 0))
                    assert abs(got - want) <= 1e-14 * max(1.0, abs(want)), (mu, var, q, got, want)
    # std-zero branch: -dmu below fmin, 0 above; sigma = 0 leaves the bound with dmu alone
    for var in (0.0, STD_ZERO ** 2 / 4):
        _, dei = _chain(0.1, var, dmu, dvar, 0, proj, amplitude, fmin_n)
        np.testing.assert_array_equal(dei, -dmu)
        _, dei = _chain(0.9, var, dmu, dvar, 0, proj, amplitude, fmin_n)
        np.testing.assert_array_equal(dei, 0.0 * dmu)
    dcb, _ = _chain(0.1, 0.0, dmu, dvar, 1, 0, amplitude, cb=cb)
    np.testing.assert_array_equal(dcb, amplitude * dmu)
    for mu, var, f in ((np.nan, 0.1, 0.0), (0.1, np.inf, 0.0), (0.1, 0.1, np.inf)):
        _, dei = _chain(mu, var, dmu, dvar, 0, proj, amplitude, f)
        assert np.isnan(dei).all()


# ------------------------------------------------------------------------------------------------ GPU


def _grad(model, xs, want_variance=True):
    return model.predict_grad(np.ascontiguousarray(xs, dtype=model.A), want_variance)


def _acq_grad(model, yn, xs, mode, param):
    """hbegp_predict_mean_ei_grad (mode 0) / hbegp_predict_confidence_bound_grad (mode 1): (out1, out2, dout1, dout2, nb)."""
    from hbetune_rs_b200._lib import check, lib
    from hbetune_rs_b200.gpr import _ptr
    A = yn.A
    xs = np.ascontiguousarray(xs, dtype=A)
    m, d = xs.shape
    o1, o2 = np.full(m, np.nan, dtype=A), np.full(m, np.nan, dtype=A)
    g1, g2 = np.full((m, d), np.nan, dtype=A), np.full((m, d), np.nan, dtype=A)
    nb = ctypes.c_long(-7)
    if mode == 0:
        check(lib.hbegp_predict_mean_ei_grad(model.single_handle(), ctypes.byref(yn._raw), m, _ptr(xs), float(param),
                                             _ptr(o1), _ptr(o2), _ptr(g1), _ptr(g2), ctypes.byref(nb)), "mean_ei_grad")
        return o1, o2, g1, g2, nb.value
    check(lib.hbegp_predict_confidence_bound_grad(model.single_handle(), ctypes.byref(yn._raw), m, _ptr(xs), float(param),
                                                  _ptr(o1), _ptr(g1), ctypes.byref(nb)), "cb_grad")
    return o1, None, g1, None, nb.value


def _bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and (a.view(np.uint8) == b.view(np.uint8)).all()


# (n, nu, noise): one tile, several tiles (one train-tile group), a padded size >= 2048 (split over grid.y)
TRUTH_CASES = [(50, 0.5, 1e-2), (50, 2.5, 1e-5), (700, 1.5, 1e-4), (700, 0.5, 1e-5), (2049, 2.5, 1e-4), (2049, 1.5, 1e-2)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,nu,noise", TRUTH_CASES)
def test_f64_gradients_against_the_truth(n, nu, noise):
    """Both paths (m = 64 latency, m = 130 throughput) at candidates on, next to and away from training points."""
    A = np.float64
    d = 3
    x, y = synth(n, d, seed=n + 7)
    theta = _rounded(random_thetas(1, d, seed=n, noise=(noise, noise * 1.01))[0], A)
    xs = _candidates(x, 130, n + 1)
    assert _predict_path(64, d, _np(n), 8) == "latency" and _predict_path(130, d, _np(n), 8) != "latency"
    rec, fails = {}, []
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        k = _gpu_k(ctx, theta, nu)
        model = ctx.model(theta, nu=nu)
        outs = {m: _grad(model, xs[:m]) for m in (64, 130)}
        model.close()
    tr = Truth(k, y, theta, x, nu)
    lap = _reference(theta, x, y, nu=nu, k=k)
    tm, tv, s_m, s_v = _grad_star(tr, theta, x, xs, nu)
    lm, lv = _grad_numpy(lap.w, lap.alpha, theta, x, xs, nu)
    slack = SLACK[("w", _family(noise))]
    for m, (mean, var, dm, dv) in outs.items():
        sl = slice(0, m)
        for key, got, want, yard, scale, sk in (("dmean", dm, tm, lm, s_m, 1.0), ("dvar", dv, tv, lv, s_v, slack)):
            live = var > 0 if key == "dvar" else np.ones(m, bool)
            if key == "dvar":
                assert (dv[~live] == 0).all()
            e_gpu = np.abs(got[live] - want[sl][live])
            e_lap = np.abs(yard[sl][live] - want[sl][live])
            bound = R * e_lap.max() + F * EPS * scale[sl][live]
            ratio = float((e_gpu / bound).max()) if e_gpu.size else 0.0
            rec[f"m={m} {key}"] = {"gpu": float(e_gpu.max()) if e_gpu.size else 0.0, "lapack": float(e_lap.max()) if e_lap.size else 0.0,
                                   "err/bound": ratio}
            if ratio > sk:
                fails.append((m, key, ratio, int(np.argmax((e_gpu / bound).max(axis=1)))))
    _record(f"f64 n={n} nu={nu} noise={noise:g}", rec)
    assert not fails, (fails, rec)


RATIO = 4.0


@pytest.mark.gpu
@pytest.mark.parametrize("nu", [0.5, 2.5])
@pytest.mark.parametrize("n", [300, 1500])
def test_f32_gradients_against_the_f64_truth(n, nu):
    """f32 within RATIO x the error of a NumPy float32 restatement (LAPACK f32 factor), both against the f64 value of the
    same rounded inputs, on both paths."""
    from scipy.linalg import cho_factor, lapack
    A = np.float32
    d = 3
    x, y = synth(n, d, seed=n + 11, A=A)
    theta = _rounded(random_thetas(1, d, seed=n + 2, noise=(1e-2, 1.01e-2))[0], A)
    xs = np.random.default_rng(n).random((130, d)).astype(A)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta, nu=nu)
        outs = {m: _grad(model, xs[:m]) for m in (40, 130)}
        model.close()
    ref = _reference(theta, x, y, nu=nu)
    tm, tv = _grad_numpy(ref.w, ref.alpha, theta, x, xs, nu)
    noise, c, ls = math.exp(theta[0]), math.exp(theta[1]), np.exp(theta[2:])
    k32 = (_kernel_f64(x, x, c, ls, nu) + noise * np.eye(n)).astype(A)
    low = np.tril(cho_factor(k32, lower=True)[0])
    w32 = np.tril(lapack.strtri(low, lower=1)[0])
    a32 = (w32.T @ (w32 @ y.astype(A))).astype(A)
    nm, nv = _grad_numpy(w32, a32, theta, x.astype(np.float64), xs.astype(np.float64), nu, dtype=A)
    rec = {}
    for m, (mean, var, dm, dv) in outs.items():
        sl = slice(0, m)
        for key, got, want, yard in (("dmean", dm, tm, nm), ("dvar", dv, tv, nv)):
            e_gpu = float(np.abs(got.astype(np.float64) - want[sl]).max())
            e_np = float(np.abs(yard[sl].astype(np.float64) - want[sl]).max())
            rec[f"m={m} {key}"] = {"gpu": e_gpu, "numpy f32": e_np, "ratio": e_gpu / e_np}
            assert e_gpu <= RATIO * e_np, (m, key, rec)
    _record(f"f32 n={n} nu={nu}", rec)


@pytest.mark.gpu
def test_defined_points_exactly():
    """nu = 1/2 on a training point: the term contributes 0 (the gradient equals the sum without that point's term);
    clamped variance (c = 1e14): dvar = 0 there; EI's std-zero branch: -dmean or 0 bit for bit; NaN rows: dEI all NaN."""
    from hbetune_rs_b200.estimator import YNormalize
    A = np.float64
    n, d = 120, 2
    x, y = synth(n, d)
    # nu = 1/2, candidate = training point 5: the host sum without j = 5 equals the device result to rounding, and
    # the j = 5 term itself is exactly 0 (dk_factor(0) = 0); checked against the f64 formula with that term dropped
    theta = _rounded(np.array([math.log(1e-2), math.log(1.3), math.log(0.4), math.log(0.7)]), A)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta, nu=0.5)
        mean, var, dm, dv = _grad(model, x[5:6])
        ref = _reference(theta, x, y, nu=0.5)
        g = _grad_kstar(x[5:6], x, math.exp(theta[1]), np.exp(theta[2:]), 0.5)
        assert all(gk[0, 5] == 0.0 for gk in g)
        want = np.array([[gk[0] @ ref.alpha for gk in g]])
        assert np.isfinite(dm).all() and np.isfinite(dv).all()
        np.testing.assert_allclose(dm, want, rtol=1e-9, atol=1e-9 * float(np.abs(ref.alpha).sum()))
        model.close()
        # clamped variances and the std-zero branch
        theta = np.array([math.log(1e-2), math.log(1e14), math.log(2.0), math.log(2.0)])
        xs = np.concatenate([x[:60], np.random.default_rng(1).random((40, d))])
        yl, yn = YNormalize.new_project_into_normalized(y + 5.0, 0)
        model = ctx.model(theta)
        mean, var, dm, dv = _grad(model, xs)
        zero = var == 0
        assert zero.any() and (dv[zero] == 0).all()
        fmin = float(yn.project_location_from_normalized(np.array([float(np.median(mean))]))[0])
        fmin_n = float(yn.project_into_normalized(np.array([fmin]))[0])
        _, ei, _, dei, _ = _acq_grad(model, yn, xs, 0, fmin)
        sd0 = np.sqrt(var) <= STD_ZERO
        below = sd0 & (mean < fmin_n)
        assert below.any() and (sd0 & ~below).any()
        assert _bits(dei[below], -dm[below]) and (dei[sd0 & ~below] == 0).all()
        _, _, dcb, _, _ = _acq_grad(model, yn, xs, 1, -1.5)
        np.testing.assert_array_equal(dcb[zero], (A(yn.amplitude) * dm)[zero])
        # NaN rows
        xn = xs[:8].copy()
        xn[3, 1] = np.nan
        _, ei, _, dei, _ = _acq_grad(model, yn, xn, 0, fmin)
        assert np.isnan(ei[3]) and np.isnan(dei[3]).all() and np.isfinite(dei[[0, 1, 2, 4, 5, 6, 7]]).all()
        model.close()


def _model_case(A, n, d, proj=0, nu=2.5):
    from hbetune_rs_b200.estimator import YNormalize
    x, yraw = synth(n, d, seed=n + 1, A=A)
    yraw = (yraw * A(3) + A(10)).astype(A)
    yl, yn = YNormalize.new_project_into_normalized(yraw, proj, A=A)
    theta = _rounded(random_thetas(1, d, seed=n, noise=(1e-2, 1.01e-2))[0], A)
    return x, yraw, yl, yn, theta


@pytest.mark.gpu
@pytest.mark.parametrize("A", [np.float64, np.float32])
@pytest.mark.parametrize("proj", [0, 1])
def test_epilogue_is_the_chain_rule_of_predict_grad(proj, A):
    """hbegp_predict_mean_ei_grad / _confidence_bound_grad against _chain on hbegp_predict_grad's own (mu, var, dmu,
    dvar), both paths; values bit for bit those of hbegp_predict_mean_ei / _confidence_bound.  F_CHAIN: the device
    evaluates each component with a handful of roundings (division, erfc and exp to 2 ulps each, the products; dsd in
    T, EI's combination in f64, then rounded to T), so F_CHAIN eps_T of the condition sum |lf dmu| + |cb lf dsd|
    (|dmu| + |dsd| + |dEI| for EI, with Phi, phi <= 1)."""
    n, d = 1100, 3
    x, yraw, yl, yn, theta = _model_case(A, n, d, proj)
    eps = float(np.finfo(A).eps) / 2
    F_CHAIN = 16.0
    fmin = float(yraw.min())
    cb = -1.5
    with _ctx(A) as ctx:
        ctx.set_data(x, yl)
        model = ctx.model(theta)
        xs = _candidates(x.astype(np.float64), 200, 9).astype(A)
        for m in (17, 200):
            mean, var, dm, dv = _grad(model, xs[:m])
            fmin_n = float(yn.project_into_normalized(np.array([fmin]))[0])
            o1, ei, g1, gei, _ = _acq_grad(model, yn, xs[:m], 0, fmin)
            r1, rei, _, _ = _acq(model, yn, xs[:m], 0, fmin)
            assert _bits(o1, r1) and _bits(ei, rei)
            c1, _, gc, _, _ = _acq_grad(model, yn, xs[:m], 1, cb)
            rc, _, _, _ = _acq(model, yn, xs[:m], 1, cb)
            assert _bits(c1, rc)
            for r in range(m):
                mu, v = float(mean[r]), float(var[r])
                dmu, dvr = dm[r].astype(np.float64), dv[r].astype(np.float64)
                wl, wei = _chain(mu, v, dmu, dvr, 0, proj, float(yn.amplitude), fmin_n)
                wc, _ = _chain(mu, v, dmu, dvr, 1, proj, float(yn.amplitude), cb=cb)
                sd = math.sqrt(v)
                dsd = np.abs(dvr) / (2 * sd) if sd > 0 else 0 * dvr
                y = mu + sd * cb
                lf0 = abs(yn.amplitude) * (1 if proj == 0 else math.exp(mu * float(yn.amplitude)))
                lf1 = abs(yn.amplitude) * (1 if proj == 0 else math.exp(y * float(yn.amplitude)))
                tol_l = F_CHAIN * eps * lf0 * np.abs(dmu) * (1 + abs(mu * float(yn.amplitude)) * proj)
                tol_c = F_CHAIN * eps * lf1 * (np.abs(dmu) + abs(cb) * dsd) * (1 + abs(y * float(yn.amplitude)) * proj)
                tol_e = F_CHAIN * eps * (np.abs(dmu) + dsd + np.abs(wei))
                assert (np.abs(g1[r] - wl) <= tol_l).all(), (m, r, g1[r], wl)
                assert (np.abs(gc[r] - wc) <= tol_c).all(), (m, r, gc[r], wc)
                assert (np.abs(gei[r] - wei) <= tol_e).all(), (m, r, gei[r], wei)
        model.close()


@pytest.mark.gpu
@pytest.mark.parametrize("A", [np.float64, np.float32])
def test_gradients_do_not_depend_on_the_other_rows(A):
    """m > 64: the same bits whether rows come together or in pieces (m = 65, 128, 129, 1000, and 1000 as 129 + 871);
    the m <= 64 path agrees with the throughput path to rounding."""
    n, d = 2100, 4
    x, yraw, yl, yn, theta = _model_case(A, n, d)
    xs = np.random.default_rng(5).random((1000, d)).astype(A)
    with _ctx(A) as ctx:
        ctx.set_data(x, yl)
        model = ctx.model(theta)
        _, _, dm_all, dv_all = _grad(model, xs)
        for m in (65, 128, 129):
            _, _, dm, dv = _grad(model, xs[:m])
            assert _bits(dm, dm_all[:m]) and _bits(dv, dv_all[:m]), m
        _, _, dm, dv = _grad(model, xs[129:])
        assert _bits(dm, dm_all[129:]) and _bits(dv, dv_all[129:])
        _, _, dm, dv = _grad(model, xs[:64])
        tol = 1e-10 if A == np.float64 else 2e-3
        for got, want in ((dm, dm_all[:64]), (dv, dv_all[:64])):
            scale = max(1.0, float(np.abs(want).max()))
            assert float(np.abs(got - want).max()) <= tol * scale
        model.close()


@pytest.mark.gpu
@pytest.mark.parametrize("nu", [0.5, 1.5, 2.5])
def test_central_differences_of_the_library(nu):
    """Central differences (h = 1e-6 relative) of hbegp_predict_mean_ei in f64 against dmean_out / dei, away from
    training points, on both paths; a wrong sign or l instead of l^2 is off by O(1)."""
    A = np.float64
    n, d = 400, 3
    x, yraw, yl, yn, theta = _model_case(A, n, d, nu=nu)
    xs = 0.2 + 0.6 * np.random.default_rng(2).random((80, d))
    fmin = float(np.median(yraw))
    with _ctx(A) as ctx:
        ctx.set_data(x, yl)
        model = ctx.model(theta, nu=nu)
        for m in (5, 80):
            _, _, gm, gei, _ = _acq_grad(model, yn, xs[:m], 0, fmin)
            for q in range(d):
                h = 1e-6
                xp, xm = xs[:m].copy(), xs[:m].copy()
                xp[:, q] += h
                xm[:, q] -= h
                mp_, ep, _, _ = _acq(model, yn, xp, 0, fmin)
                mm, em, _, _ = _acq(model, yn, xm, 0, fmin)
                fd_m, fd_e = (mp_ - mm) / (2 * h), (ep - em) / (2 * h)
                np.testing.assert_allclose(gm[:, q], fd_m, rtol=1e-4, atol=1e-6 * max(1.0, float(np.abs(fd_m).max())))
                np.testing.assert_allclose(gei[:, q], fd_e, rtol=1e-4, atol=1e-6 * max(1.0, float(np.abs(fd_e).max())))
        model.close()


@pytest.mark.gpu
def test_evicted_model_gives_the_same_gradients():
    """An evicted model (resident limit 1) rebuilds W and returns the same bits on both paths."""
    A = np.float64
    n, d = 900, 3
    x, yraw, yl, yn, theta = _model_case(A, n, d)
    xs = np.random.default_rng(4).random((150, d))
    with _ctx(A) as ctx:
        ctx.set_data(x, yl)
        m1 = ctx.model(theta)
        before = [_grad(m1, xs[:k]) for k in (10, 150)]
        ctx.set_resident_models(1)
        m2 = ctx.model(theta)
        assert ctx.model_stats()["rebuilds"] == 0
        after = [_grad(m1, xs[:k]) for k in (10, 150)]
        assert ctx.model_stats()["rebuilds"] == 1
        for b, a in zip(before, after):
            for u, v in zip(b, a):
                assert _bits(u, v)
        m2.close()
        m1.close()


@pytest.mark.gpu
def test_lockstep_ei_search_with_fit_runs_with():
    """hbegp_fit_runs_with maximising EI from 8 starts (n = 500, d = 4, bounds [0, 1]^d, maxeval 30): one
    hbegp_predict_mean_ei_grad call per round for all live runs, every run ends at EI >= its start and one strictly
    above, and a second run gives bit-identical records."""
    from hbetune_rs_b200 import _lib
    A = np.float64
    n, d = 500, 4
    x, yraw, yl, yn, theta = _model_case(A, n, d)
    fmin = float(np.median(yraw))  # EI well above 0 at most starts
    starts = np.random.default_rng(8).random((8, d))
    lo, hi = np.exp(np.zeros(d)), np.exp(np.ones(d))  # fit_runs_with takes bounds in natural units of exp(x)
    with _ctx(A) as ctx:
        ctx.set_data(x, yl)
        model = ctx.model(theta)
        _, ei0, _, _, _ = _acq_grad(model, yn, starts, 0, fmin)

        def search():
            calls = []

            def cb(_user, B, p, th, out, grad, status):
                xs = np.array([[th[b * p + k] for k in range(p)] for b in range(B)])
                _, ei, _, dei, _ = _acq_grad(model, yn, xs, 0, fmin)
                calls.append(B)
                for b in range(B):
                    status[b] = 0
                    out[b] = float(ei[b])
                    for k in range(p):
                        grad[b * p + k] = float(dei[b, k])
                return 0

            fn = _lib.BATCH_OBJECTIVE_FN(cb)
            res = (_lib.RunResult * 8)()
            best = np.empty((8, d))
            rc = _lib.lib.hbegp_fit_runs_with(fn, None, d, 8, starts.ctypes.data, lo.ctypes.data, hi.ctypes.data, 30, 0, 1,
                                              _lib.ALLREDUCE_FN(), None, res, best.ctypes.data)
            assert rc == 0
            recs = [(r.best_lml, r.best_eval, r.n_evals, r.final_f, r.status) for r in res]
            return calls, recs, best

        calls, recs, best = search()
        calls2, recs2, best2 = search()
        model.close()
    assert calls[0] == 8 and sum(calls) == sum(r[2] for r in recs)
    for r, rec in enumerate(recs):
        assert rec[4] == 0 and rec[0] >= ei0[r]
    assert any(rec[0] > ei0[r] for r, rec in enumerate(recs))
    assert calls == calls2 and recs == recs2 and _bits(best, best2)


@pytest.mark.gpu
def test_bad_arguments_and_warnings():
    """Null pointers and m < 0 are HBEGP_ERR_INVALID; m = 0 is a no-op; the calls report the warnings of predict."""
    from hbetune_rs_b200._lib import lib
    from hbetune_rs_b200.estimator import YNormalize
    from hbetune_rs_b200.gpr import _ptr
    A = np.float64
    n, d = 120, 2
    x, y = synth(n, d)
    theta = np.array([math.log(1e-2), math.log(1e14), math.log(2.0), math.log(2.0)])
    xs = np.concatenate([x[:60], np.random.default_rng(1).random((40, d))])
    yl, yn = YNormalize.new_project_into_normalized(y + 5.0, 0)
    buf = np.zeros(4 * d)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta)
        hnd = model.single_handle()
        INVALID = -1
        assert lib.hbegp_predict_grad(hnd, -1, _ptr(buf), _ptr(buf), None, _ptr(buf), None, None) == INVALID
        assert lib.hbegp_predict_grad(hnd, 1, _ptr(buf), _ptr(buf), None, None, None, None) == INVALID
        assert lib.hbegp_predict_grad(hnd, 1, None, _ptr(buf), None, _ptr(buf), None, None) == INVALID
        assert lib.hbegp_predict_grad(None, 1, _ptr(buf), _ptr(buf), None, _ptr(buf), None, None) == INVALID
        assert lib.hbegp_predict_mean_ei_grad(hnd, None, 1, _ptr(buf), 0.0, None, None, None, None, None) == INVALID
        assert lib.hbegp_predict_confidence_bound_grad(hnd, ctypes.byref(yn._raw), -1, _ptr(buf), 0.0, None, None, None) == INVALID
        assert lib.hbegp_predict_grad(hnd, 0, None, None, None, None, None, None) == 0
        model.predict(xs, warn=False)
        count, (vals, rows) = model.n_below_warn, model.warn_values(cap=4096)
        assert count > 0
        _grad(model, xs)
        assert model.n_below_warn == count
        v2, r2 = model.warn_values(cap=4096)
        np.testing.assert_array_equal(v2, vals)
        np.testing.assert_array_equal(r2, rows)
        for mode, p in ((0, 5.0), (1, -1.5)):
            *_, nb = _acq_grad(model, yn, xs, mode, p)
            assert nb == count
            v2, r2 = model.warn_values(cap=4096)
            np.testing.assert_array_equal(v2, vals)
            np.testing.assert_array_equal(r2, rows)
        model.close()
