"""The squared exponential (RBF) kernel, selected by nu = +inf: K_ij = c exp(-0.5 s_ij) + noise delta_ij with
s_ij = sum_k (x_ik / l_k - x_jk / l_k)^2 (sklearn's ``RBF``; sklearn documents ``Matern(nu=np.inf)`` as the same kernel).

The oracle restates the reference, which has no RBF (matern_kernel.rs:79 is ``unimplemented!`` there); this module
restates sklearn's RBF arithmetic on top of the oracle's Matern (``RbfMatern``) and pins it to sklearn.  The Matern
truth helpers of test_f64_truth (``_derivs``, ``_kernel_f64``, ``_dmatern_r``) treat any nu other than 1/2 and 3/2 as
5/2, so nothing here passes nu = inf to them: the RBF versions are below.  GPU results are held to an mpmath truth, to
sklearn, to LAPACK's error on the GPU's own K (the rule of test_f64_truth) and to themselves bit for bit."""
import ctypes
import math

import numpy as np
import pytest

from oracle import gpr as ogpr
from tests.test_dispatch_sweep import _ctx, _note, _np, _predict_path, _rounded
from tests.test_f64_truth import (EPS, F_K, Truth, _acc_sum, _check_lml_grad, _gpu_k, _rule, _two_prod, _two_sum,
                                  dd_matmul)
from tests.util import random_thetas, synth

INF = math.inf


# ------------------------------------------------------------------------------------------------ the formulas


class RbfMatern(ogpr.Matern):
    """oracle.gpr.Matern at nu = inf, restating sklearn's RBF (sklearn/gaussian_process/kernels.py, class RBF):
    K = exp(-0.5 sqeuclidean(X / l)), dK/dln l_k = K (x_ik - x_jk)^2 / l_k^2."""

    def __init__(self, length_scale):
        super().__init__(INF, length_scale)

    def kernel(self, x1, x2, A=np.float64):
        ls = self._ls(A)
        a, b = np.asarray(x1, dtype=A) / ls[None, :], np.asarray(x2, dtype=A) / ls[None, :]
        s = np.zeros((a.shape[0], b.shape[0]), dtype=A)
        for k in range(a.shape[1]):
            s = s + (a[:, k, None] - b[None, :, k]) ** 2
        return np.exp(A(-0.5) * s)

    def theta_grad(self, x, A=np.float64):
        x = np.asarray(x, dtype=A)
        k = self.kernel(x, x, A)
        ls = self._ls(A)
        d = (x[:, None, :] - x[None, :, :]) ** 2 / (ls * ls)[None, None, :]
        return k, (d * k[:, :, None]).astype(A, copy=False)

    def with_theta(self, theta):
        return RbfMatern([b.with_value(math.exp(t)) for t, b in zip(theta, self.length_scale)])

    def with_clamped_theta(self, theta):
        return RbfMatern([b.with_clamped_value(math.exp(t)) for t, b in zip(theta, self.length_scale)])


def rbf_kernel(theta, lo=1e-9, hi=1e9):
    c, ls = math.exp(theta[1]), [math.exp(t) for t in theta[2:]]
    bv = ogpr.BoundedValue
    return ogpr.Product(ogpr.ConstantKernel(bv(c, min(lo, c), max(hi, c))),
                        RbfMatern([bv(v, min(lo, v), max(hi, v)) for v in ls]))


def rbf_lml(theta, x, y):
    return ogpr.lml_with_gradient(rbf_kernel(theta), math.exp(theta[0]), x, y)


def _sq(x1, x2, ls):
    """s = sum_k (x1 / l - x2 / l)^2, features left to right (division first)."""
    a, b = np.asarray(x1, np.float64) / ls, np.asarray(x2, np.float64) / ls
    s = np.zeros((a.shape[0], b.shape[0]))
    for k in range(a.shape[1]):
        s += (a[:, k, None] - b[None, :, k]) ** 2
    return s


def _rbf_f64(x1, x2, c, ls):
    return c * np.exp(-0.5 * _sq(x1, x2, ls))


def _rbf_derivs(theta, x):
    """dK/dtheta in f64 for Truth.grad: noise (scalar), c M, c M (x_i - x_j)^2 / l_k^2."""
    x = np.asarray(x, dtype=np.float64)
    noise, c, ls = math.exp(theta[0]), math.exp(theta[1]), np.exp(np.asarray(theta[2:], dtype=np.float64))
    kc = _rbf_f64(x, x, c, ls)
    return [noise, kc] + [kc * ((x[:, j, None] - x[None, :, j]) / ls[j]) ** 2 for j in range(x.shape[1])]


class RbfTruth(Truth):
    """Truth (factor, K^-1, alpha, LML: nothing there depends on the kernel) with the RBF's dK/dtheta."""

    @property
    def grad(self):
        if self._grad is None:
            (ah, al), (kh, kl) = self.outer_alpha(), self.kinv
            gs, scale = [], []
            for j, g in enumerate(_rbf_derivs(self.theta, self.x)):
                if j == 0:
                    p1, e1 = _two_prod(np.diag(ah).copy(), np.full(self.n, g))
                    p2, e2 = _two_prod(-np.diag(kh).copy(), np.full(self.n, g))
                    parts = [p1, e1, p2, e2, np.diag(al) * g, -np.diag(kl) * g]
                    sc = np.abs(np.diag(ah) - np.diag(kh)).sum() * g
                else:
                    p1, e1 = _two_prod(ah, g)
                    p2, e2 = _two_prod(-kh, g)
                    parts = [p1, e1, p2, e2, al * g, -kl * g]
                    sc = float((np.abs(ah - kh) * np.abs(g)).sum())
                hi, lo = _acc_sum(np.concatenate([p.ravel() for p in parts]))
                gs.append((float(hi) / 2, float(lo) / 2))
                scale.append(sc / 2)
            self._grad = (np.array([h for h, _ in gs]), np.array([lo for _, lo in gs]), np.array(scale))
        return self._grad

    def grad_contract(self, m):
        return np.array([0.5 * (float(np.trace(m)) * g if j == 0 else float((m * np.abs(g)).sum()))
                         for j, g in enumerate(_rbf_derivs(self.theta, self.x))])


def _reference(theta, x, y, k):
    """LAPACK's LML, gradient, alpha, W and K^-1 on a given K, with the RBF's dK/dtheta (test_dispatch_sweep's
    _reference restated for the RBF)."""
    from types import SimpleNamespace

    from scipy.linalg import cho_factor, cho_solve, lapack
    n = len(y)
    low = np.tril(cho_factor(k, lower=True)[0])
    r = SimpleNamespace(k=k)
    r.alpha = cho_solve((low, True), y)
    r.w, info = lapack.dtrtri(low, lower=1)
    assert info == 0
    r.kinv = r.w.T @ r.w
    logdet = np.log(np.diag(low))
    r.lml = -0.5 * float(y @ r.alpha) - float(logdet.sum()) - n / 2.0 * math.log(2.0 * math.pi)
    r.lml_scale = 0.5 * abs(float(y @ r.alpha)) + float(np.abs(logdet).sum()) + n / 2.0 * math.log(2.0 * math.pi)
    tmp = np.outer(r.alpha, r.alpha) - r.kinv
    g = _rbf_derivs(theta, x)
    r.grad = np.array([0.5 * g[0] * float(np.trace(tmp))] + [0.5 * float((tmp * gk).sum()) for gk in g[1:]])
    return r


def _dk_kstar(xs, x, c, ls, dtype=np.float64):
    """G[k][r, j] = d k*_rj / d xs_rk = -c M(s_rj) (x~_rk - X~_jk) / l_k, in `dtype`."""
    xs, x, ls = (np.asarray(a, dtype=dtype) for a in (xs, x, ls))
    a, b = xs / ls, x / ls
    diffs = [a[:, k, None] - b[None, :, k] for k in range(a.shape[1])]
    s = sum(df * df for df in diffs)
    m = np.exp(dtype(-0.5) * s)
    return [-dtype(c) * m * df / ls[k] for k, df in enumerate(diffs)]


def _bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


# ------------------------------------------------------------------------------------------------ CPU: the oracle

skl = pytest.importorskip("sklearn.gaussian_process")
from sklearn.gaussian_process.kernels import RBF, ConstantKernel, Matern, WhiteKernel  # noqa: E402


def _golden_inputs():
    """The inputs of the reference's kernel goldens (matern_kernel.rs:189-253, product_kernel.rs:120-169)."""
    import json
    import os
    path = os.path.join(os.path.dirname(__file__), "golden", "reference_kernel_goldens.json")
    with open(path) as f:
        data = json.load(f)
    out = []

    def walk(v):
        if isinstance(v, dict):
            for key, val in v.items():
                if key in ("x", "x1", "x_train", "xs") and isinstance(val, list) and val and isinstance(val[0], list):
                    out.append(np.asarray(val, dtype=np.float64))
                else:
                    walk(val)
        elif isinstance(v, list):
            for val in v:
                walk(val)
    walk(data)
    return out


def _kernel_cases():
    cases = [(x, np.full(x.shape[1], 1.0), 1.0) for x in _golden_inputs()]
    rng = np.random.default_rng(7)
    for n, d in ((1, 1), (5, 1), (30, 3), (50, 8)):
        cases.append((rng.random((n, d)) * 3 - 1, rng.uniform(0.2, 2.0, d), rng.uniform(0.5, 3.0)))
    return cases


def test_golden_inputs_are_found():
    assert len(_golden_inputs()) >= 2


@pytest.mark.parametrize("case", range(6))
def test_oracle_kernel_and_theta_grad_match_sklearn(case):
    cases = _kernel_cases()
    if case >= len(cases):
        pytest.skip("fewer cases")
    for x, ls, c in cases[case::6]:
        ours = ogpr.Product(ogpr.ConstantKernel(ogpr.BoundedValue(c, 1e-9, 1e9)),
                            RbfMatern([ogpr.BoundedValue(v, 1e-9, 1e9) for v in ls]))
        k, g = ours.theta_grad(x)
        for sk in (ConstantKernel(c) * RBF(length_scale=ls), ConstantKernel(c) * Matern(length_scale=ls, nu=np.inf)):
            ks, gs = sk(x, eval_gradient=True)  # sklearn: [ln c, ln l_1 ..] -- our order too
            np.testing.assert_allclose(k, ks, rtol=1e-14, atol=1e-15)
            np.testing.assert_allclose(g, gs, rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(ours.kernel(x, x[::-1]), ConstantKernel(c)(x, x[::-1]) * RBF(ls)(x, x[::-1]),
                                   rtol=1e-14, atol=1e-15)


CASES = [(25, 1), (60, 3), (130, 5), (200, 8)]


def _theta(d, seed):
    rng = np.random.default_rng(seed)
    return np.concatenate([[math.log(rng.uniform(0.02, 0.5)), math.log(rng.uniform(0.5, 3.0))],
                           np.log(rng.uniform(0.3, 2.5, d) * math.sqrt(d))])


def _sklearn(theta, x, y):
    k = ConstantKernel(math.exp(theta[1])) * RBF(length_scale=np.exp(theta[2:])) + WhiteKernel(math.exp(theta[0]))
    gp = skl.GaussianProcessRegressor(kernel=k, optimizer=None, alpha=0.0).fit(x, y)
    lml, g = gp.log_marginal_likelihood(np.concatenate([theta[1:], theta[:1]]), eval_gradient=True)
    return gp, lml, np.concatenate([g[-1:], g[:-1]])


@pytest.mark.parametrize("n,d", CASES)
def test_oracle_lml_gradient_and_prediction_match_sklearn(n, d):
    x, y = synth(n, d, seed=n + d)
    theta = _theta(d, n)
    gp, lml, grad = _sklearn(theta, x, y)
    res = rbf_lml(theta, x, y)
    assert res.lml == pytest.approx(lml, rel=1e-11, abs=1e-11)
    np.testing.assert_allclose(res.lml_gradient, grad, rtol=1e-8, atol=1e-9 * np.abs(grad).max())
    xs = np.random.default_rng(1).random((40, d))
    mean, std = gp.predict(xs, return_std=True)
    var = np.empty(len(xs))
    omean = ogpr.predict(rbf_kernel(theta), res.alpha, xs, x, res.factorization.invc(), var)
    np.testing.assert_allclose(omean, mean, rtol=0, atol=1e-10 * max(1.0, np.abs(mean).max()))
    np.testing.assert_allclose(var, np.maximum(std ** 2 - math.exp(theta[0]) + 1e-5, 0.0), rtol=0, atol=1e-9)


def test_correlation_and_derivative_against_mpmath():
    """M(s) = exp(-s / 2) and dk_factor = -2 dM/ds = M, at s from 0 to where M underflows."""
    import mpmath
    s = np.concatenate([[0.0, 1e-300, 1e-8], np.geomspace(1e-3, 1400.0, 200)])
    m = np.exp(-0.5 * s)
    with mpmath.workdps(40):
        for si, mi in zip(s, m):
            want = mpmath.exp(-mpmath.mpf(float(si)) / 2)
            dwant = -2 * mpmath.diff(lambda t: mpmath.exp(-t / 2), mpmath.mpf(float(si)))
            assert abs(mpmath.mpf(float(mi)) - want) <= 2 * EPS * want + mpmath.mpf(2) ** -1074
            assert abs(dwant - want) <= mpmath.mpf(10) ** -30 * want


# ------------------------------------------------------------------------------------------------ GPU


def _problem(n, d, noise, ls_scale, seed, A=np.float64):
    x, y = synth(n, d, seed=seed)
    th = random_thetas(1, d, seed=seed + 1, noise=(noise, noise * 1.01), ls=(0.3 * ls_scale, ls_scale))[0]
    return x, y, _rounded(th, A)


def _kappa(k):
    return float(np.linalg.cond(k))


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 3, 16, 64, 65, 200])
def test_assembled_k_against_mpmath(d):
    """debug_factor's K against c exp(-s / 2) + noise in mpmath, s the host's f64 squared distance (division first,
    features left to right): within F_K eps (c + noise), and elementwise within F_K eps (|K| + (d - 1) c s e^{-s/2}):
    the GPU fuses the d - 1 additions of s with the squares (s moves by up to (d - 1) eps s, K by c M s / 2 times that).
    At d = 1 both round the one square the same way, and with l = 0.04 the exp arguments reach a few hundred, where an
    inexact exp, or s formed as sqrt(s)^2, shows."""
    import mpmath
    n = 200
    x, y = synth(n, d, seed=d)
    theta = _rounded(random_thetas(1, d, seed=d + 1, noise=(1e-4, 1e-2), ls=(0.3 * math.sqrt(d), 3 * math.sqrt(d)))[0],
                     np.float64)
    if d == 1:
        theta[2] = math.log(0.04)
    noise, c, ls = math.exp(theta[0]), math.exp(theta[1]), np.exp(theta[2:])
    with _ctx(np.float64) as ctx:
        ctx.set_data(x, y)
        out = ctx.debug_factor(theta, nu=INF, want=("k",))
    s = _sq(x, x, ls)
    rows = range(0, n, 7)
    with mpmath.workdps(30):
        err, bound = [], []
        for i in rows:
            for j in range(i + 1):
                kij = mpmath.mpf(c) * mpmath.exp(-mpmath.mpf(float(s[i, j])) / 2) + (noise if i == j else 0)
                err.append(float(abs(mpmath.mpf(float(out["k"][i, j])) - kij)))
                bound.append(F_K * EPS * (float(abs(kij)) + (d - 1) * c * s[i, j] * math.exp(-0.5 * s[i, j])))
    err, bound = np.array(err), np.array(bound)
    ulps = float(err.max() / (EPS * (c + noise)))
    _note(f"rbf K d={d}", {"max err / eps (c + noise)": ulps, "max err / elementwise bound": float((err / bound).max())})
    assert ulps <= F_K
    assert (err <= bound).all(), float((err / bound).max())
    # the diagonal is c + noise exactly as for Matern (s = 0, M = 1)
    assert (np.diag(out["k"]) == np.float64(c) + np.float64(noise)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("A", [np.float64, np.float32])
def test_kernel_matrix_and_theta_grad_against_sklearn(A):
    import hbetune_rs_b200 as h
    rng = np.random.default_rng(3)
    x1, x2 = rng.random((70, 4)).astype(A), rng.random((90, 4)).astype(A)
    c, ls = 1.7, np.array([0.3, 0.8, 1.5, 2.5])
    theta = [math.log(c)] + list(np.log(ls))
    kern = h.Product(h.ConstantKernel(h.BoundedValue(c, 1e-3, 1e3)), h.Matern(INF, [h.BoundedValue(v, 1e-3, 1e3) for v in ls]))
    sk = ConstantKernel(c) * RBF(length_scale=ls)
    tol = 1e-14 if A == np.float64 else 2e-6
    with _ctx(A) as ctx:
        k12 = kern.kernel(ctx, x1, x2)
        k, g = kern.theta_grad(ctx, x1)
    np.testing.assert_allclose(k12, sk(x1.astype(np.float64), x2.astype(np.float64)), rtol=tol, atol=tol)
    ks, gs = sk(x1.astype(np.float64), eval_gradient=True)
    np.testing.assert_allclose(k, ks, rtol=tol, atol=tol)
    np.testing.assert_allclose(g, gs, rtol=10 * tol, atol=10 * tol * c)
    assert len(theta) == g.shape[2]


# (n, d, B, noise, length-scale scale): the dispatch-sweep sizes; RBF matrices are far worse conditioned than Matern
# ones, so the length scales are short enough (and the noise large enough) for LAPACK to factorise -- kappa is recorded.
LML_CASES = [(129, 3, 5, 1e-2, 0.5), (511, 4, 3, 1e-2, 0.6), (700, 3, 5, 1e-2, 0.4), (960, 3, 33, 1e-2, 0.4),
             (1025, 3, 3, 1e-2, 0.3), (2049, 2, 9, 1e-2, 0.15), (2049, 2, 20, 3e-2, 0.15)]


def _lml_thetas(B, d, noise, ls_scale, seed, A):
    th = random_thetas(B, d, seed=seed, noise=(noise, 3 * noise), ls=(0.4 * ls_scale, ls_scale))
    return np.stack([_rounded(t, A) for t in th])


@pytest.mark.gpu
@pytest.mark.parametrize("n,d,B,noise,ls_scale", LML_CASES)
def test_lml_and_gradient(n, d, B, noise, ls_scale):
    """f64: the first, middle and last member by the rule of test_f64_truth (R x LAPACK + F eps S on the GPU's own K)
    and against sklearn at 1e-9; every member equals its B = 1 result bit for bit.  f32 within 2 x LAPACK f32's error."""
    x, y = synth(n, d)
    th = _lml_thetas(B, d, noise, ls_scale, B + n, np.float64)
    with _ctx(np.float64) as ctx:
        ctx.set_data(x, y)
        lml, grad, status = ctx.lml_grad_batch(th, INF)
        singles = [ctx.lml_grad_batch(th[b:b + 1], INF) for b in range(B)]
        check = sorted({0, B // 2, B - 1})
        ks = {b: _gpu_k(ctx, th[b], nu=INF) for b in check}
        ws = {b: ctx.debug_factor(th[b], nu=INF, want=("w",))["w"] for b in check}
    assert (status == 0).all()
    for b in range(B):
        assert _bits(lml[b], singles[b][0][0]) and _bits(grad[b], singles[b][1][0]), b
    rec, fails = {}, []
    for b in check:
        k = ks[b]
        tr = RbfTruth(k, y, th[b], x)
        lap = _reference(th[b], x, y, k)
        nz = math.exp(th[b, 0])
        _check_lml_grad(rec, fails, f"b={b}", lml[b], grad[b], tr, lap, _np(n), ws[b], nz)
        rec[f"b={b} kappa"] = _kappa(k)
        _, sk_lml, sk_grad = _sklearn(th[b], x, y)
        assert lml[b] == pytest.approx(sk_lml, rel=1e-9, abs=1e-9)
        np.testing.assert_allclose(grad[b], sk_grad, rtol=1e-7, atol=1e-9 * np.abs(sk_grad).max())
    # f32: against the f64 LAPACK reference, within twice LAPACK f32's own error (both on the f32-rounded problem)
    th32 = _lml_thetas(B, d, max(noise, 0.1), ls_scale, B + n, np.float32)
    x32, y32 = x.astype(np.float32), y.astype(np.float32)
    with _ctx(np.float32) as ctx:
        ctx.set_data(x32, y32)
        lml32, grad32, st32 = ctx.lml_grad_batch(th32, INF)
    assert (st32 == 0).all()
    for b in check:
        ref = rbf_lml(th32[b], x32.astype(np.float64), y32.astype(np.float64))
        lap32 = ogpr.lml_with_gradient(rbf_kernel(th32[b]), np.float32(math.exp(th32[b, 0])), x32, y32, np.float32)
        e_l = abs(float(lap32.lml) - ref.lml)
        e_g = np.abs(np.asarray(lap32.lml_gradient, np.float64) - ref.lml_gradient)
        floor = 64 * 2.0 ** -24
        assert abs(float(lml32[b]) - ref.lml) <= 2 * e_l + floor * abs(ref.lml), (b, lml32[b], ref.lml, e_l)
        gs = np.abs(ref.lml_gradient).max()
        assert (np.abs(grad32[b] - ref.lml_gradient) <= 2 * e_g + floor * gs).all(), (b, grad32[b], ref.lml_gradient)
    _note(f"rbf lml n={n} d={d} B={B}", rec)
    assert not fails, fails


@pytest.mark.gpu
def test_not_positive_definite_member_keeps_its_neighbours_bits():
    """Near-duplicate rows at noise 1e-20 and long length scales: HBEGP_NOT_PD, lml = -inf, a zero gradient; the other members' bits are
    those of their B = 1 evaluations."""
    n, d = 300, 2
    x, y = synth(n, d, seed=4)
    x[150:200] = x[:50] + 1e-9
    th = _lml_thetas(3, d, 1e-2, 0.3, 5, np.float64)
    th[1, 0] = math.log(1e-20)
    th[1, 2:] = math.log(3.0)
    with _ctx(np.float64) as ctx:
        ctx.set_data(x, y)
        lml, grad, status = ctx.lml_grad_batch(th, INF)
        singles = [ctx.lml_grad_batch(th[b:b + 1], INF) for b in (0, 2)]
    assert status[1] == 1 and lml[1] == -np.inf and (grad[1] == 0).all(), (status, lml)
    for b, s in zip((0, 2), singles):
        assert status[b] == 0 and _bits(lml[b], s[0][0]) and _bits(grad[b], s[1][0])


@pytest.mark.gpu
def test_fit_reaches_the_optimum_sklearn_finds():
    import hbetune_rs_b200 as h
    n, d = 80, 2
    x, y = synth(n, d, seed=21)
    bv = h.BoundedValue
    kernel = h.Product(h.ConstantKernel(bv(1.0, 1e-2, 1e2)), h.Matern(INF, [bv(1.0, 1e-2, 1e2)] * d))
    with h.Context() as ctx:
        fk = h.FittedKernel.new(ctx, kernel, x, y, h.RNG.new_with_seed(5), 10, bv(1.0, 1e-3, 1e1))
    k = (ConstantKernel(1.0, (1e-2, 1e2)) * RBF(length_scale=[1.0] * d, length_scale_bounds=(1e-2, 1e2))
         + WhiteKernel(1.0, (1e-3, 1e1)))
    gp = skl.GaussianProcessRegressor(kernel=k, alpha=0.0, n_restarts_optimizer=10, random_state=0).fit(x, y)
    sk_lml = gp.log_marginal_likelihood_value_
    assert fk.kernel.k2.nu == INF
    assert fk.lml >= sk_lml - 1e-5 * abs(sk_lml)
    assert fk.lml <= sk_lml + 1e-3 * abs(sk_lml) + 1e-3
    ours = np.array([math.log(fk.kernel.k1.constant.value)] + [math.log(v.value) for v in fk.kernel.k2.length_scale]
                    + [math.log(fk.noise.value)])
    np.testing.assert_allclose(ours, gp.kernel_.theta, atol=5e-3)


def _predict_star(tr, theta, x, xs):
    """mean* = k* alpha* and var* = c + 1e-5 - |W* k*|^2 (clamped), with their condition sums."""
    c = math.exp(theta[1])
    ks = _rbf_f64(xs, x, c, np.exp(theta[2:]))
    mh, ml = dd_matmul(ks, tuple(t[:, None] for t in tr.alpha))
    uh, ul = dd_matmul(tuple(tr.ws), ks.T)
    p, e = _two_prod(uh, uh)
    sh, sl = _acc_sum(np.concatenate([p, e, 2 * uh * ul]))
    th, tl = _two_sum(c, 1e-5)
    var = np.maximum((th - sh) + (tl - sl), 0.0)
    s_mean = np.abs(ks) @ np.abs(tr.alpha[0])
    s_var = c + 1e-5 + 2 * (np.abs(uh) * (np.abs(tr.ws[0]) @ np.abs(ks.T))).sum(axis=0)
    return (mh[:, 0], ml[:, 0]), var, s_mean, s_var, ks


def _check_predictions(rec, fails, tag, model, tr, lap, theta, x, xs, ms):
    (th, tl), tv, s_mean, s_var, ks = _predict_star(tr, theta, x, xs)
    lm = ks @ lap.alpha
    u = ks @ lap.w.T
    lv = np.maximum(math.exp(theta[1]) + 1e-5 - np.einsum("ij,ij->i", u, u), 0.0)
    for m in ms:
        mean, var = model.predict(xs[:m], warn=False)
        sl = slice(0, m)
        _rule(rec, fails, f"{tag} m={m} mean", np.abs((mean - th[sl]) - tl[sl]), np.abs((lm[sl] - th[sl]) - tl[sl]),
              s_mean[sl].max())
        _rule(rec, fails, f"{tag} m={m} var", np.abs(var - tv[sl]), np.abs(lv[sl] - tv[sl]), s_var[sl].max())


def _candidates(x, m, seed):
    rng = np.random.default_rng(seed)
    xs = rng.random((m, x.shape[1]))
    idx = rng.choice(x.shape[0], 20, replace=False)
    xs[:10] = x[idx[:10]]
    xs[10:20] = x[idx[10:]] + 1e-7 * rng.standard_normal((10, x.shape[1]))
    return xs


@pytest.mark.gpu
def test_model_paths():
    """create, extend (block append and full fallback), eviction and rebuild at nu = inf: predictions on both paths
    against the truth of the GPU's K; rows of the m > 64 path do not depend on the row count; the rebuilt model returns
    the bits it returned before its eviction (a rebuild at another nu would not)."""
    import hbetune_rs_b200 as h
    d = 3
    x, y = synth(1300, d, seed=13)
    theta = _rounded(random_thetas(1, d, seed=14, noise=(1e-3, 1.01e-3), ls=(0.2, 0.3))[0], np.float64)
    xs = _candidates(x, 300, 15)
    assert _predict_path(300, d, _np(1300), 8) == "split" and _predict_path(17, d, _np(1300), 8) == "latency"
    rec, fails = {}, []
    with _ctx(np.float64) as ctx:
        ctx.set_data(x[:1000], y[:1000])
        models = [ctx.model(theta, INF)]
        for n, appended in ((1100, True), (1300, True)):
            ctx.set_data(x[:n], y[:n])
            m = h.Model(ctx, prior=models[-1], want_kinv=True)
            assert bool(m.appended) == appended, n
            models.append(m)
            k = _gpu_k(ctx, theta, nu=INF)
            tr = RbfTruth(k, y[:n], theta, x[:n])
            lap = _reference(theta, x[:n], y[:n], k)
            _check_predictions(rec, fails, f"1000->{n}", m, tr, lap, theta, x[:n], xs, (17, 300))
            rec[f"1000->{n} kappa"] = _kappa(k)
        # the full fallback: rows in another order
        perm = np.random.default_rng(1).permutation(1300)
        ctx.set_data(x[perm], y[perm])
        full = h.Model(ctx, prior=models[-1])
        assert not full.appended
        k = _gpu_k(ctx, theta, nu=INF)
        tr = RbfTruth(k, y[perm], theta, x[perm])
        _check_predictions(rec, fails, "full", full, tr, _reference(theta, x[perm], y[perm], k), theta, x[perm], xs, (17, 300))
        # row-count independence of the m > 64 path
        mean_all, var_all = full.predict(xs, warn=False)
        mean_65, var_65 = full.predict(xs[:65], warn=False)
        assert _bits(mean_all[:65], mean_65) and _bits(var_all[:65], var_65)
        # eviction and rebuild
        before = [full.predict(xs[:k], warn=False) for k in (17, 300)] + [full.predict_grad(xs[:k]) for k in (17, 300)]
        ctx.set_resident_models(1)
        other = ctx.model(theta, INF)
        r0 = ctx.model_stats()["rebuilds"]
        after = [full.predict(xs[:k], warn=False) for k in (17, 300)] + [full.predict_grad(xs[:k]) for k in (17, 300)]
        assert ctx.model_stats()["rebuilds"] == r0 + 1
        for b, a in zip(before, after):
            for u, v in zip(b, a):
                assert _bits(u, v)
        for mdl in models + [full, other]:
            mdl.close()
    _note("rbf model paths noise=1e-3", rec)
    assert not fails, fails


@pytest.mark.gpu
@pytest.mark.parametrize("n", [50, 700])
def test_candidate_gradients(n):
    """f64 dmean and dvar on both paths against the truth's (R x LAPACK + F eps S); f32 against a float32
    restatement; central differences of the mean; a candidate on a training point (its term contributes 0, which is
    the true derivative of a smooth kernel)."""
    import mpmath
    d = 3
    x, y = synth(n, d, seed=n)
    theta = _rounded(random_thetas(1, d, seed=n + 2, noise=(1e-3, 1.01e-3), ls=(0.3, 0.5))[0], np.float64)
    c, ls = math.exp(theta[1]), np.exp(theta[2:])
    xs = 0.1 + 0.8 * np.random.default_rng(n).random((80, d))
    xs[3] = x[5]
    with _ctx(np.float64) as ctx:
        ctx.set_data(x, y)
        k = _gpu_k(ctx, theta, nu=INF)
        model = ctx.model(theta, INF)
        outs = {m: model.predict_grad(xs[:m]) for m in (5, 80)}
        model.close()
    tr = RbfTruth(k, y, theta, x)
    lap = _reference(theta, x, y, k)
    g = _dk_kstar(xs, x, c, ls)
    ks = _rbf_f64(xs, x, c, ls)
    # the truth: dmean* = G alpha*, dvar* = -2 G . (W*^T W* k*)
    dm_t = np.stack([gk @ tr.alpha[0] + gk @ sum(tr.alpha[1:]) for gk in g], axis=1)
    uh, ul = dd_matmul(tuple(tr.ws), ks.T)
    vh, vl = dd_matmul(tuple(t.T for t in tr.ws), (uh, ul))
    dv_t = np.stack([-2.0 * ((vh + vl).T * gk).sum(axis=1) for gk in g], axis=1)
    dm_l = np.stack([gk @ lap.alpha for gk in g], axis=1)
    vl_ = (ks @ lap.w.T) @ lap.w
    dv_l = np.stack([-2.0 * (vl_ * gk).sum(axis=1) for gk in g], axis=1)
    s_m = np.stack([np.abs(gk) @ np.abs(tr.alpha[0]) for gk in g], axis=1)
    w0 = np.abs(tr.ws[0])
    s_v = np.stack([2.0 * ((w0.T @ (w0 @ np.abs(ks.T))).T * np.abs(gk)).sum(axis=1) for gk in g], axis=1)
    rec, fails = {}, []
    for m, out in outs.items():
        mean, var, dmean, dvar = out
        _rule(rec, fails, f"m={m} dmean", np.abs(dmean - dm_t[:m]), np.abs(dm_l[:m] - dm_t[:m]), s_m[:m].max())
        _rule(rec, fails, f"m={m} dvar", np.abs(dvar - dv_t[:m]), np.abs(dv_l[:m] - dv_t[:m]), s_v[:m].max())
    # the truth's G against mpmath derivatives of k*
    with mpmath.workdps(30):
        for r, j in ((0, 1), (7, 20), (3, 5)):
            for q in range(d):
                def kr(t, r=r, j=j, q=q):
                    s = mpmath.fsum((((mpmath.mpf(float(xs[r, k])) + (t if k == q else 0)) / float(ls[k]))
                                     - mpmath.mpf(float(x[j, k])) / float(ls[k])) ** 2 for k in range(d))
                    return c * mpmath.exp(-s / 2)
                want = mpmath.diff(kr, 0)
                assert abs(float(want) - g[q][r, j]) <= 1e-13 * max(1.0, abs(float(want))), (r, j, q)
    # central differences of the library's own mean (away from training points)
    with _ctx(np.float64) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta, INF)
        for m in (5, 80):
            sel = [i for i in range(m) if i != 3]
            dmean = model.predict_grad(xs[:m])[2]
            for q in range(d):
                hh = 1e-6
                xp, xm = xs[:m].copy(), xs[:m].copy()
                xp[:, q] += hh
                xm[:, q] -= hh
                fd = (model.predict(xp, warn=False)[0] - model.predict(xm, warn=False)[0]) / (2 * hh)
                np.testing.assert_allclose(dmean[sel, q], fd[sel], rtol=1e-4, atol=1e-6 * max(1.0, np.abs(fd).max()))
        model.close()
    # f32 against a float32 restatement from LAPACK's factor
    x32, y32 = x.astype(np.float32), y.astype(np.float32)
    th32 = _rounded(theta, np.float32)
    with _ctx(np.float32) as ctx:
        ctx.set_data(x32, y32)
        model = ctx.model(th32, INF)
        got = {m: model.predict_grad(xs[:m].astype(np.float32)) for m in (5, 80)}
        model.close()
    c32, ls32 = np.float32(math.exp(th32[1])), np.exp(th32[2:]).astype(np.float32)
    g32 = _dk_kstar(xs.astype(np.float32), x32, c32, ls32, np.float32)
    dm32 = np.stack([gk @ lap.alpha.astype(np.float32) for gk in g32], axis=1)
    scale = np.abs(dm_t).max()
    for m, out in got.items():
        dmean = out[2]
        err = np.abs(dmean.astype(np.float64) - dm_t[:m]).max()
        err32 = np.abs(dm32[:m].astype(np.float64) - dm_t[:m]).max()
        rec[f"f32 m={m} dmean"] = {"gpu": float(err), "float32 restatement": float(err32)}
        assert err <= 4 * err32 + 1e-3 * scale, (m, err, err32)
    _note(f"rbf candidate gradients n={n}", rec)
    assert not fails, fails


@pytest.mark.gpu
@pytest.mark.parametrize("A", [np.float64, np.float32])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("S", [10, 64, 65])
def test_acquisition_search_equals_the_restatement(A, mode, S):
    from tests.test_acquire import _case, _param, _same_records, _search, _set_default_tolerances
    _set_default_tolerances()
    n, d = 500, 3
    x, yraw, yl, yn, theta = _case(A, n, d, 0, nu=INF)
    theta[2:] = np.log(0.3)
    param = _param(mode, yraw)
    rng = np.random.default_rng(S * 7 + d)
    lo, hi = np.zeros(d), np.ones(d)
    starts = rng.random((S, d)).astype(A)
    with _ctx(A) as ctx:
        ctx.set_data(x, yl)
        model = ctx.model(theta, nu=INF)
        dev = _search(model, yn, mode, param, starts, lo, hi, 150)
        ref = _search(model, yn, mode, param, starts, lo, hi, 150, restated=True)
        model.close()
    assert max(r[2] for r in ref[2]) > 1
    assert _bits(dev[0], ref[0])
    if mode == 0:
        assert _bits(dev[1], ref[1])
    assert _same_records(dev[2], ref[2])
    assert dev[3:] == ref[3:]


@pytest.mark.gpu
def test_mixed_nu_on_one_context():
    """Batches at nu = 5/2, inf, 5/2 on one context (the graph cache is keyed by nu2) each give their own bits."""
    n, d = 1025, 3
    x, y = synth(n, d)
    th = _lml_thetas(3, d, 1e-2, 0.5, 9, np.float64)
    with _ctx(np.float64) as ctx:
        ctx.set_data(x, y)
        a1 = ctx.lml_grad_batch(th, 2.5)
        b1 = ctx.lml_grad_batch(th, INF)
        a2 = ctx.lml_grad_batch(th, 2.5)
        b2 = ctx.lml_grad_batch(th, INF)
    with _ctx(np.float64) as ctx:
        ctx.set_data(x, y)
        b0 = ctx.lml_grad_batch(th, INF)
    with _ctx(np.float64) as ctx:
        ctx.set_data(x, y)
        a0 = ctx.lml_grad_batch(th, 2.5)
    for u, v, w in zip(a0, a1, a2):
        assert _bits(u, v) and _bits(u, w)
    for u, v, w in zip(b0, b1, b2):
        assert _bits(u, v) and _bits(u, w)
    assert not _bits(a0[0], b0[0])


@pytest.mark.gpu
def test_every_entry_point_accepts_inf_and_rejects_other_nus():
    import hbetune_rs_b200 as h
    from hbetune_rs_b200._lib import ALLREDUCE_FN, HbegpError, RunResult, check, lib
    from hbetune_rs_b200.gpr import _ptr
    n, d = 150, 2
    x, y = synth(n, d)
    th = _lml_thetas(2, d, 1e-2, 0.5, 3, np.float64)
    lo, hi = np.exp(th.min(axis=0) - 1), np.exp(th.max(axis=0) + 1)  # natural units
    for nu in (INF, 3.5, math.nan, -INF, 1e300):
        ok = nu == INF
        with h.Context() as ctx:
            ctx.set_data(x, y)
            calls = [
                lambda: ctx.lml_grad_batch(th, nu),
                lambda: ctx.lml_grad_batch_sharded(th, nu),
                lambda: ctx.fit_runs(th, lo, hi, nu, maxeval=3),
                lambda: check(lib.hbegp_fit_runs_sharded(ctx._h, nu, 2, _ptr(th), _ptr(lo), _ptr(hi), 3, 0, 1, ALLREDUCE_FN(), None,
                                                         (RunResult * 2)(), _ptr(np.empty_like(th))), "fit_runs_sharded"),
                lambda: ctx.model(th[0], nu).close(),
                lambda: ctx.debug_factor(th[0], nu),
                lambda: ctx.bench_phase(th, 0, 1, nu),
            ]
            for i, call in enumerate(calls):
                try:
                    call()
                    assert ok, (nu, i)
                except HbegpError as e:
                    assert not ok and e.code == -4, (nu, i, e)
            kout = np.empty((n, n))
            assert lib.hbegp_kernel_matrix(ctx._h, nu, d, _ptr(th[0][1:].copy()), n, _ptr(x), n, _ptr(x), _ptr(kout)) == (0 if ok else -4)
            gout = np.empty((n, n, d + 1))
            assert lib.hbegp_kernel_theta_grad(ctx._h, nu, d, _ptr(th[0][1:].copy()), n, _ptr(x), _ptr(kout), _ptr(gout)) == (0 if ok else -4)
            bh = ctypes.c_void_p()
            rc = lib.hbegp_batcher_create(ctx._h, nu, 2, _ptr(lo), _ptr(hi), ctypes.byref(bh))
            assert rc == (0 if ok else -4), (nu, rc)
            if ok:
                lib.hbegp_batcher_destroy(bh)


@pytest.mark.gpu
def test_multi_gpu_replica_bits():
    import torch

    import hbetune_rs_b200 as h
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    n, d = 700, 3
    x, y = synth(n, d)
    th = _lml_thetas(4, d, 1e-2, 0.4, 1, np.float64)
    xs = np.random.default_rng(0).random((300, d))
    with h.Context() as ctx:
        ctx.set_data(x, y)
        lml1, grad1, _ = ctx.lml_grad_batch(th, INF)
        m1 = ctx.model(th[0], INF)
        mean1, var1 = m1.predict(xs, warn=False)
        m1.close()
        res1, best1 = ctx.fit_runs(th, np.exp(th.min(axis=0) - 1), np.exp(th.max(axis=0) + 1), INF, maxeval=5)
    with h.MultiContext(2) as mc:
        mc.set_data(x, y)
        lml2, grad2, _ = mc.lml_grad_batch(th, INF)
        res2, best2 = mc.fit_runs(th, np.exp(th.min(axis=0) - 1), np.exp(th.max(axis=0) + 1), INF, maxeval=5)
        assert _bits(best1, best2)
        mm = mc.model(th[0], INF)
        mean2, var2 = mm.predict(xs, warn=False)
        mm.close()
    assert _bits(lml1, lml2) and _bits(grad1, grad2) and _bits(mean1, mean2) and _bits(var1, var2)
