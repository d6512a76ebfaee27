"""The f64 path against a truth far beyond double precision, held to the error LAPACK f64 makes on the same matrix.

A flat 1e-9 against LAPACK is 1e4-1e6 times looser than what f64 achieves at the noise levels of the other tests,
and at noise 1e-5 it is tighter than LAPACK's own error.  So every compared quantity X is measured against its truth
X*, computed from the matrix K the GPU itself assembled (`debug_factor`), together with LAPACK's value X_L from the
same K (`_reference`'s steps), and must satisfy

    max |X_gpu - X*| <= R max |X_L - X*| + F eps S(X),     eps = 2^-53,

where S(X) is the condition sum of X (the same expression with every term replaced by its absolute value).  It
covers what may legitimately differ: an ulp of exp between CUDA and glibc, fused against separate multiply-adds.
From a padded size of 2048 on, K^-1 is the emulated product (DESIGN K6b), and its error model, evaluated on the GPU's
own W, is added elementwise for K^-1 and contracted with |dK/dtheta| for the gradient.  Where W and K^-1 were
measured above this bound (as kappa grows), SLACK asserts the measured excess, per quantity and noise, with a 2x margin.

The LML and the noise component of the gradient are scalars that depend on W through y^T W^T W y, log det and
sum alpha_i^2 - tr K^-1.  LAPACK computes them through two triangular solves, and its error on them varies by 10x and
more between matrices one ulp apart, so a ratio to it says little.  They are held instead to what the GPU's own W
implies (`_implied_by_w`, computed to about 2^-100 from debug_factor's W, which W itself is held to LAPACK by
the factor test): |X_gpu - X(W_gpu)| <= F eps S, with S the condition sum of the GPU's finishing arithmetic.

The truth, in f64 BLAS only:
- `dd_matmul`: products to about 2^-110 of (row max x column max), from integer slices whose products are exact;
- `_refine`: one correction of LAPACK's L0 = dpotrf(K), W0 = dtrtri(L0) from the accurate residuals K - L0 L0^T and
  I - L0 W0.  What is left is of second order, (kappa eps)^2 relative;
- the derived quantities as (hi, lo) pairs or accurate sums: K^-1* = W*^T W*, alpha* by refinement, log det from the
  n logarithms in mpmath, y^T alpha* as an exact dot product, the gradient contraction and the predictions.
The CPU tests check the truth against mpmath at 40 digits and show that LAPACK's error, the yardstick, is not zero.
"""
import math
import time

import numpy as np
import pytest
from scipy.linalg import cho_factor, cho_solve, lapack

from tests.test_dispatch_sweep import (FACTOR_SHAPES, SHAPES, _ctx, _kernel_f64, _note, _np, _predict_path,
                                       _predict_truth, _reference, _rounded, _thetas, _worst_tile)
from tests.test_kinv_bits import _bits
from tests.util import random_thetas, synth

EPS = 2.0 ** -53
# error <= R * (LAPACK f64's error) + F * eps * S(X), both against the truth of the GPU's own K
R, F = 2.0, 4.0
# K: |K_gpu - K_host| <= F_K eps (c + noise), and elementwise F_K eps (|K| + (d - 1) c |M'(r)| r).  Measured on a
# B200: 4.08 eps (c + noise) at d = 3, nu = 2.5, and 0.999 of the elementwise bound at F_K = 4 for d = 1
F_K = 8.0
# Where the factor exceeds R x LAPACK + F eps S, the right-hand side is multiplied by twice the largest excess measured
# on a B200 (profiles/r07_f64_truth.json): W 1.01 at noise 1e-4 and 1.69 at 1e-5, K^-1 1.51 and 2.02.  DESIGN section 2.
SLACK = {("w", "1e-2"): 1.0, ("w", "1e-4"): 2.1, ("w", "1e-5"): 3.4,
         ("kinv", "1e-2"): 1.0, ("kinv", "1e-4"): 3.1, ("kinv", "1e-5"): 4.1}


def _family(noise):
    return "1e-2" if noise >= 5e-3 else "1e-4" if noise >= 5e-5 else "1e-5"


A = np.float64

# ------------------------------------------------------------------------------------------------ accurate arithmetic


def _dev():
    import torch
    return torch.device("cuda" if torch.cuda.is_available() else "cpu")


def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def _veltkamp(a):
    c = 134217729.0 * a  # 2^27 + 1
    hi = c - (c - a)
    return hi, a - hi


def _two_prod(a, b):
    """p + e = a b exactly (Dekker, no FMA needed)."""
    p = a * b
    ah, al = _veltkamp(a)
    bh, bl = _veltkamp(b)
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def _acc_sum(a):
    """The sum over axis 0 as (hi, lo): a cascade of TwoSums, whose errors are added up in f64.  Accurate to about
    log2(N) eps^2 of sum |a|, which is all the truth needs from a sum."""
    a = np.asarray(a, dtype=np.float64)
    err = np.zeros(a.shape[1:])
    while a.shape[0] > 1:
        h = a.shape[0] // 2
        s, e = _two_sum(a[:h], a[h:2 * h])
        err += e.sum(axis=0)
        a = np.concatenate([s, a[2 * h:]]) if a.shape[0] % 2 else s
    return _two_sum(a[0], err)


def _terms(x):
    return tuple(x) if isinstance(x, (tuple, list)) else (x,)


def _slice_terms(terms, axis, s, k):
    """The terms' sum scaled by a power of two per row (axis = 1) or column (axis = 0), so that it is below 1 there,
    cut into k integer slices of s bits: sum_t x_t = 2^e sum_q slice_q 2^-(s (q + 1)) up to 2^-(s k)."""
    import torch
    dev = _dev()
    ts = [torch.from_numpy(np.ascontiguousarray(t, dtype=np.float64)).to(dev) for t in terms]
    m = sum(t.abs() for t in ts).amax(dim=axis, keepdim=True)
    e = torch.frexp(m)[1]  # m < 2^e
    out = [torch.zeros_like(ts[0]) for _ in range(k)]
    for t in ts:
        r = torch.ldexp(t, -e)
        for q in range(k):
            r = torch.ldexp(r, torch.tensor(s, device=dev))
            sl = torch.round(r)
            r = r - sl  # exact
            out[q] += sl
    return out, e


def dd_matmul(a, b):
    """a @ b as (hi, lo), to about 2^-110 of max|a row| max|b column| per element.  a and b may be tuples of terms
    (a pair (hi, lo), say): the product of their sums.  The slices have s = floor((53 - ceil(log2 n') - 1) / 2)
    bits, n' = n times the number of term pairs, so that every slice product summed over n terms is an integer below
    2^53, hence exact; that is asserted, so a BLAS whose f64 products are not exact on integers fails here instead of
    corrupting the truth.  The partial products are combined with TwoSum.  On the GPU if there is one."""
    import torch
    a, b = _terms(a), _terms(b)
    n = a[0].shape[1]
    s = (53 - math.ceil(math.log2(n * len(a) * len(b))) - 1) // 2
    k = -(-116 // s)
    sa, ea = _slice_terms(a, 1, s, k)
    sb, eb = _slice_terms(b, 0, s, k)
    hi = torch.zeros((a[0].shape[0], b[0].shape[1]), dtype=torch.float64, device=sa[0].device)
    lo = torch.zeros_like(hi)
    for lvl in range(k - 1, -1, -1):  # smallest partial products first
        for p in range(lvl + 1):
            prod = sa[p] @ sb[lvl - p]
            assert torch.equal(prod, torch.round(prod)) and float(prod.abs().max()) < 2.0 ** 53, \
                "an f64 product of integer slices is not exact"
            v = torch.ldexp(prod, torch.tensor(-s * (lvl + 2), device=hi.device))
            t = hi + v
            bb = t - hi
            lo += (hi - (t - bb)) + (v - bb)
            hi = t
    t = hi + lo
    lo = lo - (t - hi)
    scale = ea + eb  # exact power-of-two scaling
    return torch.ldexp(t, scale).cpu().numpy(), torch.ldexp(lo, scale).cpu().numpy()


# ------------------------------------------------------------------------------------------------ the truth


def _lapack_factor(k):
    low = np.tril(cho_factor(k, lower=True)[0])
    w, info = lapack.dtrtri(low, lower=1)
    assert info == 0
    return low, np.tril(w)


def _refine(k, ls, ws):
    """One correction of L = sum(ls), W = sum(ws) for K = L L^T: E = K - L L^T (accurate), dL = L0 Phi(W0 E W0^T)
    with Phi the strict lower triangle plus half the diagonal, R = I - L W (accurate) - dL W0, dW = tril(W0 R).
    Returns the terms with dL and dW appended."""
    n = k.shape[0]
    hi, lo = dd_matmul(tuple(ls), tuple(t.T for t in ls))
    e = (k - hi) - lo
    x = ws[0] @ e @ ws[0].T
    dl = np.tril(ls[0] @ (np.tril(x, -1) + np.diag(np.diag(x)) / 2))
    hi, lo = dd_matmul(tuple(ls), tuple(ws))
    r = ((np.eye(n) - hi) - lo) - dl @ ws[0]
    return ls + [dl], ws + [np.tril(ws[0] @ r)]


def _derivs(theta, x, nu):
    """The host's f64 dK/dtheta_k of _reference: noise I (as the scalar noise), kc, f ((x_i - x_j) / l_k)^2."""
    x = np.asarray(x, dtype=np.float64)
    d = x.shape[1]
    noise, c, ls = math.exp(theta[0]), math.exp(theta[1]), np.exp(np.asarray(theta[2:], dtype=np.float64))
    kc = _kernel_f64(x, x, c, ls, nu)
    rr = np.sqrt(sum(((x[:, j, None] - x[None, :, j]) / ls[j]) ** 2 for j in range(d)))
    if nu == 0.5:
        with np.errstate(divide="ignore", invalid="ignore"):
            f = np.where(rr > 0, kc / rr, 0.0)
    elif nu == 1.5:
        f = 3.0 * c * np.exp(-math.sqrt(3.0) * rr)
    else:
        f = 5.0 / 3.0 * c * np.exp(-math.sqrt(5.0) * rr) * (math.sqrt(5.0) * rr + 1.0)
    return [noise, kc] + [f * ((x[:, j, None] - x[None, :, j]) / ls[j]) ** 2 for j in range(d)]


class Truth:
    """The exact factor, K^-1, alpha, LML and gradient of one symmetric f64 K (to about 2^-100), lazily."""

    def __init__(self, k, y, theta=None, x=None, nu=2.5, refinements=1):
        self.k, self.y = np.asarray(k, dtype=np.float64), np.asarray(y, dtype=np.float64)
        self.n = self.k.shape[0]
        self.theta, self.x, self.nu = theta, x, nu
        l0, w0 = _lapack_factor(self.k)
        self.ls, self.ws = [l0], [w0]
        for _ in range(refinements):
            self.ls, self.ws = _refine(self.k, self.ls, self.ws)
        self._kinv = self._alpha = self._lml = self._grad = None

    @property
    def w(self):
        return self.ws

    @property
    def kinv(self):
        if self._kinv is None:
            self._kinv = dd_matmul(tuple(t.T for t in self.ws), tuple(self.ws))
        return self._kinv

    @property
    def alpha(self):
        """alpha0 = cho_solve(L0, y), then two steps alpha += W0^T W0 (y - K alpha), the residual accurate."""
        if self._alpha is None:
            w0 = self.ws[0]
            terms = [cho_solve((self.ls[0], True), self.y)]
            for _ in range(2):
                hi, lo = dd_matmul(self.k, tuple(t[:, None] for t in terms))
                r = (self.y - hi[:, 0]) - lo[:, 0]
                terms.append(w0.T @ (w0 @ r))
            self._alpha = terms
        return self._alpha

    def logdet_mp(self):
        import mpmath
        with mpmath.workdps(40):
            diag = [sum(mpmath.mpf(float(t[i, i])) for t in self.ls) for i in range(self.n)]
            return 2 * mpmath.fsum(mpmath.log(v) for v in diag)

    def ya_mp(self):
        """y^T alpha* exactly (TwoProduct and math.fsum), as an mpf."""
        import mpmath
        parts = []
        for t in self.alpha:
            p, e = _two_prod(self.y, t)
            parts += p.tolist() + e.tolist()
        with mpmath.workdps(40):
            return mpmath.fsum(mpmath.mpf(v) for v in parts)

    @property
    def lml(self):
        """-1/2 y^T alpha* - 1/2 log det - n/2 ln(2 pi) as (float, mpf)."""
        if self._lml is None:
            import mpmath
            with mpmath.workdps(40):
                v = -self.ya_mp() / 2 - self.logdet_mp() / 2 - mpmath.mpf(self.n) / 2 * mpmath.log(2 * mpmath.pi)
                self._lml = (float(v), v)
        return self._lml

    def outer_alpha(self):
        a = tuple(t[:, None] for t in self.alpha)
        return dd_matmul(a, tuple(t.T for t in a))

    @property
    def grad(self):
        """1/2 sum_ij (alpha* alpha*^T - K^-1*)_ij G_k,ij for the host's f64 G_k, with its condition sum
        1/2 sum |alpha* alpha*^T - K^-1*| |G_k|, and the contraction with |G_k| of a given elementwise matrix."""
        if self._grad is None:
            (ah, al), (kh, kl) = self.outer_alpha(), self.kinv
            gs, scale = [], []
            for j, g in enumerate(_derivs(self.theta, self.x, self.nu)):
                if j == 0:  # noise I
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
        """1/2 sum_ij m_ij |G_k,ij| for an elementwise bound m."""
        out = []
        for j, g in enumerate(_derivs(self.theta, self.x, self.nu)):
            out.append(0.5 * (float(np.trace(m)) * g if j == 0 else float((m * np.abs(g)).sum())))
        return np.array(out)


def _err(got, pair):
    """|got - (hi + lo)| elementwise."""
    hi, lo = pair
    return np.abs((np.asarray(got, dtype=np.float64) - hi) - lo)


def _wsum_err(got, terms):
    """|got - sum(terms)|, the terms summed from the largest."""
    r = np.asarray(got, dtype=np.float64) - terms[0]
    for t in terms[1:]:
        r = r - t
    return np.abs(r)


# ------------------------------------------------------------------------------------------------ the rule


def _rule(rec, fails, key, e_gpu, e_lapack, scale, extra=0.0, where=None, slack=1.0):
    """max |X_gpu - X*| <= R max |X_L - X*| + F eps S(X) (+ the emulation's bound, elementwise), times SLACK where
    a measured excess is asserted instead.  Records err/bound at slack 1."""
    e_gpu = np.atleast_1d(np.asarray(e_gpu, dtype=np.float64))
    e_l = float(np.max(e_lapack))
    bound = R * e_l + F * EPS * scale + np.asarray(extra)
    excess = float(np.max(e_gpu / bound))
    rec[key] = {"gpu": float(e_gpu.max()), "lapack": e_l, "ratio": float(e_gpu.max()) / e_l if e_l else None,
                "scale": float(scale), "err/bound": excess}
    if excess > slack:
        fails.append((key, rec[key], where(e_gpu) if where is not None else None))


def _emu_bound(w, kinv, np_):
    """DESIGN K6b on the GPU's own W: |K^-1_emu - W^T W|_ij <= 2^-b (M_j |W_.i|_1 + M_i |W_.j|_1) + np 2^-2b M_i M_j
    + 2^-53 |K^-1_ij|, M_j = max_{k >= j} |W_kj|; zero below a padded size of 2048 (the DMMA product)."""
    if np_ < 2048:
        return 0.0
    b = _bits(np_)
    wl = np.abs(np.tril(w))
    m, l1 = wl.max(axis=0), wl.sum(axis=0)
    return (2.0 ** -b * (m[None, :] * l1[:, None] + m[:, None] * l1[None, :]) + np_ * 2.0 ** (-2 * b) * np.outer(m, m)
            + 2.0 ** -53 * np.abs(kinv))


def _sym(low):
    low = np.tril(low)
    return low + np.tril(low, -1).T


def _gpu_k(ctx, theta, nu=2.5):
    out = ctx.debug_factor(theta, nu=nu, want=("k",))
    assert out["status"] == 0
    return _sym(out["k"])


def _lml_err(lml, truth):
    import mpmath
    with mpmath.workdps(40):
        return float(abs(mpmath.mpf(float(lml)) - truth.lml[1]))


def _sq_sum(hi, lo):
    """sum (hi + lo)^2 over axis 0, to about eps^2 of itself, as an mpf per column."""
    import mpmath
    p, e = _two_prod(hi, hi)
    sh, sl = _acc_sum(np.concatenate([p, e, 2 * hi * lo]))
    with mpmath.workdps(40):
        return [mpmath.mpf(float(a)) + mpmath.mpf(float(b)) for a, b in zip(np.atleast_1d(sh), np.atleast_1d(sl))]


def _implied_by_w(w, y, noise):
    """The LML and the noise component of the gradient that the GPU's W implies, to about 2^-100 (mpf):
    LML(W) = -1/2 |W y|^2 + sum ln W_ii - n/2 ln 2 pi and g0(W) = 1/2 noise (|W^T W y|^2 - |W|_F^2), with the condition
    sums of the GPU's arithmetic for them (as S(var)): |W y|^T |W| |y| for the mat-vec, and one unit per pivot for the
    log-determinant, which the kernels take as -1/2 ln of a product of eight rounded pivot reciprocals: about 23
    roundings per eight pivots (a refined reciprocal within an ulp each, seven products, the logarithm), which the
    logarithm turns into absolute errors, 1.5 eps per pivot after the factor 1/2."""
    import mpmath
    n = len(y)
    wl = np.tril(w)
    uh, ul = dd_matmul(wl, y[:, None])
    ah, al = dd_matmul(wl.T, (uh, ul))
    u2 = _sq_sum(uh, ul)[0]
    a2 = _sq_sum(ah, al)[0]
    p, e = _two_prod(wl.ravel(), wl.ravel())
    fh, fl = _acc_sum(np.concatenate([p, e]))
    wy = np.abs(wl) @ np.abs(y)
    with mpmath.workdps(40):
        lnw = [mpmath.log(mpmath.mpf(float(v))) for v in np.diag(wl)]
        lml = -u2 / 2 + mpmath.fsum(lnw) - mpmath.mpf(n) / 2 * mpmath.log(2 * mpmath.pi)
        g0 = mpmath.mpf(noise) / 2 * (a2 - (mpmath.mpf(float(fh)) + mpmath.mpf(float(fl))))
        s_lml = float(np.abs(uh[:, 0]) @ wy) + float(sum(abs(v) for v in lnw)) + n + n / 2 * math.log(2 * math.pi)
    s_g0 = 0.5 * noise * (float(a2) + float(fh) + 2 * float(np.abs(ah[:, 0]) @ (np.abs(wl).T @ wy)))
    return lml, g0, s_lml, s_g0


def _check_lml_grad(rec, fails, tag, lml, grad, truth, lapack, np_, w_gpu, noise):
    """The LML and g0 against what the GPU's W implies (plus, for g0 from np 2048 on, the emulated K^-1's bound on its
    diagonal); every other gradient component by the rule against LAPACK.  The errors against the truth are recorded."""
    import mpmath
    lml_w, g0_w, s_lml, s_g0 = _implied_by_w(w_gpu, truth.y, noise)
    g_hi, g_lo, g_scale = truth.grad
    extra = np.zeros(len(g_hi))
    if np_ >= 2048:
        extra = truth.grad_contract(_emu_bound(w_gpu, truth.kinv[0], np_))
    with mpmath.workdps(40):
        g0_t = mpmath.mpf(float(g_hi[0])) + mpmath.mpf(float(g_lo[0]))
        for key, got, imp, star, lap, scale, ex in (
                ("lml", lml, lml_w, truth.lml[1], lapack.lml, s_lml, 0.0),
                ("grad[0]", grad[0], g0_w, g0_t, lapack.grad[0], s_g0, float(extra[0]))):
            e_arith = float(abs(mpmath.mpf(float(got)) - imp))
            bound = F * EPS * scale + ex
            rec[f"{tag} {key}"] = {"gpu": float(abs(mpmath.mpf(float(got)) - star)),
                                   "lapack": float(abs(mpmath.mpf(float(lap)) - star)),
                                   "implied by the GPU's W": float(abs(imp - star)),
                                   "gpu - implied": e_arith, "scale": scale, "err/bound": e_arith / bound}
            rec[f"{tag} {key}"]["ratio"] = rec[f"{tag} {key}"]["gpu"] / rec[f"{tag} {key}"]["lapack"]
            if e_arith > bound:
                fails.append((f"{tag} {key}", rec[f"{tag} {key}"]))
    for j in range(1, len(g_hi)):
        _rule(rec, fails, f"{tag} grad[{j}]", abs((grad[j] - g_hi[j]) - g_lo[j]), abs((lapack.grad[j] - g_hi[j]) - g_lo[j]),
              g_scale[j], extra[j])


# ------------------------------------------------------------------------------------------------ CPU part


def test_dd_matmul_is_exact_for_integers():
    rng = np.random.default_rng(1)
    for n in (1, 7, 64, 300):
        a = rng.integers(-(2 ** 20), 2 ** 20, (n + 3, n)).astype(np.float64)
        b = rng.integers(-(2 ** 20), 2 ** 20, (n, n + 1)).astype(np.float64)
        hi, lo = dd_matmul(a, b)
        want = a.astype(np.int64).astype(object) @ b.astype(np.int64).astype(object)
        np.testing.assert_array_equal(hi, want.astype(np.float64))
        assert (lo == 0).all()


@pytest.mark.parametrize("n", [3, 40, 130])
def test_dd_matmul_matches_python_integers(n):
    """Full-mantissa inputs with scales from 2^-30 to 2^30 per row and column, and a pair (hi, lo) as an operand:
    hi + lo within n 2^-104 of max|a row| max|b col| of the exact product (the slices keep about 116 bits)."""
    from fractions import Fraction as Fr
    rng = np.random.default_rng(n)
    a = np.ldexp(rng.standard_normal((n, n)), rng.integers(-30, 30, n)[:, None])
    b = np.ldexp(rng.standard_normal((n, n)), rng.integers(-30, 30, n)[None, :])
    b_lo = b * 2.0 ** -60 * rng.standard_normal((n, n))
    scale = np.abs(a).max(axis=1)[:, None] * np.abs(b).max(axis=0)[None, :]
    cells = [(0, 0), (n - 1, n - 1)] + [tuple(rng.integers(0, n, 2)) for _ in range(40)]
    for terms in ((b,), (b, b_lo)):
        hi, lo = dd_matmul(a, terms if len(terms) > 1 else b)
        for i, j in cells:
            want = sum(Fr(float(a[i, q])) * sum(Fr(float(t[q, j])) for t in terms) for q in range(n))
            got = Fr(float(hi[i, j])) + Fr(float(lo[i, j]))
            assert abs(got - want) <= Fr(2.0 ** -104) * Fr(float(scale[i, j])) * n, (i, j, float(got - want))


def _mp_reference(k, y, derivs):
    """Cholesky, W = L^-1, K^-1 = W^T W, alpha, log det and the gradient contraction in mpmath at 40 digits."""
    import mpmath
    n = k.shape[0]
    with mpmath.workdps(40):
        mpf = mpmath.mpf
        a = [[mpf(v) for v in row] for row in k.tolist()]
        low = [[mpf(0)] * n for _ in range(n)]
        for j in range(n):
            lj = low[j]
            lj[j] = mpmath.sqrt(a[j][j] - mpmath.fdot(lj[:j], lj[:j]))
            inv = 1 / lj[j]
            for i in range(j + 1, n):
                low[i][j] = (a[i][j] - mpmath.fdot(low[i][:j], lj[:j])) * inv
        wc = []  # wc[j][k - j] = W[k][j]
        for j in range(n):
            col = [1 / low[j][j]]
            for i in range(j + 1, n):
                col.append(-mpmath.fdot(low[i][j:i], col) / low[i][i])
            wc.append(col)
        w = [[wc[j][i - j] if i >= j else mpf(0) for j in range(n)] for i in range(n)]
        kinv = [[None] * n for _ in range(n)]
        for i in range(n):
            for j in range(i + 1):
                v = mpmath.fdot(wc[i][0:], wc[j][i - j:])
                kinv[i][j] = kinv[j][i] = v
        ym = [mpf(v) for v in y.tolist()]
        alpha = [mpmath.fdot(row, ym) for row in kinv]
        logdet = 2 * mpmath.fsum(mpmath.log(low[i][i]) for i in range(n))
        lml = -mpmath.fdot(ym, alpha) / 2 - logdet / 2 - mpf(n) / 2 * mpmath.log(2 * mpmath.pi)
        grad = []
        for j, g in enumerate(derivs):
            if j == 0:
                grad.append(mpmath.fsum((alpha[i] ** 2 - kinv[i][i]) * mpf(g) for i in range(n)) / 2)
            else:
                gl = g.tolist()
                grad.append(mpmath.fsum((alpha[i] * alpha[jj] - kinv[i][jj]) * mpf(gl[i][jj])
                                        for i in range(n) for jj in range(n)) / 2)
        return dict(w=w, kinv=kinv, alpha=alpha, logdet=logdet, lml=lml, grad=grad)


def _mp_err(got, want):
    """max |got - want| for got a float array or a list of float arrays (terms), want nested mpf lists."""
    import mpmath
    terms = [np.asarray(t, dtype=np.float64) for t in _terms(got)]
    with mpmath.workdps(40):
        if terms[0].ndim == 0:
            return float(abs(mpmath.fsum([mpmath.mpf(float(t)) for t in terms]) - want))
        flat_w = [v for row in want for v in row] if terms[0].ndim == 2 else list(want)
        flat_t = [t.ravel().tolist() for t in terms]
        return float(max(abs(mpmath.fsum([mpmath.mpf(ft[i]) for ft in flat_t]) - flat_w[i]) for i in range(len(flat_w))))


@pytest.mark.parametrize("nu", [0.5, 2.5])
@pytest.mark.parametrize("noise", [1e-2, 1e-5])
def test_truth_matches_mpmath(noise, nu):
    """n = 96: W*, K^-1*, alpha*, log det, the LML and the gradient within 1e-6 of LAPACK's error on the same K
    (plus eps^2 of the quantity's scale, in case LAPACK happens to be exact on a scalar)."""
    n, d = 96, 3
    x, y = synth(n, d, seed=11)
    theta = random_thetas(1, d, seed=12, noise=(noise, noise * 1.01))[0]
    lap = _reference(theta, x, y, nu)
    k = lap.k
    tr = Truth(k, y, theta, x, nu)
    mp = _mp_reference(k, y, _derivs(theta, x, nu))
    fails = []

    def check(key, truth_terms, lapack_val, want, scale):
        e_t, e_l = _mp_err(truth_terms, want), _mp_err(lapack_val, want)
        if not e_t <= 1e-6 * e_l + EPS ** 2 * scale:
            fails.append((key, e_t, e_l))
        return e_t, e_l

    check("w", tr.ws, lap.w, mp["w"], np.abs(lap.w).max())
    check("kinv", list(tr.kinv), lap.kinv, mp["kinv"], np.abs(lap.kinv).max())
    check("alpha", tr.alpha, lap.alpha, mp["alpha"], np.abs(lap.alpha).max())
    import mpmath
    with mpmath.workdps(40):
        e_t = float(abs(tr.logdet_mp() - mp["logdet"]))
        e_l = float(abs(mpmath.mpf(2 * float(np.log(np.diag(np.linalg.cholesky(k))).sum())) - mp["logdet"]))
        if not e_t <= 1e-6 * e_l + EPS ** 2 * lap.lml_scale:
            fails.append(("logdet", e_t, e_l))
        e_t = float(abs(tr.lml[1] - mp["lml"]))
        e_l = float(abs(mpmath.mpf(lap.lml) - mp["lml"]))
        if not e_t <= 1e-6 * e_l + EPS ** 2 * lap.lml_scale:
            fails.append(("lml", e_t, e_l))
    g_hi, g_lo, g_scale = tr.grad
    for j in range(len(g_hi)):
        check(f"grad[{j}]", [g_hi[j], g_lo[j]], lap.grad[j], mp["grad"][j], g_scale[j])
    assert not fails, fails


def test_second_refinement_changes_nothing():
    """n = 2112 at noise 1e-5: a second correction moves W* by less than 1e-6 of LAPACK's error, so the first one
    left nothing that matters."""
    n, d = 2112, 3
    x, y = synth(n, d, seed=n)
    theta = random_thetas(1, d, seed=n, noise=(1e-5, 1.01e-5))[0]
    k = _kernel_f64(x, x, math.exp(theta[1]), np.exp(theta[2:]), 2.5) + math.exp(theta[0]) * np.eye(n)
    tr = Truth(k, y)
    ls2, ws2 = _refine(k, tr.ls, tr.ws)
    _, w_l = _lapack_factor(k)
    e_l = float(_wsum_err(w_l, tr.ws).max())
    moved = float(np.abs(ws2[-1]).max())
    _note("truth: second refinement n=2112 noise=1e-5", {"moved": moved, "lapack W error": e_l,
                                                         "max|W|": float(np.abs(w_l).max())})
    assert 0 < e_l and moved <= 1e-6 * e_l, (moved, e_l)


def test_lapack_error_grows_with_kappa():
    """The yardstick measures something: LAPACK's W error against the truth is not zero and grows as the noise falls
    from 1e-2 to 1e-5 (kappa from about 1e4 to 1e7)."""
    n, d = 512, 3
    x, y = synth(n, d, seed=5)
    errs = []
    for noise in (1e-2, 1e-3, 1e-4, 1e-5):
        theta = random_thetas(1, d, seed=6, noise=(noise, noise * 1.01))[0]
        lap = _reference(theta, x, y)
        tr = Truth(lap.k, y)
        errs.append(float(_wsum_err(lap.w, tr.ws).max() / np.abs(lap.w).max()))
    _note("truth: lapack W error n=512 by noise 1e-2..1e-5", {"rel": errs})
    assert errs[0] > 0 and errs[-1] > 30 * errs[0], errs
    assert all(b > a for a, b in zip(errs, errs[1:])), errs


# ------------------------------------------------------------------------------------------------ GPU part

_CACHE = {}


def _truth_of(key, k, y, theta, x, nu=2.5):
    """Built once per matrix within the module (the n = 2112 truth is the expensive step)."""
    if key not in _CACHE:
        _CACHE[key] = Truth(k, y, theta, x, nu)
    return _CACHE[key]


def _dmatern_r(r, nu):
    """|dM/dr| r of the Matern correlation."""
    if nu == 0.5:
        return r * np.exp(-r)
    if nu == 1.5:
        t = math.sqrt(3.0) * r
        return t * t * np.exp(-t)
    t = math.sqrt(5.0) * r
    return t * t / 3 * (1 + t) * np.exp(-t)


@pytest.mark.gpu
@pytest.mark.parametrize("nu", [0.5, 1.5, 2.5])
@pytest.mark.parametrize("d", [1, 3, 16, 64, 65, 200])
def test_assembled_k_to_a_few_ulps(d, nu):
    """k_assemble against the host's kernel: within F_K ulps of c + noise, and elementwise within F_K ulps of |K_ij|
    plus what the squared distance may differ by: the GPU fuses each of its d - 1 additions with the square, which
    moves r by up to (d - 1) eps relative, and K by c |M'(r)| r times that.  At d = 1 both round the one square the
    same way, so an exp a few ulps off shows.  Duplicate rows (r = 0) under nu = 0.5."""
    n = 300
    x, y = synth(n, d, seed=d)
    if nu == 0.5:
        x[100:140] = x[:40]
    theta = _rounded(random_thetas(1, d, seed=d + 1, noise=(1e-4, 1e-2), ls=(0.05 * math.sqrt(d), 3 * math.sqrt(d)))[0], A)
    if d == 1:
        theta[2] = math.log(0.04)  # r up to 25: exp arguments of a few tens, where an exp |x| ulps off shows
    noise, c, ls = math.exp(theta[0]), math.exp(theta[1]), np.exp(theta[2:])
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        out = ctx.debug_factor(theta, nu=nu, want=("k",))
    kh = _kernel_f64(x, x, c, ls, nu) + noise * np.eye(n)
    err = np.tril(np.abs(out["k"] - kh))
    r = np.sqrt(sum(((x[:, j, None] - x[None, :, j]) / ls[j]) ** 2 for j in range(d)))
    bound = F_K * EPS * (np.abs(kh) + (d - 1) * c * _dmatern_r(r, nu))
    ulps = float(err.max() / (EPS * (c + noise)))
    rel = float(np.tril(err / bound).max())
    _note(f"K d={d} nu={nu}", {"max err / eps (c + noise)": ulps, "max err / elementwise bound": rel})
    assert ulps <= F_K, (ulps, _worst_tile(err))
    assert rel <= 1.0, (rel, _worst_tile(np.tril(err / bound)))


@pytest.mark.gpu
@pytest.mark.parametrize("noise", [1e-2, 1e-4, 1e-5])
@pytest.mark.parametrize("n,d", FACTOR_SHAPES)
def test_factor_against_the_truth(n, d, noise):
    """W and K^-1 of debug_factor against the truth of the GPU's own K: leaf, node, every GEMM class on 32x32 and
    64x64 tiles, both sides of the K^-1 emulation."""
    x, y = synth(n, d)
    theta = _rounded(random_thetas(1, d, seed=n, noise=(noise, noise * 1.01))[0], A)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        out = ctx.debug_factor(theta)
    assert out["status"] == 0
    k = _sym(out["k"])
    t0 = time.perf_counter()
    tr = _truth_of(("factor", n, d, noise), k, y, theta, x)
    kinv = tr.kinv
    t_truth = time.perf_counter() - t0
    lap = _reference(theta, x, y, k=k)
    rec, fails = {}, []
    fam = _family(noise)
    e_w = _wsum_err(np.tril(out["w"]), tr.ws)
    _rule(rec, fails, "w", e_w, _wsum_err(lap.w, tr.ws), np.abs(tr.ws[0]).max(), where=_worst_tile,
          slack=SLACK[("w", fam)])
    _rule(rec, fails, "kinv", _err(out["kinv"], kinv), _err(lap.kinv, kinv), np.abs(kinv[0]).max(),
          _emu_bound(out["w"], kinv[0], _np(n)), where=_worst_tile, slack=SLACK[("kinv", fam)])
    rec["w"]["worst tile"] = _worst_tile(e_w)
    rec["w"]["lapack worst tile"] = _worst_tile(_wsum_err(lap.w, tr.ws))
    rec["truth s"] = t_truth
    _note(f"factor n={n} d={d} noise={noise:g}", rec)
    assert not fails, fails


@pytest.mark.gpu
@pytest.mark.parametrize("n,d,B", SHAPES)
def test_lml_and_gradient_against_the_truth(n, d, B):
    """lml_grad_batch at the dispatch-sweep shapes (graphs and direct launches, stream groups, the side stream,
    padded batches): the first, middle and last member, the last at noise 1e-5, component by component."""
    x, y = synth(n, d)
    thetas = np.stack([_rounded(t, A) for t in _thetas(B, d, A, seed=B + n)])
    thetas[-1, 0] = _rounded(np.array([math.log(1e-5)]), A)[0]
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        lml, grad, status = ctx.lml_grad_batch(thetas)
        check = sorted({0, B // 2, B - 1})
        ks = {b: _gpu_k(ctx, thetas[b]) for b in check}
        ws = {b: ctx.debug_factor(thetas[b], want=("w",))["w"] for b in check}
    assert (status == 0).all()
    rec, fails = {}, []
    for b in check:
        tr = Truth(ks[b], y, thetas[b], x)
        lap = _reference(thetas[b], x, y, k=ks[b])
        noise = math.exp(thetas[b, 0])
        _check_lml_grad(rec, fails, f"b={b} noise={noise:.2g}", lml[b], grad[b], tr, lap, _np(n), ws[b], noise)
    _note(f"lml n={n} d={d} B={B}", rec)
    assert not fails, fails


def _candidates(x, m, seed):
    """m rows: 10 training points, 10 within 1e-7 of one, the rest uniform; the variance cancels at the first 20."""
    rng = np.random.default_rng(seed)
    xs = rng.random((m, x.shape[1]))
    idx = rng.choice(x.shape[0], 20, replace=False)
    xs[:10] = x[idx[:10]]
    xs[10:20] = x[idx[10:]] + 1e-7 * rng.standard_normal((10, x.shape[1]))
    return xs


def _predict_star(tr, theta, x, xs, nu=2.5):
    """mean* = k* alpha* and var* = c + 1e-5 - |W* k*|^2 (clamped at 0 like the kernels), with S(mean) and S(var)."""
    c = math.exp(theta[1])
    ks = _kernel_f64(xs, x, c, np.exp(theta[2:]), nu)
    mh, ml = dd_matmul(ks, tuple(t[:, None] for t in tr.alpha))
    uh, ul = dd_matmul(tuple(tr.ws), ks.T)
    p, e = _two_prod(uh, uh)
    sh, sl = _acc_sum(np.concatenate([p, e, 2 * uh * ul]))
    th, tl = _two_sum(c, 1e-5)
    var = np.maximum((th - sh) + (tl - sl), 0.0)
    s_mean = np.abs(ks) @ np.abs(tr.alpha[0])
    s_var = c + 1e-5 + 2 * (np.abs(uh) * (np.abs(tr.ws[0]) @ np.abs(ks.T))).sum(axis=0)
    return (mh[:, 0], ml[:, 0]), var, s_mean, s_var


def _check_predictions(rec, fails, tag, model, tr, lap, theta, x, xs, ms):
    tm, tv, s_mean, s_var = _predict_star(tr, theta, x, xs)
    lm, _ = _predict_truth(theta, x, xs, lap)
    ks = _kernel_f64(xs, x, math.exp(theta[1]), np.exp(theta[2:]), 2.5)
    u = ks @ lap.w.T  # LAPACK's variance in the kernels' form, c + 1e-5 - |W_L k*|^2
    lv = np.maximum(math.exp(theta[1]) + 1e-5 - np.einsum("ij,ij->i", u, u), 0.0)
    for m in ms:
        mean, var = model.predict(xs[:m], warn=False)
        sl = slice(0, m)
        _rule(rec, fails, f"{tag} m={m} mean", _err(mean, (tm[0][sl], tm[1][sl])), _err(lm[sl], (tm[0][sl], tm[1][sl])),
              s_mean[sl].max(), where=lambda e: f"worst candidate {int(e.argmax())}")
        _rule(rec, fails, f"{tag} m={m} var", np.abs(var - tv[sl]), np.abs(lv[sl] - tv[sl]), s_var[sl].max(),
              where=lambda e: f"worst candidate {int(e.argmax())}")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1025, 2049])
def test_predictions_against_the_truth(n):
    """The throughput path with the train tiles split over grid.y (m = 1000) and the latency path (m = 1, 17, 64),
    at candidates on, next to and away from the training points, noise 1e-4."""
    d = 3
    x, y = synth(n, d, seed=n)
    theta = _rounded(random_thetas(1, d, seed=5, noise=(1e-4, 1.01e-4))[0], A)
    xs = _candidates(x, 1000, n)
    assert _predict_path(1000, d, _np(n), 8) == "split" and _predict_path(64, d, _np(n), 8) == "latency"
    rec, fails = {}, []
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        k = _gpu_k(ctx, theta)
        tr = _truth_of(("predict", n), k, y, theta, x)
        lap = _reference(theta, x, y, k=k)
        model = ctx.model(theta)
        _check_predictions(rec, fails, f"n={n}", model, tr, lap, theta, x, xs, (1, 17, 64, 1000))
        model.close()
    _note(f"predict n={n} noise=1e-4", rec)
    assert not fails, fails


@pytest.mark.gpu
def test_append_chain_against_the_truth():
    """1000 -> 1100 -> 1300 at noise 1e-4: each appended W comes from another recursion tree (DESIGN section 3) and
    is held to the same rule: LML, alpha, K^-1 and predictions on both paths, against the truth of its K."""
    import hbetune_rs_b200 as h
    d = 3
    x, y = synth(1300, d, seed=13)
    theta = _rounded(random_thetas(1, d, seed=14, noise=(1e-4, 1.01e-4))[0], A)
    xs = _candidates(x, 300, 15)
    rec, fails = {}, []
    with _ctx(A) as ctx:
        ctx.set_data(x[:1000], y[:1000])
        models = [ctx.model(theta)]
        for n in (1100, 1300):
            ctx.set_data(x[:n], y[:n])
            m = h.Model(ctx, prior=models[-1], want_kinv=True)
            models.append(m)
            assert m.appended, n
            k = _gpu_k(ctx, theta)
            tr = Truth(k, y[:n], theta, x[:n])
            lap = _reference(theta, x[:n], y[:n], k=k)
            tag = f"1000->{n}"
            _rule(rec, fails, f"{tag} lml", _lml_err(m.lml, tr), _lml_err(lap.lml, tr), lap.lml_scale)
            s_alpha = float((np.abs(tr.ws[0]).T @ (np.abs(tr.ws[0]) @ np.abs(y[:n]))).max())
            _rule(rec, fails, f"{tag} alpha", _wsum_err(m.alpha, tr.alpha), _wsum_err(lap.alpha, tr.alpha), s_alpha)
            kinv = tr.kinv
            _rule(rec, fails, f"{tag} kinv", _err(m.k_inv, kinv), _err(lap.kinv, kinv), np.abs(kinv[0]).max(),
                  where=_worst_tile)
            _check_predictions(rec, fails, tag, m, tr, lap, theta, x[:n], xs, (17, 300))
        for m in models:
            m.close()
    _note("append chain 1000->1100->1300 noise=1e-4", rec)
    assert not fails, fails
