"""The acquisition search on the device (hbegp_acquire_ei, hbegp_acquire_confidence_bound).

The truth is tests/cpp/acquire_restatement.cpp: one BoundedLbfgs of lbfgs.h per start, compiled with the library's host
flags, driven round by round through the public hbegp_predict_mean_ei_grad / hbegp_predict_confidence_bound_grad on all
S rows.  Every output of the device search must equal it bit for bit.  The other tests check what a search must give
whatever its optimiser: points inside the box, values no worse than the starts and equal to a fresh prediction, the
best of a dense grid reached, determinism, and the edge cases of the interface.
"""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RESTATEMENT = os.path.join(ROOT, "tests", "cpp", "libacquire_restatement.so")
FTOL, GTOL = 1e-11, 1e-8  # the defaults of hbegp_lbfgs_set_tolerances


def _case(A, n, d, proj=0, nu=2.5, seed=0):
    """Synthetic data (y in [10, 17)), its normalisation, and the model's theta rounded to A."""
    from hbetune_rs_b200.estimator import YNormalize
    from tests.util import random_thetas, synth
    x, yraw = synth(n, d, seed=n + 1 + seed, A=A)
    yraw = (yraw * A(3) + A(10)).astype(A)
    yl, yn = YNormalize.new_project_into_normalized(yraw, proj, A=A)
    theta = random_thetas(1, d, seed=n + seed, noise=(1e-2, 1.01e-2))[0].astype(A).astype(np.float64)
    return x, yraw, yl, yn, theta


def _ctx(A):
    import hbetune_rs_b200 as h
    return h.Context(0, h.F64 if A == np.float64 else h.F32)


def _restatement():
    if not os.path.exists(RESTATEMENT):
        subprocess.run(["make", "-C", os.path.join(ROOT, "hbetune_rs_b200", "csrc")], check=True)
    from hbetune_rs_b200 import _lib
    lib = ctypes.CDLL(RESTATEMENT)
    lib.acq_restatement.restype = ctypes.c_int
    lib.acq_restatement.argtypes = [ctypes.c_void_p, ctypes.POINTER(_lib.YNorm), ctypes.c_int, ctypes.c_double, ctypes.c_long,
                                    ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_double,
                                    ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(_lib.AcqResult),
                                    ctypes.POINTER(ctypes.c_long), ctypes.POINTER(ctypes.c_longlong)]
    return lib


def _search(model, yn, mode, param, starts, lo, hi, maxeval, restated=False):
    """The device search (or the restatement): (x, mean, records as tuples, best_index, n_rounds)."""
    from hbetune_rs_b200 import _lib
    from hbetune_rs_b200._lib import check
    from hbetune_rs_b200.gpr import _ptr
    A = yn.A
    starts = np.ascontiguousarray(starts, dtype=A)
    S, d = starts.shape
    lo, hi = np.ascontiguousarray(lo, dtype=np.float64), np.ascontiguousarray(hi, dtype=np.float64)
    x, mean = np.full((S, d), 7, dtype=A), np.full(S, 7, dtype=A)
    res = (_lib.AcqResult * max(S, 1))()
    best, rounds = ctypes.c_long(-7), ctypes.c_longlong(-7)
    h = model.single_handle()
    if restated:
        rc = _restatement().acq_restatement(h, ctypes.byref(yn._raw), mode, float(param), S, _ptr(starts), _ptr(lo), _ptr(hi),
                                            maxeval, FTOL, GTOL, _ptr(x), _ptr(mean) if mode == 0 else None, res,
                                            ctypes.byref(best), ctypes.byref(rounds))
    elif mode == 0:
        rc = _lib.lib.hbegp_acquire_ei(h, ctypes.byref(yn._raw), float(param), S, _ptr(starts), _ptr(lo), _ptr(hi), maxeval,
                                       _ptr(x), _ptr(mean), res, ctypes.byref(best), ctypes.byref(rounds))
    else:
        rc = _lib.lib.hbegp_acquire_confidence_bound(h, ctypes.byref(yn._raw), float(param), S, _ptr(starts), _ptr(lo),
                                                     _ptr(hi), maxeval, _ptr(x), res, ctypes.byref(best), ctypes.byref(rounds))
    check(rc, "acquire")
    recs = [(r.best_value, r.best_eval, r.n_evals, r.status) for r in res[:S]]
    return x, (mean if mode == 0 else None), recs, best.value, rounds.value


def _bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def _same_records(r1, r2):
    return len(r1) == len(r2) and all(_bits(np.float64(a[0]), np.float64(b[0])) and a[1:] == b[1:] for a, b in zip(r1, r2))


def _values(model, yn, mode, param, xs):
    """hbegp_predict_mean_ei (EI) / hbegp_predict_confidence_bound (bound) of the rows, as f64."""
    from hbetune_rs_b200._lib import check, lib
    from hbetune_rs_b200.gpr import _ptr
    xs = np.ascontiguousarray(xs, dtype=yn.A)
    m = xs.shape[0]
    o1, o2 = np.empty(m, dtype=yn.A), np.empty(m, dtype=yn.A)
    if mode == 0:
        check(lib.hbegp_predict_mean_ei(model.single_handle(), ctypes.byref(yn._raw), m, _ptr(xs), float(param), _ptr(o1), _ptr(o2),
                                        None, None), "mean_ei")
        return o2.astype(np.float64), o1
    check(lib.hbegp_predict_confidence_bound(model.single_handle(), ctypes.byref(yn._raw), m, _ptr(xs), float(param), _ptr(o1),
                                             None, None), "cb")
    return o1.astype(np.float64), None


def _param(mode, yraw):
    # EI against the median of y: EI is far from negligible at most starts (with fmin = min(y) the absolute gtol ends
    # most runs at their start).  The bound: mean + 1 sd.
    return float(np.median(yraw)) if mode == 0 else 1.0


def _set_default_tolerances():
    from hbetune_rs_b200._lib import lib
    lib.hbegp_lbfgs_set_tolerances(FTOL, GTOL)


# ---------------------------------------------------------------------------------------------- bit-identity
# Every (dtype, mode, projection) with every S; nu and (n, d) rotate so that each S meets both sizes and both nus.
# S = 64 / 65 sit on both sides of the m = 64 switch between the latency and the throughput prediction paths; n = 2100
# pads its last 64-row tile.
_SIZES = [(500, 2), (2100, 8), (500, 8), (2100, 2)]
_IDENTITY = []
for _ia, _A in enumerate([np.float64, np.float32]):
    for _mode in (0, 1):
        for _proj in (0, 1):
            for _iS, _S in enumerate([1, 10, 64, 65, 200]):
                _k = _ia + 2 * _mode + _proj + _iS
                _IDENTITY.append(pytest.param(_A, _mode, _proj, _S, [0.5, 2.5][_k % 2], *_SIZES[_k % 4],
                                              id=f"{'f64' if _A == np.float64 else 'f32'}-{'ei' if _mode == 0 else 'cb'}-"
                                                 f"{'lin' if _proj == 0 else 'log'}-S{_S}-nu{[0.5, 2.5][_k % 2]}-"
                                                 f"n{_SIZES[_k % 4][0]}-d{_SIZES[_k % 4][1]}"))


@pytest.mark.gpu
@pytest.mark.parametrize("A,mode,proj,S,nu,n,d", _IDENTITY)
def test_device_search_equals_the_lbfgs_restatement(A, mode, proj, S, nu, n, d):
    """x_out, mean_out, every record, best_index and n_rounds equal the restatement built from lbfgs.h bit for bit."""
    _set_default_tolerances()
    x, yraw, yl, yn, theta = _case(A, n, d, proj)
    param = _param(mode, yraw)
    rng = np.random.default_rng(S * 7 + d)
    lo, hi = np.zeros(d), np.ones(d)
    starts = rng.random((S, d)).astype(A)
    with _ctx(A) as ctx:
        ctx.set_data(x, yl)
        model = ctx.model(theta, nu=nu)
        dev = _search(model, yn, mode, param, starts, lo, hi, 150)
        ref = _search(model, yn, mode, param, starts, lo, hi, 150, restated=True)
        model.close()
    xd, md, rd, bd, nd = dev
    xr, mr, rr, br, nr = ref
    assert any(r[3] == 0 for r in rr), "every start failed: the case checks nothing"
    assert max(r[2] for r in rr) > 1, "no start moved: the case checks nothing"
    assert _bits(xd, xr)
    if mode == 0:
        assert _bits(md, mr)
    assert _same_records(rd, rr), (rd[:3], rr[:3])
    assert (bd, nd) == (br, nr)
    print(f"S={S}: {nd} rounds, evaluations {sum(r[2] for r in rd)}, best start {bd}")


# ---------------------------------------------------------------------------------------------- properties
def _projected_gradient(model, yn, mode, param, xs, lo, hi):
    """max over free components of |objective gradient| at the rows (BoundedLbfgs's stopping measure)."""
    from tests.test_predict_grad import _acq_grad
    o1, o2, g1, g2, _ = _acq_grad(model, yn, xs, mode, param)
    g = -g2.astype(np.float64) if mode == 0 else g1.astype(np.float64)
    xs = np.asarray(xs, dtype=np.float64)
    free = ~(((xs <= lo) & (g > 0)) | ((xs >= hi) & (g < 0)))
    return np.where(free, np.abs(g), 0.0).max(axis=1)


@pytest.mark.gpu
@pytest.mark.parametrize("A", [np.float64, np.float32])
@pytest.mark.parametrize("mode", [0, 1])
def test_search_properties(A, mode):
    """n = 500, d = 4, 24 starts in [-0.25, 1.25]^4 over the box [0, 1]^4 with bounds -0.5 / 2 on one feature:
    points inside the box exactly; best values no worse than the (clamped) starts' and one strictly better; the values
    equal a fresh hbegp_predict_mean_ei / _confidence_bound of x_out (S rows) to rounding of the data type; a second
    call gives the same bits.  A start that stopped before maxeval either has a projected gradient <= gtol at its
    point, or stalled (ftol, or a line search that found no descent): a new search from its point then improves the
    value by no more than 1e-6 relative (1e-4 in f32).  The reason of each start is printed."""
    _set_default_tolerances()
    n, d, S, maxeval = 500, 4, 24, 150
    x, yraw, yl, yn, theta = _case(A, n, d, 0, seed=3)
    param = _param(mode, yraw)
    lo, hi = np.array([0.0, 0.0, -0.5, 0.0]), np.array([1.0, 1.0, 2.0, 1.0])
    starts = (np.random.default_rng(5).random((S, d)) * 1.5 - 0.25).astype(A)
    sign = 1.0 if mode == 0 else -1.0  # larger is better after the sign
    with _ctx(A) as ctx:
        ctx.set_data(x, yl)
        model = ctx.model(theta)
        xo, mo, recs, best, rounds = _search(model, yn, mode, param, starts, lo, hi, maxeval)
        again = _search(model, yn, mode, param, starts, lo, hi, maxeval)
        v0, _ = _values(model, yn, mode, param, np.clip(starts.astype(np.float64), lo, hi))
        v, mean = _values(model, yn, mode, param, xo)
        pg = _projected_gradient(model, yn, mode, param, xo, lo, hi)
        early = [i for i, r in enumerate(recs) if r[2] < maxeval]
        restart = _search(model, yn, mode, param, xo[early], lo, hi, maxeval) if early else None
        model.close()
    assert _bits(xo, again[0]) and _same_records(recs, again[2]) and (best, rounds) == again[3:]
    if mode == 0:
        assert _bits(mo, again[1])
    xo64 = xo.astype(np.float64)
    assert (xo64 >= lo).all() and (xo64 <= hi).all()
    bv = np.array([r[0] for r in recs])
    assert all(r[3] == 0 for r in recs)
    assert (sign * bv >= sign * v0).all()
    assert (sign * bv > sign * v0).any()
    eps = float(np.finfo(A).eps)
    tol = 8 * eps * np.maximum(1.0, np.abs(bv))
    assert (np.abs(v - bv) <= tol).all(), np.abs(v - bv).max()
    if mode == 0:
        assert (np.abs(mean.astype(np.float64) - mo.astype(np.float64)) <= 8 * eps * np.abs(mo.astype(np.float64))).all()
    # An f32 objective changes in steps of 2^-24 relative: two accepted steps that leave it unchanged end the run (ftol),
    # with gradients that carry f32 rounding, so a new search may still gain some hundred ulps there.
    stall_tol = 1e-6 if A == np.float64 else 1e-4
    reasons = {}
    for j, i in enumerate(early):
        if pg[i] <= GTOL:
            reasons[i] = f"gtol (projected gradient {pg[i]:.2e})"
            continue
        gain = sign * (restart[2][j][0] - bv[i])
        assert gain <= stall_tol * max(1.0, abs(bv[i])), (i, gain, pg[i])
        reasons[i] = f"stalled (projected gradient {pg[i]:.2e}, a new search gains {gain:.2e})"
    for i in range(S):
        print(f"start {i}: {recs[i][2]} evaluations, {reasons.get(i, 'maxeval')}")
    assert best == (max(i for i in range(S) if bv[i] == bv.max()) if mode == 0 else int(np.argmin(bv)))


# ---------------------------------------------------------------------------------------------- global check
@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_search_reaches_the_best_of_a_dense_grid(mode):
    """d = 2, n = 60, 64 starts on an 8 x 8 grid over [0, 1]^2: the best EI is >= the largest EI of a 201 x 201 grid
    (hbegp_predict_mean_ei), the best bound <= the grid's smallest, within 1e-9 relative.  Measured on a B200: the search
    beats the grid by 2.4e-5 relative (EI, 47 rounds) and 4.7e-6 relative (bound, 48 rounds)."""
    _set_default_tolerances()
    A, n, d = np.float64, 60, 2
    x, yraw, yl, yn, theta = _case(A, n, d, 0)
    param = _param(mode, yraw)
    g8 = (np.arange(8) + 0.5) / 8
    starts = np.array([[a, b] for a in g8 for b in g8])
    g = np.linspace(0.0, 1.0, 201)
    grid = np.array([[a, b] for a in g for b in g])
    with _ctx(A) as ctx:
        ctx.set_data(x, yl)
        model = ctx.model(theta)
        xo, _, recs, best, rounds = _search(model, yn, mode, param, starts, np.zeros(d), np.ones(d), 150)
        vg, _ = _values(model, yn, mode, param, grid)
        model.close()
    assert best >= 0
    b = recs[best][0]
    if mode == 0:
        top = vg.max()
        assert b >= top * (1 - 1e-9), (b, top)
        print(f"EI: search {b!r}, grid {top!r}, margin {(b - top) / abs(top):.3e} relative, {rounds} rounds")
    else:
        low = vg.min()
        assert b <= low + 1e-9 * abs(low), (b, low)
        print(f"bound: search {b!r}, grid {low!r}, margin {(low - b) / abs(low):.3e} relative, {rounds} rounds")


# ---------------------------------------------------------------------------------------------- edge cases
@pytest.mark.gpu
@pytest.mark.parametrize("A", [np.float64, np.float32])
def test_edge_cases(A):
    """S = 0 is a no-op; maxeval = 0 evaluates nothing (clamped starts, HBEGP_NOT_PD, best -1, 0 rounds); starts outside
    the box are clamped, with the restatement's bits; every invalid argument is HBEGP_ERR_INVALID."""
    from hbetune_rs_b200 import _lib
    from hbetune_rs_b200.gpr import _ptr
    _set_default_tolerances()
    n, d = 500, 3
    x, yraw, yl, yn, theta = _case(A, n, d, 0)
    fmin = _param(0, yraw)
    lo, hi = np.zeros(d), np.ones(d)
    starts = np.array([[-1.0, 0.5, 2.0], [0.25, 3.0, -0.5], [0.5, 0.5, 0.5]], dtype=A)
    clamped = np.clip(starts.astype(np.float64), lo, hi).astype(A)
    with _ctx(A) as ctx:
        ctx.set_data(x, yl)
        model = ctx.model(theta)
        h = model.single_handle()
        for mode in (0, 1):
            xo, _, recs, best, rounds = _search(model, yn, mode, 1.0 if mode else fmin, starts[:0], lo, hi, 150)
            assert recs == [] and best == -1 and rounds == 0
            xo, mo, recs, best, rounds = _search(model, yn, mode, 1.0 if mode else fmin, starts, lo, hi, 0)
            assert _bits(xo, clamped) and best == -1 and rounds == 0
            assert all(r[1:] == (-1, 0, 1) and math.isnan(r[0]) for r in recs)
            if mode == 0:
                assert np.isnan(mo).all()
            dev = _search(model, yn, mode, 1.0 if mode else fmin, starts, lo, hi, 150)
            ref = _search(model, yn, mode, 1.0 if mode else fmin, starts, lo, hi, 150, restated=True)
            assert _bits(dev[0], ref[0]) and _same_records(dev[2], ref[2]) and dev[3:] == ref[3:]
            assert ((dev[0] >= lo) & (dev[0] <= hi)).all() and dev[4] > 1

        INVALID = _lib.ERR_INVALID
        xo = np.empty((3, d), dtype=A)
        mo = np.empty(3, dtype=A)
        res = (_lib.AcqResult * 3)()
        best, rounds = ctypes.c_long(), ctypes.c_longlong()
        yp = ctypes.byref(yn._raw)

        def ei(model_h=h, ynp=yp, S=3, st=starts, lo_=lo, hi_=hi, maxeval=10, xo_=xo, res_=res, best_=True, rounds_=True):
            return _lib.lib.hbegp_acquire_ei(model_h, ynp, fmin, S, _ptr(st) if st is not None else None,
                                             _ptr(lo_) if lo_ is not None else None, _ptr(hi_) if hi_ is not None else None,
                                             maxeval, _ptr(xo_) if xo_ is not None else None, _ptr(mo), res_,
                                             ctypes.byref(best) if best_ else None, ctypes.byref(rounds) if rounds_ else None)

        def cb(model_h=h, ynp=yp, S=3, st=starts, lo_=lo, hi_=hi, maxeval=10, xo_=xo, res_=res, best_=True, rounds_=True):
            return _lib.lib.hbegp_acquire_confidence_bound(model_h, ynp, 1.0, S, _ptr(st) if st is not None else None,
                                                           _ptr(lo_) if lo_ is not None else None,
                                                           _ptr(hi_) if hi_ is not None else None, maxeval,
                                                           _ptr(xo_) if xo_ is not None else None, res_,
                                                           ctypes.byref(best) if best_ else None,
                                                           ctypes.byref(rounds) if rounds_ else None)

        bad_start = starts.copy()
        bad_start[1, 2] = np.nan
        inf_start = starts.copy()
        inf_start[0, 0] = np.inf
        for call in (ei, cb):
            assert call() == 0
            assert call(model_h=None) == INVALID
            assert call(ynp=None) == INVALID
            assert call(st=None) == INVALID
            assert call(lo_=None) == INVALID
            assert call(hi_=None) == INVALID
            assert call(xo_=None) == INVALID
            assert call(res_=None) == INVALID
            assert call(best_=False) == INVALID
            assert call(rounds_=False) == INVALID
            assert call(S=-1) == INVALID
            assert call(maxeval=-1) == INVALID
            assert call(st=bad_start) == INVALID
            assert call(st=inf_start) == INVALID
            assert call(lo_=np.array([0.0, -np.inf, 0.0])) == INVALID
            assert call(hi_=np.array([1.0, 1.0, np.nan])) == INVALID
            assert call(lo_=np.array([0.0, 0.6, 0.0]), hi_=np.array([1.0, 0.5, 1.0])) == INVALID
        model.close()


@pytest.mark.gpu
@pytest.mark.parametrize("A", [np.float64, np.float32])
def test_all_nan_ei(A):
    """Log projection with fmin <= expected: EI is NaN everywhere, so every start ends after its first evaluation with
    HBEGP_NOT_PD, the best index is -1, and x_out holds the (clamped) starts."""
    _set_default_tolerances()
    n, d = 500, 2
    x, yraw, yl, yn, theta = _case(A, n, d, 1)
    fmin = float(yn.expected) - 0.5
    starts = np.random.default_rng(2).random((12, d)).astype(A)
    with _ctx(A) as ctx:
        ctx.set_data(x, yl)
        model = ctx.model(theta)
        xo, mo, recs, best, rounds = _search(model, yn, 0, fmin, starts, np.zeros(d), np.ones(d), 150)
        model.close()
    assert all(r[1:] == (-1, 1, 1) and math.isnan(r[0]) for r in recs)
    assert best == -1 and rounds == 1 and _bits(xo, starts) and np.isnan(mo).all()


@pytest.mark.gpu
def test_evicted_model_and_warn_list():
    """A search on an evicted model (resident limit 1) rebuilds it and gives the bits of the search before eviction; the
    warn list of the preceding hbegp_predict is the same after a search."""
    from hbetune_rs_b200.estimator import YNormalize
    from tests.util import synth
    _set_default_tolerances()
    A, n, d = np.float64, 500, 3
    x, yraw, yl, yn, theta = _case(A, n, d, 0)
    fmin = _param(0, yraw)
    starts = np.random.default_rng(4).random((20, d))
    lo, hi = np.zeros(d), np.ones(d)
    with _ctx(A) as ctx:
        ctx.set_resident_models(1)
        ctx.set_data(x, yl)
        m1 = ctx.model(theta)
        before = [_search(m1, yn, mode, 1.0 if mode else fmin, starts, lo, hi, 150) for mode in (0, 1)]
        m2 = ctx.model(theta + np.array([0.0, 0.1] + [0.0] * d))  # evicts m1
        st0 = ctx.model_stats()
        after = [_search(m1, yn, mode, 1.0 if mode else fmin, starts, lo, hi, 150) for mode in (0, 1)]
        st1 = ctx.model_stats()
        m1.close()
        m2.close()
    assert st0["evictions"] >= 1 and st1["rebuilds"] > st0["rebuilds"]
    for b, a in zip(before, after):
        assert _bits(b[0], a[0]) and _same_records(b[2], a[2]) and b[3:] == a[3:]
        if b[1] is not None:
            assert _bits(b[1], a[1])

    # a model whose predicted variances go below -sqrt(1e-5) (a huge amplitude): the reference warns about them
    xw, yw = synth(120, 2)
    thw = np.array([math.log(1e-2), math.log(1e14), math.log(2.0), math.log(2.0)])
    xs = np.concatenate([xw[:60], np.random.default_rng(1).random((40, 2))])
    ylw, ynw = YNormalize.new_project_into_normalized(yw + 5.0, 0)
    with _ctx(A) as ctx:
        ctx.set_data(xw, yw)
        model = ctx.model(thw)
        model.predict(xs, warn=False)
        w0 = model.warn_values(cap=4096)
        assert len(w0[0]) > 0
        _search(model, ynw, 1, 1.0, xs[:10], np.zeros(2), np.ones(2), 20)
        _search(model, ynw, 0, float(np.median(yw + 5.0)), xs[:10], np.zeros(2), np.ones(2), 20)
        w1 = model.warn_values(cap=4096)
        model.close()
    assert _bits(np.asarray(w0[0]), np.asarray(w1[0])) and _bits(np.asarray(w0[1]), np.asarray(w1[1]))


@pytest.mark.gpu
def test_estimator_methods():
    """SurrogateModelGPR.acquire_ei / acquire_confidence_bound return the device search's arrays and records."""
    import hbetune_rs_b200 as h
    from hbetune_rs_b200.estimator import EstimatorGPR
    from oracle.rng import RNG
    from tests.util import synth
    _set_default_tolerances()
    n, d = 200, 3
    x, y = synth(n, d)
    with h.Context(0, h.F64) as ctx:
        est = EstimatorGPR(d, ctx=ctx)
        model = est.estimate(x, y + 5.0, None, RNG.new_with_seed(3))
        starts = np.random.default_rng(6).random((16, d))
        fmin = float(np.median(y + 5.0))
        xo, mean, recs, best, rounds = model.acquire_ei(starts, 0.0, 1.0, fmin)
        dev = _search(model.fitted.model, model.y_norm, 0, fmin, starts, np.zeros(d), np.ones(d), 150)
        xc, recc, bestc, roundsc = model.acquire_confidence_bound(starts, 0.0, 1.0, 1.0, maxeval=50)
        devc = _search(model.fitted.model, model.y_norm, 1, 1.0, starts, np.zeros(d), np.ones(d), 50)
        ei_best = model.predict_mean_ei_device(xo[best:best + 1], fmin)[1][0]
    assert _bits(xo, dev[0]) and _bits(mean, dev[1]) and (best, rounds) == dev[3:]
    assert _same_records([(r.best_value, r.best_eval, r.n_evals, r.status) for r in recs], dev[2])
    assert _bits(xc, devc[0]) and (bestc, roundsc) == devc[3:]
    assert abs(ei_best - recs[best].best_value) <= 1e-12 * abs(ei_best)
