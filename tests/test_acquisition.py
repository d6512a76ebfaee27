"""The device acquisition (k_acquisition's EI, confidence bound and de-normalisation; the arg-best pick of
launch_argbest) against an exact truth, on every prediction path and arg-best partition.

EI = -(mu - f) Phi(z) + sigma phi(z), z = -(mu - f) / sigma, is restated in mpmath at 60 digits (`_ei_exact`), and
every f64 evaluation must satisfy

    |EI - EI*| <= F eps S + F 2^-1074 (1 + |delta| + sigma),     S = (|delta| Phi(z) + sigma phi(z)) (2 + z^2),

with delta = f - mu and eps = 2^-53.  F comes from the documented maximum errors, not from measurements: erfc 5 ulps
and exp 1 ulp (the CUDA math library's table; glibc's is no larger), i.e. 10 eps and 2 eps relative.  Term by term:
- delta Phi(z): delta and the product round (2 eps), erfc (10 eps), and the argument -z / sqrt 2 carries 4 eps
  relative error (the subtraction is in delta, then the division, the constant and the product); it moves Phi by
  phi |z| 4 eps <= Phi (|z| + 1) |z| 4 eps <= Phi (6 z^2 + 2) eps (Mills' ratio phi / Phi <= |z| + 1 for z < 0).
  Together (14 + 6 z^2) eps <= 7 (2 + z^2) eps of the term.
- sigma phi(z): exp (2 eps), two constants and two products (4 eps), and the argument z^2 / 2 with 6 eps relative
  error, 3 eps z^2 absolute: (6 + 3 z^2) eps <= 4 (2 + z^2) eps of the term.
- the final sum adds eps |EI| <= eps (|delta| Phi + sigma phi).
So F = 8 covers both the device (erfc(-z * 1/sqrt 2)) and the host (erfc(-z / sqrt 2)).  The z^2 is erfc's
conditioning in the tail, where the two terms cancel.  The second term covers underflow: for |z| > 38.6, phi and Phi
are subnormal or 0, with an absolute error of a few 2^-1074, and products and sums that land among the subnormals
round to an absolute 2^-1075 each.

The std-zero branch (sigma <= 2^-52, `ei_std_is_zero`) is held bit for bit.  The library's EI is NaN exactly where the
host `hbegp_expected_improvement` is.  The arg-best rules (EI: the last maximum; confidence bound: the first minimum;
NaN never wins; -0 == +0) are restated in NumPy, and the partition is restated from the launcher's constants.

Engine tests feed `hbegp_predict_mean_ei` / `hbegp_predict_confidence_bound` candidates on, next to and away from
training points, and check that they equal, bit for bit, tests/cuda/libacq_harness.so's epilogue applied to
`hbegp_predict`'s mean and variance; in f64 also against test_f64_truth's posterior truth.
"""
import ctypes
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests.test_dispatch_sweep import _ctx, _kernel_f64, _note, _np, _predict_path, _reference, _rounded
from tests.test_f64_truth import EPS, R, F, _candidates, _gpu_k, _predict_star, _truth_of
from tests.util import random_thetas, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hbetune_rs_b200", "csrc")
HARNESS = os.path.join(ROOT, "tests", "cuda", "libacq_harness.so")

F_EI = 8.0             # see the module docstring
TINY = 2.0 ** -1074    # the subnormal quantum
STD_ZERO = 2.0 ** -52  # ei_std_is_zero: sigma <= f64::EPSILON
PHI0 = 0.4             # >= phi(0) = 0.3989..., the largest |dEI / dsigma|
# documented maximum ulp errors of exp (CUDA: exp 1 ulp, expf 2 ulps)
ULP_EXP = {np.float64: 1.0, np.float32: 2.0}
# launch_argbest's plan (kernels.cuh): at most 1024 parts, 256 threads per part
PARTS, THREADS = 1024, 256


def _name(A):
    return "f64" if A == np.float64 else "f32"


# ------------------------------------------------------------------------------------------------ the exact EI


def _ei_mp(mu, sd, f):
    """EI as an mpf, at the working precision (the caller's workdps)."""
    import mpmath
    mu, sd, f = mpmath.mpf(mu), mpmath.mpf(sd), mpmath.mpf(f)
    if sd <= STD_ZERO:
        return max(f - mu, mpmath.mpf(0))
    z = (f - mu) / sd
    cdf = mpmath.erfc(-z / mpmath.sqrt(2)) / 2
    pdf = mpmath.exp(-z * z / 2) / mpmath.sqrt(2 * mpmath.pi)
    return (f - mu) * cdf + sd * pdf


def _ei_exact(mu, sd, f):
    """EI(mu, sd, f) at 60 digits, rounded to f64, elementwise (f may be a scalar)."""
    import mpmath
    mu, sd = np.atleast_1d(np.asarray(mu, np.float64)), np.atleast_1d(np.asarray(sd, np.float64))
    f = np.broadcast_to(np.asarray(f, np.float64), mu.shape)
    out = np.empty(mu.shape)
    with mpmath.workdps(60):
        for i in range(mu.size):
            out.flat[i] = float(_ei_mp(float(mu.flat[i]), float(sd.flat[i]), float(f.flat[i])))
    return out


def _ei_bound(mu, sd, f):
    """F eps S + F 2^-1074 (1 + |delta| + sigma) at the inputs (mu, sd, f), elementwise."""
    from scipy.special import erfc
    mu, sd = np.asarray(mu, np.float64), np.asarray(sd, np.float64)
    delta = f - mu
    with np.errstate(divide="ignore", invalid="ignore", over="ignore", under="ignore"):
        z = np.where(sd > 0, delta / np.where(sd > 0, sd, 1.0), 0.0)
        cdf = 0.5 * erfc(-z / math.sqrt(2.0))
        pdf = np.exp(-0.5 * z * z) / math.sqrt(2.0 * math.pi)
        s = (np.abs(delta) * cdf + sd * pdf) * (2.0 + z * z)
    return F_EI * EPS * s + F_EI * TINY * (1.0 + np.abs(delta) + sd)


def _ratio(err, bound):
    """err / bound, 0 where both are 0 (an exact 0 whose bound underflows)."""
    err, bound = np.asarray(err, np.float64), np.asarray(bound, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(err == 0, 0.0, err / bound)


def test_exact_ei_satisfies_the_reflection_identity():
    """EI(delta) - EI(-delta) = delta, delta = f - mu, at 60 digits (the std-zero branch included)."""
    import mpmath
    rng = np.random.default_rng(1)
    with mpmath.workdps(60):
        for sd in (0.0, STD_ZERO, 1e-9, 0.3, 1.0, 40.0):
            for z in np.concatenate([rng.uniform(-40, 40, 20), [0.0, -38.9, 38.9]]):
                f = mpmath.mpf(0.25)
                delta = mpmath.mpf(float(z)) * (sd if sd > 0 else 1.0)
                lhs = _ei_mp(f - delta, sd, f) - _ei_mp(f + delta, sd, f)
                assert abs(lhs - delta) <= mpmath.mpf(10) ** -55 * (abs(delta) + sd), (sd, z)


def test_exact_ei_follows_the_tail_asymptote():
    """EI -> sigma phi(z) / z^2 (1 - 3 / z^2 + ...) as z -> -inf: the ratio lies in [1 - 3 / z^2, 1]."""
    import mpmath
    with mpmath.workdps(60):
        prev = None
        for z in (-5, -10, -20, -40, -80):
            sd, f = mpmath.mpf(1.7), mpmath.mpf(-0.5)
            ei = _ei_mp(f - z * sd, sd, f)
            asym = sd * mpmath.exp(-mpmath.mpf(z) ** 2 / 2) / mpmath.sqrt(2 * mpmath.pi) / z ** 2
            ratio = ei / asym
            assert 1 - mpmath.mpf(3) / z ** 2 <= ratio <= 1, (z, ratio)
            if prev is not None:
                assert abs(1 - ratio) < abs(1 - prev)
            prev = ratio


def _host_ei():
    import hbetune_rs_b200 as h
    from hbetune_rs_b200._lib import lib
    assert h is not None
    return lib.hbegp_expected_improvement


def test_host_ei_within_the_stated_bound():
    """hbegp_expected_improvement against _ei_exact at z in [-40, 40] (phi underflows beyond 38.6) and sigma from
    3e-16 to 1e6; the std-zero branch, subnormal sigma included, bit for bit."""
    ei = _host_ei()
    zs = np.concatenate([np.linspace(-40, 40, 161), [-38.7, 38.7, -1e-3, 1e-3]])
    worst = 0.0
    for sd in (3e-16, 1e-8, 0.37, 1.0, 13.0, 1e6):
        for f in (0.0, 0.41, -2.5):
            mu = f - zs * sd
            got = np.array([ei(float(a), sd, f) for a in mu])
            want = _ei_exact(mu, np.full_like(mu, sd), f)
            r = _ratio(np.abs(got - want), _ei_bound(mu, np.full_like(mu, sd), f))
            worst = max(worst, float(r.max()))
            assert (r <= 1.0).all(), (sd, f, zs[r.argmax()], got[r.argmax()], want[r.argmax()])
    for sd in (0.0, -0.0, 5e-324, 1e-310, STD_ZERO):
        for mu, f in ((0.3, 0.7), (0.7, 0.3), (0.5, 0.5), (-1e300, 1e300)):
            want = -(mu - f) if mu < f else 0.0
            assert np.float64(ei(mu, sd, f)).view(np.int64) == np.float64(want).view(np.int64), (mu, sd, f)
    assert ei(0.3, np.nextafter(STD_ZERO, 1.0), 0.7) == pytest.approx(0.4, abs=1e-15)
    _note("acquisition host EI", {"max err/bound": worst})


def test_host_ei_is_nan_on_every_non_finite_input():
    ei = _host_ei()
    vals = (math.nan, math.inf, -math.inf, 0.25)
    for mu in vals:
        for sd in vals + (0.0,):
            for f in vals:
                finite = all(math.isfinite(v) for v in (mu, sd, f))
                assert math.isnan(ei(mu, sd, f)) != finite, (mu, sd, f)


# ------------------------------------------------------------------------------------------------ the selection rules


def _argbest_rule(key, want_max):
    """EI: the last maximum wins (max_by); confidence bound: the first minimum wins (strict <); NaN never wins, all
    NaN gives -1; -0 and +0 tie."""
    k = np.asarray(key, dtype=np.float64)
    ok = ~np.isnan(k)
    if not ok.any():
        return -1
    v = k[ok].max() if want_max else k[ok].min()
    hit = np.flatnonzero(ok & (k == v))
    return int(hit[-1] if want_max else hit[0])


def _argbest_sequential(key, want_max):
    best, bi = None, -1
    for i, x in enumerate(key):
        if x != x:
            continue
        if bi < 0 or (x >= best if want_max else x < best):
            best, bi = x, i
    return bi


def test_selection_rules_restated():
    rng = np.random.default_rng(3)
    pool = np.array([-math.inf, -1.0, -0.0, 0.0, 1.0, math.inf, math.nan])
    for _ in range(3000):
        key = rng.choice(pool, size=int(rng.integers(1, 12)))
        for want_max in (True, False):
            assert _argbest_rule(key, want_max) == _argbest_sequential(key.tolist(), want_max), (key, want_max)
    assert _argbest_rule([math.nan] * 5, True) == -1 and _argbest_rule([math.nan], False) == -1
    assert _argbest_rule([0.0, -0.0, 0.0, -0.0], True) == 3 and _argbest_rule([-0.0, 0.0], False) == 0
    assert _argbest_rule([1.0, math.nan, 1.0], True) == 2 and _argbest_rule([1.0, math.nan, 1.0], False) == 0


def _plan(m):
    """launch_argbest's partition: (lo, hi) of every part."""
    nparts = max(1, min(PARTS, -(-m // THREADS)))
    chunk = -(-m // nparts)
    return [(min(m, p * chunk), min(m, p * chunk + chunk)) for p in range(nparts)]


def _cases(m):
    parts = _plan(m)
    chunk = parts[0][1] - parts[0][0]
    out = set()
    if len(parts) == 1:
        out.add("1 part")
    elif chunk <= THREADS:
        out.add("several parts, chunk <= 256")
    if len(parts) == PARTS and chunk > THREADS:
        out.add("1024 parts, several elements per thread")
    if any(lo == hi for lo, hi in parts):
        out.add("empty trailing parts")
    if m > 2 ** 31:
        out.add("m > 2^31")
    return out


M_GPU = [1, 200, 256, 257, 70001, 262144, 262145, 1000003, 1 << 24]
M_HUGE = 2 ** 31 + 3


def test_planned_sizes_reach_every_partition_case():
    reached = set().union(*(_cases(m) for m in M_GPU + [M_HUGE]))
    assert reached == {"1 part", "several parts, chunk <= 256", "1024 parts, several elements per thread",
                       "empty trailing parts", "m > 2^31"}, reached
    parts = _plan(262145)
    assert parts[0] == (0, 257) and [p for p, (lo, hi) in enumerate(parts) if lo == hi] == [1021, 1022, 1023]
    for m in M_GPU + [M_HUGE, 2, 255, 65536]:
        parts = _plan(m)
        assert parts[0][0] == 0 and parts[-1][1] == m
        assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))


def test_harness_builds_without_a_gpu():
    lib = _harness()
    for m in M_GPU + [M_HUGE, 2, 255, 65536]:
        assert lib.acq_argbest_parts(m) == len(_plan(m)), m
        assert lib.acq_argbest_ws_bytes(m) == 16 * len(_plan(m))


# ------------------------------------------------------------------------------------------------ the harness


def _harness():
    if not os.path.exists(HARNESS):
        nvcc = shutil.which("nvcc") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
        subprocess.run(["make", "-C", CSRC, f"NVCC={nvcc}", "../../tests/cuda/libacq_harness.so"], check=True)
    lib = ctypes.CDLL(HARNESS)
    lib.acq_argbest_parts.restype, lib.acq_argbest_parts.argtypes = ctypes.c_int, [ctypes.c_long]
    lib.acq_argbest_ws_bytes.restype, lib.acq_argbest_ws_bytes.argtypes = ctypes.c_size_t, [ctypes.c_long]
    lib.acq_epilogue.restype = ctypes.c_int
    lib.acq_epilogue.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long, ctypes.c_int, ctypes.c_int,
                                 ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_void_p,
                                 ctypes.c_void_p, ctypes.c_void_p]
    lib.acq_argbest.restype = ctypes.c_int
    lib.acq_argbest.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_long, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                ctypes.c_void_p]
    return lib


def _epilogue(mean, var, mode, proj=0, amplitude=1.0, expected=0.0, fmin_n=0.0, cb=0.0):
    """k_acquisition on device copies of mean and var (host arrays of one dtype); returns (out1, out2) on the host."""
    import torch
    lib = _harness()
    A = mean.dtype.type
    mu = torch.from_numpy(np.ascontiguousarray(mean)).cuda()
    va = torch.from_numpy(np.ascontiguousarray(var, dtype=A)).cuda()
    o1, o2 = torch.full_like(mu, math.nan), torch.full_like(mu, math.nan)
    rc = lib.acq_epilogue(0 if A == np.float64 else 1, mu.data_ptr(), va.data_ptr(), mu.numel(), mode, proj,
                          float(amplitude), float(expected), float(fmin_n), float(cb), o1.data_ptr(), o2.data_ptr(),
                          torch.cuda.current_stream().cuda_stream)
    assert rc == 0, f"k_acquisition: cudaError {rc}"
    torch.cuda.synchronize()
    return o1.cpu().numpy(), o2.cpu().numpy()


def _argbest_dev(key, want_max):
    """launch_argbest on a torch CUDA tensor; the workspace is filled with 0xFF first."""
    import torch
    lib = _harness()
    m = key.numel()
    ws = torch.full((lib.acq_argbest_ws_bytes(m),), 0xFF, dtype=torch.uint8, device="cuda")
    out = torch.full((1,), -7, dtype=torch.int64, device="cuda")
    rc = lib.acq_argbest(0 if key.dtype == torch.float64 else 1, key.data_ptr(), m, int(want_max), ws.data_ptr(),
                         out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert rc == 0, f"launch_argbest: cudaError {rc}"
    return int(out.item())


def _bits_equal(got, want):
    got, want = np.asarray(got), np.asarray(want, dtype=np.asarray(got).dtype)
    iv = np.int64 if got.dtype == np.float64 else np.int32
    return got.view(iv) == want.view(iv)


def _half_ulp32(x):
    return 0.5 * np.spacing(np.abs(np.asarray(x, dtype=np.float64)).astype(np.float32)).astype(np.float64)


def _ei_grid(A):
    """(mean, var, f) in the data type A: z in [-40, 40] at sigma from 1e-7 to 1e6, and the std-zero edges: sigma =
    2^-52 exactly and the next representable sigma above it, var = 0, subnormal var (sigma >= 1e-162 in f64; sigma
    = sqrt(var) cannot be subnormal)."""
    f = 0.41
    zs = np.concatenate([np.linspace(-40, 40, 161), [-38.7, 38.7]])
    mus, vars_ = [], []
    for sd in (1e-7, 0.37, 1.0, 13.0, 1e6):
        mus.append(f - zs * sd)
        vars_.append(np.full(zs.size, sd * sd))
    v = A(2.0 ** -104)
    assert np.sqrt(v) == A(STD_ZERO)
    above = v
    while np.sqrt(above) == A(STD_ZERO):
        above = np.nextafter(above, A(1))
    assert np.sqrt(above) == np.nextafter(A(STD_ZERO), A(1))
    tiny = np.finfo(A).smallest_subnormal
    edge_z = np.array([-3.0, -0.5, 0.0, 0.5, 3.0])
    for var in (v, above):
        s = float(np.sqrt(var))
        mus.append(f - edge_z * s)
        vars_.append(np.full(edge_z.size, var))
    for var in (0.0, -0.0, tiny, 3 * tiny):
        mus.append(np.array([f - 1.0, f - 1e-9, f, f + 1e-9, f + 1.0]))
        vars_.append(np.full(5, var))
    return np.concatenate(mus).astype(A), np.concatenate(vars_).astype(A), f


@pytest.mark.gpu
@pytest.mark.parametrize("A", [np.float64, np.float32])
def test_ei_grid_against_the_exact_value(A):
    mean, var, f = _ei_grid(A)
    _, ei = _epilogue(mean, var, 0, fmin_n=f)
    sd = np.sqrt(var).astype(np.float64)  # sqrt / sqrtf round correctly, like the kernel's
    mu = mean.astype(np.float64)
    zero = sd <= STD_ZERO
    want0 = np.where(mu < f, -(mu - f), 0.0).astype(A)
    assert _bits_equal(ei[zero], want0[zero]).all(), (mu[zero], sd[zero], ei[zero], want0[zero])
    exact = _ei_exact(mu[~zero], sd[~zero], f)
    bound = _ei_bound(mu[~zero], sd[~zero], f)
    if A == np.float32:
        bound = bound + _half_ulp32(exact)
    r = _ratio(np.abs(ei[~zero].astype(np.float64) - exact), bound)
    z = (f - mu[~zero]) / sd[~zero]
    assert np.abs(z).max() >= 38.7 and (sd == float(np.nextafter(A(STD_ZERO), A(1)))).any() and (sd == STD_ZERO).any()
    _note(f"acquisition EI grid {_name(A)}", {"max err/bound": float(r.max()), "rows": int(mean.size),
                                               "std-zero rows": int(zero.sum())})
    assert (r <= 1.0).all(), (z[r.argmax()], sd[~zero][r.argmax()], ei[~zero][r.argmax()], exact[r.argmax()])


def _ynorm(A, proj, amplitude, expected):
    from hbetune_rs_b200 import _lib
    from hbetune_rs_b200.estimator import YNormalize
    raw = _lib.YNorm()
    raw.amplitude, raw.expected, raw.projection = float(A(amplitude)), float(A(expected)), proj
    raw.dtype = _lib.F64 if A == np.float64 else _lib.F32
    return YNormalize(raw, A)


@pytest.mark.gpu
@pytest.mark.parametrize("A", [np.float64, np.float32])
def test_linear_projection_is_the_host_ynorm_bit_for_bit(A):
    """mode 0 mean and mode 1 bound = hbegp_ynorm_apply op 1 of mu and of mu + sqrt(var) cb, unfused."""
    rng = np.random.default_rng(7)
    m = 20000
    mean = rng.normal(0.3, 2.0, m).astype(A)
    var = (rng.random(m) ** 4 * 3).astype(A)
    var[:50] = 0
    for amp, exp_ in ((3.7, -1.3), (0.01234567, 1234.5678)):
        yn = _ynorm(A, 0, amp, exp_)
        o1, _ = _epilogue(mean, var, 0, 0, yn.amplitude, yn.expected, 0.2)
        assert _bits_equal(o1, yn.project_location_from_normalized(mean)).all()
        for cb in (1.5, -2.0):
            o1, _ = _epilogue(mean, var, 1, 0, yn.amplitude, yn.expected, cb=cb)
            y = mean + np.sqrt(var) * A(cb)  # NumPy rounds each operation
            assert _bits_equal(o1, yn.project_location_from_normalized(y)).all(), cb


@pytest.mark.gpu
@pytest.mark.parametrize("A", [np.float64, np.float32])
def test_log_projection_within_the_exp_bound(A):
    """exp(fl(y amp)) + expected: within ULP_EXP ulps of exp plus the final rounding of the exact value."""
    import mpmath
    rng = np.random.default_rng(8)
    m = 2000
    mean = rng.normal(0.0, 1.5, m).astype(A)
    var = (rng.random(m) * 2).astype(A)
    worst = 0.0
    for amp, exp_ in ((1.9, -3.25), (4.5, 100.0)):  # |y amp| < 50: no overflow in f32
        yn = _ynorm(A, 1, amp, exp_)
        for mode, cb in ((0, 0.0), (1, -1.5)):
            o1, _ = _epilogue(mean, var, mode, 1, yn.amplitude, yn.expected, 0.1, cb)
            y = mean if mode == 0 else mean + np.sqrt(var) * A(cb)
            p = (y * A(yn.amplitude)).astype(np.float64)
            with mpmath.workdps(40):
                e = [mpmath.exp(mpmath.mpf(float(v))) for v in p]
                err = np.array([float(abs(mpmath.mpf(float(g)) - v - mpmath.mpf(yn.expected))) for g, v in zip(o1, e)])
                e = np.array([float(v) for v in e])
            bound = ULP_EXP[A] * np.spacing(e.astype(A)).astype(np.float64) + \
                0.5 * np.spacing(np.abs(o1)).astype(np.float64)
            r = _ratio(err, bound)
            worst = max(worst, float(r.max()))
            assert (r <= 1.0).all(), (mode, amp, p[r.argmax()], o1[r.argmax()], err[r.argmax()])
    _note(f"acquisition log projection {_name(A)}", {"max err/bound": worst})


@pytest.mark.gpu
@pytest.mark.parametrize("A", [np.float64, np.float32])
def test_ei_is_nan_exactly_where_the_host_ei_is(A):
    """NaN or +-inf in the mean, the variance (var = 0 and var > 0 too) and fmin_n: EI is NaN where
    hbegp_expected_improvement is, and only there; before the finiteness test the std-zero branch answered 0 or
    -(mu - f) for a non-finite fmin_n."""
    ei = _host_ei()
    vals = [math.nan, math.inf, -math.inf, 0.2]
    mean = np.array([a for a in vals for _ in range(6)], dtype=A)
    var = np.array([0.0, 0.25, math.nan, math.inf, -math.inf, -1.0] * len(vals), dtype=A)
    with np.errstate(invalid="ignore"):
        sd = np.sqrt(var).astype(np.float64)
    for f in vals:
        _, got = _epilogue(mean, var, 0, fmin_n=f)
        want = np.array([ei(float(a), float(s), f) for a, s in zip(mean, sd)])
        assert (np.isnan(got) == np.isnan(want)).all(), (f, mean, var, got, want)
        assert np.isfinite(got[~np.isnan(want)]).all()


def _plant(m, kind, dev, dtype, rng_seed):
    """A key vector (max direction) on the device: random values in [0, 1) with the winner planted by `kind`."""
    import torch
    g = torch.Generator(device=dev).manual_seed(rng_seed)
    key = torch.rand(m, generator=g, device=dev, dtype=dtype)
    parts = [(lo, hi) for lo, hi in _plan(m) if hi > lo]
    if kind == "part edges":
        idx = torch.tensor(sorted({i for lo, hi in parts for i in (lo, hi - 1)}), device=dev)
        key[idx] = 2.0
    elif kind == "stride 256":
        lo, hi = parts[len(parts) // 2]
        assert hi - lo > THREADS + 5
        key[lo + 5] = key[lo + 5 + THREADS] = 2.0
    elif kind == "adjacent":
        i = (m - 1) // 2
        key[i] = 2.0
        if i + 1 < m:
            key[i + 1] = 2.0
    elif kind == "signed zeros":
        key = -1.0 - key
        idx = torch.randperm(m, generator=g, device=dev)[:7]
        key[idx] = 0.0
        key[idx[::2]] = -0.0
    elif kind == "infinities":
        idx = torch.randperm(m, generator=g, device=dev)[:9]
        key[idx[:3]] = math.inf
        key[idx[3:]] = -math.inf
    elif kind == "one non-NaN":
        j = int(torch.randint(m, (1,), generator=g, device=dev).item())
        key.fill_(math.nan)
        key[j] = -5.0
    elif kind == "all NaN":
        key.fill_(math.nan)
    return key


@pytest.mark.gpu
@pytest.mark.parametrize("A", [np.float64, np.float32])
@pytest.mark.parametrize("m", M_GPU)
def test_argbest_on_planted_keys(m, A):
    """Every plant in both directions (the minimum on the negated keys) against the restated rule."""
    import torch
    dtype = torch.float64 if A == np.float64 else torch.float32
    kinds = ["part edges", "adjacent", "signed zeros", "infinities", "one non-NaN", "all NaN"]
    if _plan(m)[0][1] > THREADS + 5:
        kinds.append("stride 256")
    for s, kind in enumerate(kinds):
        key = _plant(m, kind, "cuda", dtype, 1000 * m + s)
        for want_max in (True, False):
            k = key if want_max else -key
            want = _argbest_rule(k.cpu().numpy(), want_max)
            got = _argbest_dev(k, want_max)
            assert got == want, (m, kind, want_max, got, want)
            if kind == "all NaN":
                assert got == -1


@pytest.mark.gpu
def test_argbest_beyond_2_31_elements():
    """m = 2^31 + 3 in f32 (8.6 GB): the winner beyond 2^31 against an equal key at index 0, and a tie of every
    element; by construction."""
    import torch
    m = M_HUGE
    free, _ = torch.cuda.mem_get_info()
    if free < 4 * m + (1 << 30):
        pytest.skip(f"needs {4 * m / 1e9:.1f} GB of free device memory")
    w = 2 ** 31 + 1
    key = torch.zeros(m, dtype=torch.float32, device="cuda")
    assert _argbest_dev(key, True) == m - 1 and _argbest_dev(key, False) == 0
    key[0] = key[w] = 1.0
    assert _argbest_dev(key, True) == w
    key.zero_()
    key[0] = -0.5
    key[w] = key[w + 1] = -1.0
    assert _argbest_dev(key, False) == w
    key[w] = math.nan
    assert _argbest_dev(key, False) == w + 1
    del key
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ the engine


def _acq(model, yn, xs, mode, param):
    """hbegp_predict_mean_ei (mode 0, param = fmin) or hbegp_predict_confidence_bound (mode 1, param = cb)."""
    from hbetune_rs_b200._lib import check, lib
    from hbetune_rs_b200.gpr import _ptr
    A = yn.A
    xs = np.ascontiguousarray(xs, dtype=A)
    m = xs.shape[0]
    out1, out2 = np.full(m, np.nan, dtype=A), np.full(m, np.nan, dtype=A)
    best, nb = ctypes.c_long(-7), ctypes.c_long(-7)
    if mode == 0:
        check(lib.hbegp_predict_mean_ei(model.single_handle(), ctypes.byref(yn._raw), m, _ptr(xs), float(param),
                                        _ptr(out1), _ptr(out2), ctypes.byref(best), ctypes.byref(nb)), "predict_mean_ei")
    else:
        check(lib.hbegp_predict_confidence_bound(model.single_handle(), ctypes.byref(yn._raw), m, _ptr(xs), float(param),
                                                 _ptr(out1), ctypes.byref(best), ctypes.byref(nb)), "predict_cb")
    return out1, (out2 if mode == 0 else None), best.value, nb.value


def _wired(model, yn, xs, mode, param):
    """The harness epilogue on hbegp_predict's mean and variance of the same rows, with fmin projected as the library
    does (in the data type)."""
    mean, var = model.predict(np.ascontiguousarray(xs, dtype=yn.A), warn=False)
    fmin_n = float(yn.project_into_normalized(np.array([param]))[0]) if mode == 0 else 0.0
    o1, o2 = _epilogue(mean, var, mode, yn.projection, yn.amplitude, yn.expected, fmin_n, param if mode == 1 else 0.0)
    return o1, (o2 if mode == 0 else None), mean, var, fmin_n


def _assert_wired(model, yn, xs, mode, param, tag):
    got1, got2, best, _ = _acq(model, yn, xs, mode, param)
    w1, w2, mean, var, fmin_n = _wired(model, yn, xs, mode, param)
    assert _bits_equal(got1, w1).all(), (tag, "out1", np.flatnonzero(~_bits_equal(got1, w1))[:5])
    if mode == 0:
        assert _bits_equal(got2, w2).all(), (tag, "ei", np.flatnonzero(~_bits_equal(got2, w2))[:5])
    assert best == _argbest_rule(got2 if mode == 0 else got1, mode == 0), (tag, best)
    return got1, got2, best, mean, var, fmin_n


NOISE = {np.float64: 1e-4, np.float32: 1e-2}
CB = -1.5


def _fmins(yn, y, mean, var):
    """min(y); one below every mean (the far tail: z <= -6 at the median sigma, below -38 where EI underflows at the
    smallest); one above every mean; in natural units."""
    sd = np.sqrt(var.astype(np.float64))
    lo = float(mean.min()) - 6.0 * max(float(np.median(sd)), 1e-3)
    hi = float(mean.max()) + 3.0 * max(float(sd.max()), 1e-3)
    nat = yn.project_location_from_normalized(np.array([lo, hi]))
    return {"min(y)": float(y.min()), "below": float(nat[0]), "above": float(nat[1])}


def _model_case(A, n, d=3):
    """Training data, its linear normalisation (the model's y), both YNormalize records and theta."""
    from hbetune_rs_b200.estimator import LINEAR, LOGARITHMIC, YNormalize
    x, yraw = synth(n, d, seed=n + 1, A=A)
    yraw = (yraw * A(3) + A(10)).astype(A)
    yl, ynl = YNormalize.new_project_into_normalized(yraw, LINEAR, A=A)
    _, ynlog = YNormalize.new_project_into_normalized(yraw, LOGARITHMIC, A=A)
    theta = _rounded(random_thetas(1, d, seed=n, noise=(NOISE[A], NOISE[A] * 1.01))[0], A)
    return x, yraw, yl, ynl, ynlog, theta


@pytest.mark.gpu
@pytest.mark.parametrize("A", [np.float64, np.float32])
@pytest.mark.parametrize("n", [1025, 4097])
def test_acquisition_is_the_epilogue_of_predict(n, A):
    """Bit for bit on the latency path (m = 1, 17, 64) and the split path (65, 1000; f64 at n = 4097 also m = 70000,
    three variance chunks), linear and log projection, fmin at min(y), below and above every mean, and the bound;
    the returned index is the restated rule on the returned vector."""
    d = 3
    x, yraw, yl, ynl, ynlog, theta = _model_case(A, n, d)
    ms = [1, 17, 64, 65, 1000] + ([70000] if A == np.float64 and n == 4097 else [])
    xs = _candidates(x.astype(np.float64), max(ms), n).astype(A)
    for m in ms:
        assert _predict_path(m, d, _np(n), A().itemsize) == ("latency" if m <= 64 else "split")
    with _ctx(A) as ctx:
        ctx.set_data(x, yl)
        model = ctx.model(theta)
        mean_all, var_all = model.predict(xs, warn=False)
        for yn in (ynl, ynlog):
            for name, fmin in _fmins(yn, yraw, mean_all, var_all).items():
                for m in ms:
                    _assert_wired(model, yn, xs[:m], 0, fmin, f"{_name(A)} n={n} proj={yn.projection} {name} m={m}")
            for m in ms:
                _assert_wired(model, yn, xs[:m], 1, CB, f"{_name(A)} n={n} proj={yn.projection} cb m={m}")
        model.close()


def _truth_ei_check(rec, tag, got_ei, mean, var, mu_star, var_star, e_mu, e_var, fmin_n):
    """|EI - EI(mu*, sigma*)| <= E_mu + 0.4 E_sigma + the arithmetic bound, and the pick within twice the bound."""
    import mpmath
    sd, sd_star = np.sqrt(var), np.sqrt(var_star)
    e_sd = np.minimum(e_var / np.maximum(sd + sd_star, 1e-300), math.sqrt(e_var))
    with mpmath.workdps(60):
        star = np.array([float(_ei_mp(mpmath.mpf(h) + mpmath.mpf(lo), mpmath.sqrt(mpmath.mpf(v)), fmin_n))
                         for h, lo, v in zip(mu_star[0], mu_star[1], var_star)])
    bound = e_mu + PHI0 * e_sd + _ei_bound(mean, sd, fmin_n)
    err = np.abs(got_ei - star)
    r = _ratio(err, bound)
    rec[tag] = {"max err/bound": float(r.max()), "max err": float(err.max())}
    assert (r <= 1.0).all(), (tag, int(r.argmax()), float(r.max()))
    return star, bound


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1025, 4097])
def test_acquisition_against_the_posterior_truth(n):
    """f64: EI and the confidence bound against EI(mu*, sigma*) and mu* + cb sigma* of test_f64_truth's posterior,
    with E_mu and E_var its own bounds (R x LAPACK's error + F eps S).  At n = 4097 the 70000-row call is sampled at
    the variance-chunk edges (32256 rows a chunk)."""
    A, d = np.float64, 3
    x, yraw, yl, ynl, ynlog, theta = _model_case(A, n, d)
    m = 70000 if n == 4097 else 1000
    xs = _candidates(x, m, n)
    if n == 4097:
        rows = np.unique(np.concatenate([np.arange(40), 32256 + np.arange(-20, 20), 64512 + np.arange(-20, 20),
                                         m - 40 + np.arange(40)]))
    else:
        rows = np.arange(m)
    rec = {}
    c = math.exp(theta[1])
    with _ctx(A) as ctx:
        ctx.set_data(x, yl)
        k = _gpu_k(ctx, theta)
        tr = _truth_of(("acquisition", n), k, yl, theta, x)
        lap = _reference(theta, x, yl, k=k)
        model = ctx.model(theta)
        tm, tv, s_mean, s_var = _predict_star(tr, theta, x, xs[rows])
        ks = _kernel_f64(xs[rows], x, c, np.exp(theta[2:]), 2.5)
        lm = ks @ lap.alpha
        u = ks @ lap.w.T
        lv = np.maximum(c + 1e-5 - np.einsum("ij,ij->i", u, u), 0.0)
        e_mu = R * float(np.abs((lm - tm[0]) - tm[1]).max()) + F * EPS * float(s_mean.max())
        e_var = R * float(np.abs(lv - tv).max()) + F * EPS * float(s_var.max())
        for yn in (ynl, ynlog):
            mean_all, var_all = model.predict(xs, warn=False)
            for name, fmin in _fmins(yn, yraw, mean_all, var_all).items():
                _, ei, best, mean, var, fmin_n = _assert_wired(model, yn, xs, 0, fmin, f"n={n} {name}")
                star, bound = _truth_ei_check(rec, f"n={n} proj={yn.projection} EI {name}", ei[rows], mean[rows],
                                              var[rows], tm, tv, e_mu, e_var, fmin_n)
                if n == 1025:  # the pick, over every row
                    assert star[best] >= star.max() - 2 * bound.max(), (name, best, int(star.argmax()))
            # the confidence bound, in normalised units: |y - y*| <= E_mu + |cb| E_sigma + rounding of mu + cb sigma
            out, _, best, mean, var, _ = _assert_wired(model, yn, xs, 1, CB, f"n={n} cb")
            sd, sd_star = np.sqrt(var[rows]), np.sqrt(tv)
            e_sd = np.minimum(e_var / np.maximum(sd + sd_star, 1e-300), math.sqrt(e_var))
            y = mean[rows] + sd * CB
            y_star = (tm[0] + tm[1]) + CB * sd_star
            bound = e_mu + abs(CB) * e_sd + 2 * EPS * (np.abs(mean[rows]) + np.abs(sd * CB))
            err = np.abs(y - y_star)
            r = _ratio(err, bound)
            rec[f"n={n} proj={yn.projection} cb"] = {"max err/bound": float(r.max())}
            assert (r <= 1.0).all(), (yn.projection, float(r.max()))
            if n == 1025:  # the pick, in natural units: out = location_from(y), monotone in y
                amp, ex = yn.amplitude, yn.expected
                if yn.projection == 0:
                    o_star, slope = (y_star - 0.05) * amp + ex, np.full_like(y_star, amp)
                else:
                    o_star = np.exp(y_star * amp) + ex
                    slope = amp * np.exp(y_star * amp)
                o_bound = slope * bound + 8 * EPS * (np.abs(o_star) + abs(ex))
                assert o_star[best] <= o_star.min() + 2 * o_bound.max(), (best, int(o_star.argmin()))
        model.close()
    _note(f"acquisition truth n={n}", rec)


@pytest.mark.gpu
def test_f32_ei_within_twice_the_host_path_on_lapack_f32():
    """f32 at n = 1025: the device EI's error against the f64 truth of the same f32 inputs is at most 2x the error of
    the host EI fed with LAPACK f32's mean and variance, plus a floor of 4 eps32 times EI's condition sum."""
    from scipy.linalg import cho_solve, lapack

    from tests.test_dispatch_sweep import _lapack_f32
    from tests.util import oracle_kernel
    from hbetune_rs_b200._lib import lib
    from hbetune_rs_b200.gpr import _ptr
    A, n, d = np.float32, 1025, 3
    x, yraw, yl, ynl, _, theta = _model_case(A, n, d)
    xs = _candidates(x.astype(np.float64), 1000, n).astype(A)
    x64, y64, xs64 = x.astype(np.float64), yl.astype(np.float64), xs.astype(np.float64)
    truth = _reference(theta, x64, y64)
    c = math.exp(theta[1])
    ks = _kernel_f64(xs64, x64, c, np.exp(theta[2:]), 2.5)
    mu_star = ks @ truth.alpha
    u = ks @ truth.w.T
    var_star = np.maximum(c + 1e-5 - np.einsum("ij,ij->i", u, u), 0.0)
    k32, w32, _ = _lapack_f32(theta, x, 2.5)  # spotrf + strtri on the f32 oracle's K
    low32, info = lapack.spotrf(k32, lower=1, clean=1)
    assert info == 0
    alpha32 = cho_solve((low32, True), yl)
    ks32 = oracle_kernel(theta).kernel(xs, x, np.float32)
    m32 = (ks32 @ alpha32).astype(np.float32)
    u32 = ks32 @ w32.T
    v32 = np.maximum(np.float32(c) + np.float32(1e-5) - np.einsum("ij,ij->i", u32, u32), 0).astype(np.float32)
    assert m32.dtype == np.float32 and u32.dtype == np.float32
    rec = {}
    with _ctx(A) as ctx:
        ctx.set_data(x, yl)
        model = ctx.model(theta)
        mean_all, var_all = model.predict(xs, warn=False)
        for name, fmin in _fmins(ynl, yraw, mean_all, var_all).items():
            _, ei, _, _, _, fmin_n = _assert_wired(model, ynl, xs, 0, fmin, f"f32 {name}")
            star = _ei_exact(mu_star, np.sqrt(var_star), fmin_n)
            host = np.empty(1000, dtype=A)
            assert lib.hbegp_expected_improvement_a(1, 1000, _ptr(m32), _ptr(v32), fmin_n, _ptr(host)) == 0
            e_dev = np.abs(ei.astype(np.float64) - star)
            e_host = float(np.abs(host.astype(np.float64) - star).max())
            floor = 4 * 2.0 ** -24 * (_ei_bound(mu_star, np.sqrt(var_star), fmin_n) / (F_EI * EPS)).max()
            rec[name] = {"device": float(e_dev.max()), "host on LAPACK f32": e_host, "floor": float(floor)}
            assert e_dev.max() <= 2 * e_host + floor, (name, rec[name])
        model.close()
    _note("acquisition f32 n=1025", rec)


@pytest.mark.gpu
def test_rebuilt_and_appended_models_keep_the_epilogue():
    """After an eviction (one resident model, a second model built) acquisition on the rebuilt model returns the bits
    it returned before; an appended model (1000 -> 1100) is the harness epilogue of its own prediction."""
    import hbetune_rs_b200 as h
    A, d = np.float64, 3
    x, yraw, yl, ynl, ynlog, theta = _model_case(A, 1100, d)
    xs = _candidates(x, 300, 3)
    with _ctx(A) as ctx:
        ctx.set_data(x[:1000], yl[:1000])
        first = ctx.model(theta)
        before = [_acq(first, yn, xs, mode, p) for yn in (ynl, ynlog) for mode, p in ((0, float(yraw.min())), (1, CB))]
        ctx.set_resident_models(1)
        second = ctx.model(_rounded(theta + 0.1, A))
        _acq(second, ynl, xs[:5], 0, float(yraw.min()))
        after = [_acq(first, yn, xs, mode, p) for yn in (ynl, ynlog) for mode, p in ((0, float(yraw.min())), (1, CB))]
        for (a1, a2, ab, _), (b1, b2, bb, _) in zip(before, after):
            assert _bits_equal(a1, b1).all() and ab == bb
            assert a2 is None or _bits_equal(a2, b2).all()
        second.close()
        ctx.set_resident_models(8)
        ctx.set_data(x, yl)
        app = h.Model(ctx, prior=first, want_kinv=False)
        assert app.appended
        for yn in (ynl, ynlog):
            _assert_wired(app, yn, xs, 0, float(yraw.min()), "appended ei")
            _assert_wired(app, yn, xs, 1, CB, "appended cb")
        app.close()
        first.close()


@pytest.mark.gpu
def test_acquisition_reports_the_warnings_of_predict():
    """c = 1e14 (test_predict_lists_the_variances_below_the_warning_level): the same n_below_warn and the same
    hbegp_predict_warn_values as hbegp_predict on the same rows, for both acquisition calls."""
    from hbetune_rs_b200.estimator import YNormalize
    n, d = 120, 2
    x, y = synth(n, d)
    theta = np.array([math.log(1e-2), math.log(1e14), math.log(2.0), math.log(2.0)])
    xs = np.concatenate([x[:60], np.random.default_rng(1).random((140, d))])
    yl, yn = YNormalize.new_project_into_normalized(y + 5.0, 0)
    with _ctx(np.float64) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta)
        model.predict(xs, warn=False)
        count = model.n_below_warn
        vals, rows = model.warn_values(cap=4096)
        assert count > 0
        for mode, p in ((0, 5.0), (1, CB)):
            _, _, _, nb = _acq(model, yn, xs, mode, p)
            v2, r2 = model.warn_values(cap=4096)
            assert nb == count
            np.testing.assert_array_equal(v2, vals)
            np.testing.assert_array_equal(r2, rows)
        model.close()
