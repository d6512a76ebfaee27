"""The emulated f64 K^-1 = W^T W (Ozaki scheme II, hbetune_rs_b200/csrc/gemm_i8.cuh) bit for bit.

The scheme defines its result exactly: column j of W is scaled by 2^e_j and rounded once to b bits, the product of the
scaled integers is exact, and the result is rounded once to double.  `_oz_kinv_exact` restates that from the
definition (exponents, scaled integers, an exact integer product from 18-bit slices, one correct rounding through
Python integers) without the residues, the moduli or the Chinese remaindering of the kernels, and with b, E_CLAMP and
the E_BAD limit stated here rather than read from the header.  The GPU tests feed arbitrary W to the four kernels
through tests/cuda/liboz_harness.so (rounding ties, exponent extremes, non-finite columns, batches, the edges of the
CRT range, the largest size) and compare every written cell, and K^-1 of real factors through the engine.

Error model (K6b in DESIGN.md), with M_j = max_{k >= j} |W_kj|:
    |K^-1_emu - W^T W|_ij <= 2^-b (M_j |W_.i|_1 + M_i |W_.j|_1) + np 2^-2b M_i M_j + 2^-53 |K^-1_ij|
"""
import ctypes
import math
import os
import shutil
import subprocess
import time

import numpy as np
import pytest

from tests.test_dispatch_sweep import _ctx, _kernel_f64, _note, _np, _reference, _rounded
from tests.test_kinv_emulation import H, _crt, _epilogue_mod, _residue_pieces, _to_double
from tests.util import random_thetas, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hbetune_rs_b200", "csrc")
HARNESS = os.path.join(ROOT, "tests", "cuda", "liboz_harness.so")
TB, TILE = 128, 64
NP_MAX = 46016

# The scheme's parameters, stated independently of the header.  b per padded size: the largest b <= 50 with
# np 2^2b < P / 2 (P = 2^110.2, the product of the 14 moduli).
BITS_FROM = [(64, 50), (576, 49), (2304, 48), (9216, 47), (36672, 46)]
E_CLAMP = 400         # |e_j| <= 400
BAD_ABOVE = 2.0 ** 440  # a column max beyond this (or NaN / Inf) makes the column's row and column of K^-1 NaN
SENTINEL = np.array([0x7FF80000DEADBEEF], dtype=np.int64).view(np.float64)[0]  # a NaN no kernel writes


def _bits(np_):
    return [b for lo, b in BITS_FROM if np_ >= lo][-1]


# ------------------------------------------------------------------------------------------------ the exact restatement


def _oz_exponents(w, bits):
    """e_j from the NaN-propagating max over k >= j of column j; `bad` marks NaN, Inf or a max above 2^440."""
    m = np.abs(np.tril(w)).max(axis=0)
    bad = ~(m <= BAD_ABOVE)
    _, E = np.frexp(np.where(bad, 1.0, m))  # m < 2^E (subnormals included)
    e = np.clip(bits - E.astype(np.int64), -E_CLAMP, E_CLAMP)
    return np.where(bad | (m == 0), 0, e), bad


def _oz_scaled(w, e, bad):
    """W' = rint(2^e_j W_kj) on the lower triangle as exact int64 (|W'| <= 2^50); zero in non-finite columns."""
    low = np.where(bad[None, :], 0.0, np.tril(w))
    ws = np.rint(np.ldexp(low, e[None, :]))
    assert np.abs(ws).max() <= 2.0 ** 50
    return ws.astype(np.int64)


def _slices(ws):
    """W' = s0 + s1 2^18 + s2 2^36 with |s| <= 2^17: every slice product summed over <= 46016 rows is below 2^53."""
    out, rest = [], ws
    for _ in range(2):
        s = ((rest + (1 << 17)) & ((1 << 18) - 1)) - (1 << 17)
        out.append(s.astype(np.float64))
        rest = (rest - s) >> 18
    assert np.abs(rest).max() <= 1 << 17
    return out + [rest.astype(np.float64)]


def _mm(a, b):
    """a^T b of f64 integer matrices (exact: every partial sum is an integer below 2^53), on the GPU if there is one."""
    try:
        import torch
        if torch.cuda.is_available():
            return (torch.from_numpy(a).cuda().T @ torch.from_numpy(b).cuda()).cpu().numpy()
    except ImportError:
        pass
    return a.T @ b


def _limbs(sl, rows, cols):
    """C' on rows x cols (slices) as five exact int64 limbs: C' = sum_k c_k 2^(18 k)."""
    k0 = max(rows.start, cols.start)  # W' is lower triangular
    c = [np.zeros((rows.stop - rows.start, cols.stop - cols.start)) for _ in range(5)]
    for a in range(3):
        for b in range(3):
            c[a + b] += _mm(np.ascontiguousarray(sl[a][k0:, rows]), np.ascontiguousarray(sl[b][k0:, cols]))
    assert max(np.abs(x).max() for x in c) < 2.0 ** 53
    return [x.astype(np.int64) for x in c]


def _round_limbs(c, shift):
    """One correct rounding of sum_k c_k 2^(18 k) 2^-shift per element, through Python integers."""
    v = c[4].astype(object)
    for k in (3, 2, 1, 0):
        v = (v << 18) + c[k].astype(object)
    flat, sh = v.ravel(), (-shift).ravel().tolist()
    return np.array([math.ldexp(float(x), s) for x, s in zip(flat.tolist(), sh)], dtype=np.float64).reshape(v.shape)


class Exact:
    """The scheme for one np x np matrix w (only k >= j is read): exponents, scaled integers, their slices."""

    def __init__(self, w, np_=None):
        self.np = np_ or w.shape[0]
        assert w.shape == (self.np, self.np)
        self.bits = _bits(self.np)
        self.e, self.bad = _oz_exponents(w, self.bits)
        self.ws = _oz_scaled(w, self.e, self.bad)
        self.sl = _slices(self.ws)

    def block(self, rows, cols):
        """The rounded C' 2^-(e_i + e_j) on rows x cols (slices); NaN in the rows and columns of non-finite columns."""
        c = _limbs(self.sl, rows, cols)
        out = _round_limbs(c, self.e[rows][:, None] + self.e[cols][None, :])
        out[self.bad[rows], :] = np.nan
        out[:, self.bad[cols]] = np.nan
        return out


def _written(np_):
    """The cells launch_kinv writes: the lower 64 x 64 tiles (including the upper half of each diagonal 64-tile)."""
    t = np.arange(np_) // TILE
    return t[:, None] >= t[None, :]


def _oz_kinv_exact(w, np_=None):
    """Every cell launch_kinv must write for w (the lower 64 x 64 tiles, as the symmetric C'), 0 elsewhere."""
    ex = Exact(w, np_)
    out = np.zeros((ex.np, ex.np))
    for r0 in range(0, ex.np, TB):
        r1 = min(ex.np, r0 + TB)
        out[r0:r1, :r1] = ex.block(slice(r0, r1), slice(0, r1))
    return np.where(_written(ex.np), out, 0.0)


# ------------------------------------------------------------------------------------------------ inputs


def _random_w(np_, seed, lo=-300, hi=300):
    """Lower triangle of full-mantissa doubles with per-column power-of-two scales in [2^lo, 2^hi], NaN above."""
    rng = np.random.default_rng(seed)
    w = rng.standard_normal((np_, np_)) * rng.random((np_, np_))
    w = np.ldexp(w, rng.integers(lo, hi + 1, np_)[None, :])
    w[np.triu_indices(np_, 1)] = np.nan
    return w


def _edge_w(np_, seed):
    """Columns whose max is exactly 2^k or the double below it, exact half-integers after scaling (even and odd
    integer part), subnormal entries, an all-subnormal column and all-zero columns."""
    rng = np.random.default_rng(seed)
    w = _random_w(np_, seed, -40, 40)
    b = _bits(np_)
    for j in range(0, np_ - 8, 7):
        kind, k = j // 7 % 6, int(rng.integers(-200, 200))
        col = w[j:, j]
        if kind == 0:                                    # max exactly 2^k: e = b - k - 1
            col[:] = np.ldexp(rng.random(len(col)) * 0.99, k)
            col[int(rng.integers(0, len(col)))] = -2.0 ** k
        elif kind == 1:                                  # max the double below 2^k: e = b - k, W' = 2^b at the max
            col[:] = np.ldexp(rng.random(len(col)) * 0.99, k)
            col[0] = np.nextafter(2.0 ** k, 0.0)
        elif kind == 2:                                  # max 2^k, ties m + 1/2 for even and odd m
            e = b - k - 1
            m = rng.integers(-(2 ** 40), 2 ** 40, len(col))
            col[:] = np.ldexp(m + 0.5, -e)
            col[0] = 2.0 ** k
        elif kind == 3:                                  # subnormal entries under a small normal max
            col[:] = rng.integers(-1000, 1000, len(col)) * 5e-324
            col[0] = np.ldexp(1.0, -300)
        elif kind == 4:                                  # only subnormals: the exponent clamps
            col[:] = rng.integers(-(2 ** 40), 2 ** 40, len(col)) * 5e-324
        else:                                            # all zero
            col[:] = 0.0
    return w


def _clamp_w(np_, seed):
    """Column maxima from 2^(b - 461) (clamped to e = 400) to 2^440 (e = b - 441), in a random order of columns."""
    rng = np.random.default_rng(seed)
    b = _bits(np_)
    w = _random_w(np_, seed, 0, 0)
    exps = np.concatenate([np.arange(b - 460, b - 395), np.arange(-345, -335), np.arange(430, 442),
                           rng.integers(-340, 440, np_)])[:np_]
    rng.shuffle(exps)
    for j in range(np_):
        w[j:, j] = np.ldexp(w[j:, j] / np.abs(w[j:, j]).max(), int(exps[j]) - 1)
        w[j + int(rng.integers(0, np_ - j)), j] = 2.0 ** (int(exps[j]) - 1)  # the max in a random row: m = 2^(x - 1)
    return w


# ------------------------------------------------------------------------------------------------ CPU part


def test_bits_and_exponents_stated_here():
    P = math.prod(H["moduli"])
    for np_ in range(64, NP_MAX + 1, 64):
        b = _bits(np_)
        assert np_ * 2 ** (2 * b) < P // 2 and (b == 50 or np_ * 2 ** (2 * b + 2) >= P // 2), np_
    # e_j = b - E_j (max in [2^(E-1), 2^E)) for every max in [2^-340, 2^440], the max itself scaled into (2^(b-1), 2^b]
    for x in list(range(-340, 441)):
        for m in (2.0 ** x, np.nextafter(2.0 ** x, np.inf), np.nextafter(2.0 ** x, 0.0)):
            if not 2.0 ** -340 <= m <= 2.0 ** 440:
                continue
            w = np.array([[m]])
            for np_ in (64, 2304, 46016):
                e, bad = _oz_exponents(w, _bits(np_))
                E = math.frexp(m)[1]
                assert not bad[0] and e[0] == _bits(np_) - E and 2 ** (_bits(np_) - 1) <= m * 2.0 ** e[0] <= 2 ** _bits(np_)
    e, bad = _oz_exponents(np.array([[2.0 ** 440, 0, 0], [0.0, np.nextafter(2.0 ** 440, np.inf), 0], [1.0, np.nan, 0]]), 50)
    assert list(bad) == [False, True, False] and e[0] == 50 - 441 and e[2] == 0
    e, _ = _oz_exponents(np.array([[2.0 ** -700]]), 50)
    assert e[0] == E_CLAMP


def test_restatement_ignores_the_upper_triangle():
    w = _random_w(192, 1)
    w2 = w.copy()
    w2[np.triu_indices(192, 1)] = np.random.default_rng(2).standard_normal(192 * 191 // 2) * 1e300
    np.testing.assert_array_equal(_oz_kinv_exact(w), _oz_kinv_exact(w2))


def test_restatement_is_the_product_for_small_integers():
    """Integers of up to 40 bits with power-of-two column scales are exact after scaling: K^-1 = W^T W exactly."""
    rng = np.random.default_rng(3)
    for np_ in (64, 192, 640):
        a = np.tril(rng.integers(-(2 ** 20), 2 ** 20, (np_, np_))).astype(np.float64)
        s = rng.integers(-20, 20, np_)
        w = np.ldexp(a, s[None, :])
        got = _oz_kinv_exact(w)
        want = w.T @ w  # exact: every partial sum is a multiple of 2^(s_i + s_j) below 2^53 of it
        mask = _written(np_)
        np.testing.assert_array_equal(got[mask], want[mask])


@pytest.mark.parametrize("np_", [192, 640])
def test_restatement_matches_the_residue_path(np_):
    """The same bits as the per-element restatement of the kernels' arithmetic in tests/test_kinv_emulation.py:
    residues of W', per-modulus products reduced as the epilogue does, CRT merge and its single rounding."""
    w = _random_w(np_, np_, -60, 60)
    ex = Exact(w)
    got = _oz_kinv_exact(w)
    planes = [_residue_pieces(ex.ws.T, p) for p in H["moduli"]]
    prods = [_epilogue_mod(r @ r.T, p) for r, p in zip(planes, H["moduli"])]
    rng = np.random.default_rng(np_)
    cells = [(0, 0), (np_ - 1, np_ - 1), (np_ - 1, 0), (63, 0), (3, 60)]
    cells += [tuple(sorted(rng.integers(0, np_, 2))[::-1]) for _ in range(300)]
    for i, j in cells:
        c = _crt([int(pr[i, j]) for pr in prods])
        assert _to_double(c, int(ex.e[i] + ex.e[j])) == got[i, j], (i, j)


def test_rounding_of_limbs_matches_python_integers():
    rng = np.random.default_rng(4)
    c = [rng.integers(-(2 ** 52), 2 ** 52, 3000) for _ in range(5)]
    c[4][:10] = 0
    c[3][:5] = 0
    c[0][-3:] = [1, 0, -1]  # near-ties: the low limb decides
    shift = rng.integers(-400, 800, 3000)
    got = _round_limbs(c, shift)
    for t in range(3000):
        v = sum(int(c[k][t]) << (18 * k) for k in range(5))
        assert got[t] == math.ldexp(float(v), -int(shift[t])), t


def _accurate_product(w, np_):
    """W^T W to about 2^-100 of M_i M_j: W rounded to 100 bits per column max, split in six 17-bit slices, exact
    integer products combined in Python integers, then rounded once."""
    n = w.shape[0]
    wl = np.tril(w)
    _, E = np.frexp(np.abs(wl).max(axis=0))
    g = 100 - E.astype(np.int64)
    big = [[int(round(math.ldexp(float(x), int(g[j])))) if x else 0 for j, x in enumerate(row)] for row in wl.tolist()]
    big = np.array(big, dtype=object)
    sl, rest = [], big
    for _ in range(5):
        s = np.array([((int(v) + (1 << 16)) & ((1 << 17) - 1)) - (1 << 16) for v in rest.ravel()], dtype=np.int64).reshape(n, n)
        sl.append(s.astype(np.float64))
        rest = (rest - s.astype(object)) >> 17
    sl.append(np.array(rest, dtype=np.float64))
    acc = np.zeros((n, n), dtype=object)
    for a in range(6):
        for b in range(6):
            acc = acc + (np.rint(sl[a].T @ sl[b]).astype(np.int64).astype(object) << (17 * (a + b)))
    sh = (g[:, None] + g[None, :]).ravel().tolist()
    return np.array([math.ldexp(float(v), -s) for v, s in zip(acc.ravel().tolist(), sh)]).reshape(n, n)


def test_error_model_on_a_real_factor():
    """The bound of the module docstring, elementwise, on W = L^-1 at noise 1e-5 (kappa ~ 2e7), b of np 2112."""
    n, d = 700, 3
    x, y = synth(n, d, seed=n)
    theta = random_thetas(1, d, seed=n, noise=(1e-5, 1.01e-5))[0]
    w = _reference(theta, x, y).w
    np_ = 2112  # b = 49, as at n = 2049: W padded with I does not change the first n rows and columns
    wp = np.eye(np_)
    wp[:n, :n] = w
    ex = Exact(wp)
    emu = ex.block(slice(0, n), slice(0, n))
    ref = _accurate_product(w, np_)
    wl = np.abs(np.tril(w))
    M, l1 = wl.max(axis=0), wl.sum(axis=0)
    b = ex.bits
    bound = (2.0 ** -b * (M[None, :] * l1[:, None] + M[:, None] * l1[None, :]) + np_ * 2.0 ** (-2 * b) * np.outer(M, M)
             + 2.0 ** -52 * np.abs(ref))  # two roundings: the scheme's and the reference's
    err = np.abs(emu - ref)
    assert (err <= bound).all(), float((err / bound).max())
    assert (err / bound).max() > 1e-3  # the bound is not vacuous
    rel = err / np.abs(ref)
    _note("kinv bits: error model cpu n=700 noise=1e-5",
          {"max err/bound": float((err / bound).max()), "median rel": float(np.median(rel)),
           "p99 rel": float(np.quantile(rel, 0.99)), "max err/max|kinv|": float(err.max() / np.abs(ref).max())})


def test_harness_builds_without_a_gpu():
    lib = _harness()
    assert lib.oz_scale_bits(2112) == 49 and lib.oz_scale_bits(46016) == 46
    assert lib.oz_slot_bytes(128) == 2 * 14 * 128 * 128 + 128 * 128


# ------------------------------------------------------------------------------------------------ GPU part: the harness


def _harness():
    if not os.path.exists(HARNESS):
        nvcc = shutil.which("nvcc") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
        subprocess.run(["make", "-C", CSRC, f"NVCC={nvcc}", "../../tests/cuda/liboz_harness.so"], check=True)
    lib = ctypes.CDLL(HARNESS)
    lib.oz_slot_bytes.restype, lib.oz_slot_bytes.argtypes = ctypes.c_size_t, [ctypes.c_int]
    lib.oz_scale_bits.restype, lib.oz_scale_bits.argtypes = ctypes.c_int, [ctypes.c_int]
    lib.oz_kinv.restype = ctypes.c_int
    lib.oz_kinv.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                            ctypes.c_void_p]
    return lib


def _launch(lib, W, C, np_, cnt):
    """launch_kinv on torch CUDA tensors; the workspace is filled with 0xFF and C with SENTINEL first."""
    import torch
    assert lib.oz_scale_bits(np_) == _bits(np_)
    ws = torch.full((cnt * lib.oz_slot_bytes(np_),), 0xFF, dtype=torch.uint8, device="cuda")
    C.view(torch.int64).fill_(int(SENTINEL.view(np.int64)))
    rc = lib.oz_kinv(W.data_ptr(), C.data_ptr(), np_ * np_, np_, cnt, ws.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert rc == 0, f"launch_kinv: cudaError {rc}"
    torch.cuda.synchronize()
    del ws


def _run(w):
    """C for one matrix or a stack of them, as a NumPy array."""
    import torch
    lib = _harness()
    W = torch.from_numpy(np.ascontiguousarray(w)).cuda()
    C = torch.empty_like(W)
    _launch(lib, W, C, w.shape[-1], 1 if w.ndim == 2 else w.shape[0])
    return C.cpu().numpy()


def _want(exact):
    return np.where(_written(exact.shape[0]), exact, SENTINEL)


def _assert_bits(got, want, tag):
    gb, wb = got.view(np.int64), want.view(np.int64)
    bad = gb != wb
    if bad.any():
        i, j = np.argwhere(bad)[0]
        with np.errstate(invalid="ignore"):
            rel = np.nanmax(np.abs(got - want)[bad] / np.abs(want[bad])) if np.isfinite(want[bad]).any() else float("nan")
        raise AssertionError(f"{tag}: {int(bad.sum())} cells differ, first ({i}, {j}): got {got[i, j]!r}, want "
                             f"{want[i, j]!r}; max relative difference {rel:.3e}")


@pytest.mark.gpu
@pytest.mark.parametrize("np_", [64, 128, 192, 2048, 2112, 2304, 4096])
def test_random_full_mantissa(np_):
    t0 = time.perf_counter()
    w = _random_w(np_, np_)
    _assert_bits(_run(w), _want(_oz_kinv_exact(w)), f"np={np_}")
    _note(f"kinv bits: random np={np_}", {"bits": _bits(np_), "s": time.perf_counter() - t0})


@pytest.mark.gpu
@pytest.mark.parametrize("np_", [192, 2112])
def test_rounding_edges(np_):
    w = _edge_w(np_, np_ + 1)
    ex = Exact(w)
    assert (ex.e == E_CLAMP).any() and (ex.e == 0).any() and np.abs(ex.ws).max() == 2 ** ex.bits
    _assert_bits(_run(w), _want(_oz_kinv_exact(w)), f"edges np={np_}")


@pytest.mark.gpu
@pytest.mark.parametrize("np_", [640, 2304])
def test_exponent_clamp(np_):
    w = _clamp_w(np_, np_)
    ex = Exact(w)
    assert (ex.e == E_CLAMP).sum() >= 60 and (ex.e == ex.bits - 441).any() and not ex.bad.any()
    _assert_bits(_run(w), _want(_oz_kinv_exact(w)), f"clamp np={np_}")


@pytest.mark.gpu
@pytest.mark.parametrize("np_", [192, 2112])
def test_non_finite_columns(np_):
    w = _random_w(np_, np_ + 2, -20, 20)
    w[np_ - 5, 3] = np.nan                       # NaN at one k of column 3
    w[70, 64] = -np.inf                          # Inf on the diagonal tile border
    w[np_ - 1, np_ - 70] = 2.0 ** 441            # finite, beyond the limit
    w[np_ - 2, 100] = 2.0 ** 440                 # at the limit: finite result
    ex = Exact(w)
    assert list(np.flatnonzero(ex.bad)) == sorted([3, 64, np_ - 70])
    want = _want(_oz_kinv_exact(w))
    assert np.isnan(want[np_ - 1, 3]) and np.isfinite(want[np_ - 1, 100])
    _assert_bits(_run(w), want, f"non-finite np={np_}")


@pytest.mark.gpu
def test_batch_members_equal_their_single_bits():
    np_, cnt = 2112, 5
    ws = np.stack([_random_w(np_, 100 + b) for b in range(cnt)])
    ws[2, np_ - 3, 17] = np.nan
    batch = _run(ws)
    for b in range(cnt):
        want = _want(_oz_kinv_exact(ws[b]))
        _assert_bits(batch[b], want, f"batch member {b}")
        _assert_bits(_run(ws[b]), want, f"alone {b}")


@pytest.mark.gpu
def test_only_the_lower_64_tiles_are_written():
    """Every cell of the lower 64 x 64 tiles is written (no SENTINEL left), none above them, for a W whose product
    fills every tile and with a ragged last tile."""
    np_ = 320
    w = np.tril(np.ones((np_, np_)))
    got = _run(w)
    wr = _written(np_)
    assert not (got.view(np.int64)[wr] == SENTINEL.view(np.int64)).any()
    assert (got.view(np.int64)[~wr] == SENTINEL.view(np.int64)).all()
    i = np.arange(np_)
    np.testing.assert_array_equal(got[wr], (np_ - np.maximum(i[:, None], i[None, :]))[wr])


def _free_bytes():
    import torch
    return torch.cuda.mem_get_info()[0]


def _big(np_, fill, need):
    """An np x np f64 tensor on the GPU filled row block by row block by fill(r0, r1) (lower part; NaN above)."""
    import torch
    if _free_bytes() < need:
        pytest.skip(f"np={np_} needs {need / 2 ** 30:.0f} GiB of free GPU memory, {_free_bytes() / 2 ** 30:.0f} GiB are free")
    W = torch.empty((np_, np_), dtype=torch.float64, device="cuda")
    for r0 in range(0, np_, 4096):
        r1 = min(np_, r0 + 4096)
        lower = torch.ones((r1 - r0, np_), dtype=torch.bool, device="cuda").tril_(r0)
        W[r0:r1] = torch.where(lower, fill(r0, r1), float("nan"))
    return W


def _need(np_, lib):
    return 2 * np_ * np_ * 8 + lib.oz_slot_bytes(np_) + 4 * 4096 * np_ * 8 + (2 << 30)


@pytest.mark.gpu
@pytest.mark.parametrize("np_", [9152, 9216, 36608, 36672, NP_MAX])
def test_scale_against_an_exact_product(np_):
    """Integers in [-2^18, 2^18] with power-of-two column scales: W' is W exactly, and the f64 product of the lower
    triangles is exact too (every partial sum is an integer multiple of 2^(s_i + s_j) below 2^53 of it)."""
    import torch
    lib = _harness()
    g = torch.Generator(device="cuda").manual_seed(np_)
    s = torch.randint(-100, 101, (np_,), device="cuda", generator=g)
    scale = ((s + 1023) << 52).view(torch.float64)  # 2^s from its bits (exact, unlike a computed power)

    def fill(r0, r1):
        a = torch.randint(-(2 ** 18), 2 ** 18 + 1, (r1 - r0, np_), device="cuda", generator=g).to(torch.float64)
        return a * scale[None, :]

    t0 = time.perf_counter()
    W = _big(np_, fill, _need(np_, lib))
    C = torch.empty_like(W)
    _launch(lib, W, C, np_, 1)
    for r0 in range(0, np_, 4096):  # W's upper triangle (NaN) to zero for the reference
        W[r0:r0 + 4096].nan_to_num_(nan=0.0)
    sent = int(SENTINEL.view(np.int64))
    idx = torch.arange(np_, device="cuda") // TILE
    for r0 in range(0, np_, 4096):
        r1 = min(np_, r0 + 4096)
        ref = W[:, r0:r1].T @ W  # rows r0..r1 of W^T W
        wr = idx[r0:r1, None] >= idx[None, :]
        want = ref.view(torch.int64)
        want[~wr] = sent
        diff = C[r0:r1].view(torch.int64) != want
        if diff.any():
            i, j = diff.nonzero()[0].tolist()
            exact = math.fsum((W[:, r0 + i] * W[:, j]).cpu().tolist())  # exact products, one correct rounding
            raise AssertionError(f"np={np_}: {int(diff.sum())} cells differ in rows {r0}..{r1}, first ({r0 + i}, {j}): "
                                 f"kernel {C[r0 + i, j].item()!r}, f64 product {ref[i, j].item()!r}, exact {exact!r}")
    _note(f"kinv bits: scale np={np_}", {"bits": _bits(np_), "s": time.perf_counter() - t0, "ran": True})
    del W, C
    torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("np_", [4096, NP_MAX])
@pytest.mark.parametrize("signs", ["one", "per column"])
def test_crt_range_extremes(np_, signs):
    """W_kj = s_j (2^b - 128), e = 0: C'_ij = s_i s_j (np - max(i, j)) (2^b - 128)^2, the largest |C'| this np can
    give, at both signs; every residue mod 256 is -128, so |C_256| = np 128^2 (the epilogue's extreme)."""
    import torch
    lib = _harness()
    b = _bits(np_)
    v = float(2 ** b - 128)
    sg = torch.ones(np_, dtype=torch.float64, device="cuda")
    if signs == "per column":
        sg[1::2] = -1.0
        sg[2::3] *= -1.0
    W = _big(np_, lambda r0, r1: (sg * v)[None, :].expand(r1 - r0, np_).clone(), _need(np_, lib))
    C = torch.empty_like(W)
    _launch(lib, W, C, np_, 1)
    del W
    table = torch.tensor([float(k * (2 ** b - 128) ** 2) for k in range(np_ + 1)], dtype=torch.float64, device="cuda")
    idx = torch.arange(np_, device="cuda")
    sent = int(SENTINEL.view(np.int64))
    for r0 in range(0, np_, 4096):
        r1 = min(np_, r0 + 4096)
        i = idx[r0:r1, None]
        want = (sg[r0:r1, None] * sg[None, :] * table[np_ - torch.maximum(i, idx[None, :])]).view(torch.int64)
        want[~(i // TILE >= idx[None, :] // TILE)] = sent
        diff = C[r0:r1].view(torch.int64) != want
        assert not diff.any(), f"np={np_}: {int(diff.sum())} cells differ in rows {r0}..{r1}, first {diff.nonzero()[0].tolist()}"
    del C
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ GPU part: the engine


def _tiles(np_, rng):
    """Above np 4096: every diagonal tile, the first tile column, the last (ragged) tile row, 16 random tiles."""
    t = -(-np_ // TB)
    tiles = {(r, r) for r in range(t)} | {(r, 0) for r in range(t)} | {(t - 1, c) for c in range(t)}
    while len(tiles) < 3 * t + 16:
        r = int(rng.integers(0, t))
        tiles.add((r, int(rng.integers(0, r + 1))))
    return sorted(tiles)


ENGINE_CASES = [(2048, 3, 2.5, 1e-5), (2049, 3, 0.5, 1e-2), (2049, 3, 0.5, 1e-5), (2049, 3, 2.5, 1e-2),
                (2049, 3, 2.5, 1e-5), (2250, 3, 2.5, 1e-5), (4096, 16, 2.5, 1e-5), (9200, 3, 2.5, 1e-5)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,d,nu,noise", ENGINE_CASES)
def test_engine_kinv_is_the_scheme_of_its_w(n, d, nu, noise):
    """debug_factor's K^-1 equals the restatement applied to its W padded with the identity, bit for bit."""
    A = np.float64
    x, y = synth(n, d, A=A)
    theta = _rounded(random_thetas(1, d, seed=n + d, noise=(noise, noise * 1.01))[0], A)
    t0 = time.perf_counter()
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        out = ctx.debug_factor(theta, nu=nu, want=("w", "kinv"))
    dt = time.perf_counter() - t0
    assert out["status"] == 0
    np_ = _np(n)
    wp = np.eye(np_)
    wp[:n, :n] = out["w"]
    ex = Exact(wp)
    got = out["kinv"]
    if np_ <= 4096:
        want = _oz_kinv_exact(wp)[:n, :n]
        sym = np.tril(want) + np.tril(want, -1).T  # debug_factor mirrors the lower triangle
        _assert_bits(got, sym, f"n={n}")
    else:
        for r, c in _tiles(np_, np.random.default_rng(n)):
            rows, cols = slice(r * TB, min(n, (r + 1) * TB)), slice(c * TB, min(n, (c + 1) * TB))
            blk = ex.block(rows, cols)
            _assert_bits(np.ascontiguousarray(got[rows, cols]), blk, f"n={n} tile ({r}, {c})")
    _note(f"kinv bits: engine n={n} d={d} nu={nu} noise={noise:g}", {"bits": ex.bits, "factor s": dt})


def _grad(theta, x, alpha, kinv):
    """The gradient contraction of _reference (nu = 2.5) for given alpha and K^-1."""
    n, d = x.shape
    noise, c, ls = math.exp(theta[0]), math.exp(theta[1]), np.exp(theta[2:])
    kc = _kernel_f64(x, x, c, ls, 2.5)
    tmp = np.outer(alpha, alpha) - kinv
    g = [0.5 * noise * float(np.trace(tmp)), 0.5 * float((tmp * kc).sum())]
    rr = np.sqrt(sum(((x[:, j, None] - x[None, :, j]) / ls[j]) ** 2 for j in range(d)))
    f = 5.0 / 3.0 * c * np.exp(-math.sqrt(5.0) * rr) * (math.sqrt(5.0) * rr + 1.0)
    for j in range(d):
        g.append(0.5 * float((tmp * f * ((x[:, j, None] - x[None, :, j]) / ls[j]) ** 2).sum()))
    return np.array(g)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2049, 4096])
def test_gradient_at_small_noise(n):
    """kappa ~ 2e8 / 4e8: the gradient within 1e-9 of the f64 reference; the same contraction with the GPU's W and
    alpha but an f64 W^T W is recorded beside it (the cost of the emulation)."""
    A, d = np.float64, 3
    x, y = synth(n, d, A=A)
    theta = _rounded(random_thetas(1, d, seed=n, noise=(1e-5, 1.01e-5))[0], A)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        lml, grad, status = ctx.lml_grad_batch(theta[None])
        w = ctx.debug_factor(theta, want=("w",))["w"]
        m = ctx.model(theta)
        alpha = m.alpha.copy()
        m.close()
    assert status[0] == 0
    ref = _reference(theta, x, y)
    scale = np.abs(ref.grad).max()
    np.testing.assert_allclose(grad[0], ref.grad, rtol=1e-9, atol=1e-9 * scale)
    host = _grad(theta, x, alpha, w.T @ w)
    _note(f"kinv bits: gradient n={n} noise=1e-5",
          {"emulated |dg|/max|g|": float(np.abs(grad[0] - ref.grad).max() / scale),
           "f64 W^T W from the GPU's W |dg|/max|g|": float(np.abs(host - ref.grad).max() / scale)})
