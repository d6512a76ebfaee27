"""The f64 K^-1 = W^T W product on the integer tensor cores (Ozaki scheme II, hbetune_rs_b200/csrc/gemm_i8.cuh).

The CPU part restates the scheme in NumPy and Python integers: the constants of the header, the split into residues,
the per-modulus products, the Chinese-remainder merge and its single rounding, the bounds that keep every integer
exact up to the largest padded size the library accepts, and the size from which Engine::lauum takes this path.  The
GPU part compares K^-1 and the gradient with the f64 reference on both sides of that size, and checks that the
emulated product reads no stale workspace and gives every matrix of a batch the bits it has alone.
"""
import math
import os
import re

import numpy as np
import pytest

from tests.test_dispatch_sweep import _ctx, _note, _np, _reference, _rounded, _worst_tile
from tests.util import random_thetas, synth

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "hbetune_rs_b200", "csrc", "gemm_i8.cuh")
ENGINE = os.path.join(os.path.dirname(HEADER), "hbegp.cu")
TB = 128
NP_MAX = _np(46000)  # Engine::set_data accepts n <= 46000


def _src(path):
    with open(path) as f:
        return f.read()


def _header():
    src = _src(HEADER)
    mod = [int(v) for v in re.findall(r"m == \d+ \? (\d+)", src)] + [int(re.search(r": (\d+);\s*\n\}", src).group(1))]
    h = {"S": int(re.search(r"constexpr int S = (\d+);", src).group(1)), "moduli": mod}
    for name in ("P_LO", "P_HI", "HALF_LO", "HALF_HI"):
        h[name] = int(re.search(name + r" = (0x[0-9a-f]+)ull", src).group(1), 16)
    h["INV_P58"] = float(re.search(r"INV_P58 = ([0-9.e+-]+);", src).group(1))
    h["crt"] = [[int(v, 16) for v in row] for row in re.findall(r"\{(0x[0-9a-f]+)u, (0x[0-9a-f]+)u, (0x[0-9a-f]+)u, (0x[0-9a-f]+)u\}", src)]
    h["MAX_BITS"] = int(re.search(r"MAX_BITS = (\d+);", src).group(1))
    h["E_CLAMP"] = int(re.search(r"E_CLAMP = (\d+);", src).group(1))
    return h


H = _header()
P = math.prod(H["moduli"])


def _oz_min_np():
    return int(re.search(r"OZ_MIN_NP = (\d+);", _src(ENGINE)).group(1))


def _emulated(np_, f32=False):
    """Engine::kinv_emulated (hbegp.cu): f64 from OZ_MIN_NP on; depends on the type and the padded size only."""
    return not f32 and np_ >= _oz_min_np()


# ------------------------------------------------------------------------------------------------ the scheme restated


def _scale_bits(np_):
    """oz::scale_bits: the largest b <= MAX_BITS with np 2^2b < P / 2."""
    b = H["MAX_BITS"]
    while b > 0 and np_ << (2 * b) >= P // 2:
        b -= 1
    return b


def _exponents(w, bits):
    """k_oz_split pass 1: e_j = bits - E_j with max_k |W[k][j]| < 2^E_j, clamped."""
    m = np.abs(w).max(axis=0)
    _, E = np.frexp(m)
    e = np.clip(bits - E, -H["E_CLAMP"], H["E_CLAMP"])
    return np.where(m > 0, e, 0).astype(np.int64)


def _scaled(w, e):
    """W' = rn(2^e_j W[k][j]) as exact int64."""
    return np.rint(np.ldexp(w, e[None, :])).astype(np.int64)


def _residue_pieces(x, p):
    """k_oz_split's residue of x (|x| < 2^51) through u = x + 2^51 cut into 24 + 12 + 16 bits, symmetric range."""
    u = x + (1 << 51)
    lo, h0, h1 = u & 0xFFFFFF, (u >> 24) & 0xFFF, u >> 36
    t = lo + h0 * ((1 << 24) % p) + h1 * ((1 << 36) % p) + (p - (1 << 51) % p)
    assert t.max() < 1 << 26
    r = t % p
    return np.where(r > (p - 1) // 2, r - p, r)


def _epilogue_mod(v, p):
    """k_oz_syrk_i8's epilogue: v mod p through a float32 quotient, corrected by one modulus either way."""
    q = np.floor(v.astype(np.float32) * np.float32(1.0 / np.float32(p))).astype(np.int64)
    r = v - q * p
    r = np.where(r < 0, r + p, r)
    return np.where(r >= p, r - p, r)


def _crt(res):
    """k_oz_merge's C' from residues r_m in [0, p_m): limb sums, one quotient estimate, symmetric range."""
    acc = [sum(int(r) * H["crt"][m][l] for m, r in enumerate(res)) for l in range(4)]
    s = acc[0] + (acc[1] << 32) + (acc[2] << 64) + (acc[3] << 96)
    assert s < 1 << 122 and max(acc) < 1 << 64
    q = int(float(s >> 58) * H["INV_P58"])
    v = s - q * P
    if v < 0:
        v += P
    if v >= P:
        v -= P
    return v - P if v > P // 2 else v


def _to_double(v, e):
    """k_oz_merge's single rounding: the top 64 bits with a sticky bit, rounded to nearest even, times 2^(sh - e)."""
    a = abs(v)
    sh = max(0, a.bit_length() - 64)
    m = (a >> sh) | (1 if a & ((1 << sh) - 1) else 0)
    d = float(m) * 2.0 ** (sh - e)
    return -d if v < 0 else d


def test_header_constants():
    assert H["S"] == 14 and len(H["moduli"]) == 14 and len(H["crt"]) == 14
    assert H["moduli"] == sorted(H["moduli"], reverse=True) and max(H["moduli"]) <= 256
    for i, a in enumerate(H["moduli"]):
        for b in H["moduli"][i + 1:]:
            assert math.gcd(a, b) == 1, (a, b)
    # the 14 largest pairwise coprime integers <= 256, greedily from the top
    greedy, c = [], 256
    while len(greedy) < 14:
        if all(math.gcd(c, q) == 1 for q in greedy):
            greedy.append(c)
        c -= 1
    assert H["moduli"] == greedy
    assert (H["P_HI"] << 64 | H["P_LO"]) == P and (H["HALF_HI"] << 64 | H["HALF_LO"]) == P // 2
    assert H["INV_P58"] == 2.0 ** 58 / P
    for m, p in enumerate(H["moduli"]):
        c = sum(limb << (32 * l) for l, limb in enumerate(H["crt"][m]))
        assert c < P and c % p == 1 and all(c % q == 0 for q in H["moduli"] if q != p), p


def test_bounds_hold_up_to_the_largest_size():
    """int32 accumulators, P / 2, the 2^51 window of the split and the exponent range, for every padded size."""
    assert NP_MAX == 46016 and -(-NP_MAX // TB) * TB * TB * TB < 2 ** 31  # |C_m| <= np_tiles 128^2
    for np_ in range(64, -(-NP_MAX // TB) * TB + 1, 64):
        b = _scale_bits(np_)
        assert np_ * 2 ** (2 * b) < P // 2 and 0 < b <= 50, np_
    assert _scale_bits(4096) == 48 and _scale_bits(46080) == 46
    assert 14 * 255 * P < 2 ** 122  # the merge's limb sum
    # 2^(sh - e_i - e_j) stays a normal double: sh <= 46, |e| <= E_CLAMP
    assert 46 + 2 * H["E_CLAMP"] < 1022


def test_split_residues_and_epilogue_reduction():
    rng = np.random.default_rng(5)
    x = np.concatenate([rng.integers(-(2 ** 50), 2 ** 50, 4000), [0, 1, -1, 2 ** 50, -(2 ** 50)]])
    vmax = -(-NP_MAX // TB) * TB * 128 * 128  # |C_m| <= np 128^2 (exact in the float32 quotient's reach up to here)
    v = np.concatenate([rng.integers(-vmax, vmax + 1, 20000), [0, vmax, -vmax, vmax - 1, 1 - vmax]])
    for p in H["moduli"]:
        r = _residue_pieces(x, p)
        assert ((r - x) % p == 0).all() and r.min() >= -128 and r.max() <= 127, p
        assert (_epilogue_mod(v, p) == v % p).all(), p


def test_single_rounding_matches_python_float():
    rng = np.random.default_rng(6)
    vals = [int(rng.integers(0, 2 ** 62)) << int(rng.integers(0, 48)) | int(rng.integers(0, 2 ** 40)) for _ in range(2000)]
    vals += [(1 << 109) + (1 << 56) + 1, (1 << 109) + (1 << 56), (1 << 53) + 1, 2 ** 64 - 1, 0]  # ties and near-ties
    for v in vals:
        for s in (v, -v):
            assert _to_double(s, 0) == float(s), s
            assert _to_double(s, 37) == math.ldexp(float(s), -37), s


@pytest.mark.parametrize("n,noise", [(90, 1e-2), (200, 1e-4)])
def test_scheme_matches_python_integers(n, noise):
    """split -> per-modulus int64 products -> CRT merge equals W'^T W' in Python integers, and the result is
    within the truncation error of K^-1."""
    x, y = synth(n, 3, seed=n)
    theta = random_thetas(1, 3, seed=n, noise=(noise, noise * 1.01))[0]
    w = _reference(theta, x, y).w
    np_ = -(-n // TB) * TB  # the planes are padded with zeros to whole tiles
    wp = np.zeros((np_, np_))
    wp[:n, :n] = w
    e = _exponents(wp, _scale_bits(np_))
    ws = _scaled(wp, e)
    assert np.abs(ws).max() <= 2 ** _scale_bits(np_)
    planes = [_residue_pieces(ws.T, p) for p in H["moduli"]]  # R_m[j][k] = W'[k][j] mod p
    prods = [_epilogue_mod(r @ r.T, p) for r, p in zip(planes, H["moduli"])]  # int64 is exact here
    wo = ws.astype(object)
    exact = wo.T @ wo
    rng = np.random.default_rng(n)
    for i, j in [(0, 0), (n - 1, n - 1), (n - 1, 0)] + [tuple(sorted(rng.integers(0, n, 2))[::-1]) for _ in range(150)]:
        c = _crt([int(pr[i, j]) for pr in prods])
        assert c == exact[i, j], (i, j)
        got = _to_double(c, int(e[i] + e[j]))
        assert got == math.ldexp(float(exact[i, j]), -int(e[i] + e[j]))
    kinv = w.T @ w
    approx = np.ldexp(exact[:n, :n].astype(np.float64), -(e[:n, None] + e[None, :n]))
    assert np.abs(approx - kinv).max() <= 1e-13 * np.abs(kinv).max()


# the padded sizes of the GPU part, on both sides of OZ_MIN_NP; 1088 and 2112 are not multiples of 128
GPU_SHAPES = [(600, 3), (1025, 3), (2049, 2)]


def test_gpu_shapes_reach_both_paths():
    paths = {_emulated(_np(n)) for n, _ in GPU_SHAPES}
    assert paths == {False, True}
    assert any(_emulated(_np(n)) and _np(n) % TB for n, _ in GPU_SHAPES)
    assert not _emulated(4096, f32=True) and _emulated(4096) and _emulated(2112) and not _emulated(1088)


# ------------------------------------------------------------------------------------------------ GPU part


@pytest.mark.gpu
@pytest.mark.parametrize("noise", [1e-2, 1e-4])
@pytest.mark.parametrize("n,d", GPU_SHAPES)
def test_kinv_and_gradient_against_reference(n, d, noise):
    A = np.float64
    x, y = synth(n, d, A=A)
    thetas = np.stack([_rounded(t, A) for t in random_thetas(3, d, seed=n, noise=(noise, noise * 1.01))])
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        out = ctx.debug_factor(thetas[0], want=("kinv",))
        lml, grad, status = ctx.lml_grad_batch(thetas)
    assert out["status"] == 0 and (status == 0).all()
    note = {"emulated": _emulated(_np(n))}
    truth = _reference(thetas[0], x, y)
    err = np.abs(out["kinv"] - truth.kinv)
    note["kinv"] = float(err.max() / np.abs(truth.kinv).max())
    assert err.max() <= 1e-9 * np.abs(truth.kinv).max(), _worst_tile(err)
    note["grad"] = 0.0
    for b in range(3):
        ref = _reference(thetas[b], x, y)
        g_scale = np.abs(ref.grad).max()
        assert abs(lml[b] - ref.lml) <= 1e-9 * abs(ref.lml)
        np.testing.assert_allclose(grad[b], ref.grad, rtol=1e-9, atol=1e-9 * g_scale)
        note["grad"] = max(note["grad"], float(np.abs(grad[b] - ref.grad).max() / g_scale))
    _note(f"kinv emulation n={n} noise={noise:g}", note)


@pytest.mark.gpu
def test_emulated_kinv_reads_no_stale_workspace():
    """NaN-poisoned workspaces (K, W and the residue planes): the same bits as before, evaluation after evaluation."""
    A = np.float64
    n, d = 2049, 3
    x, y = synth(n, d, A=A)
    thetas = np.stack([_rounded(t, A) for t in random_thetas(4, d, seed=7)])
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        ref = ctx.debug_factor(thetas[0], want=("kinv",))["kinv"]
        ref_b = ctx.lml_grad_batch(thetas)
        for _ in range(2):
            ctx.debug_poison()
            got = ctx.debug_factor(thetas[0], want=("kinv",))["kinv"]
            np.testing.assert_array_equal(got, ref)
            ctx.debug_poison()
            lml, grad, status = ctx.lml_grad_batch(thetas)
            np.testing.assert_array_equal(lml, ref_b[0])
            np.testing.assert_array_equal(grad, ref_b[1])
    assert np.isfinite(ref).all()


@pytest.mark.gpu
@pytest.mark.parametrize("n,B", [(2049, 9), (2049, 20)])  # stream groups of 2-3 with the side stream, of 5 without
def test_batch_members_have_their_single_bits(n, B):
    A = np.float64
    x, y = synth(n, 3, A=A)
    thetas = np.stack([_rounded(t, A) for t in random_thetas(B, 3, seed=B)])
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        lml, grad, status = ctx.lml_grad_batch(thetas)
        for b in range(B):
            l1, g1, s1 = ctx.lml_grad_batch(thetas[b][None])
            assert s1[0] == status[b] == 0 and l1[0] == lml[b]
            np.testing.assert_array_equal(g1[0], grad[b])
        # a model's K^-1 is the one debug_factor computes
        m = ctx.model(thetas[0], want_alpha=False, want_kinv=True)
        np.testing.assert_array_equal(m.k_inv, ctx.debug_factor(thetas[0], want=("kinv",))["kinv"])
