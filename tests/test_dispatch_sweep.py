"""Every kernel variant the engine dispatches to, against a plain f64 reference, on both sides of each switch.

Which kernel runs a product depends on the shape: the recursion of Engine::chol_inv splits a block into a 64-wide
leaf, a 128-wide fused node or a merge of two halves; each merge issues four GEMM classes and the inverse one more,
and every GEMM runs on 32x32 tiles, 64x64 tiles or (f32) the tcgen05 3xTF32 kernel, whose 128-wide tiles are ragged
when an extent is 64 mod 128.  `_plan` restates those rules, and `test_sweep_reaches_every_variant` checks that the
shapes below reach every variant; if a threshold moves, that test fails and SHAPES has to move with it.

`_reference` evaluates the LML, its gradient, alpha, W = L^-1 and K^-1 in f64 without the oracle's (n, n, d + 1)
tensor.  f32 results are compared with the f64 truth for the f32 inputs and f32-rounded parameters (what
Engine::fill_params hands the kernels), and must be no worse than LAPACK f32 (spotrf / strtri) is on the f32 K.
"""
import json
import math
import os
from types import SimpleNamespace

import numpy as np
import pytest
from scipy.linalg import cho_factor, cho_solve, lapack

from tests.util import oracle_kernel, oracle_lml, random_thetas, synth

TILE = 64
EPS32 = float(np.finfo(np.float32).eps)

# ------------------------------------------------------------------------------------------------ dispatch restated


def _split(s):
    """Engine::chol_inv (hbegp.cu:495-498): q tiles split into q1 + (q - q1), q1 even from q >= 4 so that the
    128-multiple block comes first."""
    q = s // TILE
    q1 = (q + 1) // 2
    if q >= 4 and q1 % 2:
        q1 += 1
    if q1 >= q:
        q1 = q - 1
    return q1 * TILE, s - q1 * TILE


def _recursion(s, ops):
    """chol_inv (hbegp.cu:477-502) and merge_node (:506-547): ("leaf",), ("node",) or ("gemm", class, M, N, lower)."""
    if s == TILE:
        ops.append(("leaf",))
        return
    if s == 2 * TILE:
        ops.append(("node",))
        return
    s1, s2 = _split(s)
    _recursion(s1, ops)
    ops += [("gemm", 0, s2, s1, False), ("gemm", 1, s2, s1, False), ("gemm", 2, s2, s2, True)]
    _recursion(s2, ops)
    ops.append(("gemm", 3, s2, s1, False))


def _gemm_kind(np_, M, N, lower, batch, f32):
    if f32 and min(M, N) >= 256:  # gemm_uses_tf32 (gemm_tf32.cuh:488-490)
        return "tf32" if M % 128 == 0 and N % 128 == 0 else "tf32 ragged"
    small_ctas = 296 if np_ <= 1024 else 0  # GemmArgs::small_ctas (hbegp.cu:519, :562)
    tm, tn = M // 64, N // 64
    tiles = tm * (tm + 1) // 2 if lower else tm * tn
    return "32x32" if tiles * batch <= small_ctas else "64x64"  # launch_gemm (gemm.cuh:388-396)


def _padded(np_, cnt):
    """padded_batch (hbegp.cu:333-345) for the first request of a batch size."""
    return (cnt + 3) // 4 * 4 if np_ <= 2048 and cnt > 4 else cnt


def _groups(np_, cnt):
    """n_groups (hbegp.cu:636-648) with 16 streams, and the split of issue_chunk (:662-664)."""
    gm = 1 if np_ >= 1024 else 2
    g = min(16, max(1, cnt // gm)) if np_ <= 2048 else 4
    g = max(1, min(g, cnt))
    return [cnt // g + (i < cnt % g) for i in range(g)]


def _plan(np_, cnt, f32):
    """The set of variants one batched evaluation of `cnt` matrices of padded size np_ runs through."""
    run = _padded(np_, cnt)
    v = {"graph" if np_ <= 2048 else "direct", "one group" if len(_groups(np_, run)) == 1 else "groups"}
    if run != cnt:
        v.add("padded batch")
    for c in set(_groups(np_, run)):
        if np_ > 2048:  # pipeline (hbegp.cu:630): the side stream above 2048 only for groups of <= 4
            v.add("side stream" if c <= 4 else "no side stream")
        ops = []
        _recursion(np_, ops)
        ops.append(("gemm", 4, np_, np_, True))  # lauum (:571-581)
        for op in ops:
            v.add(op[0] if op[0] != "gemm" else (op[1], _gemm_kind(np_, op[2], op[3], op[4], c, f32)))
    return v


def _predict_path(m, d, np_, itemsize, want_var=True):
    """ModelT::predict_impl (hbegp.cu:994-1067)."""
    if m <= 64 and m * d * itemsize <= 40 * 1024:
        return "latency"
    p = "split" if np_ > 16 * TILE else "one"  # train tiles over grid.y in groups of 16
    return p + (" chunked" if not want_var and m > (1 << 20) else "")


def _np(n):
    return -(-n // TILE) * TILE


# (n, d, batch): the batched LML test runs each at `batch` and at B = 1
SHAPES = [
    (129, 3, 5),    # np 192: node then a lone leaf, 32x32 tiles, padded batch
    (511, 4, 3),    # np 512: TF32 in all five classes, full tiles
    (576, 3, 3),    # ragged TF32 in K^-1 only
    (700, 3, 5),    # np 704: ragged TF32 in all five classes
    (960, 3, 33),   # full and ragged TF32; 2-3 matrices per group: K^-1 on 32x32 and on 64x64 tiles
    (1025, 3, 3),   # np 1088: no 32x32 tiles, groups of one, graphs
    (2049, 2, 9),   # np 2112: direct launches, groups of <= 4 with the side stream
    (2049, 2, 20),  # groups of 5, no side stream
]


def _required():
    req = {"leaf", "node", "graph", "direct", "one group", "groups", "side stream", "no side stream", "padded batch"}
    for cls in range(5):
        req |= {(cls, "32x32"), (cls, "64x64"), (cls, "tf32"), (cls, "tf32 ragged")}
    return req


def test_sweep_reaches_every_variant():
    reached = {}
    for n, _, b in SHAPES:
        for f32 in (False, True):
            for cnt in (b, 1):
                for v in _plan(_np(n), cnt, f32):
                    reached.setdefault(v, set()).add((n, b, "f32" if f32 else "f64"))
    missing = sorted(map(str, _required() - set(reached)))
    assert not missing, f"no shape reaches {missing}"
    # f64 has no TF32 path: both GEMM tile sizes must be reached by f64 shapes for every class
    for cls in range(5):
        for kind in ("32x32", "64x64"):
            assert any(p == "f64" for _, _, p in reached[(cls, kind)]), (cls, kind)
    # the shape notes above stay true
    assert (_np(129), _split(192)) == (192, (128, 64))
    assert all((c, "tf32") in _plan(512, 1, True) for c in range(5))
    assert all((c, "tf32 ragged") in _plan(704, 1, True) for c in range(5))
    assert {v for v in _plan(576, 1, True) if isinstance(v, tuple) and v[1] == "tf32 ragged"} == {(4, "tf32 ragged")}
    assert {(4, "32x32"), (4, "64x64")} <= _plan(960, 33, False)
    assert not any(isinstance(v, tuple) and v[1] == "32x32" for v in _plan(1088, 3, False))


# ------------------------------------------------------------------------------------------------ the f64 reference


def _kernel_f64(x1, x2, c, ls, nu):
    """c * Matern_nu(|x1 / l - x2 / l|) in f64 (matern_kernel.rs:37-80: divide first, sum squares over features)."""
    a, b = x1 / ls, x2 / ls
    r2 = np.zeros((a.shape[0], b.shape[0]))
    for k in range(a.shape[1]):
        r2 += (a[:, k, None] - b[None, :, k]) ** 2
    r = np.sqrt(r2)
    if nu == 0.5:
        return c * np.exp(-r)
    if nu == 1.5:
        t = math.sqrt(3.0) * r
        return c * (1 + t) * np.exp(-t)
    t = math.sqrt(5.0) * r
    return c * (1 + t + t * t / 3) * np.exp(-t)


def _reference(theta, x, y, nu=2.5, k=None):
    """LML, gradient, alpha, K, W = L^-1 and K^-1 in f64 (cho_factor / dtrtri).  Gradient component k is
    1/2 tr((alpha alpha^T - K^-1) dK/dtheta_k), one n x n slice at a time (matern_kernel.rs:83-135).  A given K
    (the symmetric matrix the GPU assembled, say) replaces the host's kc + noise I in the LAPACK steps."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    n, d = x.shape
    noise, c, ls = math.exp(theta[0]), math.exp(theta[1]), np.exp(np.asarray(theta[2:], dtype=np.float64))
    kc = _kernel_f64(x, x, c, ls, nu)
    if k is None:
        k = kc.copy()
        k[np.diag_indices(n)] += noise
    low, _ = cho_factor(k, lower=True)
    low = np.tril(low)
    r = SimpleNamespace(k=k)
    r.alpha = cho_solve((low, True), y)
    r.w, info = lapack.dtrtri(low, lower=1)
    assert info == 0
    r.kinv = r.w.T @ r.w
    logdet = np.log(np.diag(low))
    r.lml = -0.5 * float(y @ r.alpha) - float(logdet.sum()) - n / 2.0 * math.log(2.0 * math.pi)
    r.lml_scale = 0.5 * abs(float(y @ r.alpha)) + float(np.abs(logdet).sum()) + n / 2.0 * math.log(2.0 * math.pi)
    tmp = np.outer(r.alpha, r.alpha) - r.kinv
    g = [0.5 * noise * float(np.trace(tmp)), 0.5 * float((tmp * kc).sum())]
    rr = np.sqrt(sum(((x[:, j, None] - x[None, :, j]) / ls[j]) ** 2 for j in range(d)))
    if nu == 0.5:
        with np.errstate(divide="ignore", invalid="ignore"):
            f = np.where(rr > 0, kc / rr, 0.0)  # the r = 0 branch (kernels.cuh:75): duplicate rows contribute 0
    elif nu == 1.5:
        f = 3.0 * c * np.exp(-math.sqrt(3.0) * rr)
    else:
        f = 5.0 / 3.0 * c * np.exp(-math.sqrt(5.0) * rr) * (math.sqrt(5.0) * rr + 1.0)
    for j in range(d):
        g.append(0.5 * float((tmp * f * ((x[:, j, None] - x[None, :, j]) / ls[j]) ** 2).sum()))
    r.grad = np.array(g)
    return r


def _rounded(theta, A):
    """theta whose natural parameters are the ones Engine::fill_params rounds to T."""
    return np.log(np.exp(np.asarray(theta, dtype=np.float64)).astype(A).astype(np.float64))


@pytest.mark.parametrize("A", [np.float64, np.float32])
@pytest.mark.parametrize("nu", [0.5, 1.5, 2.5])
def test_reference_matches_oracle(nu, A):
    for n, d, seed in ((1, 1, 1), (70, 2, 2), (200, 4, 3)):
        x, y = synth(n, d, seed=seed, A=A)
        if n > 10:
            x[7] = x[3]  # a duplicate row: the r = 0 branch of the nu = 0.5 gradient
        theta = _rounded(random_thetas(1, d, seed=seed, noise=(5e-2, 1.0))[0], A)
        x64, y64 = x.astype(np.float64), y.astype(np.float64)
        want = oracle_lml(theta, x64, y64, nu=nu)
        got = _reference(theta, x64, y64, nu)
        assert abs(got.lml - want.lml) <= 1e-12 * abs(want.lml), (n, got.lml, want.lml)
        g = np.array(want.lml_gradient)
        np.testing.assert_allclose(got.grad, g, rtol=1e-12, atol=1e-12 * np.abs(g).max())
        np.testing.assert_allclose(got.alpha, want.alpha, rtol=0, atol=1e-12 * np.abs(want.alpha).max())
        kinv = want.factorization.invc()
        np.testing.assert_allclose(got.kinv, kinv, rtol=0, atol=1e-12 * np.abs(kinv).max())


def test_plan_notes_the_predict_paths():
    assert _predict_path(64, 3, 320, 8) == "latency" and _predict_path(65, 3, 320, 8) == "one"
    assert _predict_path(60, 100, 320, 8) == "one" and _predict_path(60, 100, 320, 4) == "latency"
    assert _predict_path(60, 200, 320, 4) == "one"
    assert _predict_path(65, 3, 1088, 4) == "split"
    assert _predict_path((1 << 20) + 65, 2, 1088, 4, want_var=False) == "split chunked"


# ------------------------------------------------------------------------------------------------ GPU part

DTYPES = [np.float64, np.float32]


def _note(key, payload):
    """Adds the measured errors to the JSON file named by HBEGP_SWEEP_NOTES (profiles/r03_dispatch_sweep.json holds
    one such record); without that variable nothing is written."""
    path = os.environ.get("HBEGP_SWEEP_NOTES")
    if not path:
        return
    try:
        data = {}
        if os.path.exists(path):
            with open(path) as f:
                data = json.load(f)
        data[key] = payload
        with open(path, "w") as f:
            json.dump(data, f, indent=1, sort_keys=True)
    except (OSError, ValueError):
        pass


def _ctx(A):
    import hbetune_rs_b200 as h
    return h.Context(0, h.F64 if A == np.float64 else h.F32)


def _name(A):
    return "f64" if A == np.float64 else "f32"


def _thetas(B, d, A, seed):
    # f32 keeps the noise >= 0.1 like the other f32 parity tests (K's condition number stays within f32's reach)
    return random_thetas(B, d, seed=seed, noise=(1e-2, 1.0) if A == np.float64 else (1e-1, 1.0))


def _worst_tile(err):
    t = -(-err.shape[0] // TILE)
    pad = np.zeros((t * TILE, t * TILE))
    pad[: err.shape[0], : err.shape[1]] = err
    per = pad.reshape(t, TILE, t, TILE).max(axis=(1, 3))
    i, j = np.unravel_index(int(per.argmax()), per.shape)
    return f"worst 64x64 tile ({i}, {j}) = rows {i * TILE}.., cols {j * TILE}.., max error {per[i, j]:.3e}"


# f32 against the f64 truth: error <= RATIO * (LAPACK f32's error) + FLOOR * eps32 * scale
RATIO, FLOOR = 2.0, 4.0


def _lapack_f32(theta, x, nu):
    """K as the f32 oracle assembles it, then spotrf + strtri and W^T W in f32."""
    n = x.shape[0]
    k = oracle_kernel(theta, nu).kernel(x, x, np.float32) + np.float32(math.exp(theta[0])) * np.eye(n, dtype=np.float32)
    low, info = lapack.spotrf(k, lower=1, clean=1)
    assert info == 0
    w, info = lapack.strtri(low, lower=1)
    assert info == 0
    return k, w, w.T @ w


FACTOR_SHAPES = sorted({(n, d) for n, d, _ in SHAPES})


@pytest.mark.gpu
@pytest.mark.parametrize("A", DTYPES)
@pytest.mark.parametrize("n,d", FACTOR_SHAPES)
def test_factor_intermediates(n, d, A):
    x, y = synth(n, d, A=A)
    theta = _rounded(_thetas(1, d, A, seed=n)[0], A)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        out = ctx.debug_factor(theta)
    assert out["status"] == 0
    ref = _reference(theta, x, y)
    truth = {"k": np.tril(ref.k), "w": ref.w, "kinv": ref.kinv}
    note = {}
    if A == np.float64:
        np.testing.assert_allclose(out["k"], truth["k"], rtol=1e-12, atol=1e-14)
        for key in ("w", "kinv"):
            err = np.abs(out[key] - truth[key])
            note[key] = float(err.max() / np.abs(truth[key]).max())
            assert err.max() <= 1e-9 * np.abs(truth[key]).max(), (key, _worst_tile(err))
        _note(f"factor n={n} f64", note)
        return
    k32, w32, kinv32 = _lapack_f32(theta, x, 2.5)
    lapack32 = {"k": np.tril(k32), "w": w32, "kinv": kinv32}
    fails = []
    for key in ("k", "w", "kinv"):
        err = np.abs(out[key].astype(np.float64) - truth[key])
        e_lapack = float(np.abs(lapack32[key].astype(np.float64) - truth[key]).max())
        scale = float(np.abs(truth[key]).max())
        note[key] = {"cuda": float(err.max()), "lapack_f32": e_lapack, "ratio": float(err.max()) / e_lapack, "scale": scale}
        if err.max() > RATIO * e_lapack + FLOOR * EPS32 * scale:
            fails.append((key, note[key], _worst_tile(err)))
    _note(f"factor n={n} f32", note)
    assert not fails, fails


def _check_f32_against_truth(got_lml, got_grad, o32, truth, tag):
    """f32: the CUDA LML / gradient no further from the f64 truth than RATIO x the f32 oracle (LAPACK f32)."""
    e_lml, o_lml = abs(got_lml - truth.lml), abs(o32.lml - truth.lml)
    g32 = np.array(o32.lml_gradient)
    e_g, o_g = float(np.abs(got_grad - truth.grad).max()), float(np.abs(g32 - truth.grad).max())
    gscale = float(np.abs(truth.grad).max())
    rec = {"lml": e_lml, "lml_lapack_f32": o_lml, "grad": e_g, "grad_lapack_f32": o_g,
           "lml_scale": truth.lml_scale, "grad_scale": gscale}
    ok = (e_lml <= RATIO * o_lml + FLOOR * EPS32 * truth.lml_scale and e_g <= RATIO * o_g + FLOOR * EPS32 * gscale)
    return rec, ok


@pytest.mark.gpu
@pytest.mark.parametrize("A", DTYPES)
@pytest.mark.parametrize("n,d,B", SHAPES)
def test_batched_lml_and_gradient(n, d, B, A):
    x, y = synth(n, d, A=A)
    thetas = np.stack([_rounded(t, A) for t in _thetas(B, d, A, seed=B + n)])
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        lml, grad, status = ctx.lml_grad_batch(thetas)
        singles = [ctx.lml_grad_batch(t[None]) for t in thetas]
    assert (status == 0).all()
    for b, (l1, g1, s1) in enumerate(singles):  # the same bits whatever the batch (fit capture rule, NLopt batcher)
        assert s1[0] == 0 and l1[0] == lml[b], (b, l1[0], lml[b])
        np.testing.assert_array_equal(g1[0], grad[b])
    check = range(B) if _np(n) <= 1088 else sorted({0, B // 2, B - 1})
    worst, fails = {}, []
    for b in check:
        truth = _reference(thetas[b], x, y)
        g_scale = np.abs(truth.grad).max()
        if A == np.float64:
            assert abs(lml[b] - truth.lml) <= 1e-9 * abs(truth.lml), (b, lml[b], truth.lml)
            np.testing.assert_allclose(grad[b], truth.grad, rtol=1e-9, atol=1e-9 * g_scale)
            rel = max(abs(lml[b] - truth.lml) / abs(truth.lml), float(np.abs(grad[b] - truth.grad).max() / g_scale))
            worst["rel"] = max(worst.get("rel", 0.0), rel)
            continue
        o32 = oracle_lml(thetas[b], x, y, A=np.float32)
        assert abs(lml[b] - o32.lml) <= 1e-4 * abs(o32.lml), (b, lml[b], o32.lml)
        g32 = np.array(o32.lml_gradient)
        np.testing.assert_allclose(grad[b], g32, rtol=1e-4, atol=1e-4 * np.abs(g32).max())
        rec, ok = _check_f32_against_truth(lml[b], grad[b], o32, truth, b)
        for key, v in rec.items():
            worst[key] = max(worst.get(key, 0.0), v)
        if not ok:
            fails.append((b, rec))
    _note(f"lml n={n} B={B} {_name(A)}", worst)
    assert not fails, fails


def _predict_truth(theta, x, xs, truth, nu=2.5):
    ks = _kernel_f64(np.asarray(xs, np.float64), np.asarray(x, np.float64), math.exp(theta[1]),
                     np.exp(theta[2:]), nu)
    mean = ks @ truth.alpha
    var = math.exp(theta[1]) + 1e-5 - np.einsum("ij,ij->i", ks @ truth.kinv, ks)
    return mean, np.maximum(var, 0.0)


def _check_predict(mean, var, tm, tv, theta, A, tag):
    # f32: 2e-5 is ten times the worst error measured over these shapes on a B200 (2.1e-6, profiles/r03_dispatch_sweep.json)
    tol = 1e-9 if A == np.float64 else 2e-5
    c = math.exp(theta[1])
    e_mean = float(np.abs(mean - tm).max() / max(1.0, np.abs(tm).max()))
    rec = {"mean": e_mean}
    if var is not None:
        rec["var"] = float(np.abs(var - tv).max() / (c + 1e-5))
    _note(tag, rec)
    assert e_mean <= tol, (tag, rec)
    if var is not None:
        assert rec["var"] <= tol, (tag, rec)


@pytest.mark.gpu
@pytest.mark.parametrize("A", DTYPES)
@pytest.mark.parametrize("n", [1025, 2049])
def test_predict_with_train_tiles_split_over_grid_y(n, A):
    d = 3
    x, y = synth(n, d, A=A)
    theta = _rounded(random_thetas(1, d, seed=5, noise=(3e-2, 0.3) if A == np.float64 else (0.1, 0.5))[0], A)
    xs = np.random.default_rng(2).random((1000, d)).astype(A)
    truth = _reference(theta, x, y)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta)
        for m in (65, 300, 1000):
            assert _predict_path(m, d, _np(n), A().itemsize) == "split"
            mean, var = model.predict(xs[:m])
            tm, tv = _predict_truth(theta, x, xs[:m], truth)
            _check_predict(mean, var, tm, tv, theta, A, f"predict n={n} m={m} {_name(A)}")
        model.close()


@pytest.mark.gpu
@pytest.mark.parametrize("A", DTYPES)
def test_predict_few_rows_with_many_features_take_the_throughput_path(A):
    """m <= 64 rows whose features exceed 40 KB skip the latency path (its shared-memory copy of the rows)."""
    n, m = 300, 60
    d = 100 if A == np.float64 else 200
    assert _predict_path(m, d, _np(n), A().itemsize) == "one"
    x, y = synth(n, d, A=A)
    rng = np.random.default_rng(9)
    theta = _rounded(np.concatenate([[math.log(0.1), math.log(1.3)], rng.uniform(math.log(3.0), math.log(9.0), d)]), A)
    xs = rng.random((m, d)).astype(A)
    truth = _reference(theta, x, y)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta)
        mean, var = model.predict(xs)
        model.close()
    tm, tv = _predict_truth(theta, x, xs, truth)
    _check_predict(mean, var, tm, tv, theta, A, f"predict throughput m={m} d={d} {_name(A)}")


@pytest.mark.gpu
@pytest.mark.parametrize("A", DTYPES)
def test_predict_mean_over_chunks_of_2_20_rows(A):
    n, d, m = 1025, 2, (1 << 20) + 65
    x, y = synth(n, d, A=A)
    theta = _rounded(random_thetas(1, d, seed=6, noise=(3e-2, 0.3) if A == np.float64 else (0.1, 0.5))[0], A)
    xs = np.random.default_rng(3).random((m, d)).astype(A)
    assert _predict_path(m, d, _np(n), A().itemsize, want_var=False) == "split chunked"
    truth = _reference(theta, x, y)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta)
        mean, none = model.predict(xs, want_variance=False)
        model.close()
    assert none is None
    edge = 1 << 20
    rows = np.unique(np.concatenate([np.arange(0, 64), np.arange(edge - 200, m),
                                     np.random.default_rng(4).integers(0, m, 2000)]))
    tm, _ = _predict_truth(theta, x, xs[rows], truth)
    _check_predict(mean[rows], None, tm, None, theta, A, f"predict mean chunks m={m} {_name(A)}")


@pytest.mark.gpu
@pytest.mark.parametrize("nu", [0.5, 1.5])
def test_matern_orders_in_f32(nu):
    A, n, d, B = np.float32, 700, 3, 3
    x, y = synth(n, d, A=A)
    thetas = np.stack([_rounded(t, A) for t in _thetas(B, d, A, seed=17)])
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        lml, grad, status = ctx.lml_grad_batch(thetas, nu=nu)
    assert (status == 0).all()
    fails, worst = [], {}
    for b in range(B):
        o32 = oracle_lml(thetas[b], x, y, nu=nu, A=A)
        assert abs(lml[b] - o32.lml) <= 1e-4 * abs(o32.lml), (b, lml[b], o32.lml)
        g32 = np.array(o32.lml_gradient)
        np.testing.assert_allclose(grad[b], g32, rtol=1e-4, atol=1e-4 * np.abs(g32).max())
        rec, ok = _check_f32_against_truth(lml[b], grad[b], o32, _reference(thetas[b], x, y, nu), b)
        for key, v in rec.items():
            worst[key] = max(worst.get(key, 0.0), v)
        if not ok:
            fails.append((b, rec))
    _note(f"matern nu={nu} n={n} f32", worst)
    assert not fails, fails


@pytest.mark.gpu
@pytest.mark.parametrize("A", DTYPES)
def test_duplicate_training_rows_under_matern_0_5(A):
    """Integer search spaces repeat training rows; with noise > 0 K stays definite and the nu = 0.5 gradient takes its
    r = 0 branch (kernels.cuh:75) on every duplicate pair."""
    n, d = 300, 3
    x, y = synth(n, d, A=A)
    x[100:140] = x[:40]
    thetas = np.stack([_rounded(t, A) for t in random_thetas(3, d, seed=12, noise=(0.1, 0.1))])
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        lml, grad, status = ctx.lml_grad_batch(thetas, nu=0.5)
    assert (status == 0).all()
    for b in range(3):
        truth = _reference(thetas[b], x, y, 0.5)
        if A == np.float64:
            assert abs(lml[b] - truth.lml) <= 1e-9 * abs(truth.lml)
            np.testing.assert_allclose(grad[b], truth.grad, rtol=1e-9, atol=1e-9 * np.abs(truth.grad).max())
        else:
            o32 = oracle_lml(thetas[b], x, y, nu=0.5, A=A)
            assert abs(lml[b] - o32.lml) <= 1e-4 * abs(o32.lml)
            g32 = np.array(o32.lml_gradient)
            np.testing.assert_allclose(grad[b], g32, rtol=1e-4, atol=1e-4 * np.abs(g32).max())
            np.testing.assert_allclose(grad[b], truth.grad, rtol=1e-4, atol=1e-4 * np.abs(truth.grad).max())


@pytest.mark.gpu
@pytest.mark.parametrize("A", DTYPES)
@pytest.mark.parametrize("n", [300, 1025])
def test_prediction_does_not_depend_on_the_row_count(n, A):
    """DESIGN section 5: for m > 64 a candidate's mean and variance have the same bits however many rows are
    predicted with it (one call, chunks, shards).  f32 used to pick the variance kernel from the padded row count."""
    d = 3
    x, y = synth(n, d, A=A)
    theta = _rounded(random_thetas(1, d, seed=8, noise=(3e-2, 0.3) if A == np.float64 else (0.1, 0.5))[0], A)
    xs = np.random.default_rng(5).random((1000, d)).astype(A)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta)
        full_mean, full_var = model.predict(xs)
        for m in (65, 128, 129, 256):
            mean, var = model.predict(xs[:m])
            np.testing.assert_array_equal(mean, full_mean[:m], err_msg=f"mean, m = {m}")
            np.testing.assert_array_equal(var, full_var[:m], err_msg=f"variance, m = {m}")
        model.close()
