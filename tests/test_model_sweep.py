"""The paths a fitted model runs after the fit, against the f64 reference of tests/test_dispatch_sweep.py: extend's block
append (Engine::append_nu), the rebuild of an evicted model (ModelT::rebuild_nu) and the latency prediction path
(m <= 64: k_kstar_small, k_wmatvec_small, k_small_finish).

An append keeps the prior's W11 = L11^-1 over its first r1 rows, assembles K from tile row r1 / 64 and runs one node of
the recursion, merge_node(r1, np - r1).  `_append_plan` restates which kernels that reaches, and
`test_append_shapes_reach_every_variant` checks that APPEND_SHAPES reach each of them; if a threshold moves, that test
fails and APPEND_SHAPES has to move with it.  f64 results must be within 1e-9 of the truth; f32 results no further from
the f64 truth of the f32 inputs than RATIO x LAPACK f32 plus FLOOR f32 roundings, as in the sweep.
"""
import math

import numpy as np
import pytest

from oracle import gpr as ogpr
from oracle.gpr import BoundedValue
from tests.test_dispatch_sweep import (DTYPES, EPS32, FLOOR, RATIO, TILE, _check_predict, _ctx, _gemm_kind, _lapack_f32,
                                       _name, _note, _np, _predict_path, _predict_truth, _recursion, _reference,
                                       _rounded, _split, _thetas, _worst_tile)
from tests.test_kinv_emulation import _emulated
from tests.util import oracle_kernel, oracle_lml, random_thetas, synth

# ------------------------------------------------------------------------------------------------ dispatch restated


def _r1(n_prior, n):
    """Engine::model_extend: the prior rows an append keeps, a multiple of 128 so that the appended blocks stay
    aligned with the 128-wide tiles."""
    return min(n_prior, n) // (2 * TILE) * (2 * TILE)


def _appends(n_prior, n, evicted=False, noise=0.5, noise_clamped=0.5, prefix=True, A=np.float64):
    """The r1 model_extend appends at; 0 runs the full evaluation.  The prior's factor is only reusable if it was
    computed with the noise extend evaluates with (the clamped one), from resident W, for a prefix of the new rows."""
    if evicted or n_prior > n or A(noise_clamped) != A(noise) or not prefix:
        return 0
    return _r1(n_prior, n)


def _append_ops(n_prior, n, want_kinv=True):
    """append_nu: merge_node(r1, np - r1) (hbegp.cu, the four GEMM classes around chol_inv of the new block), then
    the lauum K^-1 = W^T W if asked for."""
    np_, s1 = _np(n), _r1(n_prior, n)
    s2 = np_ - s1
    ops = []
    if s2:
        ops += [("gemm", 0, s2, s1, False), ("gemm", 1, s2, s1, False), ("gemm", 2, s2, s2, True)]
        _recursion(s2, ops)
        ops.append(("gemm", 3, s2, s1, False))
    if want_kinv:
        ops.append(("gemm", 4, np_, np_, True))
    return ops


def _append_plan(n_prior, n, f32):
    np_, r1 = _np(n), _r1(n_prior, n)
    v = set()
    if np_ == r1:
        v.add("s2 = 0")
    if _np(n_prior) % (2 * TILE):
        v.add("prior np not a multiple of 128")
    if r1 < n_prior:
        v.add("r1 < n_prior")
    for op in _append_ops(n_prior, n):
        v.add(op[0] if op[0] != "gemm" else (op[1], _gemm_kind(np_, op[2], op[3], op[4], 1, f32)))
    if _emulated(np_, f32):  # the lauum on the integer tensor cores (tests/test_kinv_bits.py)
        v.add("K^-1 emulated")
    return v


# (n_prior, n)
APPEND_SHAPES = [
    (130, 131),    # r1 = 128, np 192: the appended block is a lone leaf
    (200, 330),    # r1 = 128, np 384: merge(128, 256) where the full recursion runs chol_inv(256), merge(256, 128)
    (300, 768),    # r1 = 256 < 300, prior np 320: full 3xTF32 tiles in classes 0-4
    (300, 800),    # np 832: ragged 3xTF32 tiles in classes 0-4
    (1000, 1100),  # np 1152: 64x64 tiles; r1 = 896 < 1000
    (1100, 1600),  # r1 = 1024, np 1600: 64x64 tiles and ragged 3xTF32 tiles
    (640, 640),    # np = r1: only the copy of W11, alpha and K^-1
    (1900, 2100),  # prior np 1920, np 2112: K^-1 emulated, the workspace of the emulation first allocated by extend
    (2100, 2300),  # r1 = 2048, np 2304: both sides emulated, b = 48
]


def test_append_shapes_reach_every_variant():
    reached = {}
    for n_prior, n in APPEND_SHAPES:
        assert _appends(n_prior, n) > 0, (n_prior, n)
        for f32 in (False, True):
            for v in _append_plan(n_prior, n, f32):
                reached.setdefault(v, set()).add((n_prior, n, "f32" if f32 else "f64"))
    req = {"leaf", "node", "s2 = 0", "prior np not a multiple of 128", "r1 < n_prior", "K^-1 emulated"}
    for cls in range(5):
        req |= {(cls, "32x32"), (cls, "64x64"), (cls, "tf32"), (cls, "tf32 ragged")}
    missing = sorted(map(str, req - set(reached)))
    assert not missing, f"no shape reaches {missing}"
    for cls in range(5):  # both f64 tile sizes in every class
        for kind in ("32x32", "64x64"):
            assert any(p == "f64" for _, _, p in reached[(cls, kind)]), (cls, kind)
    # the shape notes above stay true
    assert _append_ops(130, 131, False) == [("gemm", 0, 64, 128, False), ("gemm", 1, 64, 128, False),
                                            ("gemm", 2, 64, 64, True), ("leaf",), ("gemm", 3, 64, 128, False)]
    assert _r1(200, 330) == 128 and _split(384) == (256, 128)  # the append's tree is not the full evaluation's
    assert all((c, "tf32") in _append_plan(300, 768, True) for c in range(5))
    assert all((c, "tf32 ragged") in _append_plan(300, 800, True) for c in range(5))
    assert all((c, "64x64") in _append_plan(1000, 1100, False) for c in range(5)) and _r1(1000, 1100) == 896
    assert {(c, "tf32 ragged") for c in range(5)} <= _append_plan(1100, 1600, True)
    assert _append_ops(640, 640, False) == []
    assert not _emulated(_np(1900)) and _emulated(_np(2100)) and _r1(2100, 2300) == 2048 and _emulated(2048)


def test_append_falls_back_to_the_full_evaluation():
    assert _appends(200, 330) == 128 and _appends(1100, 1600) == 1024
    assert _appends(100, 330) == 0                      # no 128 prior rows to keep
    assert _appends(200, 330, evicted=True) == 0        # the prior's W was given back
    assert _appends(331, 330) == 0                      # fewer rows than the prior
    assert _appends(200, 330, noise=0.5, noise_clamped=0.25) == 0  # the prior evaluated outside its noise bounds
    assert _appends(200, 330, prefix=False) == 0        # the old rows changed (k_prefix_mismatch)
    # the noise comparison is in the data type: a clamp below f32 resolution still appends in f32
    assert _appends(200, 330, noise=0.5, noise_clamped=0.5 + 1e-12, A=np.float32) == 128
    assert _appends(200, 330, noise=0.5, noise_clamped=0.5 + 1e-12) == 0


@pytest.mark.parametrize("clamp", [False, True])
def test_extend_truth_matches_the_oracle(clamp):
    """The f64 truth the GPU tests compare an extended model with is the oracle's extend (fit.rs:33-68) at the
    prior's theta, with the noise it clamps to, and its prediction (predict.rs:7-52)."""
    n, d = 200, 3
    x, y = synth(n, d, seed=4)
    theta = _rounded(random_thetas(1, d, seed=9, noise=(5e-2, 1.0))[0], np.float64)
    nz = math.exp(theta[0])
    # the noise a model keeps (fit.rs:164): the value it evaluated, clamped to its bounds
    noise = BoundedValue(nz / 4, nz / 4, nz / 2).with_clamped_value(nz) if clamp else BoundedValue(nz, nz / 2, nz * 2)
    want = ogpr.fitted_kernel_extend(oracle_kernel(theta), x, y, noise)
    theta_eval = theta.copy()
    theta_eval[0] = math.log(noise.value)
    assert noise.value == (nz / 2 if clamp else nz)
    got = _reference(theta_eval, x, y)
    assert abs(got.lml - want.lml) <= 1e-12 * abs(want.lml)
    np.testing.assert_allclose(got.alpha, want.alpha, rtol=0, atol=1e-12 * np.abs(want.alpha).max())
    np.testing.assert_allclose(got.kinv, want.k_inv, rtol=0, atol=1e-12 * np.abs(want.k_inv).max())
    xs = np.random.default_rng(3).random((40, d))
    ov = np.empty(len(xs))
    om = ogpr.predict(want.kernel, want.alpha, xs, x, want.k_inv, ov)
    tm, tv = _predict_truth(theta_eval, x, xs, got)
    np.testing.assert_allclose(tm, om, rtol=0, atol=1e-12 * max(1.0, np.abs(om).max()))
    np.testing.assert_allclose(tv, np.maximum(ov, 0.0), rtol=0, atol=1e-12 * math.exp(theta[1]))


# ------------------------------------------------------------------------------------------------ GPU part


def _data(n, d, A, seed):
    """x, y of n rows, and y renormalised as the adapter does on extend (gpr.rs:293-337): the targets of the old rows
    change, X does not."""
    x, y = synth(n, d, seed=seed, A=A)
    return x, y, (y * A(1.25) + A(0.1)).astype(A)


def _extend(ctx, theta, x, y_prior, y, n_prior):
    import hbetune_rs_b200 as h
    ctx.set_data(x[:n_prior], y_prior[:n_prior])
    prior = ctx.model(theta)
    ctx.set_data(x, y)
    return prior, h.Model(ctx, prior=prior, want_kinv=True)


def _check_model(model, theta, x, y, A, tag):
    """LML, alpha and (if the model returned it) K^-1 against the f64 truth at theta; returns the truth."""
    truth = _reference(theta, x, y)
    got = {"lml": np.array([model.lml]), "alpha": model.alpha}
    want = {"lml": np.array([truth.lml]), "alpha": truth.alpha}
    scale = {"lml": truth.lml_scale, "alpha": float(np.abs(truth.alpha).max())}
    if model.k_inv is not None:
        got["kinv"], want["kinv"], scale["kinv"] = model.k_inv, truth.kinv, float(np.abs(truth.kinv).max())
    lapack = {}
    if A == np.float32:
        o32 = oracle_lml(theta, x, y, A=np.float32)
        lapack = {"lml": np.array([o32.lml]), "alpha": o32.alpha}
        if "kinv" in got:
            lapack["kinv"] = _lapack_f32(theta, x, 2.5)[2]
    note, fails = {}, []
    for key in got:
        err = np.abs(got[key].astype(np.float64) - want[key])
        if A == np.float64:
            note[key] = float(err.max() / abs(want[key]).max())
            ok = note[key] <= 1e-9
        else:
            e_lapack = float(np.abs(lapack[key].astype(np.float64) - want[key]).max())
            note[key] = {"cuda": float(err.max()), "lapack_f32": e_lapack, "scale": scale[key]}
            ok = err.max() <= RATIO * e_lapack + FLOOR * EPS32 * scale[key]
        if not ok:
            fails.append((key, note[key], _worst_tile(err) if err.ndim == 2 else f"worst index {int(err.argmax())}"))
    _note(tag, note)
    assert not fails, (tag, fails)
    return truth


def _check_predictions(model, theta, x, truth, A, ms, tag):
    d = x.shape[1]
    xs = np.random.default_rng(7).random((max(ms), d)).astype(A)
    for m in ms:
        want = "latency" if m <= 64 else ("split" if _np(x.shape[0]) > 16 * TILE else "one")
        assert _predict_path(m, d, _np(x.shape[0]), A().itemsize) == want
        mean, var = model.predict(xs[:m])
        tm, tv = _predict_truth(theta, x, xs[:m], truth)
        _check_predict(mean, var, tm, tv, theta, A, f"{tag} m={m}")


@pytest.mark.gpu
@pytest.mark.parametrize("A", DTYPES)
@pytest.mark.parametrize("n_prior,n", APPEND_SHAPES)
def test_append_matches_the_truth(n_prior, n, A):
    d = 3
    x, y, y2 = _data(n, d, A, seed=n_prior)
    theta = _rounded(_thetas(1, d, A, seed=n_prior + n)[0], A)
    with _ctx(A) as ctx:
        prior, ext = _extend(ctx, theta, x, y, y2, n_prior)
        assert ext.appended
        tag = f"append {n_prior}->{n} {_name(A)}"
        truth = _check_model(ext, theta, x, y2, A, tag)
        _check_predictions(ext, theta, x, truth, A, (1, 17, 64, 65, 300), tag)
        ext.close()
        prior.close()


def _poison_run(A, theta, x, y, y2, n_prior, poison):
    import hbetune_rs_b200 as h
    with _ctx(A) as ctx:
        ctx.set_data(x, y2)
        ctx.lml_grad_batch(theta[None], want_grad=False)  # workspaces of the extended size, kept for the smaller prior
        ctx.set_data(x[:n_prior], y[:n_prior])
        if poison:
            ctx.debug_poison()
        prior = ctx.model(theta)
        ctx.set_data(x, y2)
        if poison:
            ctx.debug_poison()
        ext = h.Model(ctx, prior=prior, want_kinv=True)
        xs = np.random.default_rng(6).random((300, x.shape[1])).astype(A)
        out = [np.array([ext.appended, ext.lml]), ext.alpha, ext.k_inv, *ext.predict(xs[:17]), *ext.predict(xs)]
        ext.close()
        prior.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("A", DTYPES)
@pytest.mark.parametrize("n_prior,n", APPEND_SHAPES)
def test_append_reads_no_stale_workspace(n_prior, n, A):
    """NaN in every cell of the workspaces the prior's recursion and then the append do not write (the upper
    triangle of the copied W11, the 128-wide tiles over it, the lauum): the same bits as without."""
    d = 3
    x, y, y2 = _data(n, d, A, seed=n_prior + 1)
    theta = _rounded(_thetas(1, d, A, seed=n)[0], A)
    clean = _poison_run(A, theta, x, y, y2, n_prior, False)
    poisoned = _poison_run(A, theta, x, y, y2, n_prior, True)
    assert clean[0][0] == 1
    for what, a, b in zip(("appended, lml", "alpha", "K^-1", "mean m=17", "var m=17", "mean", "var"), clean, poisoned):
        assert np.isfinite(b).all(), what
        np.testing.assert_array_equal(b, a, err_msg=what)


@pytest.mark.gpu
@pytest.mark.parametrize("A", DTYPES)
def test_chain_of_appends(A):
    """The tuner extends every generation from the previous model: each step against the truth, and the last model,
    evicted, rebuilds to the same bits (its W went through four appends)."""
    import hbetune_rs_b200 as h
    d = 4
    x, y = synth(700, d, seed=3, A=A)
    theta = _rounded(_thetas(1, d, A, seed=70)[0], A)
    xs = np.random.default_rng(8).random((300, d)).astype(A)
    with _ctx(A) as ctx:
        ctx.set_data(x[:150], y[:150])
        models = [ctx.model(theta)]
        for n in (200, 330, 331, 700):
            ctx.set_data(x[:n], y[:n])
            models.append(h.Model(ctx, prior=models[-1], want_kinv=True))
            assert models[-1].appended, n
            tag = f"chain 150->{n} {_name(A)}"
            truth = _check_model(models[-1], theta, x[:n], y[:n], A, tag)
            _check_predictions(models[-1], theta, x[:n], truth, A, (17, 300), tag)
        last = models[-1]
        before = [*last.predict(xs[:17]), *last.predict(xs)]
        ctx.set_resident_models(1)
        models.append(ctx.model(theta))
        assert ctx.model_stats()["rebuilds"] == 0
        after = [*last.predict(xs[:17]), *last.predict(xs)]
        assert ctx.model_stats()["rebuilds"] == 1
        for what, a, b in zip(("mean m=17", "var m=17", "mean", "var"), before, after):
            np.testing.assert_array_equal(b, a, err_msg=what)
        for m in models:
            m.close()


@pytest.mark.gpu
@pytest.mark.parametrize("A", DTYPES)
def test_extend_evaluates_at_the_clamped_noise(A):
    """The prior evaluated its unclamped noise (fit.rs:96); extend evaluates the clamped one (fit.rs:41-44), so the
    prior's factor does not apply and the full evaluation runs."""
    import hbetune_rs_b200 as h
    n_prior, n, d = 300, 400, 3
    x, y, y2 = _data(n, d, A, seed=40)
    theta = _rounded(_thetas(1, d, A, seed=41)[0], A)
    theta[0] = math.log(0.5)
    lo = np.array([0.01] + [1e-9] * (d + 1))
    hi = np.array([0.25] + [1e9] * (d + 1))
    with _ctx(A) as ctx:
        ctx.set_data(x[:n_prior], y[:n_prior])
        prior = ctx.model(theta, lo=lo, hi=hi)
        _check_model(prior, theta, x[:n_prior], y[:n_prior], A, f"clamped prior {_name(A)}")
        ctx.set_data(x, y2)
        ext = h.Model(ctx, prior=prior, want_kinv=True)
        assert not ext.appended and _appends(n_prior, n, noise=0.5, noise_clamped=0.25, A=A) == 0
        clamped = theta.copy()
        clamped[0] = math.log(0.25)
        truth = _check_model(ext, clamped, x, y2, A, f"clamped extend {_name(A)}")
        _check_predictions(ext, clamped, x, truth, A, (17, 300), f"clamped extend {_name(A)}")
        ext.close()
        prior.close()


# (n_prior or None for a created model, n, dtype)
REBUILD_CASES = [(None, 330, np.float64), (200, 330, np.float64), (None, 330, np.float32), (200, 330, np.float32),
                 (300, 768, np.float32)]


@pytest.mark.gpu
@pytest.mark.parametrize("n_prior,n,A", REBUILD_CASES)
def test_rebuilt_model_answers_with_the_same_bits(n_prior, n, A):
    """DESIGN section 3: an evicted model refactorises on its next variance request and answers with the bits it
    gave before, also when its W came from an append; a later extend appends to the rebuilt W."""
    import hbetune_rs_b200 as h
    d, n_next = 3, n + 70
    x, y, y2 = _data(n_next, d, A, seed=n)
    theta = _rounded(_thetas(1, d, A, seed=n + 1)[0], A)
    xs = np.random.default_rng(9).random((300, d)).astype(A)
    with _ctx(A) as ctx:
        if n_prior is None:
            ctx.set_data(x[:n], y2[:n])
            prior, model = None, ctx.model(theta)
        else:
            prior, model = _extend(ctx, theta, x[:n], y, y2[:n], n_prior)
            assert model.appended
        before = [*model.predict(xs[:17]), *model.predict(xs)]
        ctx.set_resident_models(1)
        other = ctx.model(theta)
        st = ctx.model_stats()
        assert st["resident"] == 1 and st["rebuilds"] == 0
        after = [*model.predict(xs[:17]), *model.predict(xs)]
        assert ctx.model_stats()["rebuilds"] == 1
        for what, a, b in zip(("mean m=17", "var m=17", "mean", "var"), before, after):
            np.testing.assert_array_equal(b, a, err_msg=what)
        ctx.set_data(x, y2)
        nxt = h.Model(ctx, prior=model, want_kinv=True)
        assert nxt.appended
        tag = f"extend after rebuild {n_prior}->{n}->{n_next} {_name(A)}"
        truth = _check_model(nxt, theta, x, y2, A, tag)
        _check_predictions(nxt, theta, x, truth, A, (17, 300), tag)
        for m in (prior, model, other, nxt):
            if m is not None:
                m.close()


def _predict_on_device(model, xs):
    import torch
    xd = torch.from_numpy(xs).cuda()
    mean = torch.empty(len(xs), dtype=xd.dtype, device=xd.device)
    var = torch.empty_like(mean)
    torch.cuda.synchronize()
    model.predict_device(len(xs), xd.data_ptr(), mean.data_ptr(), var.data_ptr())
    torch.cuda.synchronize()
    return mean.cpu().numpy(), var.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("A", DTYPES)
@pytest.mark.parametrize("n", [1025, 2049, 4097])
def test_latency_path_at_scale(n, A):
    """One point per call, as every in-tree caller of the reference predicts: 17 to 65 train tiles in k_kstar_small,
    n / 8 row blocks of W in k_wmatvec_small."""
    d = 3
    x, y = synth(n, d, seed=n, A=A)
    theta = _rounded(random_thetas(1, d, seed=5, noise=(3e-2, 0.3) if A == np.float64 else (0.1, 0.5))[0], A)
    xs = np.random.default_rng(2).random((64, d)).astype(A)
    truth = _reference(theta, x, y)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta)
        for m in (1, 16, 17, 64):
            assert _predict_path(m, d, _np(n), A().itemsize) == "latency"
            mean, var = model.predict(xs[:m])
            tm, tv = _predict_truth(theta, x, xs[:m], truth)
            _check_predict(mean, var, tm, tv, theta, A, f"latency n={n} m={m} {_name(A)}")
            dmean, dvar = _predict_on_device(model, xs[:m])
            np.testing.assert_array_equal(dmean, mean)
            np.testing.assert_array_equal(dvar, var)
        model.close()


@pytest.mark.gpu
@pytest.mark.parametrize("A,d,path", [(np.float64, 80, "latency"), (np.float64, 81, "split"),
                                      (np.float32, 160, "latency"), (np.float32, 161, "split")])
def test_latency_path_shared_memory_edge(A, d, path):
    """k_kstar_small copies the m x d candidate rows to shared memory: up to 40 KB, beyond that the throughput path."""
    n, m = 1025, 64
    assert _predict_path(m, d, _np(n), A().itemsize) == path
    x, y = synth(n, d, seed=d, A=A)
    rng = np.random.default_rng(d)
    theta = _rounded(np.concatenate([[math.log(0.1), math.log(1.3)], rng.uniform(math.log(3.0), math.log(9.0), d)]), A)
    xs = rng.random((m, d)).astype(A)
    truth = _reference(theta, x, y)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta)
        mean, var = model.predict(xs)
        model.close()
    tm, tv = _predict_truth(theta, x, xs, truth)
    _check_predict(mean, var, tm, tv, theta, A, f"predict edge m={m} d={d} {_name(A)}")
