"""GPU parity tests proper: the CUDA path (through the C ABI) against the CPU oracle on the same
seeded inputs.  Tolerances: f64 relative 1e-9, f32 relative 1e-4 (BASELINE.json north_star), with the
conditioning caveat of SURVEY.md H3: variances are compared as |d var| <= tol * (c + 1e-5), and the
synthetic thetas keep noise >= 1e-2."""
import math

import numpy as np
import pytest

from tests.util import oracle_kernel, oracle_lml, random_thetas, synth
from oracle import gpr as ogpr

pytestmark = pytest.mark.gpu

TOL = {np.float64: 1e-9, np.float32: 1e-4}


def _ctx(A):
    import hbetune_rs_b200 as h
    return h.Context(0, h.F64 if A == np.float64 else h.F32)


@pytest.mark.parametrize("n,d", [(1, 1), (3, 2), (64, 2), (65, 3), (100, 3), (200, 5), (333, 8)])
def test_factor_intermediates_f64(n, d):
    A = np.float64
    x, y = synth(n, d)
    theta = random_thetas(1, d, seed=n)[0]
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        out = ctx.debug_factor(theta)
    assert out["status"] == 0
    kern = oracle_kernel(theta)
    k_ref = kern.kernel(x, x, A) + math.exp(theta[0]) * np.eye(n)
    np.testing.assert_allclose(out["k"], np.tril(k_ref), rtol=1e-12, atol=1e-14)
    l_ref = np.linalg.cholesky(k_ref)
    w_ref = np.linalg.inv(l_ref)
    np.testing.assert_allclose(out["w"], w_ref, rtol=0, atol=1e-9 * np.abs(w_ref).max())
    kinv_ref = ogpr.factorizec(k_ref.copy(), A).invc()
    np.testing.assert_allclose(out["kinv"], kinv_ref, rtol=0, atol=1e-9 * np.abs(kinv_ref).max())


@pytest.mark.parametrize("A", [np.float64, np.float32])
@pytest.mark.parametrize("n,d,B", [(50, 2, 3), (150, 4, 5), (300, 8, 4), (90, 64, 2)])
def test_lml_and_gradient_batch(A, n, d, B):
    x, y = synth(n, d, A=A)
    thetas = random_thetas(B, d, seed=7 + n, noise=(1e-2, 1.0) if A == np.float64 else (1e-1, 1.0))
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        lml, grad, status = ctx.lml_grad_batch(thetas)
        lml_only, none, _ = ctx.lml_grad_batch(thetas, want_grad=False)
    assert none is None
    np.testing.assert_array_equal(lml, lml_only)
    tol = TOL[A]
    for b in range(B):
        ref = oracle_lml(thetas[b], x, y, A=A)
        assert status[b] == 0 and ref is not None
        assert abs(lml[b] - ref.lml) <= tol * abs(ref.lml), (b, lml[b], ref.lml)
        g_ref = np.array(ref.lml_gradient)
        scale = np.abs(g_ref).max()
        np.testing.assert_allclose(grad[b], g_ref, rtol=tol, atol=tol * scale)


@pytest.mark.parametrize("nu", [0.5, 1.5, 2.5])
def test_matern_nu_variants(nu):
    A = np.float64
    x, y = synth(90, 3)
    thetas = random_thetas(3, 3, seed=11)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        lml, grad, status = ctx.lml_grad_batch(thetas, nu=nu)
    for b in range(3):
        ref = oracle_lml(thetas[b], x, y, nu=nu)
        assert abs(lml[b] - ref.lml) <= 1e-9 * abs(ref.lml)
        g_ref = np.array(ref.lml_gradient)
        np.testing.assert_allclose(grad[b], g_ref, rtol=1e-8, atol=1e-9 * np.abs(g_ref).max())


def test_unsupported_nu_and_errors():
    import hbetune_rs_b200 as h
    x, y = synth(10, 2)
    with _ctx(np.float64) as ctx:
        with pytest.raises(h.HbegpError) as e:
            ctx.lml_grad_batch(random_thetas(1, 0))  # no data yet
        ctx.set_data(x, y)
        with pytest.raises(h.HbegpError) as e:
            ctx.lml_grad_batch(random_thetas(1, 2), nu=3.5)
        assert e.value.code == -4


def test_not_positive_definite_is_a_status_not_an_error():
    A = np.float64
    x, y = synth(20, 2)
    x[1] = x[0]  # duplicate row, zero noise, c = 1: the second pivot is exactly 0
    theta_bad = np.array([-800.0, 0.0, 0.0, 0.0])
    theta_ok = np.array([math.log(0.1), 0.0, 0.0, 0.0])
    assert oracle_lml(theta_bad, x, y) is None  # lml.rs:47-50
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        lml, grad, status = ctx.lml_grad_batch(np.stack([theta_ok, theta_bad, theta_ok]))
    assert list(status) == [0, 1, 0]
    assert lml[1] == -math.inf and (grad[1] == 0).all()  # fit.rs:103-113
    assert np.isfinite(lml[0]) and lml[0] == lml[2]


@pytest.mark.parametrize("A", [np.float64, np.float32])
@pytest.mark.parametrize("dup", [(0, 1), (5, 40), (3, 70), (64, 127), (10, 130), (200, 255), (100, 299), (1000, 2048)])
def test_singular_matrices_do_not_leak_into_their_neighbours(A, dup):
    """Duplicate training rows with zero noise make K singular at pivot max(dup): in the first or second half of a
    bottom node, in a later node, or in the trailing part of a merge.  Rounding decides whether that pivot comes out
    <= 0 (status 1, lml.rs:47-50: then lml = -inf and a zero gradient, fit.rs:103-113) or tiny positive, except for
    dup = (0, 1) where it is exactly 0.  Either way the neighbours in the batch are untouched (the second-generation
    bottom node lets non-finite values run on instead of repairing the pivot) and the context evaluates cleanly after.
    dup = (1000, 2048) at n = 2049 (np 2112) runs K^-1 of the f64 batch on the integer tensor cores, where the non-finite
    columns of a singular matrix's W are flagged per column (E_BAD in gemm_i8.cuh) next to finite neighbours."""
    if A == np.float32 and dup[1] >= 300:
        pytest.skip("the emulated K^-1 product above 2048 is f64 only")
    n, d = (300 if dup[1] < 300 else 2049), 3
    x, y = synth(n, d, A=A)
    x[dup[1]] = x[dup[0]]
    theta_bad = np.array([-800.0, 0.0, 0.0, 0.0, 0.0])
    theta_ok = np.array([math.log(0.1), 0.0, 0.0, 0.0, 0.0])
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        lml, grad, status = ctx.lml_grad_batch(np.stack([theta_ok, theta_bad, theta_ok, theta_bad, theta_ok]))
        lml2, grad2, status2 = ctx.lml_grad_batch(theta_ok[None])
    assert [status[0], status[2], status[4]] == [0, 0, 0] and list(status2) == [0]
    assert status[1] == status[3]
    if dup == (0, 1):
        assert status[1] == 1
    for b in (1, 3):
        if status[b] == 1:
            assert lml[b] == -math.inf and (grad[b] == 0).all()
    assert np.isfinite(lml[0]) and lml[0] == lml[2] == lml[4] == lml2[0]
    np.testing.assert_array_equal(grad[0], grad[2])
    np.testing.assert_array_equal(grad[0], grad2[0])
    ref = oracle_lml(theta_ok, x, y, A=A)
    tol = 1e-9 if A == np.float64 else 1e-4
    assert abs(lml[0] - ref.lml) <= tol * abs(ref.lml)


@pytest.mark.parametrize("A", [np.float64, np.float32])
def test_cached_graphs_follow_new_data_of_the_same_padded_size(A):
    """The reference's loop refits with ten more rows every generation (src/core/minimize.rs:331-407).  While the padded
    size stays the same the context keeps its CUDA graphs and patches their arguments (cudaGraphExecUpdate) instead of
    capturing new ones: every evaluation must equal, bit for bit, what a fresh context computes for the same data —
    growing within one padded size, crossing into the next, shrinking back, and with the batch sizes of a fit."""
    d = 3
    xs, ys = synth(260, d, A=A)
    thetas = random_thetas(5, d, seed=11)
    with _ctx(A) as ctx:
        for n in (130, 140, 150, 192, 193, 200, 150, 130):
            ctx.set_data(xs[:n], ys[:n])
            got = [ctx.lml_grad_batch(thetas[:b]) for b in (5, 3, 1, 5)]
            with _ctx(A) as fresh:
                fresh.set_data(xs[:n], ys[:n])
                want = [fresh.lml_grad_batch(thetas[:b]) for b in (5, 3, 1, 5)]
            for (l1, g1, s1), (l2, g2, s2) in zip(got, want):
                np.testing.assert_array_equal(l1, l2)
                np.testing.assert_array_equal(g1, g2)
                np.testing.assert_array_equal(s1, s2)
    ref = oracle_lml(thetas[0], xs[:130], ys[:130], A=A)
    tol = 1e-9 if A == np.float64 else 1e-4
    assert abs(l1[0] - ref.lml) <= tol * abs(ref.lml)


def test_theta_clamping_matches_with_clamped_theta():
    A = np.float64
    x, y = synth(40, 2)
    lo = np.array([1e-5, 0.5, 0.1, 0.1])
    hi = np.array([1e5, 2.0, 1.0, 1.0])
    theta = np.array([math.log(0.1), math.log(5.0), math.log(0.01), math.log(0.5)])  # c, l_1 out of bounds
    clamped = np.array([math.log(0.1), math.log(2.0), math.log(0.1), math.log(0.5)])
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        a, ga, _ = ctx.lml_grad_batch(theta[None], lo=lo, hi=hi)
        b, gb, _ = ctx.lml_grad_batch(clamped[None])
    assert abs(a[0] - b[0]) <= 1e-12 * abs(b[0])
    np.testing.assert_allclose(ga, gb, rtol=1e-10)


@pytest.mark.parametrize("A", [np.float64, np.float32])
@pytest.mark.parametrize("n,d,m", [(5, 1, 1), (120, 3, 300), (257, 6, 1000), (64, 2, 64), (70, 50, 130)])
def test_predict_mean_and_variance(A, n, d, m):
    x, y = synth(n, d, A=A)
    xs = np.random.default_rng(2).random((m, d)).astype(A)
    theta = random_thetas(1, d, seed=5, noise=(3e-2, 0.3) if A == np.float64 else (0.1, 0.5))[0]
    ref = oracle_lml(theta, x, y, A=A)
    kern = oracle_kernel(theta)
    kinv_ref = ref.factorization.invc()
    var_ref = np.zeros(m, dtype=A)
    mean_ref = ogpr.predict(kern, ref.alpha, xs, x, kinv_ref, var_ref, A)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta, want_kinv=True)
        mean, var = model.predict(xs)
        mean_only, none = model.predict(xs, want_variance=False)
    tol = TOL[A]
    c = math.exp(theta[1])
    assert abs(model.lml - ref.lml) <= tol * abs(ref.lml)
    np.testing.assert_allclose(model.alpha, ref.alpha, rtol=0, atol=tol * 10 * np.abs(ref.alpha).max())
    np.testing.assert_allclose(model.k_inv, kinv_ref, rtol=0, atol=tol * 10 * np.abs(kinv_ref).max())
    np.testing.assert_allclose(mean, mean_ref, rtol=0, atol=tol * max(1.0, np.abs(mean_ref).max()))
    np.testing.assert_allclose(var, var_ref, rtol=0, atol=tol * (c + 1e-5))
    np.testing.assert_array_equal(mean, mean_only)
    assert none is None and (var >= 0).all()


def test_predict_empty_and_training_points():
    A = np.float64
    x, y = synth(80, 2)
    theta = np.array([math.log(1e-2), 0.0, math.log(0.5), math.log(0.5)])
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta)
        mean, var = model.predict(np.zeros((0, 2)))
        assert mean.shape == (0,) and var.shape == (0,)
        mean, var = model.predict(x)
    # at the training points the posterior variance is below the noise level and non-negative
    assert (var >= 0).all() and (var < 2e-2).all()
    assert np.abs(mean - y).max() < 0.5


def test_inverse_round_trip_n1024():
    """Size-independent properties at a BASELINE size (C3: n = 1024, d = 8): W K W^T = I, K^-1 = W^T W, K K^-1 = I."""
    A = np.float64
    n, d = 1024, 8
    x, y = synth(n, d)
    theta = np.array([math.log(0.05), 0.0] + [math.log(0.7)] * d)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        out = ctx.debug_factor(theta)
    k = out["k"] + np.tril(out["k"], -1).T
    assert np.abs(out["w"] @ k @ out["w"].T - np.eye(n)).max() < 1e-10  # W = L^-1  <=>  W K W^T = I
    assert np.abs(out["w"].T @ out["w"] - out["kinv"]).max() < 1e-10 * np.abs(out["kinv"]).max()
    assert np.abs(out["kinv"] @ k - np.eye(n)).max() < 1e-9


@pytest.mark.parametrize("A", [np.float64, np.float32])
def test_small_batch_predict_path_matches_throughput_path_and_oracle(A):
    """m <= 64 takes the latency path (k_kstar_small / k_wmatvec_small), larger batches the GEMM path; both must
    agree with each other and with the oracle, for every m around the switch."""
    n, d = 300, 5
    x, y = synth(n, d, A=A)
    theta = random_thetas(1, d, seed=21, noise=(5e-2, 0.3) if A == np.float64 else (0.1, 0.5))[0]
    xs = np.random.default_rng(4).random((200, d)).astype(A)
    ref = oracle_lml(theta, x, y, A=A)
    var_ref = np.zeros(200, dtype=A)
    mean_ref = ogpr.predict(oracle_kernel(theta), ref.alpha, xs, x, ref.factorization.invc(), var_ref, A)
    tol = TOL[A]
    c = math.exp(theta[1])
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta)
        mean_big, var_big = model.predict(xs)
        for m in (1, 2, 15, 16, 17, 63, 64, 65):
            mean, var = model.predict(xs[:m])
            np.testing.assert_allclose(mean, mean_ref[:m], rtol=0, atol=tol * max(1.0, np.abs(mean_ref).max()))
            np.testing.assert_allclose(var, var_ref[:m], rtol=0, atol=tol * (c + 1e-5))
            # the two paths sum in different orders (f32: FFMA mat-vec vs the 3xTF32 tensor GEMM): a few ulps of c
            np.testing.assert_allclose(mean, mean_big[:m], rtol=0, atol=tol * 1e-2 * max(1.0, np.abs(mean_ref).max()))
            np.testing.assert_allclose(var, var_big[:m], rtol=0, atol=tol * (1e-2 if A == np.float64 else 5e-2) * (c + 1e-5))
            mean_only, none = model.predict(xs[:m], want_variance=False)
            np.testing.assert_array_equal(mean_only, mean)
            assert none is None


def test_workspace_limit_chunks_the_batch_bit_identically():
    """A batch larger than the workspace capacity is evaluated in chunks; results do not depend on the chunking."""
    import hbetune_rs_b200 as h
    n, d = 1500, 4
    x, y = synth(n, d)
    thetas = random_thetas(7, d, seed=9)
    with _ctx(np.float64) as ctx:
        ctx.set_data(x, y)
        a, ga, sa = ctx.lml_grad_batch(thetas)
    with _ctx(np.float64) as ctx:
        per_slot = 2 * 1536 * 1536 * 8
        ctx.set_workspace_limit(3 * per_slot + (64 << 20))  # room for 3 of the 7 evaluations at a time
        ctx.set_data(x, y)
        b, gb, sb = ctx.lml_grad_batch(thetas)
        np.testing.assert_array_equal(a, b)
        np.testing.assert_array_equal(ga, gb)
        np.testing.assert_array_equal(sa, sb)
    with _ctx(np.float64) as ctx:
        ctx.set_workspace_limit(1 << 20)  # not even one n x n evaluation fits
        ctx.set_data(x, y)
        with pytest.raises(h.HbegpError) as e:
            ctx.lml_grad_batch(thetas[:1])
        assert e.value.code == -3


def test_predict_lists_the_variances_below_the_warning_level(capfd):
    """predict.rs:39-46 prints the offending pre-clamp values; the ABI returns their count and the values
    (hbegp_predict_warn_values).  A huge amplitude makes c + 1e-5 - |W k*|^2 cancel catastrophically at the training
    points (SURVEY H3): with c = 1e14 the rounding of c - |W k*|^2 alone is ~0.1, far below -sqrt(1e-5) (the same
    formula in NumPy f64 puts 175 of these 200 values there)."""
    n, d = 120, 2
    x, y = synth(n, d)
    theta = np.array([math.log(1e-2), math.log(1e14), math.log(2.0), math.log(2.0)])
    xs = np.concatenate([x[:60], np.random.default_rng(1).random((140, d))])
    with _ctx(np.float64) as ctx:
        ctx.set_data(x, y)
        model = ctx.model(theta)
        mean, var = model.predict(xs, warn=True)
        count = model.n_below_warn
        vals, rows = model.warn_values(cap=4096)
        few, _ = model.warn_values(cap=3)
        mean2, var2 = model.predict(xs[:5] + 0.25, warn=False)  # a clean call resets the list
        vals2, _ = model.warn_values()
        count2 = model.n_below_warn
        model.close()
    assert count > 0, "expected cancellation below the warning level at c = 1e14"
    assert len(vals) == count and (vals < -math.sqrt(1e-5)).all()
    assert (np.diff(rows) > 0).all() and (var[rows] == 0).all() and (var >= 0).all()
    np.testing.assert_array_equal(few, vals[:3])
    err = capfd.readouterr().err
    assert "Variances below 0 were predicted and will be corrected: " + f"{vals[0]:.2e}" in err
    assert count2 == len(vals2)


def test_large_gemm_tile_reads_no_stale_workspace():
    """ADVICE r01: the triangular k ranges of a 128-wide GEMM tile cover the upper 64x64 block of every 128-wide
    diagonal tile of W = L^-1, which the bottom node writes as zeros.  The f32 tcgen05 kernels run on such tiles: at
    n = 384 both K^-1 = W^T W and the predictive variance (np >= 256) take them.  Poison the workspaces with NaNs
    between two evaluations: in either precision the second one must reproduce the first bit for bit and match the
    oracle."""
    for A in (np.float64, np.float32):
        x, y = synth(384, 3, A=A)
        thetas = random_thetas(3, 3, seed=21, noise=(1e-2, 1.0) if A == np.float64 else (1e-1, 1.0))
        with _ctx(A) as ctx:
            ctx.set_data(x, y)
            first = ctx.lml_grad_batch(thetas)
            ctx.debug_poison()
            second = ctx.lml_grad_batch(thetas)
            model = ctx.model(thetas[0])
            ctx.debug_poison()
            mean, var = model.predict(x[:70] + 0.01)
            model.close()
        np.testing.assert_array_equal(first[0], second[0])
        np.testing.assert_array_equal(first[1], second[1])
        assert (second[2] == 0).all() and np.isfinite(mean).all() and np.isfinite(var).all()
        tol = TOL[A]
        for b in range(3):
            ref = oracle_lml(thetas[b], x, y, A=A)
            assert abs(second[0][b] - ref.lml) <= tol * abs(ref.lml), (A, b)
            g_ref = np.array(ref.lml_gradient)
            np.testing.assert_allclose(second[1][b], g_ref, rtol=10 * tol, atol=tol * np.abs(g_ref).max())


@pytest.mark.parametrize("A,d", [(np.float64, 200), (np.float64, 65), (np.float32, 300)])
def test_many_features_are_processed_in_chunks(A, d):
    """The d x 64 operand tiles of the assembly / gradient / k* kernels are staged 64 features at a time, so d is not
    limited by shared memory (round 1 refused d > 195).  LML, every gradient component, mean and variance against the oracle."""
    n, m = 150, 130
    x, y = synth(n, d, A=A)
    rng = np.random.default_rng(9)
    theta = np.concatenate([[math.log(0.1), math.log(1.3)], rng.uniform(math.log(2.0), math.log(9.0), d)])
    xs = rng.random((m, d)).astype(A)
    ref = oracle_lml(theta, x, y, A=A)
    var_ref = np.zeros(m, dtype=A)
    mean_ref = ogpr.predict(oracle_kernel(theta), ref.alpha, xs, x, ref.factorization.invc(), var_ref, A)
    with _ctx(A) as ctx:
        ctx.set_data(x, y)
        lml, grad, status = ctx.lml_grad_batch(np.stack([theta, theta]))
        model = ctx.model(theta)
        mean, var = model.predict(xs)
        mean1, var1 = model.predict(xs[:3])  # latency path
        model.close()
    tol = TOL[A]
    assert status[0] == 0 and abs(lml[0] - ref.lml) <= tol * abs(ref.lml)
    g_ref = np.array(ref.lml_gradient)
    assert grad.shape == (2, d + 2) and (grad[0] == grad[1]).all()
    np.testing.assert_allclose(grad[0], g_ref, rtol=tol * 10, atol=tol * np.abs(g_ref).max())
    c = math.exp(theta[1])
    np.testing.assert_allclose(mean, mean_ref, rtol=0, atol=tol * max(1.0, np.abs(mean_ref).max()))
    np.testing.assert_allclose(var, var_ref, rtol=0, atol=tol * (c + 1e-5))
    np.testing.assert_allclose(mean1, mean_ref[:3], rtol=0, atol=tol * max(1.0, np.abs(mean_ref).max()))
    np.testing.assert_allclose(var1, var_ref[:3], rtol=0, atol=tol * (c + 1e-5))
