"""CPU-side tests: the C-ABI library loads and exports every declared symbol, and the host logic
(bounded L-BFGS, RNG restatement, kernel parameter objects) behaves like the reference's."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from oracle.rng import RNG
from tests.util import lib_minimizer

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from hbetune_rs_b200 import _lib
    header = open(os.path.join(ROOT, "include", "hbegp.h")).read()
    declared = set(re.findall(r"\b(hbegp_[a-z_0-9]+)\s*\(", header))
    declared -= {"hbegp_objective_fn"}
    assert declared == set(_lib.PROTOTYPES), declared ^ set(_lib.PROTOTYPES)
    for name in declared:
        assert getattr(_lib.lib, name) is not None
    assert _lib.lib.hbegp_version().startswith(b"hbegp")


def test_no_gpu_is_a_loud_error_not_a_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import hbetune_rs_b200 as h
    with pytest.raises(h.HbegpError) as e:
        h.Context()
    assert e.value.code == -2 and "no CPU fallback" in str(e.value)


def test_minimize_by_gradient_slanted_plane():
    # src/util/gradmin.rs:62-102
    minimize = lib_minimizer()
    x, f = minimize(lambda x: (float(x.sum()), np.ones(2)), [0.0, 0.0], [(-2.0, 2.0)] * 2)
    assert list(x) == [-2.0, -2.0] and f == -4.0


def test_minimize_by_gradient_rosenbrock_in_box():
    minimize = lib_minimizer(maxeval=400)

    def rosen(x):
        f = 100 * (x[1] - x[0] ** 2) ** 2 + (1 - x[0]) ** 2
        g = np.array([-400 * x[0] * (x[1] - x[0] ** 2) - 2 * (1 - x[0]), 200 * (x[1] - x[0] ** 2)])
        return float(f), g

    x, f = minimize(rosen, [-1.2, 1.0], [(-2.0, 2.0)] * 2)
    assert f < 1e-10 and np.allclose(x, [1.0, 1.0], atol=1e-4)
    x, f = minimize(rosen, [-1.2, 1.0], [(-2.0, 0.5)] * 2)  # optimum on the boundary
    assert abs(x[0] - 0.5) < 1e-6 and abs(x[1] - 0.25) < 1e-5


def test_lbfgs_tolerances_are_settable():
    """hbegp_lbfgs_set_tolerances: the stall / gradient stops stand in for NLopt's internal ones; switched off, maxeval is
    the only stop like the reference's configuration (gradmin.rs:52-54)."""
    from hbetune_rs_b200 import _lib
    counts = {}

    def quad(x):
        counts["n"] = counts.get("n", 0) + 1
        return float(((x - 0.3) ** 2).sum()), 2 * (x - 0.3)

    try:
        minimize = lib_minimizer(maxeval=60)
        counts.clear()
        x, f = minimize(quad, [1.5, -1.0, 0.7], [(-2.0, 2.0)] * 3)
        with_tol = counts["n"]
        assert f < 1e-12 and with_tol < 30  # converged and stopped on its own
        assert _lib.lib.hbegp_lbfgs_set_tolerances(0.0, 0.0) == 0
        counts.clear()
        x2, f2 = minimize(quad, [1.5, -1.0, 0.7], [(-2.0, 2.0)] * 3)
        assert f2 <= f and counts["n"] >= with_tol  # keeps going until it cannot move or maxeval
    finally:
        _lib.lib.hbegp_lbfgs_set_tolerances(1e-11, 1e-8)


def test_minimize_handles_infinite_objective():
    minimize = lib_minimizer()

    def f(x):
        if x[0] > 1.0:
            return math.inf, np.zeros(1)
        return float((x[0] - 3.0) ** 2), np.array([2 * (x[0] - 3.0)])

    x, fx = minimize(f, [0.0], [(-5.0, 5.0)])
    assert 0.9 < x[0] <= 1.0


def test_rng_matches_oracle_restatement():
    from hbetune_rs_b200 import _lib
    st = (C.c_ulonglong * 4)()
    _lib.lib.hbegp_rng_seed(17176, st)
    ref = RNG.new_with_seed(17176)
    assert list(st) == ref.s
    child = (C.c_ulonglong * 4)()
    _lib.lib.hbegp_rng_fork(st, child)
    rchild = ref.fork_random_state()
    assert list(child) == rchild.s and list(st) == ref.s
    for lo, hi in [(-2.0, 2.0), (math.log(1e-5), math.log(1e5)), (0.0, 0.0)]:
        assert _lib.lib.hbegp_rng_uniform(child, lo, hi) == rchild.uniform_inclusive(lo, hi)


def test_xoshiro_known_answer():
    # Xoshiro256** reference output for state {1, 2, 3, 4} (public test vector of the algorithm)
    r = RNG([1, 2, 3, 4])
    assert [r.next_u64() for _ in range(3)] == [11520, 0, 1509978240]


def test_kernel_parameter_objects_mirror_the_reference():
    import hbetune_rs_b200 as h
    bv = h.BoundedValue
    k = h.Product(h.ConstantKernel(bv(2.0, 1.0, 5.0)), h.Matern(2.5, [bv(1.0, 0.05, 20.0)] * 2))
    assert k.n_params() == 3 and k.theta() == [math.log(2.0), 0.0, 0.0]
    assert k.bounds()[0] == (0.0, math.log(5.0))
    k2 = k.with_clamped_theta([math.log(9.0), math.log(0.01), 0.5])
    assert k2.k1.constant.value == 5.0 and k2.k2.length_scale[0].value == 0.05
    with pytest.raises(h.BoundsError):
        k.with_theta([math.log(9.0), 0.0, 0.0])


def test_python_rng_mirror_matches_oracle_stream():
    import hbetune_rs_b200 as h
    a, b = h.RNG.new_with_seed(123), RNG.new_with_seed(123)
    assert a.state == b.s
    fa, fb = a.fork_random_state(), b.fork_random_state()
    assert fa.state == fb.s and a.state == b.s
    assert [fa.uniform_inclusive(-11.5, 11.5) for _ in range(8)] == [fb.uniform_inclusive(-11.5, 11.5) for _ in range(8)]


def test_gpu_arm_of_bench_does_not_import_the_oracle():
    """Only the cpu_baseline / --impl reference legs may touch oracle/ (via tests.util, lazily)."""
    import ast
    src = open(os.path.join(ROOT, "bench.py")).read()
    tree = ast.parse(src)
    top_level = [n for n in tree.body if isinstance(n, (ast.Import, ast.ImportFrom))]
    names = [getattr(n, "module", None) or n.names[0].name for n in top_level]
    assert not any(str(m).startswith(("oracle", "tests")) for m in names), names
    # the product package and the GPU-only probes never touch the oracle (oracle-based probes live in tests/probes)
    for sub in ("hbetune_rs_b200", "probes"):
        for fn in os.listdir(os.path.join(ROOT, sub)):
            if fn.endswith(".py"):
                text = open(os.path.join(ROOT, sub, fn)).read()
                assert "import oracle" not in text and "from oracle" not in text and "tests.util" not in text, fn
    for fn in os.listdir(os.path.join(ROOT, "hbetune_rs_b200", "csrc")) + os.listdir(os.path.join(ROOT, "include")):
        path = os.path.join(ROOT, "hbetune_rs_b200", "csrc", fn)
        if not os.path.exists(path):
            path = os.path.join(ROOT, "include", fn)
        if fn.endswith((".cu", ".cuh", ".h", ".hpp")):
            assert "oracle/" not in open(path).read(), fn


def test_bench_dump_outputs_are_float_within_budget_and_sampled_the_same_way(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    arrays = {"lml": np.arange(65.0), "status": np.zeros(65, dtype=np.int32),
              "mean": np.random.default_rng(1).random(1 << 18), "var": np.random.default_rng(2).random(1 << 18).astype(np.float32)}
    for sub in ("a", "b"):
        bench.dump_outputs(str(tmp_path / sub), arrays)
    got = {f.stem: np.load(f) for f in (tmp_path / "a").iterdir()}
    assert sorted(got) == sorted(arrays)
    assert got["status"].dtype == np.float64 and got["var"].dtype == np.float32 and got["mean"].dtype == np.float64
    np.testing.assert_array_equal(got["lml"], arrays["lml"])
    assert sum(a.nbytes for a in got.values()) <= 1 << 20
    rows = np.flatnonzero(np.isin(arrays["mean"], got["mean"]))  # a subset of the rows, in their order
    np.testing.assert_array_equal(arrays["mean"][rows], got["mean"])
    for name, a in got.items():
        np.testing.assert_array_equal(np.load(tmp_path / "b" / f"{name}.npy"), a)


def test_c_abi_rejects_bad_arguments_without_crashing():
    """Every entry point returns a status (< 0 with a message) instead of aborting (SURVEY 8 b4 / b6)."""
    from hbetune_rs_b200 import _lib
    L = _lib.lib
    null = None
    assert L.hbegp_set_data(null, 10, 2, null, null) == _lib.ERR_INVALID
    assert b"null context" in L.hbegp_last_error()
    assert L.hbegp_lml_grad_batch(null, 2.5, 1, null, null, null, null, null, null) == _lib.ERR_INVALID
    assert L.hbegp_fit_runs(null, 2.5, 1, null, null, null, 150, None, null) == _lib.ERR_INVALID
    assert L.hbegp_predict(null, 1, null, null, null, None) == _lib.ERR_INVALID
    assert L.hbegp_predict_device(null, 1, null, null, null, null) == _lib.ERR_INVALID
    assert L.hbegp_predict_mean_ei(null, None, 1, null, 0.0, null, null, None, None) == _lib.ERR_INVALID
    assert L.hbegp_ctx_destroy(null) == 0 and L.hbegp_model_destroy(null) == 0  # destroying nothing is fine
    assert L.hbegp_ctx_launch_count(null) == 0
    h = C.c_void_p()
    assert L.hbegp_ctx_create(0, 7, None, C.byref(h)) == _lib.ERR_INVALID  # bad dtype, checked before CUDA
    assert L.hbegp_ctx_create(0, 0, None, None) == _lib.ERR_INVALID
    x = (C.c_double * 2)(0.0, 0.0)
    assert L.hbegp_minimize_by_gradient(_lib.OBJECTIVE_FN(lambda a, b, c: 0.0), None, 0, x, x, x, 10, None) == _lib.ERR_INVALID
    yn = _lib.YNorm()
    y = np.ones(3)
    assert L.hbegp_ynorm_fit(0, 5, 3, y.ctypes.data_as(C.c_void_p), None, y.ctypes.data_as(C.c_void_p), C.byref(yn)) == _lib.ERR_INVALID
    assert L.hbegp_estimate_amplitude(0, 0, None, None, None) == _lib.ERR_INVALID
    res = (_lib.RunResult * 1)()
    res[0].status = 1
    assert L.hbegp_pick_best_run(1, res) == -1 and L.hbegp_pick_best_run(0, res) == -1


def test_minimizer_respects_maxeval_and_bounds():
    from hbetune_rs_b200 import _lib
    calls = []

    def f(xp, gp, _):
        calls.append((xp[0], xp[1]))
        gp[0], gp[1] = 2 * (xp[0] - 10.0), 2 * (xp[1] + 10.0)
        return (xp[0] - 10.0) ** 2 + (xp[1] + 10.0) ** 2

    x = np.array([0.0, 0.0])
    lo, hi = np.array([-1.0, -2.0]), np.array([3.0, 2.0])
    fout = C.c_double()
    n = _lib.lib.hbegp_minimize_by_gradient(_lib.OBJECTIVE_FN(f), None, 2, x.ctypes.data_as(C.c_void_p),
                                            lo.ctypes.data_as(C.c_void_p), hi.ctypes.data_as(C.c_void_p), 7, C.byref(fout))
    assert 1 <= n <= 7 and len(calls) == n
    assert all(lo[0] <= a <= hi[0] and lo[1] <= b <= hi[1] for a, b in calls)  # never evaluated outside the box
    n = _lib.lib.hbegp_minimize_by_gradient(_lib.OBJECTIVE_FN(f), None, 2, x.ctypes.data_as(C.c_void_p),
                                            lo.ctypes.data_as(C.c_void_p), hi.ctypes.data_as(C.c_void_p), 150, C.byref(fout))
    assert list(x) == [3.0, -2.0] and fout.value == 49.0 + 64.0  # the constrained optimum is the corner


# ---- hbegp_fit_runs_with: the lockstep restart loop over a host objective (gradmin.rs:7-33)
def _quadratic_objective(centers, fail_above=None):
    """lml(theta) = -sum_k w_k (theta_k - c_k)^2 (one maximum per run family); status 1 where theta_0 > fail_above."""
    from hbetune_rs_b200 import _lib
    w = np.array([1.0, 3.0, 0.5])
    calls = []

    def cb(_user, B, p, theta, lml, grad, status):
        calls.append(B)
        for b in range(B):
            th = np.array([theta[b * p + k] for k in range(p)])
            if fail_above is not None and th[0] > fail_above:
                status[b] = 1
                lml[b] = float("nan")
                continue
            status[b] = 0
            lml[b] = -float(np.sum(w * (th - centers) ** 2))
            g = -2.0 * w * (th - centers)
            for k in range(p):
                grad[b * p + k] = g[k]
        return 0
    return _lib.BATCH_OBJECTIVE_FN(cb), calls


def _run_with(objective, starts, lo, hi, rank=0, world=1, allreduce=None, maxeval=150):
    from hbetune_rs_b200 import _lib
    L = _lib.lib
    starts = np.ascontiguousarray(starts, dtype=np.float64)
    R, p = starts.shape
    res = (_lib.RunResult * R)()
    thetas = np.empty((R, p))
    ar = _lib.allreduce_callback(allreduce) if allreduce is not None else _lib.ALLREDUCE_FN()
    rc = L.hbegp_fit_runs_with(objective, None, p, R, starts.ctypes.data, lo.ctypes.data, hi.ctypes.data, maxeval, rank, world,
                               ar, None, res, thetas.ctypes.data)
    return rc, res, thetas


def test_fit_runs_with_host_objective_finds_the_maximum_and_counts_evaluations():
    centers = np.array([0.3, -0.2, 1.0])
    obj, calls = _quadratic_objective(centers)
    lo, hi = np.exp(np.array([-3.0, -3.0, -3.0])), np.exp(np.array([3.0, 3.0, 3.0]))
    starts = np.random.default_rng(3).uniform(-2.5, 2.5, (6, 3))
    rc, res, thetas = _run_with(obj, starts, lo, hi)
    assert rc == 0
    for r in range(6):
        assert res[r].status == 0 and res[r].n_evals >= 2
        np.testing.assert_allclose(thetas[r], centers, atol=1e-6)
        assert res[r].best_lml == pytest.approx(0.0, abs=1e-10)
        assert 0 <= res[r].best_eval < res[r].n_evals
    # lockstep: the first round evaluates all six runs, later rounds only the live ones
    assert calls[0] == 6 and sum(calls) == sum(res[r].n_evals for r in range(6)) and min(calls) >= 1


def test_fit_runs_with_failed_evaluations_are_infinite_cost_not_errors():
    centers = np.array([0.3, -0.2, 1.0])
    obj, _ = _quadratic_objective(centers, fail_above=1.5)
    lo, hi = np.exp(np.array([-3.0, -3.0, -3.0])), np.exp(np.array([3.0, 3.0, 3.0]))
    starts = np.array([[2.0, 0.0, 0.0], [0.0, 0.0, 0.0]])  # run 0 starts in the failing region (fit.rs:103-113)
    rc, res, thetas = _run_with(obj, starts, lo, hi)
    assert rc == 0
    assert res[1].status == 0
    np.testing.assert_allclose(thetas[1], centers, atol=1e-6)
    assert res[0].status == 1 and res[0].best_eval == -1  # zero gradient at +inf: the run stops where it started
    np.testing.assert_array_equal(thetas[0], starts[0])


def test_fit_runs_sharded_argument_validation():
    from hbetune_rs_b200 import _lib
    centers = np.zeros(3)
    obj, _ = _quadratic_objective(centers)
    lo, hi = np.full(3, 0.1), np.full(3, 10.0)
    starts = np.zeros((2, 3))
    assert _run_with(obj, starts, lo, hi, rank=2, world=2, allreduce=lambda a: None)[0] == _lib.ERR_INVALID
    assert _run_with(obj, starts, lo, hi, rank=0, world=2, allreduce=None)[0] == _lib.ERR_INVALID
    assert _run_with(obj, starts, lo, hi, rank=0, world=0)[0] == _lib.ERR_INVALID
    assert _run_with(obj, starts, np.full(3, -1.0), hi)[0] == _lib.ERR_INVALID


def test_fit_runs_with_two_simulated_ranks_match_one_process():
    """Both 'ranks' in one process, stepping in turn through a shared all-reduce: every rank must end with the
    single-process records bit for bit, and each evaluates only its round-robin share."""
    import threading
    centers = np.array([0.3, -0.2, 1.0])
    lo, hi = np.exp(np.array([-3.0, -3.0, -3.0])), np.exp(np.array([3.0, 3.0, 3.0]))
    starts = np.random.default_rng(11).uniform(-2.5, 2.5, (7, 3))
    obj, calls1 = _quadratic_objective(centers, fail_above=2.2)
    rc, ref, ref_thetas = _run_with(obj, starts, lo, hi)
    assert rc == 0
    world = 2
    barrier = threading.Barrier(world)
    pending = {}
    lock = threading.Lock()

    def make_allreduce(rank):
        def ar(a):
            with lock:
                pending[rank] = a.copy()
            barrier.wait()
            total = sum(pending[r] for r in range(world))
            barrier.wait()
            a[:] = total
        return ar

    out = {}

    def worker(rank):
        o, calls = _quadratic_objective(centers, fail_above=2.2)
        out[rank] = _run_with(o, starts, lo, hi, rank=rank, world=world, allreduce=make_allreduce(rank)) + (calls,)

    ts = [threading.Thread(target=worker, args=(r,)) for r in range(world)]
    [t.start() for t in ts]
    [t.join(60) for t in ts]
    total_calls = 0
    for rank in range(world):
        rc, res, thetas, calls = out[rank]
        assert rc == 0
        for r in range(7):
            assert res[r].best_lml == ref[r].best_lml or (np.isnan(res[r].best_lml) and np.isnan(ref[r].best_lml))
            assert (res[r].best_eval, res[r].n_evals, res[r].status) == (ref[r].best_eval, ref[r].n_evals, ref[r].status)
            assert res[r].final_f == ref[r].final_f
        np.testing.assert_array_equal(thetas, ref_thetas)
        total_calls += sum(calls)
    assert total_calls == sum(calls1)  # the evaluations were split, not duplicated
