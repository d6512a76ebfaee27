"""Cost of the squared exponential (RBF, nu = inf) against Matern 5/2 on the same workloads, the two alternated
within each repetition so that both see the same machine state; medians of --reps repetitions after one warm-up each.

  - the north-star step: one batched LML + gradient evaluation, n = 4096, d = 16, B = 65, bench.py's thetas, f64 and f32
    (host clock around hbegp_lml_grad_batch, which returns with the results on the host);
  - hbegp_bench_phase at the same shape: phase 0 (scale + assembly) and phase 3 - phase 2 (gradient contraction and
    finish), each timed by the library with CUDA events;
  - prediction of m = 2^20 device-resident candidates, mean + variance and mean only (host clock around the call and a
    device synchronise: the library predicts on its own stream, so events on torch's stream would not bracket it);
  - one-point prediction latency (host clock, hbegp_predict with host buffers);
  - hbegp_acquire_ei at n = 500, d = 16, S = 64, maxeval 150.

The card's name and power limit are read in the same run.

  python probes/rbf_bench.py [--out profiles/r11_rbf.json] [--reps 5] [--only step,predict,acquire]
"""
import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
NUS = [("matern52", 2.5), ("rbf", math.inf)]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # no nvidia-smi: say so
        return f"unavailable: {e}"


def workload(n, d, B, A, seed=0):
    """bench.py's synthetic problem and thetas (a mid-fit optimiser step)."""
    rng = np.random.default_rng(seed)
    x = rng.random((n, d)).astype(A)
    y = (np.sin(2 * np.pi * x).sum(axis=1) + 0.1 * rng.standard_normal(n)).astype(A)
    th = np.empty((B, d + 2))
    th[:, 0] = rng.uniform(math.log(0.03), math.log(1.0), B)
    th[:, 1] = rng.uniform(math.log(0.5), math.log(5.0), B)
    th[:, 2:] = rng.uniform(math.log(0.3), math.log(3.0), (B, d))
    return x, y, th


def med(v):
    return float(np.median(v))


def step_and_phases(h, A, reps):
    x, y, th = workload(4096, 16, 65, A)
    out = {}
    with h.Context(0, h.F64 if A == np.float64 else h.F32) as ctx:
        ctx.set_data(x, y)
        times = {k: {"step_ms": [], "phase0_ms": [], "phase3_minus_2_ms": []} for k, _ in NUS}
        for _, nu in NUS:  # warm-up: graphs, modules
            ctx.lml_grad_batch(th, nu)
            for ph in (0, 2, 3):
                ctx.bench_phase(th, ph, 1, nu)
        for _ in range(reps):
            for key, nu in NUS:
                t0 = time.perf_counter()
                _, _, st = ctx.lml_grad_batch(th, nu)
                times[key]["step_ms"].append((time.perf_counter() - t0) * 1e3)
                assert (st == 0).all() or key == "rbf", st
                times[key]["phase0_ms"].append(ctx.bench_phase(th, 0, 3, nu))
                times[key]["phase3_minus_2_ms"].append(ctx.bench_phase(th, 3, 3, nu) - ctx.bench_phase(th, 2, 3, nu))
        for key, nu in NUS:
            _, _, st = ctx.lml_grad_batch(th, nu)
            out[key] = {k: med(v) for k, v in times[key].items()}
            out[key]["not_pd_members"] = int((st != 0).sum())
    return out


def predict(h, A, reps):
    import torch
    n, d, m = 4096, 16, 1 << 20
    x, y, th = workload(n, d, 1, A)
    th[0, 0] = math.log(0.1)
    dt = torch.float64 if A == np.float64 else torch.float32
    xs = torch.rand((m, d), dtype=dt, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    mean, var = torch.empty(m, dtype=dt, device="cuda"), torch.empty(m, dtype=dt, device="cuda")
    out = {}
    with h.Context(0, h.F64 if A == np.float64 else h.F32) as ctx:
        ctx.set_data(x, y)
        models = {key: ctx.model(th[0], nu) for key, nu in NUS}
        one = np.random.default_rng(2).random((1, d)).astype(A)
        t = {key: {"mean_var_ms": [], "mean_only_ms": [], "one_point_ms": []} for key, _ in NUS}
        for key, mdl in models.items():  # warm-up
            mdl.predict_device(m, xs.data_ptr(), mean.data_ptr(), var.data_ptr())
            mdl.predict_device(m, xs.data_ptr(), mean.data_ptr())
            mdl.predict(one, warn=False)
        torch.cuda.synchronize()
        for _ in range(reps):
            for key, mdl in models.items():
                for name, vp in (("mean_var_ms", var.data_ptr()), ("mean_only_ms", None)):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    mdl.predict_device(m, xs.data_ptr(), mean.data_ptr(), vp)
                    torch.cuda.synchronize()
                    t[key][name].append((time.perf_counter() - t0) * 1e3)
                lat = []
                for _ in range(200):
                    t0 = time.perf_counter()
                    mdl.predict(one, warn=False)
                    lat.append((time.perf_counter() - t0) * 1e3)
                t[key]["one_point_ms"].append(med(lat))
        for key, mdl in models.items():
            out[key] = {k: med(v) for k, v in t[key].items()}
            mdl.close()
    return out


def acquire(h, A, reps):
    from hbetune_rs_b200 import _lib
    from hbetune_rs_b200.estimator import YNormalize
    from hbetune_rs_b200.gpr import _ptr
    n, d, S = 500, 16, 64
    x, y, th = workload(n, d, 1, A, seed=3)
    yraw = (y * A(3) + A(10)).astype(A)
    yl, yn = YNormalize.new_project_into_normalized(yraw, 0, A=A)
    th[0, 0] = math.log(1e-2)
    starts = np.random.default_rng(4).random((S, d)).astype(A)
    lo, hi = np.zeros(d), np.ones(d)
    xo, mo = np.empty((S, d), dtype=A), np.empty(S, dtype=A)
    res = (_lib.AcqResult * S)()
    best, rounds = ctypes.c_long(), ctypes.c_longlong()
    fmin = float(np.median(yraw))
    out = {}
    with h.Context(0, h.F64 if A == np.float64 else h.F32) as ctx:
        ctx.set_data(x, yl)
        models = {key: ctx.model(th[0], nu) for key, nu in NUS}

        def run(mdl):
            t0 = time.perf_counter()
            _lib.check(_lib.lib.hbegp_acquire_ei(mdl.single_handle(), ctypes.byref(yn._raw), fmin, S, _ptr(starts), _ptr(lo),
                                                 _ptr(hi), 150, _ptr(xo), _ptr(mo), res, ctypes.byref(best),
                                                 ctypes.byref(rounds)), "acquire_ei")
            return (time.perf_counter() - t0) * 1e3, int(rounds.value)

        for mdl in models.values():
            run(mdl)
        t = {key: [] for key in models}
        nr = {}
        for _ in range(reps):
            for key, mdl in models.items():
                ms, nr[key] = run(mdl)
                t[key].append(ms)
        for key, mdl in models.items():
            out[key] = {"acquire_ei_ms": med(t[key]), "rounds": nr[key]}
            mdl.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default="", help="comma-separated subset of step,predict,acquire")
    args = ap.parse_args()
    import hbetune_rs_b200 as h
    only = set(args.only.split(",")) if args.only else {"step", "predict", "acquire"}
    result = {"card (name, power limit, max SM clock)": card(), "reps": args.reps}
    for A, name in ((np.float64, "f64"), (np.float32, "f32")):
        result[name] = {}
        if "step" in only:
            result[name]["north-star step and phases (n 4096, d 16, B 65)"] = step_and_phases(h, A, args.reps)
        if "predict" in only:
            result[name]["predict (n 4096, d 16, m 2^20; one point)"] = predict(h, A, args.reps)
        if "acquire" in only:
            result[name]["acquire_ei (n 500, d 16, S 64)"] = acquire(h, A, args.reps)
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
