"""Cost of the candidate gradients: hbegp_predict_mean_ei_grad against hbegp_predict_mean_ei at n = 4096, d = 16,
m = 1, 8, 64 and 2^20, f64 and f32, and the device time per kernel of one gradient call (torch.profiler, a run of
its own after the timed calls).

  python probes/predict_grad_bench.py [--out profiles/r09_predict_grad_bench.json]

Call times are host clocks around the whole call, which ends in a stream synchronise (median of --reps after warm-up).
The card's name and power limit are read in the same run.  Prints one JSON object."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
N, D = 4096, 16
ROWS = [1, 8, 64, 1 << 20]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # no nvidia-smi: say so
        q = f"unavailable: {e}"
    return q


def phases(est, xs, fmin):
    """Device time per kernel name of one gradient call and one value call (ms)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for tag, fn in (("grad", lambda: est.predict_mean_ei_grad(xs, fmin)), ("values", lambda: est.predict_mean_ei_device(xs, fmin))):
        fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        per = {}
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            if t > 0:
                per[ev.key[:90]] = per.get(ev.key[:90], 0.0) + t / 1e3
        out[tag] = dict(sorted(per.items(), key=lambda kv: -kv[1]))
    return out


def measure(reps):
    sys.path.insert(0, os.path.dirname(HERE))
    import hbetune_rs_b200 as h
    from hbetune_rs_b200.estimator import LINEAR, SurrogateModelGPR, YNormalize
    res = {"card (name, power limit, max SM clock)": card(), "n": N, "d": D, "unit": "ms per call, median"}
    rng = np.random.default_rng(1)
    for name, A, dt in (("f64", np.float64, h.F64), ("f32", np.float32, h.F32)):
        x = rng.random((N, D)).astype(A)
        yraw = (np.sin(6.0 * x).sum(axis=1) + 0.1 * rng.standard_normal(N)).astype(A)
        y, yn = YNormalize.new_project_into_normalized(yraw, LINEAR, A=A)
        theta = np.array([np.log(1e-2 if A == np.float64 else 1e-1), 0.0] + [np.log(0.7)] * D)
        xs_all = rng.random((max(ROWS), D)).astype(A)
        fmin = float(yraw.min())
        rec = {}
        with h.Context(0, dt) as ctx:
            ctx.set_data(x, y)
            model = ctx.model(theta)
            est = SurrogateModelGPR.__new__(SurrogateModelGPR)
            est.fitted = type("F", (), {"model": model})()
            est.y_norm, est.A = yn, A
            for m in ROWS:
                xs = xs_all[:m]
                r = reps if m < 4096 else 3
                row = {}
                for tag, fn in (("mean_ei", lambda: est.predict_mean_ei_device(xs, fmin, want_best=False)),
                                ("mean_ei_grad", lambda: est.predict_mean_ei_grad(xs, fmin))):
                    for _ in range(3 if m >= 4096 else 20):
                        fn()
                    ts = []
                    for _ in range(r):
                        t0 = time.perf_counter()
                        fn()
                        ts.append((time.perf_counter() - t0) * 1e3)
                    row[tag] = float(np.median(ts))
                row["ratio"] = row["mean_ei_grad"] / row["mean_ei"]
                rec[f"m={m}"] = row
            rec["kernels at m=2^20 (ms, torch.profiler)"] = phases(est, xs_all, fmin)
            rec["kernels at m=1 (ms, torch.profiler)"] = phases(est, xs_all[:1], fmin)
            model.close()
        res[name] = rec
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = measure(a.reps)
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
