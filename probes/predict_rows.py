"""f32 predict call time (mean + variance, host arrays in and out) at few candidate rows, where the variance GEMM used to
switch between the FFMA kernel (m <= 128) and the 3xTF32 kernel (m > 128).

  python probes/predict_rows.py                          # the in-tree library
  python probes/predict_rows.py --libs A.so B.so         # A/B: alternating child processes (HBEGP_LIB), 2 rounds each

Prints one JSON object: milliseconds per call (median of --reps) by n and m, with the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SIZES = [(512, 8), (4096, 16)]
ROWS = [65, 128, 200]


def measure(reps):
    sys.path.insert(0, os.path.dirname(HERE))
    import hbetune_rs_b200 as h
    out = {}
    rng = np.random.default_rng(1)
    for n, d in SIZES:
        x = rng.random((n, d)).astype(np.float32)
        y = (np.sin(6.0 * x).sum(axis=1) + 0.1 * rng.standard_normal(n)).astype(np.float32)
        theta = np.array([np.log(0.1), 0.0] + [np.log(0.7)] * d)
        xs = rng.random((max(ROWS), d)).astype(np.float32)
        with h.Context(0, h.F32) as ctx:
            ctx.set_data(x, y)
            model = ctx.model(theta)
            for m in ROWS:
                for _ in range(20):
                    model.predict(xs[:m])
                ts = []
                for _ in range(reps):
                    t0 = time.perf_counter()
                    model.predict(xs[:m])  # returns host arrays: ends in a stream synchronise
                    ts.append(time.perf_counter() - t0)
                out[f"n{n}_m{m}_ms"] = round(float(np.median(ts)) * 1e3, 4)
            model.close()
    return out


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, check=True).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.CalledProcessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--libs", nargs="*", default=[])
    ap.add_argument("--reps", type=int, default=300)
    ap.add_argument("--child", action="store_true")
    a = ap.parse_args()
    if a.child or not a.libs:
        res = measure(a.reps)
        print(json.dumps(res if a.child else {"card": card(), "ms": res}))
        return
    runs = {lib: [] for lib in a.libs}
    for _ in range(2):
        for lib in a.libs:
            env = dict(os.environ, HBEGP_LIB=os.path.abspath(lib))
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--reps", str(a.reps)],
                               env=env, capture_output=True, text=True, check=True)
            runs[lib].append(json.loads(p.stdout.strip().splitlines()[-1]))
    print(json.dumps({"card": card(), "ms": runs}))


if __name__ == "__main__":
    main()
