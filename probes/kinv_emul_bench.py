"""Two builds of the library (HBEGP_LIB) side by side: the K^-1 = W^T W launches (hbegp_bench_phase 5) and the whole
evaluation (phase 3) in f64 against the padded size, alternating the builds process by process so that both see the
same machine state, and a check that the two agree on LML and alpha bit for bit and on K^-1 and the gradient within
the emulation's error.

    python probes/kinv_emul_bench.py --lib main=/path/a/libhbegp.so --lib branch=/path/b/libhbegp.so \
        --rounds 3 --out profiles/r05_kinv_emulation.json

One process per (build, round); each prints one JSON line.  --worker runs one such process.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = (512, 768, 1024, 1536, 2048, 3072, 4096)
D = 16


def _data(n, seed=1):
    rng = np.random.default_rng(seed)
    x = rng.random((n, D))
    y = np.sin(2 * np.pi * x).sum(axis=1)
    y = (y - y.min()) / (y - y.min()).mean() + 0.05
    return x, y


def _thetas(B, noise):
    rng = np.random.default_rng(B)
    th = np.empty((B, D + 2))
    th[:, 0] = math.log(noise)
    th[:, 1] = rng.uniform(-0.5, 0.5, B)
    th[:, 2:] = np.log(rng.uniform(0.8, 2.0, (B, D)))
    return th


def worker(args):
    sys.path.insert(0, ROOT)
    import hbetune_rs_b200 as h

    out = {"lib": os.environ.get("HBEGP_LIB", "")}
    if args.timing:
        rows = []
        for n in SIZES:
            x, y = _data(n)
            with h.Context(0, h.F64) as ctx:
                ctx.set_data(x, y)
                for B in (1, 65):
                    th = _thetas(B, 1e-2)
                    step = ctx.bench_phase(th, 3, 3)
                    kinv = ctx.bench_phase(th, 5, 5)
                    rows.append({"n": n, "B": B, "step_ms": step, "kinv_ms": kinv})
        out["timing"] = rows
    if args.check:
        os.makedirs(args.check, exist_ok=True)
        tag = os.path.basename(os.path.dirname(out["lib"])) or "default"
        res = {}
        for n, noise in ((1100, 1e-2), (2049, 1e-4), (4096, 1e-2)):
            x, y = _data(n, seed=n)
            th = _thetas(3, noise)
            with h.Context(0, h.F64) as ctx:
                ctx.set_data(x, y)
                lml, grad, status = ctx.lml_grad_batch(th)
                m = ctx.model(th[0], want_alpha=True, want_kinv=True)
                res[f"n{n}_lml"], res[f"n{n}_grad"], res[f"n{n}_status"] = lml, grad, status
                res[f"n{n}_alpha"], res[f"n{n}_kinv"] = m.alpha, m.k_inv
        np.savez(os.path.join(args.check, f"{tag}.npz"), **res)
        out["check"] = os.path.join(args.check, f"{tag}.npz")
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], help="name=path of a libhbegp.so")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default="")
    ap.add_argument("--check-dir", default="", help="where the workers leave their outputs (default: a temporary directory)")
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--timing", action="store_true")
    ap.add_argument("--check", default="")
    args = ap.parse_args()
    if args.worker:
        return worker(args)
    libs = [tuple(s.split("=", 1)) for s in args.lib]
    check_dir = args.check_dir or tempfile.mkdtemp(prefix="kinv_emul_")
    runs = {name: [] for name, _ in libs}
    checks = {}
    for r in range(args.rounds):
        for name, path in libs:
            cmd = [sys.executable, __file__, "--worker", "--timing"]
            if r == 0:
                cmd += ["--check", os.path.join(check_dir, name)]
            t0 = time.perf_counter()
            p = subprocess.run(cmd, env=dict(os.environ, HBEGP_LIB=os.path.abspath(path)), capture_output=True, text=True)
            if p.returncode != 0:
                sys.exit(f"{name} round {r} failed:\n{p.stdout}\n{p.stderr}")
            rec = json.loads(p.stdout.strip().splitlines()[-1])
            if "check" in rec:
                checks[name] = rec["check"]
            runs[name].append(rec["timing"])
            print(f"{name} round {r}: {time.perf_counter() - t0:.1f} s", flush=True)
    summary = {}
    for name in runs:
        for i, row in enumerate(runs[name][0]):
            key = f"n={row['n']} B={row['B']}"
            ks = [rr[i]["kinv_ms"] for rr in runs[name]]
            ss = [rr[i]["step_ms"] for rr in runs[name]]
            summary.setdefault(key, {})[name] = {"kinv_ms": ks, "step_ms": ss}
    for key, v in summary.items():
        print(key, "  ".join(f"{nm}: kinv {min(x['kinv_ms']):.3f}-{max(x['kinv_ms']):.3f} ms step {min(x['step_ms']):.2f}-"
                             f"{max(x['step_ms']):.2f} ms" for nm, x in v.items()), flush=True)
    agree = {}
    if len(checks) == 2:
        (na, pa), (nb, pb) = checks.items()
        a, b = np.load(pa), np.load(pb)
        for k in a.files:
            if k.endswith(("_lml", "_alpha", "_status")):
                agree[k] = "identical" if np.array_equal(a[k], b[k]) else f"differs by {float(np.abs(a[k] - b[k]).max()):.3e}"
            else:
                agree[k] = float(np.abs(a[k] - b[k]).max() / np.abs(a[k]).max())
        for k, v in agree.items():
            print(f"{na} vs {nb} {k}: {v}", flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"timing": summary, "agreement": agree}, f, indent=1)


if __name__ == "__main__":
    main()
