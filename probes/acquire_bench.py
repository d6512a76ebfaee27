"""Cost of a multi-start EI search (maxeval 150) per generation: the device search (hbegp_acquire_ei) with R rounds
between two looks of the host (HBEGP_ACQ_ROUNDS = 1, 4, 16, alternated), the route before it (hbegp_fit_runs_with + one
hbegp_predict_mean_ei_grad per round, box as exp(lo), exp(hi)), and, as a cost yardstick only, S x 150 one-point
hbegp_predict_mean_ei calls (the shape of BOBYQA's batch-of-1 evaluations; not a parity claim).  All three are timed
from C++ (probes/acquire_routes.cpp, compiled into a temporary directory), host clock around calls that end in a stream
synchronise; the median of --reps runs after one warm-up run.  n in {100, 500, 4096}, d in {2, 8, 16}, S in {10, 64},
f64 and f32; synthetic data, fmin = median(y), starts uniform in [0, 1]^d.  The card's name and power limit are read
in the same run.

  python probes/acquire_bench.py [--out profiles/r10_acquire_bench.json] [--reps 3]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
RS = [1, 4, 16]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # no nvidia-smi: say so
        return f"unavailable: {e}"


def routes(tmp):
    so = os.path.join(tmp, "libacquire_routes.so")
    lib_dir = os.path.join(ROOT, "hbetune_rs_b200")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"),
                    os.path.join(HERE, "acquire_routes.cpp"), "-o", so, "-L", lib_dir, "-lhbegp", "-Wl,-rpath," + lib_dir],
                   check=True)
    lib = ctypes.CDLL(so)
    from hbetune_rs_b200 import _lib
    V, P, L, LL = ctypes.c_void_p, ctypes.POINTER(_lib.YNorm), ctypes.c_long, ctypes.POINTER(ctypes.c_longlong)
    lib.time_device.restype = lib.time_fit_runs_with.restype = lib.time_one_point.restype = ctypes.c_double
    lib.time_device.argtypes = [V, P, ctypes.c_double, L, V, V, V, ctypes.c_int, LL]
    lib.time_fit_runs_with.argtypes = [V, P, ctypes.c_double, ctypes.c_int, V, V, V, ctypes.c_int, LL]
    lib.time_one_point.argtypes = [V, P, ctypes.c_double, L, V]
    return lib


def measure(reps):
    import hbetune_rs_b200 as h
    from hbetune_rs_b200.estimator import LINEAR, YNormalize
    from hbetune_rs_b200.gpr import _ptr
    h._lib.lib.hbegp_lbfgs_set_tolerances(1e-11, 1e-8)
    out = {"card (name, power limit, max SM clock)": card(), "maxeval": 150, "reps": reps,
           "unit": "ms, median of reps after one warm-up; per round = per search / rounds", "cases": []}
    with tempfile.TemporaryDirectory() as tmp:
        lib = routes(tmp)
        for name, A, dt in (("f64", np.float64, h.F64), ("f32", np.float32, h.F32)):
            for n in (100, 500, 4096):
                for d in (2, 8, 16):
                    rng = np.random.default_rng(n * 31 + d)
                    x = rng.random((n, d)).astype(A)
                    yraw = (np.sin(6.0 * x).sum(axis=1) + 0.1 * rng.standard_normal(n) + 10.0).astype(A)
                    y, yn = YNormalize.new_project_into_normalized(yraw, LINEAR, A=A)
                    theta = np.array([np.log(1e-2 if A == np.float64 else 1e-1), 0.0] + [np.log(0.3 * np.sqrt(d))] * d)
                    fmin = float(np.median(yraw))
                    lo, hi = np.zeros(d), np.ones(d)
                    with h.Context(0, dt) as ctx:
                        ctx.set_data(x, y)
                        model = ctx.model(theta)
                        hnd, ynp = model.single_handle(), ctypes.byref(yn._raw)
                        for S in (10, 64):
                            starts = np.ascontiguousarray(rng.random((S, d)))
                            starts_a = np.ascontiguousarray(starts.astype(A))
                            pts = np.ascontiguousarray(rng.random((S * 150, d)).astype(A))
                            rounds = ctypes.c_longlong(0)
                            rec = {"dtype": name, "n": n, "d": d, "S": S}
                            dev = {R: [] for R in RS}
                            dev_rounds = {}
                            for rep in range(reps + 1):  # rep 0: warm-up; R alternates within each rep
                                for R in RS:
                                    os.environ["HBEGP_ACQ_ROUNDS"] = str(R)
                                    ms = lib.time_device(hnd, ynp, fmin, S, _ptr(starts_a), _ptr(lo), _ptr(hi), 150,
                                                         ctypes.byref(rounds))
                                    assert ms >= 0, h._lib.lib.hbegp_last_error()
                                    if rep:
                                        dev[R].append(ms)
                                    dev_rounds[R] = rounds.value
                            os.environ.pop("HBEGP_ACQ_ROUNDS", None)
                            for R in RS:
                                med = float(np.median(dev[R]))
                                rec[f"device_R{R}"] = {"ms_per_search": med, "rounds": dev_rounds[R],
                                                       "ms_per_round": med / max(dev_rounds[R], 1)}
                            fr = []
                            for rep in range(reps + 1):
                                ms = lib.time_fit_runs_with(hnd, ynp, fmin, S, _ptr(starts), _ptr(lo), _ptr(hi), 150,
                                                            ctypes.byref(rounds))
                                assert ms >= 0, h._lib.lib.hbegp_last_error()
                                if rep:
                                    fr.append(ms)
                            med = float(np.median(fr))
                            rec["fit_runs_with"] = {"ms_per_search": med, "rounds": rounds.value,
                                                    "ms_per_round": med / max(rounds.value, 1)}
                            lib.time_one_point(hnd, ynp, fmin, 20, _ptr(pts))
                            ms = lib.time_one_point(hnd, ynp, fmin, S * 150, _ptr(pts))
                            assert ms >= 0, h._lib.lib.hbegp_last_error()
                            rec["one_point_x150S"] = {"ms_total": ms, "calls": S * 150, "ms_per_call": ms / (S * 150)}
                            out["cases"].append(rec)
                            print(json.dumps(rec), flush=True)
                        model.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    res = measure(args.reps)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card (name, power limit, max SM clock)"], "cases": len(res["cases"])}))


if __name__ == "__main__":
    main()
