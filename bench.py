#!/usr/bin/env python
"""Benchmark of the GP surrogate hot path (BASELINE.json metric: GP fit LML evals/s + Cholesky FP64
TFLOP/s + predict candidates/s), north-star shape: n = 4096, d = 16, 64 restarts (B = 65 thetas per
lockstep optimiser step), m = 2^20 candidates.

One JSON line on stdout (rank 0).  A "step" is ONE lockstep optimiser step of the fit: a batched
LML + gradient evaluation of all B thetas (src/gpr/lml.rs:29-79 x B), sharded over the ranks with an
all-gather of the per-theta results.  `value` = evaluations per second with X, y resident in HBM;
`e2e` = the same through the C ABI with host buffers (X, y, theta uploaded and results read back every
step).  Prediction throughput, per-phase rooflines and the whole fit + predict wall time are reported in
the same line.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    # long spellings for use under torchrun, whose own parser treats --n / --m as ambiguous abbreviations
    ap.add_argument("--n", "--train-n", dest="n", type=int, default=4096)
    ap.add_argument("--d", "--feat-d", dest="d", type=int, default=16)
    ap.add_argument("--restarts", type=int, default=64)
    ap.add_argument("--m", "--cand-m", dest="m", type=int, default=1 << 20)
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--no-full-fit", action="store_true", help="skip the whole fit+predict wall-time leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub-benchmarks", action="store_true", help="skip the C3 / other-precision / C5-shaped side measurements")
    ap.add_argument("--maxeval", type=int, default=150)
    ap.add_argument("--fit-shard", default="balanced", choices=["balanced", "static"],
                    help="multi-GPU restart loop: per-round balancing (hbegp_fit_runs_sharded) or a static split of the runs")
    ap.add_argument("--only", default="all", choices=["all", "fit-step", "predict"],
                    help="profiling aid: run just the timed fit steps or just the timed prediction, print a short line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed fit step and the last timed prediction returned as DIR/<name>.npy "
                         "(rank 0; with several ranks the prediction is rank 0's block of rows)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


DUMP_BYTES = 64 << 20


def dump_outputs(directory, arrays):
    """Writes each array as directory/<name>.npy in float64 (float32 results stay float32), DUMP_BYTES in all: an array
    whose share would be exceeded is cut to a fixed, seeded sample of its rows, so that two builds run with the same
    arguments are compared on the same entries."""
    os.makedirs(directory, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        if a.nbytes > share:
            rows = np.random.default_rng(0).choice(len(a), share // (a.nbytes // len(a)), replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(directory, f"{name}.npy"), a)


def synth(n, d, seed=1, A=np.float64):
    """X ~ U[0,1)^{n x d}; y = sum_k sin(2 pi x_k) + 0.1 N(0,1), normalised like the linear YNormalize
    (ynormalize.rs:168-173) so that mean(y) = 1.05.  (Same generator as tests/util.py; kept here so that the GPU
    arm of the benchmark imports nothing from tests/ or oracle/.)"""
    rng = np.random.default_rng(seed)
    x = rng.random((n, d))
    y = np.sin(2 * np.pi * x).sum(axis=1) + 0.1 * rng.standard_normal(n)
    y = y - y.min()
    y = y / (y.mean() if y.mean() > 0 else 1.0) + 0.05
    return x.astype(A), y.astype(A)


def workload(args):
    """SURVEY.md section 8 d2: X ~ U[0,1)^{n x d}, y = sum sin(2 pi x_k) + 0.1 N(0,1) normalised like the
    linear YNormalize; bounds as EstimatorGPR::new except noise in [1e-2, 1e1]."""
    A = np.float64 if args.dtype == "f64" else np.float32
    x, y = synth(args.n, args.d, seed=1, A=A)
    p = args.d + 2
    lo = np.array([1e-2] + [max(np.quantile(y.astype(np.float64), 0.1) ** 2 * args.n, 2e-5) / 2] + [1e-3] * args.d)
    hi = np.array([1e1] + [2 * float((y.astype(np.float64) ** 2).sum())] + [1e3] * args.d)
    rng = np.random.default_rng(7)
    B = args.restarts + 1
    # thetas of a typical mid-fit optimiser step: moderate noise / amplitude / length scales
    thetas = np.empty((B, p))
    thetas[:, 0] = rng.uniform(math.log(0.03), math.log(1.0), B)
    thetas[:, 1] = rng.uniform(math.log(0.5), math.log(5.0), B)
    thetas[:, 2:] = rng.uniform(math.log(0.3), math.log(3.0), (B, args.d))
    xs = np.random.default_rng(2).random((args.m, args.d)).astype(A)
    return A, x, y, lo, hi, thetas, xs


def base_config(args, B):
    return {"workload": f"ns_fit_n{args.n}_d{args.d}_B{B}", "n": args.n, "d": args.d, "restarts": args.restarts, "B": B,
            "m": args.m}


def ncu_traffic():
    """DRAM bytes per launch from the committed `ncu --set full` captures (profiles/r01_ncu_traffic.json)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r01_ncu_traffic.json")))
    except (OSError, ValueError):
        return {}


class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.samples, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for s in self.samples:
            f = [t.strip() for t in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
            except ValueError:
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        busy = [v for v in sm if smax and v > 0.5 * smax] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def oracle_eval_seconds(x, y, theta, A):
    """One reference-faithful LML + gradient evaluation on the host (oracle: full-square kernel,
    materialised (n, n, d+1) gradient tensor, explicit potri), timed.  The ONLY place bench.py touches oracle/
    (cpu_baseline leg and --impl reference)."""
    from tests.util import oracle_lml
    t0 = time.perf_counter()
    res = oracle_lml(theta, x, y, A=A)
    dt = time.perf_counter() - t0
    return dt, res


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (restatement oracle -- the Rust crate cannot be
    built here: no cargo/rustc) on the host; each step is ONE of the B evaluations of the repo arm's step.

    Headline = ONE BLAS thread: the reference builds OpenBLAS with USE_THREAD=0 (/root/reference Makefile:3-4) and never
    uses rayon inside src/gpr, so one core is all its gpr path can use (SURVEY F6, BASELINE.md section 4).  The same
    evaluation with every host core is reported beside it as a courtesy figure."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from threadpoolctl import threadpool_limits
    A, x, y, lo, hi, thetas, xs = workload(args)
    cores = os.cpu_count()
    warm = min(args.warmup, 1)  # a CPU path has nothing to warm beyond the first call's page faults
    times = []
    with threadpool_limits(limits=1):
        for i in range(warm + args.steps):
            dt, _ = oracle_eval_seconds(x, y, thetas[i % len(thetas)], A)
            if i >= warm:
                times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = 1e3 / ms
    all_cores = [oracle_eval_seconds(x, y, thetas[i % len(thetas)], A)[0] for i in range(2)]
    sample = (f"{len(times)} timed steps; each step = 1 of the {len(thetas)} LML+gradient evaluations of one optimiser step "
              f"(n={args.n}, d={args.d}) on 1 BLAS thread like the reference's USE_THREAD=0 OpenBLAS; restatement oracle "
              "(NumPy + OpenBLAS), not the Rust binary")
    print(json.dumps({
        "impl": "reference", "metric": "gp_fit_lml_evals_per_s", "value": value, "unit": "evals/s", "n_gpus": args.gpus,
        "steps": len(times), "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": base_config(args, len(thetas)),
        "cpu_baseline": {"value": value, "unit": "evals/s", "cores": 1, "kind": "port", "sample": sample,
                         "all_cores": {"value": 1.0 / min(all_cores), "unit": "evals/s", "cores": cores,
                                       "seconds_per_eval": min(all_cores)}},
        "e2e": {"value": value, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import hbetune_rs_b200 as h
    from hbetune_rs_b200 import dist as hd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: hbetune_rs_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG is left as the launcher set it; whatever NCCL logs goes to stderr so that stdout stays the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    A, x, y, lo, hi, thetas, xs = workload(args)
    B, p = thetas.shape
    n, d, m = args.n, args.d, args.m
    side = torch.cuda.Stream()  # a real (non-default) stream: torch events on it bracket the library's kernels
    torch.cuda.set_stream(side)
    stream = torch.cuda.current_stream().cuda_stream
    assert stream != 0
    ctx = h.Context(local_rank, h.F64 if args.dtype == "f64" else h.F32, stream=stream)
    ctx.set_data(x, y)
    hd.init_library_comm(ctx)  # N > 1: the library's own NCCL communicator (torch.distributed only carries the 128-byte id)
    mine = hd.owned_runs(B, rank, world)
    my_thetas = thetas[mine]

    def step_resident():
        # every rank evaluates thetas rank, rank + world, ...; the per-restart (lml, gradient, status) records are packed on
        # the device and exchanged inside libhbegp.so with one ncclAllGather over NVLink; every rank returns all B results
        return ctx.lml_grad_batch_sharded(thetas, lo=lo, hi=hi)

    x_pin = torch.from_numpy(x).pin_memory().numpy()  # pinned host staging for the end-to-end leg
    y_pin = torch.from_numpy(y).pin_memory().numpy()

    def step_e2e():
        ctx.set_data(x_pin, y_pin)  # host -> device copy of X, y every step (theta goes up / results come back inside)
        return step_resident()

    coll = {"ms": 0.0, "n": 0}

    def timed(fn, steps, warmup, note_collectives=False):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launch_count
        ci0 = ctx.comm_info()
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        if note_collectives:  # device time of the library's NCCL calls inside the timed steps only (warm-up pays NCCL's lazy set-up)
            ci1 = ctx.comm_info()
            coll["ms"] = ci1["collective_ms"] - ci0["collective_ms"]
            coll["n"] = ci1["n_collectives"] - ci0["n_collectives"]
        return max_over_ranks(e0.elapsed_time(e1)) / steps, ctx.launch_count - l0, out

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    def fit_outputs(gathered):
        lml, grad, status = gathered
        return {"lml": lml, "lml_grad": grad, "status": status}

    if args.only == "fit-step":
        ms_step, launches, gathered = timed(step_resident, args.steps, args.warmup)
        if rank == 0 and args.dump_outputs:
            dump_outputs(args.dump_outputs, fit_outputs(gathered))
        if rank == 0:
            print(json.dumps({"only": "fit-step", "ms_per_step": ms_step, "evals_per_s": B / (ms_step * 1e-3),
                              "gpu_launches": int(launches), "clocks": sampler.stop()}), flush=True)
        ctx.close()
        return
    if args.only != "predict":
        ms_step, launches, gathered = timed(step_resident, args.steps, args.warmup, note_collectives=True)
        coll_ms_step = coll["ms"] / max(1, coll["n"]) if world > 1 else 0.0
        ms_e2e, _, _ = timed(step_e2e, args.steps, max(1, args.warmup // 2))

    # ---- prediction: mean + variance of m candidates, rows sharded over ranks
    lo_r, hi_r = hd.row_block(m, rank, world)
    theta_model = np.array([math.log(0.1), 0.0] + [math.log(0.5)] * d)  # SURVEY.md 8 d2 (C4)
    model = ctx.model(theta_model, want_alpha=False)
    tdt = torch.float64 if A == np.float64 else torch.float32
    xs_dev = torch.from_numpy(xs[lo_r:hi_r]).cuda()
    mean_dev = torch.empty(hi_r - lo_r, dtype=tdt, device="cuda")
    var_dev = torch.empty(hi_r - lo_r, dtype=tdt, device="cuda")

    def predict_resident():
        model.predict_device(hi_r - lo_r, xs_dev.data_ptr(), mean_dev.data_ptr(), var_dev.data_ptr())

    xs_pin = torch.from_numpy(xs[lo_r:hi_r]).pin_memory()

    xs_all_pin = torch.from_numpy(xs).pin_memory() if world > 1 else xs_pin

    def predict_e2e():
        # host candidates in, host mean / variance out; N > 1: contiguous row blocks per rank, one ncclAllGather of the
        # device-resident shards inside the library
        if world > 1:
            return model.predict_sharded(xs_all_pin.numpy(), want_variance=True)
        return model.predict(xs_pin.numpy(), want_variance=True, warn=False)

    def predict_mean_resident():
        model.predict_device(hi_r - lo_r, xs_dev.data_ptr(), mean_dev.data_ptr(), None)

    psteps = max(2, min(args.steps, 3))
    ms_pred, pred_launches, _ = timed(predict_resident, psteps, 1)
    if rank == 0 and args.dump_outputs:
        outputs = {} if args.only == "predict" else fit_outputs(gathered)
        outputs.update({"predict_mean": mean_dev.cpu().numpy(), "predict_var": var_dev.cpu().numpy()})
        dump_outputs(args.dump_outputs, outputs)
    ms_pred_mean, _, _ = timed(predict_mean_resident, psteps, 1)
    if args.only == "predict":
        if rank == 0:
            print(json.dumps({"only": "predict", "ms": ms_pred, "candidates_per_s": m / (ms_pred * 1e-3),
                              "tflops_mn2": float(hi_r - lo_r) * n * n / (ms_pred * 1e-3) * 1e-12,
                              "gpu_launches": int(pred_launches), "clocks": sampler.stop()}), flush=True)
        model.close()
        ctx.close()
        return
    ms_pred_e2e, _, _ = timed(predict_e2e, psteps, 1)
    clocks = sampler.stop() if rank == 0 else None

    # ---- per-phase timings on rank 0's shard (CUDA events on the context's stream, inside the library)
    phases = None
    if rank == 0:
        reps = 2
        t0 = ctx.bench_phase(my_thetas, 0, reps)
        t1 = ctx.bench_phase(my_thetas, 1, reps)
        t2 = ctx.bench_phase(my_thetas, 2, reps)
        t3 = ctx.bench_phase(my_thetas, 3, reps)
        t5 = ctx.bench_phase(my_thetas, 5, max(reps, 3))  # only the K^-1 = W^T W launches (one per stream group)
        phases = {"assemble_ms": t0, "factor_inverse_ms": t1 - t0, "alpha_kinv_ms": t2 - t1, "grad_finish_ms": t3 - t2,
                  "eval_ms": t3, "kinv_gemm_ms": t5, "batch": len(mine)}

    # ---- peaks measured live with cuBLAS 8192^3 through torch.matmul: FP64 (DGEMM), true FP32 (SGEMM), TF32
    def gemm_peak(dt, tf32):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        a = torch.randn(8192, 8192, dtype=dt, device="cuda")
        b = torch.randn(8192, 8192, dtype=dt, device="cuda")
        torch.matmul(a, b)
        best = 1e30
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        torch.backends.cuda.matmul.allow_tf32 = False
        return 2 * 8192.0 ** 3 / best * 1e-9

    peak_tf = peak_f64 = peak_f32 = peak_tf32 = None
    if rank == 0:
        peak_f64 = gemm_peak(torch.float64, False)
        peak_f32 = gemm_peak(torch.float32, False)
        peak_tf32 = gemm_peak(torch.float32, True)
        # f32 contractions run as 3 x TF32 on tcgen05 (hbetune_rs_b200/csrc/gemm_tf32.cuh): three tensor-core products
        # per useful one, so the bound on USEFUL flops is the measured TF32 rate / 3
        tf32_on = os.environ.get("HBEGP_TF32", "1") != "0"
        peak_tf = peak_f64 if args.dtype == "f64" else (peak_tf32 / 3.0 if tf32_on else peak_f32)

    # ---- the metric's other configurations, 1 GPU, same run (VERDICT r01 item 6): C3 in both precisions, the north-star
    # step in the other precision, and the factor + inverse phase at the C5 size
    def sub_bench(nn, dd, restarts, dtype, steps, phase_only=False):
        sargs = argparse.Namespace(n=nn, d=dd, restarts=restarts, m=8, dtype=dtype)
        _, sx, sy, slo, shi, sth, _ = workload(sargs)
        sctx = h.Context(local_rank, h.F64 if dtype == "f64" else h.F32, stream=stream)
        try:
            sctx.set_data(sx, sy)
            pk = peak_f64 if dtype == "f64" else (peak_tf32 / 3.0 if os.environ.get("HBEGP_TF32", "1") != "0" else peak_f32)
            out = {"n": nn, "d": dd, "B": len(sth), "dtype": dtype, "peak_tflops": pk,
                   "peak_source": "cuBLAS DGEMM 8192^3" if dtype == "f64" else "cuBLAS TF32 GEMM 8192^3 / 3 (3xTF32 split)"}
            if phase_only:
                t0 = sctx.bench_phase(sth, 0, 2)
                t1 = sctx.bench_phase(sth, 1, 2)
                tf = 2.0 * nn ** 3 / 3.0 * len(sth) / ((t1 - t0) * 1e-3) * 1e-12
                out.update({"factor_inverse_ms": t1 - t0, "cholesky_tflops": tf, "frac": tf / pk,
                            "what": "2 n^3 / 3 FLOP per matrix (Cholesky factor + its triangular inverse), CUDA events inside the library"})
                return out
            # warm-up: the graph of the padded batch is captured on the first call and the exact-size graph on the fourth
            # consecutive call with the same batch size (Engine::padded_batch); both are one-off costs
            for _ in range(8):
                sctx.lml_grad_batch(sth, lo=slo, hi=shi)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                sctx.lml_grad_batch(sth, lo=slo, hi=shi)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            tf = 1.0 * nn ** 3 * len(sth) / (ms * 1e-3) * 1e-12
            out.update({"ms_per_step": ms, "evals_per_s": len(sth) / (ms * 1e-3), "lml_eval_n3_tflops": tf, "frac": tf / pk})
            return out
        finally:
            sctx.close()

    subs = None
    if rank == 0 and world == 1 and not args.no_sub_benchmarks:
        other = "f32" if args.dtype == "f64" else "f64"
        subs = {
            "c3_f64": sub_bench(1024, 8, 32, "f64", 50),
            "c3_f32": sub_bench(1024, 8, 32, "f32", 50),
            f"ns_{other}": sub_bench(args.n, args.d, args.restarts, other, 5),
            "c5_shape_factor_phase_f64": sub_bench(16384, 32, 1, "f64", 1, phase_only=True),
        }

    # ---- the whole north-star job once: fit (B lockstep runs, <= maxeval evaluations each) + predict
    full = None
    if not args.no_full_fit:
        bv = h.BoundedValue
        kernel = h.Product(h.ConstantKernel(bv(math.sqrt(lo[1] * hi[1]), lo[1], hi[1])),
                           h.Matern(2.5, [bv(1.0, 1e-3, 1e3)] * d))
        barrier()
        t0 = time.perf_counter()
        fk = h.FittedKernel.new(ctx, kernel, x, y, h.RNG.new_with_seed(1), args.restarts, bv(1.0, 1e-2, 1e1),
                                maxeval=args.maxeval,
                                shard=None if world == 1 else (hd.LibraryFit() if args.fit_shard == "balanced" else hd.sharded_fit_runs))
        barrier()
        t_fit = time.perf_counter() - t0
        t0 = time.perf_counter()
        if world > 1:
            mean, var = fk.model.predict_sharded(xs_all_pin.numpy(), want_variance=True)
        else:
            mean, var = fk.model.predict(xs_pin.numpy(), want_variance=True, warn=False)
        barrier()
        t_pred = time.perf_counter() - t0
        full = {"fit_s": max_over_ranks(t_fit), "predict_s": max_over_ranks(t_pred), "n_evals": int(fk.n_evals),
                "lml": fk.lml, "noise": fk.noise.value, "amplitude": fk.kernel.k1.constant.value}
        full["fit_predict_s"] = full["fit_s"] + full["predict_s"]

    if rank == 0:
        evals_per_s = B / (ms_step * 1e-3)
        out = {
            "metric": "gp_fit_lml_evals_per_s", "value": evals_per_s, "unit": "evals/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": base_config(args, B),
            "config_notes": {
                "sharding": f"restarts and candidate rows over {world} rank(s); one n x n factorisation per GPU",
                "l2": f"inputs larger than L2: per-step working set {B // world * 2 * n * n * x.itemsize / 1e9:.1f} GB per GPU vs 126 MB",
                "exchange": ("none (1 GPU)" if world == 1 else
                             "inside libhbegp.so: records packed on the device, ncclAllGather over NVLink, one device-to-host copy")},
            "e2e": {"value": B / (ms_e2e * 1e-3), "unit": "evals/s",
                    "h2d_bytes_per_step": int(x.nbytes + y.nbytes + thetas.nbytes),
                    "d2h_bytes_per_step": int(B * (p + 1) * 8 + B * 4) if world == 1 else int((B + world) * (p + 2) * 8)},
            "gpu_launches": int(launches),
            "collective": {"ms_per_step": coll_ms_step, "compute_ms_per_step": ms_step - coll_ms_step, "nccl": ctx.comm_info()["nccl_version"],
                           "ranks": ctx.comm_info()["world"],
                           "what": "device time of the ncclAllGather of one step on rank 0 (CUDA events around the call; it includes waiting "
                                   "for the slowest rank to arrive) vs the rest of the step"},
            "clocks": clocks,
            "predict": {"candidates_per_s": m / (ms_pred * 1e-3), "ms": ms_pred, "m": m,
                        "e2e_candidates_per_s": m / (ms_pred_e2e * 1e-3), "e2e_ms": ms_pred_e2e,
                        "h2d_bytes": int(xs.nbytes), "d2h_bytes": int(2 * m * xs.itemsize), "gpu_launches": int(pred_launches)},
            "fit_predict": full,
            "sub_benchmarks": subs,
            "peaks_measured": {"dgemm_tflops": peak_f64, "sgemm_fp32_tflops": peak_f32, "tf32_gemm_tflops": peak_tf32},
        }
        nb = len(mine)
        flops_fi = 2.0 * n ** 3 / 3.0 * nb  # L and L^-1 together (potrf n^3/3 + trtri n^3/3)
        tf_fi = flops_fi / (phases["factor_inverse_ms"] * 1e-3) * 1e-12
        tf_eval = 1.0 * n ** 3 * nb / (phases["eval_ms"] * 1e-3) * 1e-12
        tf_var = float(hi_r - lo_r) * n * n / (ms_pred * 1e-3) * 1e-12
        # Headline roofline: the largest single launch of the dominant kernel, gemm_kernel (DMMA.8x8x4) -- the
        # K^-1 = W^T W product (n^3/3 FLOP per matrix, one launch per stream group), timed live with CUDA events on
        # the library's stream (hbegp_bench_phase 5).  `traffic` is the ncu DRAM byte count of one such launch.
        traffic = ncu_traffic()
        tf_kinv = (n ** 3 / 3.0) * nb / (phases["kinv_gemm_ms"] * 1e-3) * 1e-12
        kt = traffic.get("kinv_gemm", {})
        out["roofline"] = {
            "bound": "tensor",
            "kernel": ("gemm_kernel<double,64,64,32,32,false,false> (DMMA.8x8x4)" if args.dtype == "f64" else
                       "gemm_tf32x3_kernel<false,false> (tcgen05.mma kind::tf32, 3xTF32 split, TMA + TMEM)")
                      + ": K^-1 = W^T W on the lower tiles",
            "achieved": tf_kinv, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf_kinv / peak_tf,
            "traffic": kt.get("traffic") if args.dtype == "f64" and n == 4096 else None,
            "algorithmic_bytes": kt.get("algorithmic_bytes") if args.dtype == "f64" and n == 4096 else None,
            "traffic_note": (f"DRAM bytes of one ncu --set full launch over {kt.get('matrices', '?')} matrices "
                             "(profiles/r01_kinv_gemm_early_ncu_raw.csv); algorithmic = 8 n (n + 1) bytes per matrix "
                             "(W lower read once, K^-1 lower written once)" if args.dtype == "f64" and n == 4096 else
                             "no ncu DRAM capture of this launch; the f32 kernel's capture is at n = 2048 over 17 matrices "
                             "(profiles/r02_tf32_gemm_ncu_raw.csv): 566 MB moved against 4 n (n + 1) x 17 = 285 MB algorithmic"),
            "launch_ms": phases["kinv_gemm_ms"], "matrices": nb,
            "peak_source": ("cuBLAS DGEMM 8192^3 (torch.matmul f64) measured in this run; MEASURED_PEAKS.json has no FP64 entry"
                            if args.dtype == "f64" else
                            "cuBLAS TF32 GEMM 8192^3 (torch.matmul, allow_tf32) measured in this run, divided by 3: every useful "
                            "product costs three tensor-core products in the 3xTF32 split"),
            "algorithmic": "n^3 / 3 FLOP per matrix (lower tiles of W^T W, K restricted to k >= row tile)",
        }
        out["phases"] = phases
        t_dense = (phases["factor_inverse_ms"] + phases["alpha_kinv_ms"]) * 1e-3
        tf_dense = 1.0 * n ** 3 * nb / t_dense * 1e-12
        out["cholesky_fp64_tflops"] = tf_fi
        out["lml_eval_fp64_tflops"] = tf_eval
        out["predict_var_fp64_tflops"] = tf_var
        out["rooflines"] = {
            "factor_inverse_phase": {"bound": "tensor", "achieved": tf_fi, "peak": peak_tf, "frac": tf_fi / peak_tf, "unit": "TFLOP/s",
                                     "what": "2 n^3 / 3 FLOP per evaluation (Cholesky factor n^3/3 + its triangular inverse n^3/3) over the "
                                             "whole recursion phase: k_node128 / k_leaf chains + 4 gemm_kernel launches per node"},
            "lml_eval_n3": {"achieved": tf_eval, "peak": peak_tf, "frac": tf_eval / peak_tf, "unit": "TFLOP/s"},
            "dense_phases_n3": {"achieved": tf_dense, "peak": peak_tf, "frac": tf_dense / peak_tf, "unit": "TFLOP/s",
                                "what": "all gemm_kernel + k_leaf launches (factor, inverse, K^-1 = W^T W): n^3 FLOP per evaluation"},
            "kinv_gemm": dict({"bound": "tensor", "unit": "TFLOP/s", "peak": peak_tf,
                               "algorithmic": "n^3/3 FLOP, 8 n^2 bytes (read W lower, write K^-1 lower) per matrix"},
                              **traffic.get("kinv_gemm", {})),
            "predict_var_gemm": dict({"bound": "tensor", "unit": "TFLOP/s", "peak": peak_tf,
                                      "algorithmic": "m n^2 FLOP per chunk of m candidates"},
                                     **traffic.get("predict_var_gemm", {})),
            "predict_var_mn2": {"achieved": tf_var * world, "peak": peak_tf * world, "frac": tf_var / peak_tf, "unit": "TFLOP/s"},
            "assemble_hbm": {"achieved": nb * (8.0 * n * d + x.itemsize * n * (n + 1) / 2) / (phases["assemble_ms"] * 1e-3) * 1e-9,
                             "peak": peaks().get("hbm_gbs"), "unit": "GB/s"},
        }
        # SURVEY 8 d3: the element-wise kernels are reported against HBM as BASELINE.json asks, with the FP64 FMA-pipe
        # bound that actually limits them beside it (approximate op counts per matrix entry: distances 3d, Matern +
        # exp + sqrt ~40; the gradient contraction re-forms the distances and adds 3d per entry).
        alu_peak = 36.7 if args.dtype == "f64" else 2 * 36.7  # TFLOP/s, profiles/r01_fp64_peak_probe.log (raw DFMA issue rate)
        isz = x.itemsize
        rl = out["rooflines"]
        rl["assemble_hbm"]["alu"] = {"achieved": nb * (3 * d + 40) * n * (n + 1) / 2 / (phases["assemble_ms"] * 1e-3) * 1e-12,
                                     "peak": alu_peak, "unit": "TFLOP/s (approx. op count)"}
        rl["grad_contract_hbm"] = {
            "achieved": nb * (isz * n * (n + 1) / 2 + isz * n * (d + 1)) / (phases["grad_finish_ms"] * 1e-3) * 1e-9,
            "peak": peaks().get("hbm_gbs"), "unit": "GB/s",
            "what": "k_grad_contract + k_finish: reads the lower tiles of K^-1 once, scaled X and alpha",
            "alu": {"achieved": nb * (6 * d + 60) * n * (n + 1) / 2 / (phases["grad_finish_ms"] * 1e-3) * 1e-12,
                    "peak": alu_peak, "unit": "TFLOP/s (approx. op count)"}}
        mm = hi_r - lo_r
        rl["predict_mean_hbm"] = {
            "achieved": (isz * mm * d + isz * n * d + isz * mm) / (ms_pred_mean * 1e-3) * 1e-9,
            "peak": peaks().get("hbm_gbs"), "unit": "GB/s", "ms": ms_pred_mean, "candidates_per_s": mm / (ms_pred_mean * 1e-3),
            "what": "k_kstar_mean without variance: k* is formed tile by tile and never written (reads X*, X, alpha; writes the mean)",
            "alu": {"achieved": mm * n * (3.0 * d + 42) / (ms_pred_mean * 1e-3) * 1e-12, "peak": alu_peak,
                    "unit": "TFLOP/s (approx. op count)"}}
        for key in ("assemble_hbm", "grad_contract_hbm", "predict_mean_hbm"):
            r = rl[key]
            if r["peak"]:
                r["frac"] = r["achieved"] / r["peak"]
            r["alu"]["frac"] = r["alu"]["achieved"] / r["alu"]["peak"]
        if not args.no_cpu_baseline and world == 1:
            # headline: ONE BLAS thread, all the reference's gpr path can use (OpenBLAS built with USE_THREAD=0,
            # /root/reference Makefile:3-4; SURVEY F6); courtesy: the same evaluation with every host core
            from threadpoolctl import threadpool_limits
            with threadpool_limits(limits=1):
                dt1, _ = oracle_eval_seconds(x, y, thetas[0], A)
            dt, _ = oracle_eval_seconds(x, y, thetas[0], A)
            out["cpu_baseline"] = {
                "value": 1.0 / dt1, "unit": "evals/s", "cores": 1, "kind": "port",
                "sample": f"1 of the {B} LML+gradient evaluations of one step (n={n}, d={d}), reference-faithful restatement "
                          f"oracle (NumPy + OpenBLAS potrf/potrs/potri, (n,n,d+1) tensor materialised) on 1 BLAS thread: {dt1:.1f} s",
                "all_cores": {"value": 1.0 / dt, "unit": "evals/s", "cores": os.cpu_count(), "seconds_per_eval": dt},
            }
        print(json.dumps(out), flush=True)
    model.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        return {"hbm_gbs": 6650.0, "hbm_source": "fallback (B200_PROFILING.md)"}


if __name__ == "__main__":
    main()
