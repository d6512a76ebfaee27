"""Time of the rebuild of an evicted model (ModelT::rebuild_nu, DESIGN section 3) at n = 4096: a created model and a
model appended to a prior of 4000 rows.  The rebuild time is the first variance request after eviction less the same
request on the resident model.  HBEGP_LIB selects the library to time (A/B builds)."""
import math
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, ".")
import hbetune_rs_b200 as h  # noqa: E402

print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip(), flush=True)
n_prior, n, d, reps = 4000, 4096, 8, 15
for dtype, A in ((h.F64, np.float64), (h.F32, np.float32)):
    rng = np.random.default_rng(2)
    x = rng.random((n, d)).astype(A)
    y = (np.sin(2 * np.pi * x).sum(axis=1) + 1.5).astype(A)
    th = np.array([math.log(0.1), 0.0] + [math.log(1.5)] * d)
    xs = np.random.default_rng(3).random((1, d)).astype(A)
    for kind in ("created", "appended"):
        with h.Context(0, dtype) as ctx:
            ctx.set_resident_models(1)
            if kind == "created":
                ctx.set_data(x, y)
                model = ctx.model(th)
            else:
                ctx.set_data(x[:n_prior], y[:n_prior])
                prior = ctx.model(th)
                ctx.set_data(x, y)
                model = h.Model(ctx, prior=prior)
                assert model.appended
            want = model.predict(xs)
            resident, rebuild, same = [], [], True
            for _ in range(reps + 1):
                t0 = time.perf_counter()
                model.predict(xs)
                resident.append(time.perf_counter() - t0)
                other = ctx.model(th)  # one resident model: `model` is evicted
                t0 = time.perf_counter()
                got = model.predict(xs)
                rebuild.append(time.perf_counter() - t0)
                other.close()
                same &= all(np.array_equal(a, b) for a, b in zip(got, want))
            ms = (np.median(rebuild[1:]) - np.median(resident[1:])) * 1e3
            print(f"{'f64' if A == np.float64 else 'f32'} {kind:8s} n={n} d={d}: rebuild {ms:.3f} ms "
                  f"(median of {reps}; rebuilds {ctx.model_stats()['rebuilds']}; same bits as before eviction: {same})", flush=True)
