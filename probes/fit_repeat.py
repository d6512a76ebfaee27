import sys, time, math
sys.path.insert(0, '.')
import numpy as np
import hbetune_rs_b200 as h
from bench import synth
n, d, restarts = 1024, 8, 32
x, y = synth(n, d)
lo_c = max(np.quantile(y, 0.1) ** 2 * n, 2e-5) / 2; hi_c = 2 * float((y ** 2).sum())
bv = h.BoundedValue
kernel = h.Product(h.ConstantKernel(bv(math.sqrt(lo_c * hi_c), lo_c, hi_c)), h.Matern(2.5, [bv(1.0, 1e-3, 1e3)] * d))
ts = []
for rep in range(6):
    ctx = h.Context()
    t0 = time.perf_counter()
    fk = h.FittedKernel.new(ctx, kernel, x, y, h.RNG.new_with_seed(1), restarts, bv(1.0, 1e-2, 1e1))
    ts.append(time.perf_counter() - t0)
    ctx.close()
print("fit seconds", [round(t, 3) for t in ts], "evals", fk.n_evals, "lml", fk.lml)
