"""Host-side mirror of the reference's ``src/gpr`` surface on top of the C ABI.

Kernel *objects* only carry hyper-parameters and bounds (``BoundedValue``, ``ConstantKernel``,
``Matern``, ``Product`` — same names and theta conventions as ``src/gpr/*_kernel.rs``); every kernel
*evaluation* happens on the GPU inside ``libhbegp.so``.
"""
from __future__ import annotations

import ctypes as C
import math
import sys
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import check, lib


class BoundsError(ValueError):
    """``src/util/bounded_value.rs:72-77``."""

    def __init__(self, value, lo, hi):
        super().__init__(f"value {value} violated bounds [{lo}, {hi}]")
        self.value, self.min, self.max = value, lo, hi


@dataclass(frozen=True)
class BoundedValue:
    """``src/util/bounded_value.rs:3-56``."""

    value: float
    min: float
    max: float

    def __post_init__(self):
        if not (self.min <= self.value <= self.max):
            raise BoundsError(self.value, self.min, self.max)

    def with_value(self, value):
        return BoundedValue(value, self.min, self.max)

    def with_clamped_value(self, value):
        if value < self.min:
            value = self.min
        elif self.max < value:
            value = self.max
        return BoundedValue(value, self.min, self.max)


class ConstantKernel:
    """``src/gpr/constant_kernel.rs:9-67`` (parameters only)."""

    def __init__(self, constant: BoundedValue):
        self.constant = constant

    def n_params(self):
        return 1

    def theta(self):
        return [math.log(self.constant.value)]

    def with_theta(self, theta):
        (t,) = theta
        return ConstantKernel(self.constant.with_value(math.exp(t)))

    def with_clamped_theta(self, theta):
        (t,) = theta
        return ConstantKernel(self.constant.with_clamped_value(math.exp(t)))

    def bounds(self):
        return [(math.log(self.constant.min), math.log(self.constant.max))]

    def natural_bounds(self):
        return [(self.constant.min, self.constant.max)]


class Matern:
    """``src/gpr/matern_kernel.rs:12-187`` (parameters only; nu in {0.5, 1.5, 2.5}, or ``math.inf`` for the squared
    exponential (RBF) kernel exp(-0.5 |x / l - x' / l|^2), sklearn's ``RBF`` and ``Matern(nu=np.inf)``)."""

    def __init__(self, nu: float, length_scale: Sequence[BoundedValue]):
        self.nu = nu
        self.length_scale = list(length_scale)

    def n_params(self):
        return len(self.length_scale)

    def theta(self):
        return [math.log(b.value) for b in self.length_scale]

    def with_theta(self, theta):
        assert len(theta) == self.n_params()
        return Matern(self.nu, [b.with_value(math.exp(t)) for t, b in zip(theta, self.length_scale)])

    def with_clamped_theta(self, theta):
        assert len(theta) == self.n_params()
        return Matern(self.nu, [b.with_clamped_value(math.exp(t)) for t, b in zip(theta, self.length_scale)])

    def bounds(self):
        return [(math.log(b.min), math.log(b.max)) for b in self.length_scale]

    def natural_bounds(self):
        return [(b.min, b.max) for b in self.length_scale]


class Product:
    """``src/gpr/product_kernel.rs:8-109`` specialised like the reference's production kernel
    ``Product<ConstantKernel, Matern>`` (``src/core/gpr.rs:51``)."""

    def __init__(self, k1: ConstantKernel, k2: Matern):
        self.k1, self.k2 = k1, k2

    def n_params(self):
        return self.k1.n_params() + self.k2.n_params()

    def theta(self):
        return self.k1.theta() + self.k2.theta()

    def with_theta(self, theta):
        assert len(theta) == self.n_params()
        return Product(self.k1.with_theta(theta[:1]), self.k2.with_theta(theta[1:]))

    def with_clamped_theta(self, theta):
        assert len(theta) == self.n_params()
        return Product(self.k1.with_clamped_theta(theta[:1]), self.k2.with_clamped_theta(theta[1:]))

    def bounds(self):
        return self.k1.bounds() + self.k2.bounds()

    def natural_bounds(self):
        return self.k1.natural_bounds() + self.k2.natural_bounds()

    # ---- trait Kernel evaluation (src/gpr/kernel.rs:8-43), on the GPU through the C ABI
    def kernel(self, ctx: "Context", x1, x2) -> np.ndarray:
        """``Kernel::kernel(x1, x2) -> (n1, n2)`` (``kernel.rs:10-14``, ``product_kernel.rs:36-38``)."""
        x1 = np.ascontiguousarray(x1, dtype=ctx.A)
        x2 = np.ascontiguousarray(x2, dtype=ctx.A)
        assert x1.ndim == 2 and x2.ndim == 2 and x1.shape[1] == x2.shape[1] == self.k2.n_params()
        out = np.empty((x1.shape[0], x2.shape[0]), dtype=ctx.A)
        theta = np.array(self.theta(), dtype=np.float64)
        check(lib.hbegp_kernel_matrix(ctx._h, self.k2.nu, x1.shape[1], _ptr(theta), x1.shape[0], _ptr(x1), x2.shape[0],
                                      _ptr(x2), _ptr(out)), "hbegp_kernel_matrix")
        return out

    def theta_grad(self, ctx: "Context", x) -> Tuple[np.ndarray, np.ndarray]:
        """``Kernel::theta_grad(x) -> ((n, n), (n, n, n_params))`` (``kernel.rs:16-21``, ``product_kernel.rs:40-70``)."""
        x = np.ascontiguousarray(x, dtype=ctx.A)
        n, d = x.shape
        assert d == self.k2.n_params()
        k = np.empty((n, n), dtype=ctx.A)
        g = np.empty((n, n, d + 1), dtype=ctx.A)
        theta = np.array(self.theta(), dtype=np.float64)
        check(lib.hbegp_kernel_theta_grad(ctx._h, self.k2.nu, d, _ptr(theta), n, _ptr(x), _ptr(k), _ptr(g)),
              "hbegp_kernel_theta_grad")
        return k, g

    def diag(self, ctx: "Context", x) -> np.ndarray:
        """``Kernel::diag(x) -> (n)`` (``kernel.rs:23-24``, ``product_kernel.rs:72-74``)."""
        n = np.asarray(x).shape[0]
        out = np.empty(n, dtype=ctx.A)
        theta = np.array(self.theta(), dtype=np.float64)
        check(lib.hbegp_kernel_diag(ctx.dtype, self.k2.n_params(), _ptr(theta), n, _ptr(out)), "hbegp_kernel_diag")
        return out


def _np_dtype(dtype: int):
    return np.float64 if dtype == _lib.F64 else np.float32


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Context:
    """One GPU context (``hbegp_ctx``).  ``stream`` is a raw ``cudaStream_t`` (e.g.
    ``torch.cuda.current_stream().cuda_stream``) or None."""

    def __init__(self, device: int = 0, dtype: int = _lib.F64, stream: Optional[int] = None):
        self.dtype = dtype
        self.A = _np_dtype(dtype)
        h = C.c_void_p()
        # stream == 0 is the legacy default stream: pass its explicit handle (cudaStreamLegacy = 0x1), since
        # NULL asks the library to create its own stream
        sh = None if stream is None else C.c_void_p(stream if stream != 0 else 1)
        check(lib.hbegp_ctx_create(device, dtype, sh, C.byref(h)), "hbegp_ctx_create")
        self._h = h
        self.n = self.d = 0

    def close(self):
        if getattr(self, "_h", None):
            lib.hbegp_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def launch_count(self) -> int:
        return int(lib.hbegp_ctx_launch_count(self._h))

    def set_resident_models(self, max_resident: int):
        """``hbegp_ctx_set_resident_models``: how many models keep their n x n factor on the device."""
        check(lib.hbegp_ctx_set_resident_models(self._h, max_resident), "hbegp_ctx_set_resident_models")

    def model_stats(self):
        live, res = C.c_int(), C.c_int()
        ev, rb = C.c_longlong(), C.c_longlong()
        check(lib.hbegp_ctx_model_stats(self._h, C.byref(live), C.byref(res), C.byref(ev), C.byref(rb)), "hbegp_ctx_model_stats")
        return {"live": live.value, "resident": res.value, "evictions": ev.value, "rebuilds": rb.value}

    def set_workspace_limit(self, nbytes: int):
        check(lib.hbegp_ctx_set_workspace_limit(self._h, nbytes), "hbegp_ctx_set_workspace_limit")

    def set_data(self, x: np.ndarray, y: np.ndarray):
        x = np.ascontiguousarray(x, dtype=self.A)
        y = np.ascontiguousarray(y, dtype=self.A)
        assert x.ndim == 2 and y.shape == (x.shape[0],)
        check(lib.hbegp_set_data(self._h, x.shape[0], x.shape[1], _ptr(x), _ptr(y)), "hbegp_set_data")
        self.n, self.d = x.shape

    def set_data_device(self, n: int, d: int, x_ptr: int, y_ptr: int):
        check(lib.hbegp_set_data_device(self._h, n, d, C.c_void_p(x_ptr), C.c_void_p(y_ptr)), "hbegp_set_data_device")
        self.n, self.d = n, d

    def lml_grad_batch(self, theta: np.ndarray, nu: float = 2.5, lo=None, hi=None, want_grad: bool = True):
        theta = np.ascontiguousarray(np.atleast_2d(theta), dtype=np.float64)
        B, p = theta.shape
        assert p == self.d + 2
        lo = None if lo is None else np.ascontiguousarray(lo, dtype=np.float64)
        hi = None if hi is None else np.ascontiguousarray(hi, dtype=np.float64)
        lml = np.empty(B)
        grad = np.empty((B, p)) if want_grad else None
        status = np.empty(B, dtype=np.int32)
        check(lib.hbegp_lml_grad_batch(self._h, nu, B, _ptr(theta), _ptr(lo), _ptr(hi), _ptr(lml), _ptr(grad),
                                       _ptr(status)), "hbegp_lml_grad_batch")
        return lml, grad, status

    # ---- exchange between GPUs inside the library (NCCL on device buffers)
    @staticmethod
    def comm_unique_id() -> bytes:
        """``hbegp_comm_unique_id``: 128 bytes rank 0 hands to every rank (over any side channel)."""
        buf = C.create_string_buffer(128)
        check(lib.hbegp_comm_unique_id(buf), "hbegp_comm_unique_id")
        return buf.raw

    def comm_init(self, world: int, rank: int, unique_id: bytes):
        """``hbegp_comm_init``: joins this context (one per process / GPU) to an NCCL communicator of ``world`` ranks."""
        check(lib.hbegp_comm_init(self._h, world, rank, C.create_string_buffer(unique_id, 128)), "hbegp_comm_init")
        self.comm_rank, self.comm_world = rank, world

    def comm_info(self):
        rank, world, ver = C.c_int(), C.c_int(), C.c_int()
        ms, cnt = C.c_double(), C.c_longlong()
        check(lib.hbegp_comm_info(self._h, C.byref(rank), C.byref(world), C.byref(ver), C.byref(ms), C.byref(cnt)), "hbegp_comm_info")
        return {"rank": rank.value, "world": world.value, "nccl_version": ver.value, "collective_ms": ms.value,
                "n_collectives": cnt.value}

    def lml_grad_batch_sharded(self, theta: np.ndarray, nu: float = 2.5, lo=None, hi=None, want_grad: bool = True):
        """``hbegp_lml_grad_batch_sharded``: every rank passes the same thetas and gets all results; rank r evaluates
        thetas r, r + world, ...; one ncclAllGather of the device-resident records."""
        theta = np.ascontiguousarray(np.atleast_2d(theta), dtype=np.float64)
        B, p = theta.shape
        lo = None if lo is None else np.ascontiguousarray(lo, dtype=np.float64)
        hi = None if hi is None else np.ascontiguousarray(hi, dtype=np.float64)
        lml = np.empty(B)
        grad = np.empty((B, p)) if want_grad else None
        status = np.empty(B, dtype=np.int32)
        check(lib.hbegp_lml_grad_batch_sharded(self._h, nu, B, _ptr(theta), _ptr(lo), _ptr(hi), _ptr(lml), _ptr(grad),
                                               _ptr(status)), "hbegp_lml_grad_batch_sharded")
        return lml, grad, status

    def fit_runs(self, starts: np.ndarray, lo, hi, nu: float = 2.5, maxeval: int = 150, rank: int = 0, world: int = 1,
                 allreduce=None):
        """``hbegp_fit_runs``; with ``world > 1`` the balanced multi-process loop (``hbegp_fit_runs_sharded``):
        ``allreduce(array)`` must sum the float64 array in place over all ranks, or None to let the library exchange
        the rounds itself over the communicator of ``comm_init`` (ncclAllReduce on the device-resident record)."""
        starts = np.ascontiguousarray(np.atleast_2d(starts), dtype=np.float64)
        R, p = starts.shape
        lo = np.ascontiguousarray(lo, dtype=np.float64)
        hi = np.ascontiguousarray(hi, dtype=np.float64)
        res = (_lib.RunResult * R)()
        best_theta = np.empty((R, p))
        if world == 1:
            check(lib.hbegp_fit_runs(self._h, nu, R, _ptr(starts), _ptr(lo), _ptr(hi), maxeval, res, _ptr(best_theta)),
                  "hbegp_fit_runs")
        else:
            cb = _lib.allreduce_callback(allreduce) if allreduce is not None else _lib.ALLREDUCE_FN()  # NULL: library NCCL
            check(lib.hbegp_fit_runs_sharded(self._h, nu, R, _ptr(starts), _ptr(lo), _ptr(hi), maxeval, rank, world, cb, None,
                                             res, _ptr(best_theta)), "hbegp_fit_runs_sharded")
        return res, best_theta

    def bench_phase(self, theta, phase: int, reps: int = 3, nu: float = 2.5) -> float:
        """Average milliseconds of a truncated batched evaluation (see hbegp_bench_phase)."""
        theta = np.ascontiguousarray(np.atleast_2d(theta), dtype=np.float64)
        ms = C.c_float()
        check(lib.hbegp_bench_phase(self._h, nu, theta.shape[0], _ptr(theta), phase, reps, C.byref(ms)), "hbegp_bench_phase")
        return float(ms.value)

    def debug_poison(self):
        check(lib.hbegp_debug_poison(self._h), "hbegp_debug_poison")

    def debug_factor(self, theta, nu: float = 2.5, want=("k", "w", "kinv")):
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        out = {k: (np.empty((self.n, self.n), dtype=self.A) if k in want else None) for k in ("k", "w", "kinv")}
        st = C.c_int(0)
        check(lib.hbegp_debug_factor(self._h, nu, _ptr(theta), _ptr(out["k"]), _ptr(out["w"]),
                                     _ptr(out["kinv"]), C.byref(st)), "hbegp_debug_factor")
        out["status"] = st.value
        return out

    def model(self, theta, nu: float = 2.5, lo=None, hi=None, want_alpha=True, want_kinv=False) -> "Model":
        return Model(self, theta, nu, lo, hi, want_alpha, want_kinv)


class Model:
    """A fitted model resident on the GPU (``hbegp_model``): X, alpha and L^-1 stay in HBM."""

    def __init__(self, ctx: Context, theta=None, nu=2.5, lo=None, hi=None, want_alpha=True, want_kinv=False,
                 prior: Optional["Model"] = None):
        self.ctx, self.A = ctx, ctx.A
        self.alpha = np.empty(ctx.n, dtype=self.A) if want_alpha else None
        self.k_inv = np.empty((ctx.n, ctx.n), dtype=self.A) if want_kinv else None
        h = C.c_void_p()
        lml = C.c_double()
        self.appended = False
        if prior is not None:
            # hbegp_model_extend: the prior's parameters on the context's current data (block append when possible)
            appended = C.c_int(0)
            rc = lib.hbegp_model_extend(ctx._h, prior._h, C.byref(h), C.byref(lml), _ptr(self.alpha), _ptr(self.k_inv),
                                        C.byref(appended))
            what = "hbegp_model_extend"
            self.appended = bool(appended.value)
        else:
            theta = np.ascontiguousarray(theta, dtype=np.float64)
            lo = None if lo is None else np.ascontiguousarray(lo, dtype=np.float64)
            hi = None if hi is None else np.ascontiguousarray(hi, dtype=np.float64)
            rc = lib.hbegp_model_create(ctx._h, nu, _ptr(theta), _ptr(lo), _ptr(hi), C.byref(h), C.byref(lml),
                                        _ptr(self.alpha), _ptr(self.k_inv))
            what = "hbegp_model_create"
        if rc == _lib.NOT_PD:
            raise np.linalg.LinAlgError("Kernel matrix must be invertible.")  # fit.rs:55 panics here
        check(rc, what)
        self._h = h
        self.lml = lml.value
        self.n, self.d = ctx.n, ctx.d

    def close(self):
        if getattr(self, "_h", None):
            lib.hbegp_model_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def predict(self, xs: np.ndarray, want_variance: bool = True, warn: bool = True):
        xs = np.ascontiguousarray(xs, dtype=self.A)
        assert xs.ndim == 2 and xs.shape[1] == self.d
        m = xs.shape[0]
        mean = np.empty(m, dtype=self.A)
        var = np.empty(m, dtype=self.A) if want_variance else None
        nb = C.c_long(0)
        check(lib.hbegp_predict(self._h, m, _ptr(xs), _ptr(mean), _ptr(var), C.byref(nb)), "hbegp_predict")
        self.n_below_warn = nb.value
        if warn and nb.value:
            # predict.rs:39-46 lists the offending values with {:.2e}
            vals, _ = self.warn_values()
            more = "" if len(vals) == nb.value else f", ... ({nb.value} in all)"
            print("Variances below 0 were predicted and will be corrected: "
                  + ", ".join(f"{v:.2e}" for v in vals) + more, file=sys.stderr)
        return mean, var

    def predict_grad(self, xs: np.ndarray, want_variance: bool = True):
        """``hbegp_predict_grad``: (mean, var, dmean, dvar) with dmean / dvar of shape (m, d), the gradients in the
        candidate (normalised units; var and dvar are None unless wanted).  Values as ``predict``."""
        xs = np.ascontiguousarray(xs, dtype=self.A)
        assert xs.ndim == 2 and xs.shape[1] == self.d
        m = xs.shape[0]
        mean = np.empty(m, dtype=self.A)
        var = np.empty(m, dtype=self.A) if want_variance else None
        dmean = np.empty((m, self.d), dtype=self.A)
        dvar = np.empty((m, self.d), dtype=self.A) if want_variance else None
        nb = C.c_long(0)
        check(lib.hbegp_predict_grad(self._h, m, _ptr(xs), _ptr(mean), _ptr(var), _ptr(dmean), _ptr(dvar), C.byref(nb)),
              "hbegp_predict_grad")
        self.n_below_warn = nb.value
        return mean, var, dmean, dvar

    def single_handle(self):
        return self._h

    def warn_values(self, cap: int = 16):
        """The pre-clamp variances below -sqrt(1e-5) of the last prediction, in row order, with their rows
        (``hbegp_predict_warn_values``; ``predict.rs:39-46``, ``:104-127``)."""
        vals = np.empty(cap)
        rows = np.empty(cap, dtype=np.int64)
        k = check(lib.hbegp_predict_warn_values(self._h, cap, _ptr(vals), _ptr(rows)), "hbegp_predict_warn_values")
        return vals[:k], rows[:k]

    def predict_sharded(self, xs: np.ndarray, want_variance: bool = True):
        """``hbegp_predict_sharded``: every rank passes all rows and gets all results; contiguous row blocks per rank,
        one ncclAllGather of the device-resident (mean, variance) shards."""
        xs = np.ascontiguousarray(xs, dtype=self.A)
        m = xs.shape[0]
        mean = np.empty(m, dtype=self.A)
        var = np.empty(m, dtype=self.A) if want_variance else None
        nb = C.c_long(0)
        check(lib.hbegp_predict_sharded(self._h, m, _ptr(xs), _ptr(mean), _ptr(var), C.byref(nb)), "hbegp_predict_sharded")
        self.n_below_warn = nb.value
        return mean, var

    def predict_device(self, m: int, xs_ptr: int, mean_ptr: int, var_ptr: Optional[int] = None):
        check(lib.hbegp_predict_device(self._h, m, C.c_void_p(xs_ptr), C.c_void_p(mean_ptr),
                                       C.c_void_p(var_ptr) if var_ptr else None, None), "hbegp_predict_device")


class MultiContext:
    """``hbegp_multi``: ONE process over several GPUs (the reference is one process, ``src/bin/hbetune/main.rs:255-355``).
    Thetas / live runs are dealt round-robin to the GPUs, candidate rows go out in contiguous blocks, data and model are
    replicated with ncclBroadcast; results are bit-identical to one GPU."""

    def __init__(self, n_gpus: int, dtype: int = _lib.F64, devices: Optional[Sequence[int]] = None):
        self.dtype, self.A = dtype, _np_dtype(dtype)
        h = C.c_void_p()
        dev = None if devices is None else np.ascontiguousarray(devices, dtype=np.int32)
        check(lib.hbegp_multi_create(n_gpus, _ptr(dev), dtype, C.byref(h)), "hbegp_multi_create")
        self._h = h
        self.n_gpus = n_gpus
        self.n = self.d = 0

    def close(self):
        if getattr(self, "_h", None):
            lib.hbegp_multi_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        self.close()

    def set_data(self, x, y):
        x = np.ascontiguousarray(x, dtype=self.A)
        y = np.ascontiguousarray(y, dtype=self.A)
        check(lib.hbegp_multi_set_data(self._h, x.shape[0], x.shape[1], _ptr(x), _ptr(y)), "hbegp_multi_set_data")
        self.n, self.d = x.shape

    def lml_grad_batch(self, theta, nu: float = 2.5, lo=None, hi=None):
        theta = np.ascontiguousarray(np.atleast_2d(theta), dtype=np.float64)
        B, p = theta.shape
        lo = None if lo is None else np.ascontiguousarray(lo, dtype=np.float64)
        hi = None if hi is None else np.ascontiguousarray(hi, dtype=np.float64)
        lml, grad, status = np.empty(B), np.empty((B, p)), np.empty(B, dtype=np.int32)
        check(lib.hbegp_multi_lml_grad_batch(self._h, nu, B, _ptr(theta), _ptr(lo), _ptr(hi), _ptr(lml), _ptr(grad), _ptr(status)),
              "hbegp_multi_lml_grad_batch")
        return lml, grad, status

    def fit_runs(self, starts, lo, hi, nu: float = 2.5, maxeval: int = 150):
        starts = np.ascontiguousarray(np.atleast_2d(starts), dtype=np.float64)
        R, p = starts.shape
        lo = np.ascontiguousarray(lo, dtype=np.float64)
        hi = np.ascontiguousarray(hi, dtype=np.float64)
        res = (_lib.RunResult * R)()
        best_theta = np.empty((R, p))
        check(lib.hbegp_multi_fit_runs(self._h, nu, R, _ptr(starts), _ptr(lo), _ptr(hi), maxeval, res, _ptr(best_theta)),
              "hbegp_multi_fit_runs")
        return res, best_theta

    def model(self, theta, nu: float = 2.5, lo=None, hi=None, want_alpha=True, want_kinv=False) -> "MultiModel":
        return MultiModel(self, theta, nu, lo, hi, want_alpha, want_kinv)


class MultiModel:
    """``hbegp_multi_model``: one evaluation on GPU 0, replicas on the other GPUs over NVLink."""

    def __init__(self, mctx: MultiContext, theta, nu=2.5, lo=None, hi=None, want_alpha=True, want_kinv=False):
        self.mctx = self.ctx = mctx
        self.A, self.n, self.d = mctx.A, mctx.n, mctx.d
        self.appended = False
        self.alpha = np.empty(mctx.n, dtype=self.A) if want_alpha else None
        self.k_inv = np.empty((mctx.n, mctx.n), dtype=self.A) if want_kinv else None
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        lo = None if lo is None else np.ascontiguousarray(lo, dtype=np.float64)
        hi = None if hi is None else np.ascontiguousarray(hi, dtype=np.float64)
        h, lml = C.c_void_p(), C.c_double()
        rc = lib.hbegp_multi_model_create(mctx._h, nu, _ptr(theta), _ptr(lo), _ptr(hi), C.byref(h), C.byref(lml),
                                          _ptr(self.alpha), _ptr(self.k_inv))
        if rc == _lib.NOT_PD:
            raise np.linalg.LinAlgError("Kernel matrix must be invertible.")
        check(rc, "hbegp_multi_model_create")
        self._h, self.lml = h, lml.value

    def close(self):
        if getattr(self, "_h", None):
            lib.hbegp_multi_model_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def single_handle(self):
        """GPU 0's replica as a plain ``hbegp_model`` (for the single-GPU acquisition epilogues)."""
        return C.c_void_p(lib.hbegp_multi_model_replica(self._h, 0))

    def predict(self, xs, want_variance: bool = True, warn: bool = True):
        xs = np.ascontiguousarray(xs, dtype=self.A)
        m = xs.shape[0]
        mean = np.empty(m, dtype=self.A)
        var = np.empty(m, dtype=self.A) if want_variance else None
        nb = C.c_long(0)
        check(lib.hbegp_multi_predict(self._h, m, _ptr(xs), _ptr(mean), _ptr(var), C.byref(nb)), "hbegp_multi_predict")
        self.n_below_warn = nb.value
        if warn and nb.value:
            print(f"Variances below 0 were predicted and will be corrected: {nb.value} value(s) over {self.mctx.n_gpus} GPUs",
                  file=sys.stderr)
        return mean, var


@dataclass
class FittedKernel:
    """``src/gpr/fit.rs:6-12``; ``model`` is the device-resident counterpart of (alpha, k_inv)."""

    kernel: Product
    noise: BoundedValue
    alpha: np.ndarray
    k_inv: Optional[np.ndarray]
    lml: float
    model: Model
    n_evals: int = 0

    @staticmethod
    def _theta_bounds(kernel: Product, noise: BoundedValue):
        lo = np.array([noise.min] + [b[0] for b in kernel.natural_bounds()])
        hi = np.array([noise.max] + [b[1] for b in kernel.natural_bounds()])
        return lo, hi

    @classmethod
    def new(cls, ctx: Context, kernel: Product, x_train, y_train, rng, n_restarts_optimizer: int,
            noise: BoundedValue, maxeval: int = 150, want_kinv: bool = False, shard=None) -> "FittedKernel":
        """``FittedKernel::new`` (``src/gpr/fit.rs:18-31, 71-176``).  ``rng`` needs ``uniform_inclusive``;
        start points are drawn in reference order (``gradmin.rs:21-24``) before any optimisation runs.
        ``shard`` (optional) distributes the runs over processes: either a callable
        ``(starts, run_fn) -> (results, thetas)`` (static split, ``dist.sharded_fit_runs``) or an object with a
        ``fit_runs(ctx, starts, lo, hi, nu, maxeval)`` method (``dist.BalancedFit``: per-round balancing)."""
        ctx.set_data(x_train, y_train)
        lo, hi = cls._theta_bounds(kernel, noise)
        tb = [(math.log(a), math.log(b)) for a, b in zip(lo, hi)]
        theta0 = [math.log(noise.value)] + kernel.theta()
        starts = [theta0] + [[rng.uniform_inclusive(a, b) for a, b in tb] for _ in range(n_restarts_optimizer)]
        starts = np.array(starts, dtype=np.float64)
        nu = kernel.k2.nu
        if shard is None:
            res, thetas = ctx.fit_runs(starts, lo, hi, nu, maxeval)
        elif hasattr(shard, "fit_runs"):
            res, thetas = shard.fit_runs(ctx, starts, lo, hi, nu, maxeval)
        else:
            res, thetas = shard(starts, lambda s: ctx.fit_runs(s, lo, hi, nu, maxeval))
        best = lib.hbegp_pick_best_run(len(res), res)
        if best < 0:
            raise RuntimeError("called `Option::unwrap()` on a `None` value")  # fit.rs:161
        theta = thetas[best]
        k = kernel.with_clamped_theta(list(theta[1:]))
        nz = noise.with_clamped_value(float(ctx.A(math.exp(theta[0]))))
        model = ctx.model(theta, nu, lo, hi, want_alpha=True, want_kinv=want_kinv)
        return cls(k, nz, model.alpha, model.k_inv, res[best].best_lml, model, sum(r.n_evals for r in res))

    @classmethod
    def extend(cls, ctx: Context, kernel: Product, x_train, y_train, noise: BoundedValue,
               want_kinv: bool = False, prior: Optional["FittedKernel"] = None) -> "FittedKernel":
        """``FittedKernel::extend`` (``src/gpr/fit.rs:33-68``): one evaluation, no optimisation.

        With ``prior`` (the fitted kernel being extended, i.e. the reference's ``self``) whose model is still
        resident on ``ctx``, the library appends the new rows to the prior factorisation when the old rows are an
        unchanged prefix of ``x_train`` (``hbegp_model_extend``) instead of refactorising everything."""
        ctx.set_data(x_train, y_train)
        theta = np.array([math.log(noise.value)] + kernel.theta())
        try:
            pm = getattr(prior, "model", None)
            if (isinstance(pm, Model) and isinstance(ctx, Context) and getattr(pm, "_h", None) and pm.ctx is ctx
                    and prior.noise.value == noise.value and prior.kernel.theta() == kernel.theta()
                    and prior.kernel.k2.nu == kernel.k2.nu):
                model = Model(ctx, want_alpha=True, want_kinv=want_kinv, prior=pm)
            else:
                model = ctx.model(theta, kernel.k2.nu, None, None, want_alpha=True, want_kinv=want_kinv)
        except np.linalg.LinAlgError:
            raise RuntimeError("Kernel matrix must be invertible.")
        return cls(kernel, noise, model.alpha, model.k_inv, model.lml, model, 1)


def predict(fitted: FittedKernel, x, want_variance: Optional[np.ndarray] = None):
    """``src/gpr/predict.rs:7-52``: returns the mean; fills ``want_variance`` in place when given."""
    mean, var = fitted.model.predict(x, want_variance is not None)
    if want_variance is not None:
        want_variance[...] = var
    return mean
