//! Raw bindings to `include/hbegp.h` (kept in the same order as the header).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_double, c_float, c_int, c_long, c_longlong, c_ulonglong, c_void};

pub const HBEGP_F64: c_int = 0;
pub const HBEGP_F32: c_int = 1;

pub const HBEGP_OK: c_int = 0;
pub const HBEGP_NOT_PD: c_int = 1;
pub const HBEGP_ERR_INVALID: c_int = -1;
pub const HBEGP_ERR_CUDA: c_int = -2;
pub const HBEGP_ERR_NOMEM: c_int = -3;
pub const HBEGP_ERR_UNSUPPORTED: c_int = -4;
pub const HBEGP_ERR_NO_CAPTURE: c_int = -5;

pub const HBEGP_PROJ_LINEAR: c_int = 0;
pub const HBEGP_PROJ_LOG: c_int = 1;

#[repr(C)]
pub struct hbegp_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct hbegp_model {
    _private: [u8; 0],
}
#[repr(C)]
pub struct hbegp_batcher {
    _private: [u8; 0],
}
#[repr(C)]
pub struct hbegp_multi {
    _private: [u8; 0],
}
#[repr(C)]
pub struct hbegp_multi_model {
    _private: [u8; 0],
}
pub const HBEGP_COMM_ID_BYTES: usize = 128;

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct hbegp_acq_result {
    pub best_value: c_double,
    pub best_eval: c_longlong,
    pub n_evals: c_longlong,
    pub status: c_int,
    pub reserved: c_int,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct hbegp_run_result {
    pub best_lml: c_double,
    pub best_eval: c_longlong,
    pub n_evals: c_longlong,
    pub final_f: c_double,
    pub status: c_int,
    pub reserved: c_int,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct hbegp_ynorm {
    pub amplitude: c_double,
    pub expected: c_double,
    pub projection: c_int,
    pub dtype: c_int,
}

pub type hbegp_objective_fn =
    Option<unsafe extern "C" fn(x: *const c_double, grad_out: *mut c_double, user: *mut c_void) -> c_double>;

/// Sums `count` doubles in place over all ranks; 0 on success.
pub type hbegp_allreduce_fn = Option<unsafe extern "C" fn(user: *mut c_void, values: *mut c_double, count: c_long) -> c_int>;
/// Batched objective of `hbegp_fit_runs_with`; 0 on success.
pub type hbegp_batch_objective_fn = Option<
    unsafe extern "C" fn(user: *mut c_void, batch: c_int, p: c_int, theta: *const c_double, lml: *mut c_double,
                         grad: *mut c_double, status: *mut c_int) -> c_int,
>;

extern "C" {
    pub fn hbegp_version() -> *const c_char;
    pub fn hbegp_last_error() -> *const c_char;

    pub fn hbegp_ctx_create(device: c_int, dtype: c_int, stream: *mut c_void, out: *mut *mut hbegp_ctx) -> c_int;
    pub fn hbegp_ctx_destroy(ctx: *mut hbegp_ctx) -> c_int;
    pub fn hbegp_ctx_set_workspace_limit(ctx: *mut hbegp_ctx, bytes: c_ulonglong) -> c_int;
    pub fn hbegp_ctx_launch_count(ctx: *mut hbegp_ctx) -> c_longlong;

    pub fn hbegp_set_data(ctx: *mut hbegp_ctx, n: c_long, d: c_int, x: *const c_void, y: *const c_void) -> c_int;
    pub fn hbegp_set_data_device(ctx: *mut hbegp_ctx, n: c_long, d: c_int, x: *const c_void, y: *const c_void) -> c_int;

    pub fn hbegp_lml_grad_batch(
        ctx: *mut hbegp_ctx, nu: c_double, b: c_int, theta: *const c_double, lo: *const c_double,
        hi: *const c_double, lml: *mut c_double, grad: *mut c_double, status: *mut c_int,
    ) -> c_int;

    pub fn hbegp_fit_runs(
        ctx: *mut hbegp_ctx, nu: c_double, n_runs: c_int, starts: *const c_double, bounds_lo: *const c_double,
        bounds_hi: *const c_double, maxeval: c_int, results: *mut hbegp_run_result, best_theta: *mut c_double,
    ) -> c_int;
    pub fn hbegp_fit_runs_sharded(
        ctx: *mut hbegp_ctx, nu: c_double, n_runs: c_int, starts: *const c_double, bounds_lo: *const c_double,
        bounds_hi: *const c_double, maxeval: c_int, rank: c_int, world: c_int, allreduce: hbegp_allreduce_fn,
        allreduce_user: *mut c_void, results: *mut hbegp_run_result, best_theta: *mut c_double,
    ) -> c_int;
    pub fn hbegp_fit_runs_with(
        objective: hbegp_batch_objective_fn, objective_user: *mut c_void, p: c_int, n_runs: c_int,
        starts: *const c_double, bounds_lo: *const c_double, bounds_hi: *const c_double, maxeval: c_int, rank: c_int,
        world: c_int, allreduce: hbegp_allreduce_fn, allreduce_user: *mut c_void, results: *mut hbegp_run_result,
        best_theta: *mut c_double,
    ) -> c_int;
    pub fn hbegp_pick_best_run(n_runs: c_int, results: *const hbegp_run_result) -> c_int;

    // batched objective for a caller-owned optimiser (NLopt, src/util/gradmin.rs:35-60)
    pub fn hbegp_batcher_create(
        ctx: *mut hbegp_ctx, nu: c_double, n_runs: c_int, bounds_lo: *const c_double, bounds_hi: *const c_double,
        out: *mut *mut hbegp_batcher,
    ) -> c_int;
    pub fn hbegp_batcher_eval(
        batcher: *mut hbegp_batcher, run: c_int, theta: *const c_double, lml: *mut c_double, grad: *mut c_double,
        status: *mut c_int,
    ) -> c_int;
    pub fn hbegp_batcher_leave(batcher: *mut hbegp_batcher, run: c_int, final_f: c_double) -> c_int;
    pub fn hbegp_batcher_results(
        batcher: *mut hbegp_batcher, results: *mut hbegp_run_result, best_theta: *mut c_double, n_rounds: *mut c_longlong,
    ) -> c_int;
    pub fn hbegp_batcher_destroy(batcher: *mut hbegp_batcher) -> c_int;
    pub fn hbegp_lbfgs_set_tolerances(ftol: c_double, gtol: c_double) -> c_int;

    // exchange between GPUs inside the library (NCCL)
    pub fn hbegp_comm_unique_id(id_out: *mut c_void) -> c_int; // 128 bytes
    pub fn hbegp_comm_init(ctx: *mut hbegp_ctx, world: c_int, rank: c_int, id: *const c_void) -> c_int;
    pub fn hbegp_comm_info(
        ctx: *mut hbegp_ctx, rank: *mut c_int, world: *mut c_int, nccl_version: *mut c_int, collective_ms: *mut c_double,
        n_collectives: *mut c_longlong,
    ) -> c_int;
    pub fn hbegp_lml_grad_batch_sharded(
        ctx: *mut hbegp_ctx, nu: c_double, b: c_int, theta: *const c_double, lo: *const c_double, hi: *const c_double,
        lml: *mut c_double, grad: *mut c_double, status: *mut c_int,
    ) -> c_int;
    pub fn hbegp_multi_create(n_gpus: c_int, devices: *const c_int, dtype: c_int, out: *mut *mut hbegp_multi) -> c_int;
    pub fn hbegp_multi_destroy(multi: *mut hbegp_multi) -> c_int;
    pub fn hbegp_multi_n_gpus(multi: *const hbegp_multi) -> c_int;
    pub fn hbegp_multi_ctx(multi: *mut hbegp_multi, i: c_int) -> *mut hbegp_ctx;
    pub fn hbegp_multi_set_data(multi: *mut hbegp_multi, n: c_long, d: c_int, x: *const c_void, y: *const c_void) -> c_int;
    pub fn hbegp_multi_lml_grad_batch(
        multi: *mut hbegp_multi, nu: c_double, b: c_int, theta: *const c_double, lo: *const c_double, hi: *const c_double,
        lml: *mut c_double, grad: *mut c_double, status: *mut c_int,
    ) -> c_int;
    pub fn hbegp_multi_fit_runs(
        multi: *mut hbegp_multi, nu: c_double, n_runs: c_int, starts: *const c_double, bounds_lo: *const c_double,
        bounds_hi: *const c_double, maxeval: c_int, results: *mut hbegp_run_result, best_theta: *mut c_double,
    ) -> c_int;
    pub fn hbegp_multi_model_create(
        multi: *mut hbegp_multi, nu: c_double, theta: *const c_double, lo: *const c_double, hi: *const c_double,
        out: *mut *mut hbegp_multi_model, lml: *mut c_double, alpha_out: *mut c_void, kinv_out: *mut c_void,
    ) -> c_int;
    pub fn hbegp_multi_model_destroy(model: *mut hbegp_multi_model) -> c_int;
    pub fn hbegp_multi_model_replica(model: *mut hbegp_multi_model, i: c_int) -> *mut hbegp_model;
    pub fn hbegp_multi_predict(
        model: *mut hbegp_multi_model, m: c_long, xs: *const c_void, mean: *mut c_void, var: *mut c_void,
        n_below_warn: *mut c_long,
    ) -> c_int;

    // retained-model policy (SURVEY F10 / H6)
    pub fn hbegp_ctx_set_resident_models(ctx: *mut hbegp_ctx, max_resident: c_int) -> c_int;
    pub fn hbegp_ctx_model_stats(
        ctx: *mut hbegp_ctx, live: *mut c_int, resident: *mut c_int, evictions: *mut c_longlong, rebuilds: *mut c_longlong,
    ) -> c_int;

    // trait Kernel standalone (src/gpr/kernel.rs:8-43)
    pub fn hbegp_kernel_matrix(
        ctx: *mut hbegp_ctx, nu: c_double, d: c_int, theta: *const c_double, n1: c_long, x1: *const c_void, n2: c_long,
        x2: *const c_void, k_out: *mut c_void,
    ) -> c_int;
    pub fn hbegp_kernel_theta_grad(
        ctx: *mut hbegp_ctx, nu: c_double, d: c_int, theta: *const c_double, n: c_long, x: *const c_void, k_out: *mut c_void,
        grad_out: *mut c_void,
    ) -> c_int;
    pub fn hbegp_kernel_diag(dtype: c_int, d: c_int, theta: *const c_double, n: c_long, diag_out: *mut c_void) -> c_int;
    pub fn hbegp_debug_poison(ctx: *mut hbegp_ctx) -> c_int;

    pub fn hbegp_model_create(
        ctx: *mut hbegp_ctx, nu: c_double, theta: *const c_double, lo: *const c_double, hi: *const c_double,
        out: *mut *mut hbegp_model, lml: *mut c_double, alpha_out: *mut c_void, kinv_out: *mut c_void,
    ) -> c_int;
    pub fn hbegp_model_extend(
        ctx: *mut hbegp_ctx, prior: *mut hbegp_model, out: *mut *mut hbegp_model, lml: *mut c_double,
        alpha_out: *mut c_void, kinv_out: *mut c_void, appended: *mut c_int,
    ) -> c_int;
    pub fn hbegp_model_destroy(model: *mut hbegp_model) -> c_int;
    pub fn hbegp_model_n(model: *const hbegp_model) -> c_long;
    pub fn hbegp_model_dim(model: *const hbegp_model) -> c_int;

    pub fn hbegp_predict(
        model: *mut hbegp_model, m: c_long, xs: *const c_void, mean: *mut c_void, var: *mut c_void,
        n_below_warn: *mut c_long,
    ) -> c_int;
    pub fn hbegp_predict_warn_values(model: *const hbegp_model, cap: c_int, values_out: *mut c_double, rows_out: *mut c_long) -> c_int;
    pub fn hbegp_predict_sharded(
        model: *mut hbegp_model, m: c_long, xs: *const c_void, mean: *mut c_void, var: *mut c_void, n_below_warn: *mut c_long,
    ) -> c_int;
    pub fn hbegp_predict_device(
        model: *mut hbegp_model, m: c_long, xs_device: *const c_void, mean_device: *mut c_void,
        var_device: *mut c_void, n_below_warn_device: *mut c_long,
    ) -> c_int;

    pub fn hbegp_predict_mean_ei(
        model: *mut hbegp_model, yn: *const hbegp_ynorm, m: c_long, xs: *const c_void, fmin: c_double,
        mean_out: *mut c_void, ei_out: *mut c_void, best_index: *mut c_long, n_below_warn: *mut c_long,
    ) -> c_int;
    pub fn hbegp_predict_confidence_bound(
        model: *mut hbegp_model, yn: *const hbegp_ynorm, m: c_long, xs: *const c_void, cb: c_double,
        out: *mut c_void, best_index: *mut c_long, n_below_warn: *mut c_long,
    ) -> c_int;

    pub fn hbegp_predict_grad(
        model: *mut hbegp_model, m: c_long, xs: *const c_void, mean: *mut c_void, var: *mut c_void, dmean: *mut c_void,
        dvar: *mut c_void, n_below_warn: *mut c_long,
    ) -> c_int;
    pub fn hbegp_predict_mean_ei_grad(
        model: *mut hbegp_model, yn: *const hbegp_ynorm, m: c_long, xs: *const c_void, fmin: c_double,
        mean_out: *mut c_void, ei_out: *mut c_void, dmean_out: *mut c_void, dei_out: *mut c_void, n_below_warn: *mut c_long,
    ) -> c_int;
    pub fn hbegp_predict_confidence_bound_grad(
        model: *mut hbegp_model, yn: *const hbegp_ynorm, m: c_long, xs: *const c_void, cb: c_double,
        out: *mut c_void, dout: *mut c_void, n_below_warn: *mut c_long,
    ) -> c_int;

    // acquisition search on the device: S bounded L-BFGS searches in lockstep (see hbegp.h)
    pub fn hbegp_acquire_ei(
        model: *mut hbegp_model, yn: *const hbegp_ynorm, fmin: c_double, n_starts: c_long, starts: *const c_void,
        lo: *const c_double, hi: *const c_double, maxeval: c_int, x_out: *mut c_void, mean_out: *mut c_void,
        results: *mut hbegp_acq_result, best_index: *mut c_long, n_rounds: *mut c_longlong,
    ) -> c_int;
    pub fn hbegp_acquire_confidence_bound(
        model: *mut hbegp_model, yn: *const hbegp_ynorm, cb: c_double, n_starts: c_long, starts: *const c_void,
        lo: *const c_double, hi: *const c_double, maxeval: c_int, x_out: *mut c_void, results: *mut hbegp_acq_result,
        best_index: *mut c_long, n_rounds: *mut c_longlong,
    ) -> c_int;

    pub fn hbegp_minimize_by_gradient(
        objective: hbegp_objective_fn, user: *mut c_void, n: c_int, x: *mut c_double, lo: *const c_double,
        hi: *const c_double, maxeval: c_int, f_out: *mut c_double,
    ) -> c_int;

    pub fn hbegp_rng_seed(seed: c_ulonglong, state: *mut c_ulonglong);
    pub fn hbegp_rng_fork(state: *mut c_ulonglong, child: *mut c_ulonglong);
    pub fn hbegp_rng_uniform(state: *mut c_ulonglong, lo: c_double, hi: c_double) -> c_double;

    pub fn hbegp_ynorm_fit(
        dtype: c_int, projection: c_int, n: c_long, y: *const c_void, known_optimum: *const c_double,
        y_normalized_out: *mut c_void, out: *mut hbegp_ynorm,
    ) -> c_int;
    pub fn hbegp_ynorm_apply(
        yn: *const hbegp_ynorm, op: c_int, n: c_long, a: *const c_void, b: *const c_void, out: *mut c_void,
    ) -> c_int;
    pub fn hbegp_estimate_amplitude(dtype: c_int, n: c_long, y: *const c_void, bounds: *const c_double, out: *mut c_double) -> c_int;
    pub fn hbegp_expected_improvement(mean: c_double, std: c_double, fmin: c_double) -> c_double;
    pub fn hbegp_expected_improvement_a(
        dtype: c_int, m: c_long, mean: *const c_void, var: *const c_void, fmin: c_double, ei_out: *mut c_void,
    ) -> c_int;
    pub fn hbegp_normal_inverse_cdf(p: c_double, mean: c_double, std: c_double) -> c_double;

    pub fn hbegp_bench_phase(
        ctx: *mut hbegp_ctx, nu: c_double, b: c_int, theta: *const c_double, phase: c_int, reps: c_int,
        ms_out: *mut c_float,
    ) -> c_int;
    pub fn hbegp_debug_factor(
        ctx: *mut hbegp_ctx, nu: c_double, theta: *const c_double, k: *mut c_void, w: *mut c_void,
        kinv: *mut c_void, status: *mut c_int,
    ) -> c_int;
}
