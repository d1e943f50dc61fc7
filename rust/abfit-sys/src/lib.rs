//! Raw bindings to `libabfit.so` — one `extern "C"` item per entry point of `include/abfit.h`.
//!
//! UNTESTED courtesy file: there is no Rust toolchain in the image the library is built in.  The contract is the C
//! header; the binding that IS exercised by the test-suite (same names, same argument order) is the ctypes mirror
//! `alphabeta-rs_b200/__init__.py`.  INTEGRATION.md shows the call-site changes in alphabeta-rs
//! (`src/ab_neutral.rs:13-142`, `src/boot_model.rs:17-115`, `src/alphabeta.rs:23-59`, `src/pedigree.rs:137-262`,
//! `src/cli/metaprofile.rs:50-72`).
//!
//! Conventions (abfit.h): plain pointers and sizes; arrays are caller-owned, row-major, f64 unless noted; every call
//! returns 0 or a negative `abfit_status`, message from `abfit_last_error()` (thread-local); nothing unwinds across the
//! boundary; one `abfit_ctx` per device and host thread; without a CUDA device every compute call fails with
//! `ABFIT_ERR_CUDA` (there is no CPU fallback).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int};

#[repr(C)]
pub struct abfit_ctx {
    _p: [u8; 0],
}
#[repr(C)]
pub struct abfit_batch {
    _p: [u8; 0],
}

pub const ABFIT_OK: c_int = 0;
pub const ABFIT_ERR_ARG: c_int = -1;
pub const ABFIT_ERR_CUDA: c_int = -2;
pub const ABFIT_ERR_TIME: c_int = -3;
pub const ABFIT_ERR_NAN: c_int = -4;
pub const ABFIT_ERR_TOO_LARGE: c_int = -5;
pub const ABFIT_ERR_STATE: c_int = -6;

/// abfit_fit.status
pub const ABFIT_TERM_SD: i32 = 1;
pub const ABFIT_TERM_MAX_ITERS: i32 = 2;
pub const ABFIT_TERM_STALLED: i32 = 3;
pub const ABFIT_TERM_TARGET_COST: i32 = 4;
pub const ABFIT_FIT_NAN: i32 = -1;

/// flags of the fit / bootstrap calls
pub const ABFIT_SHRINK_ON_FAILED_CONTRACTION: u32 = 1;
pub const ABFIT_NO_EARLY_EXIT_ON_STALL: u32 = 2;

/// `Problem` (src/structs.rs:12-19): `pedigree` is the `Pedigree(Array2<f64>)` buffer, rows `[t0, t1, t2, D]`
/// (src/pedigree.rs:32-45); p0mm = 1 - p0uu, p0um = 0 as in src/ab_neutral.rs:23-24.
#[repr(C)]
#[derive(Clone, Copy)]
pub struct abfit_problem {
    pub pedigree: *const f64,
    pub n_pairs: i32,
    pub p0uu: f64,
    pub eqp: f64,
    pub eqp_weight: f64,
}

/// One Nelder-Mead run: theta = `res.state.best_param` (alpha, beta, weight, intercept), cost = `best_cost`,
/// lse = the penalty-free least squares of src/ab_neutral.rs:88-93.
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct abfit_fit {
    pub theta: [f64; 4],
    pub cost: f64,
    pub lse: f64,
    pub iters: i32,
    pub evals: i32,
    pub status: i32,
    pub start_id: i32,
}

/// CG site / gene of the window placement (src/methylation_site.rs:32-45, src/genes.rs:59-96)
#[repr(C)]
#[derive(Clone, Copy)]
pub struct abfit_cg_site {
    pub chromosome: i32,
    pub start: u32,
    pub end: u32,
    pub strand: i32,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct abfit_gene {
    pub chromosome: i32,
    pub start: u32,
    pub end: u32,
    pub strand: i32,
}

extern "C" {
    pub fn abfit_last_error() -> *const c_char;
    pub fn abfit_version() -> *const c_char;
    pub fn abfit_device_count() -> c_int;

    // ---- context ------------------------------------------------------------------------------------------------
    pub fn abfit_ctx_create(device: c_int, out: *mut *mut abfit_ctx) -> c_int;
    pub fn abfit_ctx_destroy(ctx: *mut abfit_ctx);
    pub fn abfit_ctx_sync(ctx: *mut abfit_ctx) -> c_int;

    // ---- seeded input generators: Model::new (src/structs.rs:78-96), Model::vary (:100-128), the residual
    //      resampling of src/boot_model.rs:43-48 ---------------------------------------------------------------------
    pub fn abfit_gen_start_simplices(seed: u64, problem_id: u64, n_starts: i32, max_divergence: f64, out: *mut f64);
    pub fn abfit_gen_vary_vertices(seed: u64, problem_id: u64, n_boot: i32, best_theta: *const f64, out: *mut f64);
    pub fn abfit_gen_resample_idx(seed: u64, problem_id: u64, n_boot: i32, n_pairs: i32, out: *mut i32);

    // ---- the seams of the hot path ----------------------------------------------------------------------------------
    /// `impl CostFunction for Problem` (src/structs.rs:191-217), batched
    pub fn abfit_cost_batch(
        ctx: *mut abfit_ctx, probs: *const abfit_problem, n_probs: i32, prob_of_theta: *const i32, theta: *const f64,
        b: i32, cost_out: *mut f64, lse_out: *mut f64,
    ) -> c_int;
    /// `divergence()` (src/divergence.rs:33-94)
    pub fn abfit_model_divergence(
        ctx: *mut abfit_ctx, prob: *const abfit_problem, theta: *const f64, dt1t2_out: *mut f64, p_uu_out: *mut f64,
    ) -> c_int;
    /// `ab_neutral::run` (src/ab_neutral.rs:13-142) for n_probs windows at once
    pub fn abfit_fit_batch(
        ctx: *mut abfit_ctx, probs: *const abfit_problem, n_probs: i32, n_starts: i32, simplices: *const f64,
        max_iters: i32, sd_tol: f64, flags: u32, best_out: *mut abfit_fit, all_out: *mut abfit_fit, pred_out: *mut f64,
        resid_out: *mut f64, prob_status_out: *mut i32,
    ) -> c_int;
    /// `boot_model::run` (src/boot_model.rs:17-115) for n_probs windows at once
    pub fn abfit_boot_batch(
        ctx: *mut abfit_ctx, probs: *const abfit_problem, n_probs: i32, best: *const abfit_fit, pred: *const f64,
        resid: *const f64, n_boot: i32, resample_idx: *const i32, vary_vertices: *const f64, max_iters: i32, sd_tol: f64,
        flags: u32, rows_out: *mut f64, fits_out: *mut abfit_fit,
    ) -> c_int;
    /// `alphabeta::run` (src/alphabeta.rs:23-59) for every window of a metaprofile (src/cli/metaprofile.rs:50-72)
    pub fn abfit_alphabeta_batch(
        ctx: *mut abfit_ctx, probs: *const abfit_problem, n_probs: i32, n_starts: i32, simplices: *const f64, n_boot: i32,
        resample_idx: *const i32, vary_seed: u64, first_problem_id: u64, max_iters_fit: i32, max_iters_boot: i32,
        sd_tol: f64, flags: u32, best_out: *mut abfit_fit, pred_out: *mut f64, resid_out: *mut f64,
        prob_status_out: *mut i32, rows_out: *mut f64, analysis_out: *mut f64,
    ) -> c_int;
    /// the same with the windows sharded over several GPUs (one context per device)
    pub fn abfit_alphabeta_batch_multi(
        ctxs: *const *mut abfit_ctx, n_ctx: i32, probs: *const abfit_problem, n_probs: i32, n_starts: i32,
        simplices: *const f64, n_boot: i32, resample_idx: *const i32, vary_seed: u64, first_problem_id: u64,
        problem_ids: *const u64, max_iters_fit: i32, max_iters_boot: i32, sd_tol: f64, flags: u32,
        best_out: *mut abfit_fit, pred_out: *mut f64, resid_out: *mut f64, prob_status_out: *mut i32,
        rows_out: *mut f64, analysis_out: *mut f64,
    ) -> c_int;
    /// `DMatrix::from` (src/pedigree.rs:213-262) + per-sample statistics / p0uu (:159-183)
    pub fn abfit_divergence(
        ctx: *mut abfit_ctx, status: *const u8, posterior_max: *const f64, meth_lvl: *const f64, s: i32, l: i64,
        seg_offsets: *const i64, w: i32, thr: f64, d_out: *mut f64, diff_out: *mut u64, cnt_out: *mut u64,
        p0uu_out: *mut f64, methsum_out: *mut f64, nvalid_out: *mut i64,
    ) -> c_int;
    pub fn abfit_divergence_multi(
        ctxs: *const *mut abfit_ctx, n_ctx: i32, status: *const u8, posterior_max: *const f64, meth_lvl: *const f64,
        s: i32, l: i64, seg_offsets: *const i64, w: i32, thr: f64, d_out: *mut f64, diff_out: *mut u64,
        cnt_out: *mut u64, p0uu_out: *mut f64, methsum_out: *mut f64, nvalid_out: *mut i64,
    ) -> c_int;

    // ---- host-side pieces around the path -----------------------------------------------------------------------------
    /// `RawAnalysis::analyze` (src/analysis.rs:50-98): rows [n][7] -> out[32]
    pub fn abfit_analyze(rows: *const f64, n: i32, out: *mut f64) -> c_int;
    /// `steady_state` (src/alphabeta.rs:71-79)
    pub fn abfit_steady_state(alpha: f64, beta: f64) -> f64;
    /// `Pedigree::to_file` (src/pedigree.rs:81-90)
    pub fn abfit_write_pedigree(path: *const c_char, pedigree: *const f64, n_pairs: i32) -> c_int;
    /// `Analysis::to_file` (src/analysis.rs:102-144)
    pub fn abfit_write_analysis(path: *const c_char, analysis: *const f64) -> c_int;
    /// `write_npy` (src/cli/alphabeta.rs:34-35, src/cli/metaprofile.rs:110-111)
    pub fn abfit_write_npy_f64(path: *const c_char, data: *const f64, ndim: i32, shape: *const i64) -> c_int;
    /// `plot::metaplot` (src/plot.rs:6-82): metaplot.png; any of the four interval arrays may be null
    pub fn abfit_plot_metaplot(path: *const c_char, n_windows: i32, alpha: *const f64, beta: *const f64,
                               ci_alpha_lo: *const f64, ci_alpha_hi: *const f64, ci_beta_lo: *const f64,
                               ci_beta_hi: *const f64) -> c_int;
    /// `plot::bootstrap` (src/plot.rs:84-137): bootstrap.png from the bootstrap alphas and betas
    pub fn abfit_plot_bootstrap(path: *const c_char, alphas: *const f64, betas: *const f64, n: i32) -> c_int;
    /// `MethylationSite::from_methylome_file_line` (src/methylation_site.rs:146-362) over a whole file image, in place of
    /// the `BufRead::lines` loops of `Windows::extract` (src/windows.rs:310-330) and `Pedigree::build`
    /// (src/pedigree.rs:137-157).  Every output may be null; `capacity` = number of lines is always enough.
    pub fn abfit_parse_methylome_buffer(buf: *const c_char, len: i64, invert_strand: i32, skip_first_line: i32, capacity: i64,
                                        sites: *mut abfit_cg_site, posterior_max: *mut f64, status: *mut u8,
                                        meth_lvl: *mut f64, line_off: *mut i64, line_len: *mut i32, n_out: *mut i64) -> c_int;
}

/// Message of the last failed call on this thread.
pub fn last_error() -> String {
    unsafe {
        let p = abfit_last_error();
        if p.is_null() {
            String::new()
        } else {
            std::ffi::CStr::from_ptr(p).to_string_lossy().into_owned()
        }
    }
}
