/*
 * abfit.h — C ABI of libabfit, the B200 (sm_100a) implementation of the
 * alphabeta-rs model-fitting hot path.
 *
 * alphabeta-rs has no FFI/plugin layer; the seams this library replaces are
 * Rust function signatures (SURVEY.md §8b).  Each entry point below names the
 * reference interface it stands in for (paths relative to the alphabeta-rs
 * repository).  INTEGRATION.md shows the Rust `extern "C"` block and the
 * three call-site changes a maintainer would make.
 *
 * Conventions
 *  - plain pointers and sizes only; all arrays are caller-owned, row-major, f64
 *    unless noted;
 *  - every call returns 0 on success or a negative abfit_status; a message is
 *    available from abfit_last_error() (thread-local);
 *  - nothing here runs on the CPU: without a CUDA device every compute call
 *    fails with ABFIT_ERR_CUDA — there is no fallback path;
 *  - a context owns one CUDA device and one stream; use one context per host
 *    thread (multi-GPU = one context per device, problems sharded by window).
 *
 * Arithmetic contract: identical to the reference's operation order
 * (FMA chains only inside the 3x3 products, everything else unfused IEEE-754
 * binary64, pair sums accumulated sequentially in pedigree order), so results
 * are reproducible bit for bit against the CPU restatement in oracle/.
 */
#ifndef ABFIT_H
#define ABFIT_H
#ifndef __CUDACC_RTC__ /* the library's run-time kernel build supplies the fixed-width types itself */
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct abfit_ctx abfit_ctx;
typedef struct abfit_batch abfit_batch;

typedef enum {
    ABFIT_OK = 0,
    ABFIT_ERR_ARG = -1,      /* bad argument (null pointer, negative size, ...) */
    ABFIT_ERR_CUDA = -2,     /* CUDA runtime / no device */
    ABFIT_ERR_TIME = -3,     /* pedigree row violates 0 <= t0 <= t1,t2 <= 127 (src/divergence.rs:17-19,52) */
    ABFIT_ERR_NAN = -4,      /* a value on which the reference panics (NaN divergence, p0uu+p0mm != 1, ...) */
    ABFIT_ERR_TOO_LARGE = -5,/* per-lane model state of one problem exceeds shared memory */
    ABFIT_ERR_STATE = -6     /* batch call sequence violated (e.g. boot before fit) */
} abfit_status;

/* per-fit termination status (abfit_fit.status) */
enum {
    ABFIT_TERM_SD = 1,        /* sample sd of the simplex costs < sd_tol (argmin NelderMead::terminate) */
    ABFIT_TERM_MAX_ITERS = 2, /* iter >= max_iters (argmin Executor) */
    ABFIT_TERM_STALLED = 3,   /* failed inside contraction left the simplex unchanged: every further
                                 iteration is identical, so the fit returns what the reference returns
                                 after max_iters; iters is reported as max_iters */
    ABFIT_TERM_TARGET_COST = 4, /* best cost is -inf (argmin Executor: best_cost <= target_cost = -inf); tested
                                   after the sd and max_iters tests, so those win when they fire too */
    ABFIT_FIT_NAN = -1        /* best cost is NaN: the reference panics on best_param.unwrap().  This happens
                                 exactly when vertex 0 of the start simplex costs NaN (a NaN never moves in the
                                 stable sort, so it stays the best vertex); theta then holds that vertex, cost is
                                 NaN and lse its penalty-free cost */
};

/* flags for fit/boot calls */
enum {
    ABFIT_SHRINK_ON_FAILED_CONTRACTION = 1, /* later-argmin behaviour; default (0) = argmin 0.8.1 */
    ABFIT_NO_EARLY_EXIT_ON_STALL = 2        /* burn all max_iters iterations like the reference */
};

/* One ABneutral problem = one window's pedigree.
 * Replaces `Problem` (src/structs.rs:12-19) / the arguments of ab_neutral::run
 * (src/ab_neutral.rs:13-20): `pedigree` is the reference's `Pedigree(Array2<f64>)`
 * buffer, n_pairs rows of [t0, t1, t2, D] (src/pedigree.rs:32-45).
 * p0mm = 1 - p0uu and p0um = 0 are derived as in src/ab_neutral.rs:23-24. */
typedef struct {
    const double *pedigree; /* [n_pairs][4] */
    int32_t n_pairs;
    double p0uu;       /* Pr(UU) at G0 */
    double eqp;        /* equilibrium target of the penalty (alphabeta.rs passes p0uu) */
    double eqp_weight; /* penalty weight (alphabeta.rs passes 1.0) */
} abfit_problem;

/* Result of one Nelder-Mead run.  theta = [alpha, beta, weight, intercept] is
 * `res.state.best_param` (src/ab_neutral.rs:66), cost = state.best_cost,
 * lse = penalty-free least squares used for best-of-starts (src/ab_neutral.rs:88-93). */
typedef struct {
    double theta[4];
    double cost;
    double lse;
    int32_t iters;
    int32_t evals;    /* objective evaluations executed by this fit (for FLOP accounting) */
    int32_t status;   /* ABFIT_TERM_* / ABFIT_FIT_NAN */
    int32_t start_id; /* index of the start / replicate inside its problem */
} abfit_fit;

const char *abfit_last_error(void);
const char *abfit_version(void);

/* ---- context ------------------------------------------------------------ */
/* CUDA devices visible to this process (0 without a driver) */
int abfit_device_count(void);
int abfit_ctx_create(int device, abfit_ctx **out);
void abfit_ctx_destroy(abfit_ctx *ctx);
/* device properties the bench reports: sm count, max SM clock (kHz), HBM bytes */
int abfit_ctx_info(abfit_ctx *ctx, int32_t *sm_count, int32_t *sm_clock_khz, int64_t *mem_bytes);
/* CUDA-event stopwatch on the context stream (bench.py times its steps on the device with it) */
int abfit_ctx_timer_start(abfit_ctx *ctx);
int abfit_ctx_timer_stop(abfit_ctx *ctx, float *ms_out); /* records, synchronises, returns elapsed ms */
int abfit_ctx_sync(abfit_ctx *ctx);
/* FP64 peak micro-benchmark (independent DFMA chains on every SM); TFLOP/s, FMA = 2 */
int abfit_measure_fp64_peak(abfit_ctx *ctx, double *tflops_out);

/* ---- host-side input generators ------------------------------------------
 * `north_star`: random starts and bootstrap resamples are produced on the host
 * from a seed and fed to every implementation.  Counter-based (splitmix64 keyed
 * by seed, problem, start/replicate, vertex, coordinate), so any shard can be
 * generated independently.  Distributions follow the reference:                 */
/* Model::new (src/structs.rs:78-96): alpha, beta = 10^U(-9,-2); weight ~ U(0,0.1);
 * intercept ~ U(0, max_div) (max_div <= 0 -> 0.1); out [n_starts][5][4] */
void abfit_gen_start_simplices(uint64_t seed, uint64_t problem_id, int32_t n_starts, double max_divergence,
                               double *out);
/* Model::vary (src/structs.rs:100-128): x -> U(x-0.1|x|, x+0.1|x|) (x == 0 -> U(0.09,0.11));
 * out [n_boot][4][4] */
void abfit_gen_vary_vertices(uint64_t seed, uint64_t problem_id, int32_t n_boot, const double best_theta[4],
                             double *out);
/* the same for n_probs windows (problem ids first_problem_id + p, theta of best[p]), on all host cores;
 * out [n_probs][n_boot][4][4] */
void abfit_gen_vary_vertices_batch(uint64_t seed, uint64_t first_problem_id, int32_t n_probs, int32_t n_boot,
                                   const abfit_fit *best, double *out);
/* residual resampling with replacement (src/boot_model.rs:43-48); out [n_boot][n_pairs] */
void abfit_gen_resample_idx(uint64_t seed, uint64_t problem_id, int32_t n_boot, int32_t n_pairs, int32_t *out);

/* ---- one-shot host-buffer entry points (what the Rust FFI binds) ---------- */

/* Objective only.  Replaces `<Problem as CostFunction>::cost` (src/structs.rs:191-217).
 * theta [B][4]; prob_of_theta [B] selects the problem of each theta (NULL: all problem 0);
 * cost_out [B] (with penalty), lse_out [B] (without; may be NULL). */
int abfit_cost_batch(abfit_ctx *ctx, const abfit_problem *probs, int32_t n_probs, const int32_t *prob_of_theta,
                     const double *theta, int32_t B, double *cost_out, double *lse_out);

/* Theoretical divergence of every pair.  Replaces `divergence()` (src/divergence.rs:33-94)
 * for one problem and one theta; dt1t2_out [n_pairs], p_uu_out = p_uu_est(alpha,beta). */
int abfit_model_divergence(abfit_ctx *ctx, const abfit_problem *prob, const double theta[4], double *dt1t2_out,
                           double *p_uu_out);

/* Multi-start ABneutral fit of n_probs windows.  Replaces `ab_neutral::run`
 * (src/ab_neutral.rs:13-142), batched over windows (the reference loops windows
 * serially in src/cli/metaprofile.rs:50-72).
 *  simplices  [n_probs][n_starts][5][4]  start simplices (Model::new x 5, src/ab_neutral.rs:49-55)
 *  max_iters  10000 in the reference (src/ab_neutral.rs:61); sd_tol = DBL_EPSILON (argmin default)
 *  best_out   [n_probs]            best-of-starts by lse, ties -> lowest start id
 *  all_out    [n_probs][n_starts]  every start's result (may be NULL)
 *  pred_out / resid_out  [sum n_pairs] predicted divergence and residuals of the best
 *             model, problems concatenated (src/ab_neutral.rs:123-135; may be NULL)
 *  prob_status_out [n_probs] 0 or ABFIT_ERR_NAN where the reference would panic (may be NULL) */
int abfit_fit_batch(abfit_ctx *ctx, const abfit_problem *probs, int32_t n_probs, int32_t n_starts,
                    const double *simplices, int32_t max_iters, double sd_tol, uint32_t flags,
                    abfit_fit *best_out, abfit_fit *all_out, double *pred_out, double *resid_out,
                    int32_t *prob_status_out);

/* Bootstrap refits.  Replaces `boot_model::run` (src/boot_model.rs:17-115) up to and
 * including the raw result rows (statistics: abfit_analyze).
 *  best        [n_probs]  model to perturb (theta used)         (src/boot_model.rs:19,70)
 *  pred, resid [sum n_pairs]                                    (src/boot_model.rs:20-21)
 *  resample_idx  [n_probs][n_boot][n_pairs_p] concatenated per problem  (:43-48)
 *  vary_vertices [n_probs][n_boot][4][4]                        (:71-74)
 *  max_iters   1000 in the reference (:81)
 *  rows_out    [n_probs][n_boot][7] = alpha,beta,weight,intercept,pr_mm,pr_um,pr_uu (:86-91)
 *  fits_out    [n_probs][n_boot] (may be NULL) */
int abfit_boot_batch(abfit_ctx *ctx, const abfit_problem *probs, int32_t n_probs, const abfit_fit *best,
                     const double *pred, const double *resid, int32_t n_boot, const int32_t *resample_idx,
                     const double *vary_vertices, int32_t max_iters, double sd_tol, uint32_t flags,
                     double *rows_out, abfit_fit *fits_out);

/* Fit, then bootstrap, every window: replaces `alphabeta::run` (src/alphabeta.rs:23-59: ab_neutral::run :33-41
 * followed by boot_model::run :42-54) for all windows of a metaprofile in one call (the reference loops the
 * windows serially, src/cli/metaprofile.rs:50-72).  The vary vertices depend on each window's best model; they are
 * the numbers abfit_gen_vary_vertices(vary_seed, first_problem_id + window, ...) returns, drawn on the device right
 * behind the best-of-starts selection (same counter-based generator, same bits), so the bootstrap starts without a
 * round trip through the host.  The start simplices cross PCIe while the host compiles the pedigrees, the resample
 * indices under the multi-start kernel, and the fit results come back under the bootstrap kernel.
 *  resample_idx  as in abfit_boot_batch, or NULL: the indices are drawn on the device, as boot_model::run draws its own
 *                (src/boot_model.rs:43-48) — the numbers abfit_gen_resample_idx(vary_seed, first_problem_id + window
 *                [or problem_ids[window]], n_boot, n_pairs) returns, without generating and copying 4 n_boot n_pairs
 *                bytes per window on the host
 *  rows_out      [n_probs][n_boot][7]   (required)
 *  analysis_out  [n_probs][32]          RawAnalysis::analyze per window (may be NULL)
 *  best_out, pred_out, resid_out, prob_status_out as in abfit_fit_batch (may be NULL) */
int abfit_alphabeta_batch(abfit_ctx *ctx, const abfit_problem *probs, int32_t n_probs, int32_t n_starts,
                          const double *simplices, int32_t n_boot, const int32_t *resample_idx, uint64_t vary_seed,
                          uint64_t first_problem_id, int32_t max_iters_fit, int32_t max_iters_boot, double sd_tol,
                          uint32_t flags, abfit_fit *best_out, double *pred_out, double *resid_out,
                          int32_t *prob_status_out, double *rows_out, double *analysis_out);

/* The same over several GPUs of one box (SURVEY.md §8e; the reference's window loop src/cli/metaprofile.rs:50-72 is
 * serial): one context per device (ctxs[0..n_ctx)), one host thread per context, contiguous balanced blocks of windows;
 * every shard writes its windows' results straight into the caller's arrays, in window order.  The shards never
 * exchange data — no collective.  Window p of the call keeps its generator key whatever the sharding:
 * problem_ids[p] when given (e.g. the window's position in the genome, so that dropping an empty window does not
 * change its neighbours' bootstrap), else first_problem_id + p.  Bit-identical to one device. */
int abfit_alphabeta_batch_multi(abfit_ctx *const *ctxs, int32_t n_ctx, const abfit_problem *probs, int32_t n_probs,
                                int32_t n_starts, const double *simplices, int32_t n_boot, const int32_t *resample_idx,
                                uint64_t vary_seed, uint64_t first_problem_id, const uint64_t *problem_ids,
                                int32_t max_iters_fit, int32_t max_iters_boot, double sd_tol, uint32_t flags,
                                abfit_fit *best_out, double *pred_out, double *resid_out, int32_t *prob_status_out,
                                double *rows_out, double *analysis_out);

/* Observed pairwise divergence + p0uu.  Replaces `DMatrix::from` (src/pedigree.rs:213-262)
 * and the per-sample statistics of `Pedigree::build` (src/pedigree.rs:159-183).
 *  status        [S][L] u8: 0 = U, 1 = I, 2 = M (src/methylation_site.rs:130-136); other values are not
 *                checked and count as 2
 *  posterior_max [S][L], meth_lvl [S][L] (rc.meth.lvl)
 *  seg_offsets   [W+1] site ranges of W windows over the L axis, or NULL (one window = all sites)
 *  thr           posterior_max_filter (0.99).  A site is valid where posterior_max >= thr: a NaN posterior, or
 *                thr = NaN, makes it invalid (src/pedigree.rs:249-251); meth_lvl of an invalid site is never read
 *  D_out    [W][S(S-1)/2]  diff/(2*cnt) in pair order (0,1),(0,2)...(S-2,S-1); 0/0 = NaN
 *  diff_out, cnt_out [W][S(S-1)/2] exact integer sums (may be NULL)
 *  p0uu_out [W] = mean_s(1 - methsum/nvalid) (may be NULL)
 *  methsum_out [W][S] sum of meth_lvl over valid sites, nvalid_out [W][S] (may be NULL): the raw
 *           per-sample partials, so site-sharded callers (one shard per GPU) can add them up.
 * Windows of at most 65536 sites accumulate methsum sequentially in site order (bit-identical
 * to the reference); longer ones use a fixed-shape blocked tree (deterministic, <= 1e-12 rel). */
int abfit_divergence(abfit_ctx *ctx, const uint8_t *status, const double *posterior_max, const double *meth_lvl,
                     int32_t S, int64_t L, const int64_t *seg_offsets, int32_t W, double thr, double *D_out,
                     uint64_t *diff_out, uint64_t *cnt_out, double *p0uu_out, double *methsum_out,
                     int64_t *nvalid_out);

/* abfit_divergence over several GPUs (one context per device).  With seg_offsets the WINDOWS are sharded: every
 * shard sums meth_lvl in the tree one device picks for the whole window list, so all outputs are bit-identical to
 * abfit_divergence on one device, for any W (W = 1 runs on the first context).  seg_offsets = NULL (whole
 * methylomes, src/pedigree.rs:213-262 at 200 x 5 M sites): the SITE axis is sharded; the exact integer sums of every
 * shard are added on the host, so D is bit-identical for any number of devices, and p0uu agrees within 1e-12
 * (per-sample sums added in device order). */
int abfit_divergence_multi(abfit_ctx *const *ctxs, int32_t n_ctx, const uint8_t *status, const double *posterior_max,
                           const double *meth_lvl, int32_t S, int64_t L, const int64_t *seg_offsets, int32_t W, double thr,
                           double *D_out, uint64_t *diff_out, uint64_t *cnt_out, double *p0uu_out, double *methsum_out,
                           int64_t *nvalid_out);

/* The same with the three input arrays already in device memory (site tables that stay resident between
 * calls; bench: HBM roofline of the packing pass).  seg_offsets and all outputs are host memory.  The call runs on
 * the context's own non-blocking stream, which does not wait for work on other streams: the inputs must be complete
 * (e.g. the stream that wrote them synchronised) before the call.
 * kernel_ms[0] = device time of the packing pass (streams 17 B per sample-site), kernel_ms[1] = all-pairs
 * popcounts + finalisation; launches_out = kernels launched.  Both may be NULL. */
int abfit_divergence_device(abfit_ctx *ctx, const uint8_t *d_status, const double *d_posterior_max,
                            const double *d_meth_lvl, int32_t S, int64_t L, const int64_t *seg_offsets, int32_t W,
                            double thr, double *D_out, uint64_t *diff_out, uint64_t *cnt_out, double *p0uu_out,
                            double *methsum_out, int64_t *nvalid_out, float kernel_ms[2], int32_t *launches_out);

/* ---- staged, device-resident interface ------------------------------------
 * Same computation as abfit_fit_batch + abfit_boot_batch, split into upload /
 * run / download so a caller (bench.py, the metaprofile driver) can keep inputs
 * resident in HBM and overlap transfers.  run_* only enqueue kernels on the
 * context stream and record CUDA events around them. */
int abfit_batch_create(abfit_ctx *ctx, const abfit_problem *probs, int32_t n_probs, abfit_batch **out);
void abfit_batch_destroy(abfit_batch *b);
int abfit_batch_upload_starts(abfit_batch *b, int32_t n_starts, const double *simplices);
int abfit_batch_run_fit(abfit_batch *b, int32_t max_iters, double sd_tol, uint32_t flags);
int abfit_batch_download_fit(abfit_batch *b, abfit_fit *best_out, abfit_fit *all_out, double *pred_out,
                             double *resid_out, int32_t *prob_status_out);
/* best == NULL: use the best-of-starts already on the device (needs run_fit first) */
int abfit_batch_upload_boot(abfit_batch *b, int32_t n_boot, const abfit_fit *best, const double *pred,
                            const double *resid, const int32_t *resample_idx, const double *vary_vertices);
int abfit_batch_run_boot(abfit_batch *b, int32_t max_iters, double sd_tol, uint32_t flags);
int abfit_batch_download_boot(abfit_batch *b, double *rows_out, abfit_fit *fits_out);
/* run_fit + run_boot of an uploaded batch as ONE pipelined pass: the windows are cut into sub-batches, each a
 * fit -> select -> bootstrap chain on its own stream, so that the long fits that end every multi-start launch and the
 * bootstraps overlap with the next sub-batch's fits (what abfit_alphabeta_batch does internally).  Same results as
 * run_fit followed by run_boot.  abfit_batch_timing then reports the whole span as ms[0]. */
int abfit_batch_run_pipelined(abfit_batch *b, int32_t max_iters_fit, int32_t max_iters_boot, double sd_tol, uint32_t flags);
/* sub-batches abfit_batch_run_pipelined uses for this batch (1: no overlap possible) */
int abfit_batch_pipes(abfit_batch *b);
int abfit_batch_sync(abfit_batch *b);
/* device times of the last run_fit / run_boot (ms, CUDA events on the context stream):
 * ms[0] multi-start NM kernel, ms[1] best-of-starts select, ms[2] bootstrap NM kernel;
 * evals[0], evals[1]: objective evaluations executed by the start / bootstrap kernels;
 * launches: kernels launched by the last run_fit + run_boot. Synchronises the stream. */
int abfit_batch_timing(abfit_batch *b, float ms[3], int64_t evals[2], int32_t *launches);
/* algorithmic FLOPs of one objective evaluation of problem p:
 * 45(Tmax-1) + 56 U + 5 N + 40 (SURVEY.md §8d) */
int abfit_batch_flops_per_eval(abfit_batch *b, int32_t p, double *flops_out, int32_t *n_triples_out,
                               int32_t *tmax_out);
/* FP64 instructions one fit executes per objective evaluation of problem p (an FMA counts once).  Under the
 * bit-exact arithmetic contract only the 3x3 products are FMAs, so this is larger than flops / 2; the ratio is
 * the ceiling of the FMA-roofline fraction (bench.py: roofline.pipe_frac). */
int abfit_batch_fp64_instr_per_eval(abfit_batch *b, int32_t p, double *instr_out);
/* 1 when the batch's Nelder-Mead kernels are the run-time specialised ones (a batch whose windows all share one
 * pedigree time structure — every metaprofile — gets its micro-op program compiled to straight-line code with
 * NVRTC; policy and environment switches: csrc/abfit_api.cu::decide_jit), 0 for the interpreter kernels.  Results
 * are bit-identical either way. */
int abfit_batch_uses_specialised_kernels(abfit_batch *b);
/* why the last attempt to build or load specialised kernels failed in this process ("" if none did); the batch
 * concerned ran on the interpreter kernels */
const char *abfit_jit_last_error(void);
/* Diagnostic (no GPU needed): writes the CUDA C++ source specialised for `prob`'s pedigree to source_path and, when
 * cubin_path is not NULL, compiles it with NVRTC for sm_100a and writes the cubin (tests build the same source
 * for the host and compare it with the oracle; cuobjdump -sass on the cubin shows what the GPU runs). */
int abfit_jit_dump(const abfit_problem *prob, const char *source_path, const char *cubin_path, double *compile_seconds);

/* ---- site -> window assignment (host) ---------------------------------------
 * Replaces MethylationSite::is_in_gene / find_gene / place_in_windows (src/methylation_site.rs:368-490),
 * Windows::new (src/windows.rs:28-44), the gene-caching loop of Windows::extract (src/windows.rs:331-337)
 * and Windows::distribution (src/windows.rs:158-165).  Integer and f64-compare logic, bit-exact.
 * chromosome: Chromosome::Numbered(n) -> n, Mitochondrial -> 256, Chloroplast -> 257 (src/methylation_site.rs:49-68);
 * strand: +1 Sense, -1 Antisense, 0 Unknown ('*', equal to anything: src/genes.rs:88-96). */
typedef struct {
    int32_t chromosome;
    uint32_t start, end;
    int32_t strand;
} abfit_gene; /* `Gene` (src/genes.rs:117-125), annotation order */
typedef struct {
    int32_t chromosome;
    uint32_t start, end;
    int32_t strand;
} abfit_cg_site; /* `MethylationSite` (src/methylation_site.rs:32-45), file order */
typedef struct {
    uint32_t window_size, window_step; /* step 0 = window_size (src/extract.rs:26-28) */
    uint32_t cutoff;
    uint32_t max_gene_length; /* 100 unless absolute (src/extract.rs:49-58) */
    int32_t absolute, cutoff_gene_length;
} abfit_window_args; /* the fields of `arguments::Windows` the placement reads (src/arguments.rs:14-55) */
/* windows per region: upstream, gene, downstream (Windows::new) */
int abfit_window_counts(const abfit_window_args *args, int32_t n_windows_out[3]);
/* distribution_out [n_up + n_gene + n_down]: sites per window, upstream || gene || downstream;
 * the optional assignment list (site index, flat window index) holds every (site, window) hit in site
 * order — n_assign_out returns how many there are, at most assign_cap are written. */
int abfit_place_sites(const abfit_gene *genes, int32_t n_genes, const abfit_cg_site *sites, int64_t n_sites,
                      const abfit_window_args *args, int32_t *distribution_out, int64_t *n_assign_out,
                      int64_t assign_cap, int64_t *assign_site, int32_t *assign_window);

/* ---- post-processing ------------------------------------------------------ */
/* Replaces RawAnalysis::analyze (src/analysis.rs:50-98). rows [n][7] -> out[32]: 8 means,
 * 8 sds (ddof 1), 8 (q0.025, q0.975) pairs, field order alpha, beta, beta/alpha, weight,
 * intercept, pr_mm, pr_um, pr_uu. Host only (O(n) per window). */
int abfit_analyze(const double *rows, int32_t n, double out[32]);

/* ---- input files (host parsing; the observed divergence of the pedigree runs on the GPU) ------------
 * MethylationSite::from_methylome_file_line (src/methylation_site.rs:146-362): 0 = parsed, 1 = not a site
 * (header, non-CG context, malformed), < 0 = error.  status_out: 0 U / 1 I / 2 M. */
int abfit_parse_methylome_line(const char *line, int32_t invert_strand, abfit_cg_site *site_out, double *posterior_max_out,
                               int32_t *status_out, double *meth_lvl_out);
/* Pedigree::build (src/pedigree.rs:92-193) + DMatrix::convert (:264-337): nodelist + edgelist + the methylome files the
 * nodelist names (relative to the CWD, as in the reference) -> pedigree rows [t0, t1, t2, D] and p0uu. */
/* The same parser over a whole file image (the reference reads its methylome files line by line on rayon threads,
 * src/extract.rs:75, src/windows.rs:310-330, src/pedigree.rs:137-157).  Lines are split like BufRead::lines ('\n', one
 * trailing '\r' stripped); skip_first_line != 0 drops the header row unparsed (Windows::extract, src/windows.rs:322).
 * Every output may be NULL; each has room for `capacity` entries (the number of lines is always enough).  status: 0 U /
 * 1 I / 2 M.  line_off / line_len: where each accepted line sits in buf.  *n_out = accepted lines, in file order; with
 * all outputs NULL the call only counts.  Host only, multi-threaded (ABFIT_HOST_THREADS overrides the thread count).
 * Returns ABFIT_ERR_ARG when capacity is too small (*n_out is still set). */
int abfit_parse_methylome_buffer(const char *buf, int64_t len, int32_t invert_strand, int32_t skip_first_line, int64_t capacity,
                                 abfit_cg_site *sites, double *posterior_max, uint8_t *status, double *meth_lvl,
                                 int64_t *line_off, int32_t *line_len, int64_t *n_out);
typedef struct abfit_pedigree abfit_pedigree;
int abfit_pedigree_build(abfit_ctx *ctx, const char *nodelist_path, const char *edgelist_path, double posterior_max_filter,
                         abfit_pedigree **out);
int abfit_pedigree_info(const abfit_pedigree *p, int32_t *n_pairs, double *p0uu, int32_t *n_samples, int64_t *n_sites);
const double *abfit_pedigree_rows(const abfit_pedigree *p); /* [n_pairs][4] */
/* The graph part alone (metaprofile: same nodes and edges for every window, only D changes): the measured nodes' file
 * names ('\n'-separated, nodelist order) and per pedigree row (i, j, t0, t1, t2), i < j sample indices. */
int abfit_pedigree_graph(const char *nodelist_path, const char *edgelist_path, int32_t *n_samples_out, char *files_out,
                         int32_t files_cap, int32_t *n_pairs_out, double *pairs_out /*[n_pairs][5]*/, int32_t pairs_cap);
/* Gene::from_annotation_file_line (src/genes.rs:166-216): 0 = parsed, 1 = not a gene line */
int abfit_parse_annotation_line(const char *line, int32_t invert_strand, abfit_gene *gene_out);
const char *abfit_pedigree_warnings(const abfit_pedigree *p);
void abfit_pedigree_free(abfit_pedigree *p);

/* ---- result files of the reference, byte for byte (host) ------------------------
 * f64 exactly as Rust's `{}` prints it (shortest round-trip digits, never scientific, "1" not "1.0", "NaN", "inf");
 * returns the length or ABFIT_ERR_ARG when buf is too small */
int abfit_format_f64(double v, char *buf, int32_t cap);
/* steady_state (src/alphabeta.rs:71-79) */
double abfit_steady_state(double alpha, double beta);
/* Pedigree::to_file (src/pedigree.rs:81-90): "time0\ttime1\ttime2\tD.value" + one row per pair */
int abfit_write_pedigree(const char *path, const double *pedigree, int32_t n_pairs);
/* Analysis::to_file / Display (src/analysis.rs:102-187) from abfit_analyze's out[32] */
int abfit_write_analysis(const char *path, const double analysis[32]);
int abfit_format_analysis(const double analysis[32], char *buf, int32_t cap);
/* write_npy of raw.npy (src/cli/alphabeta.rs:34-35; 3-D in src/cli/metaprofile.rs:110-111): NPY v1.0, '<f8', C order */
int abfit_write_npy_f64(const char *path, const double *data, int32_t ndim, const int64_t *shape);
/* results.txt of `metaprofile ... alphabeta` (src/cli/metaprofile.rs:74-99); region 0/1/2 = upstream/gene/downstream,
 * analysis [n_windows][32] from abfit_analyze / abfit_alphabeta_batch */
int abfit_write_metaprofile_results(const char *path, const char *run_name, int32_t n_windows, const int32_t *cg_count,
                                    const int32_t *region, const abfit_fit *best, const double *analysis,
                                    const double *obs_steady_state);

/* ---- simulated methylomes under ABneutral (data with known epimutation rates) --------------------------
 * A pedigree forest: every node has at most one parent, generations do not decrease from parent to child and lie in
 * 0..127 (the `as i8` time cast of src/divergence.rs:52).  A root at generation g draws its state (UU, UM, MM) from
 * sv0.G^g with sv0 = [p0uu, w(1-p0uu), (1-w)(1-p0uu)] (divergence()'s sv0 with p0mm = 1 - p0uu, p0um = 0,
 * src/ab_neutral.rs:23-24); a child draws from row state(parent) of G^(gen(child) - gen(parent)), G = genmatrix(alpha,
 * beta), powers by matrix_power's chain under the arithmetic contract above.  Every sampled node gives one output row:
 * status 0/1/2 (U/I/M), meth_lvl = status / 2, posterior_max = 1, or 0.5 with probability missing_rate (independent per
 * sample and site).  Measurement error (the fit's intercept) is not simulated.
 * Randomness is counter-based: every draw is keyed by (seed, node index, global site index), so a site range gives the
 * same bits whether it is simulated in one call, in several calls (first_site) or on several devices. */
typedef struct abfit_sim_tree abfit_sim_tree;
typedef struct {
    double alpha, beta;  /* per-generation gain / loss rates, [0, 1] */
    double weight, p0uu; /* founder distribution (see above), [0, 1]; abfit_sim_equilibrium gives the steady state */
    double missing_rate; /* [0, 1] */
    uint64_t seed;
} abfit_sim_params;
/* nodelist + edgelist (the files abfit_pedigree_build reads; an edge's `from` is the parent).  Refused with
 * ABFIT_ERR_ARG: a node with two parents, a cycle, gen(from) > gen(to), a generation above 127, an edge naming an
 * unknown node.  Sampled nodes (meth == Y) give the output rows, in nodelist order. */
int abfit_sim_tree_build(const char *nodelist_path, const char *edgelist_path, abfit_sim_tree **out);
/* the same from arrays: parent [n_nodes] (-1 = root), generation [n_nodes], sampled [n_nodes] (0 / 1) */
int abfit_sim_tree_from_arrays(int32_t n_nodes, const int32_t *parent, const int32_t *generation, const uint8_t *sampled,
                               abfit_sim_tree **out);
int abfit_sim_tree_info(const abfit_sim_tree *t, int32_t *n_nodes, int32_t *n_samples, int32_t *n_pairs);
/* pedigree rows (i, j, t0, t1, t2) of the sampled nodes, in the order and with the values abfit_pedigree_graph gives
 * for the same files: the D column of pair (i, j) is entry (i, j) of abfit_divergence on the simulated rows */
int abfit_sim_tree_pairs(const abfit_sim_tree *t, double *pairs_out /*[n_pairs][5]*/, int32_t pairs_cap);
/* the per-node draw table [n_nodes][6]: for parent state k the pair (c0, c1) = (r0, r0 + r1) of row k of G^delta; a
 * root's pair (of sv0.G^g) is stored three times.  A draw u in [0, 1) gives u < c0 ? 0 : u < c1 ? 1 : 2. */
int abfit_sim_tree_thresholds(const abfit_sim_tree *t, const abfit_sim_params *params, double *out);
void abfit_sim_tree_free(abfit_sim_tree *t);
/* the founders at the model's steady state: p0uu = p_uu_est(alpha, beta), weight = p_um / (p_um + p_mm)
 * (src/alphabeta.rs:62-79, src/structs.rs:146-159) */
int abfit_sim_equilibrium(double alpha, double beta, double *p0uu_out, double *weight_out);
/* sites [first_site, first_site + L) of every sampled node into host arrays status [S][L] u8, posterior_max [S][L],
 * meth_lvl [S][L] (the layout abfit_divergence reads) */
int abfit_simulate(abfit_ctx *ctx, const abfit_sim_tree *tree, const abfit_sim_params *params, int64_t first_site, int64_t L,
                   uint8_t *status, double *posterior_max, double *meth_lvl);
/* the same into device arrays (e.g. the inputs of abfit_divergence_device: 17 bytes per sample-site never cross
 * PCIe); runs on the context stream and returns when the arrays are written.  kernel_ms: device time of the
 * simulation kernel (may be NULL). */
int abfit_simulate_device(abfit_ctx *ctx, const abfit_sim_tree *tree, const abfit_sim_params *params, int64_t first_site,
                          int64_t L, uint8_t *d_status, double *d_posterior_max, double *d_meth_lvl, float *kernel_ms);

/* ---- the reference's pictures (host; src/plot.rs) ------------------------------------
 * 1280 x 960 PNG files with the reference's series, colours, axis ranges and captions (not its pixels: own
 * rasteriser and bitmap font, see csrc/abfit_plot.cu).
 * metaplot.png of `metaprofile ... alphabeta` (src/plot.rs:6-82, called at src/cli/metaprofile.rs:113): alpha (red)
 * and beta (blue) per window, x = 0..300, y = 0..0.01, 95 % bands from ci_*_lo / ci_*_hi (any of the four may be NULL) */
int abfit_plot_metaplot(const char *path, int32_t n_windows, const double *alpha, const double *beta,
                        const double *ci_alpha_lo, const double *ci_alpha_hi, const double *ci_beta_lo,
                        const double *ci_beta_hi);
/* bootstrap.png of every alphabeta run (src/plot.rs:84-137, called at src/boot_model.rs:105-109): box plots of the
 * n bootstrap alphas and betas (columns 0 and 1 of the bootstrap rows), y = 0 .. 1.3 max */
int abfit_plot_bootstrap(const char *path, const double *alphas, const double *betas, int32_t n);

#ifdef __cplusplus
}
#endif
#endif
