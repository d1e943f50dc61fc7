/*
 * abref — CPU ORACLE for the ABneutral hot path of alphabeta-rs.
 *
 * THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, the smoke check
 * in __graft_entry__.py and bench.py's cpu_baseline / --impl reference legs may
 * load this library.  Nothing under alphabeta-rs_b200/ links, imports or calls it.
 *
 * It is a plain-C restatement, function by function, of the Rust reference
 * (crate `alphabeta` v0.2.1).  The reference cannot be compiled in this image
 * (no cargo/rustc), so there is no oracle/_ref build; instead this restatement
 * is pinned against every golden vector the reference ships for the path
 * (tests/test_oracle_golden.py):
 *   - src/structs.rs:233      cost KAT 0.0006700888539608879  (bit-exact)
 *   - data/divergence.txt     351 dt1t2 values of src/divergence.rs:139-161
 *   - data/pedigree_generated.txt  6 rows of src/pedigree.rs:345-358 (bit-exact)
 *   - data/desired_output/    R-original pedigree (5 decimals) and fit (10 %)
 * Parity status of the optimiser: the Nelder-Mead iteration itself lives in the
 * third-party crate argmin 0.8.1 (+ argmin-math 0.3.0), whose source is NOT in
 * /root/reference and which none of the reference's enabled tests exercise:
 * "parity unpinned" for the NM trajectory (restated from the published 0.8.1
 * algorithm, see abref_nelder_mead).
 *
 * Arithmetic contract ("ref-order"): every 3x3 inner product is an FMA chain
 * over k ascending (what matrixmultiply 0.3.2's FMA micro-kernel does and the
 * only pattern that reproduces the cost KAT); every other operation is a plain
 * IEEE-754 binary64 mul/add/sub/div/sqrt in source order.  Compile with
 * -ffp-contract=off.
 */
#ifndef ABREF_H
#define ABREF_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* src/structs.rs:12-19 `Problem` (pedigree rows are [t0,t1,t2,D], row-major) */
typedef struct {
    const double *ped; /* [n][4] */
    int32_t n;
    double p_mm, p_um, p_uu; /* state probabilities at G0 */
    double eqp, eqp_weight;
} abref_problem;

enum {
    ABREF_NM_SHRINK_ON_FAILED_CONTRACTION = 1, /* later-argmin semantics; default off = 0.8.1 */
    ABREF_NM_EARLY_EXIT_ON_STALL = 2,          /* result-identical short-cut, see abref_nelder_mead */
    ABREF_FAST_DIVERGENCE = 4,                 /* power table + same chain: bit-identical, less work */
    ABREF_LITERAL_SORT = 8                     /* best-of-starts by the reference's own sort_by whose comparator
                                                  re-evaluates divergence() twice per comparison (src/ab_neutral.rs:83-101);
                                                  same winner, the reference's serial tail is paid */
};

enum {
    ABREF_OK = 0,
    ABREF_TERM_SD = 1,        /* sd of simplex costs < sd_tolerance */
    ABREF_TERM_MAX_ITERS = 2, /* iter >= max_iters */
    ABREF_TERM_STALLED = 3,   /* ABREF_NM_EARLY_EXIT_ON_STALL fired; iters reported = max_iters */
    ABREF_TERM_TARGET_COST = 4, /* best_cost <= target_cost (-inf) */
    ABREF_ERR_NAN = -1,       /* reference would panic (NaN cost / best_param None) */
    ABREF_ERR_TIME = -2       /* t0>t1 or t0>t2 or outside i8: reference takes the matrix-inverse path */
};

typedef struct {
    double theta[4]; /* alpha, beta, weight, intercept = state.best_param */
    double cost;     /* state.best_cost */
    double lse;      /* penalty-free least squares of theta (src/ab_neutral.rs:88-93) */
    int32_t iters, evals, status, start_id;
} abref_fit;

/* src/divergence.rs:96-114 */
void abref_genmatrix(double alpha, double beta, double G[9]);
/* src/divergence.rs:16-31 (power >= 0 only) */
void abref_matrix_power(const double M[9], int power, double out[9]);
/* src/alphabeta.rs:62-79, src/structs.rs:146-158 */
double abref_p_uu_est(double alpha, double beta);
double abref_p_mm_est(double alpha, double beta);
double abref_p_um_est(double alpha, double beta);
double abref_steady_state(double alpha, double beta);
/* src/divergence.rs:33-94; returns 0 or ABREF_ERR_TIME */
int abref_divergence(const double *ped, int n, double p_mm, double p_um, double p_uu, double alpha,
                     double beta, double weight, int flags, double *dt1t2, double *p_uu_out);
/* src/structs.rs:191-217 */
double abref_cost(const abref_problem *pb, const double theta[4], int flags);
/* src/ab_neutral.rs:88-93 */
double abref_lse(const abref_problem *pb, const double theta[4], int flags);
/* argmin 0.8.1 NelderMead + Executor, call sites src/ab_neutral.rs:49-64, src/boot_model.rs:69-84 */
int abref_nelder_mead(const abref_problem *pb, const double simplex[20], int max_iters, double sd_tol,
                      int flags, abref_fit *out);
/* src/ab_neutral.rs:13-142 with the start simplices passed in ([n_starts][5][4]).
 * all_out may be NULL, else [n_starts]. pred/resid are [n]. n_threads<=1: serial. */
int abref_ab_neutral(const abref_problem *pb, int n_starts, const double *simplices, int max_iters,
                     double sd_tol, int flags, int n_threads, abref_fit *best, abref_fit *all_out,
                     double *pred, double *resid);
/* src/boot_model.rs:17-115 with resample indices [n_boot][n] and vary vertices [n_boot][4][4]
 * passed in; rows_out [n_boot][7], fits_out optional [n_boot]. */
int abref_boot_model(const abref_problem *pb, const double best_theta[4], const double *pred,
                     const double *resid, int n_boot, const int32_t *resample_idx,
                     const double *vary_vertices, int max_iters, double sd_tol, int flags,
                     int n_threads, double *rows_out, abref_fit *fits_out);
/* src/pedigree.rs:213-262: status [S][L] (0=U,1=I,2=M), posterior_max [S][L];
 * pair order (0,1),(0,2)..(S-2,S-1); D_out/diff_out/cnt_out are [S(S-1)/2]. */
void abref_dmatrix(const uint8_t *status, const double *posterior_max, int S, int64_t L, double thr,
                   double *D_out, uint64_t *diff_out, uint64_t *cnt_out);
/* src/pedigree.rs:159-183: per-sample rc = sum_valid(meth_lvl)/n_valid; p0uu = mean(1-rc). */
double abref_p0uu(const double *posterior_max, const double *meth_lvl, int S, int64_t L, double thr,
                  double *rc_out, int64_t *nvalid_out);
/* src/analysis.rs:50-98: rows [n][7] -> out[32]: 8 means, 8 sds, 8 (lo,hi) pairs in the
 * field order of `Analysis` (alpha,beta,alphabeta,weight,intercept,pr_mm,pr_um,pr_uu). */
void abref_analyze(const double *rows, int n, double out[32]);

int abref_hw_threads(void);

#ifdef __cplusplus
}
#endif
#endif
