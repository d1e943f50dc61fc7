/*
 * abref.c — CPU ORACLE (test infrastructure only; see abref.h for the contract
 * and the list of golden vectors that pin it).  Each function cites the
 * reference lines it restates (paths relative to the alphabeta-rs repo root).
 *
 * Build: gcc -O2 -std=c11 -ffp-contract=off -fPIC -shared -pthread abref.c -lm
 */
#define _GNU_SOURCE
#include "abref.h"

#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

/* ------------------------------------------------------------------------- */
/* 3x3 products.  ndarray 0.15.6 sends mat*mat with every dim <= 7 to          */
/* matrixmultiply 0.3.2, whose x86-64 dgemm micro-kernel accumulates           */
/*   c[i][j] = fma(a[i][k], b[k][j], c[i][j])   for k = 0,1,2                  */
/* (FMA variant selected at run time).  That pattern is the only one that      */
/* reproduces src/structs.rs:233 bit for bit; a non-fused product is 4 ulp off.*/
/* ------------------------------------------------------------------------- */

static inline double fma_chain3(double a0, double b0, double a1, double b1, double a2, double b2)
{
    double acc = a0 * b0;
    acc = __builtin_fma(a1, b1, acc);
    acc = __builtin_fma(a2, b2, acc);
    return acc;
}

#define MAT3_BODY                                                                              \
    double r[9];                                                                               \
    for (int i = 0; i < 3; ++i)                                                                \
        for (int j = 0; j < 3; ++j)                                                            \
            r[3 * i + j] = fma_chain3(A[3 * i], B[j], A[3 * i + 1], B[3 + j], A[3 * i + 2], B[6 + j]); \
    memcpy(out, r, sizeof r);

static void mat3_mul_generic(const double A[9], const double B[9], double out[9]) { MAT3_BODY }

#if defined(__x86_64__)
__attribute__((target("fma"))) static void mat3_mul_hwfma(const double A[9], const double B[9],
                                                          double out[9])
{
    MAT3_BODY
}
#endif

typedef void (*mat3_fn)(const double *, const double *, double *);
static mat3_fn mat3_mul_ptr = 0;

static mat3_fn pick_mat3(void)
{
#if defined(__x86_64__)
    __builtin_cpu_init();
    if (__builtin_cpu_supports("fma")) return mat3_mul_hwfma;
#endif
    return mat3_mul_generic;
}

static inline void mat3_mul(const double A[9], const double B[9], double out[9])
{
    if (!mat3_mul_ptr) mat3_mul_ptr = pick_mat3();
    mat3_mul_ptr(A, B, out);
}

/* 1x3 . 3x3 (src/divergence.rs:55).  Same FMA chain, chosen for uniformity; the
 * mode does not influence any golden vector (t0 == 0 multiplies by the identity). */
static inline void vec3_mat3(const double v[3], const double M[9], double out[3])
{
    for (int j = 0; j < 3; ++j) out[j] = fma_chain3(v[0], M[j], v[1], M[3 + j], v[2], M[6 + j]);
}

/* src/divergence.rs:96-114 — powi(2) is x*x */
void abref_genmatrix(double alpha, double beta, double G[9])
{
    double oma = 1.0 - alpha, omb = 1.0 - beta;
    double b1a = beta + 1.0 - alpha; /* (beta + 1.0) - alpha */
    double a1b = alpha + 1.0 - beta;
    G[0] = oma * oma;
    G[1] = 2.0 * oma * alpha;
    G[2] = alpha * alpha;
    G[3] = 0.25 * (b1a * b1a);
    G[4] = 0.5 * b1a * a1b;
    G[5] = 0.25 * (a1b * a1b);
    G[6] = beta * beta;
    G[7] = 2.0 * omb * beta;
    G[8] = omb * omb;
}

/* src/divergence.rs:16-31 — power 0 = identity, else R = M; (power-1) x R = R.M */
void abref_matrix_power(const double M[9], int power, double out[9])
{
    if (power == 0) {
        static const double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
        memcpy(out, I, sizeof I);
        return;
    }
    double R[9];
    memcpy(R, M, sizeof R);
    for (int k = 1; k < power; ++k) mat3_mul(R, M, R);
    memcpy(out, R, sizeof R);
}

/* src/alphabeta.rs:62-65 == src/structs.rs:156-159 */
double abref_p_uu_est(double a, double b)
{
    double omb = 1.0 - b, oma = 1.0 - a, s = a + b, sm1 = s - 1.0;
    return (b * (omb * omb - oma * oma - 1.0)) / (s * (sm1 * sm1 - 2.0));
}
/* src/alphabeta.rs:68-71 == src/structs.rs:146-149 */
double abref_p_mm_est(double a, double b)
{
    double omb = 1.0 - b, oma = 1.0 - a, s = a + b, sm1 = s - 1.0;
    return (a * (oma * oma - omb * omb - 1.0)) / (s * (sm1 * sm1 - 2.0));
}
/* src/structs.rs:151-154 */
double abref_p_um_est(double a, double b)
{
    double s = a + b, sm1 = s - 1.0;
    return (4.0 * a * b * (s - 2.0)) / (s * (sm1 * sm1 - 2.0));
}
/* src/alphabeta.rs:74-79 */
double abref_steady_state(double a, double b)
{
    double pi_2 = abref_p_um_est(a, b);
    return abref_p_mm_est(a, b) + 0.5 * pi_2;
}

/* `x as i8` for f64 in Rust: saturating, NaN -> 0 (src/divergence.rs:52) */
static inline int as_i8(double x)
{
    if (x != x) return 0;
    if (x >= 127.0) return 127;
    if (x <= -128.0) return -128;
    return (int)x; /* truncation toward zero */
}

/* src/divergence.rs:68-87: one conditional divergence from row k of A and B */
static inline double cond_div(const double *a, const double *b)
{
    return 0.5 * (a[0] * b[1] + a[1] * b[0] + a[1] * b[2] + a[2] * b[1]) + (a[0] * b[2] + a[2] * b[0]);
}

/* src/divergence.rs:33-94 */
int abref_divergence(const double *ped, int n, double p_mm, double p_um, double p_uu, double alpha,
                     double beta, double weight, int flags, double *dt1t2, double *p_uu_out)
{
    (void)p_um;
    double sv0[3] = {p_uu, weight * p_mm, (1.0 - weight) * p_mm};
    double G[9];
    abref_genmatrix(alpha, beta, G);

    double table[128][9];
    int have = -1;
    if (flags & ABREF_FAST_DIVERGENCE) {
        /* same left-associated chain as matrix_power, shared between pairs */
        int tmax = 0;
        for (int i = 0; i < n; ++i) {
            int t0 = as_i8(ped[4 * i]), t1 = as_i8(ped[4 * i + 1]), t2 = as_i8(ped[4 * i + 2]);
            if (t0 < 0 || t1 < t0 || t2 < t0) return ABREF_ERR_TIME;
            if (t0 > tmax) tmax = t0;
            if (t1 - t0 > tmax) tmax = t1 - t0;
            if (t2 - t0 > tmax) tmax = t2 - t0;
        }
        abref_matrix_power(G, 0, table[0]);
        if (tmax >= 1) memcpy(table[1], G, sizeof G);
        for (int k = 2; k <= tmax; ++k) mat3_mul(table[k - 1], G, table[k]);
        have = tmax;
    }

    for (int i = 0; i < n; ++i) {
        int t0 = as_i8(ped[4 * i]), t1 = as_i8(ped[4 * i + 1]), t2 = as_i8(ped[4 * i + 2]);
        if (t0 < 0 || t1 < t0 || t2 < t0) return ABREF_ERR_TIME;
        double P0[9], A[9], B[9];
        const double *p0 = P0, *a = A, *b = B;
        if (have >= 0) {
            p0 = table[t0];
            a = table[t1 - t0];
            b = table[t2 - t0];
        } else {
            abref_matrix_power(G, t0, P0);
            abref_matrix_power(G, t1 - t0, A);
            abref_matrix_power(G, t2 - t0, B);
        }
        double s[3];
        vec3_mat3(sv0, p0, s);
        double d_mm = cond_div(a + 6, b + 6);
        double d_um = cond_div(a + 3, b + 3);
        double d_uu = cond_div(a, b);
        dt1t2[i] = s[0] * d_uu + s[1] * d_um + s[2] * d_mm;
    }
    if (p_uu_out) *p_uu_out = abref_p_uu_est(alpha, beta);
    return 0;
}

#define STACK_N 4096

/* src/structs.rs:191-217 — the penalty term sits inside the per-pair loop */
double abref_cost(const abref_problem *pb, const double th[4], int flags)
{
    int n = pb->n;
    double stackbuf[STACK_N];
    double *dt = n <= STACK_N ? stackbuf : (double *)malloc(sizeof(double) * (size_t)n);
    double puu;
    if (abref_divergence(pb->ped, n, pb->p_mm, pb->p_um, pb->p_uu, th[0], th[1], th[2], flags, dt, &puu)) {
        if (dt != stackbuf) free(dt);
        return NAN;
    }
    double sq = 0.0;
    for (int i = 0; i < n; ++i) {
        double r = pb->ped[4 * i + 3] - th[3] - dt[i];
        double dq = puu - pb->eqp;
        sq += r * r + pb->eqp_weight * (double)n * (dq * dq);
    }
    if (dt != stackbuf) free(dt);
    return sq;
}

/* src/ab_neutral.rs:88-93 */
double abref_lse(const abref_problem *pb, const double th[4], int flags)
{
    int n = pb->n;
    double stackbuf[STACK_N];
    double *dt = n <= STACK_N ? stackbuf : (double *)malloc(sizeof(double) * (size_t)n);
    if (abref_divergence(pb->ped, n, pb->p_mm, pb->p_um, pb->p_uu, th[0], th[1], th[2], flags, dt, 0)) {
        if (dt != stackbuf) free(dt);
        return NAN;
    }
    double s = 0.0;
    for (int i = 0; i < n; ++i) {
        double r = pb->ped[4 * i + 3] - th[3] - dt[i];
        s += r * r;
    }
    if (dt != stackbuf) free(dt);
    return s;
}

/* ------------------------------------------------------------------------- */
/* Nelder-Mead as in argmin 0.8.1 `solver::neldermead::NelderMead` driven by   */
/* `core::Executor` (third-party, pinned in Cargo.lock, source not vendored;   */
/* restated from the published 0.8.1 algorithm):                               */
/*   new(): alpha=1, gamma=2, rho=0.5, sigma=0.5, sd_tolerance=EPSILON         */
/*   init(): cost of the 5 vertices in the given order, stable sort ascending  */
/*           (partial_cmp, incomparable -> Equal)                              */
/*   Executor loop, top of every iteration: solver.terminate() [sample sd of   */
/*           the costs < sd_tolerance], then iter >= max_iters, then           */
/*           best_cost <= target_cost(-inf)                                    */
/*   next_iter(): x0 = (x0+x1+x2+x3) * (1/4); xr = x0 + (x0 - x4)*1;           */
/*       fr <  c[3] && fr >= c[0] : worst <- xr                                */
/*       fr <  c[0]               : xe = x0 + (xr - x0)*2; worst <- fe<fr?xe:xr*/
/*       fr >= c[3]               : xc = x0 + (x4 - x0)*0.5;                   */
/*                                  worst <- xc only if fc < c[4]; ELSE NOTHING*/
/*       otherwise (NaN fr)       : shrink all towards x[0] by 0.5             */
/*     stable re-sort; state.param = x[0], state.cost = c[0]                   */
/*   IterState::update(): best_param <- param iff cost < best_cost (or both    */
/*           infinite with the same sign)                                      */
/* A failed inside contraction leaves the simplex untouched, and next_iter is  */
/* a pure function of the simplex, so every later iteration repeats it until   */
/* max_iters: ABREF_NM_EARLY_EXIT_ON_STALL returns at that point with the      */
/* identical best_param/best_cost and iters = max_iters.                       */
/* ------------------------------------------------------------------------- */

typedef struct {
    double x[4];
    double c;
} vertex;

static void sort_vertices(vertex *v, int n)
{
    /* stable insertion sort; is_less(a,b) := partial_cmp(a,b) == Less */
    for (int i = 1; i < n; ++i) {
        vertex t = v[i];
        int j = i;
        while (j > 0 && t.c < v[j - 1].c) {
            v[j] = v[j - 1];
            --j;
        }
        v[j] = t;
    }
}

int abref_nelder_mead(const abref_problem *pb, const double simplex[20], int max_iters, double sd_tol,
                      int flags, abref_fit *out)
{
    vertex v[5];
    int evals = 0, iters = 0, status = ABREF_TERM_MAX_ITERS;
    for (int k = 0; k < 5; ++k) {
        memcpy(v[k].x, simplex + 4 * k, sizeof v[k].x);
        v[k].c = abref_cost(pb, v[k].x, flags);
        ++evals;
    }
    sort_vertices(v, 5);

    double best_cost = INFINITY, best[4] = {NAN, NAN, NAN, NAN};
    int have_best = 0;
#define UPDATE_BEST()                                                                    \
    do {                                                                                 \
        double c_ = v[0].c;                                                              \
        if (c_ < best_cost || (isinf(c_) && isinf(best_cost) && (c_ > 0) == (best_cost > 0))) { \
            memcpy(best, v[0].x, sizeof best);                                           \
            best_cost = c_;                                                              \
            have_best = 1;                                                               \
        }                                                                                \
    } while (0)
    UPDATE_BEST();

    for (;;) {
        /* NelderMead::terminate */
        double sum = 0.0;
        for (int k = 0; k < 5; ++k) sum += v[k].c;
        double c0 = sum / 5.0;
        double ss = 0.0;
        for (int k = 0; k < 5; ++k) {
            double d = v[k].c - c0;
            ss += d * d;
        }
        double s = sqrt(1.0 / (5.0 - 1.0) * ss);
        if (s < sd_tol) {
            status = ABREF_TERM_SD;
            break;
        }
        if (iters >= max_iters) {
            status = ABREF_TERM_MAX_ITERS;
            break;
        }
        if (best_cost <= -INFINITY) {
            status = ABREF_TERM_TARGET_COST;
            break;
        }

        /* next_iter */
        double x0[4], xr[4];
        for (int j = 0; j < 4; ++j) {
            double a = v[0].x[j];
            a = a + v[1].x[j];
            a = a + v[2].x[j];
            a = a + v[3].x[j];
            x0[j] = a * (1.0 / 4.0);
        }
        for (int j = 0; j < 4; ++j) xr[j] = x0[j] + (x0[j] - v[4].x[j]) * 1.0;
        double fr = abref_cost(pb, xr, flags);
        ++evals;
        int stalled = 0;
        if (fr < v[3].c && fr >= v[0].c) {
            memcpy(v[4].x, xr, sizeof xr);
            v[4].c = fr;
        } else if (fr < v[0].c) {
            double xe[4];
            for (int j = 0; j < 4; ++j) xe[j] = x0[j] + (xr[j] - x0[j]) * 2.0;
            double fe = abref_cost(pb, xe, flags);
            ++evals;
            if (fe < fr) {
                memcpy(v[4].x, xe, sizeof xe);
                v[4].c = fe;
            } else {
                memcpy(v[4].x, xr, sizeof xr);
                v[4].c = fr;
            }
        } else if (fr >= v[3].c) {
            double xc[4];
            for (int j = 0; j < 4; ++j) xc[j] = x0[j] + (v[4].x[j] - x0[j]) * 0.5;
            double fc = abref_cost(pb, xc, flags);
            ++evals;
            if (fc < v[4].c) {
                memcpy(v[4].x, xc, sizeof xc);
                v[4].c = fc;
            } else if (flags & ABREF_NM_SHRINK_ON_FAILED_CONTRACTION) {
                goto shrink;
            } else {
                stalled = 1;
            }
        } else {
        shrink:
            for (int k = 1; k < 5; ++k) {
                for (int j = 0; j < 4; ++j) v[k].x[j] = v[0].x[j] + (v[k].x[j] - v[0].x[j]) * 0.5;
                v[k].c = abref_cost(pb, v[k].x, flags);
                ++evals;
            }
        }
        sort_vertices(v, 5);
        UPDATE_BEST();
        ++iters;
        if (stalled && (flags & ABREF_NM_EARLY_EXIT_ON_STALL)) {
            /* the sd test above did not fire for this simplex and never will */
            status = ABREF_TERM_STALLED;
            iters = max_iters;
            break;
        }
    }
#undef UPDATE_BEST
    if (!have_best) {
        /* best_param stays None and the reference panics.  v[0] is the start's vertex 0 (its NaN cost never moves
         * in the stable sort): report it with its NaN cost, as the library's records do (include/abfit.h) */
        memcpy(best, v[0].x, sizeof best);
        best_cost = v[0].c;
    }
    memcpy(out->theta, best, sizeof best);
    out->cost = best_cost;
    out->iters = iters;
    out->evals = evals;
    out->lse = NAN;
    out->start_id = -1;
    out->status = have_best ? status : ABREF_ERR_NAN;
    return out->status;
}

/* ------------------------------------------------------------------------- */
/* thread pool helper (rayon into_par_iter().for_each analogue:                */
/* src/ab_neutral.rs:37, src/boot_model.rs:41)                                 */
/* ------------------------------------------------------------------------- */
typedef void (*task_fn)(void *ctx, int idx);
typedef struct {
    task_fn fn;
    void *ctx;
    int n;
    int next;
    pthread_mutex_t mu;
} pool_job;

static void *pool_worker(void *arg)
{
    pool_job *job = (pool_job *)arg;
    for (;;) {
        pthread_mutex_lock(&job->mu);
        int i = job->next++;
        pthread_mutex_unlock(&job->mu);
        if (i >= job->n) break;
        job->fn(job->ctx, i);
    }
    return 0;
}

static void parallel_for(int n, int n_threads, task_fn fn, void *ctx)
{
    if (n_threads <= 1 || n <= 1) {
        for (int i = 0; i < n; ++i) fn(ctx, i);
        return;
    }
    if (n_threads > 256) n_threads = 256;
    pool_job job = {fn, ctx, n, 0, PTHREAD_MUTEX_INITIALIZER};
    pthread_t th[256];
    int started = 0;
    for (int t = 0; t < n_threads; ++t)
        if (pthread_create(&th[started], 0, pool_worker, &job) == 0) ++started;
    if (!started) pool_worker(&job);
    for (int t = 0; t < started; ++t) pthread_join(th[t], 0);
}

int abref_hw_threads(void)
{
    long n = sysconf(_SC_NPROCESSORS_ONLN);
    return n > 0 ? (int)n : 1;
}

/* ------------------------------------------------------------------------- */
/* src/ab_neutral.rs:13-142                                                    */
/* ------------------------------------------------------------------------- */
typedef struct {
    const abref_problem *pb;
    const double *simplices;
    int max_iters;
    double sd_tol;
    int flags;
    abref_fit *fits;
} start_ctx;

static void start_task(void *c, int i)
{
    start_ctx *s = (start_ctx *)c;
    /* src/ab_neutral.rs:40-47: every start owns a clone of the pedigree */
    abref_problem local = *s->pb;
    double *copy = 0;
    if (!(s->flags & ABREF_FAST_DIVERGENCE)) {
        copy = (double *)malloc(sizeof(double) * 4 * (size_t)local.n);
        memcpy(copy, s->pb->ped, sizeof(double) * 4 * (size_t)local.n);
        local.ped = copy;
    }
    abref_nelder_mead(&local, s->simplices + 20 * (size_t)i, s->max_iters, s->sd_tol, s->flags, &s->fits[i]);
    s->fits[i].start_id = i;
    free(copy);
}

/* src/ab_neutral.rs:83-101, literally: `results.sort_by(|a, b| { let pedigree = pedigree.clone();
 * divergence(a); divergence(b); lse_a.partial_cmp(&lse_b).unwrap() })` — slice::sort_by is a stable
 * merge sort (insertion sort on short runs); ~ n log2 n comparisons, two objective evaluations each.
 * The comparison count of this top-down merge sort (runs of <= 20 by insertion) is within a few
 * per cent of Rust's; the ORDER it produces is the same (any stable sort gives one order). */
typedef struct {
    const abref_problem *pb;
    abref_fit *fits;
    int flags;
    int nan;
    long n_cmp;
} literal_sort_ctx;

static int literal_less(literal_sort_ctx *c, int a, int b)
{
    /* let pedigree = pedigree.clone(); */
    abref_problem local = *c->pb;
    size_t bytes = sizeof(double) * 4 * (size_t)local.n;
    double *copy = (double *)malloc(bytes);
    memcpy(copy, c->pb->ped, bytes);
    local.ped = copy;
    double la = abref_lse(&local, c->fits[a].theta, c->flags);
    double lb = abref_lse(&local, c->fits[b].theta, c->flags);
    free(copy);
    ++c->n_cmp;
    if (la != la || lb != lb) c->nan = 1; /* partial_cmp().unwrap() panics */
    return la < lb;
}

static void literal_merge_sort(literal_sort_ctx *c, int *v, int *tmp, int lo, int hi)
{
    if (hi - lo <= 20) {
        for (int i = lo + 1; i < hi; ++i) {
            int x = v[i], j = i;
            while (j > lo && literal_less(c, x, v[j - 1])) {
                v[j] = v[j - 1];
                --j;
            }
            v[j] = x;
        }
        return;
    }
    int mid = lo + (hi - lo) / 2;
    literal_merge_sort(c, v, tmp, lo, mid);
    literal_merge_sort(c, v, tmp, mid, hi);
    int i = lo, j = mid, k = lo;
    while (i < mid && j < hi) tmp[k++] = literal_less(c, v[j], v[i]) ? v[j++] : v[i++]; /* stable */
    while (i < mid) tmp[k++] = v[i++];
    while (j < hi) tmp[k++] = v[j++];
    memcpy(v + lo, tmp + lo, sizeof(int) * (size_t)(hi - lo));
}

int abref_ab_neutral(const abref_problem *pb, int n_starts, const double *simplices, int max_iters,
                     double sd_tol, int flags, int n_threads, abref_fit *best, abref_fit *all_out,
                     double *pred, double *resid)
{
    int n = pb->n;
    /* :25-29 max_by(partial_cmp().unwrap()) panics on NaN */
    for (int i = 0; i < n; ++i)
        if (pb->ped[4 * i + 3] != pb->ped[4 * i + 3]) return ABREF_ERR_NAN;
    /* :31 */
    if (pb->p_mm + pb->p_uu + pb->p_um != 1.0) return ABREF_ERR_NAN;

    abref_fit *fits = all_out ? all_out : (abref_fit *)malloc(sizeof(abref_fit) * (size_t)n_starts);
    start_ctx ctx = {pb, simplices, max_iters, sd_tol, flags, fits};
    parallel_for(n_starts, n_threads, start_task, &ctx);

    /* :83-101 stable sort by penalty-free LSE, first element wins; the reference
     * re-evaluates divergence() inside the comparator, the value is the same.
     * Result order in the reference is completion order; here: start id. */
    int rc = 0, arg = -1, literal_first = -1;
    if (flags & ABREF_LITERAL_SORT) {
        /* the reference's own work: a stable merge sort whose comparator clones the pedigree and
         * evaluates divergence() + the LSE sum for BOTH operands of every comparison (serial). */
        for (int i = 0; i < n_starts; ++i)
            if (fits[i].status < 0) rc = ABREF_ERR_NAN;
        if (rc == 0) {
            int *ord = (int *)malloc(sizeof(int) * (size_t)n_starts);
            int *tmp = (int *)malloc(sizeof(int) * (size_t)n_starts);
            for (int i = 0; i < n_starts; ++i) ord[i] = i;
            literal_sort_ctx lc = {pb, fits, flags, 0, 0};
            literal_merge_sort(&lc, ord, tmp, 0, n_starts);
            if (lc.nan) rc = ABREF_ERR_NAN;
            literal_first = ord[0];
            free(ord);
            free(tmp);
        }
    }
    for (int i = 0; i < n_starts; ++i) {
        fits[i].lse = abref_lse(pb, fits[i].theta, flags);
        if (fits[i].status < 0) {
            rc = ABREF_ERR_NAN; /* :64,66 expect()/unwrap() panic */
            continue;
        }
        if (fits[i].lse != fits[i].lse) rc = ABREF_ERR_NAN; /* :100 unwrap panic */
        if (arg < 0 || fits[i].lse < fits[arg].lse) arg = i;
    }
    if (rc == 0 && literal_first >= 0 && literal_first != arg) return ABREF_ERR_TIME - 100; /* cannot happen: both are the stable minimum */
    if (rc == 0 && arg >= 0) {
        *best = fits[arg];
        /* :108-135 */
        double *dt = (double *)malloc(sizeof(double) * (size_t)n);
        abref_divergence(pb->ped, n, pb->p_mm, pb->p_um, pb->p_uu, best->theta[0], best->theta[1],
                         best->theta[2], flags, dt, 0);
        for (int i = 0; i < n; ++i) {
            double p = best->theta[3] + dt[i];
            if (pred) pred[i] = p;
            if (resid) resid[i] = pb->ped[4 * i + 3] - p;
        }
        free(dt);
    } else if (rc == 0) {
        rc = ABREF_ERR_NAN;
    }
    if (!all_out) free(fits);
    return rc;
}

/* ------------------------------------------------------------------------- */
/* src/boot_model.rs:17-115                                                    */
/* ------------------------------------------------------------------------- */
typedef struct {
    const abref_problem *pb;
    const double *best_theta, *pred, *resid;
    const int32_t *idx;
    const double *vary;
    int max_iters;
    double sd_tol;
    int flags;
    double *rows;
    abref_fit *fits;
} boot_ctx;

static void boot_task(void *c, int b)
{
    boot_ctx *s = (boot_ctx *)c;
    int n = s->pb->n;
    /* :50-57 pedigree clone with column 3 <- pred + resampled residual */
    double *ped = (double *)malloc(sizeof(double) * 4 * (size_t)n);
    memcpy(ped, s->pb->ped, sizeof(double) * 4 * (size_t)n);
    for (int i = 0; i < n; ++i) ped[4 * i + 3] = s->pred[i] + s->resid[s->idx[(size_t)b * n + i]];
    abref_problem local = *s->pb;
    local.ped = ped;
    /* :69-75 */
    double simplex[20];
    memcpy(simplex, s->best_theta, sizeof(double) * 4);
    memcpy(simplex + 4, s->vary + 16 * (size_t)b, sizeof(double) * 16);
    abref_fit f;
    abref_nelder_mead(&local, simplex, s->max_iters, s->sd_tol, s->flags, &f);
    f.start_id = b;
    /* :86-96 */
    double *r = s->rows + 7 * (size_t)b;
    r[0] = f.theta[0];
    r[1] = f.theta[1];
    r[2] = f.theta[2];
    r[3] = f.theta[3];
    r[4] = abref_p_mm_est(f.theta[0], f.theta[1]);
    r[5] = abref_p_um_est(f.theta[0], f.theta[1]);
    r[6] = abref_p_uu_est(f.theta[0], f.theta[1]);
    if (s->fits) s->fits[b] = f;
    free(ped);
}

int abref_boot_model(const abref_problem *pb, const double best_theta[4], const double *pred,
                     const double *resid, int n_boot, const int32_t *resample_idx,
                     const double *vary_vertices, int max_iters, double sd_tol, int flags,
                     int n_threads, double *rows_out, abref_fit *fits_out)
{
    if (pb->p_mm + pb->p_uu + pb->p_um != 1.0) return ABREF_ERR_NAN; /* :35 */
    boot_ctx ctx = {pb, best_theta, pred, resid, resample_idx, vary_vertices, max_iters, sd_tol, flags,
                    rows_out, fits_out};
    parallel_for(n_boot, n_threads, boot_task, &ctx);
    return 0;
}

/* ------------------------------------------------------------------------- */
/* src/pedigree.rs:213-262, src/methylation_site.rs:130-136                    */
/* ------------------------------------------------------------------------- */
void abref_dmatrix(const uint8_t *status, const double *post, int S, int64_t L, double thr,
                   double *D_out, uint64_t *diff_out, uint64_t *cnt_out)
{
    size_t p = 0;
    for (int i = 0; i < S; ++i)
        for (int j = i + 1; j < S; ++j, ++p) {
            uint64_t div = 0, cnt = 0;
            const uint8_t *si = status + (size_t)i * L, *sj = status + (size_t)j * L;
            const double *pi = post + (size_t)i * L, *pj = post + (size_t)j * L;
            for (int64_t k = 0; k < L; ++k) {
                /* src/pedigree.rs:249-251 keeps a site when post_i >= thr && post_j >= thr: a NaN posterior (or
                 * thr = NaN) fails the test, as in abref_p0uu */
                if (!(pi[k] >= thr && pj[k] >= thr)) continue;
                int a = si[k], b = sj[k];
                div += (uint64_t)(a > b ? a - b : b - a);
                cnt += 1;
            }
            if (diff_out) diff_out[p] = div;
            if (cnt_out) cnt_out[p] = cnt;
            D_out[p] = (double)div / (2.0 * (double)cnt); /* 0/0 -> NaN as in the reference */
        }
}

/* src/pedigree.rs:159-183 */
double abref_p0uu(const double *post, const double *meth, int S, int64_t L, double thr, double *rc_out,
                  int64_t *nvalid_out)
{
    double acc = 0.0;
    for (int i = 0; i < S; ++i) {
        double s = 0.0;
        int64_t nv = 0;
        for (int64_t k = 0; k < L; ++k)
            if (post[(size_t)i * L + k] >= thr) {
                s += meth[(size_t)i * L + k];
                ++nv;
            }
        double rc = s / (double)nv;
        if (rc_out) rc_out[i] = rc;
        if (nvalid_out) nvalid_out[i] = nv;
        acc += 1.0 - rc;
    }
    return acc / (double)S;
}

/* ------------------------------------------------------------------------- */
/* src/analysis.rs:50-98.  Third-party pieces restated as published:           */
/*  ndarray 0.15.6 `mean` = sum/n where `sum` of a strided column view is a    */
/*  sequential fold and `sum` of an owned contiguous array (beta/alpha) is the */
/*  8-lane unrolled fold; `std(1.0)` = sqrt of Welford variance with           */
/*  mul_add; ndarray-stats 0.5.1 `quantiles_mut(.., &Linear)`: index q*(n-1),  */
/*  lower + (higher-lower)*fract.  ("parity unpinned": no reference test)      */
/* ------------------------------------------------------------------------- */
static double seq_sum(const double *x, int n, int stride)
{
    double s = 0.0;
    for (int i = 0; i < n; ++i) s += x[(size_t)i * stride];
    return s;
}
static double unrolled_sum(const double *x, int n)
{
    double p[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int i = 0;
    for (; n - i >= 8; i += 8)
        for (int k = 0; k < 8; ++k) p[k] += x[i + k];
    double acc = 0.0;
    acc += p[0] + p[4];
    acc += p[1] + p[5];
    acc += p[2] + p[6];
    acc += p[3] + p[7];
    for (; i < n; ++i) acc += x[i];
    return acc;
}
static double welford_std(const double *x, int n, int stride, double ddof)
{
    double mean = 0.0, sum_sq = 0.0;
    for (int i = 0; i < n; ++i) {
        double v = x[(size_t)i * stride];
        double count = (double)(i + 1);
        double delta = v - mean;
        mean = mean + delta / count;
        sum_sq = fma(v - mean, delta, sum_sq);
    }
    return sqrt(sum_sq / ((double)n - ddof));
}
static int cmp_double(const void *a, const void *b)
{
    double x = *(const double *)a, y = *(const double *)b;
    return (x > y) - (x < y);
}
static void quantile_pair(const double *x, int n, int stride, double out[2])
{
    double *tmp = (double *)malloc(sizeof(double) * (size_t)n);
    for (int i = 0; i < n; ++i) tmp[i] = x[(size_t)i * stride];
    qsort(tmp, (size_t)n, sizeof(double), cmp_double);
    const double qs[2] = {0.025, 0.975};
    for (int k = 0; k < 2; ++k) {
        double pos = (double)(n - 1) * qs[k];
        double lo = floor(pos), hi = ceil(pos);
        double frac = pos - trunc(pos);
        double a = tmp[(int)lo], b = tmp[(int)hi];
        out[k] = a + (b - a) * frac;
    }
    free(tmp);
}

void abref_analyze(const double *rows, int n, double out[32])
{
    double *ab = (double *)malloc(sizeof(double) * (size_t)n);
    for (int i = 0; i < n; ++i) ab[i] = rows[7 * (size_t)i + 1] / rows[7 * (size_t)i];
    /* field order of Analysis: alpha, beta, alphabeta, weight, intercept, pr_mm, pr_um, pr_uu */
    const int col[8] = {0, 1, -1, 2, 3, 4, 5, 6};
    for (int f = 0; f < 8; ++f) {
        if (col[f] < 0) {
            out[f] = unrolled_sum(ab, n) / (double)n;
            out[8 + f] = welford_std(ab, n, 1, 1.0);
            quantile_pair(ab, n, 1, out + 16 + 2 * f);
        } else {
            out[f] = seq_sum(rows + col[f], n, 7) / (double)n;
            out[8 + f] = welford_std(rows + col[f], n, 7, 1.0);
            quantile_pair(rows + col[f], n, 7, out + 16 + 2 * f);
        }
    }
    free(ab);
}
