// abfit_nm.cuh — Nelder-Mead (argmin 0.8.1 semantics) as a per-lane state machine.
#pragma once
#include "abfit_model.cuh"

namespace abfit {

// ---------------------------------------------------------------------------------
// Nelder-Mead, argmin 0.8.1 semantics (call sites src/ab_neutral.rs:49-64 and
// src/boot_model.rs:69-84), as a per-lane state machine: every trip of the warp loop
// evaluates exactly one trial point per active lane, so lanes in different NM phases
// (reflect / expand / contract / ...) still share the objective's instruction stream.
// ---------------------------------------------------------------------------------
enum Phase : int {
    PH_IDLE = 0,  // needs a new fit
    PH_INIT,      // evaluating initial vertex k
    PH_REFLECT,
    PH_EXPAND,
    PH_CONTRACT,
    PH_SHRINK,  // evaluating shrunk vertex k (sorted position)
    PH_LSE      // final penalty-free evaluation of the best vertex
};

struct LaneNM {
    double xt[4];  // trial point of the current evaluation
    double fr;     // reflection cost kept across the expansion evaluation
    int phase, k;
    uint32_t ord;  // 5 x 3 bits: physical slot of the sorted vertex at position p
    int iters, evals, status;
    int fit_id;
};

// per-lane simplex storage in shared memory: X[(slot*4+j)*32 + lane], C[slot*32 + lane]
struct LaneSimplex {
    double *X;
    double *C;
    __device__ __forceinline__ double &x(int slot, int j) const { return X[(slot * 4 + j) * 32]; }
    __device__ __forceinline__ double &c(int slot) const { return C[slot * 32]; }
};

__device__ __forceinline__ int ord_at(uint32_t ord, int p) { return (ord >> (3 * p)) & 7; }

// stable insertion sort of the five vertices by cost (sort_by(partial_cmp().unwrap_or(Equal)))
// written as a fixed compare-exchange sequence; with strict '<' it performs exactly the
// swaps the insertion sort would (see DESIGN.md), NaNs included.  The sorted costs are returned in c[].
//
// FULL = false: only the vertex at sorted position 4 (the one an iteration replaces) may be out of place.  The
// first four come out of an earlier call, i.e. no adjacent pair of them satisfies c[j] < c[j-1], so the six
// compare-exchanges of insertion steps 1..3 would not swap anything: only step 4 is executed.  Same result.
template <bool FULL>
__device__ __forceinline__ uint32_t sort5(const LaneSimplex &S, uint32_t ord, double c[5])
{
    int o[5];
#pragma unroll
    for (int p = 0; p < 5; ++p) {
        o[p] = ord_at(ord, p);
        c[p] = S.c(o[p]);
    }
#pragma unroll
    for (int i = FULL ? 1 : 4; i < 5; ++i)
#pragma unroll
        for (int j = i; j >= 1; --j) {
            const bool sw = c[j] < c[j - 1];
            const double tc = sw ? c[j - 1] : c[j];
            c[j - 1] = sw ? c[j] : c[j - 1];
            c[j] = tc;
            const int to = sw ? o[j - 1] : o[j];
            o[j - 1] = sw ? o[j] : o[j - 1];
            o[j] = to;
        }
    uint32_t r = 0;
#pragma unroll
    for (int p = 0; p < 5; ++p) r |= (uint32_t)o[p] << (3 * p);
    return r;
}

// x0 = (x[0]+x[1]+x[2]+x[3]) * (1/4)   (NelderMead::calculate_centroid)
__device__ __forceinline__ void centroid(const LaneSimplex &S, uint32_t ord, double x0[4])
{
    const int a = ord_at(ord, 0), b = ord_at(ord, 1), c = ord_at(ord, 2), d = ord_at(ord, 3);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        double v = S.x(a, j);
        v = v + S.x(b, j);
        v = v + S.x(c, j);
        v = v + S.x(d, j);
        x0[j] = v * (1.0 / 4.0);
    }
}

// xr = x0 + (x0 - x[4]) * alpha, alpha = 1   (NelderMead::reflect)
__device__ __forceinline__ void reflect_point(const LaneSimplex &S, uint32_t ord, double xr[4])
{
    double x0[4];
    centroid(S, ord, x0);
    const int w = ord_at(ord, 4);
#pragma unroll
    for (int j = 0; j < 4; ++j) xr[j] = x0[j] + (x0[j] - S.x(w, j)) * 1.0;
}

// shrink point for sorted position k: x[0] + (x[k] - x[0]) * sigma, sigma = 0.5
__device__ __forceinline__ void shrink_point(const LaneSimplex &S, uint32_t ord, int k, double xs[4])
{
    const int b = ord_at(ord, 0), s = ord_at(ord, k);
#pragma unroll
    for (int j = 0; j < 4; ++j) xs[j] = S.x(b, j) + (S.x(s, j) - S.x(b, j)) * 0.5;
}

struct NMParams {
    int max_iters;
    double sd_tol;
    uint32_t flags;
    // largest y with sqrt(y) < sd_tol (host: nm_var_threshold).  IEEE sqrt is correctly rounded and
    // therefore monotonic, so  sqrt(y) < sd_tol  <=>  y <= var_thr  and the kernels never take the root.
    double var_thr;
    // Quick reject of the termination test (host: nm_range_threshold): when the spread of the sorted costs,
    // c[4] - c[0], exceeds this, 0.25 * ss > var_thr is certain — whatever the mean rounds to, one of the two
    // extreme costs is at least half the spread away from it — and the exact test (a division and ~25 dependent
    // FP64 operations per iteration) is skipped.  The decision is the same as the exact test's, always.
    double range_thr;
};

// Consume the objective value f of the lane's current trial point and advance the
// state machine to the next trial point.  Returns true when the fit has finished
// (lane.phase == PH_IDLE, result in `res`).
//
// `amask` = lanes of the warp that are inside this call.  The phase switch is divergent by nature;
// the sort / termination test / reflection that follows is common to every lane that completed an
// iteration, so the lanes are re-converged before it (ncu: without the barrier the tail ran ~2.5x
// per evaluation at ~5 active lanes).
__device__ __forceinline__ bool nm_advance(LaneNM &L, const LaneSimplex &S, const NMParams &P, double f,
                                           abfit_fit &res, unsigned amask)
{
    bool iter_done = false;   // an NM iteration (or init) completed: sort + termination test follow
    bool full_sort = false;   // ... and more than the worst vertex changed (init, shrink)
    bool finish = false;      // go to the final LSE evaluation
    bool done = false;        // the fit has ended (result in `res`)
    const int ph = L.phase;
    // ---- reflect / expand / contract: ~99 % of all evaluations --------------------------------------
    // The lanes of a warp are spread over these three phases and their outcomes.  Written as ONE region with
    // per-lane predicates (instead of one switch arm per phase and outcome) so that the lanes share its
    // instruction stream: one centroid, one vertex replacement, one next trial point — whoever needs them.
    if (ph == PH_REFLECT || ph == PH_EXPAND || ph == PH_CONTRACT) {
        ++L.evals;
        const int w = ord_at(L.ord, 4);
        const bool is_r = ph == PH_REFLECT, is_e = ph == PH_EXPAND, is_c = ph == PH_CONTRACT;
        const double c0 = S.c(ord_at(L.ord, 0)), c3 = S.c(ord_at(L.ord, 3)), cw = S.c(w);
        const bool r_accept = is_r && (f < c3 && f >= c0);              // Action::Reflection
        const bool r_expand = is_r && !r_accept && (f < c0);            // Action::Expansion
        const bool r_contract = is_r && !r_accept && !r_expand && (f >= c3);  // Action::ContractionInside
        const bool r_nan = is_r && !r_accept && !r_expand && !r_contract;     // NaN reflection cost: Action::Shrink
        const bool e_take = is_e && (f < L.fr);
        const bool e_keep = is_e && !e_take;  // keep the reflection point (recomputed from the untouched simplex: same bits)
        const bool c_take = is_c && (f < cw);
        const bool c_fail = is_c && !c_take;
        double x0[4] = {0.0, 0.0, 0.0, 0.0};
        if (r_expand || r_contract || e_keep) centroid(S, L.ord, x0);
        if (r_accept || e_take || c_take || e_keep) {  // replace the worst vertex
            double v[4], cost = e_keep ? L.fr : f;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const double xr = x0[j] + (x0[j] - S.x(w, j)) * 1.0;  // NelderMead::reflect
                v[j] = e_keep ? xr : L.xt[j];
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) S.x(w, j) = v[j];
            S.c(w) = cost;
            iter_done = true;
        }
        if (r_expand || r_contract) {
            // xe = x0 + (xr - x0) * 2   /   xc = x0 + (x[4] - x0) * 0.5
            const double coef = r_expand ? 2.0 : 0.5;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const double from = r_expand ? L.xt[j] : S.x(w, j);
                L.xt[j] = x0[j] + (from - x0[j]) * coef;
            }
            if (r_expand) L.fr = f;
            L.phase = r_expand ? PH_EXPAND : PH_CONTRACT;
        }
        if (r_nan || (c_fail && (P.flags & ABFIT_SHRINK_ON_FAILED_CONTRACTION))) {
            L.k = 1;
            shrink_point(S, L.ord, 1, L.xt);
            L.phase = PH_SHRINK;
        } else if (c_fail) {
            if (P.flags & ABFIT_NO_EARLY_EXIT_ON_STALL) {
                iter_done = true;  // argmin 0.8.1: nothing replaced, iteration counted
            } else {
                // Simplex unchanged and next_iter is a pure function of it: all remaining
                // iterations repeat this one.  Same best vertex as after max_iters.
                L.iters = P.max_iters;
                L.status = ABFIT_TERM_STALLED;
                finish = true;
            }
        }
    }
    switch (ph) {
        case PH_INIT: {
            // NOTE: written as "load vertex k+1 relative to k, then bump k" on purpose.  ptxas 12.9 folds
            // `++k; load x[k]` into an LDS with the +1 in the immediate offset AND reads the already
            // incremented register (off-by-one vertex; caught by the bit-exact parity tests).
            const int k = L.k;
            S.c(k) = f;
            ++L.evals;
            L.k = k + 1;
            if (k < 4) {
                const double *nx = S.X + k * 128;  // vertex k; the next one is 128 doubles further
                L.xt[0] = nx[128];
                L.xt[1] = nx[160];
                L.xt[2] = nx[192];
                L.xt[3] = nx[224];
            } else {
                iter_done = true;  // sort + termination test of the Executor's first loop pass
                full_sort = true;
                L.iters = -1;      // the shared tail below counts an iteration; init is not one
            }
            break;
        }
        case PH_SHRINK: {
            ++L.evals;
            const int k = L.k;
            const int s = ord_at(L.ord, k);
#pragma unroll
            for (int j = 0; j < 4; ++j) S.x(s, j) = L.xt[j];
            S.c(s) = f;
            L.k = k + 1;
            if (k < 4) {
                shrink_point(S, L.ord, k + 1, L.xt);
            } else {
                iter_done = true;
                full_sort = true;
            }
            break;
        }
        case PH_LSE: {
            const int b = ord_at(L.ord, 0);
#pragma unroll
            for (int j = 0; j < 4; ++j) res.theta[j] = S.x(b, j);
            res.cost = S.c(b);
            res.lse = f;
            res.iters = L.iters;
            res.evals = L.evals;
            // IterState::update never accepts a NaN cost: best_param stays None and the
            // reference panics on unwrap (src/ab_neutral.rs:66)
            res.status = (res.cost != res.cost) ? ABFIT_FIT_NAN : L.status;
            res.start_id = L.fit_id;
            L.phase = PH_IDLE;
            done = true;
            break;
        }
        default: break;
    }

    __syncwarp(amask);
    if (iter_done) {
        double c[5];
        L.ord = full_sort ? sort5<true>(S, L.ord, c) : sort5<false>(S, L.ord, c);  // sort_param_vecs (stable)
        ++L.iters;
        // Executor: terminate_internal at the top of the next iteration
        bool sd_small = false;
        if (!(c[4] - c[0] > P.range_thr)) {  // else: certainly not converged (NMParams::range_thr)
            double sum = 0.0;
#pragma unroll
            for (int p = 0; p < 5; ++p) sum += c[p];
            const double c0 = sum / 5.0;
            double ss = 0.0;
#pragma unroll
            for (int p = 0; p < 5; ++p) {
                const double d = c[p] - c0;
                ss += d * d;
            }
            // sd = sqrt(1/(n-1) * ss) < sd_tolerance, evaluated without the root (see NMParams::var_thr)
            sd_small = 1.0 / (5.0 - 1.0) * ss <= P.var_thr;
        }
        if (sd_small) {
            L.status = ABFIT_TERM_SD;
            finish = true;
        } else if (L.iters >= P.max_iters) {
            L.status = ABFIT_TERM_MAX_ITERS;
            finish = true;
        } else if (c[0] < -1.7976931348623157e308) {
            // Executor: best_cost <= target_cost (-inf).  The sorted best equals the Executor's best_cost here: a
            // -inf cost always replaces best_cost, and a NaN at position 0 is never the Executor's best.
            L.status = ABFIT_TERM_TARGET_COST;
            finish = true;
        } else {
            reflect_point(S, L.ord, L.xt);
            L.phase = PH_REFLECT;
        }
    }
    if (finish) {
        const int b = ord_at(L.ord, 0);
#pragma unroll
        for (int j = 0; j < 4; ++j) L.xt[j] = S.x(b, j);
        L.phase = PH_LSE;
    }
    return done;
}

// Bootstrap index-tile kernel: resid and pred sit at the very start of dynamic shared memory (so the
// gather address is the byte offset stored in the tile plus a link-time constant); doubles reserved.
__host__ __device__ inline int boot_gather_lead(int n_pairs)
{
    const int npad = (n_pairs + 1) & ~1;
    return (2 * npad + 31) & ~31;
}

// start a new fit on this lane from a 5x4 simplex in global memory
__device__ __forceinline__ void nm_begin(LaneNM &L, const LaneSimplex &S, int fit_id)
{
    L.phase = PH_INIT;
    L.k = 0;
    L.ord = 0u | (1u << 3) | (2u << 6) | (3u << 9) | (4u << 12);
    L.iters = 0;
    L.evals = 0;
    L.status = 0;
    L.fit_id = fit_id;
    L.fr = 0.0;
#pragma unroll
    for (int j = 0; j < 4; ++j) L.xt[j] = S.x(0, j);
}

}  // namespace abfit
