// abfit_kernels.cu — sm_100a kernels of the ABneutral fit path.
//
//   k_fit_starts   multi-start Nelder-Mead      (src/ab_neutral.rs:37-78)
//   k_select       best-of-starts + pred/resid  (src/ab_neutral.rs:83-135)
//   k_fit_boot     bootstrap refits             (src/boot_model.rs:41-100)
//   k_cost_batch   objective only               (src/structs.rs:191-217)
//   k_model_div    dt1t2 per pair               (src/divergence.rs:33-94)
//   k_fp64_peak    DFMA roofline micro-benchmark
//
// Grid shape: one block per work item; an item is a chunk of consecutive starts /
// replicates of ONE window, so all warps of the block share the staged pedigree (D column,
// per-pair offsets, micro-op program) and every warp runs a perfectly uniform objective on 32
// different thetas.  Lanes that finish a fit pull the next start of the chunk from a
// block-wide counter (one shared-memory atomic per warp refill), which takes the 2-4x
// spread in Nelder-Mead iteration counts off the warp's critical path.  The kernel is bound by
// FP64 issue latency, so the per-fit on-chip footprint (shared bytes per lane) is what
// buys throughput: see DESIGN.md for the accounting.
#include <cstdio>
#include <cstdlib>

#include "abfit_internal.h"
#include "abfit_fitkernels.cuh"
#include "abfit_wide.cuh"

namespace abfit {

// ---------------------------------------------------------------------------------
// the generic objective: interprets the window's micro-op program (abfit_model.cuh)
// ---------------------------------------------------------------------------------
struct InterpObjective {
    static constexpr int N_LANE = -1;
    static constexpr bool NEEDS_PROGRAM = true;
    template <class DAcc>
    static __device__ __forceinline__ double eval(const WarpCtx &c, const DAcc &Dat, int lane, double alpha,
                                                  double beta, double weight, double icpt, bool penalty)
    {
        return objective(c, Dat, lane, alpha, beta, weight, icpt, penalty);
    }
};

template <bool D_SHARED, bool X_GLOBAL, bool BIG>
__global__ void __launch_bounds__(128, X_GLOBAL ? 4 : 3)
k_fit_starts(DevicePools P, const WorkItem *__restrict__ items, const double *__restrict__ simplices,
             int n_starts, NMParams nm, abfit_fit *__restrict__ all_out,
             unsigned long long *__restrict__ evals_per_prob, double *x_scratch, double *lm_scratch,
             size_t lm_stride)
{
    fit_starts_body<InterpObjective, D_SHARED, X_GLOBAL, BIG>(P, items, simplices, n_starts, nm, all_out, evals_per_prob,
                                                             x_scratch, lm_scratch, lm_stride);
}

__global__ void __launch_bounds__(32)
k_fit_boot_gather(DevicePools P, const WorkItem *__restrict__ items, int n_boot, const abfit_fit *__restrict__ best,
                  const double *__restrict__ pred, const double *__restrict__ resid,
                  const int32_t *__restrict__ resample_idx, const double *__restrict__ vary,
                  uint2 *__restrict__ idx_scratch, long long scratch_stride, NMParams nm,
                  double *__restrict__ rows_out, abfit_fit *__restrict__ fits_out,
                  unsigned long long *__restrict__ evals_per_prob, int *__restrict__ err_flag, double *x_scratch)
{
    fit_boot_gather_body<InterpObjective>(P, items, n_boot, best, pred, resid, resample_idx, vary, idx_scratch,
                                          scratch_stride, nm, rows_out, fits_out, evals_per_prob, err_flag, x_scratch);
}

// ---------------------------------------------------------------------------------
// best-of-starts (warp-shuffle argmin) + predicted divergence / residuals of the best
// ---------------------------------------------------------------------------------
template <bool D_SHARED, bool BIG>
__global__ void __launch_bounds__(32)
k_select(DevicePools P, int p_base, int n_starts, const abfit_fit *__restrict__ all, abfit_fit *__restrict__ best_out,
         double *__restrict__ pred, double *__restrict__ resid, int32_t *__restrict__ prob_status,
         double *lm_scratch, size_t lm_stride)
{
    const int lane = threadIdx.x;
    const int p = p_base + blockIdx.x;
    const DevProblem pb = P.probs[p];
    Carved cv = BIG ? carve_big(pb, P, false, nullptr, lm_scratch, lm_stride) : carve_and_stage<InterpObjective, D_SHARED>(pb, P, 0);
    __syncwarp();
    const WarpCtx &c = cv.ctx;

    // src/ab_neutral.rs:83-101: ascending stable sort by LSE, first element wins.
    // Ties go to the lowest start id; a NaN anywhere makes the reference panic (:100).
    const abfit_fit *mine = all + (size_t)p * n_starts;
    double best_lse = 0.0;
    int best_id = -1;
    int bad = 0;
    for (int s = lane; s < n_starts; s += 32) {
        const double lse = mine[s].lse;
        const int st = mine[s].status;
        if (st < 0 || lse != lse) {
            bad = 1;
            continue;
        }
        if (best_id < 0 || lse < best_lse) {
            best_lse = lse;
            best_id = s;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ol = __shfl_down_sync(FULL, best_lse, o);
        const int oi = __shfl_down_sync(FULL, best_id, o);
        bad |= __shfl_down_sync(FULL, bad, o);
        if (oi >= 0 && (best_id < 0 || ol < best_lse || (ol == best_lse && oi < best_id))) {
            best_lse = ol;
            best_id = oi;
        }
    }
    best_id = __shfl_sync(FULL, best_id, 0);
    bad = __shfl_sync(FULL, bad, 0);
    if (lane == 0 && prob_status) prob_status[p] = (bad || best_id < 0) ? ABFIT_ERR_NAN : 0;

    if (best_id < 0) {
        if (lane == 0) {
            abfit_fit r;
            r.theta[0] = r.theta[1] = r.theta[2] = r.theta[3] = nan("");
            r.cost = r.lse = nan("");
            r.iters = r.evals = 0;
            r.status = ABFIT_FIT_NAN;
            r.start_id = -1;
            store_fit(best_out + p, r);
        }
        return;
    }
    const abfit_fit b = mine[best_id];
    if (lane == 0) store_fit(best_out + p, b);
    if (!pred && !resid) return;

    // src/ab_neutral.rs:108-135 (every lane computes the same dt table; pairs are strided)
    model_divergence(c, lane, b.theta[0], b.theta[1], b.theta[2]);
    __syncwarp();
    for (int i = lane; i < c.n_pairs; i += 32) {
        const double pr = b.theta[3] + c.lm[(c.offs[i] >> 8) * 32 + lane];
        if (pred) pred[pb.pair_off + i] = pr;
        if (resid) resid[pb.pair_off + i] = c.D[i] - pr;
    }
}

// ---------------------------------------------------------------------------------
// bootstrap refits: each lane owns a replicate with its own D* column
//   D*_i = pred_i + resid[idx_i]      (src/boot_model.rs:50-57)
// The column is built cooperatively by the warp into a [n_pairs][32] scratch tile
// (coalesced on the lane axis), then read once per evaluation.
// ---------------------------------------------------------------------------------
template <bool BIG>
__global__ void __launch_bounds__(32)
k_fit_boot(DevicePools P, const WorkItem *__restrict__ items, int n_boot, const abfit_fit *__restrict__ best,
           const double *__restrict__ pred, const double *__restrict__ resid,
           const int32_t *__restrict__ resample_idx, const double *__restrict__ vary,
           double *__restrict__ dstar_scratch, long long scratch_stride, NMParams nm,
           double *__restrict__ rows_out, abfit_fit *__restrict__ fits_out,
           unsigned long long *__restrict__ evals_per_prob, int *__restrict__ err_flag, double *x_scratch,
           double *lm_scratch, size_t lm_stride)
{
    const int lane = threadIdx.x;
    const WorkItem it = items[blockIdx.x];
    const DevProblem pb = P.probs[it.prob];
    Carved cv = BIG ? carve_big(pb, P, true, x_scratch, lm_scratch, lm_stride) : carve_and_stage<InterpObjective, false>(pb, P, 25);
    __syncwarp();
    const WarpCtx &c = cv.ctx;
    const LaneSimplex &S = cv.simplex;
    double *tile = dstar_scratch + (size_t)blockIdx.x * (size_t)scratch_stride;
    const DLaneColumn Dat{tile + lane};
    const double *predp = pred + pb.pair_off;
    const double *residp = resid + pb.pair_off;
    const int32_t *idxp = resample_idx + (size_t)pb.pair_off * n_boot;  // [n_boot][n_pairs] of this problem
    const abfit_fit bm = best[it.prob];

    LaneNM L;
    lane_nm_reset(L);
    int next = it.first;
    const int end = it.first + it.count;
    unsigned long long my_evals = 0;

    for (;;) {
        const bool need = (L.phase == PH_IDLE);
        const unsigned m = __ballot_sync(FULL, need);
        if (m && next < end) {
            const int rank = __popc(m & ((1u << lane) - 1u));
            const int idx = next + rank;
            const bool take = need && idx < end;
            // cooperative build of the D* column of every lane that takes a replicate
            unsigned tm = __ballot_sync(FULL, take);
            while (tm) {
                const int tl = __ffs(tm) - 1;
                tm &= tm - 1;
                const int b = __shfl_sync(FULL, idx, tl);
                const int32_t *ib = idxp + (size_t)b * pb.n_pairs;
                for (int i = lane; i < pb.n_pairs; i += 32) {
                    uint32_t ix = (uint32_t)ib[i];
                    if (ix >= (uint32_t)pb.n_pairs) {  // reported by download_boot; keeps the gather in bounds
                        ix = 0u;
                        *err_flag = 1;
                    }
                    tile[(size_t)i * 32 + tl] = predp[i] + residp[ix];
                }
            }
            __syncwarp();
            if (take) {
                // simplex = [best, vary x 4]  (src/boot_model.rs:69-75)
                const double *vv = vary + ((size_t)it.prob * n_boot + idx) * 16;
#pragma unroll
                for (int q = 0; q < 4; ++q) S.X[q * 32] = bm.theta[q];
#pragma unroll
                for (int q = 0; q < 16; ++q) S.X[(4 + q) * 32] = vv[q];
                nm_begin(L, S, idx);
            }
            next += __popc(m);
        }
        const bool active = (L.phase != PH_IDLE);
        const unsigned amask = __ballot_sync(FULL, active);
        if (!amask) break;
        if (active) {
            const double f =
                objective(c, Dat, lane, L.xt[0], L.xt[1], L.xt[2], L.xt[3], L.phase != PH_LSE);
            abfit_fit res;
            if (nm_advance(L, S, nm, f, res, amask)) {
                my_evals += (unsigned long long)res.evals;
                const size_t o = (size_t)it.prob * n_boot + res.start_id;
                // src/boot_model.rs:86-91
                double *row = rows_out + o * 7;
                row[0] = res.theta[0];
                row[1] = res.theta[1];
                row[2] = res.theta[2];
                row[3] = res.theta[3];
                row[4] = p_mm_est(res.theta[0], res.theta[1]);
                row[5] = p_um_est(res.theta[0], res.theta[1]);
                row[6] = p_uu_est(res.theta[0], res.theta[1]);
                if (fits_out) store_fit(fits_out + o, res);
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) my_evals += __shfl_down_sync(FULL, my_evals, o);
    if (lane == 0 && evals_per_prob) atomicAdd(evals_per_prob + it.prob, my_evals);
}

// ---------------------------------------------------------------------------------
// warp-per-fit Nelder-Mead (abfit_wide.cuh) for pedigrees with thousands of pairs: one block = one
// warp = one fit at a time.  Every lane carries the same Nelder-Mead state (the state machine of
// abfit_nm.cuh run redundantly, so the control flow is warp-uniform by construction) and the
// 32 lanes share the work of each objective evaluation.  BOOT: bootstrap replicates
// (src/boot_model.rs:41-100) — the warp first materialises D*_i = pred_i + resid[idx_i] as a row of
// the scratch area, then fits it like an observed column.
// ---------------------------------------------------------------------------------
struct WideBoot {
    const abfit_fit *best;
    const double *pred, *resid;
    const int32_t *resample_idx;
    const double *vary;
    double *dstar;  // [block][stride]
    long long stride;
    double *rows_out;
    int *err_flag;
};

// EXPERIMENT (ABFIT_EXPERIMENT_SUFFSTATS=1): per-triple statistics of every problem's observed column, once per batch.
// One block per problem, one thread per triple walking the pairs in pedigree order; thread 0 adds the centred sums.
// out (per problem, at ss_off[p]): [mean_u][count_u][Q]
__global__ void k_wide_stats(DevicePools P, const long long *__restrict__ ss_off, double *__restrict__ out)
{
    const DevProblem pb = P.probs[blockIdx.x];
    const double *D = P.D + pb.d_off;
    const uint32_t *tid = P.wtid + pb.wtid_off;
    double *o = out + ss_off[blockIdx.x];
    extern __shared__ double q_u[];
    for (int u = threadIdx.x; u < pb.n_trip; u += blockDim.x) {
        double s1 = 0.0;
        int n = 0;
        for (int i = 0; i < pb.n_pairs; ++i)
            if (tid[i] == (uint32_t)u) {
                s1 += D[i];
                ++n;
            }
        const double m = s1 / (double)n;
        double q = 0.0;
        for (int i = 0; i < pb.n_pairs; ++i)
            if (tid[i] == (uint32_t)u) {
                const double e = D[i] - m;
                q += e * e;
            }
        o[u] = m;
        o[pb.n_trip + u] = (double)n;
        q_u[u] = q;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double Q = 0.0;
        for (int u = 0; u < pb.n_trip; ++u) Q += q_u[u];
        o[2 * pb.n_trip] = Q;
    }
}

template <bool BOOT>
__global__ void __launch_bounds__(32)
k_fit_wide(DevicePools P, const WorkItem *__restrict__ items, const double *__restrict__ simplices, int n_per_prob,
           NMParams nm, abfit_fit *__restrict__ fits_out, unsigned long long *__restrict__ evals_per_prob, WideBoot B,
           const long long *__restrict__ ss_off, const double *__restrict__ ss_all)
{
    extern __shared__ double smem[];
    const int lane = threadIdx.x;
    const WorkItem it = items[blockIdx.x];
    const DevProblem pb = P.probs[it.prob];
    WideCtx c;
    double *after = wide_carve(c, smem, pb.tmax, pb.n_trip);
    LaneSimplex S;
    S.X = after + lane;
    S.C = S.X + 20 * 32;
    uint32_t *trip = reinterpret_cast<uint32_t *>(after + 25 * 32);
    for (int i = lane; i < pb.n_trip; i += 32) trip[i] = P.wtrip[pb.wtrip_off + i];
    c.trip = trip;
    c.tid = P.wtid + pb.wtid_off;
    c.D = P.D + pb.d_off;
    c.n_pairs = pb.n_pairs;
    c.n_trip = pb.n_trip;
    c.tmax = pb.tmax;
    c.p_uu0 = pb.p_uu0;
    c.p_mm0 = pb.p_mm0;
    c.eqp = pb.eqp;
    c.penw = pb.penw;
    c.ss = nullptr;
    if (!BOOT && ss_all) {  // experiment: the statistics of this problem, staged behind the triple table
        double *ss = reinterpret_cast<double *>(trip + ((pb.n_trip + 1) & ~1));
        const double *g = ss_all + ss_off[it.prob];
        for (int i = lane; i < 2 * pb.n_trip + 1; i += 32) ss[i] = g[i];
        c.ss = ss;
    }
    __syncwarp();
    double *drow = BOOT ? B.dstar + (size_t)blockIdx.x * (size_t)B.stride : nullptr;
    unsigned long long my_evals = 0;

    for (int f = it.first; f < it.first + it.count; ++f) {
        if (BOOT) {
            const int32_t *ib = B.resample_idx + (size_t)pb.pair_off * n_per_prob + (size_t)f * pb.n_pairs;
            const double *predp = B.pred + pb.pair_off, *residp = B.resid + pb.pair_off;
            for (int i = lane; i < pb.n_pairs; i += 32) {
                uint32_t ix = (uint32_t)ib[i];
                if (ix >= (uint32_t)pb.n_pairs) {  // reported by download_boot; keeps the gather in bounds
                    ix = 0u;
                    *B.err_flag = 1;
                }
                drow[i] = predp[i] + residp[ix];  // src/boot_model.rs:50-57
            }
            c.D = drow;
            // simplex = [best, vary x 4]  (src/boot_model.rs:69-75)
            const abfit_fit bm = B.best[it.prob];
            const double *vv = B.vary + ((size_t)it.prob * n_per_prob + f) * 16;
#pragma unroll
            for (int q = 0; q < 4; ++q) S.X[q * 32] = bm.theta[q];
#pragma unroll
            for (int q = 0; q < 16; ++q) S.X[(4 + q) * 32] = vv[q];
        } else {
            const double *sx = simplices + ((size_t)it.prob * n_per_prob + f) * 20;
#pragma unroll
            for (int q = 0; q < 20; ++q) S.X[q * 32] = sx[q];
        }
        __syncwarp();
        LaneNM L;
        lane_nm_reset(L);
        nm_begin(L, S, f);
        for (;;) {
            const double v = objective_wide(c, lane, L.xt[0], L.xt[1], L.xt[2], L.xt[3], L.phase != PH_LSE);
            abfit_fit res;
            if (nm_advance(L, S, nm, v, res, FULL)) {
                if (lane == 0) {
                    my_evals += (unsigned long long)res.evals;
                    const size_t o = (size_t)it.prob * n_per_prob + res.start_id;
                    if (BOOT) {
                        double *row = B.rows_out + o * 7;  // src/boot_model.rs:86-91
                        row[0] = res.theta[0];
                        row[1] = res.theta[1];
                        row[2] = res.theta[2];
                        row[3] = res.theta[3];
                        row[4] = p_mm_est(res.theta[0], res.theta[1]);
                        row[5] = p_um_est(res.theta[0], res.theta[1]);
                        row[6] = p_uu_est(res.theta[0], res.theta[1]);
                    }
                    if (fits_out) store_fit(fits_out + o, res);
                }
                break;
            }
        }
        __syncwarp();  // every lane is done with this replicate's D* row and simplex
    }
    if (lane == 0 && evals_per_prob && my_evals) atomicAdd(evals_per_prob + it.prob, my_evals);
}

// ---------------------------------------------------------------------------------
// objective only (test hook / CostFunction seam)
// ---------------------------------------------------------------------------------
template <bool D_SHARED, bool BIG>
__global__ void __launch_bounds__(32)
k_cost_batch(DevicePools P, const WorkItem *__restrict__ items, const double *__restrict__ theta,
             double *__restrict__ cost_out, double *__restrict__ lse_out, double *lm_scratch, size_t lm_stride)
{
    const int lane = threadIdx.x;
    const WorkItem it = items[blockIdx.x];
    const DevProblem pb = P.probs[it.prob];
    Carved cv = BIG ? carve_big(pb, P, false, nullptr, lm_scratch, lm_stride) : carve_and_stage<InterpObjective, D_SHARED>(pb, P, 0);
    __syncwarp();
    const DBroadcast Dat{cv.ctx.D};
    if (lane < it.count) {
        const double *th = theta + (size_t)(it.first + lane) * 4;
        const double a = th[0], b = th[1], w = th[2], ic = th[3];
        cost_out[it.first + lane] = objective(cv.ctx, Dat, lane, a, b, w, ic, true);
        if (lse_out) lse_out[it.first + lane] = objective(cv.ctx, Dat, lane, a, b, w, ic, false);
    }
}

template <bool BIG>
__global__ void __launch_bounds__(32)
k_model_div(DevicePools P, const double *__restrict__ theta4, double *__restrict__ dt_out,
            double *__restrict__ puu_out, double *lm_scratch, size_t lm_stride)
{
    const int lane = threadIdx.x;
    const DevProblem pb = P.probs[0];
    Carved cv = BIG ? carve_big(pb, P, false, nullptr, lm_scratch, lm_stride) : carve_and_stage<InterpObjective, false>(pb, P, 0);
    __syncwarp();
    const WarpCtx &c = cv.ctx;
    model_divergence(c, lane, theta4[0], theta4[1], theta4[2]);
    __syncwarp();
    for (int i = lane; i < c.n_pairs; i += 32) dt_out[i] = c.lm[(c.offs[i] >> 8) * 32 + lane];
    if (lane == 0 && puu_out) *puu_out = p_uu_est(theta4[0], theta4[1]);
}

// ---------------------------------------------------------------------------------
// FP64 roofline micro-benchmark: 8 independent DFMA chains per thread
// ---------------------------------------------------------------------------------
// Model::vary x 4 per bootstrap replicate (src/boot_model.rs:69-75, src/structs.rs:100-128), one thread per coordinate
__global__ void k_gen_vary(uint64_t seed, uint64_t first_problem_id, const unsigned long long *__restrict__ ids,
                           int n_probs, int n_boot, const abfit_fit *__restrict__ best, double *__restrict__ out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t per_prob = (size_t)n_boot * 16;
    if (i >= (size_t)n_probs * per_prob) return;
    const int p = (int)(i / per_prob);
    const size_t r = i - (size_t)p * per_prob;
    const int b = (int)(r >> 4), v = (int)((r >> 2) & 3), j = (int)(r & 3);
    const uint64_t key = ids ? (uint64_t)ids[p] : first_problem_id + (uint64_t)p;
    out[i] = vary_coordinate(seed, key, (uint64_t)b, v, j, best[p].theta[j]);
}

// Resample indices of every (window, replicate, pair) drawn on the device (src/boot_model.rs:43-48: the reference draws
// them inside boot_model::run): the numbers abfit_gen_resample_idx gives on the host — integer hashing and one
// double multiplication — in the layout abfit_boot_batch takes, out[pair_off * n_boot + b * n_pairs + i].
// Blocks walk over the windows, threads over a window's n_boot * n_pairs entries.
__global__ void k_gen_resample(uint64_t seed, uint64_t first_problem_id, const unsigned long long *__restrict__ ids,
                               const DevProblem *__restrict__ probs, int n_probs, int n_boot, int32_t *__restrict__ out)
{
    for (int p = blockIdx.x; p < n_probs; p += gridDim.x) {
        const int n_pairs = probs[p].n_pairs;
        const uint64_t key = ids ? (uint64_t)ids[p] : first_problem_id + (uint64_t)p;
        int32_t *o = out + (size_t)probs[p].pair_off * n_boot;
        const size_t n = (size_t)n_boot * n_pairs;
        for (size_t e = threadIdx.x; e < n; e += blockDim.x) {
            const uint64_t b = e / (size_t)n_pairs, i = e - b * (size_t)n_pairs;
            int32_t k = (int32_t)(u01(seed, 3, key, b, i) * (double)n_pairs);
            if (k >= n_pairs) k = n_pairs - 1;
            o[e] = k;
        }
    }
}

// ---------------------------------------------------------------------------------
// RawAnalysis::analyze (src/analysis.rs:50-98) on the device: one thread per (window, statistic column), the same
// sequential sums, Welford updates and linear quantiles as the host's abfit_analyze (csrc/abfit_api.cu) — same
// operations in the same order, same bits.  The column is copied to a scratch segment of its own and heap-sorted there.
// rows [n_probs][n_boot][7], out [n_probs][32], scratch [n_probs * 8][n_boot]
// ---------------------------------------------------------------------------------
__global__ void k_analyze(const double *__restrict__ rows, int n_probs, int n, double *__restrict__ out, double *__restrict__ scratch)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_probs * 8) return;
    const int p = t >> 3, f = t & 7;
    const double *r = rows + (size_t)p * n * 7;
    double *col = scratch + (size_t)t * n;
    double *o = out + (size_t)p * 32;
    const int src = f < 2 ? f : f - 1;  // columns alpha, beta, beta / alpha, weight, intercept, pr_mm, pr_um, pr_uu
    double sum = 0.0;
    if (f == 2) {
        for (int i = 0; i < n; ++i) col[i] = r[7 * (size_t)i + 1] / r[7 * (size_t)i];
        double q[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        int i = 0;
        for (; n - i >= 8; i += 8)
#pragma unroll
            for (int k = 0; k < 8; ++k) q[k] += col[i + k];
        sum += q[0] + q[4];
        sum += q[1] + q[5];
        sum += q[2] + q[6];
        sum += q[3] + q[7];
        for (; i < n; ++i) sum += col[i];
    } else {
        for (int i = 0; i < n; ++i) {
            col[i] = r[7 * (size_t)i + src];
            sum += col[i];
        }
    }
    o[f] = sum / (double)n;
    double mean = 0.0, ssq = 0.0;
    for (int i = 0; i < n; ++i) {
        const double delta = col[i] - mean;
        mean = mean + delta / (double)(i + 1);
        ssq = fma(col[i] - mean, delta, ssq);
    }
    o[8 + f] = sqrt(ssq / ((double)n - 1.0));
    // heap sort, ascending (the order of equal values does not matter for the quantiles)
    for (int start = n / 2 - 1; start >= 0; --start) {
        int root = start;
        const double v = col[root];
        for (;;) {
            int child = 2 * root + 1;
            if (child >= n) break;
            if (child + 1 < n && col[child] < col[child + 1]) ++child;
            if (!(v < col[child])) break;
            col[root] = col[child];
            root = child;
        }
        col[root] = v;
    }
    for (int end = n - 1; end > 0; --end) {
        const double v = col[end];
        col[end] = col[0];
        int root = 0;
        for (;;) {
            int child = 2 * root + 1;
            if (child >= end) break;
            if (child + 1 < end && col[child] < col[child + 1]) ++child;
            if (!(v < col[child])) break;
            col[root] = col[child];
            root = child;
        }
        col[root] = v;
    }
    const double qs[2] = {0.025, 0.975};
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const double pos = (double)(n - 1) * qs[k];
        const double lo = floor(pos), hi = ceil(pos);
        const double a = col[(size_t)lo], b2 = col[(size_t)hi];
        o[16 + 2 * f + k] = a + (b2 - a) * (pos - trunc(pos));
    }
}

int launch_analyze(cudaStream_t st, const double *rows, int n_probs, int n_boot, double *out, double *scratch)
{
    if (n_probs <= 0) return 0;
    k_analyze<<<(n_probs * 8 + 63) / 64, 64, 0, st>>>(rows, n_probs, n_boot, out, scratch);
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

__global__ void k_fp64_peak(int iters, double *sink)
{
    double a0 = 1.0 + threadIdx.x * 1e-9, a1 = a0 + 1e-9, a2 = a0 + 2e-9, a3 = a0 + 3e-9;
    double a4 = a0 + 4e-9, a5 = a0 + 5e-9, a6 = a0 + 6e-9, a7 = a0 + 7e-9;
    const double m = 0.9999999, d = 1e-7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            a0 = __fma_rn(a0, m, d); a1 = __fma_rn(a1, m, d); a2 = __fma_rn(a2, m, d); a3 = __fma_rn(a3, m, d);
            a4 = __fma_rn(a4, m, d); a5 = __fma_rn(a5, m, d); a6 = __fma_rn(a6, m, d); a7 = __fma_rn(a7, m, d);
        }
    }
    const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 123.456) sink[0] = s;  // never true; keeps the chains alive
}

// ---------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------
int max_dynamic_smem(int device)
{
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, device) != cudaSuccess) return 0;
    return v;
}

template <class K>
static int prep_kernel(K kernel, size_t smem_bytes, bool max_shared = true)
{
    if (smem_bytes > 48 * 1024)
        ABFIT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
    // prefer the largest shared-memory carve-out: these kernels keep all per-lane state in shared (the
    // warp-per-fit kernels stream D and the triple ids through L1 instead and leave the split to the driver)
    if (max_shared)
        ABFIT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                        cudaSharedmemCarveoutMaxShared));
    return 0;
}

template <bool D_SHARED, bool X_GLOBAL, bool BIG>
static int launch_fit_starts_t(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items, int n_warps,
                               const double *simplices, int n_starts, NMParams nm, abfit_fit *all_out,
                               unsigned long long *evals_per_prob, size_t smem_bytes, double *x_scratch,
                               const BigScratch &big)
{
    if (int rc = prep_kernel(k_fit_starts<D_SHARED, X_GLOBAL, BIG>, smem_bytes)) return rc;
    if (getenv("ABFIT_DEV_VERBOSE")) {
        int nb = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_fit_starts<D_SHARED, X_GLOBAL, BIG>, 32 * n_warps, smem_bytes);
        fprintf(stderr, "[abfit] k_fit_starts<D_SHARED=%d,X_GLOBAL=%d,BIG=%d>: %d blocks x %d warps, %zu B smem/block, %d blocks/SM\n",
                (int)D_SHARED, (int)X_GLOBAL, (int)BIG, n_items, n_warps, smem_bytes, nb);
    }
    k_fit_starts<D_SHARED, X_GLOBAL, BIG><<<n_items, 32 * n_warps, smem_bytes, st>>>(
        P, items, simplices, n_starts, nm, all_out, evals_per_prob, x_scratch, big.lm, big.lm_stride);
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

int launch_fit_starts(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items, int n_warps,
                      const double *simplices, int n_starts, NMParams nm, abfit_fit *all_out,
                      unsigned long long *evals_per_prob, size_t smem_bytes, bool d_in_shared, double *x_scratch,
                      const BigScratch &big)
{
    if (n_items <= 0) return 0;
    if (const char *pad = getenv("ABFIT_DEV_SMEM_PAD")) smem_bytes += (size_t)atoi(pad);  // occupancy experiments
#define ABFIT_FS(DS, XG, BG)                                                                                         \
    launch_fit_starts_t<DS, XG, BG>(st, P, items, n_items, n_warps, simplices, n_starts, nm, all_out, evals_per_prob, \
                                    smem_bytes, x_scratch, big)
    if (big.lm) return ABFIT_FS(false, true, true);
    if (d_in_shared) return x_scratch ? ABFIT_FS(true, true, false) : ABFIT_FS(true, false, false);
    return x_scratch ? ABFIT_FS(false, true, false) : ABFIT_FS(false, false, false);
#undef ABFIT_FS
}

int launch_select(cudaStream_t st, const DevicePools &P, int n_probs, int n_starts, const abfit_fit *all,
                  abfit_fit *best_out, double *pred, double *resid, int32_t *prob_status, size_t smem_bytes,
                  bool d_in_shared, const BigScratch &big, int p_base)
{
    if (n_probs <= 0) return 0;
    if (big.lm) {
        if (int rc = prep_kernel(k_select<false, true>, smem_bytes)) return rc;
        k_select<false, true><<<n_probs, 32, smem_bytes, st>>>(P, p_base, n_starts, all, best_out, pred, resid, prob_status,
                                                               big.lm, big.lm_stride);
    } else if (d_in_shared) {
        if (int rc = prep_kernel(k_select<true, false>, smem_bytes)) return rc;
        k_select<true, false><<<n_probs, 32, smem_bytes, st>>>(P, p_base, n_starts, all, best_out, pred, resid, prob_status,
                                                               nullptr, 0);
    } else {
        if (int rc = prep_kernel(k_select<false, false>, smem_bytes)) return rc;
        k_select<false, false><<<n_probs, 32, smem_bytes, st>>>(P, p_base, n_starts, all, best_out, pred, resid, prob_status,
                                                                nullptr, 0);
    }
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

int launch_fit_boot(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items, int n_boot,
                    const abfit_fit *best, const double *pred, const double *resid, const int32_t *resample_idx,
                    const double *vary, double *dstar_scratch, int64_t scratch_stride, NMParams nm,
                    double *rows_out, abfit_fit *fits_out, unsigned long long *evals_per_prob, size_t smem_bytes,
                    int *err_flag, const BigScratch &big)
{
    if (n_items <= 0) return 0;
    if (getenv("ABFIT_DEV_VERBOSE"))
        fprintf(stderr, "[abfit] k_fit_boot<BIG=%d>: %d blocks x 1 warp, %zu B smem/block\n", big.lm ? 1 : 0, n_items,
                smem_bytes);
    if (big.lm) {
        if (int rc = prep_kernel(k_fit_boot<true>, smem_bytes)) return rc;
        k_fit_boot<true><<<n_items, 32, smem_bytes, st>>>(P, items, n_boot, best, pred, resid, resample_idx, vary,
                                                          dstar_scratch, (long long)scratch_stride, nm, rows_out,
                                                          fits_out, evals_per_prob, err_flag, big.x, big.lm, big.lm_stride);
    } else {
        if (int rc = prep_kernel(k_fit_boot<false>, smem_bytes)) return rc;
        k_fit_boot<false><<<n_items, 32, smem_bytes, st>>>(P, items, n_boot, best, pred, resid, resample_idx, vary,
                                                           dstar_scratch, (long long)scratch_stride, nm, rows_out,
                                                           fits_out, evals_per_prob, err_flag, nullptr, nullptr, 0);
    }
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

int launch_fit_boot_gather(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items, int n_boot,
                           const abfit_fit *best, const double *pred, const double *resid, const int32_t *resample_idx,
                           const double *vary, void *idx_scratch, int64_t scratch_stride, NMParams nm,
                           double *rows_out, abfit_fit *fits_out, unsigned long long *evals_per_prob, size_t smem_bytes,
                           int *err_flag, double *x_scratch)
{
    if (n_items <= 0) return 0;
    if (int rc = prep_kernel(k_fit_boot_gather, smem_bytes)) return rc;
    if (getenv("ABFIT_DEV_VERBOSE"))
        fprintf(stderr, "[abfit] k_fit_boot_gather: %d blocks x 1 warp, %zu B smem/block%s\n", n_items, smem_bytes,
                x_scratch ? " (vertices in global scratch)" : "");
    k_fit_boot_gather<<<n_items, 32, smem_bytes, st>>>(P, items, n_boot, best, pred, resid, resample_idx, vary,
                                                       static_cast<uint2 *>(idx_scratch), (long long)scratch_stride, nm,
                                                       rows_out, fits_out, evals_per_prob, err_flag, x_scratch);
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

int launch_wide_stats(cudaStream_t st, const DevicePools &P, int n_probs, int max_trip, const long long *ss_off, double *out)
{
    if (n_probs <= 0) return 0;
    k_wide_stats<<<n_probs, 256, (size_t)std::max(max_trip, 1) * 8, st>>>(P, ss_off, out);
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

int launch_fit_starts_wide(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items,
                           const double *simplices, int n_starts, NMParams nm, abfit_fit *all_out,
                           unsigned long long *evals_per_prob, size_t smem_bytes, const long long *ss_off,
                           const double *ss_all, int max_trip)
{
    if (n_items <= 0) return 0;
    if (ss_all) smem_bytes += (size_t)(2 * max_trip + 2) * 8;  // experiment: [mean][count][Q] behind the triple table
    if (int rc = prep_kernel(k_fit_wide<false>, smem_bytes, false)) return rc;
    if (getenv("ABFIT_DEV_VERBOSE"))
        fprintf(stderr, "[abfit] k_fit_wide<starts>: %d blocks x 1 warp, %zu B smem/block%s\n", n_items, smem_bytes,
                ss_all ? " (EXPERIMENT: sufficient statistics)" : "");
    k_fit_wide<false><<<n_items, 32, smem_bytes, st>>>(P, items, simplices, n_starts, nm, all_out, evals_per_prob,
                                                       WideBoot{}, ss_off, ss_all);
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

int launch_fit_boot_wide(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items, int n_boot,
                         const abfit_fit *best, const double *pred, const double *resid, const int32_t *resample_idx,
                         const double *vary, double *dstar_scratch, int64_t scratch_stride, NMParams nm,
                         double *rows_out, abfit_fit *fits_out, unsigned long long *evals_per_prob, size_t smem_bytes,
                         int *err_flag)
{
    if (n_items <= 0) return 0;
    if (int rc = prep_kernel(k_fit_wide<true>, smem_bytes, false)) return rc;
    if (getenv("ABFIT_DEV_VERBOSE"))
        fprintf(stderr, "[abfit] k_fit_wide<boot>: %d blocks x 1 warp, %zu B smem/block\n", n_items, smem_bytes);
    WideBoot B{best, pred, resid, resample_idx, vary, dstar_scratch, (long long)scratch_stride, rows_out, err_flag};
    k_fit_wide<true><<<n_items, 32, smem_bytes, st>>>(P, items, nullptr, n_boot, nm, fits_out, evals_per_prob, B, nullptr, nullptr);
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

int launch_cost_batch(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items,
                      const double *theta, double *cost_out, double *lse_out, size_t smem_bytes, bool d_in_shared,
                      const BigScratch &big)
{
    if (n_items <= 0) return 0;
    if (big.lm) {
        if (int rc = prep_kernel(k_cost_batch<false, true>, smem_bytes)) return rc;
        k_cost_batch<false, true><<<n_items, 32, smem_bytes, st>>>(P, items, theta, cost_out, lse_out, big.lm, big.lm_stride);
    } else if (d_in_shared) {
        if (int rc = prep_kernel(k_cost_batch<true, false>, smem_bytes)) return rc;
        k_cost_batch<true, false><<<n_items, 32, smem_bytes, st>>>(P, items, theta, cost_out, lse_out, nullptr, 0);
    } else {
        if (int rc = prep_kernel(k_cost_batch<false, false>, smem_bytes)) return rc;
        k_cost_batch<false, false><<<n_items, 32, smem_bytes, st>>>(P, items, theta, cost_out, lse_out, nullptr, 0);
    }
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

int launch_model_divergence(cudaStream_t st, const DevicePools &P, const double *theta4, double *dt_out,
                            double *puu_out, size_t smem_bytes, const BigScratch &big)
{
    if (big.lm) {
        if (int rc = prep_kernel(k_model_div<true>, smem_bytes)) return rc;
        k_model_div<true><<<1, 32, smem_bytes, st>>>(P, theta4, dt_out, puu_out, big.lm, big.lm_stride);
    } else {
        if (int rc = prep_kernel(k_model_div<false>, smem_bytes)) return rc;
        k_model_div<false><<<1, 32, smem_bytes, st>>>(P, theta4, dt_out, puu_out, nullptr, 0);
    }
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

int launch_gen_vary(cudaStream_t st, uint64_t seed, uint64_t first_problem_id, const unsigned long long *ids, int n_probs,
                    int n_boot, const abfit_fit *best, double *out)
{
    const size_t n = (size_t)n_probs * n_boot * 16;
    if (n == 0) return 0;
    k_gen_vary<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(seed, first_problem_id, ids, n_probs, n_boot, best, out);
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

int launch_gen_resample(cudaStream_t st, uint64_t seed, uint64_t first_problem_id, const unsigned long long *ids,
                        const DevProblem *probs, int n_probs, int n_boot, int32_t *out)
{
    if (n_probs <= 0 || n_boot <= 0) return 0;
    k_gen_resample<<<(unsigned)std::min(n_probs, 148 * 16), 256, 0, st>>>(seed, first_problem_id, ids, probs, n_probs, n_boot, out);
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

int launch_fp64_peak(cudaStream_t st, int blocks, int threads, int iters, double *sink)
{
    k_fp64_peak<<<blocks, threads, 0, st>>>(iters, sink);
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace abfit
