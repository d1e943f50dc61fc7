// abfit_fitkernels.cuh — device code of the two throughput kernels of the ABneutral fit path, written against an
// OBJECTIVE POLICY so that the same source serves two builds:
//
//   * the ahead-of-time build (abfit_kernels.cu): `InterpObjective` interprets the per-window micro-op program
//     (abfit_model.cuh) — any pedigree, any mix of pedigrees in one batch;
//   * the run-time build (abfit_jit.cu, NVRTC): when a whole batch shares one program — every window of a
//     metaprofile does — the host emits that program as straight-line code (`SpecObjective`): no dispatch, no
//     per-lane shared-memory traffic for the model state (everything lives in registers), the pair loop unrolled with
//     each pair's dt1t2 named directly.  Same operations in the same order: same bits.
//
//   fit_starts_body        multi-start Nelder-Mead      (src/ab_neutral.rs:37-78)
//   fit_boot_gather_body   bootstrap refits, index tile (src/boot_model.rs:41-100)
//
// An objective policy provides
//   static constexpr int  N_LANE          doubles of per-lane shared storage it needs (-1: DevProblem::n_lane)
//   static constexpr bool NEEDS_PROGRAM   stage the window's offsets + micro-ops in shared memory
//   template <class DAcc> static double eval(const WarpCtx &, const DAcc &, int lane, alpha, beta, weight, icpt, penalty)
//
// Grid shape: one block per work item; an item is a chunk of consecutive starts / replicates of ONE window, so all
// warps of the block share the staged pedigree and every warp runs a perfectly uniform objective on 32 different
// thetas.  Lanes that finish a fit pull the next start of the chunk from a block-wide counter.
#pragma once
#include "abfit_fitkernels_host.h"
#include "abfit_nm.cuh"

namespace abfit {

template <class OBJ>
__device__ __forceinline__ int obj_n_lane(const DevProblem &pb)
{
    return OBJ::N_LANE >= 0 ? OBJ::N_LANE : pb.n_lane;
}

// ---------------------------------------------------------------------------------
// shared-memory carve-up
//   [ per warp: (n_lane + simplex_doubles) x 32 doubles ] [ D ] [ offs ] [ ops ] [ queue ]
// simplex_doubles: 0 = no Nelder-Mead state, 25 = vertices X (20) + costs C (5) in shared memory,
// 5 = only the costs in shared memory, the vertices in a global (L2-resident) scratch area — they are
// touched once per evaluation, and giving up their 5 KB per warp is what lets 16 warps share an SM.
// ---------------------------------------------------------------------------------
struct Carved {
    WarpCtx ctx;
    LaneSimplex simplex;
    int *queue;
};

template <class OBJ, bool D_SHARED>
__device__ __forceinline__ Carved carve_and_stage(const DevProblem &pb, const DevicePools &P, int simplex_doubles,
                                                  double *x_scratch = nullptr, int lead_doubles = 0)
{
    extern __shared__ double smem[];
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int warp = tid >> 5, lane = tid & 31, n_warps = nthr >> 5;
    const int n_lane = obj_n_lane<OBJ>(pb);
    const int per_warp = (n_lane + simplex_doubles) * 32;
    Carved cv;
    double *mine = smem + lead_doubles + (size_t)warp * per_warp;  // lead_doubles: multiple of 32
    cv.ctx.lm = mine;
    if (simplex_doubles == 25) {
        cv.simplex.X = mine + n_lane * 32 + lane;
        cv.simplex.C = cv.simplex.X + 20 * 32;
    } else if (simplex_doubles == 5) {
        cv.simplex.X = x_scratch + ((size_t)blockIdx.x * n_warps + warp) * (20 * 32) + lane;
        cv.simplex.C = mine + n_lane * 32 + lane;
    } else {
        cv.simplex.X = nullptr;
        cv.simplex.C = nullptr;
    }
    double *p = smem + lead_doubles + (size_t)n_warps * per_warp;  // multiple of 256 bytes
    const double *Dg = P.D + pb.d_off;
    if (D_SHARED) {
        double *Ds = p;
        p += (pb.n_pairs + 1) & ~1;
        for (int i = tid; i < pb.n_pairs; i += nthr) Ds[i] = Dg[i];
        cv.ctx.D = Ds;
    } else {
        cv.ctx.D = Dg;  // pool offsets are even: 16-byte aligned
    }
    if (OBJ::NEEDS_PROGRAM) {
        uint32_t *offs = reinterpret_cast<uint32_t *>(p);  // 16-byte aligned; n_offs is a multiple of 4
        OpWord *ops = reinterpret_cast<OpWord *>(offs + pb.n_offs);
        cv.queue = reinterpret_cast<int *>(ops + pb.n_ops);
        for (int i = tid; i < pb.n_offs; i += nthr) offs[i] = P.offs[pb.offs_off + i];
        for (int i = tid; i < pb.n_ops; i += nthr) ops[i] = P.ops[pb.ops_off + i];
        cv.ctx.offs = offs;
        cv.ctx.ops = ops;
    } else {  // a specialised objective carries the program in its code
        cv.queue = reinterpret_cast<int *>(p);
        cv.ctx.offs = nullptr;
        cv.ctx.ops = nullptr;
    }
    cv.ctx.n_pairs = pb.n_pairs;
    cv.ctx.n_ops = pb.n_ops;
    cv.ctx.p_uu0 = pb.p_uu0;
    cv.ctx.p_mm0 = pb.p_mm0;
    cv.ctx.eqp = pb.eqp;
    cv.ctx.penw = pb.penw;
    return cv;
}

// Pedigrees whose per-lane model state does not fit in shared memory (hundreds of distinct triples: C5's
// 19 900-pair pedigree needs 836 doubles per lane): lane state, simplex vertices, D and the pair offsets all
// live in global memory (an L2-resident scratch, [index][32 lanes] so every access is one coalesced 256-byte
// request); only the simplex costs, the program and the queue stay in shared memory.  Same code, same bits —
// just slower per evaluation.
__device__ __forceinline__ Carved carve_big(const DevProblem &pb, const DevicePools &P, bool with_nm,
                                            double *x_scratch, double *lm_scratch, size_t lm_stride)
{
    extern __shared__ double smem[];
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int warp = tid >> 5, lane = tid & 31, n_warps = nthr >> 5;
    const size_t slot = (size_t)blockIdx.x * n_warps + warp;
    Carved cv;
    cv.ctx.lm = lm_scratch + slot * lm_stride;
    if (with_nm) {
        cv.simplex.X = x_scratch + slot * (20 * 32) + lane;
        cv.simplex.C = smem + (size_t)warp * (5 * 32) + lane;
    } else {
        cv.simplex.X = nullptr;
        cv.simplex.C = nullptr;
    }
    OpWord *ops = reinterpret_cast<OpWord *>(smem + (with_nm ? (size_t)n_warps * (5 * 32) : 0));
    cv.queue = reinterpret_cast<int *>(ops + pb.n_ops);
    for (int i = tid; i < pb.n_ops; i += nthr) ops[i] = P.ops[pb.ops_off + i];
    cv.ctx.D = P.D + pb.d_off;
    cv.ctx.offs = P.offs + pb.offs_off;
    cv.ctx.ops = ops;
    cv.ctx.n_pairs = pb.n_pairs;
    cv.ctx.n_ops = pb.n_ops;
    cv.ctx.p_uu0 = pb.p_uu0;
    cv.ctx.p_mm0 = pb.p_mm0;
    cv.ctx.eqp = pb.eqp;
    cv.ctx.penw = pb.penw;
    return cv;
}

__device__ __forceinline__ void store_fit(abfit_fit *dst, const abfit_fit &r)
{
    // 64-byte record written as four 16-byte vector stores (dst is 64-byte aligned)
    double2 *d = reinterpret_cast<double2 *>(dst);
    d[0] = make_double2(r.theta[0], r.theta[1]);
    d[1] = make_double2(r.theta[2], r.theta[3]);
    d[2] = make_double2(r.cost, r.lse);
    d[3] = make_double2(__hiloint2double(r.evals, r.iters), __hiloint2double(r.start_id, r.status));
}

__device__ __forceinline__ void lane_nm_reset(LaneNM &L)
{
    L.phase = PH_IDLE;
    L.k = 0; L.ord = 0; L.iters = 0; L.evals = 0; L.status = 0; L.fit_id = -1; L.fr = 0.0;
    L.xt[0] = L.xt[1] = L.xt[2] = L.xt[3] = 0.0;
}

// take `count` consecutive fit ids for the idle lanes in mask m; returns this lane's id (or >= end)
__device__ __forceinline__ int queue_take(int *queue, unsigned m, int lane, int end, bool &drained)
{
    int base = end;
    if (!drained) {
        if (lane == 0) base = atomicAdd(queue, __popc(m));
        base = __shfl_sync(FULL, base, 0);
        if (base >= end) drained = true;  // warp-uniform
    }
    return base + __popc(m & ((1u << lane) - 1u));
}

// ---------------------------------------------------------------------------------
// Tail hand-off.  Once a block's queue is drained its warps thin out: Nelder-Mead run lengths spread 4x, so
// a warp keeps executing full-width instructions for a handful of long fits (simulation on the C4 shape:
// 89 % of the issued lanes do useful work with 3 warps per block, 95 % with hand-off).  A warp with few
// active lanes therefore hands them to a sibling warp of the same block that has room, and exits.
//
// Mailbox protocol (one shared int `mb`, one published active-lane count per warp; all offers are
// targeted, every take goes through a CAS, only the donor withdraws):
//   donor     drained, 0 < active <= HANDOFF_MAX, mb == 0, a live sibling r with nact[r] + active <= 32:
//             CAS mb 0 -> OFFER(donor, r, count); park the lane states in its own (now idle) lane_mem;
//             fence; wait: mb == 0 -> taken, exit;  nact[r] < 0 (r has exited) -> CAS OFFER -> 0, resume.
//   receiver  sees OFFER targeted at it (every loop trip, and once more after announcing its exit):
//             CAS OFFER -> TAKING; idle lanes load the parked states and copy the simplices; mb = 0.
// Active-lane counts only fall after the drain, so the room the donor saw is still there when the receiver
// looks.  The moved state is the complete LaneNM + simplex, so results are unchanged bit for bit.
// ---------------------------------------------------------------------------------
constexpr int HANDOFF_MAX = 16;
constexpr int MB_OFFER = 1 << 30, MB_TAKING = 1 << 29;
__device__ __forceinline__ int mb_offer(int donor, int target, int count) { return MB_OFFER | donor | (target << 4) | (count << 8); }

struct HandoffCtx {
    volatile int *mb;            // mailbox word
    volatile signed char *nact;  // [n_warps] published active-lane counts (-1: exited)
    double *lm_base;             // shared: start of warp 0's per-warp region
    int per_warp;                // doubles per warp region
    int n_lane;                  // doubles of lane state (simplex X follows)
};

__device__ __forceinline__ void handoff_park(const LaneNM &L, double *ent, int lane)
{
    ent[0] = L.xt[0]; ent[1] = L.xt[1]; ent[2] = L.xt[2]; ent[3] = L.xt[3];
    ent[4] = L.fr;
    ent[5] = __hiloint2double(L.phase, L.k);
    ent[6] = __hiloint2double((int)L.ord, L.iters);
    ent[7] = __hiloint2double(L.evals, L.status);
    ent[8] = __hiloint2double(L.fit_id, lane);
}
__device__ __forceinline__ int handoff_unpark(LaneNM &L, const double *ent)
{
    L.xt[0] = ent[0]; L.xt[1] = ent[1]; L.xt[2] = ent[2]; L.xt[3] = ent[3];
    L.fr = ent[4];
    L.phase = __double2hiint(ent[5]); L.k = __double2loint(ent[5]);
    L.ord = (uint32_t)__double2hiint(ent[6]); L.iters = __double2loint(ent[6]);
    L.evals = __double2hiint(ent[7]); L.status = __double2loint(ent[7]);
    L.fit_id = __double2hiint(ent[8]);
    return __double2loint(ent[8]);  // the donor lane that owns the simplex
}

// receiver side: returns true when lanes were taken over
__device__ __forceinline__ bool handoff_try_take(const HandoffCtx &H, int warp, int lane, LaneNM &L, const LaneSimplex &S)
{
    const unsigned idle = __ballot_sync(FULL, L.phase == PH_IDLE);
    int v = 0;
    if (lane == 0) {
        v = *H.mb;
        if (!((v & MB_OFFER) && ((v >> 4) & 15) == warp && ((v >> 8) & 63) <= __popc(idle) &&
              atomicCAS(const_cast<int *>(H.mb), v, MB_TAKING) == v))
            v = 0;
    }
    v = __shfl_sync(FULL, v, 0);
    if (!v) return false;
    __threadfence_block();
    const int donor = v & 15, count = (v >> 8) & 63;
    const int rank = __popc(idle & ((1u << lane) - 1u));
    if (L.phase == PH_IDLE && rank < count) {
        const double *dbase = H.lm_base + (size_t)donor * H.per_warp;
        const int dl = handoff_unpark(L, dbase + rank * 16);
        const double *dX = dbase + H.n_lane * 32 + dl;  // donor lane's simplex: X[20], C[5] at stride 32
#pragma unroll
        for (int q = 0; q < 20; ++q) S.X[q * 32] = dX[q * 32];
#pragma unroll
        for (int q = 0; q < 5; ++q) S.C[q * 32] = dX[(20 + q) * 32];
    }
    const unsigned now = __ballot_sync(FULL, L.phase != PH_IDLE);
    if (lane == 0) {
        H.nact[warp] = (signed char)__popc(now);  // published before the mailbox is released: the next donor sees it
        __threadfence_block();
        *H.mb = 0;
    }
    return true;
}

// donor side: returns true when the lanes were taken (the warp is empty now), false when it keeps them
__device__ __forceinline__ bool handoff_try_give(const HandoffCtx &H, int warp, int n_warps, int lane, LaneNM &L,
                                                 unsigned amask, double *my_lm)
{
    const int n_act = __popc(amask);
    int offer = 0;
    if (lane == 0 && *H.mb == 0) {
        int target = -1, best = 0;
        for (int r = 0; r < n_warps; ++r) {
            const int a = H.nact[r];
            if (r != warp && a > best && a + n_act <= 32) {
                best = a;
                target = r;
            }
        }
        if (target >= 0) {
            offer = mb_offer(warp, target, n_act);
            if (atomicCAS(const_cast<int *>(H.mb), 0, MB_TAKING) != 0) offer = 0;  // reserved while the states are parked
            else H.nact[warp] = 0;  // not a target for anybody while it is giving its lanes away
        }
    }
    offer = __shfl_sync(FULL, offer, 0);
    if (!offer) return false;
    if (L.phase != PH_IDLE) handoff_park(L, my_lm + __popc(amask & ((1u << lane) - 1u)) * 16, lane);
    __syncwarp();
    __threadfence_block();
    const int target = (offer >> 4) & 15;
    int taken = 0;  // 1 taken, 2 withdrawn
    if (lane == 0) {
        atomicExch(const_cast<int *>(H.mb), offer);
        for (;;) {
            const int v = *H.mb;
            if (v == 0) {
                taken = 1;
                break;
            }
            if (v == offer && H.nact[target] < 0 && atomicCAS(const_cast<int *>(H.mb), offer, 0) == offer) {
                taken = 2;
                break;
            }
            __nanosleep(256);
        }
    }
    taken = __shfl_sync(FULL, taken, 0);
    if (taken == 1) {
        L.phase = PH_IDLE;  // the fits live on in the receiver
        return true;
    }
    return false;  // withdrawn: registers still hold the states
}

// ---------------------------------------------------------------------------------
// multi-start Nelder-Mead
// ---------------------------------------------------------------------------------
template <class OBJ, bool D_SHARED, bool X_GLOBAL, bool BIG>
__device__ __forceinline__ void fit_starts_body(const DevicePools &P, const WorkItem *__restrict__ items,
                                                const double *__restrict__ simplices, int n_starts, const NMParams &nm,
                                                abfit_fit *__restrict__ all_out,
                                                unsigned long long *__restrict__ evals_per_prob, double *x_scratch,
                                                double *lm_scratch, size_t lm_stride)
{
    constexpr bool HANDOFF = !X_GLOBAL && !BIG;  // the simplex of a moved lane is copied between shared regions
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const WorkItem it = items[blockIdx.x];
    const DevProblem pb = P.probs[it.prob];
    Carved cv = BIG ? carve_big(pb, P, true, x_scratch, lm_scratch, lm_stride)
                    : carve_and_stage<OBJ, D_SHARED>(pb, P, X_GLOBAL ? 5 : 25, x_scratch);
    const int n_lane = obj_n_lane<OBJ>(pb);
    if (threadIdx.x == 0) {
        cv.queue[0] = it.first;
        cv.queue[1] = 0;           // mailbox
        cv.queue[2] = 0x20202020;  // published active-lane counts: everybody full
    }
    __syncthreads();
    const WarpCtx &c = cv.ctx;
    const LaneSimplex &S = cv.simplex;
    const DBroadcast Dat{c.D};
    HandoffCtx H;
    H.mb = cv.queue + 1;
    H.nact = reinterpret_cast<volatile signed char *>(cv.queue + 2);
    H.per_warp = (n_lane + 25) * 32;
    H.lm_base = c.lm - (size_t)warp * H.per_warp;
    H.n_lane = n_lane;

    LaneNM L;
    lane_nm_reset(L);
    const int end = it.first + it.count;
    bool drained = false;
    unsigned long long my_evals = 0;

    for (;;) {
        // ---- refill idle lanes from the block's chunk ----
        const bool need = (L.phase == PH_IDLE);
        const unsigned m = __ballot_sync(FULL, need);
        if (m && !drained) {
            const int idx = queue_take(cv.queue, m, lane, end, drained);
            if (need && idx < end) {
                const double *sx = simplices + ((size_t)it.prob * n_starts + idx) * 20;
#pragma unroll
                for (int q = 0; q < 20; ++q) S.X[q * 32] = sx[q];
                nm_begin(L, S, idx);
            }
        }
        unsigned amask = __ballot_sync(FULL, L.phase != PH_IDLE);
        if (HANDOFF && drained && n_warps > 1 && n_lane * 32 >= HANDOFF_MAX * 16) {
            if (lane == 0) H.nact[warp] = (signed char)__popc(amask);
            if (amask != FULL && handoff_try_take(H, warp, lane, L, S)) {
                amask = __ballot_sync(FULL, L.phase != PH_IDLE);
            } else if (amask && __popc(amask) <= HANDOFF_MAX && handoff_try_give(H, warp, n_warps, lane, L, amask, c.lm)) {
                amask = 0;
            }
        }
        if (!amask) {
            if (HANDOFF && n_warps > 1 && n_lane * 32 >= HANDOFF_MAX * 16) {
                // announce the exit, then look once more: an offer posted in between is either taken here or
                // withdrawn by its donor (whoever wins the CAS)
                if (lane == 0) H.nact[warp] = -1;
                __threadfence_block();
                if (handoff_try_take(H, warp, lane, L, S)) continue;
            }
            break;
        }
        const bool active = (L.phase != PH_IDLE);
        if (active) {
            const double f =
                OBJ::eval(c, Dat, lane, L.xt[0], L.xt[1], L.xt[2], L.xt[3], L.phase != PH_LSE);
            abfit_fit res;
            if (nm_advance(L, S, nm, f, res, amask)) {
                my_evals += (unsigned long long)res.evals;
                store_fit(all_out + (size_t)it.prob * n_starts + res.start_id, res);
            }
        }
    }
    // FLOP accounting: objective evaluations actually executed (excludes the LSE pass)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) my_evals += __shfl_down_sync(FULL, my_evals, o);
    if (lane == 0 && evals_per_prob) atomicAdd(evals_per_prob + it.prob, my_evals);
}

// ---------------------------------------------------------------------------------
// bootstrap refits, index-tile variant (n_pairs <= 8191): D* is never materialised; each lane keeps the
// u16 resample indices of its replicate in an L2-resident tile and gathers resid from shared memory
// (see DGather).  Cuts the per-evaluation L2 traffic of k_fit_boot by 4x.
// ---------------------------------------------------------------------------------
template <class OBJ>
__device__ __forceinline__ void fit_boot_gather_body(const DevicePools &P, const WorkItem *__restrict__ items, int n_boot,
                                                     const abfit_fit *__restrict__ best, const double *__restrict__ pred,
                                                     const double *__restrict__ resid,
                                                     const int32_t *__restrict__ resample_idx,
                                                     const double *__restrict__ vary, uint2 *__restrict__ idx_scratch,
                                                     long long scratch_stride, const NMParams &nm,
                                                     double *__restrict__ rows_out, abfit_fit *__restrict__ fits_out,
                                                     unsigned long long *__restrict__ evals_per_prob,
                                                     int *__restrict__ err_flag, double *x_scratch)
{
    const int lane = threadIdx.x;
    const WorkItem it = items[blockIdx.x];
    const DevProblem pb = P.probs[it.prob];
    Carved cv = carve_and_stage<OBJ, false>(pb, P, x_scratch ? 5 : 25, x_scratch, boot_gather_lead(pb.n_pairs));
    // resid / pred of this window at the start of shared memory
    extern __shared__ double smem_lead[];
    const int npad = (pb.n_pairs + 1) & ~1;
    double *sresid = smem_lead;
    double *spred = smem_lead + npad;
    for (int i = lane; i < pb.n_pairs; i += 32) {
        spred[i] = pred[pb.pair_off + i];
        sresid[i] = resid[pb.pair_off + i];
    }
    __syncwarp();
    const WarpCtx &c = cv.ctx;
    const LaneSimplex &S = cv.simplex;
    uint2 *tile = idx_scratch + (size_t)blockIdx.x * (size_t)scratch_stride + lane;
    const DGather Dat{tile, spred, reinterpret_cast<const char *>(sresid), nullptr};
    const int32_t *idxp = resample_idx + (size_t)pb.pair_off * n_boot;  // [n_boot][n_pairs] of this problem
    const abfit_fit bm = best[it.prob];
    const int ng4 = (pb.n_pairs + 3) >> 2;

    LaneNM L;
    lane_nm_reset(L);
    int next = it.first;
    const int end = it.first + it.count;
    unsigned long long my_evals = 0;

    for (;;) {
        const bool need = (L.phase == PH_IDLE);
        const unsigned m = __ballot_sync(FULL, need);
        if (m && next < end) {
            const int idx = next + __popc(m & ((1u << lane) - 1u));
            if (need && idx < end) {
                // pack this replicate's indices into the lane's tile column (read back by this lane only)
                const int32_t *ib = idxp + (size_t)idx * pb.n_pairs;
                for (int g = 0; g < ng4; ++g) {
                    uint32_t v[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        v[q] = (4 * g + q < pb.n_pairs) ? (uint32_t)ib[4 * g + q] : 0u;
                        if (v[q] >= (uint32_t)pb.n_pairs) {  // reported by download_boot; keeps the gather in bounds
                            v[q] = 0u;
                            *err_flag = 1;
                        }
                        v[q] *= 8u;  // byte offset into resid (n_pairs <= 8191)
                    }
                    tile[(size_t)g * 32] = make_uint2(v[0] | (v[1] << 16), v[2] | (v[3] << 16));
                }
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
                OBJ::eval(c, Dat, lane, L.xt[0], L.xt[1], L.xt[2], L.xt[3], L.phase != PH_LSE);
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
// Continuous lane scheduling ("v2" bodies; specialised objectives, batches whose windows share one program).
//
// The block-per-item bodies above keep a whole block on ONE window: when its queue drains the warps thin out
// (a handful of long fits keep full-width instructions issuing; the hand-off only consolidates them), and a batch
// with few windows per SM slot ends in a ragged last wave — at 1 250 windows per GPU (10 000 sharded over 8) the
// multi-start kernel ran 15-20 % below its large-batch rate; the bootstrap's 100 replicates per window left
// 21.5 of 32 lanes busy.  Here a block is ONE warp that lives for the whole launch (grid = resident warps):
//
//   * work items are chunks of one window's fits, opened one after the other from a global cursor; their
//     sizes follow guided self-scheduling on the host (large first, 32 at the end: make_items_guided), so all
//     warps run out of work within about one fit of each other;
//   * a lane that finishes a fit takes the next fit of the open item AT ONCE, even when the item belongs to
//     another window than the fits still running on its neighbours: a warp keeps V2_SLOTS window slots in shared
//     memory (D column + the window's scalars), every lane points at the slot of its own window.  The objective
//     is the same instruction stream for every lane — only the broadcast loads of D become multi-address loads
//     while windows overlap;
//   * a new item is opened into a slot that has no running fits; with four slots even an item of one fit per
//     lane finds one (measured with two: mid-sized items kept idle lanes waiting for a predecessor's long fits).
//
// No block-wide synchronisation, no inter-block waiting (the cursor is only ever incremented).  A fit's arithmetic
// does not depend on which lane, warp or slot runs it: same bits as the block-per-item kernels.
// ---------------------------------------------------------------------------------

__device__ __forceinline__ WarpCtx v2_ctx(const double *D, const double *scal, int n_pairs)
{
    WarpCtx c;
    c.D = D;
    c.offs = nullptr;
    c.ops = nullptr;
    c.lm = nullptr;
    c.n_pairs = n_pairs;
    c.n_ops = 0;
    c.p_uu0 = scal[0];
    c.p_mm0 = scal[1];
    c.eqp = scal[2];
    c.penw = scal[3];
    return c;
}

// warp-uniform bookkeeping of the open item
struct V2Queue {
    int cur = 0;  // slot being filled from
    int next = 0, end = 0, prob = 0;
    bool exhausted = false;
};

// Opens the next item when the current one is used up.  Returns false when idle lanes have to wait (every slot
// still has running fits) or no items are left.  `busy`: bit s set = slot s has running fits.
template <int NSLOTS, class STAGE>
__device__ __forceinline__ bool v2_open_next(V2Queue &q, const WorkItem *__restrict__ items, int n_items, int *cursor,
                                             int lane, unsigned busy, STAGE stage)
{
    if (q.exhausted) return false;
    const int slot = __ffs(~busy) - 1;  // first slot without running fits
    if (slot >= NSLOTS) return false;
    int idx = 0;
    if (lane == 0) idx = atomicAdd(cursor, 1);
    idx = __shfl_sync(FULL, idx, 0);
    if (idx >= n_items) {
        q.exhausted = true;
        return false;
    }
    const WorkItem it = items[idx];
    q.cur = slot;
    q.next = it.first;
    q.end = it.first + it.count;
    q.prob = it.prob;
    stage(slot, it.prob);
    return true;
}

// bit s = some lane runs a fit on slot s
template <int NSLOTS>
__device__ __forceinline__ unsigned v2_busy_slots(bool active, int my_slot)
{
    unsigned busy = 0;
#pragma unroll
    for (int s = 0; s < NSLOTS; ++s) busy |= (__ballot_sync(FULL, active && my_slot == s) ? 1u : 0u) << s;
    return busy;
}

// ---------------------------------------------------------------------------------
// Drain merging (multi-start kernel, V2_FIT_WARPS > 1).  When the item cursor runs dry every lane still finishes its
// fit, and Nelder-Mead run lengths spread 3.5x: for the last ~20 ms of a launch the machine is full of warps with a few
// live lanes each, and a warp instruction costs the FP64 pipe the same whether 3 or 32 of its lanes are live.  With
// V2_FIT_WARPS warps per block (still independent: own queue state, own slots, NO barrier per evaluation) the warps of
// a block MERGE at that point: the emptiest warp hands its running fits to idle lanes of the fullest warp that has
// room for all of them, and exits.  Everything a fit owns is in shared memory or registers: the receiver lane copies
// the 25-double simplex, takes the LaneNM registers through its own (unused) simplex storage, and keeps reading the
// window's D column from the DONOR's slot — a block's shared memory outlives the warps that filled it.
//
// Protocol (barriers, no polling): a warp that can start no further fit (cursor dry, own item used up) registers in
// `counts`; once all live warps of the block are registered — a condition that stays true: registration is permanent
// and an exiting warp leaves both counts at once — every live warp enters a merge round every V2_MERGE_EVERY
// evaluations: barrier, publish the running lanes, barrier, the same plan computed by every warp, donor parks,
// barrier, receiver adopts.  bar.sync counts exited warps as arrived, so a warp may leave between rounds.
// A fit's arithmetic does not depend on the lane that runs it: same bits.
// ---------------------------------------------------------------------------------
constexpr int V2_MERGE_EVERY = 8;
struct V2MergeCtl {
    int counts;         // (live warps << 8) | registered warps
    int nact[8];        // per merge round: running fits of warp w (0: exited)
    unsigned amask[8];  // ... and the lanes that run them
};
static_assert(sizeof(V2MergeCtl) <= V2_FIT_CTL_BYTES && V2_FIT_WARPS <= 8, "control words of a merging block");

// One merge round; called by every live warp of the block.  my_slot is the BLOCK-wide slot index (warp * V2_SLOTS + s).
template <int FW>
__device__ __forceinline__ void v2_merge_round(V2MergeCtl *ctl, double *smem_block, int warp_doubles, int warp, int lane,
                                               LaneNM &L, const LaneSimplex &S, int &my_slot, int &my_prob)
{
    __syncthreads();
    const unsigned am = __ballot_sync(FULL, L.phase != PH_IDLE);
    if (lane == 0) {
        ctl->nact[warp] = __popc(am);
        ctl->amask[warp] = am;
    }
    __syncthreads();
    int d = -1, r = -1, nd = 33, nr = 0;
#pragma unroll
    for (int w = 0; w < FW; ++w) {
        const int n = ctl->nact[w];
        if (n > 0 && n < nd) {
            d = w;
            nd = n;
        }
    }
#pragma unroll
    for (int w = 0; w < FW; ++w) {
        const int n = ctl->nact[w];
        if (w != d && n > 0 && n + nd <= 32 && n > nr) {
            r = w;
            nr = n;
        }
    }
    if (d < 0 || r < 0) return;  // (block-uniform: every warp read the same words)
    const unsigned dmask = ctl->amask[d], rfree = ~ctl->amask[r];
    if (warp == d && ((dmask >> lane) & 1u)) {
        // park the registers in the simplex storage of the receiver's idle lane that takes this fit over
        const int tl = __fns(rfree, 0, __popc(dmask & ((1u << lane) - 1u)) + 1);
        double *ent = smem_block + (size_t)r * warp_doubles + tl;
        ent[0 * 32] = L.xt[0]; ent[1 * 32] = L.xt[1]; ent[2 * 32] = L.xt[2]; ent[3 * 32] = L.xt[3];
        ent[4 * 32] = L.fr;
        ent[5 * 32] = __hiloint2double(L.phase, L.k);
        ent[6 * 32] = __hiloint2double((int)L.ord, L.iters);
        ent[7 * 32] = __hiloint2double(L.evals, L.status);
        ent[8 * 32] = __hiloint2double(L.fit_id, lane);
        ent[9 * 32] = __hiloint2double(my_prob, my_slot);
    }
    __syncthreads();
    if (warp == r && ((rfree >> lane) & 1u)) {
        const int rank = __popc(rfree & ((1u << lane) - 1u));
        if (rank < nd) {
            const double e5 = S.X[5 * 32], e6 = S.X[6 * 32], e7 = S.X[7 * 32], e8 = S.X[8 * 32], e9 = S.X[9 * 32];
            L.xt[0] = S.X[0 * 32]; L.xt[1] = S.X[1 * 32]; L.xt[2] = S.X[2 * 32]; L.xt[3] = S.X[3 * 32];
            L.fr = S.X[4 * 32];
            L.phase = __double2hiint(e5); L.k = __double2loint(e5);
            L.ord = (uint32_t)__double2hiint(e6); L.iters = __double2loint(e6);
            L.evals = __double2hiint(e7); L.status = __double2loint(e7);
            L.fit_id = __double2hiint(e8);
            my_prob = __double2hiint(e9);
            my_slot = __double2loint(e9);
            const double *src = smem_block + (size_t)d * warp_doubles + __double2loint(e8);  // the donor lane's simplex
#pragma unroll
            for (int k = 0; k < 25; ++k) S.X[k * 32] = src[k * 32];  // X[20] and C[5] are contiguous
        }
    }
    if (warp == d) lane_nm_reset(L);  // handed over; the warp leaves through the regular exit
}

template <class OBJ>
__device__ __forceinline__ void fit_starts_body_v2(const DevicePools &P, const WorkItem *__restrict__ items, int n_items,
                                                   int *cursor, const double *__restrict__ simplices, int n_starts,
                                                   const NMParams &nm, abfit_fit *__restrict__ all_out,
                                                   unsigned long long *__restrict__ evals_per_prob,
                                                   const int *__restrict__ sx_ready)
{
    extern __shared__ double smem_block[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_pairs = P.probs[items[0].prob].n_pairs;  // one program for the whole batch (host: jit_eligible)
    const int npad = (n_pairs + 1) & ~1;
    const int slot_doubles = v2_fit_slot_doubles(n_pairs);
    constexpr int FW = V2_FIT_WARPS;              // > 1: the block's warps merge when the launch drains (see above)
    constexpr int NW = FW > 1 ? FW : V2_WARPS;    // warps per block
    const int warp_doubles = 25 * 32 + V2_SLOTS * slot_doubles;
    double *smem = smem_block + (size_t)warp * warp_doubles;  // this warp's own region
    V2MergeCtl *ctl = reinterpret_cast<V2MergeCtl *>(smem_block + (size_t)NW * warp_doubles);
    if (FW > 1) {
        if (threadIdx.x == 0) ctl->counts = FW << 8;
        if (threadIdx.x < 8) ctl->nact[threadIdx.x] = 0;
        __syncthreads();
    }
    LaneSimplex S;
    S.X = smem + lane;
    S.C = S.X + 20 * 32;
    double *slots = smem + 25 * 32;
    auto stage = [&](int slot, int prob) {
        const DevProblem pb = P.probs[prob];
        double *sl = slots + slot * slot_doubles;
        const double *Dg = P.D + pb.d_off;
        if (sx_ready) {
            // abfit_alphabeta_batch starts this kernel while the start simplices are still crossing PCIe: *sx_ready is
            // the number of windows whose simplices have landed (written by small copies between the chunks of the
            // upload, in stream order).  Windows are opened in order, the upload is ~50 x faster than the fits.
            if (lane == 0) {
                int have;
                do {
                    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(have) : "l"(sx_ready) : "memory");
                    if (have <= prob) __nanosleep(2000);
                } while (have <= prob);
            }
            __syncwarp();
        }
        if (DBroadcast::SUFF) OBJ::stage_stats(Dg, sl, lane);  // experiment: per-triple statistics instead of the column
        else
            for (int i = lane; i < pb.n_pairs; i += 32) sl[i] = Dg[i];
        if (lane == 0) {
            sl[npad] = pb.p_uu0;
            sl[npad + 1] = pb.p_mm0;
            sl[npad + 2] = pb.eqp;
            sl[npad + 3] = pb.penw;
        }
        __syncwarp();
    };

    LaneNM L;
    lane_nm_reset(L);
    int my_slot = 0, my_prob = 0;  // my_slot: FW > 1: block-wide index, warp * V2_SLOTS + slot
    V2Queue q;
    bool registered = false;  // FW > 1: this warp can start no further fit and is counted in ctl->counts
    int since = 0;
    for (;;) {
        // warps of a block stay in phase (shared instruction-cache lines); a warp that has left the loop has exited
        if (FW == 1 && V2_WARPS > 1) __syncthreads();
        else __syncwarp();
        if (FW > 1 && registered && ++since >= V2_MERGE_EVERY) {
            since = 0;
            int c = 0;
            if (lane == 0) c = *reinterpret_cast<volatile int *>(&ctl->counts);
            c = __shfl_sync(FULL, c, 0);
            if ((c >> 8) == (c & 0xff) && (c >> 8) > 1)
                v2_merge_round<FW>(ctl, smem_block, warp_doubles, warp, lane, L, S, my_slot, my_prob);
        }
        unsigned idle = __ballot_sync(FULL, L.phase == PH_IDLE);
        while (idle) {
            if (q.next >= q.end) {
                if (!v2_open_next<V2_SLOTS>(q, items, n_items, cursor, lane,
                                            v2_busy_slots<V2_SLOTS>(L.phase != PH_IDLE, FW > 1 ? my_slot - warp * V2_SLOTS : my_slot), stage))
                    break;
            }
            const int take = min(__popc(idle), q.end - q.next);
            const int rank = __popc(idle & ((1u << lane) - 1u));
            if (((idle >> lane) & 1u) && rank < take) {
                const int id = q.next + rank;
                const double *sx = simplices + ((size_t)q.prob * n_starts + id) * 20;
                // read-only path although, under the upload watch, a copy engine is still writing other windows'
                // simplices: see DESIGN §2.10 for why no stale sector can be read
#pragma unroll
                for (int k = 0; k < 20; ++k) S.X[k * 32] = sx[k];
                nm_begin(L, S, id);
                my_slot = FW > 1 ? warp * V2_SLOTS + q.cur : q.cur;
                my_prob = q.prob;
            }
            q.next += take;
            idle = __ballot_sync(FULL, L.phase == PH_IDLE);
        }
        const bool active = (L.phase != PH_IDLE);
        const unsigned amask = __ballot_sync(FULL, active);
        if (FW > 1 && !registered && q.exhausted && q.next >= q.end) {
            registered = true;
            if (lane == 0) atomicAdd(&ctl->counts, 1);
        }
        if (!amask) {  // nothing runs and nothing could be started: the launch's work is done
            if (FW > 1 && lane == 0) {
                ctl->nact[warp] = 0;
                __threadfence_block();
                atomicSub(&ctl->counts, registered ? 0x101 : 0x100);
            }
            break;
        }
        if (active) {
            const double *sl = FW > 1 ? smem_block + (size_t)(my_slot / V2_SLOTS) * warp_doubles + 25 * 32 + (my_slot % V2_SLOTS) * slot_doubles
                                      : slots + my_slot * slot_doubles;
            const WarpCtx c = v2_ctx(sl, sl + npad, n_pairs);
            const DBroadcast Dat{sl};
            const double f = OBJ::eval(c, Dat, lane, L.xt[0], L.xt[1], L.xt[2], L.xt[3], L.phase != PH_LSE);
            abfit_fit res;
            if (nm_advance(L, S, nm, f, res, amask)) {
                store_fit(all_out + (size_t)my_prob * n_starts + res.start_id, res);
                // FLOP accounting: objective evaluations actually executed (excludes the LSE pass)
                if (evals_per_prob) atomicAdd(evals_per_prob + my_prob, (unsigned long long)res.evals);
            }
        }
    }
}

// bootstrap refits (src/boot_model.rs:41-100), index-tile formulation (see DGather): a slot holds the window's
// residuals, predictions, scalars and best model; the lane's resample indices are packed as SHARED-MEMORY BYTE
// OFFSETS of the residuals in the lane's slot, so the gather address is again "tile value + link-time constant".
template <class OBJ>
__device__ __forceinline__ void fit_boot_gather_body_v2(const DevicePools &P, const WorkItem *__restrict__ items, int n_items,
                                                        int *cursor, int n_boot, const abfit_fit *__restrict__ best,
                                                        const double *__restrict__ pred, const double *__restrict__ resid,
                                                        const int32_t *__restrict__ resample_idx,
                                                        const double *__restrict__ vary, uint2 *__restrict__ idx_scratch,
                                                        long long scratch_stride, const NMParams &nm,
                                                        double *__restrict__ rows_out, abfit_fit *__restrict__ fits_out,
                                                        unsigned long long *__restrict__ evals_per_prob,
                                                        int *__restrict__ err_flag)
{
    extern __shared__ double smem_block[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_pairs = P.probs[items[0].prob].n_pairs;
    const int npad = (n_pairs + 1) & ~1;
    const int slot_doubles = v2_boot_slot_doubles(n_pairs);
    double *smem = smem_block + (size_t)warp * (25 * 32 + V2_BOOT_SLOTS * slot_doubles);  // this warp's own region
    LaneSimplex S;
    S.X = smem + lane;
    S.C = S.X + 20 * 32;
    double *slots = smem + 25 * 32;
    const int ng4 = (n_pairs + 3) >> 2;
    uint2 *tile = idx_scratch + ((size_t)blockIdx.x * V2_WARPS + warp) * (size_t)scratch_stride + lane;
    // slot: [resid npad][pred npad][p_uu0, p_mm0, eqp, penw][best theta 4]
    auto stage = [&](int slot, int prob) {
        const DevProblem pb = P.probs[prob];
        double *sl = slots + slot * slot_doubles;
        for (int i = lane; i < pb.n_pairs; i += 32) {
            sl[i] = resid[pb.pair_off + i];
            sl[npad + i] = pred[pb.pair_off + i];
        }
        if (lane == 0) {
            const abfit_fit bm = best[prob];
            sl[2 * npad] = pb.p_uu0;
            sl[2 * npad + 1] = pb.p_mm0;
            sl[2 * npad + 2] = pb.eqp;
            sl[2 * npad + 3] = pb.penw;
#pragma unroll
            for (int k = 0; k < 4; ++k) sl[2 * npad + 4 + k] = bm.theta[k];
        }
        __syncwarp();
    };

    LaneNM L;
    lane_nm_reset(L);
    int my_slot = 0, my_prob = 0;
    // EXPERIMENT (ABFIT_EXPERIMENT_SUFFSTATS): per-triple statistics of the lane's replicate, built when it starts
    double boot_st[OBJ::N_BOOT_STAT > 0 ? OBJ::N_BOOT_STAT : 1];
    V2Queue q;
    for (;;) {
        // warps of a block stay in phase (shared instruction-cache lines); a warp that has left the loop has exited
        if (V2_WARPS > 1) __syncthreads();
        else __syncwarp();
        unsigned idle = __ballot_sync(FULL, L.phase == PH_IDLE);
        while (idle) {
            if (q.next >= q.end) {
                if (!v2_open_next<V2_BOOT_SLOTS>(q, items, n_items, cursor, lane, v2_busy_slots<V2_BOOT_SLOTS>(L.phase != PH_IDLE, my_slot), stage)) break;
            }
            const int take = min(__popc(idle), q.end - q.next);
            const int rank = __popc(idle & ((1u << lane) - 1u));
            if (((idle >> lane) & 1u) && rank < take) {
                const int id = q.next + rank;
                const DevProblem pb = P.probs[q.prob];
                const double *sl = slots + q.cur * slot_doubles;
                // this replicate's resample indices -> byte offsets of its residuals in shared memory
                const uint32_t base = (uint32_t)((const char *)sl - (const char *)smem_block);
                const int32_t *ib = resample_idx + (size_t)pb.pair_off * n_boot + (size_t)id * pb.n_pairs;
                for (int g = 0; g < ng4; ++g) {
                    uint32_t v[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        v[k] = (4 * g + k < pb.n_pairs) ? (uint32_t)ib[4 * g + k] : 0u;
                        if (v[k] >= (uint32_t)pb.n_pairs) {  // reported by download_boot; keeps the gather in bounds
                            v[k] = 0u;
                            *err_flag = 1;
                        }
                        v[k] = base + v[k] * 8u;  // < 64 KB: the host checks the footprint
                    }
                    tile[(size_t)g * 32] = make_uint2(v[0] | (v[1] << 16), v[2] | (v[3] << 16));
                }
                if (DGather::SUFF) {
                    const DGather Dst{tile, sl + npad, reinterpret_cast<const char *>(smem_block), nullptr};
                    OBJ::boot_stats(Dst, boot_st);
                }
                // simplex = [best, vary x 4]  (src/boot_model.rs:69-75)
                const double *vv = vary + ((size_t)q.prob * n_boot + id) * 16;
#pragma unroll
                for (int k = 0; k < 4; ++k) S.X[k * 32] = sl[2 * npad + 4 + k];
#pragma unroll
                for (int k = 0; k < 16; ++k) S.X[(4 + k) * 32] = vv[k];
                nm_begin(L, S, id);
                my_slot = q.cur;
                my_prob = q.prob;
            }
            q.next += take;
            idle = __ballot_sync(FULL, L.phase == PH_IDLE);
        }
        const bool active = (L.phase != PH_IDLE);
        const unsigned amask = __ballot_sync(FULL, active);
        if (!amask) break;
        if (active) {
            const double *sl = slots + my_slot * slot_doubles;
            const WarpCtx c = v2_ctx(nullptr, sl + 2 * npad, n_pairs);
            const DGather Dat{tile, sl + npad, reinterpret_cast<const char *>(smem_block), boot_st};
            const double f = OBJ::eval(c, Dat, lane, L.xt[0], L.xt[1], L.xt[2], L.xt[3], L.phase != PH_LSE);
            abfit_fit res;
            if (nm_advance(L, S, nm, f, res, amask)) {
                if (evals_per_prob) atomicAdd(evals_per_prob + my_prob, (unsigned long long)res.evals);
                const size_t o = (size_t)my_prob * n_boot + res.start_id;
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
}

}  // namespace abfit
