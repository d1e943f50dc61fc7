// abfit_internal.h — host-side declarations shared by the API layer and the kernel launchers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <string>
#include <vector>

#include "abfit_nm.cuh"
#include "abfit_rng.h"

namespace abfit {

// dynamic shared memory of one block working on problem pb (matches carve_and_stage)
// simplex_doubles: 0 (no NM state), 25 (vertices + costs in shared) or 5 (costs only; vertices in global scratch)
size_t smem_need(const DevProblem &pb, int simplex_doubles, bool d_shared, int n_warps);

void set_error(const std::string &msg);
int cuda_fail(cudaError_t e, const char *what);
#define ABFIT_CUDA(call)                                           \
    do {                                                           \
        cudaError_t e_ = (call);                                   \
        if (e_ != cudaSuccess) return ::abfit::cuda_fail(e_, #call); \
    } while (0)

// scratch of the large-pedigree variants (lane state in global memory); lm == nullptr: regular kernels
struct BigScratch {
    double *lm = nullptr;   // [slot][lm_stride] doubles, slot = block * warps + warp
    size_t lm_stride = 0;   // n_lane_max * 32
    double *x = nullptr;    // simplex vertices [slot][20 * 32]
};

// ---- launchers (abfit_kernels.cu) ---------------------------------------------------
int launch_fit_starts(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items, int n_warps,
                      const double *simplices, int n_starts, NMParams nm, abfit_fit *all_out,
                      unsigned long long *evals_per_prob, size_t smem_bytes, bool d_in_shared, double *x_scratch,
                      const BigScratch &big);
int launch_select(cudaStream_t st, const DevicePools &P, int n_probs, int n_starts, const abfit_fit *all,
                  abfit_fit *best_out, double *pred, double *resid, int32_t *prob_status, size_t smem_bytes,
                  bool d_in_shared, const BigScratch &big, int p_base = 0);  // windows [p_base, p_base + n_probs)
int launch_fit_boot(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items, int n_boot,
                    const abfit_fit *best, const double *pred, const double *resid, const int32_t *resample_idx,
                    const double *vary, double *dstar_scratch, int64_t scratch_stride, NMParams nm,
                    double *rows_out, abfit_fit *fits_out, unsigned long long *evals_per_prob, size_t smem_bytes,
                    int *err_flag, const BigScratch &big);
// index-tile variant (n_pairs <= 8191): idx_scratch holds scratch_stride uint2 per block, scratch_stride >= 32 * ceil(N/4)
size_t smem_need_boot_gather(const DevProblem &pb, int simplex_doubles);
int launch_fit_boot_gather(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items, int n_boot,
                           const abfit_fit *best, const double *pred, const double *resid, const int32_t *resample_idx,
                           const double *vary, void *idx_scratch, int64_t scratch_stride, NMParams nm,
                           double *rows_out, abfit_fit *fits_out, unsigned long long *evals_per_prob, size_t smem_bytes,
                           int *err_flag, double *x_scratch);
// warp-per-fit variants (abfit_wide.cuh): one warp per block; dstar_scratch holds scratch_stride doubles per block
int launch_fit_starts_wide(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items,
                           const double *simplices, int n_starts, NMParams nm, abfit_fit *all_out,
                           unsigned long long *evals_per_prob, size_t smem_bytes, const long long *ss_off = nullptr,
                           const double *ss_all = nullptr, int max_trip = 0);  // ss_*: the sufficient-statistics EXPERIMENT
int launch_wide_stats(cudaStream_t st, const DevicePools &P, int n_probs, int max_trip, const long long *ss_off, double *out);
int launch_fit_boot_wide(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items, int n_boot,
                         const abfit_fit *best, const double *pred, const double *resid, const int32_t *resample_idx,
                         const double *vary, double *dstar_scratch, int64_t scratch_stride, NMParams nm,
                         double *rows_out, abfit_fit *fits_out, unsigned long long *evals_per_prob, size_t smem_bytes,
                         int *err_flag);
int launch_cost_batch(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items,
                      const double *theta, double *cost_out, double *lse_out, size_t smem_bytes, bool d_in_shared,
                      const BigScratch &big);
int launch_model_divergence(cudaStream_t st, const DevicePools &P, const double *theta4, double *dt_out,
                            double *puu_out, size_t smem_bytes, const BigScratch &big);
// vary vertices of every (window, replicate) drawn on the device from the best fits (same numbers as
// abfit_gen_vary_vertices): out[n_probs][n_boot][4][4]
// (ids: optional device array of per-window generator keys, else first_problem_id + window)
int launch_gen_vary(cudaStream_t st, uint64_t seed, uint64_t first_problem_id, const unsigned long long *ids, int n_probs,
                    int n_boot, const abfit_fit *best, double *out);
// resample indices of every (window, replicate, pair) drawn on the device (same numbers as abfit_gen_resample_idx):
// out[pair_off * n_boot + b * n_pairs + i]
int launch_gen_resample(cudaStream_t st, uint64_t seed, uint64_t first_problem_id, const unsigned long long *ids,
                        const DevProblem *probs, int n_probs, int n_boot, int32_t *out);
int launch_fp64_peak(cudaStream_t st, int blocks, int threads, int iters, double *sink);
// RawAnalysis::analyze of every window's bootstrap rows on the device (same bits as the host's abfit_analyze):
// rows [n_probs][n_boot][7] -> out [n_probs][32]; scratch [n_probs * 8 * n_boot] doubles
int launch_analyze(cudaStream_t st, const double *rows, int n_probs, int n_boot, double *out, double *scratch);
int max_dynamic_smem(int device);

// ---- divergence (abfit_divergence.cu) -------------------------------------------------
// grow-only device arena for the pass-to-pass scratch (bit-planes, tables): owned by the context, so repeated
// calls stop paying cudaMalloc / cudaFree (tens of milliseconds against a few milliseconds of kernels)
struct DivArena {
    void *p = nullptr;
    size_t cap = 0;
    // second stream + events of the overlapped pack / pair passes (created at first use)
    static constexpr int MAX_CHUNKS = 16;
    cudaStream_t st2 = nullptr;
    cudaEvent_t ev_start = nullptr, ev_pack_end = nullptr;
    cudaEvent_t ev_pack[MAX_CHUNKS] = {};
};
void div_arena_release(DivArena &a);
// h_seg is a HOST array [W+1]; every other pointer is device memory. d_p0uu [W] may be null.
int run_divergence(cudaStream_t st, const uint8_t *d_status, const double *d_post, const double *d_meth, int S,
                   int64_t L, const int64_t *h_seg, int W, double thr, double *d_D, unsigned long long *d_diff,
                   unsigned long long *d_cnt, double *d_methsum, long long *d_nvalid, double *d_p0uu,
                   int *launches, float *ms /* optional [2]: pack pass, pair pass + finalisation */,
                   DivArena *arena = nullptr /* null: allocate and free inside the call */,
                   int long_windows = -1 /* 0 / 1: what div_long_windows said of the whole call, -1: of h_seg */);
// The window list qualifies for the fused kernel: 1 to 64 windows, each of more than 65 536 sites.  The fused and the
// two-pass path sum meth_lvl in different trees, so a call that is split over devices decides this once, for all of
// its windows, and passes the answer to every shard: each window then gets the bits one device gives it.
bool div_long_windows(const int64_t *h_seg, int W);

// ---- pedigree lists (abfit_inputs.cu) ---------------------------------------------------
struct ListNode {
    size_t id;  // line index after the header
    std::string file, name;
    uint32_t generation;
    bool meth;
};
// the parsed nodelist (lines that do not parse are skipped, as the reference skips them) and the (from, to) names of
// every edgelist line; ABFIT_ERR_ARG when a file cannot be read or no node parses
int read_node_edge_lists(const char *nodelist_path, const char *edgelist_path, std::vector<ListNode> &nodes,
                         std::vector<std::pair<std::string, std::string>> &edges);

// ---- simulation (abfit_simulate.cu) ------------------------------------------------------
// sites [first_site, first_site + L) of every sampled node of `tree` into status / posterior_max / meth_lvl, which are
// device arrays (device_out) or host arrays (staged through device buffers); kernel_ms optional
int run_simulate(cudaStream_t st, int n_sms, const abfit_sim_tree *tree, const abfit_sim_params *params, int64_t first_site,
                 int64_t L, uint8_t *status, double *posterior_max, double *meth_lvl, bool device_out, float *kernel_ms);

}  // namespace abfit
