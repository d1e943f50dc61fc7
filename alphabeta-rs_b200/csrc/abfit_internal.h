// abfit_internal.h — host-side declarations shared by the API layer and the kernel launchers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <string>
#include <string_view>
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
// site-block bootstrap refits (abfit_site_boot_batch): the same kernels fitting a given D* matrix
// dstar[pair_off * n_boot + b * n_pairs + i]; a replicate with a NaN D* is not fitted (NaN row, ABFIT_FIT_NAN)
int launch_fit_boot_given(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items, int n_boot,
                          const abfit_fit *best, const double *dstar, const double *vary, double *tile_scratch,
                          int64_t scratch_stride, NMParams nm, double *rows_out, abfit_fit *fits_out,
                          unsigned long long *evals_per_prob, size_t smem_bytes, const BigScratch &big);
int launch_fit_boot_wide_given(cudaStream_t st, const DevicePools &P, const WorkItem *items, int n_items, int n_boot,
                               const abfit_fit *best, const double *dstar, const double *vary, NMParams nm,
                               double *rows_out, abfit_fit *fits_out, unsigned long long *evals_per_prob, size_t smem_bytes);
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
// windows of at most this many sites sum meth_lvl sequentially in site order (bit-identical to the reference)
constexpr int64_t DIV_EXACT_MAX = 65536;

// ---- site-block bootstrap (abfit_siteboot.cu) ---------------------------------------------
constexpr int SB_THREADS = 128;  // pedigree rows per block of k_siteboot_dstar
constexpr int SB_TB = 16;        // replicates per block (u64 accumulators per thread: 2 * SB_TB)
constexpr int SB_KC = 256;       // blocks of counts staged in shared memory at a time
struct SiteBootItem {
    int32_t prob, r0, n_rows, n_pairs;  // pedigree rows [r0, r0 + n_rows) of window prob
    int64_t pair_off;                   // first pedigree row of the window in the concatenated rows
    int64_t blk0;                       // first block of the window in the block list
    int32_t n_blk, pad;
};
// partials[k][P] = (diff, cnt) of block k from the u64 sums of run_divergence
int launch_siteboot_pack(cudaStream_t st, const unsigned long long *diff, const unsigned long long *cnt, int64_t n, uint2 *out);
// counts[blk_off[p] * n_boot + b * n_blk + k]: multiplicity of block k of window p in replicate b (counts zeroed first)
int launch_siteboot_counts(cudaStream_t st, uint64_t seed, uint64_t first_problem_id, const unsigned long long *ids,
                           const long long *blk_off, int n_probs, int n_boot, int64_t n_blk_total, uint32_t *counts);
// dstar[pair_off * n_boot + b * n_pairs + r]; nan_rep[p * n_boot + b] = 1 when a pair of the replicate has no site
int launch_siteboot_dstar(cudaStream_t st, const SiteBootItem *items, int n_items, int n_boot, const uint2 *partials,
                          int64_t P, const uint32_t *counts, const int32_t *row_pair, double *dstar, uint8_t *nan_rep);

// ---- per-region divergence (abfit_regions.cu) ---------------------------------------------
// Regions of at most DIV_EXACT_MAX sites get their diff / cnt from prefix sums over the pieces between region endpoints
// and their methsum from a sequential pass; longer ones run through run_divergence alone (its long-window tree).
struct RegionEdge {
    int32_t region, lo_row, hi_row, pad;  // rows of this chunk's prefix sums to subtract / add (-1: in another chunk)
};
struct RegionPlan {
    std::vector<int64_t> cuts;                    // sorted, unique endpoints of the non-empty short regions
    std::vector<int32_t> longs;                   // regions of more than DIV_EXACT_MAX sites
    std::vector<std::vector<RegionEdge>> edges;   // per chunk of pieces
    int64_t chunk = 1;                            // pieces per run_divergence call
    size_t max_edges = 0;
    size_t bytes = 0;                             // device scratch of the call (outputs and inputs not included)
};
// lo / hi: host arrays [W], already checked to be ranges of [0, L]
int plan_regions(int S, int64_t L, const int64_t *lo, const int64_t *hi, int W, RegionPlan &plan);
// every pointer but h_lo / h_hi is device memory; outputs [W][P] / [W][S] / [W]
int run_region_divergence(cudaStream_t st, DivArena *arena, const RegionPlan &plan, const uint8_t *d_status,
                          const double *d_post, const double *d_meth, int S, int64_t L, const int64_t *h_lo,
                          const int64_t *h_hi, int W, double thr, double *d_D, unsigned long long *d_diff,
                          unsigned long long *d_cnt, double *d_methsum, long long *d_nvalid, double *d_p0uu, int *launches);

// ---- pedigree lists (abfit_inputs.cu) ---------------------------------------------------
// the methylome parser's chromosome rule (Numbered(n) -> n, M -> 256, C -> 257, "chr" prefixes dropped) and its u32
bool parse_chromosome_name(std::string_view s, int32_t &c);
bool parse_u32_field(std::string_view s, uint32_t &v);
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
// the walk order of k_simulate: per walk position its parent's position (-1: root) and node index; per sampled row its
// walk position
void sim_walk(const abfit_sim_tree *tree, std::vector<int32_t> &parent_pos, std::vector<int32_t> &node_id,
              std::vector<int32_t> &row_pos);
// abfit_sim_tree_thresholds in walk order: out [n_nodes][6] (ABFIT_ERR_ARG for parameters outside [0, 1])
int sim_thresholds_walk(const abfit_sim_tree *tree, const abfit_sim_params *params, double *out);

// ---- parametric bootstrap (abfit_psim.cu) -------------------------------------------------
struct PsimItem {
    int32_t prob, n_tiles;  // tiles [tile0, tile0 + n_tiles) of window prob, n_tiles <= PSIM_MAX_TILES
    int64_t tile0;
    int64_t L;              // sites of the window
};
// sums [n_probs][n_boot][R] packed cnt << 32 | diff, zeroed first; grid = n_items x n_boot
int launch_psim_counts(cudaStream_t st, const PsimItem *items, int n_items, const double *thr6, const int32_t *parent_pos,
                       const int32_t *node_id, int n, const int32_t *row_pos, const double *miss, int S,
                       const int32_t *row_ij, int R, double thr, uint64_t seed, const unsigned long long *keys, int n_boot,
                       unsigned long long *sums);
// in place: sums -> D* = diff / (2.0 * cnt) + theta3[p] (doubles, layout of the site bootstrap's D*); nan_rep zeroed first
int launch_psim_dstar(cudaStream_t st, unsigned long long *sums, int64_t total, int R, int n_boot, const double *theta3,
                      uint8_t *nan_rep);

}  // namespace abfit
