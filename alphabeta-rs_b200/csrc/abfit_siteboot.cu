// abfit_siteboot.cu — sm_100a kernels of the site-block bootstrap (abfit_site_boot_batch).
//
//   k_siteboot_pack    per-block partial sums (u64 diff / cnt of abfit_divergence over the block list) -> u32 pairs
//   k_siteboot_counts  multiplicity of every block in every replicate (generator stream 5, abfit_gen_site_boot_counts)
//   k_siteboot_dstar   D*[b][row] = sum_k count[b][k] diff[k][pair(row)] / (2 sum_k count[b][k] cnt[k][pair(row)])
//
// A replicate's pair sums are integer combinations of the per-block partials, so every D* is exact: the product is
// accumulated in u64 (IMAD.WIDE on u32 operands) and finalised with k_finalize_pairs' expression.  The partials of a
// window are read once per tile of SB_TB replicates, never once per draw.
#include <cstdio>
#include <cstdlib>

#include "abfit_internal.h"

namespace abfit {

__global__ void k_siteboot_pack(const unsigned long long *__restrict__ diff, const unsigned long long *__restrict__ cnt,
                                int64_t n, uint2 *__restrict__ out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = make_uint2((uint32_t)diff[i], (uint32_t)cnt[i]);  // both < 2 * block_sites < 2^32
}

// A grid-stride loop over the draws of every window (window p owns draws [blk_off[p] n_boot, blk_off[p+1] n_boot)), so
// one long window spreads over the whole device; integer atomics, so the counts do not depend on the order of the draws.
// counts must be zero on entry.
__global__ void k_siteboot_counts(uint64_t seed, uint64_t first_problem_id, const unsigned long long *__restrict__ ids,
                                  const long long *__restrict__ blk_off, int n_probs, int n_boot,
                                  uint32_t *__restrict__ counts)
{
    const long long total = blk_off[n_probs] * n_boot;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long blk = e / n_boot;  // blk_off[p] <= blk < blk_off[p + 1]
        int lo = 0, hi = n_probs - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (blk_off[mid] <= blk) lo = mid;
            else hi = mid - 1;
        }
        const int p = lo;
        const long long b0 = blk_off[p];
        const int n_blk = (int)(blk_off[p + 1] - b0);
        const long long r = e - b0 * n_boot;
        const int b = (int)(r / n_blk), d = (int)(r - (long long)b * n_blk);
        const uint64_t key = ids ? (uint64_t)ids[p] : first_problem_id + (uint64_t)p;
        atomicAdd(counts + b0 * n_boot + (size_t)b * n_blk + site_boot_block(seed, key, (uint64_t)b, (uint64_t)d, n_blk), 1u);
    }
}

// One thread per pedigree row, SB_TB replicates per block; the counts of the tile are staged SB_KC blocks at a time.
__global__ void __launch_bounds__(SB_THREADS)
k_siteboot_dstar(const SiteBootItem *__restrict__ items, int n_boot, const uint2 *__restrict__ partials, int64_t P,
                 const uint32_t *__restrict__ counts, const int32_t *__restrict__ row_pair, double *__restrict__ dstar,
                 uint8_t *__restrict__ nan_rep)
{
    __shared__ uint32_t cs[SB_TB][SB_KC];
    const SiteBootItem it = items[blockIdx.x];
    const int b0 = blockIdx.y * SB_TB;
    const int nb = min(SB_TB, n_boot - b0);
    const int r = it.r0 + threadIdx.x;
    const bool live = threadIdx.x < it.n_rows;
    const int64_t j = live ? row_pair[it.pair_off + r] : 0;
    const uint2 *part = partials + it.blk0 * P + j;
    const uint32_t *cw = counts + it.blk0 * n_boot + (size_t)b0 * it.n_blk;
    unsigned long long sd[SB_TB], sc[SB_TB];
#pragma unroll
    for (int t = 0; t < SB_TB; ++t) sd[t] = sc[t] = 0ull;
    for (int k0 = 0; k0 < it.n_blk; k0 += SB_KC) {
        const int kc = min(SB_KC, it.n_blk - k0);
        __syncthreads();
        for (int e = threadIdx.x; e < SB_TB * SB_KC; e += SB_THREADS) {
            const int t = e / SB_KC, kk = e - t * SB_KC;
            cs[t][kk] = (t < nb && kk < kc) ? cw[(size_t)t * it.n_blk + k0 + kk] : 0u;
        }
        __syncthreads();
        if (live)
            for (int kk = 0; kk < kc; ++kk) {
                const uint2 x = part[(int64_t)(k0 + kk) * P];
#pragma unroll
                for (int t = 0; t < SB_TB; ++t) {
                    const uint32_t c = cs[t][kk];
                    sd[t] += (unsigned long long)c * x.x;
                    sc[t] += (unsigned long long)c * x.y;
                }
            }
    }
    if (!live) return;
#pragma unroll
    for (int t = 0; t < SB_TB; ++t) {
        if (t >= nb) break;
        const int b = b0 + t;
        dstar[it.pair_off * n_boot + (int64_t)b * it.n_pairs + r] = (double)sd[t] / (2.0 * (double)sc[t]);  // k_finalize_pairs
        if (sc[t] == 0ull) nan_rep[(size_t)it.prob * n_boot + b] = 1;
    }
}

int launch_siteboot_pack(cudaStream_t st, const unsigned long long *diff, const unsigned long long *cnt, int64_t n, uint2 *out)
{
    if (n <= 0) return 0;
    k_siteboot_pack<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(diff, cnt, n, out);
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

int launch_siteboot_counts(cudaStream_t st, uint64_t seed, uint64_t first_problem_id, const unsigned long long *ids,
                           const long long *blk_off, int n_probs, int n_boot, int64_t n_blk_total, uint32_t *counts)
{
    if (n_probs <= 0 || n_boot <= 0) return 0;
    const int64_t blocks = std::min<int64_t>((n_blk_total * n_boot + 255) / 256, 148 * 32);
    k_siteboot_counts<<<(unsigned)std::max<int64_t>(blocks, 1), 256, 0, st>>>(seed, first_problem_id, ids, blk_off, n_probs,
                                                                             n_boot, counts);
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

int launch_siteboot_dstar(cudaStream_t st, const SiteBootItem *items, int n_items, int n_boot, const uint2 *partials,
                          int64_t P, const uint32_t *counts, const int32_t *row_pair, double *dstar, uint8_t *nan_rep)
{
    if (n_items <= 0 || n_boot <= 0) return 0;
    const dim3 grid((unsigned)n_items, (unsigned)((n_boot + SB_TB - 1) / SB_TB));
    if (getenv("ABFIT_DEV_VERBOSE"))
        fprintf(stderr, "[abfit] k_siteboot_dstar: %u x %u blocks x %d threads\n", grid.x, grid.y, SB_THREADS);
    k_siteboot_dstar<<<grid, SB_THREADS, 0, st>>>(items, n_boot, partials, P, counts, row_pair, dstar, nan_rep);
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace abfit
