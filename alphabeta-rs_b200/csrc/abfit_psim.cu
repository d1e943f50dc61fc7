// abfit_psim.cu — sm_100a kernels of the parametric bootstrap (abfit_param_boot_batch).
//
//   k_psim_counts  simulates replicate sites of the fitted model and reduces them to exact per-row sums in one pass:
//                  the node walk of k_simulate, the bit-planes of k_pack and the popcounts of k_pairs, all in shared
//                  memory (abfit_psim.cuh holds the tile body); the 17 bytes per sample-site that the materialising
//                  route writes and reads again never reach HBM
//   k_psim_dstar   D*[b][row] = diff / (2.0 * cnt) + theta3, in place over the sums
//
// One block = up to PSIM_MAX_TILES tiles of PSIM_TILE sites of one (window, replicate).  Row counters are packed u32
// (cnt << 16 | diff) in shared memory, one run of rows per thread, and are added at the end of the block to the
// window's packed u64 sums (cnt << 32 | diff) with integer atomics, so the sums do not depend on the grid.  The host
// checks every size the kernel relies on before the launch (abfit_api.cu, abfit_param_boot_batch).
#include <cstdio>
#include <cstdlib>

#include "abfit_internal.h"
#include "abfit_psim.cuh"

namespace abfit {

__global__ void __launch_bounds__(PSIM_TILE)
k_psim_counts(const PsimItem *__restrict__ items, const double *__restrict__ thr6, const int32_t *__restrict__ parent_pos,
              const int32_t *__restrict__ node_id, int n, const int32_t *__restrict__ row_pos,
              const double *__restrict__ miss, int S, const int32_t *__restrict__ row_ij, int R, double thr, uint64_t seed,
              const unsigned long long *__restrict__ keys, int n_boot, unsigned long long *__restrict__ sums)
{
    extern __shared__ unsigned long long psim_smem[];
    uint64_t *ks = reinterpret_cast<uint64_t *>(psim_smem);
    uint64_t *km = ks + n;
    uint32_t *sV = reinterpret_cast<uint32_t *>(km + S);
    uint32_t *sA = sV + S * PSIM_WORDS, *sB = sA + S * PSIM_WORDS;
    uint32_t *ctr = sB + S * PSIM_WORDS;
    uint8_t *st = reinterpret_cast<uint8_t *>(ctr + R);
    const PsimItem it = items[blockIdx.x];
    const int b = blockIdx.y, t = threadIdx.x, lane = t & 31, wid = t >> 5;
    const uint64_t rs = param_boot_seed(seed, keys[it.prob], (uint64_t)b);
    for (int i = t; i < n; i += PSIM_TILE) ks[i] = sim_key(rs, node_id[i], 0);
    for (int s = t; s < S; s += PSIM_TILE) km[s] = sim_key(rs, node_id[row_pos[s]], 1);
    for (int r = t; r < R; r += PSIM_TILE) ctr[r] = 0u;
    const double *th = thr6 + (size_t)it.prob * n * 6;
    const double *mr = miss + (size_t)it.prob * S;
    int r0, r1;
    psim_row_range(R, t, PSIM_TILE, r0, r1);
    __syncthreads();
    for (int k = 0; k < it.n_tiles; ++k) {
        const int64_t site = (it.tile0 + k) * PSIM_TILE + t;
        const bool in = site < it.L;
        if (in) psim_walk(th, parent_pos, n, ks, (uint64_t)site, st, t);
        for (int s = 0; s < S; ++s) {
            const unsigned bits = in ? psim_bits(st[row_pos[s] * PSIM_TILE + t], km[s], (uint64_t)site, mr[s], thr) : 0u;
            const unsigned v = __ballot_sync(0xffffffffu, bits & 1u), a = __ballot_sync(0xffffffffu, bits & 2u),
                           c = __ballot_sync(0xffffffffu, bits & 4u);
            if (lane == 0) {
                sV[s * PSIM_WORDS + wid] = v;
                sA[s * PSIM_WORDS + wid] = a;
                sB[s * PSIM_WORDS + wid] = c;
            }
        }
        __syncthreads();
        psim_pairs(sV, sA, sB, row_ij, r0, r1, ctr);
        __syncthreads();  // the planes are rewritten by the next tile
    }
    unsigned long long *out = sums + ((size_t)it.prob * n_boot + b) * R;
    for (int r = r0; r < r1; ++r) {
        const uint32_t c = ctr[r];
        if (c) atomicAdd(out + r, ((unsigned long long)(c >> 16) << 32) | (c & 0xffffu));
    }
}

// in place: sums[e] (cnt << 32 | diff) -> D* as a double; nan_rep[p * n_boot + b] = 1 when a row of the replicate has
// no valid site
__global__ void k_psim_dstar(unsigned long long *__restrict__ sums, int64_t total, int R, int n_boot,
                             const double *__restrict__ theta3, uint8_t *__restrict__ nan_rep)
{
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const unsigned long long u = sums[e];
        const unsigned long long cnt = u >> 32, diff = u & 0xffffffffull;
        const int64_t pb = e / R;  // p * n_boot + b
        const double d = (double)diff / (2.0 * (double)cnt);  // k_finalize_pairs
        reinterpret_cast<double *>(sums)[e] = d + theta3[pb / n_boot];
        if (cnt == 0ull) nan_rep[pb] = 1;
    }
}

int launch_psim_counts(cudaStream_t st, const PsimItem *items, int n_items, const double *thr6, const int32_t *parent_pos,
                       const int32_t *node_id, int n, const int32_t *row_pos, const double *miss, int S,
                       const int32_t *row_ij, int R, double thr, uint64_t seed, const unsigned long long *keys, int n_boot,
                       unsigned long long *sums)
{
    if (n_items <= 0 || n_boot <= 0) return 0;
    const size_t smem = (size_t)psim_smem_bytes(n, S, R);
    ABFIT_CUDA(cudaFuncSetAttribute(k_psim_counts, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const dim3 grid((unsigned)n_items, (unsigned)n_boot);
    if (getenv("ABFIT_DEV_VERBOSE"))
        fprintf(stderr, "[abfit] k_psim_counts: %u x %u blocks x %d threads, %zu B smem/block\n", grid.x, grid.y, PSIM_TILE,
                smem);
    k_psim_counts<<<grid, PSIM_TILE, smem, st>>>(items, thr6, parent_pos, node_id, n, row_pos, miss, S, row_ij, R, thr, seed,
                                                 keys, n_boot, sums);
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

int launch_psim_dstar(cudaStream_t st, unsigned long long *sums, int64_t total, int R, int n_boot, const double *theta3,
                      uint8_t *nan_rep)
{
    if (total <= 0) return 0;
    const int64_t blocks = std::min<int64_t>((total + 255) / 256, 148 * 32);
    k_psim_dstar<<<(unsigned)blocks, 256, 0, st>>>(sums, total, R, n_boot, theta3, nan_rep);
    ABFIT_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace abfit
