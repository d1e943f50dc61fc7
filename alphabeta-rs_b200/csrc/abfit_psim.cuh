// abfit_psim.cuh — the tile body of k_psim_counts (abfit_psim.cu), the parametric bootstrap's fused simulate-and-count
// kernel.  Plain functions of one thread's work, so that tests/host_emul builds the same source for the CPU and checks
// it against the CPU oracle of the simulation and of the observed divergence without a GPU.
//
// One tile = PSIM_TILE consecutive sites of one replicate, one site per thread:
//   psim_walk   the node walk of k_simulate: every node's state of the site into st[node][PSIM_TILE] bytes
//   psim_bits   the three bits k_pack would make of a sampled row's site: valid (posterior_max >= thr), status >= 1,
//               status >= 2 (|a - b| = [a >= 1 differs] + [a >= 2 differs])
//   psim_pairs  the popcounts of k_pairs over the tile's bit-planes [S][PSIM_WORDS] of 32-site words (word w holds sites
//               32 w .. 32 w + 31 of the tile, bit l = site 32 w + l), added to packed counters cnt << 16 | diff
#pragma once
#include <stdint.h>

#include "abfit_rng.h"

namespace abfit {

constexpr int PSIM_TILE = 256;                    // sites per tile = threads per block
constexpr int PSIM_WORDS = PSIM_TILE / 32;        // 32-site words per sample and plane
constexpr int PSIM_MAX_S = 200;                   // samples (the C5 design)
constexpr int PSIM_MAX_TILES = 64;                // tiles between flushes: cnt <= 16384, diff <= 32768 fit 16 bits each
constexpr uint64_t SIM_STREAM = 4;                // generator stream of the simulator (abfit_rng.h lists the others)

// dynamic shared memory of one k_psim_counts block: state keys [n] and missingness keys [S] (u64), the three planes
// [S][PSIM_WORDS] and the row counters [R] (u32), the node states [n][PSIM_TILE] (u8)
ABFIT_HD inline uint64_t psim_smem_bytes(int n_nodes, int S, int n_rows)
{
    return 8ull * n_nodes + 8ull * S + 12ull * PSIM_WORDS * S + 4ull * n_rows + (uint64_t)PSIM_TILE * n_nodes;
}

// the simulator's uniform draw of one key at one global site index: top 53 bits of splitmix64(key ^ site) / 2^53
ABFIT_HD inline double sim_u01(uint64_t key, uint64_t site) { return (double)(mix64(key ^ site) >> 11) * (1.0 / 9007199254740992.0); }

// draw key of node `node` (index in the forest's node list): which = 0 state, 1 missingness
ABFIT_HD inline uint64_t sim_key(uint64_t seed, int node, uint64_t which)
{
    uint64_t h = mix64(seed ^ (SIM_STREAM * 0xd1342543de82ef95ull));
    h = mix64(h ^ (uint64_t)node);
    return mix64(h ^ which);
}

ABFIT_HD inline int psim_popc(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}

// thr6 [n][6] draw thresholds in walk order (parents before children), parent_pos [n] (-1 for a root), key_state [n]
ABFIT_HD inline void psim_walk(const double *__restrict__ thr6, const int32_t *__restrict__ parent_pos, int n,
                               const uint64_t *__restrict__ key_state, uint64_t site, uint8_t *__restrict__ st, int t)
{
    for (int i = 0; i < n; ++i) {
        const int p = parent_pos[i];
        const int ps = p < 0 ? 0 : st[p * PSIM_TILE + t];
        const double u = sim_u01(key_state[i], site);
        const double *c = thr6 + 6 * i + 2 * ps;
        st[i * PSIM_TILE + t] = (uint8_t)(u < c[0] ? 0 : u < c[1] ? 1 : 2);
    }
}

// bit 0: valid, bit 1: status >= 1, bit 2: status >= 2.  posterior_max is 0.5 where the missingness draw < rate, else 1
// (abfit_simulate's rule with a per-sample rate; no draw is made at rate 0)
ABFIT_HD inline unsigned psim_bits(int s, uint64_t key_miss, uint64_t site, double rate, double thr)
{
    const double post = rate > 0.0 && sim_u01(key_miss, site) < rate ? 0.5 : 1.0;
    return (post >= thr ? 1u : 0u) | (s >= 1 ? 2u : 0u) | (s >= 2 ? 4u : 0u);
}

// rows [r0, r1): row r is the pair row_ij[r] = i | j << 16 of samples; ctr[r] += cnt << 16 | diff over the tile
ABFIT_HD inline void psim_pairs(const uint32_t *__restrict__ sV, const uint32_t *__restrict__ sA,
                                const uint32_t *__restrict__ sB, const int32_t *__restrict__ row_ij, int r0, int r1,
                                uint32_t *__restrict__ ctr)
{
    int ci = -1;
    uint32_t vi[PSIM_WORDS], ai[PSIM_WORDS], bi[PSIM_WORDS];
    for (int r = r0; r < r1; ++r) {
        const int32_t ij = row_ij[r];
        const int i = ij & 0xffff, j = ij >> 16;
        if (i != ci) {  // rows come in runs of one first sample
            ci = i;
            for (int w = 0; w < PSIM_WORDS; ++w) {
                vi[w] = sV[i * PSIM_WORDS + w];
                ai[w] = sA[i * PSIM_WORDS + w];
                bi[w] = sB[i * PSIM_WORDS + w];
            }
        }
        uint32_t acc = 0;
        for (int w = 0; w < PSIM_WORDS; ++w) {
            const uint32_t m = vi[w] & sV[j * PSIM_WORDS + w];
            acc += ((uint32_t)psim_popc(m) << 16) + (uint32_t)psim_popc((ai[w] ^ sA[j * PSIM_WORDS + w]) & m) +
                   (uint32_t)psim_popc((bi[w] ^ sB[j * PSIM_WORDS + w]) & m);
        }
        ctr[r] += acc;
    }
}

// rows of thread t of T: a contiguous run, so that psim_pairs reloads the first sample's planes rarely
ABFIT_HD inline void psim_row_range(int n_rows, int t, int T, int &r0, int &r1)
{
    r0 = (int)((int64_t)n_rows * t / T);
    r1 = (int)((int64_t)n_rows * (t + 1) / T);
}

}  // namespace abfit
