// emul_psim.cpp — HOST build of the tile body of k_psim_counts (alphabeta-rs_b200/csrc/abfit_psim.cuh).
//
// TEST INFRASTRUCTURE ONLY (never loaded by the product package).  Runs the header's node walk, bit construction and
// pair popcounts one "thread" at a time, with the kernel's tiles, warp words, row runs and flush points, so that the CPU
// suite checks the same source against the oracle (abref_simulate, one run per missing rate, + abref_dmatrix).
//   g++ -O1 -std=c++17 -ffp-contract=off -shared -fPIC -o libemul_psim.so emul_psim.cpp   (tests/test_parametric_bootstrap.py)
#include <cstring>
#include <queue>
#include <vector>

#include "../../alphabeta-rs_b200/csrc/abfit_psim.cuh"

using namespace abfit;

extern "C" {

// One replicate of one window: the forest (parent [n], -1 = root; sampled [n]), its draw table in node order (thr_node
// [n][6], abfit_sim_tree_thresholds), per-sample missing rates [S], the replicate's simulator seed, L sites, R rows
// (row_ij[r] = i | j << 16).  -> diff_out / cnt_out [R], the u64 sums the kernel adds up.
int emul_psim_counts(int n, const int32_t *parent, const uint8_t *sampled, const double *thr_node, const double *rates,
                     double thr, uint64_t rep_seed, int64_t L, int R, const int32_t *row_ij, uint64_t *diff_out,
                     uint64_t *cnt_out)
{
    // a walk with parents before children (any such order gives the same draws: they are keyed by node)
    std::vector<std::vector<int>> kids(n);
    std::vector<int> order;
    std::queue<int> q;
    for (int v = 0; v < n; ++v) {
        if (parent[v] < 0) q.push(v);
        else kids[parent[v]].push_back(v);
    }
    while (!q.empty()) {
        const int v = q.front();
        q.pop();
        order.push_back(v);
        for (int c : kids[v]) q.push(c);
    }
    if ((int)order.size() != n) return -1;
    std::vector<int32_t> pos(n), parent_pos(n);
    for (int i = 0; i < n; ++i) pos[order[i]] = i;
    std::vector<double> thr6((size_t)n * 6);
    std::vector<uint64_t> ks(n);
    for (int i = 0; i < n; ++i) {
        const int v = order[i];
        parent_pos[i] = parent[v] < 0 ? -1 : pos[parent[v]];
        std::memcpy(&thr6[(size_t)i * 6], thr_node + (size_t)v * 6, 6 * sizeof(double));
        ks[i] = sim_key(rep_seed, v, 0);
    }
    std::vector<int32_t> row_pos;
    std::vector<uint64_t> km;
    for (int v = 0; v < n; ++v)
        if (sampled[v]) {
            row_pos.push_back(pos[v]);
            km.push_back(sim_key(rep_seed, v, 1));
        }
    const int S = (int)row_pos.size();
    std::vector<uint8_t> st((size_t)n * PSIM_TILE);
    std::vector<uint32_t> sV((size_t)S * PSIM_WORDS), sA(sV.size()), sB(sV.size()), ctr(R, 0u);
    for (int r = 0; r < R; ++r) diff_out[r] = cnt_out[r] = 0;
    const int64_t tiles = (L + PSIM_TILE - 1) / PSIM_TILE;
    for (int64_t tile = 0; tile < tiles; ++tile) {
        std::fill(sV.begin(), sV.end(), 0u);
        std::fill(sA.begin(), sA.end(), 0u);
        std::fill(sB.begin(), sB.end(), 0u);
        for (int t = 0; t < PSIM_TILE; ++t) {
            const int64_t site = tile * PSIM_TILE + t;
            if (site >= L) continue;  // bits 0, as the ballots of out-of-range lanes
            psim_walk(thr6.data(), parent_pos.data(), n, ks.data(), (uint64_t)site, st.data(), t);
            for (int s = 0; s < S; ++s) {
                const unsigned bits = psim_bits(st[(size_t)row_pos[s] * PSIM_TILE + t], km[s], (uint64_t)site, rates[s], thr);
                const uint32_t bit = 1u << (t & 31);
                const int w = s * PSIM_WORDS + (t >> 5);
                if (bits & 1u) sV[w] |= bit;
                if (bits & 2u) sA[w] |= bit;
                if (bits & 4u) sB[w] |= bit;
            }
        }
        for (int t = 0; t < PSIM_TILE; ++t) {
            int r0, r1;
            psim_row_range(R, t, PSIM_TILE, r0, r1);
            psim_pairs(sV.data(), sA.data(), sB.data(), row_ij, r0, r1, ctr.data());
        }
        if ((tile + 1) % PSIM_MAX_TILES == 0 || tile + 1 == tiles) {  // end of a block's run of tiles
            for (int r = 0; r < R; ++r) {
                cnt_out[r] += ctr[r] >> 16;
                diff_out[r] += ctr[r] & 0xffffu;
                ctr[r] = 0u;
            }
        }
    }
    return 0;
}

uint64_t emul_param_boot_seed(uint64_t seed, uint64_t key, uint64_t b) { return param_boot_seed(seed, key, b); }
uint64_t emul_psim_smem_bytes(int n, int S, int R) { return psim_smem_bytes(n, S, R); }
}
