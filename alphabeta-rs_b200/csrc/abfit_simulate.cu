// abfit_simulate.cu — methylomes simulated under ABneutral on a pedigree forest (include/abfit.h, "simulated
// methylomes").  The host builds the forest, its pedigree rows and a per-node table of draw thresholds (3x3 matrix
// powers under the library's arithmetic contract); the device only compares counter-based uniforms with those
// thresholds, so its output is fixed by the table and the key scheme alone.
//
// Kernel shape: one thread per site.  A thread walks the nodes in topological order, keeping every node's state of its
// site in a byte of shared memory ([node][tile] bytes per block), and stores the sampled rows — 17 bytes per sample-site,
// coalesced across the warp.  Forests whose state does not fit a block's shared memory keep it in a global [block][node]
// [tile] scratch instead.
#include <cmath>
#include <cstring>
#include <map>
#include <memory>
#include <queue>
#include <string>

#include "abfit_internal.h"
#include "abfit_psim.cuh"

struct abfit_sim_tree {
    std::vector<int32_t> parent, gen;
    std::vector<uint8_t> sampled;
    std::vector<int32_t> order;  // topological order (parents before children)
    std::vector<double> pairs;   // [n_pairs][5]
    int32_t n_samples = 0;
};

namespace abfit {
namespace {

constexpr int SIM_TILE = 256;                   // sites per block = threads per block
constexpr int SIM_SMEM_MAX_NODES = 400;         // 100 KB of node states per block; larger forests use global scratch

struct SimNode {
    double c[6];                   // (c0, c1) per parent state
    unsigned long long key_state;  // draw keys of this node
    unsigned long long key_miss;
    int32_t parent_pos;            // position of the parent in the walk, -1 for a root
    int32_t out_row;               // output row, -1 when not sampled
};

__global__ void __launch_bounds__(SIM_TILE) k_simulate(const SimNode *__restrict__ nodes, int n_nodes, int64_t first_site,
                                                        int64_t L, double missing_rate, int with_missing,
                                                        uint8_t *__restrict__ scratch, uint8_t *__restrict__ status,
                                                        double *__restrict__ post, double *__restrict__ meth)
{
    extern __shared__ uint8_t sim_smem[];
    uint8_t *st = scratch ? scratch + (size_t)blockIdx.x * n_nodes * SIM_TILE : sim_smem;
    const int t = threadIdx.x;
    for (int64_t k = (int64_t)blockIdx.x * SIM_TILE + t; k < L; k += (int64_t)gridDim.x * SIM_TILE) {
        const uint64_t site = (uint64_t)(first_site + k);
        for (int i = 0; i < n_nodes; ++i) {
            const SimNode *nd = nodes + i;
            const int p = nd->parent_pos;
            const int ps = p < 0 ? 0 : st[p * SIM_TILE + t];
            const double u = sim_u01(nd->key_state, site);
            const int s = u < nd->c[2 * ps] ? 0 : u < nd->c[2 * ps + 1] ? 1 : 2;
            st[i * SIM_TILE + t] = (uint8_t)s;
            const int row = nd->out_row;
            if (row >= 0) {
                const size_t o = (size_t)row * (size_t)L + (size_t)k;
                status[o] = (uint8_t)s;
                post[o] = with_missing && sim_u01(nd->key_miss, site) < missing_rate ? 0.5 : 1.0;
                meth[o] = (double)s * 0.5;
            }
        }
    }
}

// ---- host arithmetic of the threshold table (same operations as divergence(): FMA chains in the 3x3 products) ----
void genmatrix_h(double a, double b, double G[9])  // src/divergence.rs:96-114
{
    const double oma = 1.0 - a, omb = 1.0 - b;
    const double b1a = b + 1.0 - a, a1b = a + 1.0 - b;
    G[0] = oma * oma;
    G[1] = 2.0 * oma * a;
    G[2] = a * a;
    G[3] = 0.25 * (b1a * b1a);
    G[4] = 0.5 * b1a * a1b;
    G[5] = 0.25 * (a1b * a1b);
    G[6] = b * b;
    G[7] = 2.0 * omb * b;
    G[8] = omb * omb;
}
inline double fma_chain3(double a0, double b0, double a1, double b1, double a2, double b2)
{
    double acc = a0 * b0;
    acc = std::fma(a1, b1, acc);
    return std::fma(a2, b2, acc);
}

bool in01(double x) { return x >= 0.0 && x <= 1.0; }  // false for NaN

int check_params(const abfit_sim_params *p)
{
    if (!p) return ABFIT_ERR_ARG;
    if (!in01(p->alpha) || !in01(p->beta) || !in01(p->weight) || !in01(p->p0uu) || !in01(p->missing_rate)) {
        set_error("simulation parameters: alpha, beta, weight, p0uu and missing_rate must lie in [0, 1]");
        return ABFIT_ERR_ARG;
    }
    return 0;
}

// [n_nodes][6] in node order
void thresholds(const abfit_sim_tree &t, const abfit_sim_params &p, double *out)
{
    int tmax = 0;
    for (size_t v = 0; v < t.gen.size(); ++v) tmax = std::max(tmax, t.gen[v]);
    // powers G^0..G^tmax by matrix_power's chain R <- R.G (src/divergence.rs:16-31)
    std::vector<double> P((size_t)(tmax + 1) * 9);
    const double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    std::memcpy(P.data(), I, sizeof I);
    double G[9];
    genmatrix_h(p.alpha, p.beta, G);
    if (tmax >= 1) std::memcpy(&P[9], G, sizeof G);
    for (int k = 2; k <= tmax; ++k) {
        const double *R = &P[(size_t)(k - 1) * 9];
        double *N = &P[(size_t)k * 9];
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) N[3 * i + j] = fma_chain3(R[3 * i], G[j], R[3 * i + 1], G[3 + j], R[3 * i + 2], G[6 + j]);
    }
    const double p_mm = 1.0 - p.p0uu;
    const double sv0[3] = {p.p0uu, p.weight * p_mm, (1.0 - p.weight) * p_mm};
    for (size_t v = 0; v < t.gen.size(); ++v) {
        double *c = out + 6 * v;
        if (t.parent[v] < 0) {
            const double *M = &P[(size_t)t.gen[v] * 9];
            double s[3];
            for (int j = 0; j < 3; ++j) s[j] = fma_chain3(sv0[0], M[j], sv0[1], M[3 + j], sv0[2], M[6 + j]);
            for (int k = 0; k < 3; ++k) {
                c[2 * k] = s[0];
                c[2 * k + 1] = s[0] + s[1];
            }
        } else {
            const double *M = &P[(size_t)(t.gen[v] - t.gen[t.parent[v]]) * 9];
            for (int k = 0; k < 3; ++k) {
                c[2 * k] = M[3 * k];
                c[2 * k + 1] = M[3 * k] + M[3 * k + 1];
            }
        }
    }
}

// validates the forest, orders it and lists its pairs
int make_tree(int32_t n, const int32_t *parent, const int32_t *gen, const uint8_t *sampled, abfit_sim_tree **out)
{
    auto fail = [](const std::string &m) {
        set_error("simulation pedigree: " + m);
        return ABFIT_ERR_ARG;
    };
    if (n <= 0) return fail("no nodes");
    std::unique_ptr<abfit_sim_tree> t(new abfit_sim_tree());
    t->parent.assign(parent, parent + n);
    t->gen.assign(gen, gen + n);
    t->sampled.resize(n);
    std::vector<std::vector<int32_t>> kids(n);
    for (int32_t v = 0; v < n; ++v) {
        t->sampled[v] = sampled[v] ? 1 : 0;
        if (gen[v] < 0 || gen[v] > 127) return fail("node " + std::to_string(v) + ": generation " + std::to_string(gen[v]) + " outside 0..127");
        const int32_t p = parent[v];
        if (p < -1 || p >= n || p == v) return fail("node " + std::to_string(v) + ": parent index " + std::to_string(p) + " is not a node");
        if (p >= 0) {
            if (gen[p] > gen[v])
                return fail("edge " + std::to_string(p) + " -> " + std::to_string(v) + " goes back in time (generation " +
                            std::to_string(gen[p]) + " -> " + std::to_string(gen[v]) + ")");
            kids[p].push_back(v);
        }
    }
    std::vector<int32_t> depth(n, 0), root(n, -1);
    std::queue<int32_t> q;
    for (int32_t v = 0; v < n; ++v)
        if (parent[v] < 0) {
            q.push(v);
            root[v] = v;
        }
    while (!q.empty()) {
        const int32_t v = q.front();
        q.pop();
        t->order.push_back(v);
        for (int32_t c : kids[v]) {
            depth[c] = depth[v] + 1;
            root[c] = root[v];
            q.push(c);
        }
    }
    if ((int32_t)t->order.size() != n) return fail("the edges form a cycle");
    std::vector<int32_t> meas;
    for (int32_t v = 0; v < n; ++v)
        if (t->sampled[v]) meas.push_back(v);
    t->n_samples = (int32_t)meas.size();
    // pedigree rows: pairs of one tree; the path between two samples runs through their most recent common ancestor,
    // whose generation is the smallest on the path (DMatrix::convert's t0, src/pedigree.rs:264-337)
    for (size_t a = 0; a < meas.size(); ++a)
        for (size_t b = a + 1; b < meas.size(); ++b) {
            int32_t x = meas[a], y = meas[b];
            if (root[x] != root[y]) continue;
            while (depth[x] > depth[y]) x = parent[x];
            while (depth[y] > depth[x]) y = parent[y];
            while (x != y) x = parent[x], y = parent[y];
            const double row[5] = {(double)a, (double)b, (double)gen[x], (double)gen[meas[a]], (double)gen[meas[b]]};
            t->pairs.insert(t->pairs.end(), row, row + 5);
        }
    *out = t.release();
    return 0;
}

}  // namespace

void sim_walk(const abfit_sim_tree *t, std::vector<int32_t> &parent_pos, std::vector<int32_t> &node_id,
              std::vector<int32_t> &row_pos)
{
    const int n = (int)t->parent.size();
    std::vector<int32_t> pos(n);
    for (int i = 0; i < n; ++i) pos[t->order[i]] = i;
    parent_pos.resize(n);
    node_id.assign(t->order.begin(), t->order.end());
    row_pos.clear();
    for (int i = 0; i < n; ++i) parent_pos[i] = t->parent[t->order[i]] < 0 ? -1 : pos[t->parent[t->order[i]]];
    for (int v = 0; v < n; ++v)
        if (t->sampled[v]) row_pos.push_back(pos[v]);
}

int sim_thresholds_walk(const abfit_sim_tree *t, const abfit_sim_params *params, double *out)
{
    if (int rc = check_params(params)) return rc;
    const int n = (int)t->parent.size();
    std::vector<double> thr((size_t)n * 6);
    thresholds(*t, *params, thr.data());
    for (int i = 0; i < n; ++i) std::memcpy(out + (size_t)i * 6, &thr[(size_t)t->order[i] * 6], 6 * sizeof(double));
    return 0;
}

int run_simulate(cudaStream_t st, int n_sms, const abfit_sim_tree *tree, const abfit_sim_params *params, int64_t first_site,
                 int64_t L, uint8_t *status, double *posterior_max, double *meth_lvl, bool device_out, float *kernel_ms)
{
    if (kernel_ms) *kernel_ms = 0.0f;
    if (!tree || first_site < 0 || L < 0) return ABFIT_ERR_ARG;
    if (int rc = check_params(params)) return rc;
    const int n = (int)tree->parent.size();
    const int64_t S = tree->n_samples;
    if (S > 0 && L > 0 && (!status || !posterior_max || !meth_lvl)) return ABFIT_ERR_ARG;
    if (S == 0 || L == 0) return 0;
    // node table in walk order
    std::vector<double> thr((size_t)n * 6);
    thresholds(*tree, *params, thr.data());
    std::vector<int32_t> pos(n), row(n, -1);
    for (int i = 0; i < n; ++i) pos[tree->order[i]] = i;
    for (int v = 0, r = 0; v < n; ++v)
        if (tree->sampled[v]) row[v] = r++;
    std::vector<SimNode> nodes(n);
    for (int i = 0; i < n; ++i) {
        const int v = tree->order[i];
        SimNode &nd = nodes[i];
        std::memcpy(nd.c, &thr[(size_t)v * 6], sizeof nd.c);
        nd.key_state = sim_key(params->seed, v, 0);
        nd.key_miss = sim_key(params->seed, v, 1);
        nd.parent_pos = tree->parent[v] < 0 ? -1 : pos[tree->parent[v]];
        nd.out_row = row[v];
    }
    const int64_t tiles = (L + SIM_TILE - 1) / SIM_TILE;
    const bool in_smem = n <= SIM_SMEM_MAX_NODES;
    const int grid = (int)std::min<int64_t>(tiles, in_smem ? (int64_t)INT32_MAX : (int64_t)std::max(1, n_sms) * 4);
    const size_t smem = in_smem ? (size_t)n * SIM_TILE : 0;
    const size_t scratch_bytes = in_smem ? 0 : (size_t)grid * n * SIM_TILE;
    const size_t SL = (size_t)S * (size_t)L;
    // device buffers of this call, stream-ordered (no device-wide synchronisation from cudaFree)
    char *buf = nullptr;
    const size_t nodes_bytes = (sizeof(SimNode) * n + 255) & ~(size_t)255;
    const size_t scratch_pad = (scratch_bytes + 255) & ~(size_t)255;
    const size_t out_bytes = device_out ? 0 : ((SL + 255) & ~(size_t)255) + 16 * SL;
    ABFIT_CUDA(cudaMallocAsync((void **)&buf, nodes_bytes + scratch_pad + out_bytes, st));
    int rc = 0;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    do {
        SimNode *d_nodes = reinterpret_cast<SimNode *>(buf);
        uint8_t *d_scratch = in_smem ? nullptr : reinterpret_cast<uint8_t *>(buf + nodes_bytes);
        uint8_t *o_status = status;
        double *o_post = posterior_max, *o_meth = meth_lvl;
        if (!device_out) {
            char *o = buf + nodes_bytes + scratch_pad;
            o_status = reinterpret_cast<uint8_t *>(o);
            o_post = reinterpret_cast<double *>(o + ((SL + 255) & ~(size_t)255));
            o_meth = o_post + SL;
        }
        cudaError_t e = cudaMemcpyAsync(d_nodes, nodes.data(), sizeof(SimNode) * n, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess && smem > 48 * 1024)
            e = cudaFuncSetAttribute(k_simulate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess && kernel_ms) {
            e = cudaEventCreate(&e0);
            if (e == cudaSuccess) e = cudaEventCreate(&e1);
            if (e == cudaSuccess) e = cudaEventRecord(e0, st);
        }
        if (e != cudaSuccess) {
            rc = cuda_fail(e, "simulation setup");
            break;
        }
        k_simulate<<<grid, SIM_TILE, smem, st>>>(d_nodes, n, first_site, L, params->missing_rate,
                                                  params->missing_rate > 0.0 ? 1 : 0, d_scratch, o_status, o_post, o_meth);
        if ((e = cudaGetLastError()) != cudaSuccess) {
            rc = cuda_fail(e, "k_simulate launch");
            break;
        }
        if (kernel_ms && (e = cudaEventRecord(e1, st)) != cudaSuccess) {
            rc = cuda_fail(e, "cudaEventRecord");
            break;
        }
        if (!device_out) {
            e = cudaMemcpyAsync(status, o_status, SL, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaMemcpyAsync(posterior_max, o_post, SL * 8, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaMemcpyAsync(meth_lvl, o_meth, SL * 8, cudaMemcpyDeviceToHost, st);
            if (e != cudaSuccess) {
                rc = cuda_fail(e, "simulation download");
                break;
            }
        }
    } while (false);
    cudaFreeAsync(buf, st);
    const cudaError_t es = cudaStreamSynchronize(st);
    if (!rc && es != cudaSuccess) rc = cuda_fail(es, "k_simulate");
    if (!rc && kernel_ms) cudaEventElapsedTime(kernel_ms, e0, e1);
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    return rc;
}

}  // namespace abfit

using namespace abfit;

extern "C" {

int abfit_sim_tree_from_arrays(int32_t n_nodes, const int32_t *parent, const int32_t *generation, const uint8_t *sampled,
                               abfit_sim_tree **out)
{
    if (!out || n_nodes <= 0 || !parent || !generation || !sampled) return ABFIT_ERR_ARG;
    *out = nullptr;
    return make_tree(n_nodes, parent, generation, sampled, out);
}

int abfit_sim_tree_build(const char *nodelist_path, const char *edgelist_path, abfit_sim_tree **out)
{
    if (!nodelist_path || !edgelist_path || !out) return ABFIT_ERR_ARG;
    *out = nullptr;
    std::vector<ListNode> nodes;
    std::vector<std::pair<std::string, std::string>> edges;
    if (int rc = read_node_edge_lists(nodelist_path, edgelist_path, nodes, edges)) return rc;
    const int32_t n = (int32_t)nodes.size();
    std::map<std::string, int32_t> by_name;  // the first node of a name, as the pedigree builder resolves names
    std::vector<int32_t> parent(n, -1), gen(n);
    std::vector<uint8_t> sampled(n);
    for (int32_t v = 0; v < n; ++v) {
        by_name.emplace(nodes[v].name, v);
        if (nodes[v].generation > 127) {
            set_error("simulation pedigree: node " + nodes[v].name + ": generation " + std::to_string(nodes[v].generation) +
                      " outside 0..127");
            return ABFIT_ERR_ARG;
        }
        gen[v] = (int32_t)nodes[v].generation;
        sampled[v] = nodes[v].meth ? 1 : 0;
    }
    for (auto &e : edges) {
        auto a = by_name.find(e.first), b = by_name.find(e.second);
        if (a == by_name.end() || b == by_name.end()) {
            set_error("simulation pedigree: edge " + e.first + " -> " + e.second + " names a node that is not in the nodelist");
            return ABFIT_ERR_ARG;
        }
        int32_t &p = parent[b->second];
        if (p >= 0 && p != a->second) {
            set_error("simulation pedigree: node " + e.second + " has two parents (" + nodes[p].name + " and " + e.first + ")");
            return ABFIT_ERR_ARG;
        }
        p = a->second;
    }
    return make_tree(n, parent.data(), gen.data(), sampled.data(), out);  // node indices count the parsed nodelist lines
}

int abfit_sim_tree_info(const abfit_sim_tree *t, int32_t *n_nodes, int32_t *n_samples, int32_t *n_pairs)
{
    if (!t) return ABFIT_ERR_ARG;
    if (n_nodes) *n_nodes = (int32_t)t->parent.size();
    if (n_samples) *n_samples = t->n_samples;
    if (n_pairs) *n_pairs = (int32_t)(t->pairs.size() / 5);
    return 0;
}

int abfit_sim_tree_pairs(const abfit_sim_tree *t, double *pairs_out, int32_t pairs_cap)
{
    if (!t || !pairs_out) return ABFIT_ERR_ARG;
    if ((int64_t)(t->pairs.size() / 5) > (int64_t)pairs_cap) {
        set_error("abfit_sim_tree_pairs: pairs_out is too small");
        return ABFIT_ERR_ARG;
    }
    if (!t->pairs.empty()) std::memcpy(pairs_out, t->pairs.data(), t->pairs.size() * sizeof(double));
    return 0;
}

int abfit_sim_tree_thresholds(const abfit_sim_tree *t, const abfit_sim_params *params, double *out)
{
    if (!t || !out) return ABFIT_ERR_ARG;
    if (int rc = check_params(params)) return rc;
    thresholds(*t, *params, out);
    return 0;
}

void abfit_sim_tree_free(abfit_sim_tree *t) { delete t; }

int abfit_sim_equilibrium(double alpha, double beta, double *p0uu_out, double *weight_out)
{
    // src/alphabeta.rs:62-71, src/structs.rs:151-154
    const double omb = 1.0 - beta, oma = 1.0 - alpha, s = alpha + beta, sm1 = s - 1.0;
    const double p_uu = (beta * (omb * omb - oma * oma - 1.0)) / (s * (sm1 * sm1 - 2.0));
    const double p_mm = (alpha * (oma * oma - omb * omb - 1.0)) / (s * (sm1 * sm1 - 2.0));
    const double p_um = (4.0 * alpha * beta * (s - 2.0)) / (s * (sm1 * sm1 - 2.0));
    const double w = p_um / (p_um + p_mm);
    if (!in01(alpha) || !in01(beta) || !in01(p_uu) || !in01(w)) {
        set_error("abfit_sim_equilibrium: no steady state for these rates (alpha and beta in [0, 1], not both 0)");
        return ABFIT_ERR_ARG;
    }
    if (p0uu_out) *p0uu_out = p_uu;
    if (weight_out) *weight_out = w;
    return 0;
}

}  // extern "C"
