// abfit_regions.cu — the observed divergence of arbitrary genomic regions (BED lines) over the resident site arrays.
//
// A region over a sorted site list is a contiguous range [lo, hi) of site indices, and its diff / cnt sums are integer
// sums over its sites, so they add exactly over disjoint pieces.  Every output of region w equals, bit for bit, what
// abfit_divergence returns for the single window {lo_w, hi_w}; regions may overlap, nest, repeat or be empty, and no
// site is copied.
//
//   host            abfit_parse_region_line (BED line -> chromosome, start0, end), abfit_region_ranges (binary search)
//   pieces          the site axis is cut at the sorted, unique endpoints of every non-empty region of at most
//                   DIV_EXACT_MAX sites; run_divergence gives the u64 diff / cnt of the pieces between cuts, a chunk of
//                   pieces at a time (fused / two-pass decided once for the whole piece list)
//   k_region_scan_* running u64 prefix sums over the pieces, per pair: group totals, an exclusive scan of the groups
//                   that carries across chunks, the prefix inside every group
//   k_region_gather region w = pre[cut of hi_w] - pre[cut of lo_w], added as the chunks holding its cuts pass (u64
//                   arithmetic modulo 2^64, exact for the final non-negative sums)
//   k_region_finalize_pairs   D = diff / (2.0 * cnt), k_finalize_pairs' expression
//   k_region_methsum, k_region_p0uu   k_finalize_samples' sequential meth_lvl sum per (region, sample) and k_p0uu
//   long regions    (more than DIV_EXACT_MAX sites, e.g. whole chromosomes) run_divergence on {lo, hi} alone, which keeps
//                   the long-window path's own blocked summation tree
#include <algorithm>
#include <cstring>
#include <map>
#include <string>
#include <thread>

#include "abfit_internal.h"

namespace abfit {

constexpr int REG_GROUP = 32;     // pieces per group of the prefix scan
constexpr int REG_FIN_WARPS = 4;  // warps per block of k_region_methsum

// per (group, pair): the u64 sums of the group's pieces
__global__ void k_region_scan_groups(const unsigned long long *__restrict__ diff, const unsigned long long *__restrict__ cnt,
                                     int64_t C, int64_t P, unsigned long long *__restrict__ gd, unsigned long long *__restrict__ gc)
{
    const int64_t ng = (C + REG_GROUP - 1) / REG_GROUP;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ng * P) return;
    const int64_t g = i / P, p = i - g * P, j1 = min(C, (g + 1) * REG_GROUP);
    unsigned long long d = 0, c = 0;
    for (int64_t j = g * REG_GROUP; j < j1; ++j) {
        d += diff[j * P + p];
        c += cnt[j * P + p];
    }
    gd[i] = d;
    gc[i] = c;
}

// per pair: exclusive scan of the group sums, starting from the sums of the earlier chunks (carry), which it advances
__global__ void k_region_scan_carry(unsigned long long *__restrict__ gd, unsigned long long *__restrict__ gc, int64_t ng,
                                    int64_t P, unsigned long long *__restrict__ carry_d, unsigned long long *__restrict__ carry_c)
{
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    unsigned long long d = carry_d[p], c = carry_c[p];
    for (int64_t g = 0; g < ng; ++g) {
        const unsigned long long xd = gd[g * P + p], xc = gc[g * P + p];
        gd[g * P + p] = d;
        gc[g * P + p] = c;
        d += xd;
        c += xc;
    }
    carry_d[p] = d;
    carry_c[p] = c;
}

// in place: piece j of the chunk -> the running sum through piece j, i.e. the prefix at cut (first piece + j + 1)
__global__ void k_region_scan_apply(unsigned long long *__restrict__ diff, unsigned long long *__restrict__ cnt, int64_t C,
                                    int64_t P, const unsigned long long *__restrict__ gd, const unsigned long long *__restrict__ gc)
{
    const int64_t ng = (C + REG_GROUP - 1) / REG_GROUP;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ng * P) return;
    const int64_t g = i / P, p = i - g * P, j1 = min(C, (g + 1) * REG_GROUP);
    unsigned long long d = gd[i], c = gc[i];
    for (int64_t j = g * REG_GROUP; j < j1; ++j) {
        d += diff[j * P + p];
        c += cnt[j * P + p];
        diff[j * P + p] = d;
        cnt[j * P + p] = c;
    }
}

// per (edge, pair): region += prefix row hi_row - prefix row lo_row of this chunk; a region has one edge per chunk
__global__ void k_region_gather(const RegionEdge *__restrict__ edges, int64_t n_edges, int64_t P,
                                const unsigned long long *__restrict__ pre_d, const unsigned long long *__restrict__ pre_c,
                                unsigned long long *__restrict__ diff, unsigned long long *__restrict__ cnt)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_edges * P) return;
    const int64_t q = i / P, p = i - q * P;
    const RegionEdge e = edges[q];
    const size_t o = (size_t)e.region * P + p;
    unsigned long long d = diff[o], c = cnt[o];
    if (e.hi_row >= 0) {
        d += pre_d[(size_t)e.hi_row * P + p];
        c += pre_c[(size_t)e.hi_row * P + p];
    }
    if (e.lo_row >= 0) {
        d -= pre_d[(size_t)e.lo_row * P + p];
        c -= pre_c[(size_t)e.lo_row * P + p];
    }
    diff[o] = d;
    cnt[o] = c;
}

// k_finalize_pairs' expression (src/pedigree.rs:257, 0/0 -> NaN)
__global__ void k_region_finalize_pairs(const unsigned long long *__restrict__ diff, const unsigned long long *__restrict__ cnt,
                                        int64_t n, double *__restrict__ D)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) D[i] = (double)diff[i] / (2.0 * (double)cnt[i]);
}

// per (region, sample) of a region of at most DIV_EXACT_MAX sites: k_finalize_samples' sequential pass, operation for
// operation (32 sites at a time, +0.0 for a filtered or out-of-range site, every lane adding the 32 values in site order)
__global__ void __launch_bounds__(32 * REG_FIN_WARPS)
k_region_methsum(const double *__restrict__ post, const double *__restrict__ meth, int64_t L, const int64_t *__restrict__ lo,
                 const int64_t *__restrict__ hi, int W, int S, double thr, double *__restrict__ methsum,
                 long long *__restrict__ nvalid)
{
    __shared__ __align__(16) double xch[REG_FIN_WARPS][2][32];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long idx = (long long)blockIdx.x * REG_FIN_WARPS + wib;
    if (idx >= (long long)W * S) return;  // whole warps leave together
    const int w = (int)(idx / S), s = (int)(idx - (long long)w * S);
    const int64_t a = lo[w], b = hi[w];
    if (b - a > DIV_EXACT_MAX) return;  // long regions: run_divergence on the region alone
    double acc = 0.0;
    long long nv = 0;
    const double *po = post + (size_t)s * L, *me = meth + (size_t)s * L;
    int buf = 0;
    for (int64_t i0 = a; i0 < b; i0 += 32, buf ^= 1) {
        const int64_t i = i0 + lane;
        const bool valid = i < b && po[i] >= thr;
        const double m = valid ? me[i] : 0.0;
        nv += __popc(__ballot_sync(FULL, valid));
        xch[wib][buf][lane] = m;
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 32; q += 2) {
            const double2 v = *reinterpret_cast<const double2 *>(&xch[wib][buf][q]);
            acc += v.x;
            acc += v.y;
        }
    }
    if (lane == 0) {
        methsum[idx] = acc;
        nvalid[idx] = nv;
    }
}

// k_p0uu: mean over samples of (1 - methsum / nvalid), summed in sample order
__global__ void k_region_p0uu(const double *__restrict__ methsum, const long long *__restrict__ nvalid,
                              const int64_t *__restrict__ lo, const int64_t *__restrict__ hi, int W, int S,
                              double *__restrict__ p0uu)
{
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W || hi[w] - lo[w] > DIV_EXACT_MAX) return;
    double acc = 0.0;
    for (int s = 0; s < S; ++s) {
        const double rc = methsum[(size_t)w * S + s] / (double)nvalid[(size_t)w * S + s];
        acc += 1.0 - rc;
    }
    p0uu[w] = acc / (double)S;
}

int plan_regions(int S, int64_t L, const int64_t *lo, const int64_t *hi, int W, RegionPlan &plan)
{
    plan = RegionPlan();
    const int64_t P = (int64_t)S * (S - 1) / 2;
    for (int w = 0; w < W; ++w) {
        const int64_t len = hi[w] - lo[w];
        if (len > DIV_EXACT_MAX) plan.longs.push_back(w);
        else if (len > 0 && P > 0) {
            plan.cuts.push_back(lo[w]);
            plan.cuts.push_back(hi[w]);
        }
    }
    std::sort(plan.cuts.begin(), plan.cuts.end());
    plan.cuts.erase(std::unique(plan.cuts.begin(), plan.cuts.end()), plan.cuts.end());
    const int64_t K = plan.cuts.empty() ? 0 : (int64_t)plan.cuts.size() - 1;  // pieces
    // pieces per chunk: about 1 GiB of per-piece sums (diff, cnt and the D the divergence path writes)
    plan.chunk = std::max<int64_t>(1, std::min<int64_t>(std::max<int64_t>(K, 1), ((int64_t)1 << 30) / std::max<int64_t>(P * 24, 1)));
    const int64_t n_chunks = K ? (K + plan.chunk - 1) / plan.chunk : 0;
    plan.edges.assign((size_t)n_chunks, {});
    if (K) {
        auto cut_of = [&](int64_t x) {
            return (int64_t)(std::lower_bound(plan.cuts.begin(), plan.cuts.end(), x) - plan.cuts.begin());
        };
        for (int w = 0; w < W; ++w) {
            const int64_t len = hi[w] - lo[w];
            if (len <= 0 || len > DIV_EXACT_MAX) continue;
            // prefix at cut k >= 1 is row (k - 1) % chunk of chunk (k - 1) / chunk; the prefix at cut 0 is zero
            const int64_t a = cut_of(lo[w]), b = cut_of(hi[w]);
            const int64_t cb = (b - 1) / plan.chunk;
            RegionEdge eb{w, -1, (int32_t)((b - 1) % plan.chunk), 0};
            if (a >= 1) {
                const int64_t ca = (a - 1) / plan.chunk;
                const int32_t ra = (int32_t)((a - 1) % plan.chunk);
                if (ca == cb) eb.lo_row = ra;
                else plan.edges[(size_t)ca].push_back(RegionEdge{w, ra, -1, 0});
            }
            plan.edges[(size_t)cb].push_back(eb);
        }
    }
    for (auto &e : plan.edges) plan.max_edges = std::max(plan.max_edges, e.size());
    // scratch: the chunk's outputs of the divergence path, the scan's group sums and carries, the edge list, the
    // divergence path's bit-planes (a piece takes at least one 64-site word) and per-super-block partials, region bounds
    const int64_t C = K ? plan.chunk : 0, ng = (C + REG_GROUP - 1) / REG_GROUP;
    const size_t words = (size_t)(L / 64 + 2 * C + 2);
    plan.bytes = (size_t)C * (P * 24 + S * 16) + (size_t)ng * P * 16 + (size_t)P * 16 + plan.max_edges * sizeof(RegionEdge) +
                 (size_t)S * words * 24 + (size_t)S * (words / 64 + C + 2) * 16 + (size_t)W * 16 + ((size_t)64 << 20);
    return 0;
}

namespace {
// device allocation freed on every way out
template <class T>
struct Mem {
    T *p = nullptr;
    ~Mem()
    {
        if (p) cudaFree(p);
    }
    int alloc(size_t n)
    {
        ABFIT_CUDA(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)));
        return 0;
    }
};
unsigned grid_of(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }
}  // namespace

int run_region_divergence(cudaStream_t st, DivArena *arena, const RegionPlan &plan, const uint8_t *d_status,
                          const double *d_post, const double *d_meth, int S, int64_t L, const int64_t *h_lo,
                          const int64_t *h_hi, int W, double thr, double *d_D, unsigned long long *d_diff,
                          unsigned long long *d_cnt, double *d_methsum, long long *d_nvalid, double *d_p0uu, int *launches)
{
    const int64_t P = (int64_t)S * (S - 1) / 2;
    const int64_t K = plan.cuts.empty() ? 0 : (int64_t)plan.cuts.size() - 1;
    *launches = 0;
    Mem<int64_t> d_lo, d_hi;
    if (int rc = d_lo.alloc(W)) return rc;
    if (int rc = d_hi.alloc(W)) return rc;
    ABFIT_CUDA(cudaMemcpyAsync(d_lo.p, h_lo, (size_t)W * 8, cudaMemcpyHostToDevice, st));
    ABFIT_CUDA(cudaMemcpyAsync(d_hi.p, h_hi, (size_t)W * 8, cudaMemcpyHostToDevice, st));
    if (P > 0) {
        ABFIT_CUDA(cudaMemsetAsync(d_diff, 0, (size_t)W * P * 8, st));
        ABFIT_CUDA(cudaMemsetAsync(d_cnt, 0, (size_t)W * P * 8, st));
    }
    if (P > 0 && K > 0) {
        const int64_t C = plan.chunk, ng = (C + REG_GROUP - 1) / REG_GROUP;
        Mem<double> t_D, t_ms;
        Mem<unsigned long long> t_diff, t_cnt, g_d, g_c, carry;
        Mem<long long> t_nv;
        Mem<RegionEdge> d_edges;
        if (int rc = t_D.alloc((size_t)C * P)) return rc;
        if (int rc = t_diff.alloc((size_t)C * P)) return rc;
        if (int rc = t_cnt.alloc((size_t)C * P)) return rc;
        if (int rc = t_ms.alloc((size_t)C * S)) return rc;
        if (int rc = t_nv.alloc((size_t)C * S)) return rc;
        if (int rc = g_d.alloc((size_t)ng * P)) return rc;
        if (int rc = g_c.alloc((size_t)ng * P)) return rc;
        if (int rc = carry.alloc((size_t)2 * P)) return rc;
        if (int rc = d_edges.alloc(plan.max_edges)) return rc;
        ABFIT_CUDA(cudaMemsetAsync(carry.p, 0, (size_t)2 * P * 8, st));
        // the fused / two-pass choice is made once for the whole piece list, as one abfit_divergence call would
        const int long_windows = div_long_windows(plan.cuts.data(), (int)std::min<int64_t>(K, INT32_MAX)) ? 1 : 0;
        for (int64_t k0 = 0, c = 0; k0 < K; k0 += C, ++c) {
            const int Wc = (int)std::min<int64_t>(C, K - k0);
            int l = 0;
            if (int rc = run_divergence(st, d_status, d_post, d_meth, S, L, plan.cuts.data() + k0, Wc, thr, t_D.p, t_diff.p,
                                        t_cnt.p, t_ms.p, t_nv.p, nullptr, &l, nullptr, arena, long_windows))
                return rc;
            *launches += l;
            const int64_t ngc = (Wc + REG_GROUP - 1) / REG_GROUP;
            k_region_scan_groups<<<grid_of(ngc * P, 256), 256, 0, st>>>(t_diff.p, t_cnt.p, Wc, P, g_d.p, g_c.p);
            ABFIT_CUDA(cudaGetLastError());
            k_region_scan_carry<<<grid_of(P, 128), 128, 0, st>>>(g_d.p, g_c.p, ngc, P, carry.p, carry.p + P);
            ABFIT_CUDA(cudaGetLastError());
            k_region_scan_apply<<<grid_of(ngc * P, 256), 256, 0, st>>>(t_diff.p, t_cnt.p, Wc, P, g_d.p, g_c.p);
            ABFIT_CUDA(cudaGetLastError());
            *launches += 3;
            const std::vector<RegionEdge> &e = plan.edges[(size_t)c];
            if (!e.empty()) {
                ABFIT_CUDA(cudaMemcpyAsync(d_edges.p, e.data(), e.size() * sizeof(RegionEdge), cudaMemcpyHostToDevice, st));
                k_region_gather<<<grid_of((int64_t)e.size() * P, 256), 256, 0, st>>>(d_edges.p, (int64_t)e.size(), P, t_diff.p,
                                                                                     t_cnt.p, d_diff, d_cnt);
                ABFIT_CUDA(cudaGetLastError());
                ++*launches;
            }
        }
        ABFIT_CUDA(cudaStreamSynchronize(st));  // the temporaries are freed at the end of this scope
    }
    if (P > 0) {
        k_region_finalize_pairs<<<grid_of((int64_t)W * P, 256), 256, 0, st>>>(d_diff, d_cnt, (int64_t)W * P, d_D);
        ABFIT_CUDA(cudaGetLastError());
        ++*launches;
    }
    k_region_methsum<<<grid_of((int64_t)W * S, REG_FIN_WARPS), 32 * REG_FIN_WARPS, 0, st>>>(d_post, d_meth, L, d_lo.p, d_hi.p, W, S,
                                                                                           thr, d_methsum, d_nvalid);
    ABFIT_CUDA(cudaGetLastError());
    k_region_p0uu<<<grid_of(W, 128), 128, 0, st>>>(d_methsum, d_nvalid, d_lo.p, d_hi.p, W, S, d_p0uu);
    ABFIT_CUDA(cudaGetLastError());
    *launches += 2;
    // regions of more than DIV_EXACT_MAX sites: the single-window call itself, written into the region's rows
    for (const int32_t w : plan.longs) {
        const int64_t seg[2] = {h_lo[w], h_hi[w]};
        int l = 0;
        if (int rc = run_divergence(st, d_status, d_post, d_meth, S, L, seg, 1, thr, d_D + (size_t)w * P, d_diff + (size_t)w * P,
                                    d_cnt + (size_t)w * P, d_methsum + (size_t)w * S, d_nvalid + (size_t)w * S, d_p0uu + w, &l,
                                    nullptr, arena, -1))
            return rc;
        *launches += l;
    }
    ABFIT_CUDA(cudaStreamSynchronize(st));
    return 0;
}

}  // namespace abfit

// ---------------------------------------------------------------------------------------
// host: BED lines and site ranges
// ---------------------------------------------------------------------------------------
using namespace abfit;

static unsigned region_threads()
{
    unsigned hw = std::thread::hardware_concurrency();
    if (const char *e = getenv("ABFIT_HOST_THREADS")) hw = (unsigned)std::max(1, atoi(e));
    return hw ? hw : 1;
}

extern "C" {

int abfit_parse_region_line(const char *line, int32_t *chrom_out, int64_t *start0_out, int64_t *end_out)
{
    if (!line || !chrom_out || !start0_out || !end_out) return ABFIT_ERR_ARG;
    std::string_view s(line);
    while (!s.empty() && (s.back() == '\n' || s.back() == '\r')) s.remove_suffix(1);
    std::vector<std::string_view> f;
    for (size_t i = 0; i < s.size();) {  // fields: runs of anything but blanks and tabs
        while (i < s.size() && (s[i] == ' ' || s[i] == '\t')) ++i;
        const size_t b = i;
        while (i < s.size() && s[i] != ' ' && s[i] != '\t') ++i;
        if (i > b) f.push_back(s.substr(b, i - b));
    }
    if (f.empty() || f[0][0] == '#' || f[0] == "track" || f[0] == "browser") return 1;
    if (f.size() < 3) {
        set_error("region line: fewer than three columns: " + std::string(s));
        return ABFIT_ERR_ARG;
    }
    int32_t c = 0;
    uint32_t a = 0, b = 0;
    if (!parse_chromosome_name(f[0], c)) {
        set_error("region line: not a chromosome name: " + std::string(f[0]));
        return ABFIT_ERR_ARG;
    }
    if (!parse_u32_field(f[1], a) || !parse_u32_field(f[2], b)) {
        set_error("region line: start and end must be integers in [0, 2^32): " + std::string(s));
        return ABFIT_ERR_ARG;
    }
    if (b < a) {
        set_error("region line: end < start: " + std::string(s));
        return ABFIT_ERR_ARG;
    }
    *chrom_out = c;
    *start0_out = a;
    *end_out = b;
    return 0;
}

int abfit_region_ranges(const abfit_cg_site *sites, int64_t n_sites, const int32_t *chrom, const int64_t *start0,
                        const int64_t *end, int32_t W, int64_t *lo_out, int64_t *hi_out)
{
    if ((!sites && n_sites > 0) || n_sites < 0 || W < 0 || (W > 0 && (!chrom || !start0 || !end || !lo_out || !hi_out))) {
        set_error("region ranges: missing or out-of-range argument");
        return ABFIT_ERR_ARG;
    }
    // every chromosome one run of sites, positions non-decreasing inside it
    std::map<int32_t, std::pair<int64_t, int64_t>> runs;
    for (int64_t i = 0; i < n_sites;) {
        int64_t j = i + 1;
        while (j < n_sites && sites[j].chromosome == sites[i].chromosome) {
            if (sites[j].start < sites[j - 1].start) {
                set_error("region ranges: positions decrease on chromosome " + std::to_string(sites[i].chromosome) + " at site " +
                          std::to_string(j));
                return ABFIT_ERR_ARG;
            }
            ++j;
        }
        if (!runs.emplace(sites[i].chromosome, std::make_pair(i, j)).second) {
            set_error("region ranges: chromosome " + std::to_string(sites[i].chromosome) + " appears again at site " +
                      std::to_string(i) + " after another chromosome; the sites must be grouped by chromosome");
            return ABFIT_ERR_ARG;
        }
        i = j;
    }
    for (int32_t w = 0; w < W; ++w)
        if (end[w] < start0[w]) {
            set_error("region ranges: region " + std::to_string(w) + " has end < start");
            return ABFIT_ERR_ARG;
        }
    // site positions start0 + 1 .. end (1-based) of the region's chromosome: the first site past start0 and past end
    auto range = [&](int32_t w) {
        const auto it = runs.find(chrom[w]);
        if (it == runs.end()) {
            lo_out[w] = hi_out[w] = 0;
            return;
        }
        const abfit_cg_site *b = sites + it->second.first, *e = sites + it->second.second;
        auto past = [&](int64_t x) {
            return (int64_t)(std::upper_bound(b, e, x, [](int64_t v, const abfit_cg_site &q) { return v < (int64_t)q.start; }) - sites);
        };
        lo_out[w] = past(start0[w]);
        hi_out[w] = past(end[w]);
    };
    const unsigned nt = std::min<unsigned>(region_threads(), (unsigned)std::max(1, W / 16384));
    if (nt <= 1) {
        for (int32_t w = 0; w < W; ++w) range(w);
    } else {
        std::vector<std::thread> th;
        for (unsigned t = 0; t < nt; ++t)
            th.emplace_back([&, t]() {
                for (int32_t w = (int32_t)((int64_t)W * t / nt); w < (int32_t)((int64_t)W * (t + 1) / nt); ++w) range(w);
            });
        for (auto &x : th) x.join();
    }
    return 0;
}

}  // extern "C"
