// abfit_inputs.cu — the input side of `alphabeta` (host): nodelist / edgelist / methylome parsing and
// the pedigree builder, restated from the reference so that real files can be fed end to end
// (SURVEY.md §8f rank 2).  The O(S^2 L) part — the observed pairwise divergence — runs on the GPU
// (abfit_divergence); everything here is O(input) text handling and a shortest-path search on a graph
// of a few hundred nodes.
//
//   MethylationSite::from_methylome_file_line   src/methylation_site.rs:146-362
//   Chromosome::try_from                        src/methylation_site.rs:57-68
//   Pedigree::build                             src/pedigree.rs:92-193
//   DMatrix::convert (shortest path, t0 rule)   src/pedigree.rs:264-337
#include <atomic>
#include <charconv>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <memory>
#include <queue>
#include <sstream>
#include <string>
#include <string_view>
#include <thread>
#include <vector>

#include "abfit_internal.h"

namespace {

std::vector<std::string> split_any(const std::string &s, const char *seps)
{
    std::vector<std::string> out;
    std::string cur;
    for (char ch : s) {
        if (std::strchr(seps, ch)) {
            out.push_back(cur);
            cur.clear();
        } else {
            cur += ch;
        }
    }
    out.push_back(cur);
    return out;
}

// <u32 as FromStr>: optional '+', ASCII digits, no overflow
bool parse_u32(std::string_view s, uint32_t &v)
{
    size_t i = (!s.empty() && s[0] == '+') ? 1 : 0;
    if (i >= s.size()) return false;
    uint64_t acc = 0;
    for (; i < s.size(); ++i) {
        if (s[i] < '0' || s[i] > '9') return false;
        acc = acc * 10 + (uint64_t)(s[i] - '0');
        if (acc > 0xFFFFFFFFull) return false;
    }
    v = (uint32_t)acc;
    return true;
}

inline bool is_digit(char c) { return c >= '0' && c <= '9'; }
inline bool word_is(std::string_view s, const char *w)  // ASCII case-insensitive
{
    size_t k = 0;
    for (; k < s.size() && w[k]; ++k)
        if ((char)(s[k] | 0x20) != w[k]) return false;
    return k == s.size() && !w[k];
}

// <f64 as FromStr>: [+-] (digits [. digits] | . digits) [e[+-]digits] | inf | infinity | nan  (case-insensitive words).
// The grammar is checked here; the value comes from std::from_chars (correctly rounded, like Rust's and glibc's
// strtod), with strtod as the fallback for what from_chars reports as out of range (Rust: inf / 0 / subnormal).
bool parse_f64(std::string_view s, double &v)
{
    size_t i = 0;
    bool neg = false;
    if (i < s.size() && (s[i] == '+' || s[i] == '-')) neg = s[i] == '-', ++i;
    const std::string_view w = s.substr(i);
    if (word_is(w, "inf") || word_is(w, "infinity")) {
        v = neg ? -HUGE_VAL : HUGE_VAL;
        return true;
    }
    if (word_is(w, "nan")) {
        v = std::strtod(neg ? "-nan" : "nan", nullptr);
        return true;
    }
    const size_t num0 = i;
    size_t nd = 0;
    while (i < s.size() && is_digit(s[i])) ++i, ++nd;
    if (i < s.size() && s[i] == '.') {
        ++i;
        while (i < s.size() && is_digit(s[i])) ++i, ++nd;
    }
    if (nd == 0) return false;
    if (i < s.size() && (s[i] == 'e' || s[i] == 'E')) {
        ++i;
        if (i < s.size() && (s[i] == '+' || s[i] == '-')) ++i;
        size_t ne = 0;
        while (i < s.size() && is_digit(s[i])) ++i, ++ne;
        if (ne == 0) return false;
    }
    if (i != s.size()) return false;
    double mag;
    const auto r = std::from_chars(s.data() + num0, s.data() + s.size(), mag);
    if (r.ec == std::errc() && r.ptr == s.data() + s.size()) {
        v = neg ? -mag : mag;
        return true;
    }
    const std::string z(s);
    v = std::strtod(z.c_str(), nullptr);
    return true;
}

// Chromosome::try_from: Numbered(n) -> n, Mitochondrial -> 256, Chloroplast -> 257
bool parse_chromosome(std::string_view s, int32_t &c)
{
    while (s.substr(0, 3) == "chr") s.remove_prefix(3);  // trim_start_matches("chr")
    if (s == "M") { c = 256; return true; }
    if (s == "C") { c = 257; return true; }
    uint32_t v;
    if (!parse_u32(s, v) || v > 255) return false;
    c = (int32_t)v;
    return true;
}

struct Site {
    int32_t chromosome;
    uint32_t start, end;
    int32_t strand;
    double posteriormax, meth_lvl;
    uint8_t status;
};

uint8_t status_of(char c) { return c == 'M' ? 2 : c == 'I' ? 1 : 0; }  // anything else parses as U (with a warning)

typedef std::string_view SV;
bool cg_fields(const SV *f, size_t i_chr, SV start, const SV *end, size_t i_strand, size_t i_cm, size_t i_ct, size_t i_post,
               size_t i_status, size_t i_lvl, bool invert, Site &o)
{
    uint32_t cm, ct;
    if (!parse_chromosome(f[i_chr], o.chromosome)) return false;
    if (!parse_u32(start, o.start)) return false;
    if (end) {
        if (!parse_u32(*end, o.end)) return false;
    } else {
        o.end = o.start + 1;
    }
    o.strand = ((f[i_strand] == "+") ^ invert) ? 1 : -1;
    if (!parse_u32(f[i_cm], cm) || !parse_u32(f[i_ct], ct)) return false;
    if (!parse_f64(f[i_post], o.posteriormax)) return false;
    if (f[i_status].empty()) return false;
    o.status = status_of(f[i_status][0]);
    if (!parse_f64(f[i_lvl], o.meth_lvl)) return false;
    return true;
}

// splits like str::split: n separators -> n + 1 fields; the first `cap` fields are stored, all are counted
template <class IsSep>
inline int split_view(SV line, IsSep is_sep, SV *out, int cap)
{
    int n = 0;
    size_t b = 0;
    for (size_t i = 0; i <= line.size(); ++i)
        if (i == line.size() || is_sep(line[i])) {
            if (n < cap) out[n] = line.substr(b, i - b);
            ++n;
            b = i + 1;
        }
    return n;
}

// the six formats, tried in the reference's order; 4-field lines all end in the chromatin-state reading.
// No allocation per line: the methylome files of one run hold 10^8-10^9 lines.
bool parse_methylome_line(SV line, bool invert, Site &o)
{
    SV f[12];
    const int nf = split_view(line, [](char c) { return c == '\t'; }, f, 12);
    if (nf == 9 && f[3] == "CG" && cg_fields(f, 0, f[1], nullptr, 2, 4, 5, 6, 7, 8, invert, o)) return true;
    if (nf == 10 && f[3] == "CG" && cg_fields(f, 0, f[1], nullptr, 2, 4, 5, 6, 7, 8, invert, o)) return true;
    if (nf == 11 && f[3] == "CG" && cg_fields(f, 0, f[1], &f[2], 5, 6, 7, 8, 9, 10, invert, o)) return true;
    SV g[4];
    if (split_view(line, [](char c) { return c == '\t' || c == ' '; }, g, 4) == 4) {
        if (parse_chromosome(g[0], o.chromosome) && parse_u32(g[1], o.start) && parse_u32(g[2], o.end)) {
            o.strand = 0;
            o.posteriormax = 0.0;
            o.meth_lvl = 0.0;
            o.status = 0;
            return true;
        }
    }
    return false;
}

// One chunk of a file image, lines split like BufRead::lines ('\n'; one trailing '\r' stripped).
struct ParsedChunk {
    std::vector<abfit_cg_site> sites;
    std::vector<double> post, lvl;
    std::vector<uint8_t> status;
    std::vector<int64_t> off;
    std::vector<int32_t> len;
};
void parse_chunk(const char *buf, int64_t lo, int64_t hi, bool invert, bool want_lines, ParsedChunk &out)
{
    Site s;
    int64_t b = lo;
    while (b < hi) {
        const char *nl = static_cast<const char *>(std::memchr(buf + b, '\n', (size_t)(hi - b)));
        const int64_t e = nl ? (int64_t)(nl - buf) : hi;
        int64_t n = e - b;
        if (n > 0 && buf[b + n - 1] == '\r') --n;
        if (parse_methylome_line(SV(buf + b, (size_t)n), invert, s)) {
            out.sites.push_back(abfit_cg_site{s.chromosome, s.start, s.end, s.strand});
            out.post.push_back(s.posteriormax);
            out.lvl.push_back(s.meth_lvl);
            out.status.push_back(s.status);
            if (want_lines) {
                out.off.push_back(b);
                out.len.push_back((int32_t)n);
            }
        }
        b = e + 1;
    }
}

bool read_file(const char *path, std::string &out)
{
    FILE *f = std::fopen(path, "rb");
    if (!f) return false;
    out.clear();
    char buf[1 << 16];
    size_t n;
    while ((n = std::fread(buf, 1, sizeof buf, f)) > 0) out.append(buf, n);
    std::fclose(f);
    return true;
}

typedef abfit::ListNode Node;


// nodelist + edgelist -> measured nodes and, for every pair of them connected in the pedigree graph, (i, j, t0, t1, t2)
struct PedGraph {
    std::vector<Node> meas;
    struct Pair {
        int i, j;
        double t0, t1, t2;
    };
    std::vector<Pair> pairs;
};

}  // namespace

bool abfit::parse_chromosome_name(std::string_view s, int32_t &c) { return parse_chromosome(s, c); }
bool abfit::parse_u32_field(std::string_view s, uint32_t &v) { return parse_u32(s, v); }

// nodes: split on \n and \r, skip the header, id = index after the header (src/pedigree.rs:99-116); edges: the first
// two fields of every line after the header (src/pedigree.rs:123-135), names not yet resolved
int abfit::read_node_edge_lists(const char *nodelist_path, const char *edgelist_path, std::vector<ListNode> &nodes,
                                std::vector<std::pair<std::string, std::string>> &edges)
{
    std::string ntext, etext;
    if (!read_file(nodelist_path, ntext) || !read_file(edgelist_path, etext)) {
        abfit::set_error("cannot read the nodelist or the edgelist");
        return ABFIT_ERR_ARG;
    }
    {
        const std::vector<std::string> lines = split_any(ntext, "\n\r");
        for (size_t li = 1; li < lines.size(); ++li) {
            const std::vector<std::string> e = split_any(lines[li], ",\t ");
            uint32_t gen;
            if (e.size() < 4 || !parse_u32(e[2], gen)) continue;
            nodes.push_back(ListNode{li - 1, e[0], e[1], gen, e[3] == "Y"});
        }
    }
    if (nodes.empty()) {
        abfit::set_error("No nodes could be parsed from the nodelist");
        return ABFIT_ERR_ARG;
    }
    {
        const std::vector<std::string> lines = split_any(etext, "\n\r");
        for (size_t li = 1; li < lines.size(); ++li) {
            const std::vector<std::string> e = split_any(lines[li], "\t ,");
            if (e.size() >= 2) edges.emplace_back(e[0], e[1]);
        }
    }
    return 0;
}

namespace {

int build_graph(const char *nodelist_path, const char *edgelist_path, PedGraph &g)
{
    std::vector<Node> nodes;
    std::vector<std::pair<std::string, std::string>> names;
    if (int rc = abfit::read_node_edge_lists(nodelist_path, edgelist_path, nodes, names)) return rc;
    struct Edge {
        const Node *from, *to;
    };
    std::vector<Edge> edges;  // src/pedigree.rs:123-135: edges naming an unknown node are dropped
    for (auto &e : names) {
        const Node *a = nullptr, *b = nullptr;
        for (auto &n : nodes)
            if (!a && n.name == e.first) a = &n;
        for (auto &n : nodes)
            if (!b && n.name == e.second) b = &n;
        if (a && b) edges.push_back(Edge{a, b});
    }
    for (auto &n : nodes)
        if (n.meth) g.meas.push_back(n);
    const int S = (int)g.meas.size();
    // DMatrix::convert: undirected graph, edge weight |generation difference|, shortest path, t0 = smallest
    // generation on the path (src/pedigree.rs:264-337).  petgraph's astar with a zero heuristic is Dijkstra;
    // pedigrees are trees, so the path is unique.
    std::map<size_t, std::vector<std::pair<size_t, uint64_t>>> adj;
    std::map<size_t, uint32_t> gen_of;
    for (auto &e : edges) {
        const uint64_t w = e.from->generation > e.to->generation ? e.from->generation - e.to->generation
                                                                 : e.to->generation - e.from->generation;
        adj[e.from->id].push_back({e.to->id, w});
        adj[e.to->id].push_back({e.from->id, w});
        gen_of.emplace(e.from->id, e.from->generation);
        gen_of.emplace(e.to->id, e.to->generation);
    }
    for (int i = 0; i < S; ++i)
        for (int j = i + 1; j < S; ++j) {
            const size_t src = g.meas[i].id, dst = g.meas[j].id;
            if (!adj.count(src)) continue;
            std::map<size_t, uint64_t> dist;
            std::map<size_t, size_t> prev;
            typedef std::pair<uint64_t, size_t> QE;
            std::priority_queue<QE, std::vector<QE>, std::greater<QE>> pq;
            dist[src] = 0;
            pq.push({0, src});
            bool found = false;
            while (!pq.empty()) {
                const QE top = pq.top();
                pq.pop();
                if (top.second == dst) {
                    found = true;
                    break;
                }
                if (top.first > dist[top.second]) continue;
                for (auto &nb : adj[top.second]) {
                    const uint64_t nd = top.first + nb.second;
                    auto it = dist.find(nb.first);
                    if (it == dist.end() || nd < it->second) {
                        dist[nb.first] = nd;
                        prev[nb.first] = top.second;
                        pq.push({nd, nb.first});
                    }
                }
            }
            if (!found) continue;
            uint32_t t0 = gen_of[dst];
            for (size_t u = dst;;) {
                t0 = std::min(t0, gen_of[u]);
                auto it = prev.find(u);
                if (u == src || it == prev.end()) break;
                u = it->second;
            }
            const double t1 = (double)g.meas[i].generation, t2 = (double)g.meas[j].generation;
            if ((double)dist[dst] != t1 - (double)t0 + t2 - (double)t0) {
                abfit::set_error("pedigree graph: path length does not match the generation times (the reference asserts here)");
                return ABFIT_ERR_ARG;
            }
            g.pairs.push_back(PedGraph::Pair{i, j, (double)t0, t1, t2});
        }
    return 0;
}

}  // namespace

struct abfit_pedigree {
    std::vector<double> rows;  // [n_pairs][4]
    double p0uu = 0.0;
    int32_t n_samples = 0;
    int64_t n_sites = 0;
    std::string warnings;
};

extern "C" {

int abfit_parse_methylome_line(const char *line, int32_t invert_strand, abfit_cg_site *site_out, double *posterior_max_out,
                               int32_t *status_out, double *meth_lvl_out)
{
    if (!line) return ABFIT_ERR_ARG;
    Site s;
    if (!parse_methylome_line(line, invert_strand != 0, s)) return 1;  // not a site (header, other context, malformed)
    if (site_out) {
        site_out->chromosome = s.chromosome;
        site_out->start = s.start;
        site_out->end = s.end;
        site_out->strand = s.strand;
    }
    if (posterior_max_out) *posterior_max_out = s.posteriormax;
    if (status_out) *status_out = s.status;
    if (meth_lvl_out) *meth_lvl_out = s.meth_lvl;
    return 0;
}

static unsigned host_threads()
{
    unsigned hw = std::thread::hardware_concurrency();
    if (const char *e = getenv("ABFIT_HOST_THREADS")) hw = (unsigned)std::max(1, atoi(e));
    return hw ? hw : 1;
}

// max_threads: upper bound for this call (callers that already run one call per file on their own threads pass their share)
static int parse_buffer(const char *buf, int64_t len, int32_t invert_strand, int32_t skip_first_line, int64_t capacity,
                        abfit_cg_site *sites, double *posterior_max, uint8_t *status, double *meth_lvl, int64_t *line_off,
                        int32_t *line_len, int64_t *n_out, unsigned max_threads, std::string *err)
{
    if ((!buf && len > 0) || len < 0 || !n_out || capacity < 0) return ABFIT_ERR_ARG;
    *n_out = 0;
    int64_t lo = 0;
    if (skip_first_line) {
        const char *nl = len > 0 ? static_cast<const char *>(std::memchr(buf, '\n', (size_t)len)) : nullptr;
        lo = nl ? (int64_t)(nl - buf) + 1 : len;
    }
    // chunks of ~4 MB cut at line ends, parsed by up to 16 threads, concatenated in file order
    const int64_t body = len - lo;
    const int n_thr = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<unsigned>(std::max(1u, max_threads), 16u), body / (1 << 20)));
    const int n_chunks = n_thr == 1 ? 1 : (int)std::min<int64_t>(4096, std::max<int64_t>(n_thr, body / (4 << 20)));
    std::vector<int64_t> cut(n_chunks + 1, len);
    cut[0] = lo;
    for (int c = 1; c < n_chunks; ++c) {
        int64_t at = std::max(cut[c - 1], lo + body * c / n_chunks);
        const char *nl = at < len ? static_cast<const char *>(std::memchr(buf + at, '\n', (size_t)(len - at))) : nullptr;
        cut[c] = nl ? (int64_t)(nl - buf) + 1 : len;
    }
    const bool want_lines = line_off || line_len;
    std::vector<ParsedChunk> parts(n_chunks);
    if (n_thr == 1) {
        for (int c = 0; c < n_chunks; ++c) parse_chunk(buf, cut[c], cut[c + 1], invert_strand != 0, want_lines, parts[c]);
    } else {
        std::atomic<int> next{0};
        std::vector<std::thread> th;
        for (int t = 0; t < n_thr; ++t)
            th.emplace_back([&]() {
                for (int c; (c = next.fetch_add(1)) < n_chunks;)
                    parse_chunk(buf, cut[c], cut[c + 1], invert_strand != 0, want_lines, parts[c]);
            });
        for (auto &x : th) x.join();
    }
    int64_t total = 0;
    for (auto &pc : parts) total += (int64_t)pc.sites.size();
    *n_out = total;
    if (!sites && !posterior_max && !status && !meth_lvl && !want_lines) return ABFIT_OK;  // counting call
    if (total > capacity) {
        if (err) *err = "abfit_parse_methylome_buffer: " + std::to_string(total) + " sites, room for " + std::to_string(capacity);
        return ABFIT_ERR_ARG;
    }
    int64_t at = 0;
    for (auto &pc : parts) {
        const size_t n = pc.sites.size();
        if (n == 0) continue;
        if (sites) std::memcpy(sites + at, pc.sites.data(), n * sizeof(abfit_cg_site));
        if (posterior_max) std::memcpy(posterior_max + at, pc.post.data(), n * sizeof(double));
        if (status) std::memcpy(status + at, pc.status.data(), n);
        if (meth_lvl) std::memcpy(meth_lvl + at, pc.lvl.data(), n * sizeof(double));
        if (line_off) std::memcpy(line_off + at, pc.off.data(), n * sizeof(int64_t));
        if (line_len) std::memcpy(line_len + at, pc.len.data(), n * sizeof(int32_t));
        at += (int64_t)n;
    }
    return ABFIT_OK;
}

int abfit_parse_methylome_buffer(const char *buf, int64_t len, int32_t invert_strand, int32_t skip_first_line, int64_t capacity,
                                 abfit_cg_site *sites, double *posterior_max, uint8_t *status, double *meth_lvl,
                                 int64_t *line_off, int32_t *line_len, int64_t *n_out)
{
    std::string err;
    const int rc = parse_buffer(buf, len, invert_strand, skip_first_line, capacity, sites, posterior_max, status, meth_lvl, line_off,
                                line_len, n_out, host_threads(), &err);
    if (rc && !err.empty()) abfit::set_error(err);
    return rc;
}

int abfit_pedigree_build(abfit_ctx *ctx, const char *nodelist_path, const char *edgelist_path, double posterior_max_filter,
                         abfit_pedigree **out)
{
    if (!ctx || !nodelist_path || !edgelist_path || !out) return ABFIT_ERR_ARG;
    *out = nullptr;
    PedGraph g;
    if (int rc = build_graph(nodelist_path, edgelist_path, g)) return rc;
    // measured nodes and their site tables (src/pedigree.rs:137-177); node.file is relative to the CWD
    const int S = (int)g.meas.size();
    std::vector<std::vector<uint8_t>> st(S);
    std::vector<std::vector<double>> po(S), me(S);
    // one file per host thread (the reference: rayon, src/pedigree.rs:137-157), the parser splits a file over the rest
    {
        const unsigned hw = host_threads();
        const unsigned outer = (unsigned)std::max(1, std::min<int>(std::min<int>(S, (int)hw), 16));
        const unsigned inner = std::max(1u, hw / outer);
        std::vector<std::string> errs(S);
        std::vector<int> rcs(S, 0);
        std::atomic<int> next{0};
        auto load = [&](int s) {
            std::string image;
            if (!read_file(g.meas[s].file.c_str(), image)) {
                errs[s] = "Could not open node file: " + g.meas[s].file;
                rcs[s] = ABFIT_ERR_ARG;
                return;
            }
            // every line that parses as a CG site, header row included in the attempt (BufRead::lines strips \r\n)
            int64_t cap = 1, n = 0;
            for (char ch : image) cap += ch == '\n';
            st[s].resize((size_t)cap);
            po[s].resize((size_t)cap);
            me[s].resize((size_t)cap);
            rcs[s] = parse_buffer(image.data(), (int64_t)image.size(), 0, 0, cap, nullptr, po[s].data(), st[s].data(), me[s].data(),
                                  nullptr, nullptr, &n, inner, &errs[s]);
            st[s].resize((size_t)n);
            po[s].resize((size_t)n);
            me[s].resize((size_t)n);
            // (cap counted every line of the file, CG or not: give the difference back before the next file is read)
            st[s].shrink_to_fit();
            po[s].shrink_to_fit();
            me[s].shrink_to_fit();
        };
        std::vector<std::thread> pool;
        for (unsigned t = 0; t < outer; ++t)
            pool.emplace_back([&]() {
                for (int s; (s = next.fetch_add(1)) < S;) load(s);
            });
        for (auto &th : pool) th.join();
        for (int s = 0; s < S; ++s)
            if (rcs[s]) {
                abfit::set_error(errs[s]);
                return rcs[s];
            }
    }
    std::unique_ptr<abfit_pedigree> ped(new abfit_pedigree());
    ped->n_samples = S;
    // observed divergence + per-sample methylation level on the GPU, one call per group of samples with equally long
    // site lists (pairs of unequal length get D = 0 with a warning, src/pedigree.rs:222-230)
    std::vector<double> Dfull((size_t)S * S, 0.0);  // [i][j] for i < j
    std::vector<double> rc(S, 0.0);
    std::map<size_t, std::vector<int>> by_len;
    for (int s = 0; s < S; ++s) by_len[st[s].size()].push_back(s);
    if (by_len.size() > 1) ped->warnings += "Lengths do not match, all bets are off: pairs of samples with different site counts get D = 0\n";
    for (auto &kv : by_len) {
        const std::vector<int> &grp = kv.second;
        const int G = (int)grp.size();
        const int64_t L = (int64_t)kv.first;
        ped->n_sites = std::max(ped->n_sites, L);
        // [G][L] staging of the three columns: written in full below (no zero-fill: 17 bytes per sample-site, 17 GB for 200
        // methylomes of 5 M sites), copied on the host threads, every sample's own table released as soon as it is copied
        const size_t GL = std::max<size_t>(1, (size_t)G * (size_t)L);
        std::unique_ptr<uint8_t[]> gs(new uint8_t[GL]);
        std::unique_ptr<double[]> gp(new double[GL]), gm(new double[GL]);
        {
            std::atomic<int> next{0};
            auto copy_rows = [&]() {
                for (int q; (q = next.fetch_add(1)) < G;) {
                    const int s = grp[q];
                    if (L > 0) {
                        std::memcpy(gs.get() + (size_t)q * L, st[s].data(), (size_t)L);
                        std::memcpy(gp.get() + (size_t)q * L, po[s].data(), (size_t)L * sizeof(double));
                        std::memcpy(gm.get() + (size_t)q * L, me[s].data(), (size_t)L * sizeof(double));
                    }
                    std::vector<uint8_t>().swap(st[s]);
                    std::vector<double>().swap(po[s]);
                    std::vector<double>().swap(me[s]);
                }
            };
            const int nt = std::max(1, std::min<int>(std::min<int>(G, (int)host_threads()), 16));
            std::vector<std::thread> pool;
            for (int t = 1; t < nt; ++t) pool.emplace_back(copy_rows);
            copy_rows();
            for (auto &th : pool) th.join();
        }
        const size_t P = (size_t)G * (G - 1) / 2;
        std::vector<double> D(std::max<size_t>(P, 1)), methsum(G);
        std::vector<int64_t> nvalid(G);
        if (int rc2 = abfit_divergence(ctx, gs.get(), gp.get(), gm.get(), G, L, nullptr, 1, posterior_max_filter, D.data(),
                                       nullptr, nullptr, nullptr, methsum.data(), nvalid.data()))
            return rc2;
        size_t p = 0;
        for (int a = 0; a < G; ++a) {
            rc[grp[a]] = methsum[a] / (double)nvalid[a];  // src/pedigree.rs:171-172 (0/0 = NaN)
            for (int b = a + 1; b < G; ++b) {
                const int i = std::min(grp[a], grp[b]), j = std::max(grp[a], grp[b]);
                Dfull[(size_t)i * S + j] = D[p++];
            }
        }
    }
    {
        double acc = 0.0;  // src/pedigree.rs:179-183
        for (int s = 0; s < S; ++s) acc += 1.0 - rc[s];
        ped->p0uu = acc / (double)S;
    }
    for (auto &pr : g.pairs) {
        ped->rows.push_back(pr.t0);
        ped->rows.push_back(pr.t1);
        ped->rows.push_back(pr.t2);
        ped->rows.push_back(Dfull[(size_t)pr.i * S + pr.j]);
    }
    *out = ped.release();
    return 0;
}

// The graph part alone (metaprofile: the same nodes and edges for every window, only D changes).
//   files_out: the measured nodes' file names, '\n'-separated, in nodelist order (caller-owned buffer of files_cap bytes)
//   pairs_out [n_pairs][5]: i, j (sample indices, i < j), t0, t1, t2 in pedigree row order; D of row r is D[pair index of (i, j)]
int abfit_pedigree_graph(const char *nodelist_path, const char *edgelist_path, int32_t *n_samples_out, char *files_out,
                         int32_t files_cap, int32_t *n_pairs_out, double *pairs_out, int32_t pairs_cap)
{
    if (!nodelist_path || !edgelist_path) return ABFIT_ERR_ARG;
    PedGraph g;
    if (int rc = build_graph(nodelist_path, edgelist_path, g)) return rc;
    if (n_samples_out) *n_samples_out = (int32_t)g.meas.size();
    if (n_pairs_out) *n_pairs_out = (int32_t)g.pairs.size();
    if (files_out) {
        std::string all;
        for (auto &n : g.meas) all += n.file + "\n";
        if ((int64_t)all.size() + 1 > (int64_t)files_cap) {
            abfit::set_error("abfit_pedigree_graph: files_out is too small for the measured nodes' file names");
            return ABFIT_ERR_ARG;
        }
        std::memcpy(files_out, all.c_str(), all.size() + 1);
    }
    if (pairs_out) {
        if ((int64_t)g.pairs.size() > (int64_t)pairs_cap) {
            abfit::set_error("abfit_pedigree_graph: pairs_out is too small (call with null outputs first for the counts)");
            return ABFIT_ERR_ARG;
        }
        for (size_t r = 0; r < g.pairs.size(); ++r) {
            pairs_out[5 * r + 0] = g.pairs[r].i;
            pairs_out[5 * r + 1] = g.pairs[r].j;
            pairs_out[5 * r + 2] = g.pairs[r].t0;
            pairs_out[5 * r + 3] = g.pairs[r].t1;
            pairs_out[5 * r + 4] = g.pairs[r].t2;
        }
    }
    return 0;
}

// Gene::from_annotation_file_line (src/genes.rs:166-216): `chr start end name annotation strand` or
// `chr start end width strand name`, separated by blanks or tabs.  0 = parsed, 1 = not a gene line.
int abfit_parse_annotation_line(const char *line, int32_t invert_strand, abfit_gene *gene_out)
{
    if (!line || !gene_out) return ABFIT_ERR_ARG;
    const std::vector<std::string> f = split_any(line, " \t");
    if (f.size() != 6) return 1;
    auto strand_of = [](const std::string &s) { return s == "+" ? 1 : s == "-" ? -1 : s == "*" ? 0 : 2; };
    int sd = strand_of(f[5]);
    if (sd == 2) sd = strand_of(f[4]);
    if (sd == 2) return 1;
    if (!parse_chromosome(f[0], gene_out->chromosome) || !parse_u32(f[1], gene_out->start) || !parse_u32(f[2], gene_out->end))
        return 1;
    gene_out->strand = invert_strand ? -sd : sd;
    return 0;
}

int abfit_pedigree_info(const abfit_pedigree *p, int32_t *n_pairs, double *p0uu, int32_t *n_samples, int64_t *n_sites)
{
    if (!p) return ABFIT_ERR_ARG;
    if (n_pairs) *n_pairs = (int32_t)(p->rows.size() / 4);
    if (p0uu) *p0uu = p->p0uu;
    if (n_samples) *n_samples = p->n_samples;
    if (n_sites) *n_sites = p->n_sites;
    return 0;
}

const double *abfit_pedigree_rows(const abfit_pedigree *p) { return p ? p->rows.data() : nullptr; }
const char *abfit_pedigree_warnings(const abfit_pedigree *p) { return p ? p->warnings.c_str() : ""; }
void abfit_pedigree_free(abfit_pedigree *p) { delete p; }

}  // extern "C"
