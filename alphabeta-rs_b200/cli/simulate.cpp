// simulate — methylomes with known epimutation rates: the ABneutral model run forward on a pedigree (libabfit,
// abfit_simulate), written as files the `alphabeta` front end reads as they are.
//
//   simulate -n nodelist.txt -e edgelist.txt --alpha A --beta B --sites L [--weight W --p0uu P] [--missing-rate M]
//            [--seed N] [--device 0] -o out/
//
// out/ receives one methylome file per sampled node (10-column format: 1 <pos> + CG <status> 2 <posteriorMax> <U|I|M>
// <meth_lvl> CGN), a nodelist whose file column names them by absolute path, a copy of the edgelist and truth.txt with
// the parameters.  Then `alphabeta -n out/nodelist.txt -e out/edgelist.txt -o fit/` fits them.
#include <cerrno>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <sys/stat.h>
#include <vector>

#include "../../include/abfit.h"

static std::string f64s(double v)
{
    char buf[512];
    abfit_format_f64(v, buf, sizeof buf);
    return buf;
}

static std::vector<std::string> split_any(const std::string &s, const char *seps)
{
    std::vector<std::string> out(1);
    for (char ch : s) {
        if (std::strchr(seps, ch)) out.emplace_back();
        else out.back() += ch;
    }
    return out;
}

static bool read_text(const std::string &path, std::string &out)
{
    std::ifstream f(path, std::ios::binary);
    if (!f) return false;
    std::ostringstream ss;
    ss << f.rdbuf();
    out = ss.str();
    return true;
}

static bool parse_num(const char *s, double &v)
{
    char *end = nullptr;
    errno = 0;
    v = std::strtod(s, &end);
    return *s && end && *end == '\0' && errno == 0;
}

static int usage_error(const std::string &msg)
{
    std::fprintf(stderr, "error: %s\n(see simulate --help)\n", msg.c_str());
    return 2;
}

int main(int argc, char **argv)
{
    std::string nodes, edges, output;
    double alpha = -1.0, beta = -1.0, weight = -1.0, p0uu = -1.0, missing = 0.0;
    long long sites = -1;
    unsigned long long seed = 0xAB0B200ull;
    int device = 0;
    bool have_alpha = false, have_beta = false, have_weight = false, have_p0uu = false;
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto val = [&](const char *name) -> const char * {
            if (i + 1 >= argc) {
                std::fprintf(stderr, "error: a value is required for '%s'\n", name);
                std::exit(2);
            }
            return argv[++i];
        };
        auto num = [&](const char *name) -> double {
            const char *s = val(name);
            double v;
            if (!parse_num(s, v)) {
                std::fprintf(stderr, "error: invalid number '%s' for '%s'\n", s, name);
                std::exit(2);
            }
            return v;
        };
        if (a == "-n" || a == "--nodes") nodes = val("--nodes");
        else if (a == "-e" || a == "--edges") edges = val("--edges");
        else if (a == "-o" || a == "--output") output = val("--output");
        else if (a == "--alpha") alpha = num("--alpha"), have_alpha = true;
        else if (a == "--beta") beta = num("--beta"), have_beta = true;
        else if (a == "--weight") weight = num("--weight"), have_weight = true;
        else if (a == "--p0uu") p0uu = num("--p0uu"), have_p0uu = true;
        else if (a == "--missing-rate") missing = num("--missing-rate");
        else if (a == "--sites") {
            const double v = num("--sites");
            if (!(v >= 1 && v <= 9e15 && v == (double)(long long)v)) return usage_error("--sites must be a positive integer");
            sites = (long long)v;
        } else if (a == "--seed") {
            const char *s = val("--seed");
            char *end = nullptr;
            errno = 0;
            seed = std::strtoull(s, &end, 0);
            if (!*s || *end || errno) return usage_error(std::string("invalid seed '") + s + "'");
        } else if (a == "--device") {
            double v;
            const char *s = val("--device");
            if (!parse_num(s, v) || v < 0 || v != (double)(int)v) return usage_error(std::string("invalid device '") + s + "'");
            device = (int)v;
        } else if (a == "-h" || a == "--help") {
            std::printf("Usage: simulate -n <NODES> -e <EDGES> --alpha <A> --beta <B> --sites <L> -o <OUTPUT> [OPTIONS]\n\n"
                        "Simulates methylomes under the ABneutral model on the pedigree of the nodelist / edgelist and\n"
                        "writes them with a nodelist, an edgelist and truth.txt that `alphabeta` reads as they are.\n\n"
                        "Options:\n"
                        "  -n, --nodes <NODES>        nodelist (file,node,generation,meth); meth == Y nodes are written\n"
                        "  -e, --edges <EDGES>        edgelist (from to); `from` is the parent, every node has at most one\n"
                        "      --alpha <A>            gain rate per generation, [0, 1]\n"
                        "      --beta <B>             loss rate per generation, [0, 1]\n"
                        "      --weight <W>           founder share of UM among non-UU states [default: steady state]\n"
                        "      --p0uu <P>             founder Pr(UU) [default: steady state p_uu_est(alpha, beta)]\n"
                        "      --sites <L>            CG sites per methylome\n"
                        "      --missing-rate <M>     share of sample-sites written with posteriorMax 0.5 [default: 0]\n"
                        "      --seed <SEED>          seed of the draws [default: 0xAB0B200]\n"
                        "      --device <N>           CUDA device [default: 0]\n"
                        "  -o, --output <OUTPUT>      output directory (created if missing)\n");
            return 0;
        } else {
            return usage_error("unexpected argument '" + a + "'");
        }
    }
    if (nodes.empty() || edges.empty() || output.empty()) return usage_error("-n, -e and -o are required");
    if (!have_alpha || !have_beta) return usage_error("--alpha and --beta are required");
    if (sites < 0) return usage_error("--sites is required");
    if (!have_weight || !have_p0uu) {
        double p_eq, w_eq;
        if (abfit_sim_equilibrium(alpha, beta, &p_eq, &w_eq)) return usage_error(abfit_last_error());
        if (!have_weight) weight = w_eq;
        if (!have_p0uu) p0uu = p_eq;
    }
    const abfit_sim_params params{alpha, beta, weight, p0uu, missing, (uint64_t)seed};
    abfit_sim_tree *tree = nullptr;
    if (abfit_sim_tree_build(nodes.c_str(), edges.c_str(), &tree)) {
        std::fprintf(stderr, "error: %s\n", abfit_last_error());
        return 2;
    }
    {  // parameter check before anything is written
        int32_t n_nodes = 0;
        abfit_sim_tree_info(tree, &n_nodes, nullptr, nullptr);
        std::vector<double> thr((size_t)n_nodes * 6);
        if (abfit_sim_tree_thresholds(tree, &params, thr.data())) return usage_error(abfit_last_error());
    }
    mkdir(output.c_str(), 0777);
    char absbuf[PATH_MAX];
    if (!realpath(output.c_str(), absbuf)) {
        std::fprintf(stderr, "error: cannot create the output directory %s\n", output.c_str());
        return 2;
    }
    const std::string out = absbuf;
    // the nodelist as the library parses it (abfit_sim_tree_build): its sampled lines, in order, are the output rows
    std::string ntext, etext;
    if (!read_text(nodes, ntext) || !read_text(edges, etext)) {
        std::fprintf(stderr, "error: cannot read the nodelist or the edgelist\n");
        return 2;
    }
    struct Row {
        std::string name, gen;
        bool meth;
    };
    std::vector<Row> rows;
    {
        const std::vector<std::string> lines = split_any(ntext, "\n\r");
        for (size_t li = 1; li < lines.size(); ++li) {
            const std::vector<std::string> e = split_any(lines[li], ",\t ");
            if (e.size() < 4 || e[2].empty() || e[2].find_first_not_of("+0123456789") != std::string::npos) continue;
            rows.push_back(Row{e[1], std::to_string(std::strtoul(e[2].c_str(), nullptr, 10)), e[3] == "Y"});
        }
    }
    int32_t S = 0;
    abfit_sim_tree_info(tree, nullptr, &S, nullptr);
    std::vector<std::string> files;
    std::string nl = "filename,node,gen,meth\n";
    for (auto &r : rows) {
        std::string file = "-";
        if (r.meth) {
            file = out + "/methylome_" + std::to_string(files.size()) + ".txt";
            files.push_back(file);
        }
        nl += file + "," + r.name + "," + r.gen + "," + (r.meth ? "Y" : "N") + "\n";
    }
    if ((int32_t)files.size() != S) {
        std::fprintf(stderr, "error: the nodelist's sampled lines could not be matched to the pedigree's samples\n");
        return 2;
    }
    abfit_ctx *ctx = nullptr;
    if (abfit_ctx_create(device, &ctx)) {
        std::fprintf(stderr, "error: %s\n", abfit_last_error());
        return 1;
    }
    std::vector<FILE *> fh(S);
    for (int s = 0; s < S; ++s) {
        fh[s] = std::fopen(files[s].c_str(), "wb");
        if (!fh[s]) {
            std::fprintf(stderr, "error: cannot create %s\n", files[s].c_str());
            return 1;
        }
        std::fputs("seqnames\tstart\tstrand\tcontext\tcounts.methylated\tcounts.total\tposteriorMax\tstatus\trc.meth.lvl\tcontext.trinucleotide\n", fh[s]);
    }
    // chunks of sites: the draws are keyed by the global site index, so the chunking does not change the data
    const int64_t chunk = std::min<int64_t>(sites, std::max<int64_t>(1, (int64_t)(1 << 26) / std::max(1, S)));
    std::vector<uint8_t> st((size_t)S * chunk);
    std::vector<double> po((size_t)S * chunk), me((size_t)S * chunk);
    const std::string pm_txt[2] = {f64s(0.5), f64s(1.0)}, lvl_txt[3] = {f64s(0.0), f64s(0.5), f64s(1.0)};
    const char code[3] = {'U', 'I', 'M'};
    std::string line;
    for (int64_t first = 0; first < sites; first += chunk) {
        const int64_t n = std::min<int64_t>(chunk, sites - first);
        if (abfit_simulate(ctx, tree, &params, first, n, st.data(), po.data(), me.data())) {
            std::fprintf(stderr, "error: %s\n", abfit_last_error());
            return 1;
        }
        for (int s = 0; s < S; ++s) {
            std::string buf;
            for (int64_t k = 0; k < n; ++k) {
                const size_t o = (size_t)s * n + k;
                const int v = st[o];
                buf += "1\t" + std::to_string(first + k + 1) + "\t+\tCG\t" + std::to_string(v) + "\t2\t" + pm_txt[po[o] == 1.0] + "\t" +
                       code[v] + "\t" + lvl_txt[v] + "\tCGN\n";
            }
            if (std::fwrite(buf.data(), 1, buf.size(), fh[s]) != buf.size()) {
                std::fprintf(stderr, "error: short write to %s\n", files[s].c_str());
                return 1;
            }
        }
    }
    for (int s = 0; s < S; ++s)
        if (std::fclose(fh[s])) {
            std::fprintf(stderr, "error: cannot write %s\n", files[s].c_str());
            return 1;
        }
    const std::string truth = "alpha\t" + f64s(alpha) + "\nbeta\t" + f64s(beta) + "\nweight\t" + f64s(weight) + "\np0uu\t" + f64s(p0uu) +
                              "\nmissing_rate\t" + f64s(missing) + "\nseed\t" + std::to_string(seed) + "\nsites\t" +
                              std::to_string(sites) + "\n";
    const std::pair<std::string, const std::string *> outs[3] = {
        {out + "/nodelist.txt", &nl}, {out + "/edgelist.txt", &etext}, {out + "/truth.txt", &truth}};
    for (auto &o : outs) {
        std::ofstream f(o.first, std::ios::binary);
        f << *o.second;
        if (!f) {
            std::fprintf(stderr, "error: cannot write %s\n", o.first.c_str());
            return 1;
        }
    }
    std::printf("%d methylomes of %lld sites written to %s (alpha %s, beta %s, weight %s, p0uu %s)\n", S, sites, out.c_str(),
                f64s(alpha).c_str(), f64s(beta).c_str(), f64s(weight).c_str(), f64s(p0uu).c_str());
    abfit_sim_tree_free(tree);
    abfit_ctx_destroy(ctx);
    return 0;
}
