// metaprofile — front end with the flags of the reference's `metaprofile` binary (src/cli/metaprofile.rs:14-114,
// src/arguments.rs:9-62, src/extract.rs:17-155) on top of libabfit, FUSED: sites are binned once in memory, the observed
// divergence of every window is one abfit_divergence call (segment offsets) and all windows are fitted by one
// abfit_alphabeta_batch call — instead of one directory of re-written methylome files and one serial alphabeta::run
// per window (src/cli/metaprofile.rs:50-72).
//
//   metaprofile -m <methylome dir> -g <annotation> [-w 5] [-s 0] [-o .] [-a] [-c 2048] [-i] [--name N]
//               [--cutoff-gene-length] [--iterations 100] [--seed N] [--device 0 | --devices 0-7] [--write-windows]
//               [--site-bootstrap BLOCK_SITES]
//               [alphabeta --nodes <nodelist> --edges <edgelist>]
//
// Files written (formats of the reference): distribution_<file>, distributions.txt, steady_state_methylation.txt,
// all_steady_state_methylation.txt and, with the sub-command, results.txt, raw.npy (iterations x 7 x windows) and
// metaplot.png (src/plot.rs:6-82: same series, colours and ranges, own rasteriser); a progress bar on stderr when it
// is a terminal (cli/progress.h).
// --write-windows additionally writes the reference's per-window directory tree ({region}/{window * step}/{file},
// nodelist.txt / edgelist.txt per directory; src/setup.rs:5-74, src/windows.rs:259-285) — the fused pipeline does not
// read it; with the sub-command every window directory also gets its bootstrap.png (src/boot_model.rs:105-109).
// Deliberate differences: methylome files are processed in name order (the reference uses the directory's own order); every window is fitted on ITS OWN sites
// (the reference only does that when the nodelist holds absolute, tab-separated paths: src/setup.rs:48-58), the
// measured nodes being matched to the methylome files by file name; the windows looped over are those of
// Windows::new (the reference's loop `(0..max).step_by(step)` can run one directory past them); seeded RNG.
// Like the reference, a window that cannot be fitted prints an error and is skipped, and results.txt pairs the
// i-th fitted window with the i-th distribution entry (src/cli/metaprofile.rs:76-77).  A window in which the samples
// list DIFFERENT numbers of sites is kept, as in the reference: "Lengths do not match, all bets are off", D = 0 for
// every pair of unequal length (src/pedigree.rs:222-230; one console line per window here, one per pair there).
#include <algorithm>
#include <atomic>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dirent.h>
#include <fstream>
#include <map>
#include <memory>
#include <sstream>
#include <string>
#include <sys/stat.h>
#include <thread>
#include <vector>

#include "../../include/abfit.h"
#include "progress.h"

static std::string f64s(double v)
{
    char buf[512];
    abfit_format_f64(v, buf, sizeof buf);
    return buf;
}
static bool exists(const std::string &p)
{
    struct stat st;
    return stat(p.c_str(), &st) == 0;
}
static std::string base_name(const std::string &p)
{
    const size_t k = p.find_last_of('/');
    return k == std::string::npos ? p : p.substr(k + 1);
}
static void mkdirs(const std::string &path)  // fs::create_dir_all
{
    for (size_t i = 1; i <= path.size(); ++i)
        if (i == path.size() || path[i] == '/') mkdir(path.substr(0, i).c_str(), 0755);
}

static int write_text(const std::string &path, const std::string &c)
{
    FILE *f = std::fopen(path.c_str(), "wb");
    if (!f) return 1;
    std::fwrite(c.data(), 1, c.size(), f);
    std::fclose(f);
    return 0;
}

struct Sample {
    std::string name;
    std::vector<abfit_cg_site> sites;
    std::vector<uint8_t> status;
    std::vector<double> post, meth;
    std::vector<int32_t> dist;
    std::vector<int64_t> order, seg;  // sites of window w: order[seg[w] .. seg[w+1]) (file order)
    // --write-windows: the parsed lines as read (MethylationSite::original) = slices of the file image
    std::string image;
    std::vector<int64_t> line_off;
    std::vector<int32_t> line_len;
    std::string original(size_t i) const { return image.substr((size_t)line_off[i], (size_t)line_len[i]); }
};

static bool read_whole_file(const std::string &path, std::string &out)
{
    FILE *f = std::fopen(path.c_str(), "rb");
    if (!f) return false;
    out.clear();
    struct stat st;
    if (fstat(fileno(f), &st) == 0 && st.st_size > 0) out.reserve((size_t)st.st_size);
    char buf[1 << 16];
    size_t n;
    while ((n = std::fread(buf, 1, sizeof buf, f)) > 0) out.append(buf, n);
    std::fclose(f);
    return true;
}

// independent iterations on the host threads (blocks of 8 from a shared counter)
template <class F>
static void parallel_for(size_t n, F f)
{
    const size_t nt = std::min<size_t>(std::min<size_t>(std::max(1u, std::thread::hardware_concurrency()), 32), (n + 7) / 8);
    if (nt <= 1) {
        for (size_t i = 0; i < n; ++i) f(i);
        return;
    }
    std::atomic<size_t> next{0};
    std::vector<std::thread> pool;
    for (size_t t = 0; t < nt; ++t)
        pool.emplace_back([&]() {
            for (size_t b; (b = next.fetch_add(8)) < n;)
                for (size_t i = b; i < std::min(n, b + 8); ++i) f(i);
        });
    for (auto &th : pool) th.join();
}

int main(int argc, char **argv)
{
    std::string methylome, genome, output = ".", name, nodes, edges;
    uint32_t window_size = 5, window_step = 0, cutoff = 2048;
    bool absolute = false, invert = false, cutoff_gene_length = false, sub = false, write_windows = false;
    long iterations = 100;
    unsigned long long seed = 0xAB0B200ull;
    int device = 0;
    std::vector<int> devices;  // --devices 0-7 / 0,2,5: windows sharded over several GPUs (abfit_alphabeta_batch_multi)
    long long site_boot = 0;   // --site-bootstrap N: site-block bootstrap of N-site blocks (0: the residual bootstrap)
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto val = [&]() -> const char * {
            if (i + 1 >= argc) {
                std::fprintf(stderr, "error: a value is required for '%s'\n", a.c_str());
                std::exit(2);
            }
            return argv[++i];
        };
        if (a == "alphabeta") sub = true;
        else if (sub && (a == "-n" || a == "--nodes")) nodes = val();
        else if (sub && (a == "-e" || a == "--edges")) edges = val();
        else if (sub && (a == "-i" || a == "--iterations" || a == "-p" || a == "--posterior-max-filter" || a == "-o" || a == "--output")) val();  // parsed and ignored, like the reference (src/arguments.rs:142-152)
        else if (a == "-m" || a == "--methylome") methylome = val();
        else if (a == "-g" || a == "--genome") genome = val();
        else if (a == "-w" || a == "--window-size") window_size = (uint32_t)std::strtoul(val(), nullptr, 10);
        else if (a == "-s" || a == "--window-step") window_step = (uint32_t)std::strtoul(val(), nullptr, 10);
        else if (a == "-o" || a == "--output-dir") output = val();
        else if (a == "-a" || a == "--absolute") absolute = true;
        else if (a == "-c" || a == "--cutoff") cutoff = (uint32_t)std::strtoul(val(), nullptr, 10);
        else if (a == "-i" || a == "--invert") invert = true;
        else if (a == "--name") name = val();
        else if (a == "-f" || a == "--force") {}
        else if (a == "--cutoff-gene-length") cutoff_gene_length = true;
        else if (a == "--iterations") iterations = std::atol(val());
        else if (a == "--seed") seed = std::strtoull(val(), nullptr, 0);
        else if (a == "--device") device = std::atoi(val());
        else if (a == "--write-windows") write_windows = true;
        else if (a == "--site-bootstrap") {
            site_boot = std::atoll(val());
            if (site_boot < 1) {
                std::fprintf(stderr, "error: --site-bootstrap needs a block size of at least one site\n");
                return 2;
            }
        }
        else if (a == "--devices") {
            const std::string v = val();
            size_t pos = 0;
            while (pos < v.size()) {
                size_t e = v.find(',', pos);
                if (e == std::string::npos) e = v.size();
                const std::string tok = v.substr(pos, e - pos);
                const size_t dash = tok.find('-');
                const int lo = std::atoi(tok.c_str()), hi = dash == std::string::npos ? lo : std::atoi(tok.c_str() + dash + 1);
                for (int d = lo; d <= hi; ++d) devices.push_back(d);
                pos = e + 1;
            }
        }
        else {
            std::fprintf(stderr, "error: unexpected argument '%s' found\n", a.c_str());
            return 2;
        }
    }
    if (methylome.empty() || genome.empty()) {
        std::fprintf(stderr, "error: the following required arguments were not provided:\n  --methylome <METHYLOME>\n  --genome <GENOME>\n");
        return 2;
    }
    if (site_boot > 0 && devices.size() > 1) {
        std::fprintf(stderr, "error: --site-bootstrap runs on one device; --devices names %zu\n", devices.size());
        return 2;
    }
    std::printf("Starting run %s\n", name.c_str());
    if (window_step == 0) window_step = window_size;  // src/cli/metaprofile.rs:18-20
    if (window_step == 0 || iterations <= 0) {
        std::printf("Error: window size / step and iterations must be positive\n");
        return 1;
    }

    // ---- extract (src/extract.rs:17-155) -----------------------------------------------------------------------
    std::vector<std::string> files;  // load_methylome (src/files.rs:23-38)
    if (DIR *d = opendir(methylome.c_str())) {
        while (dirent *e = readdir(d)) {
            const std::string fn = e->d_name;
            const size_t dot = fn.find_last_of('.');
            if (fn == "." || fn == ".." || dot == std::string::npos || dot == 0) continue;
            const std::string ext = fn.substr(dot + 1);
            if (ext.find("tsv") != std::string::npos || ext.find("fn") != std::string::npos) continue;
            files.push_back(fn);
        }
        closedir(d);
    }
    if (files.empty()) {
        std::printf("Error: Could not find any files in the methylome directory. Please check your input. Files with .tsv or .fn extensions are ignored.\n");
        return 1;
    }
    std::sort(files.begin(), files.end());
    std::vector<abfit_gene> genes;
    {
        std::ifstream f(genome);
        if (!f) {
            std::printf("Error: Error while reading genome annotation file: %s\n", genome.c_str());
            return 1;
        }
        std::string line;
        abfit_gene g;
        while (std::getline(f, line)) {
            if (!line.empty() && line.back() == '\r') line.pop_back();
            if (abfit_parse_annotation_line(line.c_str(), invert, &g) == 0) genes.push_back(g);
        }
    }
    if (genes.empty()) {
        std::printf("Error: Could not parse a single annotation from the annotation file. Please check your input or add a parser implemenation for your data format.\n");
        return 1;
    }
    uint32_t max_gene_length = 100;  // src/extract.rs:49-58
    if (absolute) {
        max_gene_length = 0;
        for (auto &g : genes) max_gene_length = std::max(max_gene_length, (uint32_t)(g.end - g.start));
        std::printf("The maximum gene length is %u bp\n", max_gene_length);
    }
    if (!exists(output)) {
        std::printf("Error: output directory %s does not exist\n", output.c_str());
        return 1;
    }
    abfit_window_args wa{window_size, window_step, cutoff, max_gene_length, absolute ? 1 : 0, cutoff_gene_length ? 1 : 0};
    int32_t nwin[3];
    if (abfit_window_counts(&wa, nwin)) {
        std::printf("Error: %s\n", abfit_last_error());
        return 1;
    }
    const int n_total = nwin[0] + nwin[1] + nwin[2];

    // One methylome file = one independent unit of work (the reference: rayon par_iter over the files,
    // src/extract.rs:75): files are loaded, parsed and binned on a small pool of host threads, and the parser itself
    // splits a file over the threads that are left.
    std::vector<Sample> samples(files.size());
    std::vector<std::string> load_error(files.size());
    const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
    const unsigned outer = (unsigned)std::max<size_t>(1, std::min<size_t>(std::min<size_t>(files.size(), hw), 16));
    if (!getenv("ABFIT_HOST_THREADS")) setenv("ABFIT_HOST_THREADS", std::to_string(std::max(1u, hw / outer)).c_str(), 0);
    auto load_sample = [&](size_t fi) -> bool {
        Sample &S = samples[fi];
        S.name = files[fi];
        // the whole file in one call (parsed on several threads); Windows::extract skips the header row (src/windows.rs:322)
        if (read_whole_file(methylome + "/" + files[fi], S.image)) {
            int64_t cap = 1, n = 0;
            for (char ch : S.image) cap += ch == '\n';
            S.sites.resize((size_t)cap);
            S.status.resize((size_t)cap);
            S.post.resize((size_t)cap);
            S.meth.resize((size_t)cap);
            if (write_windows) {
                S.line_off.resize((size_t)cap);
                S.line_len.resize((size_t)cap);
            }
            if (abfit_parse_methylome_buffer(S.image.data(), (int64_t)S.image.size(), invert, 1, cap, S.sites.data(), S.post.data(),
                                             S.status.data(), S.meth.data(), write_windows ? S.line_off.data() : nullptr,
                                             write_windows ? S.line_len.data() : nullptr, &n)) {
                load_error[fi] = abfit_last_error();
                return false;
            }
            S.sites.resize((size_t)n);
            S.status.resize((size_t)n);
            S.post.resize((size_t)n);
            S.meth.resize((size_t)n);
            S.line_off.resize(write_windows ? (size_t)n : 0);
            S.line_len.resize(write_windows ? (size_t)n : 0);
            // (cap counted every line of the file, CG or not: give the difference back)
            S.sites.shrink_to_fit();
            S.status.shrink_to_fit();
            S.post.shrink_to_fit();
            S.meth.shrink_to_fit();
            S.line_off.shrink_to_fit();
            S.line_len.shrink_to_fit();
            if (!write_windows) std::string().swap(S.image);
        }
        S.dist.assign(n_total, 0);
        int64_t n_assign = 0;
        abfit_place_sites(genes.data(), (int32_t)genes.size(), S.sites.data(), (int64_t)S.sites.size(), &wa, S.dist.data(), &n_assign, 0,
                          nullptr, nullptr);
        std::vector<int64_t> asite((size_t)n_assign);
        std::vector<int32_t> awin((size_t)n_assign);
        abfit_place_sites(genes.data(), (int32_t)genes.size(), S.sites.data(), (int64_t)S.sites.size(), &wa, S.dist.data(), &n_assign,
                          n_assign, asite.data(), awin.data());
        if (invert) {
            // Windows::inverse (src/windows.rs:87-92), quirk included: upstream <- reversed downstream, gene reversed,
            // downstream <- reversed NEW upstream = the old downstream
            auto remap = [&](int32_t w) -> std::vector<int32_t> {
                std::vector<int32_t> out;
                if (w >= nwin[0] && w < nwin[0] + nwin[1]) out.push_back(nwin[0] + (nwin[1] - 1 - (w - nwin[0])));
                if (w >= nwin[0] + nwin[1]) {
                    const int i = w - nwin[0] - nwin[1];
                    out.push_back(nwin[0] - 1 - i);        // new upstream
                    out.push_back(nwin[0] + nwin[1] + i);  // new downstream = old downstream
                }
                return out;  // old upstream sites are dropped
            };
            std::vector<int64_t> a2;
            std::vector<int32_t> w2;
            for (int64_t q = 0; q < n_assign; ++q)
                for (int32_t nw : remap(awin[q])) {
                    a2.push_back(asite[q]);
                    w2.push_back(nw);
                }
            asite.swap(a2);
            awin.swap(w2);
            std::fill(S.dist.begin(), S.dist.end(), 0);
            for (int32_t w : awin) ++S.dist[w];
        }
        // stable counting sort of the hits by window: file order inside every window
        S.seg.assign(n_total + 1, 0);
        for (int32_t w : awin) ++S.seg[w + 1];
        for (int w = 0; w < n_total; ++w) S.seg[w + 1] += S.seg[w];
        S.order.resize(asite.size());
        std::vector<int64_t> cur(S.seg.begin(), S.seg.end() - 1);
        for (size_t q = 0; q < asite.size(); ++q) S.order[(size_t)cur[awin[q]]++] = asite[q];
        return true;
    };
    {
        std::atomic<size_t> next{0};
        std::atomic<bool> ok{true};
        std::vector<std::thread> pool;
        for (unsigned t = 0; t < outer; ++t)
            pool.emplace_back([&]() {
                for (size_t fi; (fi = next.fetch_add(1)) < files.size();)
                    if (!load_sample(fi)) ok = false;
            });
        for (auto &th : pool) th.join();
        if (!ok) {
            for (auto &e : load_error)
                if (!e.empty()) std::printf("Error: %s\n", e.c_str());
            return 1;
        }
    }
    // distribution / steady-state files (src/extract.rs:100-151, src/windows.rs:94-176,245-257)
    std::vector<std::vector<double>> ss(samples.size(), std::vector<double>(n_total));
    for (size_t fi = 0; fi < samples.size(); ++fi)
        for (int w = 0; w < n_total; ++w) {
            double acc = 0.0;
            for (int64_t q = samples[fi].seg[w]; q < samples[fi].seg[w + 1]; ++q) acc = acc + samples[fi].meth[(size_t)samples[fi].order[q]];
            ss[fi][w] = acc / (double)(samples[fi].seg[w + 1] - samples[fi].seg[w]);
        }
    std::vector<double> avg(n_total, 0.0);
    for (size_t fi = 0; fi < samples.size(); ++fi)
        for (int w = 0; w < n_total; ++w) avg[w] += ss[fi][w] / (double)samples.size();
    std::string all_d, all_s, avg_s;
    for (size_t fi = 0; fi < samples.size(); ++fi) {
        std::string one;
        all_d += samples[fi].name + ";";
        all_s += samples[fi].name + ";";
        for (int w = 0; w < n_total; ++w) {
            one += std::to_string(samples[fi].dist[w]) + "\n";
            all_d += std::to_string(samples[fi].dist[w]) + ";";
            all_s += f64s(ss[fi][w]) + ";";
        }
        all_d += "\n";
        all_s += "\n";
        write_text(output + "/distribution_" + samples[fi].name, one);
    }
    for (int w = 0; w < n_total; ++w) avg_s += f64s(avg[w]) + "\n";
    write_text(output + "/steady_state_methylation.txt", avg_s);
    write_text(output + "/all_steady_state_methylation.txt", all_s);
    write_text(output + "/distributions.txt", all_d);
    if (write_windows) {
        // The per-window directory tree of the reference (setup_output_dir src/setup.rs:5-74, Windows::save
        // src/windows.rs:259-285): {output}/{upstream,gene,downstream}/{window * step}/{methylome file} holding the
        // header row and the window's original lines; with the sub-command every directory also gets the edgelist and
        // the nodelist, whose '/'-led tab-separated lines are re-pathed into the directory (src/setup.rs:48-58).  The
        // fused pipeline below does not read any of it — this is for tools that consume the reference's layout.
        static const char *HEADER = "seqnames\tstart\tstrand\tcontext\tcounts.methylated\tcounts.total\tposteriorMax\tstatus\trc.meth.lvl\tcontext.trinucleotide\n";
        const char *side_name[3] = {"upstream", "gene", "downstream"};
        const uint32_t side_max[3] = {absolute ? cutoff : 100u, absolute ? max_gene_length : 100u, absolute ? cutoff : 100u};
        std::string nodes_text, edges_text;
        if (sub) {
            std::ifstream fn(nodes), fe(edges);
            std::stringstream a, b;
            a << fn.rdbuf();
            b << fe.rdbuf();
            nodes_text = a.str();
            edges_text = b.str();
        }
        for (int side = 0; side < 3; ++side)
            for (uint32_t window = 0; window < side_max[side]; window += window_step) {
                const std::string dir = output + "/" + side_name[side] + "/" + std::to_string(window);
                mkdirs(dir);
                if (!sub) continue;
                std::string nodelist;
                size_t pos = 0;
                for (;;) {  // nodes.split('\n'): a trailing newline yields a last empty piece, which also gets its "\n"
                    const size_t e = nodes_text.find('\n', pos);
                    std::string line = nodes_text.substr(pos, e == std::string::npos ? std::string::npos : e - pos);
                    if (!line.empty() && line[0] == '/') {
                        const std::string old_file = line.substr(0, line.find('\t'));
                        const std::string fname = old_file.substr(old_file.find_last_of('/') + 1);
                        const std::string repl = dir + "/" + fname;
                        std::string out;
                        size_t q = 0;
                        for (;;) {  // str::replace: every occurrence
                            const size_t h = line.find(old_file, q);
                            if (h == std::string::npos) break;
                            out += line.substr(q, h - q) + repl;
                            q = h + old_file.size();
                        }
                        line = out + line.substr(q);
                    }
                    nodelist += line + "\n";
                    if (e == std::string::npos) break;
                    pos = e + 1;
                }
                write_text(dir + "/nodelist.txt", nodelist);
                write_text(dir + "/edgelist.txt", edges_text);
            }
        for (const Sample &A : samples) {
            int w = 0;
            for (int side = 0; side < 3; ++side)
                for (int i = 0; i < nwin[side]; ++i, ++w) {
                    const std::string dir = output + "/" + side_name[side] + "/" + std::to_string((uint64_t)i * window_step);
                    mkdirs(dir);
                    std::string text = HEADER;
                    for (int64_t q = A.seg[w]; q < A.seg[w + 1]; ++q) {
                        if (q > A.seg[w]) text += "\n";
                        text += A.original((size_t)A.order[(size_t)q]);
                    }
                    write_text(dir + "/" + A.name, text);
                }
        }
    }
    if (!sub) {
        std::printf("Done\n");
        return 0;
    }

    // ---- alphabeta_multiple (src/cli/metaprofile.rs:33-114), fused ----------------------------------------------
    if (nodes.empty() || edges.empty()) {
        std::printf("Error: the alphabeta sub-command needs --nodes and --edges\n");
        return 1;
    }
    int32_t S = 0, n_pairs = 0;
    // sizes first (no outputs), then the graph itself: any number of samples and pairs
    if (abfit_pedigree_graph(nodes.c_str(), edges.c_str(), &S, nullptr, 0, &n_pairs, nullptr, 0)) {
        std::printf("Error: Error while building pedigree: %s\n", abfit_last_error());
        return 1;
    }
    if (S < 2 || n_pairs < 1) {
        std::printf("Error: Error while building pedigree: the nodelist has fewer than two measured samples\n");
        return 1;
    }
    std::vector<char> fbuf((size_t)S * 4097 + 1);  // PATH_MAX + '\n' per measured node
    std::vector<double> pairs((size_t)5 * n_pairs);
    if (abfit_pedigree_graph(nodes.c_str(), edges.c_str(), &S, fbuf.data(), (int32_t)std::min<size_t>(fbuf.size(), 0x7fffffff), &n_pairs,
                             pairs.data(), n_pairs)) {
        std::printf("Error: Error while building pedigree: %s\n", abfit_last_error());
        return 1;
    }
    std::vector<int> sample_of(S, -1);  // measured node -> methylome file, by file name
    {
        std::string all(fbuf.data());
        size_t pos = 0;
        for (int s = 0; s < S; ++s) {
            const size_t e = all.find('\n', pos);
            const std::string bn = base_name(all.substr(pos, e - pos));
            pos = e + 1;
            for (size_t fi = 0; fi < samples.size(); ++fi)
                if (samples[fi].name == bn) sample_of[s] = (int)fi;
            if (sample_of[s] < 0) {
                std::printf("Error: Error while building pedigree: Could not open node file: %s\n", bn.c_str());
                return 1;
            }
        }
    }
    if (S <= 0 || n_pairs <= 0) {  // the reference fails here too: nothing to compare (src/pedigree.rs:92-193)
        std::printf("Error: Error while building pedigree: the nodelist has fewer than two measured samples\n");
        return 1;
    }
    // Windows whose samples all list the same number of sites ("regular") go into ONE divergence call.  A window whose
    // samples list different numbers of sites is kept, as in the reference: DMatrix::from prints "Lengths do not match, all
    // bets are off" and leaves D = 0 for every pair of unequal length (src/pedigree.rs:222-230); pairs of equal length are
    // compared index by index, every sample's methylation level comes from its own sites (one small divergence call per
    // group of equally long samples of such a window, on the first device).
    std::vector<int> usable;       // every window that gets a pedigree, in window order
    std::vector<int> reg_of;       // usable index -> index among the regular windows, -1: unequal site counts
    std::vector<int> reg_windows;  // the regular windows
    std::vector<int64_t> seg{0};   // their segment offsets
    auto win_len = [&](int s, int w) { return samples[sample_of[s]].seg[w + 1] - samples[sample_of[s]].seg[w]; };
    for (int w = 0; w < n_total; ++w) {
        const int64_t len = win_len(0, w);
        bool same = true, any = len > 0;
        for (int s = 1; s < S; ++s) {
            same &= win_len(s, w) == len;
            any |= win_len(s, w) > 0;
        }
        if (!any) {
            std::printf("Error: Model failed: window %d is empty\n", w);
            continue;
        }
        usable.push_back(w);
        if (same) {
            reg_of.push_back((int)reg_windows.size());
            reg_windows.push_back(w);
            seg.push_back(seg.back() + len);
        } else {
            reg_of.push_back(-1);
        }
    }
    if (site_boot > 0)  // DMatrix::from sets D = 0 for pairs of unequal length: a site bootstrap of such a window is undefined
        for (size_t k = 0; k < usable.size(); ++k)
            if (reg_of[k] < 0) {
                std::printf("Error: --site-bootstrap: the samples of window %d list different numbers of sites\n", usable[k]);
                return 1;
            }
    if (devices.empty()) devices.push_back(device);
    std::vector<abfit_ctx *> ctxs(devices.size(), nullptr);
    for (size_t d = 0; d < devices.size(); ++d)
        if (abfit_ctx_create(devices[d], &ctxs[d])) {
            std::printf("Error: %s\n", abfit_last_error());
            return 1;
        }
    const int64_t L = seg.back();
    const int W = (int)usable.size(), WR = (int)reg_windows.size();
    const size_t P = (size_t)S * (S - 1) / 2;
    std::vector<double> D((size_t)std::max(W, 1) * std::max<size_t>(P, 1), 0.0), p0uu(std::max(W, 1));
    std::vector<uint8_t> st((size_t)S * L);  // the regular windows' sites (kept for --site-bootstrap)
    std::vector<double> po((size_t)S * L), me((size_t)S * L);
    {
        parallel_for((size_t)S * 8, [&](size_t job) {  // eight slices of the window list per sample
            const size_t s = job / 8, part = job % 8;
            const Sample &A = samples[sample_of[s]];
            const size_t k0 = reg_windows.size() * part / 8, k1 = reg_windows.size() * (part + 1) / 8;
            int64_t o = seg[k0];
            for (size_t k = k0; k < k1; ++k)
                for (int64_t q = A.seg[reg_windows[k]]; q < A.seg[reg_windows[k] + 1]; ++q, ++o) {
                    st[s * L + o] = A.status[(size_t)A.order[q]];
                    po[s * L + o] = A.post[(size_t)A.order[q]];
                    me[s * L + o] = A.meth[(size_t)A.order[q]];
                }
        });
        std::vector<double> Dr((size_t)std::max(WR, 1) * std::max<size_t>(P, 1)), p0r(std::max(WR, 1));
        if (WR > 0 && abfit_divergence_multi(ctxs.data(), (int32_t)ctxs.size(), st.data(), po.data(), me.data(), S, L, seg.data(), WR,
                                             0.99, Dr.data(), nullptr, nullptr, p0r.data(), nullptr, nullptr)) {
            std::printf("Error: %s\n", abfit_last_error());
            return 1;
        }
        for (int k = 0; k < W; ++k)
            if (reg_of[k] >= 0) {
                std::copy(Dr.begin() + (size_t)reg_of[k] * P, Dr.begin() + (size_t)(reg_of[k] + 1) * P, D.begin() + (size_t)k * P);
                p0uu[k] = p0r[reg_of[k]];
            }
    }
    for (int k = 0; k < W; ++k) {
        if (reg_of[k] >= 0) continue;
        const int w = usable[k];
        std::printf("Lengths do not match, all bets are off: window %d (pairs of samples with different site counts get D = 0)\n", w);
        std::map<int64_t, std::vector<int>> by_len;
        for (int s = 0; s < S; ++s) by_len[win_len(s, w)].push_back(s);
        std::vector<double> level(S, 0.0);  // mean rc.meth.lvl of every sample's own sites (src/pedigree.rs:171-172)
        for (auto &kv : by_len) {
            const std::vector<int> &grp = kv.second;
            const int G = (int)grp.size();
            const int64_t len = kv.first;
            if (len == 0) {
                for (int s : grp) level[s] = 0.0 / 0.0;  // 0 / 0 = NaN, as in the reference
                continue;
            }
            std::vector<uint8_t> gs((size_t)G * len);
            std::vector<double> gp((size_t)G * len), gm((size_t)G * len);
            for (int q = 0; q < G; ++q) {
                const Sample &A = samples[sample_of[grp[q]]];
                int64_t o = 0;
                for (int64_t i = A.seg[w]; i < A.seg[w + 1]; ++i, ++o) {
                    gs[(size_t)q * len + o] = A.status[(size_t)A.order[i]];
                    gp[(size_t)q * len + o] = A.post[(size_t)A.order[i]];
                    gm[(size_t)q * len + o] = A.meth[(size_t)A.order[i]];
                }
            }
            const size_t PG = (size_t)G * (G - 1) / 2;
            std::vector<double> Dg(std::max<size_t>(PG, 1)), methsum(G);
            std::vector<int64_t> nvalid(G);
            if (abfit_divergence(ctxs[0], gs.data(), gp.data(), gm.data(), G, len, nullptr, 1, 0.99, Dg.data(), nullptr, nullptr, nullptr,
                                 methsum.data(), nvalid.data())) {
                std::printf("Error: %s\n", abfit_last_error());
                return 1;
            }
            size_t p = 0;
            for (int a = 0; a < G; ++a) {
                level[grp[a]] = methsum[a] / (double)nvalid[a];
                for (int b = a + 1; b < G; ++b) {
                    const int i = grp[a], j = grp[b];  // ascending sample order inside a group
                    D[(size_t)k * P + (size_t)i * S - (size_t)i * (i + 1) / 2 + (size_t)(j - i - 1)] = Dg[p++];
                }
            }
        }
        double acc = 0.0;  // src/pedigree.rs:179-183
        for (int s = 0; s < S; ++s) acc += 1.0 - level[s];
        p0uu[k] = acc / (double)S;
    }
    // one problem per window whose pedigree has no NaN (the reference panics on those, src/ab_neutral.rs:28)
    std::vector<int> fitted;
    std::vector<std::vector<double>> peds;
    {
        std::vector<std::vector<double>> all((size_t)W);
        std::vector<uint8_t> good((size_t)W, 0);
        parallel_for((size_t)W, [&](size_t k) {
            std::vector<double> ped((size_t)n_pairs * 4);
            bool ok = n_pairs > 0 && p0uu[k] == p0uu[k];
            for (int r = 0; r < n_pairs; ++r) {
                const int i = (int)pairs[5 * r], j = (int)pairs[5 * r + 1];
                const size_t p = (size_t)i * S - (size_t)i * (i + 1) / 2 + (size_t)(j - i - 1);
                ped[4 * r + 0] = pairs[5 * r + 2];
                ped[4 * r + 1] = pairs[5 * r + 3];
                ped[4 * r + 2] = pairs[5 * r + 4];
                ped[4 * r + 3] = D[k * P + p];
                ok &= ped[4 * r + 3] == ped[4 * r + 3];
            }
            good[k] = ok;
            if (ok) all[k] = std::move(ped);
        });
        for (int k = 0; k < W; ++k) {
            if (!good[(size_t)k]) {
                std::printf("Error: Model failed: window %d has too few valid sites (NaN divergence)\n", usable[k]);
                continue;
            }
            fitted.push_back(k);
            peds.push_back(std::move(all[(size_t)k]));
        }
    }
    const int F = (int)fitted.size();
    const int n = (int)iterations;
    std::vector<abfit_problem> probs(F);
    // (written in full by the generator below: no zero-fill of gigabytes first)
    std::unique_ptr<double[]> simplices(new double[std::max<size_t>(1, (size_t)F * n * 20)]);
    std::vector<double> rows((size_t)F * n * 7), analysis((size_t)F * 32);
    std::vector<int32_t> status(F);
    std::vector<abfit_fit> best(F);
    std::vector<uint64_t> ids(F);  // every window's generator key is its position in the genome-wide window list
    parallel_for((size_t)F, [&](size_t f) {
        const int k = fitted[f];
        ids[f] = (uint64_t)usable[k];
        probs[f] = abfit_problem{peds[f].data(), n_pairs, p0uu[k], p0uu[k], 1.0};
        double max_div = peds[f][3];
        for (int r = 1; r < n_pairs; ++r) max_div = std::max(max_div, peds[f][4 * r + 3]);
        abfit_gen_start_simplices(seed, (uint64_t)usable[k], n, max_div, simplices.get() + (size_t)f * n * 20);
    });
    // start simplices, resample indices and vary vertices of a window are all keyed by (seed, window id): its result
    // does not depend on which other windows are fitted with it, nor on how the windows are sharded over the GPUs.
    // The resample indices (4 x iterations x pairs bytes per window: 14 GB for 10 000 windows at -i 1000) are drawn on
    // the device (resample_idx = NULL): the numbers abfit_gen_resample_idx(seed, window id, ...) gives.
    // progress::multi(total_steps) (src/cli/metaprofile.rs:46): one step per window; the windows are fitted in one batched
    // call, so the bar stands at the windows prepared so far while the GPUs work and jumps to the end afterwards
    progress::Bar pb("Progress ", (unsigned long long)n_total, true);
    pb.set((unsigned long long)(n_total - F));
    if (F > 0 && site_boot > 0) {
        // the fit of abfit_alphabeta_batch, then the site-block bootstrap of every fitted window on its own sites (the
        // fitted windows' sites copied next to each other: window f = problem f)
        std::vector<int64_t> fseg(F + 1, 0);
        for (int f = 0; f < F; ++f) {
            const int r = reg_of[fitted[f]];
            fseg[f + 1] = fseg[f] + seg[r + 1] - seg[r];
        }
        const int64_t LF = fseg[F];
        std::vector<uint8_t> fst((size_t)S * LF);
        std::vector<double> fpo((size_t)S * LF), fme((size_t)S * LF);
        parallel_for((size_t)S, [&](size_t s) {
            for (int f = 0; f < F; ++f) {
                const int r = reg_of[fitted[f]];
                const int64_t len = seg[r + 1] - seg[r];
                std::copy_n(st.begin() + s * L + seg[r], len, fst.begin() + s * LF + fseg[f]);
                std::copy_n(po.begin() + s * L + seg[r], len, fpo.begin() + s * LF + fseg[f]);
                std::copy_n(me.begin() + s * L + seg[r], len, fme.begin() + s * LF + fseg[f]);
            }
        });
        std::vector<int32_t> rp((size_t)F * n_pairs * 2);
        for (int f = 0; f < F; ++f)
            for (int q = 0; q < n_pairs; ++q) {
                rp[((size_t)f * n_pairs + q) * 2] = (int32_t)pairs[5 * q];
                rp[((size_t)f * n_pairs + q) * 2 + 1] = (int32_t)pairs[5 * q + 1];
            }
        std::vector<int32_t> nan_reps(F);
        if (abfit_fit_batch(ctxs[0], probs.data(), F, n, simplices.get(), 10000, DBL_EPSILON, 0, best.data(), nullptr, nullptr,
                            nullptr, status.data()) ||
            abfit_site_boot_batch(ctxs[0], probs.data(), F, rp.data(), fst.data(), fpo.data(), fme.data(), S, LF, fseg.data(), 0.99,
                                  site_boot, best.data(), n, seed, 0, ids.data(), 1000, DBL_EPSILON, 0, rows.data(), nullptr,
                                  analysis.data(), nullptr, nan_reps.data())) {
            std::printf("Error: %s\n", abfit_last_error());
            return 1;
        }
        for (int f = 0; f < F; ++f)
            if (nan_reps[f])
                std::printf("Site bootstrap: window %d: %d of %d replicates left a pair without valid sites (NaN rows)\n",
                            usable[fitted[f]], nan_reps[f], n);
    } else if (F > 0 && abfit_alphabeta_batch_multi(ctxs.data(), (int32_t)ctxs.size(), probs.data(), F, n, simplices.get(), n, nullptr,
                                                    seed, 0, ids.data(), 10000, 1000, DBL_EPSILON, 0, best.data(), nullptr, nullptr,
                                                    status.data(), rows.data(), analysis.data())) {
        std::printf("Error: %s\n", abfit_last_error());
        return 1;
    }
    pb.finish();
    std::vector<int32_t> cg, region;
    std::vector<abfit_fit> rbest;
    std::vector<double> ranalysis, robs, raw;
    std::vector<int> keep;
    for (int f = 0; f < F; ++f) {
        if (status[f] != 0) {
            std::printf("Error: Model failed: window %d\n", usable[fitted[f]]);
            continue;
        }
        keep.push_back(f);
    }
    const int R = (int)keep.size();
    for (int q = 0; q < R; ++q) {
        const int f = keep[q], w = usable[fitted[f]];
        cg.push_back(samples[0].dist[(size_t)q]);  // the i-th result meets the i-th distribution entry (src/cli/metaprofile.rs:76-77)
        region.push_back(w < nwin[0] ? 0 : w < nwin[0] + nwin[1] ? 1 : 2);
        rbest.push_back(best[f]);
        ranalysis.insert(ranalysis.end(), analysis.begin() + (size_t)f * 32, analysis.begin() + (size_t)f * 32 + 32);
        robs.push_back(1.0 - p0uu[fitted[f]]);
    }
    raw.resize((size_t)n * 7 * R);  // [iteration][column][window]
    for (int q = 0; q < R; ++q)
        for (int it = 0; it < n; ++it)
            for (int c = 0; c < 7; ++c) raw[((size_t)it * 7 + c) * R + q] = rows[((size_t)keep[q] * n + it) * 7 + c];
    const std::string rp = output + "/results.txt";
    if (abfit_write_metaprofile_results(rp.c_str(), name.c_str(), R, cg.data(), region.data(), rbest.data(), ranalysis.data(), robs.data())) {
        std::printf("Error: %s\n", abfit_last_error());
        return 1;
    }
    {
        std::ifstream f(rp);
        std::string line;
        while (std::getline(f, line)) std::printf("%s\n", line.c_str());
        std::printf("\n");
    }
    const int64_t shape[3] = {n, 7, R};
    if (abfit_write_npy_f64((output + "/raw.npy").c_str(), raw.data(), 3, shape)) {
        std::printf("Error: %s\n", abfit_last_error());
        return 1;
    }
    if (write_windows) {  // boot_model::run draws bootstrap.png into every window's own directory (src/boot_model.rs:105-109)
        const char *side_name[3] = {"upstream", "gene", "downstream"};
        std::vector<double> al(n), be(n);
        for (int q = 0; q < R; ++q) {
            const int f = keep[q], w = usable[fitted[f]];
            const int side = w < nwin[0] ? 0 : w < nwin[0] + nwin[1] ? 1 : 2;
            const int i = w - (side == 0 ? 0 : side == 1 ? nwin[0] : nwin[0] + nwin[1]);
            for (int it = 0; it < n; ++it) {
                al[it] = rows[((size_t)f * n + it) * 7];
                be[it] = rows[((size_t)f * n + it) * 7 + 1];
            }
            const std::string png = output + "/" + side_name[side] + "/" + std::to_string((uint64_t)i * window_step) + "/bootstrap.png";
            if (abfit_plot_bootstrap(png.c_str(), al.data(), be.data(), n)) std::printf("Error: %s\n", abfit_last_error());
        }
    }
    {  // plot::metaplot(&analyses, &args) (src/cli/metaprofile.rs:113): alpha, beta and their 95 % intervals per fitted window
        std::vector<double> al(R), be(R), al_lo(R), al_hi(R), be_lo(R), be_hi(R);
        for (int q = 0; q < R; ++q) {
            al[q] = rbest[q].theta[0];
            be[q] = rbest[q].theta[1];
            al_lo[q] = ranalysis[(size_t)q * 32 + 16];
            al_hi[q] = ranalysis[(size_t)q * 32 + 17];
            be_lo[q] = ranalysis[(size_t)q * 32 + 18];
            be_hi[q] = ranalysis[(size_t)q * 32 + 19];
        }
        if (abfit_plot_metaplot((output + "/metaplot.png").c_str(), R, al.data(), be.data(), al_lo.data(), al_hi.data(), be_lo.data(), be_hi.data())) {
            std::printf("Error: %s\n", abfit_last_error());
            return 1;
        }
    }
    for (abfit_ctx *c : ctxs) abfit_ctx_destroy(c);
    return 0;
}
