// regions — epimutation rates in arbitrary genomic regions: one ABneutral fit (and bootstrap) per line of a BED file,
// on top of libabfit.
//
//   regions -n nodelist.txt -e edgelist.txt -r regions.bed [-i 100] [-p 0.99] [-o .] [--seed N]
//           [--device 0 | --devices 0-7] [--site-bootstrap BLOCK_SITES]
//
// The measured samples' methylome files are read as `alphabeta --site-bootstrap` reads them (cli/sites.h); they must list
// the same (chromosome, position) sequence, grouped by chromosome with positions non-decreasing.  Every BED line is a
// region (abfit_parse_region_line: 0-based, half-open, both strands; column 4 is its name), turned into a range of site
// indices (abfit_region_ranges).  One abfit_region_divergence call gives the observed divergence and p0uu of every region
// without copying sites; every fittable region is then fitted and bootstrapped by one abfit_alphabeta_batch_multi call.
// A region is keyed by its line index in the BED file (start simplices, resamples, vary vertices): dropping or adding a
// region changes no other region's result, and --devices gives the same bits as one device.
// --site-bootstrap BLOCK_SITES: abfit_fit_batch, then abfit_site_boot_batch on the fitted regions' sites (gathered next to
// each other on the host, the only mode that copies sites); one device.
//
// Files written to the output directory:
//   regions.tsv  one row per BED region, in file order: name, chromosome, start, end, sites, p0uu, alpha, beta, weight,
//                intercept, the bootstrap's sd and 95 % bounds of alpha and beta, status ("ok", or why the region was not
//                fitted: "no sites", "pair without valid sites", "sample without valid sites", "fit failed")
//   raw.npy      bootstrap rows [n_fitted][n_boot][7] of the "ok" regions, in file order
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <memory>
#include <sstream>
#include <string>
#include <sys/stat.h>
#include <vector>

#include "../../include/abfit.h"
#include "sites.h"

static bool exists(const std::string &p)
{
    struct stat st;
    return stat(p.c_str(), &st) == 0;
}

static std::string f64s(double v)
{
    char buf[512];
    abfit_format_f64(v, buf, sizeof buf);
    return buf;
}

struct Region {
    std::string name, chrom_text;
    int32_t chrom = 0;
    int64_t start0 = 0, end = 0, line = 0;  // line: index of the line in the BED file (the region's generator key)
};

int main(int argc, char **argv)
{
    long iterations = 100;
    std::string edges = "./edgelist.txt", nodes = "./nodelist.txt", output = ".", bed;
    double filter = 0.99;
    unsigned long long seed = 0xAB0B200ull;
    int device = 0;
    std::vector<int> devices;
    long long site_boot = 0;
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto val = [&]() -> const char * {
            if (i + 1 >= argc) {
                std::fprintf(stderr, "error: a value is required for '%s'\n", a.c_str());
                std::exit(2);
            }
            return argv[++i];
        };
        if (a == "-i" || a == "--iterations") iterations = std::atol(val());
        else if (a == "-e" || a == "--edges") edges = val();
        else if (a == "-n" || a == "--nodes") nodes = val();
        else if (a == "-r" || a == "--regions") bed = val();
        else if (a == "-p" || a == "--posterior-max-filter") filter = std::atof(val());
        else if (a == "-o" || a == "--output") output = val();
        else if (a == "--seed") seed = std::strtoull(val(), nullptr, 0);
        else if (a == "--device") device = std::atoi(val());
        else if (a == "--site-bootstrap") {
            site_boot = std::atoll(val());
            if (site_boot < 1) {
                std::fprintf(stderr, "error: --site-bootstrap needs a block size of at least one site\n");
                return 2;
            }
        } else if (a == "--devices") {
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
        } else if (a == "-h" || a == "--help") {
            std::printf("Usage: regions -n <NODES> -e <EDGES> -r <REGIONS.bed> [OPTIONS]\n\nOptions:\n"
                        "  -i, --iterations <N>           Random starts and bootstrap replicates per region [default: 100]\n"
                        "  -e, --edges <EDGES>            Relative or absolute path to an edgelist [default: ./edgelist.txt]\n"
                        "  -n, --nodes <NODES>            Relative or absolute path to a nodelist [default: ./nodelist.txt]\n"
                        "  -r, --regions <BED>            Regions, one per line: chromosome, 0-based start, end [, name, ...]\n"
                        "  -p, --posterior-max-filter <P> Minimum posterior probability for a basepair read [default: 0.99]\n"
                        "  -o, --output <OUTPUT>          Output directory, must exist [default: .]\n"
                        "      --seed <SEED>              Seed of the random starts and resamples [default: 0xAB0B200]\n"
                        "      --device <N>               CUDA device [default: 0]\n"
                        "      --devices <LIST>           Fit the regions on several devices, e.g. 0-7 or 0,2,5\n"
                        "      --site-bootstrap <SITES>   Bootstrap by resampling blocks of SITES consecutive sites (one device)\n");
            return 0;
        } else {
            std::fprintf(stderr, "error: unexpected argument '%s' found\n", a.c_str());
            return 2;
        }
    }
    if (bed.empty()) {
        std::fprintf(stderr, "error: the following required argument was not provided:\n  --regions <REGIONS.bed>\n");
        return 2;
    }
    for (const std::string *f : {&edges, &nodes, &bed})
        if (!exists(*f)) {
            std::fprintf(stderr, "error: Please provide a valid file path: %s does not exist.\n", f->c_str());
            return 2;
        }
    if (!exists(output)) {
        std::fprintf(stderr, "error: Please provide a valid output directory: %s does not exist.\n", output.c_str());
        return 2;
    }
    if (iterations <= 0) {
        std::fprintf(stderr, "error: --iterations must be positive\n");
        return 2;
    }
    if (site_boot > 0 && devices.size() > 1) {
        std::fprintf(stderr, "error: --site-bootstrap runs on one device; --devices names %zu\n", devices.size());
        return 2;
    }
    if (devices.empty()) devices.push_back(device);

    // ---- regions
    std::vector<Region> regs;
    {
        std::ifstream f(bed, std::ios::binary);
        std::string line;
        for (int64_t ln = 0; std::getline(f, line); ++ln) {
            Region r;
            const int rc = abfit_parse_region_line(line.c_str(), &r.chrom, &r.start0, &r.end);
            if (rc == 1) continue;
            if (rc) {
                std::printf("Error: %s line %lld: %s\n", bed.c_str(), (long long)ln + 1, abfit_last_error());
                return 1;
            }
            std::istringstream fs(line);
            std::string c, s, e, name;
            fs >> c >> s >> e >> name;
            r.chrom_text = c;
            r.name = name.empty() ? "." : name;
            r.line = ln;
            regs.push_back(r);
        }
    }
    const int32_t W = (int32_t)regs.size();
    if (W == 0) {
        std::printf("Error: %s holds no region\n", bed.c_str());
        return 1;
    }

    // ---- pedigree graph and sites
    int32_t S = 0, n_pairs = 0;
    if (abfit_pedigree_graph(nodes.c_str(), edges.c_str(), &S, nullptr, 0, &n_pairs, nullptr, 0)) {
        std::printf("Error: Error while building pedigree: %s\n", abfit_last_error());
        return 1;
    }
    if (S < 2 || n_pairs < 1) {
        std::printf("Error: Error while building pedigree: the nodelist has fewer than two measured samples\n");
        return 1;
    }
    std::vector<double> graph((size_t)n_pairs * 5);
    if (abfit_pedigree_graph(nodes.c_str(), edges.c_str(), &S, nullptr, 0, &n_pairs, graph.data(), n_pairs)) {
        std::printf("Error: Error while building pedigree: %s\n", abfit_last_error());
        return 1;
    }
    int64_t L = 0;
    std::vector<uint8_t> st;
    std::vector<double> po, me;
    std::vector<int32_t> pairs;
    std::vector<abfit_cg_site> sites;
    if (!read_sites(nodes, edges, n_pairs, S, L, st, po, me, pairs, "regions", &sites)) return 1;
    std::vector<int64_t> lo(W), hi(W);
    {
        std::vector<int32_t> ch(W);
        std::vector<int64_t> a(W), b(W);
        for (int32_t w = 0; w < W; ++w) {
            ch[w] = regs[w].chrom;
            a[w] = regs[w].start0;
            b[w] = regs[w].end;
        }
        if (abfit_region_ranges(sites.data(), (int64_t)sites.size(), ch.data(), a.data(), b.data(), W, lo.data(), hi.data())) {
            std::printf("Error: %s\n", abfit_last_error());
            return 1;
        }
    }

    std::vector<abfit_ctx *> ctxs(devices.size(), nullptr);
    for (size_t d = 0; d < devices.size(); ++d)
        if (abfit_ctx_create(devices[d], &ctxs[d])) {
            std::printf("Error: %s\n", abfit_last_error());
            return 1;
        }
    const int64_t P = (int64_t)S * (S - 1) / 2;
    std::vector<double> D((size_t)W * P), p0uu(W);
    if (abfit_region_divergence(ctxs[0], st.data(), po.data(), me.data(), S, L, lo.data(), hi.data(), W, filter, D.data(), nullptr,
                                nullptr, p0uu.data(), nullptr, nullptr)) {
        std::printf("Error: %s\n", abfit_last_error());
        return 1;
    }

    // ---- pedigree rows of every region; the fittable ones
    std::vector<std::string> why(W);
    std::vector<int32_t> fitted;  // region of every problem
    std::vector<double> peds;
    for (int32_t w = 0; w < W; ++w) {
        if (hi[w] == lo[w]) {
            why[w] = "no sites";
            continue;
        }
        const size_t off = peds.size();
        bool nan = false;
        for (int32_t q = 0; q < n_pairs; ++q) {
            const int64_t i = (int64_t)graph[5 * q], j = (int64_t)graph[5 * q + 1];
            const double d = D[(size_t)w * P + (size_t)(i * S - i * (i + 1) / 2 + (j - i - 1))];
            nan |= std::isnan(d);
            peds.insert(peds.end(), {graph[5 * q + 2], graph[5 * q + 3], graph[5 * q + 4], d});
        }
        if (nan || std::isnan(p0uu[w])) {
            why[w] = nan ? "pair without valid sites" : "sample without valid sites";
            peds.resize(off);
            continue;
        }
        fitted.push_back(w);
    }
    const int F = (int)fitted.size();
    const int n = (int)iterations;
    std::vector<abfit_problem> probs(F);
    std::vector<uint64_t> ids(F);
    std::unique_ptr<double[]> simplices(new double[std::max<size_t>(1, (size_t)F * n * 20)]);
    for (int f = 0; f < F; ++f) {
        const int32_t w = fitted[f];
        const double *ped = peds.data() + (size_t)f * n_pairs * 4;
        probs[f] = abfit_problem{ped, n_pairs, p0uu[w], p0uu[w], 1.0};  // eqp = p0uu, eqp_weight = 1 (src/alphabeta.rs:33-37)
        ids[f] = (uint64_t)regs[w].line;
        double max_div = ped[3];
        for (int32_t q = 1; q < n_pairs; ++q) max_div = std::max(max_div, ped[4 * q + 3]);  // src/ab_neutral.rs:25-29
        abfit_gen_start_simplices(seed, ids[f], n, max_div, simplices.get() + (size_t)f * n * 20);
    }
    std::vector<abfit_fit> best(F);
    std::vector<int32_t> status(F);
    std::vector<double> rows((size_t)F * n * 7), analysis((size_t)F * 32);
    std::printf("Regions: %d in %s, %d fitted, %d samples, %lld sites\n", W, bed.c_str(), F, S, (long long)L);
    if (F > 0 && site_boot > 0) {
        std::vector<int64_t> fseg(F + 1, 0);
        for (int f = 0; f < F; ++f) fseg[f + 1] = fseg[f] + hi[fitted[f]] - lo[fitted[f]];
        const int64_t LF = fseg[F];
        std::vector<uint8_t> fst((size_t)S * LF);
        std::vector<double> fpo((size_t)S * LF), fme((size_t)S * LF);
        for (int32_t s = 0; s < S; ++s)
            for (int f = 0; f < F; ++f) {
                const int32_t w = fitted[f];
                const size_t src = (size_t)s * L + lo[w], dst = (size_t)s * LF + fseg[f], len = hi[w] - lo[w];
                std::copy_n(st.begin() + src, len, fst.begin() + dst);
                std::copy_n(po.begin() + src, len, fpo.begin() + dst);
                std::copy_n(me.begin() + src, len, fme.begin() + dst);
            }
        std::vector<int32_t> rp((size_t)F * n_pairs * 2);
        for (int f = 0; f < F; ++f)
            for (int32_t q = 0; q < n_pairs; ++q) {
                rp[((size_t)f * n_pairs + q) * 2] = pairs[2 * q];
                rp[((size_t)f * n_pairs + q) * 2 + 1] = pairs[2 * q + 1];
            }
        std::vector<int32_t> nan_reps(F);
        if (abfit_fit_batch(ctxs[0], probs.data(), F, n, simplices.get(), 10000, DBL_EPSILON, 0, best.data(), nullptr, nullptr,
                            nullptr, status.data()) ||
            abfit_site_boot_batch(ctxs[0], probs.data(), F, rp.data(), fst.data(), fpo.data(), fme.data(), S, LF, fseg.data(), filter,
                                  site_boot, best.data(), n, seed, 0, ids.data(), 1000, DBL_EPSILON, 0, rows.data(), nullptr,
                                  analysis.data(), nullptr, nan_reps.data())) {
            std::printf("Error: %s\n", abfit_last_error());
            return 1;
        }
        for (int f = 0; f < F; ++f)
            if (nan_reps[f])
                std::printf("Site bootstrap: region %s (line %lld): %d of %d replicates left a pair without valid sites (NaN rows)\n",
                            regs[fitted[f]].name.c_str(), (long long)regs[fitted[f]].line + 1, nan_reps[f], n);
    } else if (F > 0 && abfit_alphabeta_batch_multi(ctxs.data(), (int32_t)ctxs.size(), probs.data(), F, n, simplices.get(), n, nullptr,
                                                    seed, 0, ids.data(), 10000, 1000, DBL_EPSILON, 0, best.data(), nullptr, nullptr,
                                                    status.data(), rows.data(), analysis.data())) {
        std::printf("Error: %s\n", abfit_last_error());
        return 1;
    }

    // ---- regions.tsv, raw.npy
    std::vector<int> fit_of(W, -1);
    for (int f = 0; f < F; ++f) {
        if (status[f] != 0) why[fitted[f]] = "fit failed";
        else fit_of[fitted[f]] = f;
    }
    std::string tsv = "name\tchromosome\tstart\tend\tsites\tp0uu\talpha\tbeta\tweight\tintercept\talpha_sd\talpha_lo\talpha_hi\t"
                      "beta_sd\tbeta_lo\tbeta_hi\tstatus\n";
    std::vector<double> raw;
    const double nan = std::nan("");
    for (int32_t w = 0; w < W; ++w) {
        const Region &r = regs[w];
        const int f = fit_of[w];
        double v[10];
        for (double &x : v) x = nan;
        if (f >= 0) {
            const abfit_fit &b = best[f];
            const double *a = analysis.data() + (size_t)f * 32;  // means, sds, (q0.025, q0.975): alpha, beta, ...
            const double vv[10] = {b.theta[0], b.theta[1], b.theta[2], b.theta[3], a[8], a[16], a[17], a[9], a[18], a[19]};
            std::copy(vv, vv + 10, v);
            raw.insert(raw.end(), rows.begin() + (size_t)f * n * 7, rows.begin() + (size_t)(f + 1) * n * 7);
        }
        tsv += r.name + "\t" + r.chrom_text + "\t" + std::to_string(r.start0) + "\t" + std::to_string(r.end) + "\t" +
               std::to_string(hi[w] - lo[w]) + "\t" + f64s(hi[w] > lo[w] ? p0uu[w] : nan);
        for (double x : v) tsv += "\t" + f64s(x);
        tsv += "\t" + (f >= 0 ? std::string("ok") : why[w]) + "\n";
    }
    const std::string tp = output + "/regions.tsv", rp = output + "/raw.npy";
    std::printf("Writing regions to file: %s\n", tp.c_str());
    FILE *fo = std::fopen(tp.c_str(), "wb");
    if (!fo || std::fwrite(tsv.data(), 1, tsv.size(), fo) != tsv.size()) {
        std::printf("Error: could not write %s\n", tp.c_str());
        return 1;
    }
    std::fclose(fo);
    std::printf("Writing bootstrap rows to file: %s\n", rp.c_str());
    const int64_t shape[3] = {(int64_t)(raw.size() / ((size_t)n * 7)), n, 7};
    if (abfit_write_npy_f64(rp.c_str(), raw.data(), 3, shape)) {
        std::printf("Error: %s\n", abfit_last_error());
        return 1;
    }
    for (abfit_ctx *c : ctxs) abfit_ctx_destroy(c);
    return 0;
}
