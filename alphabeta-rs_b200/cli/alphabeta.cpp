// alphabeta — command-line front end with the flags, console block and output files of the reference's
// `alphabeta` binary (src/cli/alphabeta.rs:8-38, src/arguments.rs:96-114, src/alphabeta.rs:23-59), on top of libabfit.
//
//   alphabeta -n nodelist.txt -e edgelist.txt [-i 1000] [-p 0.99] [-o .] [--seed N] [--device 0 | --devices 0-7]
//             [--site-bootstrap BLOCK_SITES | --parametric-bootstrap N]
//
// --site-bootstrap replaces the reference's residual bootstrap with the site-block bootstrap (abfit_site_boot_batch): the
// replicates resample blocks of BLOCK_SITES consecutive sites of the methylome files, and the output files are written
// from those rows.
// --parametric-bootstrap replaces it with N replicates simulated from the fitted model on the pedigree forest of the same
// nodelist and edgelist, with the methylomes' number of sites and each sample's share of missing sites
// (abfit_param_boot_batch); the output files are written from those rows, and goodness_of_fit.txt ranks the observed LSE
// among the replicates' (a p-value of the model's fit).
//
// Differences that are deliberate: the random starts / resamples come from a seed (default 0xAB0B200,
// `--seed` is an extra flag; the reference uses an unseeded thread_rng), the two progress bars advance per stage
// of the batched call instead of per start (cli/progress.h), bootstrap.png is drawn by the library's own rasteriser
// (same content as src/plot.rs:84-137, not the same pixels), and a window on which the reference panics reports an
// error instead.
#include <cfloat>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <sys/stat.h>
#include <vector>

#include "../../include/abfit.h"
#include "progress.h"
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

int main(int argc, char **argv)
{
    long iterations = 1000;
    std::string edges = "./edgelist.txt", nodes = "./nodelist.txt", output = ".";
    double filter = 0.99;
    unsigned long long seed = 0xAB0B200ull;
    int device = 0;
    long long site_boot = 0;  // 0: the residual bootstrap of the reference
    long param_boot = 0;      // replicates of the parametric bootstrap, 0: none
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto val = [&](const char *name) -> const char * {
            if (i + 1 >= argc) {
                std::fprintf(stderr, "error: a value is required for '%s'\n", name);
                std::exit(2);
            }
            return argv[++i];
        };
        if (a == "-i" || a == "--iterations") iterations = std::atol(val("--iterations"));
        else if (a == "-e" || a == "--edges") edges = val("--edges");
        else if (a == "-n" || a == "--nodes") nodes = val("--nodes");
        else if (a == "-p" || a == "--posterior-max-filter") filter = std::atof(val("--posterior-max-filter"));
        else if (a == "-o" || a == "--output") output = val("--output");
        else if (a == "--seed") seed = std::strtoull(val("--seed"), nullptr, 0);
        else if (a == "--device") device = std::atoi(val("--device"));
        else if (a == "--site-bootstrap") {
            site_boot = std::atoll(val("--site-bootstrap"));
            if (site_boot < 1) {
                std::fprintf(stderr, "error: --site-bootstrap needs a block size of at least one site\n");
                return 2;
            }
        }
        else if (a == "--parametric-bootstrap") {
            param_boot = std::atol(val("--parametric-bootstrap"));
            if (param_boot < 1 || param_boot > 65535) {
                std::fprintf(stderr, "error: --parametric-bootstrap needs between 1 and 65535 replicates\n");
                return 2;
            }
        }
        else if (a == "--devices") device = std::atoi(val("--devices"));  // one pedigree = one window: its starts and replicates stay on the first listed GPU
        else if (a == "-h" || a == "--help") {
            std::printf("Usage: alphabeta [OPTIONS]\n\nOptions:\n"
                        "  -i, --iterations <ITERATIONS>  Number of iterations to run for Nelder-Mead optimization [default: 1000]\n"
                        "  -e, --edges <EDGES>            Relative or absolute path to an edgelist [default: ./edgelist.txt]\n"
                        "  -n, --nodes <NODES>            Relative or absolute path to a nodelist [default: ./nodelist.txt]\n"
                        "  -p, --posterior-max-filter <P> Minimum posterior probability for a basepair read [default: 0.99]\n"
                        "  -o, --output <OUTPUT>          Output directory, must exist [default: .]\n"
                        "      --seed <SEED>              Seed of the random starts and resamples [default: 0xAB0B200]\n"
                        "      --device <N>               CUDA device [default: 0]\n"
                        "      --site-bootstrap <SITES>   Bootstrap by resampling blocks of SITES consecutive sites instead of pair residuals\n"
                        "      --parametric-bootstrap <N> Bootstrap by N data sets simulated from the fitted model; adds goodness_of_fit.txt\n");
            return 0;
        } else {
            std::fprintf(stderr, "error: unexpected argument '%s' found\n", a.c_str());
            return 2;
        }
    }
    // validators of src/arguments.rs:116-140
    for (const std::string *f : {&edges, &nodes}) {
        if (!exists(*f)) {
            std::fprintf(stderr, "error: Please provide a valid file path. By default, we fill try %s, which does not exist.\n", f->c_str());
            return 2;
        }
        std::printf("Using default file: %s\n", f->c_str());
    }
    if (!exists(output)) {
        std::fprintf(stderr, "error: Please provide a valid output directory. By default, we fill try %s, which does not exist.\n", output.c_str());
        return 2;
    }
    if (iterations <= 0) {
        std::fprintf(stderr, "error: --iterations must be positive\n");
        return 2;
    }
    if (site_boot > 0 && param_boot > 0) {
        std::fprintf(stderr, "error: --site-bootstrap and --parametric-bootstrap cannot be used together\n");
        return 2;
    }
    abfit_sim_tree *tree = nullptr;  // the pedigree forest the parametric bootstrap simulates on
    if (param_boot > 0 && abfit_sim_tree_build(nodes.c_str(), edges.c_str(), &tree)) {
        std::printf("Error: --parametric-bootstrap: %s\n", abfit_last_error());
        return 1;
    }
    abfit_ctx *ctx = nullptr;
    if (abfit_ctx_create(device, &ctx)) {
        std::printf("Error: %s\n", abfit_last_error());
        return 1;
    }
    std::printf("Building pedigree...\n");
    abfit_pedigree *ped = nullptr;
    if (abfit_pedigree_build(ctx, nodes.c_str(), edges.c_str(), filter, &ped)) {
        std::printf("Error: Error while building pedigree: %s\n", abfit_last_error());
        return 1;
    }
    std::fputs(abfit_pedigree_warnings(ped), stdout);
    int32_t n_pairs = 0;
    double p0uu = 0.0;
    abfit_pedigree_info(ped, &n_pairs, &p0uu, nullptr, nullptr);
    const double *rows = abfit_pedigree_rows(ped);
    if (n_pairs <= 0) {
        std::printf("Error: Model failed: the pedigree has no pairs\n");
        return 1;
    }
    double max_div = rows[3];
    for (int i = 1; i < n_pairs; ++i) max_div = rows[4 * i + 3] > max_div ? rows[4 * i + 3] : max_div;  // src/ab_neutral.rs:25-29
    const int n = (int)iterations;
    const int n_boot = param_boot > 0 ? (int)param_boot : n;
    std::vector<double> simplices((size_t)n * 20), rows_out((size_t)n_boot * 7), pred(n_pairs), resid(n_pairs), analysis(32);
    std::vector<int32_t> idx((size_t)n * n_pairs);
    abfit_gen_start_simplices(seed, 0, n, max_div, simplices.data());
    abfit_gen_resample_idx(seed, 0, n, n_pairs, idx.data());
    abfit_problem prob{rows, n_pairs, p0uu, p0uu, 1.0};  // eqp = p0uu, eqp_weight = 1 (src/alphabeta.rs:33-37)
    abfit_fit best;
    int32_t status = 0;
    progress::Bar pb_neutral("ABNeutral", (unsigned long long)n, false), pb_boot("BootModel", (unsigned long long)n_boot, false);  // src/progress.rs:5-23
    pb_neutral.tick();
    int rc = 0;
    double gof_p = 0.0;
    int32_t gof_fitted = 0, gof_nan = 0;
    if (param_boot > 0) {
        // fit as abfit_alphabeta_batch does, then replicates of the fitted model with the methylomes' design
        int32_t S = 0;
        int64_t L = 0;
        std::vector<uint8_t> st;
        std::vector<double> po, me;
        std::vector<int32_t> pairs;
        if (!read_sites(nodes, edges, n_pairs, S, L, st, po, me, pairs, "--parametric-bootstrap")) return 1;
        if (L <= 0) {
            std::printf("Error: --parametric-bootstrap: the methylome files hold no sites\n");
            return 1;
        }
        std::vector<double> missing(S);
        for (int32_t s = 0; s < S; ++s) {
            int64_t nvalid = 0;
            for (int64_t k = 0; k < L; ++k) nvalid += po[(size_t)s * L + k] >= filter ? 1 : 0;
            missing[s] = 1.0 - (double)nvalid / (double)L;
        }
        rc = abfit_fit_batch(ctx, &prob, 1, n, simplices.data(), 10000, DBL_EPSILON, 0, &best, nullptr, nullptr, nullptr, &status);
        std::vector<abfit_fit> fits(n_boot);
        int32_t wstat = 0;
        if (!rc && !status)
            rc = abfit_param_boot_batch(ctx, tree, &prob, 1, &L, missing.data(), filter, &best, n_boot, seed, 0, nullptr, 1000,
                                        DBL_EPSILON, 0, rows_out.data(), fits.data(), analysis.data(), nullptr, nullptr,
                                        &gof_p, &wstat, &gof_nan);
        if (!rc && !status && wstat) {
            std::printf("Error: Model failed: the fitted alpha, beta or weight lie outside [0, 1], so the model cannot be simulated\n");
            return 1;
        }
        for (const abfit_fit &f : fits) gof_fitted += f.status != ABFIT_FIT_NAN ? 1 : 0;
    } else if (site_boot > 0) {
        // fit as abfit_alphabeta_batch does, then the site-block bootstrap on the methylomes' own sites
        int32_t S = 0;
        int64_t L = 0;
        std::vector<uint8_t> st;
        std::vector<double> po, me;
        std::vector<int32_t> pairs;
        if (!read_sites(nodes, edges, n_pairs, S, L, st, po, me, pairs)) return 1;
        rc = abfit_fit_batch(ctx, &prob, 1, n, simplices.data(), 10000, DBL_EPSILON, 0, &best, nullptr, nullptr, nullptr, &status);
        const int64_t seg[2] = {0, L};
        int32_t nan_reps = 0;
        if (!rc && !status)
            rc = abfit_site_boot_batch(ctx, &prob, 1, pairs.data(), st.data(), po.data(), me.data(), S, L, seg, filter, site_boot,
                                       &best, n, seed, 0, nullptr, 1000, DBL_EPSILON, 0, rows_out.data(), nullptr, analysis.data(),
                                       nullptr, &nan_reps);
        if (!rc && nan_reps)
            std::printf("Site bootstrap: %d of %d replicates left a pair without valid sites (NaN rows)\n", nan_reps, n);
    } else {
        rc = abfit_alphabeta_batch(ctx, &prob, 1, n, simplices.data(), n, idx.data(), seed, 0, 10000, 1000, DBL_EPSILON, 0, &best,
                                   pred.data(), resid.data(), &status, rows_out.data(), analysis.data());
    }
    if (rc || status) {
        std::printf("Error: Model failed: %s\n", rc ? abfit_last_error() : "NaN in the pedigree or in every fit (the reference panics here)");
        return 1;
    }
    pb_neutral.finish();
    pb_boot.finish();
    char text[8192];
    abfit_format_analysis(analysis.data(), text, sizeof text);
    std::printf("##########\nResults:\n\n");
    std::printf("Model:\n\tAlpha: %s\n\tBeta: %s\n\tWeight: %s\n\tIntercept: %s\n", f64s(best.theta[0]).c_str(), f64s(best.theta[1]).c_str(),
                f64s(best.theta[2]).c_str(), f64s(best.theta[3]).c_str());
    std::printf("%s\n", text);
    std::printf("Estimated steady state %s\n", f64s(abfit_steady_state(best.theta[0], best.theta[1])).c_str());
    std::printf("Observed steady state methylation %s\n", f64s(1.0 - p0uu).c_str());
    std::printf("##########\n");
    const std::string pp = output + "/pedigree.txt", ap = output + "/analysis.txt", rp = output + "/raw.npy";
    std::printf("Writing pedigree to file: %s\n", pp.c_str());
    std::printf("Writing model to file: %s\n", ap.c_str());
    const int64_t shape[2] = {n_boot, 7};
    if (abfit_write_pedigree(pp.c_str(), rows, n_pairs) || abfit_write_analysis(ap.c_str(), analysis.data()) ||
        abfit_write_npy_f64(rp.c_str(), rows_out.data(), 2, shape)) {
        std::printf("Error: %s\n", abfit_last_error());
        return 1;
    }
    if (param_boot > 0) {
        const std::string gp = output + "/goodness_of_fit.txt";
        std::printf("Goodness of fit: p = %s (observed LSE %s, %d replicates fitted, %d NaN replicates)\n", f64s(gof_p).c_str(),
                    f64s(best.lse).c_str(), gof_fitted, gof_nan);
        std::printf("Writing goodness of fit to file: %s\n", gp.c_str());
        std::ofstream g(gp);
        g << "observed_lse\t" << f64s(best.lse) << "\np\t" << f64s(gof_p) << "\nreplicates_fitted\t" << gof_fitted
          << "\nnan_replicates\t" << gof_nan << "\n";
        if (!g) {
            std::printf("Error: cannot write %s\n", gp.c_str());
            return 1;
        }
    }
    {  // plot::bootstrap(results.column(0), results.column(1), output_dir)  (src/boot_model.rs:105-109)
        std::vector<double> alphas(n_boot), betas(n_boot);
        for (int i = 0; i < n_boot; ++i) {
            alphas[i] = rows_out[(size_t)i * 7];
            betas[i] = rows_out[(size_t)i * 7 + 1];
        }
        if (abfit_plot_bootstrap((output + "/bootstrap.png").c_str(), alphas.data(), betas.data(), n_boot)) {
            std::printf("Error: %s\n", abfit_last_error());
            return 1;
        }
    }
    abfit_pedigree_free(ped);
    abfit_sim_tree_free(tree);
    abfit_ctx_destroy(ctx);
    return 0;
}
