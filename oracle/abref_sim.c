/*
 * abref_sim.c — CPU ORACLE of the ABneutral methylome simulation (test infrastructure only, like abref.c, whose
 * abref_genmatrix / abref_matrix_power it uses; built with abref.c into one library by abref_sim_py.py).
 *
 * Model, on a forest (parent[v] = -1 for roots, gen(parent) <= gen(v) <= 127): a root at generation g draws its state
 * from sv0.G^g, sv0 = [p0uu, w(1-p0uu), (1-w)(1-p0uu)]; a child draws from row state(parent) of
 * G^(gen(child) - gen(parent)) (abref_matrix_power's chain; the 1x3 . 3x3 product is the FMA chain of divergence()).
 * thresholds [n][6]: per parent state k the pair (r0, r0 + r1) of the row; a root stores its pair three times.
 * Draw of node v at global site i: u = top 53 bits of splitmix64(key ^ i) / 2^53, with
 * key = mix(mix(mix(seed ^ 4 * 0xd1342543de82ef95) ^ v) ^ which), which = 0 (state) or 1 (missingness);
 * state = u < c0 ? 0 : u < c1 ? 1 : 2.  Outputs [n_sampled][L], rows in node order: status, posterior_max = 1
 * (0.5 when the missingness draw < missing_rate), meth_lvl = status / 2.
 *
 * Build: gcc -O2 -std=c11 -ffp-contract=off -fPIC -shared abref.c abref_sim.c -lm
 */
#include <stdint.h>
#include <stdlib.h>

#include "abref.h"

void abref_sim_thresholds(int n, const int32_t *parent, const int32_t *gen, double alpha, double beta, double weight,
                          double p0uu, double *out);
void abref_simulate(int n, const int32_t *parent, const int32_t *gen, const uint8_t *sampled, double alpha, double beta,
                    double weight, double p0uu, double missing_rate, uint64_t seed, int64_t first_site, int64_t L,
                    uint8_t *status, double *posterior_max, double *meth_lvl);

/* 1x3 . 3x3 as abref.c's vec3_mat3: a*b, then two fused multiply-adds (correctly rounded in hardware or software) */
static void vec3_mat3(const double v[3], const double M[9], double out[3])
{
    for (int j = 0; j < 3; ++j) {
        double acc = v[0] * M[j];
        acc = __builtin_fma(v[1], M[3 + j], acc);
        out[j] = __builtin_fma(v[2], M[6 + j], acc);
    }
}
static uint64_t sim_mix64(uint64_t z)
{
    z += 0x9e3779b97f4a7c15ull;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

static uint64_t sim_key(uint64_t seed, int node, uint64_t which)
{
    uint64_t h = sim_mix64(seed ^ (4ull * 0xd1342543de82ef95ull));
    h = sim_mix64(h ^ (uint64_t)node);
    return sim_mix64(h ^ which);
}

static double sim_u01(uint64_t key, uint64_t site) { return (double)(sim_mix64(key ^ site) >> 11) * (1.0 / 9007199254740992.0); }

void abref_sim_thresholds(int n, const int32_t *parent, const int32_t *gen, double alpha, double beta, double weight,
                          double p0uu, double *out)
{
    double G[9], P[9];
    abref_genmatrix(alpha, beta, G);
    const double p_mm = 1.0 - p0uu;
    const double sv0[3] = {p0uu, weight * p_mm, (1.0 - weight) * p_mm};
    for (int v = 0; v < n; ++v) {
        double *c = out + 6 * (size_t)v;
        if (parent[v] < 0) {
            double s[3];
            abref_matrix_power(G, gen[v], P);
            vec3_mat3(sv0, P, s);
            for (int k = 0; k < 3; ++k) {
                c[2 * k] = s[0];
                c[2 * k + 1] = s[0] + s[1];
            }
        } else {
            abref_matrix_power(G, gen[v] - gen[parent[v]], P);
            for (int k = 0; k < 3; ++k) {
                c[2 * k] = P[3 * k];
                c[2 * k + 1] = P[3 * k] + P[3 * k + 1];
            }
        }
    }
}

void abref_simulate(int n, const int32_t *parent, const int32_t *gen, const uint8_t *sampled, double alpha, double beta,
                    double weight, double p0uu, double missing_rate, uint64_t seed, int64_t first_site, int64_t L,
                    uint8_t *status, double *posterior_max, double *meth_lvl)
{
    double *thr = malloc(sizeof(double) * 6 * (size_t)(n > 0 ? n : 1));
    uint64_t *ks = malloc(sizeof(uint64_t) * 2 * (size_t)(n > 0 ? n : 1));
    int *depth = malloc(sizeof(int) * (size_t)(n > 0 ? n : 1)), *row = malloc(sizeof(int) * (size_t)(n > 0 ? n : 1));
    uint8_t *st = malloc((size_t)(n > 0 ? n : 1));
    abref_sim_thresholds(n, parent, gen, alpha, beta, weight, p0uu, thr);
    int max_depth = 0, n_rows = 0;
    for (int v = 0; v < n; ++v) {
        ks[2 * v] = sim_key(seed, v, 0);
        ks[2 * v + 1] = sim_key(seed, v, 1);
        int d = 0;
        for (int u = parent[v]; u >= 0; u = parent[u]) ++d;
        depth[v] = d;
        if (d > max_depth) max_depth = d;
        row[v] = sampled[v] ? n_rows++ : -1;
    }
    for (int64_t k = 0; k < L; ++k) {
        const uint64_t site = (uint64_t)(first_site + k);
        for (int d = 0; d <= max_depth; ++d) /* parents before children */
            for (int v = 0; v < n; ++v) {
                if (depth[v] != d) continue;
                const int ps = parent[v] < 0 ? 0 : st[parent[v]];
                const double u = sim_u01(ks[2 * v], site);
                const double *c = thr + 6 * (size_t)v + 2 * ps;
                const int s = u < c[0] ? 0 : u < c[1] ? 1 : 2;
                st[v] = (uint8_t)s;
                if (row[v] >= 0) {
                    const size_t o = (size_t)row[v] * (size_t)L + (size_t)k;
                    status[o] = (uint8_t)s;
                    posterior_max[o] = sim_u01(ks[2 * v + 1], site) < missing_rate ? 0.5 : 1.0;
                    meth_lvl[o] = (double)s * 0.5;
                }
            }
    }
    free(thr);
    free(ks);
    free(depth);
    free(row);
    free(st);
}
