// abfit_rng.h — the counter-based generator behind the seeded inputs (start simplices, vary vertices, resample
// indices).  One definition for host and device: the vary vertices of abfit_alphabeta_batch are drawn on the GPU
// (they depend on each window's best fit, which is already there) and must be the very numbers the host entry
// point abfit_gen_vary_vertices returns.  Integer hashing and IEEE double operations only (device code is built
// with -fmad=false, host code with -ffp-contract=off), so both sides produce the same bits.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define ABFIT_HD __host__ __device__
#else
#define ABFIT_HD
#endif

namespace abfit {

ABFIT_HD inline uint64_t mix64(uint64_t z)
{
    z += 0x9e3779b97f4a7c15ull;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}
ABFIT_HD inline double u01(uint64_t seed, uint64_t stream, uint64_t problem, uint64_t item, uint64_t sub)
{
    uint64_t h = mix64(seed ^ (stream * 0xd1342543de82ef95ull));
    h = mix64(h ^ problem);
    h = mix64(h ^ item);
    h = mix64(h ^ sub);
    return (double)(h >> 11) * (1.0 / 9007199254740992.0);  // [0,1)
}
ABFIT_HD inline double uniform(double lo, double hi, double u) { return lo + (hi - lo) * u; }

// Model::vary (src/structs.rs:100-128): coordinate j of vary vertex v of replicate b around best_j
ABFIT_HD inline double vary_coordinate(uint64_t seed, uint64_t problem_id, uint64_t b, int v, int j, double best_j)
{
    double n = best_j;
    if (n == 0.0) n = 0.1;  // src/structs.rs:105-108
    const double a = n < 0.0 ? -n : n;
    double lo = n - a * 0.1, hi = n + a * 0.1;
    if (lo >= hi) {  // src/structs.rs:113-115
        const double t = lo;
        lo = hi;
        hi = t;
    }
    return uniform(lo, hi, u01(seed, 2, problem_id, b, (uint64_t)(v * 4 + j)));
}

// site-block bootstrap: draw d of replicate b picks one of the window's n_blocks blocks (stream 5; streams 1-3 are
// starts, vary vertices and resamples, 4 the simulator)
ABFIT_HD inline int32_t site_boot_block(uint64_t seed, uint64_t problem_id, uint64_t b, uint64_t d, int32_t n_blocks)
{
    int32_t k = (int32_t)(u01(seed, 5, problem_id, b, d) * (double)n_blocks);
    if (k >= n_blocks) k = n_blocks - 1;
    return k;
}

// parametric bootstrap: the simulator seed of replicate b of window problem_id (stream 6)
ABFIT_HD inline uint64_t param_boot_seed(uint64_t seed, uint64_t problem_id, uint64_t b)
{
    uint64_t h = mix64(seed ^ (6 * 0xd1342543de82ef95ull));
    h = mix64(h ^ problem_id);
    return mix64(h ^ b);
}

}  // namespace abfit
