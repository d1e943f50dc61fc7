// abfit_divergence.cu — observed pairwise methylation divergence + per-sample methylation level.
//
// Replaces DMatrix::from (src/pedigree.rs:213-262) and the valid-site statistics of
// Pedigree::build (src/pedigree.rs:159-183), batched over windows (site segments).
//
// HBM-bound design (SURVEY.md §8d: 17 bytes per sample-site are algorithmic):
//   pass 1  k_pack      streams posteriorMax (f64), rc.meth.lvl (f64) and status (u8) ONCE, fully
//                       coalesced on the site axis, and emits three bit-planes per sample —
//                       valid = post >= thr, t1 = status >= 1, t2 = status >= 2 (thermometer code,
//                       |a-b| = popc(t1a^t1b) + popc(t2a^t2b)) — plus blocked partial sums of
//                       meth_lvl over valid sites.  3 bits/site leave HBM again (2 % of the input).
//   pass 2  k_pairs     all-pairs popcount over the bit-planes staged in shared memory, 4 x 4 sample tiles
//                       in registers (POPC-bound); exact u64
//                       sums, so D = diff / (2 cnt) is bit-identical to the reference for any
//                       sharding of the site axis.
//   pass 3  k_finalize  D = diff/(2 cnt), per-sample methsum / nvalid, p0uu per window.
#include "abfit_internal.h"

namespace abfit {

constexpr int SB_WORDS = 64;           // words (64 sites) per super-block = one warp's share in k_pack
constexpr int64_t EXACT_MAX = 65536;   // windows up to this many sites: sequential (bit-exact) methsum
constexpr int FIN_WARPS = 4;           // warps per block of the per-sample finalisation kernels

struct SuperBlock {
    int32_t window;
    int32_t n_words;      // <= SB_WORDS
    int64_t first_word;   // global packed word index
    int64_t first_site;   // site index on the L axis
    int64_t end_site;     // end of the window
};

// pass 1 ------------------------------------------------------------------------------
// 56 registers: two 128-thread blocks fit in the 14 K registers a k_pairs block leaves free on an SM
__global__ void __maxnreg__(56)
k_pack(const uint8_t *__restrict__ status, const double *__restrict__ post, const double *__restrict__ meth,
       int64_t L, int64_t total_words, const SuperBlock *__restrict__ sbs, int n_sb, int sb_first, int sb_end, int S,
       double thr, unsigned long long *__restrict__ V, unsigned long long *__restrict__ T1,
       unsigned long long *__restrict__ T2, double *__restrict__ methpart, long long *__restrict__ nvpart)
{
    // Work unit = one super-block of one sample; units of this launch: super-blocks [sb_first, sb_end) x S samples,
    // unit u = sample u / n_sbc, super-block sb_first + u % n_sbc (consecutive warps read consecutive memory).  A
    // launch either has a warp per unit, or — the overlapped mode of run_divergence, where the pair pass of one chunk
    // of sites runs while the next chunk is being packed — a fixed number of blocks per SM that loop over the units,
    // so that the packing never takes more of an SM than the registers the pair kernel leaves free.
    const int lane = threadIdx.x & 31;
    const int n_sbc = sb_end - sb_first;
    const long long n_units = (long long)n_sbc * S;
    const long long n_warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long u = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; u < n_units; u += n_warps) {
    const int s = (int)(u / n_sbc);
    const int warp = sb_first + (int)(u - (long long)s * n_sbc);
    const SuperBlock sb = sbs[warp];
    const uint8_t *st = status + (size_t)s * L;
    const double *po = post + (size_t)s * L;
    const double *me = meth + (size_t)s * L;
    unsigned long long *Vs = V + (size_t)s * total_words + sb.first_word;
    unsigned long long *T1s = T1 + (size_t)s * total_words + sb.first_word;
    unsigned long long *T2s = T2 + (size_t)s * total_words + sb.first_word;

    double acc = 0.0;  // lane-local, in site order within the lane
    int nv = 0;
    // Lane l owns the two adjacent sites 2l, 2l+1 of every 64-site word, so one 16-byte load per lane and
    // array covers the word (512 contiguous bytes per warp request).  Bit b < 32 of a packed word is site 2b,
    // bit 32 + b is site 2b + 1: any fixed permutation of the sites inside a word is as good as any other for
    // the popcounts of pass 2, as long as every sample and plane uses the same one.
    const bool vec = ((reinterpret_cast<uintptr_t>(po + sb.first_site) | reinterpret_cast<uintptr_t>(me + sb.first_site)) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(st + sb.first_site) & 1) == 0;
#pragma unroll 4
    for (int w = 0; w < sb.n_words; ++w) {
        const int64_t i0 = sb.first_site + (int64_t)w * 64 + 2 * lane, i1 = i0 + 1;
        const bool in0 = i0 < sb.end_site, in1 = i1 < sb.end_site;
        double p0 = -1.0, p1 = -1.0, m0 = 0.0, m1 = 0.0;
        int s0 = 0, s1 = 0;
        if (vec && in1) {
            const double2 pp = __ldcs(reinterpret_cast<const double2 *>(po + i0));
            const double2 mm = __ldcs(reinterpret_cast<const double2 *>(me + i0));
            const unsigned short ss = __ldcs(reinterpret_cast<const unsigned short *>(st + i0));
            p0 = pp.x; p1 = pp.y; m0 = mm.x; m1 = mm.y;
            s0 = ss & 0xff; s1 = ss >> 8;
        } else {
            if (in0) { p0 = __ldcs(po + i0); m0 = __ldcs(me + i0); s0 = (int)__ldcs(st + i0); }
            if (in1) { p1 = __ldcs(po + i1); m1 = __ldcs(me + i1); s1 = (int)__ldcs(st + i1); }
        }
        const bool v0 = in0 && (p0 >= thr), v1 = in1 && (p1 >= thr);
        const unsigned bv0 = __ballot_sync(FULL, v0), bv1 = __ballot_sync(FULL, v1);
        const unsigned b10 = __ballot_sync(FULL, s0 >= 1), b11 = __ballot_sync(FULL, s1 >= 1);
        const unsigned b20 = __ballot_sync(FULL, s0 >= 2), b21 = __ballot_sync(FULL, s1 >= 2);
        if (v0) { acc += m0; ++nv; }
        if (v1) { acc += m1; ++nv; }
        if (lane == 0) {
            Vs[w] = (unsigned long long)bv0 | ((unsigned long long)bv1 << 32);
            T1s[w] = (unsigned long long)b10 | ((unsigned long long)b11 << 32);
            T2s[w] = (unsigned long long)b20 | ((unsigned long long)b21 << 32);
        }
    }
    // fixed-shape tree over lanes: deterministic for a given (L, segmentation)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        acc += __shfl_down_sync(FULL, acc, o);
        nv += __shfl_down_sync(FULL, nv, o);
    }
    if (lane == 0) {
        methpart[(size_t)s * n_sb + warp] = acc;
        nvpart[(size_t)s * n_sb + warp] = nv;
    }
    }  // units
}

// pass 2 ------------------------------------------------------------------------------
struct PairItem {
    int32_t window;
    int32_t n_words;     // words of this chunk
    int64_t first_word;  // global packed word index
    int32_t single;      // 1: the only chunk of its window -> plain store, else atomicAdd
    int32_t pad;
};

// Register-tiled all-pairs popcount.  A thread owns up to two 4 x 4 tiles of the (i, j) sample matrix (16 pairs
// each, upper triangle incl. the diagonal blocks): per 64-site word it reads the three bit-planes of its 4 row
// samples (6 x 16-byte loads, a broadcast inside a warp, whose lanes share the row block) and of its 4 column
// samples, and updates 16 packed counters (cnt << 16 | diff: an item has at most 256 words, so diff <= 32 768 and
// cnt <= 16 384).  0.75 shared-memory loads per pair and word instead of 6, and one atomic per pair and item of
// up to 256 words instead of one per 34 words: the pass is bound by the POPC pipe, not by the LSU.
// Shared layout: plane[w * Sp + s] (word-major: the samples of a tile are adjacent), Sp = padded S + 2.
constexpr int PAIR_ITEM_WORDS = 256;
constexpr int PAIR_THREADS_MAX = 640;

// one 4 x 4 sample tile over nw staged words (plane[w * Sp + s]); 16 packed counters (cnt << 16 | diff)
__device__ __forceinline__ void pair_tile(const unsigned long long *__restrict__ sV, const unsigned long long *__restrict__ sA,
                                          const unsigned long long *__restrict__ sB, int Sp, int nw, const ushort2 T,
                                          unsigned acc[16])
{
    for (int w = 0; w < nw; ++w) {
        const size_t r = (size_t)w * Sp + 4 * T.x, c = (size_t)w * Sp + 4 * T.y;
        unsigned long long vi[4], ai[4], bi[4];
        {
            const ulonglong2 v0 = *reinterpret_cast<const ulonglong2 *>(sV + r), v1 = *reinterpret_cast<const ulonglong2 *>(sV + r + 2);
            const ulonglong2 a0 = *reinterpret_cast<const ulonglong2 *>(sA + r), a1 = *reinterpret_cast<const ulonglong2 *>(sA + r + 2);
            const ulonglong2 b0 = *reinterpret_cast<const ulonglong2 *>(sB + r), b1 = *reinterpret_cast<const ulonglong2 *>(sB + r + 2);
            vi[0] = v0.x; vi[1] = v0.y; vi[2] = v1.x; vi[3] = v1.y;
            ai[0] = a0.x; ai[1] = a0.y; ai[2] = a1.x; ai[3] = a1.y;
            bi[0] = b0.x; bi[1] = b0.y; bi[2] = b1.x; bi[3] = b1.y;
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {  // two column samples per 16-byte load
            const ulonglong2 vj = *reinterpret_cast<const ulonglong2 *>(sV + c + 2 * h);
            const ulonglong2 aj = *reinterpret_cast<const ulonglong2 *>(sA + c + 2 * h);
            const ulonglong2 bj = *reinterpret_cast<const ulonglong2 *>(sB + c + 2 * h);
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                const unsigned long long m0 = vi[a] & vj.x, m1 = vi[a] & vj.y;
                acc[4 * a + 2 * h] += ((unsigned)__popcll(m0) << 16) + (unsigned)__popcll((ai[a] ^ aj.x) & m0) +
                                      (unsigned)__popcll((bi[a] ^ bj.x) & m0);
                acc[4 * a + 2 * h + 1] += ((unsigned)__popcll(m1) << 16) + (unsigned)__popcll((ai[a] ^ aj.y) & m1) +
                                          (unsigned)__popcll((bi[a] ^ bj.y) & m1);
            }
        }
    }
}

// counters of one tile into the window's exact u64 sums (pair index of the reference: i < j, row-major upper triangle)
__device__ __forceinline__ void pair_flush(const ushort2 T, const unsigned acc[16], int S, bool single,
                                           unsigned long long *__restrict__ dw, unsigned long long *__restrict__ cw)
{
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int i = 4 * T.x + a, j = 4 * T.y + b;
            if (i < j && j < S) {
                const size_t p = (size_t)i * S - (size_t)i * (i + 1) / 2 + (size_t)(j - i - 1);
                const unsigned long long d = acc[4 * a + b] & 0xffffu, c = acc[4 * a + b] >> 16;
                if (single) {
                    dw[p] = d;
                    cw[p] = c;
                } else {
                    atomicAdd(dw + p, d);
                    atomicAdd(cw + p, c);
                }
            }
        }
}

// 80 registers (instead of the 96 a 640-thread launch bound allows): 51 K of the SM's 64 K registers, so that one
// 256-thread block of k_pack (52 registers) fits beside a block of this kernel and the two passes overlap
__global__ void __maxnreg__(80)
k_pairs(const unsigned long long *__restrict__ V, const unsigned long long *__restrict__ T1,
        const unsigned long long *__restrict__ T2, int64_t total_words, int S, int P,
        const PairItem *__restrict__ items, const ushort2 *__restrict__ tiletab, int n_tiles, int Sp, int sw,
        unsigned long long *__restrict__ diff, unsigned long long *__restrict__ cnt)
{
    extern __shared__ unsigned long long sh[];
    const PairItem it = items[blockIdx.x];
    const size_t plane = (size_t)sw * Sp;
    unsigned long long *sV = sh, *sA = sh + plane, *sB = sh + 2 * plane;
    // rows S .. Sp-1 stay zero: valid = 0, they add nothing
    {
        const int npad = Sp - S;
        for (int q = threadIdx.x; q < sw * npad; q += blockDim.x) {
            const size_t o = (size_t)(q / npad) * Sp + S + (q % npad);
            sV[o] = 0ull;
            sA[o] = 0ull;
            sB[o] = 0ull;
        }
    }
    unsigned long long *dw = diff + (size_t)it.window * P, *cw = cnt + (size_t)it.window * P;
    const int nthr = blockDim.x;
    for (int pass = 0; pass < n_tiles; pass += 2 * nthr) {
        const int ta = pass + threadIdx.x, tb = ta + nthr;
        const bool has_a = ta < n_tiles, has_b = tb < n_tiles;
        const ushort2 A = has_a ? tiletab[ta] : make_ushort2(0, 0), B = has_b ? tiletab[tb] : make_ushort2(0, 0);
        unsigned acc_a[16], acc_b[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) acc_a[k] = acc_b[k] = 0u;
        for (int w0 = 0; w0 < it.n_words; w0 += sw) {
            const int nw = min(sw, it.n_words - w0);
            __syncthreads();  // the previous sub-chunk has been consumed (and the zero fill is complete)
            // coalesced on the word axis in global memory
            for (int q = threadIdx.x; q < S * nw; q += nthr) {
                const int s = q / nw, w = q - s * nw;
                const size_t g = (size_t)s * total_words + it.first_word + w0 + w;
                sV[(size_t)w * Sp + s] = V[g];
                sA[(size_t)w * Sp + s] = T1[g];
                sB[(size_t)w * Sp + s] = T2[g];
            }
            __syncthreads();
            if (has_a) pair_tile(sV, sA, sB, Sp, nw, A, acc_a);
            if (has_b) pair_tile(sV, sA, sB, Sp, nw, B, acc_b);
        }
        if (has_a) pair_flush(A, acc_a, S, it.single, dw, cw);
        if (has_b) pair_flush(B, acc_b, S, it.single, dw, cw);
    }
}

// fused pass (whole methylomes) ----------------------------------------------------------
// k_pack is bound by HBM and k_pairs by the POPC pipe; run one after the other (or on two streams: the pair kernel
// leaves a 4-warp packing block no room to keep enough bytes in flight) each leaves the other's resource idle.  Here
// one persistent CTA per SM does both, warp-specialised:
//   * 8 packer warps stream the raw inputs with bulk asynchronous copies (cp.async.bulk -> shared memory, completion
//     on an mbarrier): a unit is one sample x FUSED_GW words (512 sites: 4 KB posteriorMax + 4 KB rc.meth.lvl + 512 B
//     status), every packer warp owns 2 ring slots and keeps the next unit's copies in flight while it packs — the
//     bytes in flight that HBM needs (~70 KB per SM) live in shared memory instead of in the registers of 64 resident
//     warps;
//   * a packer turns a landed unit into the three bit-plane words per 64 sites (the same thermometer code as k_pack;
//     bit b of a word is site b) and writes them into one of two bit-plane stages [word][sample] — the planes never
//     go to HBM;
//   * the consumer warps (the register-tiled all-pairs popcount of k_pairs) work on the other stage; full / empty
//     mbarriers per stage.  Counters are flushed to the exact u64 sums every <= 32 groups (packed 16-bit counters).
// meth_lvl sums: per (sample, group) every lane adds its own 16 sites in a fixed order, then the fixed shuffle tree —
// k_finalize_grouped adds the group partials in a fixed order: deterministic for a given (L, window), independent of
// the grid.  (Not the same rounding as the 64-word super-blocks of k_pack: both are within 1e-12 of the sequential
// sum; windows up to EXACT_MAX sites never come here.)
constexpr int FUSED_GW = 8;            // words per group (= bit-plane stage depth)
// packer warps x ring slots per packer warp are template parameters of k_fused (default 8 x 2, measured: run_divergence)
constexpr int FUSED_FLUSH_GROUPS = 32; // 256 words: cnt <= 16 384, diff <= 32 768 fit the packed counters
constexpr int FUSED_RAW_F64 = FUSED_GW * 64 * 8 + 16;   // one f64 array of a unit + alignment slack
constexpr int FUSED_RAW_U8 = FUSED_GW * 64 + 16;
constexpr int FUSED_SLOT = (2 * FUSED_RAW_F64 + FUSED_RAW_U8 + 127) & ~127;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "W_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra D_%=;\n\t"
        "bra W_%=;\n\t"
        "D_%=:\n\t}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ double2 lds_f64x2(uint32_t addr)
{
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint4 lds_u32x4(uint32_t addr)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
// acc += m where p (asks for one predicated DADD; ptxas may still turn it into an add and two selects)
__device__ __forceinline__ void dadd_if(double &acc, double m, bool p)
{
    asm("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q add.rn.f64 %0, %0, %1;\n\t}" : "+d"(acc) : "d"(m), "r"((unsigned)p));
}
// waiting without taking issue slots from the warps that are being waited for
__device__ __forceinline__ void mbar_wait_backoff(uint64_t *bar, unsigned parity)
{
    unsigned done;
    for (;;) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (done) break;
        __nanosleep(100);
    }
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

struct FusedArgs {
    const uint8_t *status;
    const double *post, *meth;
    int64_t L, site0, end_site;   // the window's sites [site0, end_site) of every sample's row
    int64_t n_groups;             // ceil(words / FUSED_GW)
    int S, Sp, n_tiles, n_cons;   // n_cons consumer threads (warp multiple) + FUSED_PACK_WARPS packer warps
    double thr;
    const ushort2 *tiletab;
    unsigned long long *diff, *cnt;
    double *methpart;             // [S][n_groups]
    int32_t *nvpart;              // [S][n_groups]
};

template <int FUSED_PACK_WARPS, int FUSED_RING>
__global__ void __launch_bounds__(PAIR_THREADS_MAX + 32 * FUSED_PACK_WARPS, 1)
k_fused(const FusedArgs a)
{
    extern __shared__ __align__(128) unsigned char fsm[];
    // layout: raw ring | two bit-plane stages | barriers
    unsigned char *raw = fsm;
    const size_t stage_words = (size_t)3 * FUSED_GW * a.Sp;
    unsigned long long *stage0 = reinterpret_cast<unsigned long long *>(fsm + (size_t)FUSED_PACK_WARPS * FUSED_RING * FUSED_SLOT);
    uint64_t *bars = reinterpret_cast<uint64_t *>(stage0 + 2 * stage_words);
    uint64_t *bar_full = bars, *bar_empty = bars + 2, *bar_raw = bars + 4;   // [2], [2], [PACK_WARPS * RING]
    const int tid = threadIdx.x, lane = tid & 31;
    const int n_cons_warps = a.n_cons >> 5;

    // this CTA's contiguous share of the groups
    const int64_t g0 = a.n_groups * blockIdx.x / gridDim.x, g1 = a.n_groups * (blockIdx.x + 1) / gridDim.x;
    const int n_gl = (int)(g1 - g0);
    const int64_t n_words = (a.end_site - a.site0 + 63) / 64;

    if (tid == 0) {
        mbar_init(bar_full + 0, FUSED_PACK_WARPS);
        mbar_init(bar_full + 1, FUSED_PACK_WARPS);
        mbar_init(bar_empty + 0, n_cons_warps);
        mbar_init(bar_empty + 1, n_cons_warps);
        for (int i = 0; i < FUSED_PACK_WARPS * FUSED_RING; ++i) mbar_init(bar_raw + i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // padding rows S .. Sp-1 of both stages stay zero (valid = 0: they add nothing)
    {
        const int npad = a.Sp - a.S;
        for (int q = tid; q < 2 * 3 * FUSED_GW * npad; q += blockDim.x) stage0[(size_t)(q / npad) * a.Sp + a.S + (q % npad)] = 0ull;
    }
    __syncthreads();

    if (tid >= a.n_cons) {
        // ------------------------------------------------------------------ packer warp
        // The units (group, sample) of the CTA, numbered group-major, are dealt to the packer warps round robin: this
        // warp's k-th unit lives in ring slot k % RING.  Two cursors walk the same sequence: the copy cursor runs RING
        // units ahead of the work cursor.
        const int pw = (tid - a.n_cons) >> 5;
        unsigned char *ring = raw + (size_t)pw * FUSED_RING * FUSED_SLOT;
        uint64_t *rbar = bar_raw + pw * FUSED_RING;
        const unsigned lo_post = (unsigned)(reinterpret_cast<uintptr_t>(a.post) >> 3) & 1u;   // in elements, mod 2
        const unsigned lo_meth = (unsigned)(reinterpret_cast<uintptr_t>(a.meth) >> 3) & 1u;
        const unsigned lo_st = (unsigned)reinterpret_cast<uintptr_t>(a.status) & 15u;
        const int64_t site_first = a.site0 + g0 * (int64_t)(FUSED_GW * 64);

        int c_gl = 0, c_s = pw, c_slot = 0;   // copy cursor: group, sample, ring slot
        while (c_s >= a.S) {
            c_s -= a.S;
            ++c_gl;
        }
        // start the copies of the unit under the copy cursor and advance it (all lanes call it; lane 0 issues)
        auto issue = [&]() {
            const int sm = c_s;
            const int64_t c_site = site_first + (int64_t)c_gl * (FUSED_GW * 64);
            const int nsites = (int)min((int64_t)(FUSED_GW * 64), a.end_site - c_site);
            const int64_t off = (int64_t)sm * a.L + c_site;   // element index of the unit's first site
            unsigned char *slot = ring + c_slot * FUSED_SLOT;
            uint64_t *bar = rbar + c_slot;
            // bytes in front of the first element down to the 16-byte boundary (bulk copies move aligned 16-byte pieces)
            const unsigned op = ((lo_post + (unsigned)off) & 1u) * 8u, om = ((lo_meth + (unsigned)off) & 1u) * 8u;
            const unsigned os = (lo_st + (unsigned)off) & 15u;
            // the rounded ranges leave the arrays only at the very first and the very last unit (conservative test)
            const bool edge = (sm == 0 && c_site < 16) || (sm == a.S - 1 && c_site + nsites + 16 > a.L);
            if (!edge) {
                if (lane == 0) {
                    const unsigned np = (op + (unsigned)nsites * 8u + 15u) & ~15u, nm = (om + (unsigned)nsites * 8u + 15u) & ~15u;
                    const unsigned ns = (os + (unsigned)nsites + 15u) & ~15u;
                    mbar_expect_tx(bar, np + nm + ns);
                    bulk_g2s(slot, reinterpret_cast<const unsigned char *>(a.post + off) - op, np, bar);
                    bulk_g2s(slot + FUSED_RAW_F64, reinterpret_cast<const unsigned char *>(a.meth + off) - om, nm, bar);
                    bulk_g2s(slot + 2 * FUSED_RAW_F64, a.status + off - os, ns, bar);
                }
            } else {
                // element-wise copy to the same places
                double *sp = reinterpret_cast<double *>(slot + op), *sq = reinterpret_cast<double *>(slot + FUSED_RAW_F64 + om);
                unsigned char *ss = slot + 2 * FUSED_RAW_F64 + os;
                for (int i = lane; i < nsites; i += 32) {
                    sp[i] = a.post[off + i];
                    sq[i] = a.meth[off + i];
                    ss[i] = a.status[off + i];
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // later bulk copies reuse the slot
                __syncwarp();
                if (lane == 0) mbar_arrive(bar);
            }
            c_s += FUSED_PACK_WARPS;
            while (c_s >= a.S) {
                c_s -= a.S;
                ++c_gl;
            }
            if (++c_slot == FUSED_RING) c_slot = 0;
        };
        for (int q = 0; q < FUSED_RING && c_gl < n_gl; ++q) issue();

        int w_slot = 0, w_s = pw;   // work cursor: ring slot, sample (the group is the loop variable)
        unsigned w_par = 0;
        int64_t site = site_first;
        for (int gl = 0; gl < n_gl; ++gl, site += FUSED_GW * 64) {
            const int nsites = (int)min((int64_t)(FUSED_GW * 64), a.end_site - site);
            const int nw = (nsites + 63) >> 6;
            const int b = gl & 1;
            const int64_t g = g0 + gl;
            unsigned short *sV = reinterpret_cast<unsigned short *>(stage0 + (size_t)b * stage_words);
            unsigned short *sA = sV + 4 * FUSED_GW * a.Sp, *sB = sA + 4 * FUSED_GW * a.Sp;   // planes, in 16-bit pieces
            mbar_wait(bar_empty + b, ((gl >> 1) & 1) ^ 1);   // the consumers are done with this stage
            for (; w_s < a.S; w_s += FUSED_PACK_WARPS) {
                const int sm = w_s;
                const unsigned char *slot = ring + w_slot * FUSED_SLOT;
                const int64_t off = (int64_t)sm * a.L + site;
                const unsigned op = ((lo_post + (unsigned)off) & 1u) * 8u, om = ((lo_meth + (unsigned)off) & 1u) * 8u;
                const unsigned os = (lo_st + (unsigned)off) & 15u;
                mbar_wait(rbar + w_slot, w_par);
                // Lane l owns the 16 consecutive sites 16 l .. 16 l + 15 of the unit, i.e. a quarter of a 64-site word:
                // it builds its own 16 bits of the three planes (no warp votes) and stores them as the l % 4-th 16-bit
                // piece of word l / 4.  The eight 16-byte chunks of a lane are visited in the order j ^ (l % 8), so that
                // the lanes of a quarter warp read eight different bank groups although each lane's data is contiguous.
                const unsigned l7 = lane & 7;
                double acc = 0.0;
                unsigned vb = 0u, ab = 0u, bb = 0u;
                if ((op | om | os) == 0 && nsites == FUSED_GW * 64) {
                    const uint32_t sl = smem_u32(slot);
                    const uint4 st4 = lds_u32x4(sl + 2 * FUSED_RAW_F64 + 16 * lane);
                    const uint32_t bx = (sl + 128 * lane) ^ (16 * l7);   // the slot is 128-byte aligned
                    unsigned vs = 0u;   // pair j of vs = sites of chunk j ^ l7
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const double2 pp = lds_f64x2(bx ^ (16 * j));
                        const double2 mm = lds_f64x2((bx ^ (16 * j)) + FUSED_RAW_F64);
                        const bool v0 = pp.x >= a.thr, v1 = pp.y >= a.thr;
                        dadd_if(acc, mm.x, v0);
                        dadd_if(acc, mm.y, v1);
                        vs |= (v0 ? (1u << (2 * j)) : 0u) | (v1 ? (2u << (2 * j)) : 0u);
                    }
                    // pair j -> pair j ^ l7: three conditional swaps
                    if (l7 & 1) vs = ((vs & 0x3333u) << 2) | ((vs >> 2) & 0x3333u);
                    if (l7 & 2) vs = ((vs & 0x0f0fu) << 4) | ((vs >> 4) & 0x0f0fu);
                    if (l7 & 4) vs = ((vs & 0x00ffu) << 8) | ((vs >> 8) & 0x00ffu);
                    vb = vs;
                    const unsigned xs[4] = {st4.x, st4.y, st4.z, st4.w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        // per byte: bit 7 of ((b & 0x7f) + 0x7f) | b is set iff b >= 1, of ((b & 0x7f) + 0x7e) | b iff
                        // b >= 2; the multiplication gathers bits 0, 8, 16, 24 into bits 24 .. 27
                        const unsigned x = xs[q], lo = x & 0x7f7f7f7fu;
                        const unsigned g1 = (((lo + 0x7f7f7f7fu) | x) >> 7) & 0x01010101u, g2 = (((lo + 0x7e7e7e7eu) | x) >> 7) & 0x01010101u;
                        ab |= ((g1 * 0x01020408u) >> 24) << (4 * q);
                        bb |= ((g2 * 0x01020408u) >> 24) << (4 * q);
                    }
                } else {
                    // rows that are not 16-byte aligned (odd L) and the last, partial group of the window: same order
                    const unsigned char *bp = slot + op + 128 * lane, *bm = slot + FUSED_RAW_F64 + om + 128 * lane;
                    const unsigned char *bs = slot + 2 * FUSED_RAW_F64 + os + 16 * lane;
                    const int base = 16 * lane;
#pragma unroll 2
                    for (int j = 0; j < 8; ++j) {
                        const int c = j ^ (int)l7, i0 = base + 2 * c;
                        const bool in0 = i0 < nsites, in1 = i0 + 1 < nsites;
                        const double p0 = *reinterpret_cast<const double *>(bp + 16 * c), p1 = *reinterpret_cast<const double *>(bp + 16 * c + 8);
                        const double m0 = *reinterpret_cast<const double *>(bm + 16 * c), m1 = *reinterpret_cast<const double *>(bm + 16 * c + 8);
                        const unsigned s0 = bs[2 * c], s1 = bs[2 * c + 1];
                        const bool v0 = in0 && p0 >= a.thr, v1 = in1 && p1 >= a.thr;
                        if (v0) acc += m0;
                        if (v1) acc += m1;
                        vb |= ((v0 ? 1u : 0u) | (v1 ? 2u : 0u)) << (2 * c);
                        ab |= ((in0 && s0 >= 1 ? 1u : 0u) | (in1 && s1 >= 1 ? 2u : 0u)) << (2 * c);
                        bb |= ((in0 && s0 >= 2 ? 1u : 0u) | (in1 && s1 >= 2 ? 2u : 0u)) << (2 * c);
                    }
                }
                __syncwarp();   // every lane has its values in registers: the slot may be overwritten
                if (c_gl < n_gl) issue();
                if ((lane >> 2) < nw) {
                    const int o = ((lane >> 2) * a.Sp + sm) * 4 + (lane & 3);
                    sV[o] = (unsigned short)vb;
                    sA[o] = (unsigned short)ab;
                    sB[o] = (unsigned short)bb;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(FULL, acc, o);
                const int nv = __reduce_add_sync(FULL, __popc(vb));
                if (lane == 0) {
                    a.methpart[(size_t)sm * a.n_groups + g] = acc;
                    a.nvpart[(size_t)sm * a.n_groups + g] = nv;
                }
                if (++w_slot == FUSED_RING) {
                    w_slot = 0;
                    w_par ^= 1u;
                }
            }
            w_s -= a.S;
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_full + b);   // this warp's units of the group are in the stage
        }
    } else {
        // ------------------------------------------------------------------ consumer warps
        const int ta = tid, tb = tid + a.n_cons;
        const bool has_a = ta < a.n_tiles, has_b = tb < a.n_tiles;
        const ushort2 A = has_a ? a.tiletab[ta] : make_ushort2(0, 0), B = has_b ? a.tiletab[tb] : make_ushort2(0, 0);
        unsigned acc_a[16], acc_b[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) acc_a[q] = acc_b[q] = 0u;
        for (int gl = 0; gl < n_gl; ++gl) {
            const int b = gl & 1;
            const int nw = (int)min((int64_t)FUSED_GW, n_words - (g0 + gl) * FUSED_GW);
            const unsigned long long *sV = stage0 + (size_t)b * stage_words, *sA = sV + (size_t)FUSED_GW * a.Sp, *sB = sA + (size_t)FUSED_GW * a.Sp;
            mbar_wait_backoff(bar_full + b, (unsigned)((gl >> 1) & 1));
            if (has_a) pair_tile(sV, sA, sB, a.Sp, nw, A, acc_a);
            if (has_b) pair_tile(sV, sA, sB, a.Sp, nw, B, acc_b);
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_empty + b);
            // staggered over the CTAs so that the atomics of a flush do not all reach L2 at once
            if (gl == n_gl - 1 || ((gl + blockIdx.x) % FUSED_FLUSH_GROUPS) == FUSED_FLUSH_GROUPS - 1) {
                if (has_a) pair_flush(A, acc_a, a.S, false, a.diff, a.cnt);
                if (has_b) pair_flush(B, acc_b, a.S, false, a.diff, a.cnt);
#pragma unroll
                for (int q = 0; q < 16; ++q) acc_a[q] = acc_b[q] = 0u;
            }
        }
    }
}

// per sample: sum of the group partials of k_fused.  One block per sample; thread t adds its contiguous share of the
// groups in order, then a fixed tree over the 256 threads: the order depends on the number of groups only.
constexpr int FING_THREADS = 256;
__global__ void __launch_bounds__(FING_THREADS)
k_finalize_grouped(const double *__restrict__ methpart, const int32_t *__restrict__ nvpart, int64_t n_groups, int S,
                   double *__restrict__ methsum, long long *__restrict__ nvalid)
{
    __shared__ double sacc[FING_THREADS];
    __shared__ long long snv[FING_THREADS];
    const int s = blockIdx.x, t = threadIdx.x;
    const int64_t per = (n_groups + FING_THREADS - 1) / FING_THREADS, q0 = min(n_groups, per * t), q1 = min(n_groups, q0 + per);
    double acc = 0.0;
    long long nv = 0;
    for (int64_t q = q0; q < q1; ++q) {
        acc += methpart[(size_t)s * n_groups + q];
        nv += nvpart[(size_t)s * n_groups + q];
    }
    sacc[t] = acc;
    snv[t] = nv;
    __syncthreads();
    for (int o = FING_THREADS / 2; o > 0; o >>= 1) {
        if (t < o) {
            sacc[t] += sacc[t + o];
            snv[t] += snv[t + o];
        }
        __syncthreads();
    }
    if (t == 0) {
        methsum[s] = sacc[0];
        nvalid[s] = snv[0];
    }
}

// pass 3 ------------------------------------------------------------------------------
__global__ void k_finalize_pairs(const unsigned long long *__restrict__ diff,
                                 const unsigned long long *__restrict__ cnt, int64_t n, double *__restrict__ D)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) D[i] = (double)diff[i] / (2.0 * (double)cnt[i]);  // src/pedigree.rs:257 (0/0 -> NaN)
}

// per (window, sample): valid-site count and sum of meth_lvl (src/pedigree.rs:159-172)
// One WARP per (window, sample).  Windows up to EXACT_MAX sites are summed in the reference's own order — one
// sequential pass over the window's sites (src/pedigree.rs:171-172) — but read 32 sites at a time, coalesced:
// every lane contributes its site's value (+0.0 when the site is filtered out: x + 0.0 == x, and the sum can never
// be -0.0), the 32 values are exchanged through shared memory and every lane adds them in site order.  (One
// thread per (window, sample) walking its own row thrashed L1: 5.3 ms for 10 000 windows x 1000 sites x 27 samples.)
__global__ void __launch_bounds__(32 * FIN_WARPS)
k_finalize_samples(const double *__restrict__ post, const double *__restrict__ meth, int64_t L,
                   const int64_t *__restrict__ seg, int W, int S, double thr,
                   const double *__restrict__ methpart, const long long *__restrict__ nvpart,
                   const int32_t *__restrict__ sb_first, int n_sb, double *__restrict__ methsum,
                   long long *__restrict__ nvalid)
{
    __shared__ __align__(16) double xch[FIN_WARPS][2][32];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long idx = (long long)blockIdx.x * FIN_WARPS + wib;
    if (idx >= (long long)W * S) return;  // whole warps leave together
    const int w = (int)(idx / S), s = (int)(idx - (long long)w * S);
    const int64_t a = seg[w], b = seg[w + 1];
    double acc = 0.0;
    long long nv = 0;
    if (b - a <= EXACT_MAX) {
        const double *po = post + (size_t)s * L, *me = meth + (size_t)s * L;
        int buf = 0;
        for (int64_t i0 = a; i0 < b; i0 += 32, buf ^= 1) {
            const int64_t i = i0 + lane;
            const bool valid = i < b && po[i] >= thr;
            const double m = valid ? me[i] : 0.0;
            nv += __popc(__ballot_sync(FULL, valid));
            xch[wib][buf][lane] = m;
            __syncwarp();
            // sites beyond the window's end hold +0.0 as well, so every chunk adds all 32 slots
#pragma unroll
            for (int q = 0; q < 32; q += 2) {
                const double2 v = *reinterpret_cast<const double2 *>(&xch[wib][buf][q]);
                acc += v.x;
                acc += v.y;
            }
            // the other buffer is written next; this one again only after the following __syncwarp
        }
    } else {
        for (int q = sb_first[w]; q < sb_first[w + 1]; ++q) {
            acc += methpart[(size_t)s * n_sb + q];
            nv += nvpart[(size_t)s * n_sb + q];
        }
    }
    if (lane == 0) {
        methsum[idx] = acc;
        nvalid[idx] = nv;
    }
}

// p0uu = mean over samples of (1 - rc_meth_lvl), summed in sample order (src/pedigree.rs:179-183)
__global__ void k_p0uu(const double *__restrict__ methsum, const long long *__restrict__ nvalid, int W, int S,
                       double *__restrict__ p0uu)
{
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    double acc = 0.0;
    for (int s = 0; s < S; ++s) {
        const double rc = methsum[(size_t)w * S + s] / (double)nvalid[(size_t)w * S + s];
        acc += 1.0 - rc;
    }
    p0uu[w] = acc / (double)S;
}

void div_arena_release(DivArena &a)
{
    if (a.p) cudaFree(a.p);
    if (a.st2) cudaStreamDestroy(a.st2);
    if (a.ev_start) cudaEventDestroy(a.ev_start);
    if (a.ev_pack_end) cudaEventDestroy(a.ev_pack_end);
    for (auto &e : a.ev_pack)
        if (e) cudaEventDestroy(e);
    a = DivArena();
}

// whole methylome (one window of millions of sites): the fused kernel + finalisation
static int run_fused(cudaStream_t st, const uint8_t *d_status, const double *d_post, const double *d_meth, int S, int64_t L,
                     int64_t site0, int64_t end_site, double thr, double *d_D, unsigned long long *d_diff,
                     unsigned long long *d_cnt, double *d_methsum, long long *d_nvalid, double *d_p0uu, int *launches,
                     float *ms, DivArena *ar, int n_sm, int pack_warps, int ring, size_t smem_bytes)
{
    const int P = S * (S - 1) / 2;
    const int Sp = ((S + 3) & ~3) + 2;
    const int nb = (S + 3) / 4, n_tiles = nb * (nb + 1) / 2;
    const int n_cons = std::min(PAIR_THREADS_MAX, std::max(32, (((n_tiles + 1) / 2) + 31) & ~31));
    const int64_t TW = (end_site - site0 + 63) / 64, NG = (TW + FUSED_GW - 1) / FUSED_GW;
    std::vector<ushort2> pairtab((size_t)n_tiles);
    {
        size_t t = 0;
        for (int i = 0; i < nb; ++i)
            for (int j = i; j < nb; ++j) pairtab[t++] = make_ushort2((unsigned short)i, (unsigned short)j);
    }
    size_t off = 0;
    auto take = [&](size_t bytes) {
        const size_t o = off;
        off += (std::max<size_t>(bytes, 1) + 255) & ~(size_t)255;
        return o;
    };
    const size_t o_mp = take((size_t)S * NG * 8), o_nv = take((size_t)S * NG * 4), o_pt = take(pairtab.size() * sizeof(ushort2));
    if (off > ar->cap) {
        if (ar->p) {
            ABFIT_CUDA(cudaStreamSynchronize(st));
            ABFIT_CUDA(cudaFree(ar->p));
            ar->p = nullptr;
            ar->cap = 0;
        }
        ABFIT_CUDA(cudaMalloc(&ar->p, off));
        ar->cap = off;
    }
    char *base = static_cast<char *>(ar->p);
    FusedArgs a;
    a.status = d_status;
    a.post = d_post;
    a.meth = d_meth;
    a.L = L;
    a.site0 = site0;
    a.end_site = end_site;
    a.n_groups = NG;
    a.S = S;
    a.Sp = Sp;
    a.n_tiles = n_tiles;
    a.n_cons = n_cons;
    a.thr = thr;
    a.tiletab = reinterpret_cast<ushort2 *>(base + o_pt);
    a.diff = d_diff;
    a.cnt = d_cnt;
    a.methpart = reinterpret_cast<double *>(base + o_mp);
    a.nvpart = reinterpret_cast<int32_t *>(base + o_nv);
    ABFIT_CUDA(cudaMemcpyAsync(base + o_pt, pairtab.data(), pairtab.size() * sizeof(ushort2), cudaMemcpyHostToDevice, st));
    ABFIT_CUDA(cudaMemsetAsync(d_diff, 0, (size_t)P * 8, st));
    ABFIT_CUDA(cudaMemsetAsync(d_cnt, 0, (size_t)P * 8, st));
    struct Events {  // destroyed on every way out
        cudaEvent_t e[3] = {nullptr, nullptr, nullptr};
        ~Events()
        {
            for (auto &x : e)
                if (x) cudaEventDestroy(x);
        }
    } evs;
    cudaEvent_t *ev = evs.e;
    if (ms) {
        for (int i = 0; i < 3; ++i) ABFIT_CUDA(cudaEventCreate(&ev[i]));
        ABFIT_CUDA(cudaEventRecord(ev[0], st));
    }
    int grid = (int)std::min<int64_t>(n_sm, NG);
    if (const char *e = getenv("ABFIT_DEV_DIV_FUSED_GRID")) grid = std::max(1, std::min<int>(atoi(e), (int)std::min<int64_t>(NG, 1 << 20)));
    auto launch = [&](auto kern) -> int {
        ABFIT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
        kern<<<grid, n_cons + 32 * pack_warps, smem_bytes, st>>>(a);
        ABFIT_CUDA(cudaGetLastError());
        return 0;
    };
    int lrc;
    if (pack_warps == 4 && ring == 3) lrc = launch(k_fused<4, 3>);
    else if (pack_warps == 6 && ring == 2) lrc = launch(k_fused<6, 2>);
    else if (pack_warps == 8 && ring == 2) lrc = launch(k_fused<8, 2>);
    else if (pack_warps == 8 && ring == 1) lrc = launch(k_fused<8, 1>);
    else if (pack_warps == 4 && ring == 2) lrc = launch(k_fused<4, 2>);
    else if (pack_warps == 3 && ring == 4) lrc = launch(k_fused<3, 4>);
    else {
        set_error("k_fused: unsupported packer shape");
        return ABFIT_ERR_ARG;
    }
    if (lrc) return lrc;
    *launches = 1;
    if (ms) ABFIT_CUDA(cudaEventRecord(ev[1], st));
    k_finalize_pairs<<<(unsigned)((P + 255) / 256), 256, 0, st>>>(d_diff, d_cnt, P, d_D);
    ABFIT_CUDA(cudaGetLastError());
    k_finalize_grouped<<<S, FING_THREADS, 0, st>>>(a.methpart, a.nvpart, NG, S, d_methsum, d_nvalid);
    ABFIT_CUDA(cudaGetLastError());
    *launches += 2;
    if (d_p0uu) {
        k_p0uu<<<1, 128, 0, st>>>(d_methsum, d_nvalid, 1, S, d_p0uu);
        ABFIT_CUDA(cudaGetLastError());
        ++*launches;
    }
    if (ms) ABFIT_CUDA(cudaEventRecord(ev[2], st));
    ABFIT_CUDA(cudaStreamSynchronize(st));
    if (ms) {
        // ms[0] = the fused pack + pair kernel (all of the HBM traffic), ms[1] = finalisation
        cudaEventElapsedTime(&ms[0], ev[0], ev[1]);
        cudaEventElapsedTime(&ms[1], ev[1], ev[2]);
    }
    return 0;
}

// bytes of dynamic shared memory of k_fused for S samples
static size_t fused_smem(int S, int pack_warps, int ring)
{
    const int Sp = ((S + 3) & ~3) + 2;
    return (size_t)pack_warps * ring * FUSED_SLOT + (size_t)2 * 3 * FUSED_GW * Sp * 8 + (size_t)(4 + pack_warps * ring) * 8;
}

bool div_long_windows(const int64_t *h_seg, int W)
{
    // (a few long windows — chromosomes — run the kernel once each)
    bool all_long = W >= 1 && W <= 64;
    for (int w = 0; w < W && all_long; ++w) all_long = h_seg[w + 1] - h_seg[w] > EXACT_MAX;
    return all_long;
}

// -------------------------------------------------------------------------------------
int run_divergence(cudaStream_t st, const uint8_t *d_status, const double *d_post, const double *d_meth, int S,
                   int64_t L, const int64_t *h_seg, int W, double thr, double *d_D, unsigned long long *d_diff,
                   unsigned long long *d_cnt, double *d_methsum, long long *d_nvalid, double *d_p0uu,
                   int *launches, float *ms, DivArena *arena, int long_windows)
{
    // host-side segmentation tables
    std::vector<SuperBlock> sbs;
    std::vector<int32_t> sb_first(W + 1, 0);
    std::vector<int64_t> woff(W + 1, 0);
    for (int w = 0; w < W; ++w) {
        const int64_t len = h_seg[w + 1] - h_seg[w];
        if (len < 0) {
            set_error("seg_offsets must be non-decreasing");
            return ABFIT_ERR_ARG;
        }
        const int64_t nw = (len + 63) / 64;
        woff[w + 1] = woff[w] + nw;
        sb_first[w] = (int32_t)sbs.size();
        for (int64_t f = 0; f < nw; f += SB_WORDS) {
            SuperBlock sb;
            sb.window = w;
            sb.n_words = (int32_t)std::min<int64_t>(SB_WORDS, nw - f);
            sb.first_word = woff[w] + f;
            sb.first_site = h_seg[w] + f * 64;
            sb.end_site = h_seg[w + 1];
            sbs.push_back(sb);
        }
    }
    sb_first[W] = (int32_t)sbs.size();
    const int64_t TW = woff[W];
    const int n_sb = (int)sbs.size();
    const int P = S * (S - 1) / 2;
    *launches = 0;

    int n_sm = 148, smem_optin = 0;
    {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
        cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    }
    // Windows of more than EXACT_MAX sites whose sample tiles fit one CTA (S <= 200): the fused kernel.
    {
        int pack_warps = 8, ring = 2;
        if (const char *e = getenv("ABFIT_DEV_DIV_FUSED_SHAPE")) sscanf(e, "%dx%d", &pack_warps, &ring);
        const int nb_f = (S + 3) / 4, n_tiles_f = nb_f * (nb_f + 1) / 2;
        const bool all_long = long_windows >= 0 ? long_windows != 0 : div_long_windows(h_seg, W);
        const bool can = all_long && P > 0 && n_tiles_f <= 2 * PAIR_THREADS_MAX && fused_smem(S, pack_warps, ring) <= (size_t)smem_optin;
        bool fused = can;
        if (const char *e = getenv("ABFIT_DEV_DIV_FUSED")) fused = atoi(e) != 0 && can;
        if (fused) {
            DivArena local;
            DivArena *ar = arena ? arena : &local;
            int rc = 0;
            if (ms) ms[0] = ms[1] = 0.f;
            for (int w = 0; w < W && rc == 0; ++w) {
                int l1 = 0;
                float m1[2] = {0.f, 0.f};
                rc = run_fused(st, d_status, d_post, d_meth, S, L, h_seg[w], h_seg[w + 1], thr, d_D + (size_t)w * P, d_diff + (size_t)w * P,
                               d_cnt + (size_t)w * P, d_methsum + (size_t)w * S, d_nvalid + (size_t)w * S, d_p0uu ? d_p0uu + w : nullptr, &l1,
                               ms ? m1 : nullptr, ar, n_sm, pack_warps, ring, fused_smem(S, pack_warps, ring));
                *launches += l1;
                if (ms) {
                    ms[0] += m1[0];
                    ms[1] += m1[1];
                }
            }
            if (!arena) div_arena_release(local);
            return rc;
        }
    }

    // pair pass: items of at most PAIR_ITEM_WORDS words (packed 16-bit counters), staged through shared memory
    // `sw` words at a time; 4 x 4 sample tiles, two per thread
    const int Sp = ((S + 3) & ~3) + 2;  // even (16-byte loads), and w * Sp walks through 8 different bank pairs
    const int nb = (S + 3) / 4;
    const int n_tiles = nb * (nb + 1) / 2;
    const size_t smem_cap = 200 * 1024;
    int sw = (int)std::min<size_t>(32, smem_cap / ((size_t)Sp * 24));
    if (sw < 1) {
        set_error("too many samples for the shared-memory pair kernel");
        return ABFIT_ERR_TOO_LARGE;
    }
    const int pair_threads = std::min(PAIR_THREADS_MAX, std::max(32, (((n_tiles + 1) / 2) + 31) & ~31));
    std::vector<PairItem> items;
    // enough items to give every SM a block, never more than PAIR_ITEM_WORDS words each
    const int64_t chunk_target = std::max<int64_t>(8, std::min<int64_t>(PAIR_ITEM_WORDS, (TW + n_sm - 1) / n_sm));
    for (int w = 0; w < W; ++w) {
        const int64_t nw = woff[w + 1] - woff[w];
        if (nw <= 0) continue;
        int64_t n_chunks = (nw + chunk_target - 1) / chunk_target;
        // one long window (a whole methylome): whole waves of one block per SM
        if (W == 1 && n_chunks > n_sm / 2) n_chunks = ((n_chunks + n_sm - 1) / n_sm) * n_sm;
        const int64_t chunk = (nw + n_chunks - 1) / n_chunks;
        for (int64_t f = 0; f < nw; f += chunk) {
            PairItem it;
            it.window = w;
            it.n_words = (int32_t)std::min<int64_t>(chunk, nw - f);
            it.first_word = woff[w] + f;
            it.single = nw <= chunk;
            it.pad = 0;
            items.push_back(it);
        }
    }
    {
        int32_t longest = 1;
        for (auto &it : items) longest = std::max(longest, it.n_words);
        sw = std::min(sw, (int)longest);  // thousands of one-word windows: a block stages one word, not 32
    }
    std::vector<ushort2> pairtab((size_t)n_tiles);  // tile -> (row block, column block), row-major: a warp shares its rows
    {
        size_t t = 0;
        for (int i = 0; i < nb; ++i)
            for (int j = i; j < nb; ++j) pairtab[t++] = make_ushort2((unsigned short)i, (unsigned short)j);
    }

    // device scratch: one arena, carved at 256-byte boundaries
    unsigned long long *d_V = nullptr, *d_T1 = nullptr, *d_T2 = nullptr;
    double *d_methpart = nullptr;
    long long *d_nvpart = nullptr;
    SuperBlock *d_sbs = nullptr;
    int32_t *d_sbfirst = nullptr;
    int64_t *d_seg = nullptr;
    PairItem *d_items = nullptr;
    ushort2 *d_pairtab = nullptr;
    int rc = 0;
    DivArena local_arena;
    DivArena *ar = arena ? arena : &local_arena;
    auto cleanup = [&]() {
        if (!arena) div_arena_release(local_arena);
    };
#define DV_CUDA(call)                                   \
    do {                                                \
        cudaError_t e_ = (call);                        \
        if (e_ != cudaSuccess) {                        \
            rc = cuda_fail(e_, #call);                  \
            cleanup();                                  \
            return rc;                                  \
        }                                               \
    } while (0)
    const size_t plane = (size_t)S * (size_t)std::max<int64_t>(TW, 1) * 8;
    {
        size_t off = 0;
        auto take = [&](size_t bytes) {
            const size_t o = off;
            off += (std::max<size_t>(bytes, 1) + 255) & ~(size_t)255;
            return o;
        };
        const size_t o_V = take(plane), o_T1 = take(plane), o_T2 = take(plane);
        const size_t o_mp = take((size_t)S * std::max(n_sb, 1) * 8), o_nv = take((size_t)S * std::max(n_sb, 1) * 8);
        const size_t o_sbs = take(sbs.size() * sizeof(SuperBlock)), o_sbf = take((size_t)(W + 1) * 4);
        const size_t o_seg = take((size_t)(W + 1) * 8), o_it = take(items.size() * sizeof(PairItem));
        const size_t o_pt = take(pairtab.size() * sizeof(ushort2));
        if (off > ar->cap) {
            if (ar->p) {
                DV_CUDA(cudaStreamSynchronize(st));  // earlier work on this stream may still read the old arena
                DV_CUDA(cudaFree(ar->p));
                ar->p = nullptr;
                ar->cap = 0;
            }
            DV_CUDA(cudaMalloc(&ar->p, off));
            ar->cap = off;
        }
        char *base = static_cast<char *>(ar->p);
        d_V = reinterpret_cast<unsigned long long *>(base + o_V);
        d_T1 = reinterpret_cast<unsigned long long *>(base + o_T1);
        d_T2 = reinterpret_cast<unsigned long long *>(base + o_T2);
        d_methpart = reinterpret_cast<double *>(base + o_mp);
        d_nvpart = reinterpret_cast<long long *>(base + o_nv);
        d_sbs = reinterpret_cast<SuperBlock *>(base + o_sbs);
        d_sbfirst = reinterpret_cast<int32_t *>(base + o_sbf);
        d_seg = reinterpret_cast<int64_t *>(base + o_seg);
        d_items = reinterpret_cast<PairItem *>(base + o_it);
        d_pairtab = reinterpret_cast<ushort2 *>(base + o_pt);
    }
    if (!sbs.empty())
        DV_CUDA(cudaMemcpyAsync(d_sbs, sbs.data(), sbs.size() * sizeof(SuperBlock), cudaMemcpyHostToDevice, st));
    DV_CUDA(cudaMemcpyAsync(d_sbfirst, sb_first.data(), (size_t)(W + 1) * 4, cudaMemcpyHostToDevice, st));
    DV_CUDA(cudaMemcpyAsync(d_seg, h_seg, (size_t)(W + 1) * 8, cudaMemcpyHostToDevice, st));
    if (!items.empty())
        DV_CUDA(cudaMemcpyAsync(d_items, items.data(), items.size() * sizeof(PairItem), cudaMemcpyHostToDevice, st));
    if (!pairtab.empty())
        DV_CUDA(cudaMemcpyAsync(d_pairtab, pairtab.data(), pairtab.size() * sizeof(ushort2),
                                cudaMemcpyHostToDevice, st));
    if (P > 0) {
        DV_CUDA(cudaMemsetAsync(d_diff, 0, (size_t)W * P * 8, st));
        DV_CUDA(cudaMemsetAsync(d_cnt, 0, (size_t)W * P * 8, st));
    }

    // ---- pass 1 and pass 2, overlapped ---------------------------------------------------------------------------
    // k_pack is bound by HBM, k_pairs by the POPC pipe: run back to back they leave each other's resource idle (2.9 +
    // 2.5 ms on the C5 shape).  A long site axis is therefore cut into chunks (whole pair items / whole super-blocks):
    // chunk c's pair pass runs on the main stream while chunk c+1 is packed on a second stream, the two kernels sharing
    // every SM (k_pairs: 640 threads x 80 registers, k_pack: 128-thread blocks in the register space that is left).
    int n_chunks = 1;
    // (only whole methylomes of millions of sites: measured on 625 000 sites and on 10 000 windows of 1000 sites the
    // plain sequence is faster)
    if (P > 0 && !items.empty() && n_sb > 0 && W == 1 && TW >= 65536) n_chunks = 4;
    if (const char *e = getenv("ABFIT_DEV_DIV_CHUNKS")) n_chunks = std::max(1, std::min(DivArena::MAX_CHUNKS, atoi(e)));
    n_chunks = (int)std::min<size_t>((size_t)std::max(n_chunks, 1), std::max<size_t>(items.size(), 1));
    if (P == 0 || items.empty() || n_sb == 0) n_chunks = 1;
    cudaStream_t st2 = st;
    cudaEvent_t ev_start = nullptr, ev_pack[DivArena::MAX_CHUNKS] = {};
    if (n_chunks > 1) {
        if (!ar->st2) {
            DV_CUDA(cudaStreamCreateWithFlags(&ar->st2, cudaStreamNonBlocking));
            DV_CUDA(cudaEventCreateWithFlags(&ar->ev_start, cudaEventDisableTiming));
            for (auto &e : ar->ev_pack) DV_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            DV_CUDA(cudaEventCreate(&ar->ev_pack_end));
        }
        st2 = ar->st2;
        ev_start = ar->ev_start;
        for (int c = 0; c < n_chunks; ++c) ev_pack[c] = ar->ev_pack[c];
    }
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    if (ms) {
        for (auto &e : ev) DV_CUDA(cudaEventCreate(&e));
        DV_CUDA(cudaEventRecord(ev[0], st));
    }
    const size_t pair_smem = (size_t)sw * Sp * 24;
    if (P > 0 && !items.empty() && pair_smem > 48 * 1024)
        DV_CUDA(cudaFuncSetAttribute(k_pairs, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pair_smem));
    if (n_chunks == 1) {
        if (n_sb > 0) {
            const long long units = (long long)n_sb * S;
            k_pack<<<(unsigned)((units + 7) / 8), 256, 0, st>>>(d_status, d_post, d_meth, L, TW, d_sbs, n_sb, 0, n_sb, S, thr,
                                                                d_V, d_T1, d_T2, d_methpart, d_nvpart);
            DV_CUDA(cudaGetLastError());
            ++*launches;
        }
        if (ms) DV_CUDA(cudaEventRecord(ev[1], st));
        if (P > 0 && !items.empty()) {
            k_pairs<<<(unsigned)items.size(), pair_threads, pair_smem, st>>>(d_V, d_T1, d_T2, TW, S, P, d_items, d_pairtab,
                                                                            n_tiles, Sp, sw, d_diff, d_cnt);
            DV_CUDA(cudaGetLastError());
            ++*launches;
        }
    } else {
        // chunk c = items [i0, i1) and every super-block that starts before the chunk's last word
        DV_CUDA(cudaEventRecord(ev_start, st));
        DV_CUDA(cudaStreamWaitEvent(st2, ev_start, 0));
        std::vector<int> item_end(n_chunks), sb_end(n_chunks);
        for (int c = 0; c < n_chunks; ++c) {
            // whole waves of one pair block per SM where the item count allows
            int64_t e = (int64_t)items.size() * (c + 1) / n_chunks;
            if (c + 1 < n_chunks && e > n_sm) e = (e / n_sm) * n_sm;
            item_end[c] = (int)e;
        }
        item_end[n_chunks - 1] = (int)items.size();
        for (int c = 0, q = 0; c < n_chunks; ++c) {
            const int64_t last_word = c + 1 < n_chunks ? items[(size_t)item_end[c]].first_word : TW;
            while (q < n_sb && sbs[(size_t)q].first_word < last_word) ++q;
            sb_end[c] = c + 1 < n_chunks ? q : n_sb;
        }
        // 128-thread blocks (4 warps x 56 registers) slip into the registers a k_pairs block leaves free.  Measured on
        // the C5 shape: a warp per unit 5.02 ms for both passes (4 chunks; 5.40 back to back); a FIXED number of looping
        // blocks per SM, which would guarantee the pair kernel its room, starves the packing instead — it needs
        // ~64 resident warps per SM to stream at HBM speed (2 / 4 blocks per SM: 8.4 / 4.7 ms for the packing alone).
        const int pack_threads = 128;
        long long pack_blocks = 1ll << 40;
        if (const char *e = getenv("ABFIT_DEV_DIV_PACK_BLOCKS")) pack_blocks = (long long)std::max(1, atoi(e)) * n_sm;
        for (int c = 0; c < n_chunks; ++c) {
            const int s0 = c ? sb_end[c - 1] : 0, s1 = sb_end[c];
            if (s1 > s0) {
                const long long units = (long long)(s1 - s0) * S;
                const unsigned grid = (unsigned)std::min<long long>(pack_blocks, (units + pack_threads / 32 - 1) / (pack_threads / 32));
                k_pack<<<grid, pack_threads, 0, st2>>>(d_status, d_post, d_meth, L, TW, d_sbs, n_sb, s0, s1, S, thr, d_V, d_T1, d_T2,
                                                        d_methpart, d_nvpart);
                DV_CUDA(cudaGetLastError());
                ++*launches;
            }
            DV_CUDA(cudaEventRecord(ev_pack[c], st2));
        }
        if (ms) DV_CUDA(cudaEventRecord(ar->ev_pack_end, st2));
        for (int c = 0; c < n_chunks; ++c) {
            const int i0 = c ? item_end[c - 1] : 0, i1 = item_end[c];
            DV_CUDA(cudaStreamWaitEvent(st, ev_pack[c], 0));
            if (i1 > i0) {
                k_pairs<<<(unsigned)(i1 - i0), pair_threads, pair_smem, st>>>(d_V, d_T1, d_T2, TW, S, P, d_items + i0, d_pairtab,
                                                                            n_tiles, Sp, sw, d_diff, d_cnt);
                DV_CUDA(cudaGetLastError());
                ++*launches;
            }
        }
        if (ms) DV_CUDA(cudaEventRecord(ev[1], st));  // end of the pair pass (the packing ended earlier, on st2)
    }
    if (P > 0) {
        const int64_t n = (int64_t)W * P;
        k_finalize_pairs<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_diff, d_cnt, n, d_D);
        DV_CUDA(cudaGetLastError());
        ++*launches;
    }
    {
        const int n = W * S;
        k_finalize_samples<<<(n + FIN_WARPS - 1) / FIN_WARPS, 32 * FIN_WARPS, 0, st>>>(
            d_post, d_meth, L, d_seg, W, S, thr, d_methpart, d_nvpart, d_sbfirst, n_sb, d_methsum, d_nvalid);
        DV_CUDA(cudaGetLastError());
        ++*launches;
        if (d_p0uu) {
            k_p0uu<<<(W + 127) / 128, 128, 0, st>>>(d_methsum, d_nvalid, W, S, d_p0uu);
            DV_CUDA(cudaGetLastError());
            ++*launches;
        }
    }
    if (ms) DV_CUDA(cudaEventRecord(ev[2], st));
    DV_CUDA(cudaStreamSynchronize(st));
    if (ms) {
        // one chunk: ms[0] = k_pack (the HBM-bound pass), ms[1] = all-pairs popcount + finalisation.
        // overlapped: ms[0] = until the last chunk was packed, ms[1] = the rest (pair pass of the last chunks +
        // finalisation); ms[0] + ms[1] is the duration of the call's kernels either way
        if (n_chunks > 1) {
            float total = 0.f;
            cudaEventElapsedTime(&ms[0], ev[0], ar->ev_pack_end);
            cudaEventElapsedTime(&total, ev[0], ev[2]);
            ms[1] = total - ms[0];
        } else {
            cudaEventElapsedTime(&ms[0], ev[0], ev[1]);
            cudaEventElapsedTime(&ms[1], ev[1], ev[2]);
        }
        for (auto &e : ev) cudaEventDestroy(e);
    }
    cleanup();
#undef DV_CUDA
    return 0;
}

}  // namespace abfit
