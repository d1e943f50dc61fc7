// abfit_api.cu — C ABI of libabfit (include/abfit.h): context, problem compilation,
// device-resident batches, host-buffer one-shot entry points, input generators.
//
// Host work here is O(input) bookkeeping only (validation, run/triple tables, copies);
// every numerical result comes from the kernels in abfit_kernels.cu / abfit_divergence.cu.
// There is deliberately no CPU implementation of the objective or the optimiser in this
// library: without a CUDA device all compute calls fail.
#include <chrono>
#include <cmath>
#include <cstring>
#include <map>
#include <memory>
#include <thread>
#include <tuple>

#include "abfit_jit.h"
#include "abfit_plan.h"
#include "abfit_psim.cuh"

namespace abfit {

static thread_local std::string g_last_error;
void set_error(const std::string &msg) { g_last_error = msg; }
int cuda_fail(cudaError_t e, const char *what)
{
    set_error(std::string("CUDA error: ") + cudaGetErrorString(e) + " at " + what);
    return ABFIT_ERR_CUDA;
}

template <class T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    ~DevBuf() { release(); }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
    int ensure(size_t count)
    {
        if (count <= n && p) return 0;
        release();
        if (count == 0) count = 1;
        ABFIT_CUDA(cudaMalloc(&p, count * sizeof(T)));
        n = count;
        return 0;
    }
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
};

}  // namespace abfit

using namespace abfit;

struct abfit_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;  // H2D of the bootstrap inputs while the multi-start kernel runs
    cudaEvent_t copy_done = nullptr;
    // abfit_alphabeta_batch: the start simplices are uploaded in chunks; behind every chunk a 4-byte copy raises a device
    // counter the multi-start kernel watches, so that it starts on the first windows while the rest is still on the bus
    static constexpr int SX_CHUNKS = 64;
    int *h_sx_counts = nullptr;  // pinned [SX_CHUNKS]
    int *d_sx_ready = nullptr;
    cudaEvent_t sx_reset = nullptr;  // recorded behind the counter's reset: the watching kernel's stream waits on it
    cudaDeviceProp prop{};
    int smem_optin = 0;
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    // pipelined fit -> bootstrap (run_pipelined): one stream per sub-batch of windows
    static constexpr int MAX_PIPES = 8;
    cudaStream_t pipe_stream[MAX_PIPES] = {};
    cudaEvent_t pipe_done[MAX_PIPES] = {};
    cudaEvent_t pipe_start = nullptr, idx_done = nullptr;
    // workspace of the one-shot host-buffer calls: device buffers are kept between calls
    // (cudaMalloc/cudaFree of multi-GB buffers costs more than the kernels of a small batch)
    abfit_batch *scratch = nullptr;
    // observed divergence: pass-to-pass scratch and result buffers, kept between calls
    DivArena div_arena;
    DevBuf<double> dv_D, dv_methsum, dv_p0uu;
    DevBuf<unsigned long long> dv_diff, dv_cnt;
    DevBuf<long long> dv_nvalid;
};

struct abfit_batch {
    abfit_ctx *ctx = nullptr;
    HostPlan hp;
    LaunchShape shape;
    int n_probs = 0;
    int64_t total_pairs = 0;
    DevBuf<DevProblem> d_probs;
    DevBuf<double> d_D;
    DevBuf<uint32_t> d_offs;
    DevBuf<OpWord> d_ops;
    DevBuf<uint32_t> d_wtrip, d_wtid;
    DevicePools pools{};
    // fit
    int n_starts = 0;
    DevBuf<double> d_simplices, d_xscratch;
    DevBuf<double> d_lm;  // lane state of the large-pedigree variants (shape.big)
    DevBuf<WorkItem> d_items;
    int n_items = 0;
    DevBuf<abfit_fit> d_all, d_best;
    DevBuf<double> d_pred, d_resid;
    DevBuf<int32_t> d_status;
    DevBuf<unsigned long long> d_evals_fit, d_evals_boot;
    bool fit_done = false;
    // boot
    int n_boot = 0;
    DevBuf<int32_t> d_idx;
    DevBuf<double> d_vary, d_scratch, d_rows;
    DevBuf<abfit_fit> d_bootfits;
    DevBuf<int> d_booterr;
    DevBuf<WorkItem> d_boot_items;
    int n_boot_items = 0;
    bool boot_uploaded = false, boot_done = false;
    // specialised kernels of this batch's program (abfit_jit.cu); nullptr: interpreter kernels
    const JitModule *jit = nullptr;
    bool jit_decided = false;
    int64_t jit_fits_seen = 0;
    bool boot_items_v2 = false;  // the bootstrap items were built for the continuous-scheduling kernel
    DevBuf<unsigned long long> d_ids;  // per-window generator keys of abfit_alphabeta_batch_multi
    DevBuf<int> d_cursor;  // item cursors of the continuous-scheduling kernels: [0] multi-start, [1] bootstrap
    DevBuf<double> d_analysis, d_analysis_scratch;  // bootstrap statistics on the device (abfit_alphabeta_batch)
    DevBuf<double> d_wide_ss;      // EXPERIMENT (ABFIT_EXPERIMENT_SUFFSTATS): per-triple statistics of the warp-per-fit kernels
    DevBuf<long long> d_wide_ss_off;
    const int *sx_ready = nullptr;  // set by abfit_alphabeta_batch for ONE run_fit: the simplices are still being uploaded
    int jit_warps_fit = 0, jit_warps_boot = 0;  // resident warps = grid of a full machine
    // pipelined fit -> select -> bootstrap: sub-batches of windows, each with its own guided item lists and cursors
    struct Pipe {
        int p0 = 0, n = 0, fit_item0 = 0, fit_items = 0, boot_item0 = 0, boot_items = 0;
    };
    std::vector<Pipe> pipes;
    DevBuf<WorkItem> d_pipe_items;
    DevBuf<int> d_pipe_cursor;
    int pipes_n_starts = -1, pipes_n_boot = -1;
    bool pipelined_timing = false;
    // timing
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    bool ev_fit = false, ev_boot = false;
    int launches_fit = 0, launches_boot = 0;
};

// run f(i) for i in [0, n) on the host's cores (input generation and statistics of large batches)
template <class F>
static void parallel_for(int32_t n, F f)
{
    const int nt = (int)std::max(1u, std::min<unsigned>(std::thread::hardware_concurrency(), (unsigned)std::max(1, n / 64)));
    if (nt <= 1) {
        for (int32_t i = 0; i < n; ++i) f(i);
        return;
    }
    std::vector<std::thread> th;
    for (int t = 0; t < nt; ++t)
        th.emplace_back([=]() {
            for (int32_t i = t; i < n; i += nt) f(i);
        });
    for (auto &x : th) x.join();
}

// scratch of the large-pedigree kernels for `slots` warps (grows only); {nullptr} when the batch is not big
static int big_scratch(abfit_batch *b, size_t slots, BigScratch &out)
{
    out = BigScratch();
    if (!b->shape.big) return 0;
    const size_t stride = (size_t)std::max(b->shape.n_lane_max, 1) * 32;
    if (int rc = b->d_lm.ensure(slots * stride)) return rc;
    if (int rc = b->d_xscratch.ensure(slots * 20 * 32)) return rc;
    out.lm = b->d_lm.p;
    out.lm_stride = stride;
    out.x = b->d_xscratch.p;
    return 0;
}

// Specialised kernels for this batch?  Policy: the batch must share one pedigree program (jit_eligible) and be large
// enough to repay a compilation — unless the module is already loaded or sits in the disk cache, which costs
// milliseconds.  ABFIT_JIT=0 never, ABFIT_JIT=1 always (tests), unset: batches of >= ABFIT_JIT_MIN_FITS fits
// (default 200 000: a compilation takes 2-4 s once per pedigree shape and machine — the cubin is cached on disk —
// and the specialised kernels run 1.4x faster).
static void decide_jit(abfit_batch *b, int64_t fits_per_prob)
{
    // decided once per loaded batch; a later request with more fits per window may still turn specialisation ON
    if (b->jit_decided && (b->jit || fits_per_prob <= b->jit_fits_seen)) return;
    b->jit_decided = true;
    b->jit_fits_seen = fits_per_prob;
    b->jit = nullptr;
    const char *env = getenv("ABFIT_JIT");
    if (env && atoi(env) == 0) return;
    std::string why;
    if (!jit_eligible(b->hp, b->shape, &why)) {
        if (getenv("ABFIT_DEV_VERBOSE")) fprintf(stderr, "[abfit] interpreter kernels: %s\n", why.c_str());
        return;
    }
    const bool force = env && atoi(env) != 0;
    if (!force && !jit_is_cached(b->hp, 0)) {
        const char *mf = getenv("ABFIT_JIT_MIN_FITS");
        const int64_t min_fits = mf ? atoll(mf) : 200000;
        if ((int64_t)b->n_probs * fits_per_prob < min_fits) return;
    }
    std::string note;
    const JitModule *m = nullptr;
    if (jit_get_module(b->hp, 0, &m, &note) == 0) {
        b->jit = m;
    } else if (!note.empty()) {
        static bool warned = false;
        if (!warned || getenv("ABFIT_DEV_VERBOSE"))
            fprintf(stderr, "[abfit] specialised kernels unavailable, using the interpreter kernels: %s\n", note.c_str());
        warned = true;
    }
}

extern "C" {

const char *abfit_last_error(void) { return g_last_error.c_str(); }
const char *abfit_version(void) { return "abfit-b200 0.1 (sm_100a)"; }

int abfit_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return n;
}

int abfit_ctx_create(int device, abfit_ctx **out)
{
    if (!out) return ABFIT_ERR_ARG;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        set_error(std::string("no CUDA device available: ") + (e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e)) +
                  " — libabfit has no CPU fallback");
        return ABFIT_ERR_CUDA;
    }
    if (device < 0 || device >= n) {
        set_error("device index out of range");
        return ABFIT_ERR_ARG;
    }
    ABFIT_CUDA(cudaSetDevice(device));
    abfit_ctx *c = new abfit_ctx();
    c->device = device;
    if (cudaGetDeviceProperties(&c->prop, device) != cudaSuccess) {
        delete c;
        return cuda_fail(cudaGetLastError(), "cudaGetDeviceProperties");
    }
    c->smem_optin = max_dynamic_smem(device);
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete c;
        return cuda_fail(cudaGetLastError(), "cudaStreamCreate");
    }
    if (cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&c->copy_done, cudaEventDisableTiming) != cudaSuccess) {
        abfit_ctx_destroy(c);
        return cuda_fail(cudaGetLastError(), "cudaStreamCreate (copy stream)");
    }
    *out = c;
    return 0;
}

void abfit_ctx_destroy(abfit_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->scratch) abfit_batch_destroy(ctx->scratch);
    div_arena_release(ctx->div_arena);
    if (ctx->t0) cudaEventDestroy(ctx->t0);
    if (ctx->t1) cudaEventDestroy(ctx->t1);
    for (int k = 0; k < abfit_ctx::MAX_PIPES; ++k) {
        if (ctx->pipe_stream[k]) cudaStreamDestroy(ctx->pipe_stream[k]);
        if (ctx->pipe_done[k]) cudaEventDestroy(ctx->pipe_done[k]);
    }
    if (ctx->pipe_start) cudaEventDestroy(ctx->pipe_start);
    if (ctx->idx_done) cudaEventDestroy(ctx->idx_done);
    if (ctx->copy_done) cudaEventDestroy(ctx->copy_done);
    if (ctx->sx_reset) cudaEventDestroy(ctx->sx_reset);
    if (ctx->h_sx_counts) cudaFreeHost(ctx->h_sx_counts);
    if (ctx->d_sx_ready) cudaFree(ctx->d_sx_ready);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int abfit_ctx_info(abfit_ctx *ctx, int32_t *sm_count, int32_t *sm_clock_khz, int64_t *mem_bytes)
{
    if (!ctx) return ABFIT_ERR_ARG;
    if (sm_count) *sm_count = ctx->prop.multiProcessorCount;
    if (sm_clock_khz) {
        int khz = 0;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device);
        *sm_clock_khz = khz;
    }
    if (mem_bytes) *mem_bytes = (int64_t)ctx->prop.totalGlobalMem;
    return 0;
}

int abfit_ctx_timer_start(abfit_ctx *ctx)
{
    if (!ctx) return ABFIT_ERR_ARG;
    ABFIT_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->t0) {
        ABFIT_CUDA(cudaEventCreate(&ctx->t0));
        ABFIT_CUDA(cudaEventCreate(&ctx->t1));
    }
    ABFIT_CUDA(cudaEventRecord(ctx->t0, ctx->stream));
    return 0;
}

int abfit_ctx_timer_stop(abfit_ctx *ctx, float *ms_out)
{
    if (!ctx || !ms_out || !ctx->t0) return ABFIT_ERR_ARG;
    ABFIT_CUDA(cudaSetDevice(ctx->device));
    ABFIT_CUDA(cudaEventRecord(ctx->t1, ctx->stream));
    ABFIT_CUDA(cudaEventSynchronize(ctx->t1));
    ABFIT_CUDA(cudaEventElapsedTime(ms_out, ctx->t0, ctx->t1));
    return 0;
}

int abfit_ctx_sync(abfit_ctx *ctx)
{
    if (!ctx) return ABFIT_ERR_ARG;
    ABFIT_CUDA(cudaSetDevice(ctx->device));
    ABFIT_CUDA(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int abfit_measure_fp64_peak(abfit_ctx *ctx, double *tflops_out)
{
    if (!ctx || !tflops_out) return ABFIT_ERR_ARG;
    ABFIT_CUDA(cudaSetDevice(ctx->device));
    DevBuf<double> sink;
    if (int rc = sink.ensure(1)) return rc;
    cudaEvent_t a, b;
    ABFIT_CUDA(cudaEventCreate(&a));
    ABFIT_CUDA(cudaEventCreate(&b));
    const int blocks = ctx->prop.multiProcessorCount * 8, threads = 256, iters = 2048;
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {
        ABFIT_CUDA(cudaEventRecord(a, ctx->stream));
        if (int rc = launch_fp64_peak(ctx->stream, blocks, threads, iters, sink.p)) return rc;
        ABFIT_CUDA(cudaEventRecord(b, ctx->stream));
        ABFIT_CUDA(cudaEventSynchronize(b));
        float ms = 0.f;
        ABFIT_CUDA(cudaEventElapsedTime(&ms, a, b));
        const double flops = (double)blocks * threads * (double)iters * 64.0 * 2.0;
        if (rep > 0 && ms > 0.f) best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    *tflops_out = best;
    return 0;
}

// ---------------------------------------------------------------------------------------
// input generators (host; counter-based so shards can be produced independently)
// ---------------------------------------------------------------------------------------
void abfit_gen_start_simplices(uint64_t seed, uint64_t problem_id, int32_t n_starts, double max_divergence,
                               double *out)
{
    double mx = max_divergence;
    if (max_divergence <= 0.0) mx = 0.1;  // src/structs.rs:80-83
    for (int32_t s = 0; s < n_starts; ++s)
        for (int v = 0; v < 5; ++v) {
            double *x = out + ((size_t)s * 5 + v) * 4;
            x[0] = std::pow(10.0, uniform(-9.0, -2.0, u01(seed, 1, problem_id, (uint64_t)s, v * 4 + 0)));
            x[1] = std::pow(10.0, uniform(-9.0, -2.0, u01(seed, 1, problem_id, (uint64_t)s, v * 4 + 1)));
            x[2] = uniform(0.0, 0.1, u01(seed, 1, problem_id, (uint64_t)s, v * 4 + 2));
            x[3] = uniform(0.0, mx, u01(seed, 1, problem_id, (uint64_t)s, v * 4 + 3));
        }
}

void abfit_gen_vary_vertices(uint64_t seed, uint64_t problem_id, int32_t n_boot, const double best_theta[4],
                             double *out)
{
    for (int32_t b = 0; b < n_boot; ++b)
        for (int v = 0; v < 4; ++v)
            for (int j = 0; j < 4; ++j) {
                out[((size_t)b * 4 + v) * 4 + j] = vary_coordinate(seed, problem_id, (uint64_t)b, v, j, best_theta[j]);
            }
}

void abfit_gen_resample_idx(uint64_t seed, uint64_t problem_id, int32_t n_boot, int32_t n_pairs, int32_t *out)
{
    for (int32_t b = 0; b < n_boot; ++b)
        for (int32_t i = 0; i < n_pairs; ++i) {
            int32_t k = (int32_t)(u01(seed, 3, problem_id, (uint64_t)b, (uint64_t)i) * (double)n_pairs);
            if (k >= n_pairs) k = n_pairs - 1;
            out[(size_t)b * n_pairs + i] = k;
        }
}

// ---------------------------------------------------------------------------------------
// batches
// ---------------------------------------------------------------------------------------
// (re)load a batch object with a new set of problems; device buffers only ever grow, so a batch that
// is reused (the context's workspace behind the one-shot calls) stops paying cudaMalloc / cudaFree
static int batch_load(abfit_batch *b, const abfit_problem *probs, int32_t n_probs)
{
    abfit_ctx *ctx = b->ctx;
    if (int rc = compile_problems(probs, n_probs, b->hp)) return rc;
    HostPlan &hp = b->hp;
    b->n_probs = n_probs;
    b->total_pairs = hp.total_pairs;
    b->n_starts = b->n_boot = 0;
    b->n_items = b->n_boot_items = 0;
    b->fit_done = b->boot_uploaded = b->boot_done = false;
    b->ev_fit = b->ev_boot = false;
    b->jit = nullptr;
    b->jit_decided = false;
    b->jit_fits_seen = 0;
    b->pipes.clear();
    b->pipes_n_starts = b->pipes_n_boot = -1;
    b->pipelined_timing = false;
    // aux kernels (select / cost / model divergence) only need the one-warp, simplex-free shape;
    // the fit shape is chosen in upload_starts / upload_boot when the number of fits is known
    if (int rc = choose_launch_shape(hp, (size_t)ctx->smem_optin, (size_t)ctx->prop.sharedMemPerMultiprocessor, 1,
                                     b->shape))
        return rc;
    if (int rc = b->d_probs.ensure(hp.probs.size())) return rc;
    if (int rc = b->d_D.ensure(hp.D.size())) return rc;
    if (int rc = b->d_offs.ensure(hp.offs.size())) return rc;
    if (int rc = b->d_ops.ensure(hp.ops.size())) return rc;
    if (int rc = b->d_wtrip.ensure(hp.wtrip.size())) return rc;
    if (int rc = b->d_wtid.ensure(hp.wtid.size())) return rc;
    cudaStream_t st = ctx->stream;
    ABFIT_CUDA(cudaMemcpyAsync(b->d_probs.p, hp.probs.data(), hp.probs.size() * sizeof(DevProblem), cudaMemcpyHostToDevice, st));
    ABFIT_CUDA(cudaMemcpyAsync(b->d_D.p, hp.D.data(), hp.D.size() * 8, cudaMemcpyHostToDevice, st));
    ABFIT_CUDA(cudaMemcpyAsync(b->d_offs.p, hp.offs.data(), hp.offs.size() * 4, cudaMemcpyHostToDevice, st));
    if (!hp.ops.empty())
        ABFIT_CUDA(cudaMemcpyAsync(b->d_ops.p, hp.ops.data(), hp.ops.size() * sizeof(OpWord), cudaMemcpyHostToDevice, st));
    ABFIT_CUDA(cudaMemcpyAsync(b->d_wtrip.p, hp.wtrip.data(), hp.wtrip.size() * 4, cudaMemcpyHostToDevice, st));
    ABFIT_CUDA(cudaMemcpyAsync(b->d_wtid.p, hp.wtid.data(), hp.wtid.size() * 4, cudaMemcpyHostToDevice, st));
    ABFIT_CUDA(cudaStreamSynchronize(st));  // hp vectors are pageable: make the copies complete here
    b->pools = DevicePools{b->d_probs.p, b->d_D.p, b->d_offs.p, b->d_ops.p, b->d_wtrip.p, b->d_wtid.p};
    if (!b->ev[0])
        for (auto &e : b->ev) ABFIT_CUDA(cudaEventCreate(&e));
    if (int rc = b->d_evals_fit.ensure(n_probs)) return rc;
    if (int rc = b->d_evals_boot.ensure(n_probs)) return rc;
    ABFIT_CUDA(cudaMemsetAsync(b->d_evals_fit.p, 0, (size_t)n_probs * 8, st));
    ABFIT_CUDA(cudaMemsetAsync(b->d_evals_boot.p, 0, (size_t)n_probs * 8, st));
    return 0;
}

int abfit_batch_create(abfit_ctx *ctx, const abfit_problem *probs, int32_t n_probs, abfit_batch **out)
{
    if (!ctx || !out) return ABFIT_ERR_ARG;
    *out = nullptr;
    ABFIT_CUDA(cudaSetDevice(ctx->device));
    std::unique_ptr<abfit_batch> b(new abfit_batch());
    b->ctx = ctx;
    if (int rc = batch_load(b.get(), probs, n_probs)) {
        abfit_batch_destroy(b.release());
        return rc;
    }
    *out = b.release();
    return 0;
}

// the context's reusable workspace for the one-shot host-buffer calls
static int workspace(abfit_ctx *ctx, const abfit_problem *probs, int32_t n_probs, abfit_batch **out)
{
    if (!ctx) return ABFIT_ERR_ARG;
    ABFIT_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->scratch) {
        ctx->scratch = new abfit_batch();
        ctx->scratch->ctx = ctx;
    }
    *out = ctx->scratch;
    return batch_load(ctx->scratch, probs, n_probs);
}

void abfit_batch_destroy(abfit_batch *b)
{
    if (!b) return;
    cudaSetDevice(b->ctx->device);
    cudaStreamSynchronize(b->ctx->stream);
    for (auto &e : b->ev)
        if (e) cudaEventDestroy(e);
    delete b;
}

// simplices == nullptr: the caller has already put them into b->d_simplices (abfit_alphabeta_batch starts that
// copy before the pedigrees are compiled)
static int upload_starts_impl(abfit_batch *b, int32_t n_starts, const double *simplices)
{
    ABFIT_CUDA(cudaSetDevice(b->ctx->device));
    const size_t n = (size_t)b->n_probs * n_starts * 20;
    if (simplices) {
        if (int rc = b->d_simplices.ensure(n)) return rc;
        ABFIT_CUDA(cudaMemcpyAsync(b->d_simplices.p, simplices, n * 8, cudaMemcpyHostToDevice, b->ctx->stream));
    }
    if (n_starts != b->n_starts) {
        b->n_starts = n_starts;
        if (int rc = choose_launch_shape(b->hp, (size_t)b->ctx->smem_optin,
                                         (size_t)b->ctx->prop.sharedMemPerMultiprocessor, n_starts, b->shape))
            return rc;
        decide_jit(b, n_starts);
        const int n_sm = b->ctx->prop.multiProcessorCount;
        std::vector<WorkItem> items;
        if (b->jit && b->jit->sched == 2) {
            if (int rc = b->d_cursor.ensure(2)) return rc;
            b->jit_warps_fit = jit_resident_warps(b->jit, false, b->hp.probs[0], n_sm);
            if (b->jit_warps_fit <= 0) return cuda_fail(cudaGetLastError(), "occupancy of the specialised multi-start kernel");
            items = make_items_guided(b->hp, n_starts, b->jit_warps_fit, 256, true);
        } else {
            items = b->shape.wide ? make_items_wide(b->hp, n_starts, n_sm, true)
                                  : make_items(b->hp, n_starts, n_sm, b->shape.n_warps, true);
        }
        b->n_items = (int)items.size();
        if (int rc = b->d_items.ensure(items.size())) return rc;
        if (!items.empty())
            ABFIT_CUDA(cudaMemcpyAsync(b->d_items.p, items.data(), items.size() * sizeof(WorkItem),
                                       cudaMemcpyHostToDevice, b->ctx->stream));
        ABFIT_CUDA(cudaStreamSynchronize(b->ctx->stream));
        if (b->shape.x_global && !b->shape.big)
            if (int rc = b->d_xscratch.ensure((size_t)std::max(b->n_items, 1) * b->shape.n_warps * 20 * 32)) return rc;
        if (int rc = b->d_all.ensure((size_t)b->n_probs * n_starts)) return rc;
        if (int rc = b->d_best.ensure(b->n_probs)) return rc;
        if (int rc = b->d_pred.ensure((size_t)b->total_pairs)) return rc;
        if (int rc = b->d_resid.ensure((size_t)b->total_pairs)) return rc;
        if (int rc = b->d_status.ensure(b->n_probs)) return rc;
    }
    b->fit_done = false;
    return 0;
}

int abfit_batch_upload_starts(abfit_batch *b, int32_t n_starts, const double *simplices)
{
    if (!b || !simplices || n_starts <= 0) return ABFIT_ERR_ARG;
    return upload_starts_impl(b, n_starts, simplices);
}

int abfit_batch_run_fit(abfit_batch *b, int32_t max_iters, double sd_tol, uint32_t flags)
{
    if (!b || b->n_starts <= 0 || max_iters < 0) {
        set_error("run_fit: upload_starts first");
        return ABFIT_ERR_STATE;
    }
    ABFIT_CUDA(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->ctx->stream;
    const NMParams nm = nm_params(max_iters, sd_tol, flags);
    // records of skipped (NaN) problems read back as status -1 / NaN
    ABFIT_CUDA(cudaMemsetAsync(b->d_all.p, 0xFF, (size_t)b->n_probs * b->n_starts * sizeof(abfit_fit), st));
    ABFIT_CUDA(cudaMemsetAsync(b->d_evals_fit.p, 0, (size_t)b->n_probs * 8, st));
    ABFIT_CUDA(cudaEventRecord(b->ev[0], st));
    BigScratch big;
    if (int rc = big_scratch(b, (size_t)std::max(std::max(b->n_items, 1) * b->shape.n_warps, b->n_probs), big)) return rc;
    if (b->shape.wide) {
        const long long *ss_off = nullptr;
        const double *ss_all = nullptr;
        int max_trip = 0;
        const char *ess = getenv("ABFIT_EXPERIMENT_SUFFSTATS");
        if (ess && atoi(ess) != 0) {
            // EXPERIMENT, never the default (DESIGN.md §2.13): per-triple statistics of every problem, once per launch
            std::vector<long long> off(b->n_probs);
            long long total = 0;
            for (int p = 0; p < b->n_probs; ++p) {
                off[p] = total;
                total += 2 * (long long)b->hp.probs[p].n_trip + 1;
                max_trip = std::max(max_trip, (int)b->hp.probs[p].n_trip);
            }
            if (int rc = b->d_wide_ss.ensure((size_t)total)) return rc;
            if (int rc = b->d_wide_ss_off.ensure((size_t)b->n_probs)) return rc;
            ABFIT_CUDA(cudaMemcpyAsync(b->d_wide_ss_off.p, off.data(), (size_t)b->n_probs * 8, cudaMemcpyHostToDevice, st));
            ABFIT_CUDA(cudaStreamSynchronize(st));  // `off` is pageable
            if (b->shape.smem_wide + (size_t)(2 * max_trip + 2) * 8 <= (size_t)b->ctx->smem_optin) {
                if (int rc = launch_wide_stats(st, b->pools, b->n_probs, max_trip, b->d_wide_ss_off.p, b->d_wide_ss.p)) return rc;
                ss_off = b->d_wide_ss_off.p;
                ss_all = b->d_wide_ss.p;
            }
        }
        if (int rc = launch_fit_starts_wide(st, b->pools, b->d_items.p, b->n_items, b->d_simplices.p, b->n_starts, nm,
                                            b->d_all.p, b->d_evals_fit.p, b->shape.smem_wide, ss_off, ss_all, max_trip))
            return rc;
    } else if (b->jit && b->jit->sched == 2) {
        if (int rc = jit_launch_fit_starts_v2(b->jit, st, b->pools, b->d_items.p, b->n_items,
                                              (int64_t)b->n_probs * b->n_starts, b->jit_warps_fit, b->d_cursor.p,
                                              b->d_simplices.p, b->n_starts, nm, b->d_all.p, b->d_evals_fit.p,
                                              jit_smem_fit_v2(b->jit, b->hp.probs[0]), b->sx_ready))
            return rc;
    } else if (b->jit) {
        if (int rc = jit_launch_fit_starts(b->jit, st, b->pools, b->d_items.p, b->n_items, b->shape.n_warps,
                                           b->d_simplices.p, b->n_starts, nm, b->d_all.p, b->d_evals_fit.p,
                                           jit_smem_fit(b->hp.probs[0], b->shape.n_warps)))
            return rc;
    } else if (int rc = launch_fit_starts(st, b->pools, b->d_items.p, b->n_items, b->shape.n_warps, b->d_simplices.p,
                                          b->n_starts, nm, b->d_all.p, b->d_evals_fit.p, b->shape.smem_fit,
                                          b->shape.d_shared, b->shape.x_global ? b->d_xscratch.p : nullptr, big))
        return rc;
    ABFIT_CUDA(cudaEventRecord(b->ev[1], st));
    if (int rc = launch_select(st, b->pools, b->n_probs, b->n_starts, b->d_all.p, b->d_best.p, b->d_pred.p,
                               b->d_resid.p, b->d_status.p, b->shape.smem_aux, b->shape.d_shared_aux, big))
        return rc;
    ABFIT_CUDA(cudaEventRecord(b->ev[2], st));
    b->ev_fit = true;
    b->fit_done = true;
    b->pipelined_timing = false;
    b->launches_fit = (b->n_items > 0 ? 1 : 0) + 1;
    return 0;
}

int abfit_batch_download_fit(abfit_batch *b, abfit_fit *best_out, abfit_fit *all_out, double *pred_out,
                             double *resid_out, int32_t *prob_status_out)
{
    if (!b || !b->fit_done) {
        set_error("download_fit: run_fit first");
        return ABFIT_ERR_STATE;
    }
    ABFIT_CUDA(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->ctx->stream;
    if (best_out)
        ABFIT_CUDA(cudaMemcpyAsync(best_out, b->d_best.p, (size_t)b->n_probs * sizeof(abfit_fit), cudaMemcpyDeviceToHost, st));
    if (all_out)
        ABFIT_CUDA(cudaMemcpyAsync(all_out, b->d_all.p, (size_t)b->n_probs * b->n_starts * sizeof(abfit_fit),
                                   cudaMemcpyDeviceToHost, st));
    if (pred_out)
        ABFIT_CUDA(cudaMemcpyAsync(pred_out, b->d_pred.p, (size_t)b->total_pairs * 8, cudaMemcpyDeviceToHost, st));
    if (resid_out)
        ABFIT_CUDA(cudaMemcpyAsync(resid_out, b->d_resid.p, (size_t)b->total_pairs * 8, cudaMemcpyDeviceToHost, st));
    if (prob_status_out)
        ABFIT_CUDA(cudaMemcpyAsync(prob_status_out, b->d_status.p, (size_t)b->n_probs * 4, cudaMemcpyDeviceToHost, st));
    ABFIT_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// buffers and work items of a bootstrap with n_boot replicates per window (synchronises the stream when it
// has to rebuild the items, so callers that overlap do this before they enqueue kernels)
static int boot_alloc(abfit_batch *b, int32_t n_boot)
{
    cudaStream_t st = b->ctx->stream;
    const size_t n_idx = (size_t)b->total_pairs * n_boot, n_vary = (size_t)b->n_probs * n_boot * 16;
    if (int rc = b->d_idx.ensure(n_idx)) return rc;
    if (int rc = b->d_vary.ensure(n_vary)) return rc;
    decide_jit(b, n_boot);  // a bootstrap-only batch has not been through upload_starts
    const bool want_v2 = b->jit && b->jit->sched == 2 && b->shape.smem_boot_gather;
    if (n_boot != b->n_boot || want_v2 != b->boot_items_v2) {
        b->n_boot = n_boot;
        b->boot_items_v2 = want_v2;
        b->pipes_n_boot = -1;
        const bool v2 = want_v2;
        std::vector<WorkItem> items;
        if (v2) {
            if (int rc = b->d_cursor.ensure(2)) return rc;
            b->jit_warps_boot = jit_resident_warps(b->jit, true, b->hp.probs[0], b->ctx->prop.multiProcessorCount);
            if (b->jit_warps_boot <= 0) return cuda_fail(cudaGetLastError(), "occupancy of the specialised bootstrap kernel");
            items = make_items_guided(b->hp, n_boot, b->jit_warps_boot, 256, true);
        } else {
            items = b->shape.wide ? make_items_wide(b->hp, n_boot, b->ctx->prop.multiProcessorCount, true)
                                  : make_items(b->hp, n_boot, b->ctx->prop.multiProcessorCount, 1, true);
        }
        b->n_boot_items = (int)items.size();
        if (int rc = b->d_boot_items.ensure(items.size())) return rc;
        if (!items.empty())
            ABFIT_CUDA(cudaMemcpyAsync(b->d_boot_items.p, items.data(), items.size() * sizeof(WorkItem),
                                       cudaMemcpyHostToDevice, st));
        ABFIT_CUDA(cudaStreamSynchronize(st));
        // stored-D* tile: N x 32 doubles per block; index tile: ceil(N/4) x 32 x 8 bytes (+ one tile of slack for
        // the L1 prefetch that runs 4 groups ahead)
        const size_t per_block = b->shape.wide ? (size_t)((b->hp.max_pairs + 1) & ~1)  // one D* row per warp
                                 : b->shape.smem_boot_gather ? (size_t)((b->hp.max_pairs + 3) / 4) * 32
                                                             : (size_t)b->hp.max_pairs * 32;
        // (continuous scheduling: one index tile per persistent warp)
        const size_t n_tiles = v2 ? (size_t)b->jit_warps_boot : (size_t)std::max(b->n_boot_items, 1);
        if (int rc = b->d_scratch.ensure((n_tiles + 1) * per_block)) return rc;
        if (int rc = b->d_rows.ensure((size_t)b->n_probs * n_boot * 7)) return rc;
        if (int rc = b->d_bootfits.ensure((size_t)b->n_probs * n_boot)) return rc;
    }
    return 0;
}

int abfit_batch_upload_boot(abfit_batch *b, int32_t n_boot, const abfit_fit *best, const double *pred,
                            const double *resid, const int32_t *resample_idx, const double *vary_vertices)
{
    if (!b || n_boot <= 0 || !resample_idx || !vary_vertices) return ABFIT_ERR_ARG;
    ABFIT_CUDA(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->ctx->stream;
    if (best) {
        if (!pred || !resid) {
            set_error("upload_boot: best given without pred/resid");
            return ABFIT_ERR_ARG;
        }
        if (int rc = b->d_best.ensure(b->n_probs)) return rc;
        if (int rc = b->d_pred.ensure((size_t)b->total_pairs)) return rc;
        if (int rc = b->d_resid.ensure((size_t)b->total_pairs)) return rc;
        ABFIT_CUDA(cudaMemcpyAsync(b->d_best.p, best, (size_t)b->n_probs * sizeof(abfit_fit), cudaMemcpyHostToDevice, st));
        ABFIT_CUDA(cudaMemcpyAsync(b->d_pred.p, pred, (size_t)b->total_pairs * 8, cudaMemcpyHostToDevice, st));
        ABFIT_CUDA(cudaMemcpyAsync(b->d_resid.p, resid, (size_t)b->total_pairs * 8, cudaMemcpyHostToDevice, st));
    } else if (!b->fit_done) {
        set_error("upload_boot: no best model on the device (run_fit first or pass best/pred/resid)");
        return ABFIT_ERR_STATE;
    }
    if (int rc = boot_alloc(b, n_boot)) return rc;
    const size_t n_idx = (size_t)b->total_pairs * n_boot, n_vary = (size_t)b->n_probs * n_boot * 16;
    ABFIT_CUDA(cudaMemcpyAsync(b->d_idx.p, resample_idx, n_idx * 4, cudaMemcpyHostToDevice, st));
    ABFIT_CUDA(cudaMemcpyAsync(b->d_vary.p, vary_vertices, n_vary * 8, cudaMemcpyHostToDevice, st));
    b->boot_uploaded = true;
    b->boot_done = false;
    return 0;
}

int abfit_batch_run_boot(abfit_batch *b, int32_t max_iters, double sd_tol, uint32_t flags)
{
    if (!b || !b->boot_uploaded) {
        set_error("run_boot: upload_boot first");
        return ABFIT_ERR_STATE;
    }
    ABFIT_CUDA(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->ctx->stream;
    if (int rc = boot_alloc(b, b->n_boot)) return rc;  // no-op unless the kernel family changed since the upload
    const NMParams nm = nm_params(max_iters, sd_tol, flags);
    ABFIT_CUDA(cudaMemsetAsync(b->d_rows.p, 0xFF, (size_t)b->n_probs * b->n_boot * 7 * 8, st));
    ABFIT_CUDA(cudaMemsetAsync(b->d_bootfits.p, 0xFF, (size_t)b->n_probs * b->n_boot * sizeof(abfit_fit), st));
    ABFIT_CUDA(cudaMemsetAsync(b->d_evals_boot.p, 0, (size_t)b->n_probs * 8, st));
    ABFIT_CUDA(cudaEventRecord(b->ev[3], st));
    if (int rc = b->d_booterr.ensure(1)) return rc;
    ABFIT_CUDA(cudaMemsetAsync(b->d_booterr.p, 0, sizeof(int), st));
    if (b->shape.wide) {
        if (int rc = launch_fit_boot_wide(st, b->pools, b->d_boot_items.p, b->n_boot_items, b->n_boot, b->d_best.p,
                                          b->d_pred.p, b->d_resid.p, b->d_idx.p, b->d_vary.p, b->d_scratch.p,
                                          (int64_t)((b->hp.max_pairs + 1) & ~1), nm, b->d_rows.p, b->d_bootfits.p,
                                          b->d_evals_boot.p, b->shape.smem_wide, b->d_booterr.p))
            return rc;
    } else if (b->shape.smem_boot_gather && b->jit && b->jit->sched == 2) {
        if (int rc = jit_launch_fit_boot_gather_v2(b->jit, st, b->pools, b->d_boot_items.p, b->n_boot_items,
                                                   (int64_t)b->n_probs * b->n_boot, b->jit_warps_boot, b->d_cursor.p + 1,
                                                   b->n_boot, b->d_best.p, b->d_pred.p, b->d_resid.p, b->d_idx.p,
                                                   b->d_vary.p, b->d_scratch.p, (int64_t)((b->hp.max_pairs + 3) / 4) * 32,
                                                   nm, b->d_rows.p, b->d_bootfits.p, b->d_evals_boot.p,
                                                   jit_smem_boot_v2(b->jit, b->hp.probs[0]), b->d_booterr.p))
            return rc;
    } else if (b->shape.smem_boot_gather && b->jit) {
        // specialised index-tile kernel: 33 doubles of shared memory per lane, the simplex always fits
        if (int rc = jit_launch_fit_boot_gather(b->jit, st, b->pools, b->d_boot_items.p, b->n_boot_items, b->n_boot,
                                                b->d_best.p, b->d_pred.p, b->d_resid.p, b->d_idx.p, b->d_vary.p,
                                                b->d_scratch.p, (int64_t)((b->hp.max_pairs + 3) / 4) * 32, nm, b->d_rows.p,
                                                b->d_bootfits.p, b->d_evals_boot.p,
                                                jit_smem_boot_gather(b->hp.probs[0], false), b->d_booterr.p, nullptr))
            return rc;
    } else if (b->shape.smem_boot_gather) {
        double *bx = nullptr;
        if (b->shape.boot_x_global) {
            if (int rc = b->d_xscratch.ensure((size_t)std::max(b->n_boot_items, 1) * 20 * 32)) return rc;
            bx = b->d_xscratch.p;
        }
        if (int rc = launch_fit_boot_gather(st, b->pools, b->d_boot_items.p, b->n_boot_items, b->n_boot, b->d_best.p,
                                            b->d_pred.p, b->d_resid.p, b->d_idx.p, b->d_vary.p, b->d_scratch.p,
                                            (int64_t)((b->hp.max_pairs + 3) / 4) * 32, nm, b->d_rows.p, b->d_bootfits.p,
                                            b->d_evals_boot.p, b->shape.smem_boot_gather, b->d_booterr.p, bx))
            return rc;
    } else {
        BigScratch big;
        if (int rc = big_scratch(b, (size_t)std::max(b->n_boot_items, 1), big)) return rc;
        if (int rc = launch_fit_boot(st, b->pools, b->d_boot_items.p, b->n_boot_items, b->n_boot, b->d_best.p,
                                     b->d_pred.p, b->d_resid.p, b->d_idx.p, b->d_vary.p, b->d_scratch.p,
                                     (int64_t)b->hp.max_pairs * 32, nm, b->d_rows.p, b->d_bootfits.p,
                                     b->d_evals_boot.p, b->shape.smem_boot, b->d_booterr.p, big))
            return rc;
    }
    ABFIT_CUDA(cudaEventRecord(b->ev[4], st));
    b->ev_boot = true;
    b->boot_done = true;
    b->launches_boot = b->n_boot_items > 0 ? 1 : 0;
    return 0;
}

// ---------------------------------------------------------------------------------------
// pipelined fit -> select -> bootstrap
//
// A multi-start launch cannot end before its longest fit does, and among a million fits some run for thousands of
// iterations: ~30 ms at the end of every launch during which the machine drains (measured: launch time =
// 0.162 ms x windows + 32 ms).  Only a window's OWN best-of-starts gates its bootstrap, so the batch is cut into
// sub-batches of windows, each a fit -> select -> (vary) -> bootstrap chain on its own stream: while the last long
// fits of one sub-batch finish, the freed warps already run the next sub-batch's fits, and the bootstraps fill what
// is left.  Same kernels, same items-to-fits mapping inside a sub-batch: same bits.
// ---------------------------------------------------------------------------------------
static int plan_pipes(abfit_batch *b)
{
    abfit_ctx *ctx = b->ctx;
    const bool v2 = b->jit && b->jit->sched == 2 && b->shape.smem_boot_gather && !b->shape.wide && !b->shape.big;
    if (!v2 || b->n_starts <= 0 || b->n_boot <= 0) {
        b->pipes.clear();
        return 0;
    }
    if (b->pipes_n_starts == b->n_starts && b->pipes_n_boot == b->n_boot && !b->pipes.empty()) return 0;
    int K = 1;
    if (const char *e = getenv("ABFIT_DEV_PIPES")) K = std::max(1, std::min<int>(abfit_ctx::MAX_PIPES, atoi(e)));
    K = std::min(K, b->n_probs);
    b->pipes.assign(K, abfit_batch::Pipe());
    std::vector<WorkItem> all;
    for (int k = 0; k < K; ++k) {
        abfit_batch::Pipe &pp = b->pipes[k];
        pp.p0 = (int)((int64_t)b->n_probs * k / K);
        pp.n = (int)((int64_t)b->n_probs * (k + 1) / K) - pp.p0;
        std::vector<WorkItem> it = make_items_guided(b->hp, b->n_starts, b->jit_warps_fit, 256, true, pp.p0, pp.p0 + pp.n);
        pp.fit_item0 = (int)all.size();
        pp.fit_items = (int)it.size();
        all.insert(all.end(), it.begin(), it.end());
    }
    for (int k = 0; k < K; ++k) {
        abfit_batch::Pipe &pp = b->pipes[k];
        std::vector<WorkItem> it = make_items_guided(b->hp, b->n_boot, b->jit_warps_boot, 256, true, pp.p0, pp.p0 + pp.n);
        pp.boot_item0 = (int)all.size();
        pp.boot_items = (int)it.size();
        all.insert(all.end(), it.begin(), it.end());
    }
    if (int rc = b->d_pipe_items.ensure(all.size())) return rc;
    if (int rc = b->d_pipe_cursor.ensure(2 * abfit_ctx::MAX_PIPES)) return rc;
    if (!all.empty())
        ABFIT_CUDA(cudaMemcpyAsync(b->d_pipe_items.p, all.data(), all.size() * sizeof(WorkItem), cudaMemcpyHostToDevice, ctx->stream));
    ABFIT_CUDA(cudaStreamSynchronize(ctx->stream));  // `all` is pageable host memory
    for (int k = 0; k < K; ++k) {
        if (!ctx->pipe_stream[k]) ABFIT_CUDA(cudaStreamCreateWithFlags(&ctx->pipe_stream[k], cudaStreamNonBlocking));
        if (!ctx->pipe_done[k]) ABFIT_CUDA(cudaEventCreateWithFlags(&ctx->pipe_done[k], cudaEventDisableTiming));
    }
    if (!ctx->pipe_start) ABFIT_CUDA(cudaEventCreateWithFlags(&ctx->pipe_start, cudaEventDisableTiming));
    b->pipes_n_starts = b->n_starts;
    b->pipes_n_boot = b->n_boot;
    return 0;
}

// gen_vary: draw the vary vertices on the device behind each sub-batch's selection (abfit_alphabeta_batch), else the
// uploaded ones are used.  before_boot: optional event the bootstraps have to wait for (the resample indices' H2D copy).
static int run_pipelined_impl(abfit_batch *b, int32_t max_iters_fit, int32_t max_iters_boot, double sd_tol, uint32_t flags,
                              bool gen_vary, uint64_t vary_seed, uint64_t first_problem_id, const unsigned long long *d_ids,
                              cudaEvent_t before_boot)
{
    abfit_ctx *ctx = b->ctx;
    if (int rc = plan_pipes(b)) return rc;
    cudaStream_t st = ctx->stream;
    if (b->pipes.size() <= 1) {  // nothing to overlap (or not the continuous-scheduling kernels): one after the other
        if (int rc = abfit_batch_run_fit(b, max_iters_fit, sd_tol, flags)) return rc;
        if (gen_vary)
            if (int rc = launch_gen_vary(st, vary_seed, first_problem_id, d_ids, b->n_probs, b->n_boot, b->d_best.p, b->d_vary.p))
                return rc;
        if (before_boot) ABFIT_CUDA(cudaStreamWaitEvent(st, before_boot, 0));
        b->boot_uploaded = true;
        return abfit_batch_run_boot(b, max_iters_boot, sd_tol, flags);
    }
    const NMParams nm_fit = nm_params(max_iters_fit, sd_tol, flags), nm_boot = nm_params(max_iters_boot, sd_tol, flags);
    if (b->sx_ready) ABFIT_CUDA(cudaStreamWaitEvent(st, ctx->copy_done, 0));  // the sub-batch launches do not watch the upload
    ABFIT_CUDA(cudaMemsetAsync(b->d_all.p, 0xFF, (size_t)b->n_probs * b->n_starts * sizeof(abfit_fit), st));
    ABFIT_CUDA(cudaMemsetAsync(b->d_evals_fit.p, 0, (size_t)b->n_probs * 8, st));
    ABFIT_CUDA(cudaMemsetAsync(b->d_rows.p, 0xFF, (size_t)b->n_probs * b->n_boot * 7 * 8, st));
    ABFIT_CUDA(cudaMemsetAsync(b->d_bootfits.p, 0xFF, (size_t)b->n_probs * b->n_boot * sizeof(abfit_fit), st));
    ABFIT_CUDA(cudaMemsetAsync(b->d_evals_boot.p, 0, (size_t)b->n_probs * 8, st));
    if (int rc = b->d_booterr.ensure(1)) return rc;
    ABFIT_CUDA(cudaMemsetAsync(b->d_booterr.p, 0, sizeof(int), st));
    ABFIT_CUDA(cudaEventRecord(b->ev[0], st));
    ABFIT_CUDA(cudaEventRecord(ctx->pipe_start, st));
    BigScratch none;
    const DevProblem &pb0 = b->hp.probs[0];
    const int64_t tile_stride = (int64_t)((b->hp.max_pairs + 3) / 4) * 32;
    // every sub-batch's bootstrap kernel gets its own range of index tiles
    if (int rc = b->d_scratch.ensure(((size_t)b->jit_warps_boot * b->pipes.size() + 1) * (size_t)tile_stride)) return rc;
    for (size_t k = 0; k < b->pipes.size(); ++k) {
        const abfit_batch::Pipe &pp = b->pipes[k];
        cudaStream_t ps = ctx->pipe_stream[k];
        ABFIT_CUDA(cudaStreamWaitEvent(ps, ctx->pipe_start, 0));
        if (int rc = jit_launch_fit_starts_v2(b->jit, ps, b->pools, b->d_pipe_items.p + pp.fit_item0, pp.fit_items,
                                              (int64_t)pp.n * b->n_starts, b->jit_warps_fit, b->d_pipe_cursor.p + 2 * k,
                                              b->d_simplices.p, b->n_starts, nm_fit, b->d_all.p, b->d_evals_fit.p,
                                              jit_smem_fit_v2(b->jit, pb0)))
            return rc;
        if (int rc = launch_select(ps, b->pools, pp.n, b->n_starts, b->d_all.p, b->d_best.p, b->d_pred.p, b->d_resid.p,
                                   b->d_status.p, b->shape.smem_aux, b->shape.d_shared_aux, none, pp.p0))
            return rc;
        if (gen_vary)
            if (int rc = launch_gen_vary(ps, vary_seed, first_problem_id + (uint64_t)pp.p0, d_ids ? d_ids + pp.p0 : nullptr, pp.n,
                                         b->n_boot, b->d_best.p + pp.p0, b->d_vary.p + (size_t)pp.p0 * b->n_boot * 16))
                return rc;
        if (before_boot) ABFIT_CUDA(cudaStreamWaitEvent(ps, before_boot, 0));
        if (int rc = jit_launch_fit_boot_gather_v2(
                b->jit, ps, b->pools, b->d_pipe_items.p + pp.boot_item0, pp.boot_items, (int64_t)pp.n * b->n_boot,
                b->jit_warps_boot, b->d_pipe_cursor.p + 2 * k + 1, b->n_boot, b->d_best.p, b->d_pred.p, b->d_resid.p, b->d_idx.p,
                b->d_vary.p, reinterpret_cast<uint2 *>(b->d_scratch.p) + (size_t)k * b->jit_warps_boot * tile_stride, tile_stride,
                nm_boot, b->d_rows.p, b->d_bootfits.p, b->d_evals_boot.p, jit_smem_boot_v2(b->jit, pb0), b->d_booterr.p))
            return rc;
        ABFIT_CUDA(cudaEventRecord(ctx->pipe_done[k], ps));
        ABFIT_CUDA(cudaStreamWaitEvent(st, ctx->pipe_done[k], 0));
    }
    for (int e = 1; e <= 4; ++e) ABFIT_CUDA(cudaEventRecord(b->ev[e], st));
    b->ev_fit = b->ev_boot = true;
    b->pipelined_timing = true;
    b->fit_done = b->boot_done = b->boot_uploaded = true;
    b->launches_fit = 2 * (int)b->pipes.size();
    b->launches_boot = (int)b->pipes.size() * (gen_vary ? 2 : 1);
    return 0;
}

int abfit_batch_run_pipelined(abfit_batch *b, int32_t max_iters_fit, int32_t max_iters_boot, double sd_tol, uint32_t flags)
{
    if (!b || b->n_starts <= 0 || !b->boot_uploaded) {
        set_error("run_pipelined: upload_starts and upload_boot first");
        return ABFIT_ERR_STATE;
    }
    ABFIT_CUDA(cudaSetDevice(b->ctx->device));
    return run_pipelined_impl(b, max_iters_fit, max_iters_boot, sd_tol, flags, false, 0, 0, nullptr, nullptr);
}

int abfit_batch_pipes(abfit_batch *b)
{
    return b ? (int)std::max<size_t>(1, b->pipes.size()) : 0;
}

int abfit_batch_download_boot(abfit_batch *b, double *rows_out, abfit_fit *fits_out)
{
    if (!b || !b->boot_done) {
        set_error("download_boot: run_boot first");
        return ABFIT_ERR_STATE;
    }
    ABFIT_CUDA(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->ctx->stream;
    if (rows_out)
        ABFIT_CUDA(cudaMemcpyAsync(rows_out, b->d_rows.p, (size_t)b->n_probs * b->n_boot * 7 * 8, cudaMemcpyDeviceToHost, st));
    if (fits_out)
        ABFIT_CUDA(cudaMemcpyAsync(fits_out, b->d_bootfits.p, (size_t)b->n_probs * b->n_boot * sizeof(abfit_fit),
                                   cudaMemcpyDeviceToHost, st));
    int err = 0;
    ABFIT_CUDA(cudaMemcpyAsync(&err, b->d_booterr.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    ABFIT_CUDA(cudaStreamSynchronize(st));
    if (err) {
        set_error("resample_idx contains an index outside [0, n_pairs)");
        return ABFIT_ERR_ARG;
    }
    return 0;
}

int abfit_batch_sync(abfit_batch *b)
{
    if (!b) return ABFIT_ERR_ARG;
    ABFIT_CUDA(cudaSetDevice(b->ctx->device));
    ABFIT_CUDA(cudaStreamSynchronize(b->ctx->stream));
    return 0;
}

int abfit_batch_timing(abfit_batch *b, float ms[3], int64_t evals[2], int32_t *launches)
{
    if (!b) return ABFIT_ERR_ARG;
    ABFIT_CUDA(cudaSetDevice(b->ctx->device));
    ABFIT_CUDA(cudaStreamSynchronize(b->ctx->stream));
    if (ms) {
        ms[0] = ms[1] = ms[2] = 0.f;
        if (b->pipelined_timing) {
            // the sub-batches' kernels overlap: only the whole span is meaningful, reported as ms[0]
            ABFIT_CUDA(cudaEventElapsedTime(&ms[0], b->ev[0], b->ev[4]));
        } else if (b->ev_fit) {
            ABFIT_CUDA(cudaEventElapsedTime(&ms[0], b->ev[0], b->ev[1]));
            ABFIT_CUDA(cudaEventElapsedTime(&ms[1], b->ev[1], b->ev[2]));
        }
        if (b->ev_boot && !b->pipelined_timing) ABFIT_CUDA(cudaEventElapsedTime(&ms[2], b->ev[3], b->ev[4]));
    }
    if (evals) {
        std::vector<unsigned long long> h(b->n_probs);
        evals[0] = evals[1] = 0;
        ABFIT_CUDA(cudaMemcpy(h.data(), b->d_evals_fit.p, (size_t)b->n_probs * 8, cudaMemcpyDeviceToHost));
        for (auto v : h) evals[0] += (int64_t)v;
        ABFIT_CUDA(cudaMemcpy(h.data(), b->d_evals_boot.p, (size_t)b->n_probs * 8, cudaMemcpyDeviceToHost));
        for (auto v : h) evals[1] += (int64_t)v;
    }
    if (launches) *launches = (b->ev_fit ? b->launches_fit : 0) + (b->ev_boot ? b->launches_boot : 0);
    return 0;
}

int abfit_batch_flops_per_eval(abfit_batch *b, int32_t p, double *flops_out, int32_t *n_triples_out,
                               int32_t *tmax_out)
{
    if (!b || p < 0 || p >= b->n_probs) return ABFIT_ERR_ARG;
    if (flops_out) *flops_out = b->hp.flops[p];
    if (n_triples_out) *n_triples_out = b->hp.n_triples[p];
    if (tmax_out) *tmax_out = b->hp.tmax[p];
    return 0;
}

int abfit_jit_dump(const abfit_problem *prob, const char *source_path, const char *cubin_path, double *compile_seconds)
{
    if (!prob) return ABFIT_ERR_ARG;
    HostPlan hp;
    if (int rc = compile_problems(prob, 1, hp)) return rc;
    const std::string src = jit_generate_source(hp, 0, jit_default_sched());
    if (source_path) {
        FILE *f = fopen(source_path, "wb");
        if (!f) {
            set_error(std::string("cannot write ") + source_path);
            return ABFIT_ERR_ARG;
        }
        fwrite(src.data(), 1, src.size(), f);
        fclose(f);
    }
    if (compile_seconds) *compile_seconds = 0.0;
    if (cubin_path) {
        std::string cubin, log;
        bool disk = false;
        if (int rc = jit_compile(src, cubin, log, compile_seconds, &disk)) {
            set_error(log);
            return rc;
        }
        FILE *f = fopen(cubin_path, "wb");
        if (!f) {
            set_error(std::string("cannot write ") + cubin_path);
            return ABFIT_ERR_ARG;
        }
        fwrite(cubin.data(), 1, cubin.size(), f);
        fclose(f);
    }
    return 0;
}

int abfit_batch_uses_specialised_kernels(abfit_batch *b)
{
    return b && b->jit ? 1 : 0;
}

const char *abfit_jit_last_error(void)
{
    static thread_local std::string s;
    s = jit_last_note();
    return s.c_str();
}

int abfit_batch_fp64_instr_per_eval(abfit_batch *b, int32_t p, double *instr_out)
{
    if (!b || p < 0 || p >= b->n_probs || !instr_out) return ABFIT_ERR_ARG;
    *instr_out = b->hp.fp64_instr[p];
    return 0;
}

// ---------------------------------------------------------------------------------------
// one-shot host-buffer entry points
// ---------------------------------------------------------------------------------------
int abfit_fit_batch(abfit_ctx *ctx, const abfit_problem *probs, int32_t n_probs, int32_t n_starts,
                    const double *simplices, int32_t max_iters, double sd_tol, uint32_t flags,
                    abfit_fit *best_out, abfit_fit *all_out, double *pred_out, double *resid_out,
                    int32_t *prob_status_out)
{
    abfit_batch *b = nullptr;
    if (int rc = workspace(ctx, probs, n_probs, &b)) return rc;
    if (int rc = abfit_batch_upload_starts(b, n_starts, simplices)) return rc;
    if (int rc = abfit_batch_run_fit(b, max_iters, sd_tol, flags)) return rc;
    return abfit_batch_download_fit(b, best_out, all_out, pred_out, resid_out, prob_status_out);
}

int abfit_boot_batch(abfit_ctx *ctx, const abfit_problem *probs, int32_t n_probs, const abfit_fit *best,
                     const double *pred, const double *resid, int32_t n_boot, const int32_t *resample_idx,
                     const double *vary_vertices, int32_t max_iters, double sd_tol, uint32_t flags,
                     double *rows_out, abfit_fit *fits_out)
{
    if (!best || !pred || !resid) {
        set_error("boot_batch: best, pred and resid are required");
        return ABFIT_ERR_ARG;
    }
    abfit_batch *b = nullptr;
    if (int rc = workspace(ctx, probs, n_probs, &b)) return rc;
    if (int rc = abfit_batch_upload_boot(b, n_boot, best, pred, resid, resample_idx, vary_vertices)) return rc;
    if (int rc = abfit_batch_run_boot(b, max_iters, sd_tol, flags)) return rc;
    return abfit_batch_download_boot(b, rows_out, fits_out);
}

void abfit_gen_vary_vertices_batch(uint64_t seed, uint64_t first_problem_id, int32_t n_probs, int32_t n_boot,
                                   const abfit_fit *best, double *out)
{
    parallel_for(n_probs, [=](int32_t p) {
        abfit_gen_vary_vertices(seed, first_problem_id + (uint64_t)p, n_boot, best[p].theta, out + (size_t)p * n_boot * 16);
    });
}

static int alphabeta_impl(abfit_ctx *ctx, const abfit_problem *probs, int32_t n_probs, int32_t n_starts,
                          const double *simplices, int32_t n_boot, const int32_t *resample_idx, uint64_t vary_seed,
                          uint64_t first_problem_id, const uint64_t *problem_ids, int32_t max_iters_fit,
                          int32_t max_iters_boot, double sd_tol, uint32_t flags, abfit_fit *best_out, double *pred_out,
                          double *resid_out, int32_t *prob_status_out, double *rows_out, double *analysis_out)
{
    if (!simplices || n_starts <= 0 || n_boot <= 0 || !rows_out) return ABFIT_ERR_ARG;  // (resample_idx NULL: drawn on the device)
    if (!ctx || n_probs <= 0) return ABFIT_ERR_ARG;
    ABFIT_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->scratch) {
        ctx->scratch = new abfit_batch();
        ctx->scratch->ctx = ctx;
    }
    abfit_batch *b = ctx->scratch;
    cudaStream_t st = ctx->stream;
    // ABFIT_DEV_VERBOSE: host-side phases of the call (wall clock)
    const bool verbose = getenv("ABFIT_DEV_VERBOSE") != nullptr;
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto t_prev = now();
    const auto t_first = t_prev;
    auto phase = [&](const char *name) {
        if (!verbose) return;
        const auto t = now();
        fprintf(stderr, "[abfit] alphabeta_batch: %-28s %8.2f ms (at %8.2f)\n", name, std::chrono::duration<double, std::milli>(t - t_prev).count(),
                std::chrono::duration<double, std::milli>(t - t_first).count());
        t_prev = t;
    };
    // the start simplices (the bulk of the fit's input) cross PCIe while the host compiles the pedigrees
    const size_t n_sx = (size_t)n_probs * n_starts * 20;
    if (b->d_simplices.n < n_sx || !b->d_simplices.p) {
        ABFIT_CUDA(cudaStreamSynchronize(st));  // the buffer is about to be reallocated
        if (int rc = b->d_simplices.ensure(n_sx)) return rc;
    }
    if (!ctx->h_sx_counts) {
        ABFIT_CUDA(cudaHostAlloc(&ctx->h_sx_counts, abfit_ctx::SX_CHUNKS * sizeof(int), cudaHostAllocDefault));
        ABFIT_CUDA(cudaMalloc(&ctx->d_sx_ready, sizeof(int)));
    }
    if (!ctx->sx_reset) ABFIT_CUDA(cudaEventCreateWithFlags(&ctx->sx_reset, cudaEventDisableTiming));
    {
        const int per = std::max(256, (n_probs + abfit_ctx::SX_CHUNKS - 1) / abfit_ctx::SX_CHUNKS);  // windows per chunk
        ABFIT_CUDA(cudaMemsetAsync(ctx->d_sx_ready, 0, sizeof(int), ctx->copy_stream));
        ABFIT_CUDA(cudaEventRecord(ctx->sx_reset, ctx->copy_stream));
        int c = 0;
        for (int p0 = 0; p0 < n_probs; p0 += per, ++c) {
            const int p1 = std::min(n_probs, p0 + per);
            const size_t o = (size_t)p0 * n_starts * 20, cnt = (size_t)(p1 - p0) * n_starts * 20;
            ABFIT_CUDA(cudaMemcpyAsync(b->d_simplices.p + o, simplices + o, cnt * 8, cudaMemcpyHostToDevice, ctx->copy_stream));
            ctx->h_sx_counts[c] = p1;
            ABFIT_CUDA(cudaMemcpyAsync(ctx->d_sx_ready, ctx->h_sx_counts + c, sizeof(int), cudaMemcpyHostToDevice, ctx->copy_stream));
        }
    }
    ABFIT_CUDA(cudaEventRecord(ctx->copy_done, ctx->copy_stream));
    phase("enqueue simplices copy");
    if (int rc = workspace(ctx, probs, n_probs, &b)) return rc;
    phase("compile pedigrees + pools");
    decide_jit(b, (int64_t)n_starts + n_boot);  // one decision for both phases of this batch
    phase("decide_jit");
    if (int rc = upload_starts_impl(b, n_starts, nullptr)) return rc;  // before any kernel is enqueued: these may synchronise
    phase("plan multi-start items");
    if (int rc = boot_alloc(b, n_boot)) return rc;
    if (analysis_out) {  // (allocations before any kernel is enqueued: cudaFree synchronises)
        if (int rc = b->d_analysis.ensure((size_t)n_probs * 32)) return rc;
        if (int rc = b->d_analysis_scratch.ensure((size_t)n_probs * 8 * std::max(n_boot, 1))) return rc;
    }
    phase("plan bootstrap items");
    // the continuous-scheduling kernel watches the upload's counter; every other kernel family waits for the whole copy
    const bool watch_upload = b->jit && b->jit->sched == 2 && !b->shape.wide && !getenv("ABFIT_DEV_NO_UPLOAD_WATCH");
    // watching: the counter still holds the previous call's count until its reset lands, so the kernel waits for that
    ABFIT_CUDA(cudaStreamWaitEvent(st, watch_upload ? ctx->sx_reset : ctx->copy_done, 0));
    if (verbose && watch_upload) fprintf(stderr, "[abfit] alphabeta_batch: the multi-start kernel watches the upload\n");
    b->sx_ready = watch_upload ? ctx->d_sx_ready : nullptr;
    const unsigned long long *d_ids = nullptr;
    if (problem_ids) {  // every window keeps its own key, whatever its position in this batch
        if (int rc = b->d_ids.ensure(n_probs)) return rc;
        ABFIT_CUDA(cudaMemcpyAsync(b->d_ids.p, problem_ids, (size_t)n_probs * 8, cudaMemcpyHostToDevice, st));
        d_ids = b->d_ids.p;
    }
    if (!ctx->idx_done) ABFIT_CUDA(cudaEventCreateWithFlags(&ctx->idx_done, cudaEventDisableTiming));
    if (resample_idx) {
        // the resample indices (the bulk of the bootstrap's input) cross PCIe under the multi-start kernels
        ABFIT_CUDA(cudaMemcpyAsync(b->d_idx.p, resample_idx, (size_t)b->total_pairs * n_boot * 4, cudaMemcpyHostToDevice,
                                   ctx->copy_stream));
        ABFIT_CUDA(cudaEventRecord(ctx->idx_done, ctx->copy_stream));
    } else {
        // ... or are drawn on the device (boot_model::run draws them itself, src/boot_model.rs:43-48): the numbers of
        // abfit_gen_resample_idx(vary_seed, window key, ...), ahead of the fit kernels on the same stream
        if (int rc = launch_gen_resample(st, vary_seed, first_problem_id, d_ids, b->pools.probs, n_probs, n_boot, b->d_idx.p)) return rc;
        ABFIT_CUDA(cudaEventRecord(ctx->idx_done, st));
    }
    // fit -> select -> Model::vary x 4 per replicate around each window's best model (src/boot_model.rs:69-75: drawn on
    // the device right behind the selection kernel — the same numbers abfit_gen_vary_vertices gives on the host — so
    // the bootstrap starts without a round trip through the host) -> bootstrap, pipelined over sub-batches of windows
    b->boot_uploaded = true;
    b->boot_done = false;
    if (int rc = run_pipelined_impl(b, max_iters_fit, max_iters_boot, sd_tol, flags, true, vary_seed, first_problem_id, d_ids,
                                    ctx->idx_done)) {
        b->sx_ready = nullptr;
        return rc;
    }
    b->sx_ready = nullptr;
    phase("enqueue kernels");
    if (best_out)
        ABFIT_CUDA(cudaMemcpyAsync(best_out, b->d_best.p, (size_t)n_probs * sizeof(abfit_fit), cudaMemcpyDeviceToHost, st));
    if (pred_out)
        ABFIT_CUDA(cudaMemcpyAsync(pred_out, b->d_pred.p, (size_t)b->total_pairs * 8, cudaMemcpyDeviceToHost, st));
    if (resid_out)
        ABFIT_CUDA(cudaMemcpyAsync(resid_out, b->d_resid.p, (size_t)b->total_pairs * 8, cudaMemcpyDeviceToHost, st));
    if (prob_status_out)
        ABFIT_CUDA(cudaMemcpyAsync(prob_status_out, b->d_status.p, (size_t)n_probs * 4, cudaMemcpyDeviceToHost, st));
    // bootstrap statistics (RawAnalysis::analyze) behind the bootstrap kernel, on the device: the same operations in the
    // same order as abfit_analyze (tests/test_gpu_parity.py::test_device_statistics_equal_host_statistics)
    const bool dev_stats = analysis_out && n_boot >= 2 && !getenv("ABFIT_DEV_HOST_STATS");
    if (dev_stats) {
        if (int rc = launch_analyze(st, b->d_rows.p, n_probs, n_boot, b->d_analysis.p, b->d_analysis_scratch.p)) return rc;
        ABFIT_CUDA(cudaMemcpyAsync(analysis_out, b->d_analysis.p, (size_t)n_probs * 32 * 8, cudaMemcpyDeviceToHost, st));
    }
    if (int rc = abfit_batch_download_boot(b, rows_out, nullptr)) return rc;
    phase("kernels + downloads");
    if (analysis_out && !dev_stats) {
        std::vector<int> rcs(n_probs, 0);
        parallel_for(n_probs, [&](int32_t p) {
            rcs[p] = abfit_analyze(rows_out + (size_t)p * n_boot * 7, n_boot, analysis_out + (size_t)p * 32);
        });
    }
    phase("bootstrap statistics");
    return 0;
}

int abfit_alphabeta_batch(abfit_ctx *ctx, const abfit_problem *probs, int32_t n_probs, int32_t n_starts,
                          const double *simplices, int32_t n_boot, const int32_t *resample_idx, uint64_t vary_seed,
                          uint64_t first_problem_id, int32_t max_iters_fit, int32_t max_iters_boot, double sd_tol,
                          uint32_t flags, abfit_fit *best_out, double *pred_out, double *resid_out,
                          int32_t *prob_status_out, double *rows_out, double *analysis_out)
{
    return alphabeta_impl(ctx, probs, n_probs, n_starts, simplices, n_boot, resample_idx, vary_seed, first_problem_id,
                          nullptr, max_iters_fit, max_iters_boot, sd_tol, flags, best_out, pred_out, resid_out,
                          prob_status_out, rows_out, analysis_out);
}

// contiguous, balanced block of `n` units for shard r of `world`
static void shard_range(int64_t n, int r, int world, int64_t &first, int64_t &count)
{
    const int64_t base = n / world, extra = n % world;
    first = (int64_t)r * base + std::min<int64_t>(r, extra);
    count = base + (r < extra ? 1 : 0);
}

int abfit_alphabeta_batch_multi(abfit_ctx *const *ctxs, int32_t n_ctx, const abfit_problem *probs, int32_t n_probs,
                                int32_t n_starts, const double *simplices, int32_t n_boot, const int32_t *resample_idx,
                                uint64_t vary_seed, uint64_t first_problem_id, const uint64_t *problem_ids,
                                int32_t max_iters_fit, int32_t max_iters_boot, double sd_tol, uint32_t flags,
                                abfit_fit *best_out, double *pred_out, double *resid_out, int32_t *prob_status_out,
                                double *rows_out, double *analysis_out)
{
    if (!ctxs || n_ctx <= 0 || !probs || n_probs <= 0 || !simplices || !rows_out) return ABFIT_ERR_ARG;
    for (int r = 0; r < n_ctx; ++r)
        if (!ctxs[r]) return ABFIT_ERR_ARG;
    const int world = std::min<int>(n_ctx, n_probs);
    std::vector<int64_t> pair_off((size_t)n_probs + 1, 0);
    for (int p = 0; p < n_probs; ++p) pair_off[p + 1] = pair_off[p] + std::max(probs[p].n_pairs, 0);
    std::vector<int> rcs(world, 0);
    std::vector<std::string> errs(world);
    auto work = [&](int r) {
        int64_t first, count;
        shard_range(n_probs, r, world, first, count);
        const int64_t po = pair_off[first];
        rcs[r] = alphabeta_impl(ctxs[r], probs + first, (int32_t)count, n_starts, simplices + (size_t)first * n_starts * 20,
                                n_boot, resample_idx ? resample_idx + (size_t)po * n_boot : nullptr, vary_seed,
                                first_problem_id + (uint64_t)first,
                                problem_ids ? problem_ids + first : nullptr, max_iters_fit, max_iters_boot, sd_tol, flags,
                                best_out ? best_out + first : nullptr, pred_out ? pred_out + po : nullptr,
                                resid_out ? resid_out + po : nullptr, prob_status_out ? prob_status_out + first : nullptr,
                                rows_out + (size_t)first * n_boot * 7, analysis_out ? analysis_out + (size_t)first * 32 : nullptr);
        if (rcs[r]) errs[r] = g_last_error;  // thread-local: carry it over to the caller's thread
    };
    // one host thread + context per device; the shards never exchange data (SURVEY.md §8e)
    std::vector<std::thread> th;
    for (int r = 1; r < world; ++r) th.emplace_back(work, r);
    work(0);
    for (auto &t : th) t.join();
    for (int r = 0; r < world; ++r)
        if (rcs[r]) {
            set_error("device shard " + std::to_string(r) + ": " + errs[r]);
            return rcs[r];
        }
    return 0;
}

int abfit_cost_batch(abfit_ctx *ctx, const abfit_problem *probs, int32_t n_probs, const int32_t *prob_of_theta,
                     const double *theta, int32_t B, double *cost_out, double *lse_out)
{
    if (!theta || !cost_out || B <= 0) return ABFIT_ERR_ARG;
    abfit_batch *b = nullptr;
    if (int rc = workspace(ctx, probs, n_probs, &b)) return rc;
    // group thetas by problem (stable), 32 per warp
    std::vector<int32_t> order(B);
    std::vector<std::vector<int32_t>> by_prob(n_probs);
    for (int32_t i = 0; i < B; ++i) {
        const int32_t p = prob_of_theta ? prob_of_theta[i] : 0;
        if (p < 0 || p >= n_probs) {
            set_error("prob_of_theta out of range");
            return ABFIT_ERR_ARG;
        }
        by_prob[p].push_back(i);
    }
    std::vector<double> th((size_t)B * 4);
    std::vector<WorkItem> items;
    int32_t pos = 0;
    for (int32_t p = 0; p < n_probs; ++p) {
        const auto &v = by_prob[p];
        for (size_t f = 0; f < v.size(); f += 32) {
            WorkItem it{p, pos, (int32_t)std::min<size_t>(32, v.size() - f), 0};
            for (int32_t q = 0; q < it.count; ++q) {
                order[pos] = v[f + q];
                std::memcpy(&th[(size_t)pos * 4], theta + (size_t)v[f + q] * 4, 32);
                ++pos;
            }
            items.push_back(it);
        }
    }
    cudaStream_t st = ctx->stream;
    DevBuf<double> d_th, d_cost, d_lse;
    DevBuf<WorkItem> d_items;
    if (int rc = d_th.ensure((size_t)B * 4)) return rc;
    if (int rc = d_cost.ensure(B)) return rc;
    if (int rc = d_lse.ensure(B)) return rc;
    if (int rc = d_items.ensure(items.size())) return rc;
    ABFIT_CUDA(cudaMemcpyAsync(d_th.p, th.data(), (size_t)B * 32, cudaMemcpyHostToDevice, st));
    ABFIT_CUDA(cudaMemcpyAsync(d_items.p, items.data(), items.size() * sizeof(WorkItem), cudaMemcpyHostToDevice, st));
    BigScratch big;
    if (int rc = big_scratch(b, std::max<size_t>(items.size(), 1), big)) return rc;
    if (int rc = launch_cost_batch(st, b->pools, d_items.p, (int)items.size(), d_th.p, d_cost.p, d_lse.p,
                                   b->shape.smem_aux, b->shape.d_shared_aux, big))
        return rc;
    std::vector<double> hc(B), hl(B);
    ABFIT_CUDA(cudaMemcpyAsync(hc.data(), d_cost.p, (size_t)B * 8, cudaMemcpyDeviceToHost, st));
    ABFIT_CUDA(cudaMemcpyAsync(hl.data(), d_lse.p, (size_t)B * 8, cudaMemcpyDeviceToHost, st));
    ABFIT_CUDA(cudaStreamSynchronize(st));
    for (int32_t i = 0; i < B; ++i) {
        cost_out[order[i]] = hc[i];
        if (lse_out) lse_out[order[i]] = hl[i];
    }
    return 0;
}

int abfit_model_divergence(abfit_ctx *ctx, const abfit_problem *prob, const double theta[4], double *dt1t2_out,
                           double *p_uu_out)
{
    if (!prob || !theta || !dt1t2_out) return ABFIT_ERR_ARG;
    abfit_batch *wb = nullptr;
    if (int rc = workspace(ctx, prob, 1, &wb)) return rc;
    cudaStream_t st = ctx->stream;
    DevBuf<double> d_th, d_dt, d_puu;
    if (int rc = d_th.ensure(4)) return rc;
    if (int rc = d_dt.ensure(prob->n_pairs)) return rc;
    if (int rc = d_puu.ensure(1)) return rc;
    ABFIT_CUDA(cudaMemcpyAsync(d_th.p, theta, 32, cudaMemcpyHostToDevice, st));
    BigScratch big;
    if (int rc = big_scratch(wb, 1, big)) return rc;
    if (int rc = launch_model_divergence(st, wb->pools, d_th.p, d_dt.p, d_puu.p,
                                         wb->shape.big ? wb->shape.smem_aux : smem_need(wb->hp.probs[0], 0, false, 1), big))
        return rc;
    ABFIT_CUDA(cudaMemcpyAsync(dt1t2_out, d_dt.p, (size_t)prob->n_pairs * 8, cudaMemcpyDeviceToHost, st));
    if (p_uu_out) ABFIT_CUDA(cudaMemcpyAsync(p_uu_out, d_puu.p, 8, cudaMemcpyDeviceToHost, st));
    ABFIT_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// pitch: row stride (in sites) of the three HOST arrays when they are column slices of wider matrices (0: L)
// long_windows: run_divergence's argument (a shard of abfit_divergence_multi passes its whole call's div_long_windows)
static int divergence_impl(abfit_ctx *ctx, bool device_inputs, const uint8_t *status, const double *posterior_max,
                           const double *meth_lvl, int32_t S, int64_t L, const int64_t *seg_offsets, int32_t W,
                           double thr, double *D_out, uint64_t *diff_out, uint64_t *cnt_out, double *p0uu_out,
                           double *methsum_out, int64_t *nvalid_out, float *ms_out, int32_t *launches_out,
                           int64_t pitch = 0, int long_windows = -1)
{
    if (!ctx || !status || !posterior_max || !meth_lvl || S <= 0 || L < 0 || S > 65535) return ABFIT_ERR_ARG;
    int64_t whole[2] = {0, L};
    if (!seg_offsets) {
        seg_offsets = whole;
        W = 1;
    }
    if (W <= 0) return ABFIT_ERR_ARG;
    if (seg_offsets[0] < 0 || seg_offsets[W] > L) {
        set_error("seg_offsets outside [0, L]");
        return ABFIT_ERR_ARG;
    }
    ABFIT_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t n = (size_t)S * (size_t)L;
    const size_t P = (size_t)S * (S - 1) / 2;
    DevBuf<uint8_t> d_status;  // host-input path: freed at the end of the call (whole methylomes can be many GB)
    DevBuf<double> d_post, d_meth;
    DevBuf<double> &d_D = ctx->dv_D, &d_methsum = ctx->dv_methsum, &d_p0uu = ctx->dv_p0uu;
    DevBuf<unsigned long long> &d_diff = ctx->dv_diff, &d_cnt = ctx->dv_cnt;
    DevBuf<long long> &d_nvalid = ctx->dv_nvalid;
    if (!device_inputs) {
        if (int rc = d_status.ensure(n)) return rc;
        if (int rc = d_post.ensure(n)) return rc;
        if (int rc = d_meth.ensure(n)) return rc;
    }
    if (int rc = d_D.ensure((size_t)W * P)) return rc;
    if (int rc = d_diff.ensure((size_t)W * P)) return rc;
    if (int rc = d_cnt.ensure((size_t)W * P)) return rc;
    if (int rc = d_methsum.ensure((size_t)W * S)) return rc;
    if (int rc = d_nvalid.ensure((size_t)W * S)) return rc;
    if (int rc = d_p0uu.ensure(W)) return rc;
    if (n && !device_inputs) {
        if (pitch > L) {  // a site range of wider host matrices: row by row into dense device matrices
            ABFIT_CUDA(cudaMemcpy2DAsync(d_status.p, (size_t)L, status, (size_t)pitch, (size_t)L, S, cudaMemcpyHostToDevice, st));
            ABFIT_CUDA(cudaMemcpy2DAsync(d_post.p, (size_t)L * 8, posterior_max, (size_t)pitch * 8, (size_t)L * 8, S,
                                         cudaMemcpyHostToDevice, st));
            ABFIT_CUDA(cudaMemcpy2DAsync(d_meth.p, (size_t)L * 8, meth_lvl, (size_t)pitch * 8, (size_t)L * 8, S,
                                         cudaMemcpyHostToDevice, st));
        } else {
            ABFIT_CUDA(cudaMemcpyAsync(d_status.p, status, n, cudaMemcpyHostToDevice, st));
            ABFIT_CUDA(cudaMemcpyAsync(d_post.p, posterior_max, n * 8, cudaMemcpyHostToDevice, st));
            ABFIT_CUDA(cudaMemcpyAsync(d_meth.p, meth_lvl, n * 8, cudaMemcpyHostToDevice, st));
        }
    }
    int launches = 0;
    if (int rc = run_divergence(st, device_inputs ? status : d_status.p, device_inputs ? posterior_max : d_post.p,
                                device_inputs ? meth_lvl : d_meth.p, S, L, seg_offsets, W, thr, d_D.p, d_diff.p,
                                d_cnt.p, d_methsum.p, d_nvalid.p, d_p0uu.p, &launches, ms_out, &ctx->div_arena,
                                long_windows))
        return rc;
    if (launches_out) *launches_out = launches;
    if (D_out && P) ABFIT_CUDA(cudaMemcpyAsync(D_out, d_D.p, (size_t)W * P * 8, cudaMemcpyDeviceToHost, st));
    if (diff_out && P) ABFIT_CUDA(cudaMemcpyAsync(diff_out, d_diff.p, (size_t)W * P * 8, cudaMemcpyDeviceToHost, st));
    if (cnt_out && P) ABFIT_CUDA(cudaMemcpyAsync(cnt_out, d_cnt.p, (size_t)W * P * 8, cudaMemcpyDeviceToHost, st));
    if (p0uu_out) ABFIT_CUDA(cudaMemcpyAsync(p0uu_out, d_p0uu.p, (size_t)W * 8, cudaMemcpyDeviceToHost, st));
    if (methsum_out) ABFIT_CUDA(cudaMemcpyAsync(methsum_out, d_methsum.p, (size_t)W * S * 8, cudaMemcpyDeviceToHost, st));
    if (nvalid_out) ABFIT_CUDA(cudaMemcpyAsync(nvalid_out, d_nvalid.p, (size_t)W * S * 8, cudaMemcpyDeviceToHost, st));
    ABFIT_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int abfit_divergence(abfit_ctx *ctx, const uint8_t *status, const double *posterior_max, const double *meth_lvl,
                     int32_t S, int64_t L, const int64_t *seg_offsets, int32_t W, double thr, double *D_out,
                     uint64_t *diff_out, uint64_t *cnt_out, double *p0uu_out, double *methsum_out,
                     int64_t *nvalid_out)
{
    return divergence_impl(ctx, false, status, posterior_max, meth_lvl, S, L, seg_offsets, W, thr, D_out, diff_out,
                           cnt_out, p0uu_out, methsum_out, nvalid_out, nullptr, nullptr);
}

int abfit_divergence_multi(abfit_ctx *const *ctxs, int32_t n_ctx, const uint8_t *status, const double *posterior_max,
                           const double *meth_lvl, int32_t S, int64_t L, const int64_t *seg_offsets, int32_t W, double thr,
                           double *D_out, uint64_t *diff_out, uint64_t *cnt_out, double *p0uu_out, double *methsum_out,
                           int64_t *nvalid_out)
{
    if (!ctxs || n_ctx <= 0 || !status || !posterior_max || !meth_lvl || S <= 0 || L < 0) return ABFIT_ERR_ARG;
    for (int r = 0; r < n_ctx; ++r)
        if (!ctxs[r]) return ABFIT_ERR_ARG;
    const size_t P = (size_t)S * (S - 1) / 2;
    if (seg_offsets) {
        // windows are independent: every device takes a contiguous block of windows (and the site range they cover).
        // Results are per window, and every shard sums meth_lvl in the tree one device would choose for the whole
        // window list (div_long_windows), so this is the single-device result bit for bit.  One window stays on one
        // device: only seg_offsets == NULL shards the site axis.
        if (W <= 0) return ABFIT_ERR_ARG;
        if (seg_offsets[0] < 0 || seg_offsets[W] > L) {
            set_error("seg_offsets outside [0, L]");
            return ABFIT_ERR_ARG;
        }
        const int long_windows = div_long_windows(seg_offsets, W) ? 1 : 0;
        const int world = std::min<int>(n_ctx, W);
        std::vector<int> rcs(world, 0);
        std::vector<std::string> errs(world);
        auto work = [&](int r) {
            int64_t w0, wc;
            shard_range(W, r, world, w0, wc);
            const int64_t a = seg_offsets[w0], b = seg_offsets[w0 + wc];
            std::vector<int64_t> seg((size_t)wc + 1);
            for (int64_t k = 0; k <= wc; ++k) seg[k] = seg_offsets[w0 + k] - a;
            rcs[r] = divergence_impl(ctxs[r], false, status + a, posterior_max + a, meth_lvl + a, S, b - a, seg.data(), (int32_t)wc,
                                     thr, D_out ? D_out + (size_t)w0 * P : nullptr, diff_out ? diff_out + (size_t)w0 * P : nullptr,
                                     cnt_out ? cnt_out + (size_t)w0 * P : nullptr, p0uu_out ? p0uu_out + w0 : nullptr,
                                     methsum_out ? methsum_out + (size_t)w0 * S : nullptr,
                                     nvalid_out ? nvalid_out + (size_t)w0 * S : nullptr, nullptr, nullptr, L, long_windows);
            if (rcs[r]) errs[r] = g_last_error;
        };
        std::vector<std::thread> th;
        for (int r = 1; r < world; ++r) th.emplace_back(work, r);
        work(0);
        for (auto &t : th) t.join();
        for (int r = 0; r < world; ++r)
            if (rcs[r]) {
                set_error("device shard " + std::to_string(r) + ": " + errs[r]);
                return rcs[r];
            }
        return 0;
    }
    // no seg_offsets: one window = all sites (whole methylomes, BASELINE configs[4]): the SITE axis is sharded in
    // 64-site words; the integer partial sums add up exactly, so D = diff / (2 cnt) (src/pedigree.rs:257) does not
    // depend on the number of devices; the per-sample methylation sums are added in device order (p0uu within 1e-12 of
    // one device)
    const int64_t words = (L + 63) / 64;
    const int world = (int)std::max<int64_t>(1, std::min<int64_t>(n_ctx, words));
    std::vector<std::vector<uint64_t>> pd(world, std::vector<uint64_t>(P)), pc(world, std::vector<uint64_t>(P));
    std::vector<std::vector<double>> pm(world, std::vector<double>(S));
    std::vector<std::vector<int64_t>> pn(world, std::vector<int64_t>(S));
    std::vector<int> rcs(world, 0);
    std::vector<std::string> errs(world);
    auto work = [&](int r) {
        int64_t w0, wc;
        shard_range(words, r, world, w0, wc);
        const int64_t a = std::min(w0 * 64, L), b = std::min((w0 + wc) * 64, L);
        rcs[r] = divergence_impl(ctxs[r], false, status + a, posterior_max + a, meth_lvl + a, S, b - a, nullptr, 1, thr, nullptr,
                                 pd[r].data(), pc[r].data(), nullptr, pm[r].data(), pn[r].data(), nullptr, nullptr, L);
        if (rcs[r]) errs[r] = g_last_error;
    };
    std::vector<std::thread> th;
    for (int r = 1; r < world; ++r) th.emplace_back(work, r);
    work(0);
    for (auto &t : th) t.join();
    for (int r = 0; r < world; ++r)
        if (rcs[r]) {
            set_error("device shard " + std::to_string(r) + ": " + errs[r]);
            return rcs[r];
        }
    for (size_t p = 0; p < P; ++p) {
        uint64_t d = 0, c = 0;
        for (int r = 0; r < world; ++r) {
            d += pd[r][p];
            c += pc[r][p];
        }
        if (diff_out) diff_out[p] = d;
        if (cnt_out) cnt_out[p] = c;
        if (D_out) D_out[p] = (double)d / (2.0 * (double)c);  // src/pedigree.rs:257 (0/0 -> NaN)
    }
    double acc = 0.0;
    for (int s = 0; s < S; ++s) {
        double m = 0.0;
        int64_t nv = 0;
        for (int r = 0; r < world; ++r) {
            m += pm[r][s];
            nv += pn[r][s];
        }
        if (methsum_out) methsum_out[s] = m;
        if (nvalid_out) nvalid_out[s] = nv;
        acc += 1.0 - m / (double)nv;  // src/pedigree.rs:179-183
    }
    if (p0uu_out) *p0uu_out = acc / (double)S;
    return 0;
}

int abfit_divergence_device(abfit_ctx *ctx, const uint8_t *d_status, const double *d_posterior_max,
                            const double *d_meth_lvl, int32_t S, int64_t L, const int64_t *seg_offsets, int32_t W,
                            double thr, double *D_out, uint64_t *diff_out, uint64_t *cnt_out, double *p0uu_out,
                            double *methsum_out, int64_t *nvalid_out, float kernel_ms[2], int32_t *launches_out)
{
    return divergence_impl(ctx, true, d_status, d_posterior_max, d_meth_lvl, S, L, seg_offsets, W, thr, D_out, diff_out,
                           cnt_out, p0uu_out, methsum_out, nvalid_out, kernel_ms, launches_out);
}

// ---------------------------------------------------------------------------------------
// per-region divergence (abfit_regions.cu): every region = the single window {lo, hi} of abfit_divergence
// ---------------------------------------------------------------------------------------
static int region_divergence_impl(abfit_ctx *ctx, bool device_inputs, const uint8_t *status, const double *posterior_max,
                                  const double *meth_lvl, int32_t S, int64_t L, const int64_t *lo, const int64_t *hi, int32_t W,
                                  double thr, double *D_out, uint64_t *diff_out, uint64_t *cnt_out, double *p0uu_out,
                                  double *methsum_out, int64_t *nvalid_out, float *ms_out, int32_t *launches_out)
{
    // every refusal that needs no device comes first
    if (!ctx || !status || !posterior_max || !meth_lvl || S <= 0 || S > 65535 || L < 0 || !lo || !hi || W <= 0) {
        set_error("region divergence: missing or out-of-range argument");
        return ABFIT_ERR_ARG;
    }
    for (int32_t w = 0; w < W; ++w)
        if (lo[w] < 0 || lo[w] > hi[w] || hi[w] > L) {
            set_error("region divergence: region " + std::to_string(w) + " [" + std::to_string(lo[w]) + ", " +
                      std::to_string(hi[w]) + ") is not a site range of [0, " + std::to_string(L) + ")");
            return ABFIT_ERR_ARG;
        }
    RegionPlan plan;
    if (int rc = plan_regions(S, L, lo, hi, W, plan)) return rc;
    const size_t P = (size_t)S * (S - 1) / 2, n = (size_t)S * (size_t)L;
    ABFIT_CUDA(cudaSetDevice(ctx->device));
    {
        const size_t need = (size_t)W * P * 24 + (size_t)W * S * 16 + (size_t)W * 8 + plan.bytes + (device_inputs ? 0 : n * 17);
        size_t fr = 0, tot = 0;
        ABFIT_CUDA(cudaMemGetInfo(&fr, &tot));
        if (need > fr) {
            set_error("region divergence: " + std::to_string(W) + " regions x " + std::to_string(P) + " pairs need about " +
                      std::to_string(need >> 20) + " MiB of device memory, " + std::to_string(fr >> 20) + " MiB are free");
            return ABFIT_ERR_TOO_LARGE;
        }
    }
    cudaStream_t st = ctx->stream;
    DevBuf<uint8_t> d_status;
    DevBuf<double> d_post, d_meth, d_D, d_methsum, d_p0uu;
    DevBuf<unsigned long long> d_diff, d_cnt;
    DevBuf<long long> d_nvalid;
    if (!device_inputs) {
        if (int rc = d_status.ensure(n)) return rc;
        if (int rc = d_post.ensure(n)) return rc;
        if (int rc = d_meth.ensure(n)) return rc;
        if (n) {
            ABFIT_CUDA(cudaMemcpyAsync(d_status.p, status, n, cudaMemcpyHostToDevice, st));
            ABFIT_CUDA(cudaMemcpyAsync(d_post.p, posterior_max, n * 8, cudaMemcpyHostToDevice, st));
            ABFIT_CUDA(cudaMemcpyAsync(d_meth.p, meth_lvl, n * 8, cudaMemcpyHostToDevice, st));
        }
        status = d_status.p;
        posterior_max = d_post.p;
        meth_lvl = d_meth.p;
    }
    if (int rc = d_D.ensure((size_t)W * P)) return rc;
    if (int rc = d_diff.ensure((size_t)W * P)) return rc;
    if (int rc = d_cnt.ensure((size_t)W * P)) return rc;
    if (int rc = d_methsum.ensure((size_t)W * S)) return rc;
    if (int rc = d_nvalid.ensure((size_t)W * S)) return rc;
    if (int rc = d_p0uu.ensure(W)) return rc;
    struct Events {  // destroyed on every way out
        cudaEvent_t e[2] = {nullptr, nullptr};
        ~Events()
        {
            for (auto &x : e)
                if (x) cudaEventDestroy(x);
        }
    } ev;
    if (ms_out) {
        ABFIT_CUDA(cudaEventCreate(&ev.e[0]));
        ABFIT_CUDA(cudaEventCreate(&ev.e[1]));
        ABFIT_CUDA(cudaEventRecord(ev.e[0], st));
    }
    int launches = 0;
    if (int rc = run_region_divergence(st, &ctx->div_arena, plan, status, posterior_max, meth_lvl, S, L, lo, hi, W, thr, d_D.p,
                                       d_diff.p, d_cnt.p, d_methsum.p, d_nvalid.p, d_p0uu.p, &launches))
        return rc;
    if (ms_out) {
        ABFIT_CUDA(cudaEventRecord(ev.e[1], st));
        ABFIT_CUDA(cudaEventSynchronize(ev.e[1]));
        ABFIT_CUDA(cudaEventElapsedTime(ms_out, ev.e[0], ev.e[1]));
    }
    if (launches_out) *launches_out = launches;
    if (D_out && P) ABFIT_CUDA(cudaMemcpyAsync(D_out, d_D.p, (size_t)W * P * 8, cudaMemcpyDeviceToHost, st));
    if (diff_out && P) ABFIT_CUDA(cudaMemcpyAsync(diff_out, d_diff.p, (size_t)W * P * 8, cudaMemcpyDeviceToHost, st));
    if (cnt_out && P) ABFIT_CUDA(cudaMemcpyAsync(cnt_out, d_cnt.p, (size_t)W * P * 8, cudaMemcpyDeviceToHost, st));
    if (p0uu_out) ABFIT_CUDA(cudaMemcpyAsync(p0uu_out, d_p0uu.p, (size_t)W * 8, cudaMemcpyDeviceToHost, st));
    if (methsum_out) ABFIT_CUDA(cudaMemcpyAsync(methsum_out, d_methsum.p, (size_t)W * S * 8, cudaMemcpyDeviceToHost, st));
    if (nvalid_out) ABFIT_CUDA(cudaMemcpyAsync(nvalid_out, d_nvalid.p, (size_t)W * S * 8, cudaMemcpyDeviceToHost, st));
    ABFIT_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int abfit_region_divergence(abfit_ctx *ctx, const uint8_t *status, const double *posterior_max, const double *meth_lvl,
                            int32_t S, int64_t L, const int64_t *region_lo, const int64_t *region_hi, int32_t W, double thr,
                            double *D_out, uint64_t *diff_out, uint64_t *cnt_out, double *p0uu_out, double *methsum_out,
                            int64_t *nvalid_out)
{
    return region_divergence_impl(ctx, false, status, posterior_max, meth_lvl, S, L, region_lo, region_hi, W, thr, D_out,
                                  diff_out, cnt_out, p0uu_out, methsum_out, nvalid_out, nullptr, nullptr);
}

int abfit_region_divergence_device(abfit_ctx *ctx, const uint8_t *d_status, const double *d_posterior_max,
                                   const double *d_meth_lvl, int32_t S, int64_t L, const int64_t *region_lo,
                                   const int64_t *region_hi, int32_t W, double thr, double *D_out, uint64_t *diff_out,
                                   uint64_t *cnt_out, double *p0uu_out, double *methsum_out, int64_t *nvalid_out,
                                   float *kernel_ms, int32_t *launches_out)
{
    return region_divergence_impl(ctx, true, d_status, d_posterior_max, d_meth_lvl, S, L, region_lo, region_hi, W, thr, D_out,
                                  diff_out, cnt_out, p0uu_out, methsum_out, nvalid_out, kernel_ms, launches_out);
}

// ---------------------------------------------------------------------------------------
// site-block bootstrap: per-block partial sums (the observed-divergence path over a list of block windows) -> D* of
// every replicate (k_siteboot_dstar) -> the bootstrap refit kernels on the given D* (DGIVEN instantiations)
// ---------------------------------------------------------------------------------------
void abfit_gen_site_boot_counts(uint64_t seed, uint64_t problem_key, int32_t n_boot, int32_t n_blocks, uint32_t *counts_out)
{
    if (!counts_out || n_boot <= 0 || n_blocks <= 0) return;
    std::fill(counts_out, counts_out + (size_t)n_boot * n_blocks, 0u);
    for (int32_t b = 0; b < n_boot; ++b)
        for (int32_t d = 0; d < n_blocks; ++d)
            ++counts_out[(size_t)b * n_blocks + site_boot_block(seed, problem_key, (uint64_t)b, (uint64_t)d, n_blocks)];
}

// The refit of given D* replicates, shared by the site-block and the parametric bootstrap: d_dstar [pair_off * n_boot +
// b * n_pairs + i] and d_nan [n_probs][n_boot] (1: a pair of the replicate has no valid site) are on the device, filled
// on the context stream.  Replicates start from [best, vary x 4], vary drawn on the device from the window keys (d_ids,
// else first_problem_id + p), and run on the mapping abfit_boot_batch's planner picks for b's pedigrees.
static int refit_given_dstar(abfit_ctx *ctx, abfit_batch *b, int32_t n_probs, const abfit_fit *best, int32_t n_boot,
                             uint64_t seed, uint64_t first_problem_id, const unsigned long long *d_ids, const double *d_dstar,
                             const uint8_t *d_nan, int64_t total_pairs, int32_t max_iters, double sd_tol, uint32_t flags,
                             double *rows_out, abfit_fit *fits_out, double *analysis_out, double *dstar_out,
                             int32_t *nan_reps_out)
{
    cudaStream_t st = ctx->stream;
    // the mapping abfit_boot_batch's planner picks for these pedigrees: warp-per-fit, else the stored-D* tile
    const int n_sm = ctx->prop.multiProcessorCount;
    std::vector<WorkItem> items = b->shape.wide ? make_items_wide(b->hp, n_boot, n_sm, false)
                                                : make_items(b->hp, n_boot, n_sm, 1, false);
    DevBuf<WorkItem> d_items;
    DevBuf<double> d_rows, d_tile, d_an, d_an_scratch;
    DevBuf<abfit_fit> d_fits;
    if (int rc = d_items.ensure(items.size())) return rc;
    if (int rc = d_rows.ensure((size_t)n_probs * n_boot * 7)) return rc;
    if (int rc = d_fits.ensure((size_t)n_probs * n_boot)) return rc;
    if (int rc = b->d_best.ensure(n_probs)) return rc;
    if (int rc = b->d_vary.ensure((size_t)n_probs * n_boot * 16)) return rc;
    if (!b->shape.wide)
        if (int rc = d_tile.ensure((items.size() + 1) * (size_t)b->hp.max_pairs * 32)) return rc;
    const bool dev_stats = analysis_out && n_boot >= 2;
    if (dev_stats) {
        if (int rc = d_an.ensure((size_t)n_probs * 32)) return rc;
        if (int rc = d_an_scratch.ensure((size_t)n_probs * 8 * n_boot)) return rc;
    }
    BigScratch big;
    if (!b->shape.wide)
        if (int rc = big_scratch(b, std::max<size_t>(items.size(), 1), big)) return rc;
    if (!items.empty())
        ABFIT_CUDA(cudaMemcpyAsync(d_items.p, items.data(), items.size() * sizeof(WorkItem), cudaMemcpyHostToDevice, st));
    ABFIT_CUDA(cudaMemcpyAsync(b->d_best.p, best, (size_t)n_probs * sizeof(abfit_fit), cudaMemcpyHostToDevice, st));
    ABFIT_CUDA(cudaMemsetAsync(d_rows.p, 0xFF, (size_t)n_probs * n_boot * 7 * 8, st));
    ABFIT_CUDA(cudaMemsetAsync(d_fits.p, 0xFF, (size_t)n_probs * n_boot * sizeof(abfit_fit), st));
    ABFIT_CUDA(cudaMemsetAsync(b->d_evals_boot.p, 0, (size_t)n_probs * 8, st));
    if (int rc = launch_gen_vary(st, seed, first_problem_id, d_ids, n_probs, n_boot, b->d_best.p, b->d_vary.p)) return rc;
    const NMParams nm = nm_params(max_iters, sd_tol, flags);
    if (b->shape.wide) {
        if (int rc = launch_fit_boot_wide_given(st, b->pools, d_items.p, (int)items.size(), n_boot, b->d_best.p, d_dstar,
                                                b->d_vary.p, nm, d_rows.p, d_fits.p, b->d_evals_boot.p, b->shape.smem_wide))
            return rc;
    } else if (int rc = launch_fit_boot_given(st, b->pools, d_items.p, (int)items.size(), n_boot, b->d_best.p, d_dstar,
                                              b->d_vary.p, d_tile.p, (int64_t)b->hp.max_pairs * 32, nm, d_rows.p, d_fits.p,
                                              b->d_evals_boot.p, b->shape.smem_boot, big)) {
        return rc;
    }
    if (dev_stats) {
        if (int rc = launch_analyze(st, d_rows.p, n_probs, n_boot, d_an.p, d_an_scratch.p)) return rc;
        ABFIT_CUDA(cudaMemcpyAsync(analysis_out, d_an.p, (size_t)n_probs * 32 * 8, cudaMemcpyDeviceToHost, st));
    }
    std::vector<uint8_t> nan_rep((size_t)n_probs * n_boot);
    ABFIT_CUDA(cudaMemcpyAsync(rows_out, d_rows.p, (size_t)n_probs * n_boot * 7 * 8, cudaMemcpyDeviceToHost, st));
    if (fits_out)
        ABFIT_CUDA(cudaMemcpyAsync(fits_out, d_fits.p, (size_t)n_probs * n_boot * sizeof(abfit_fit), cudaMemcpyDeviceToHost, st));
    if (dstar_out)
        ABFIT_CUDA(cudaMemcpyAsync(dstar_out, d_dstar, (size_t)total_pairs * n_boot * 8, cudaMemcpyDeviceToHost, st));
    ABFIT_CUDA(cudaMemcpyAsync(nan_rep.data(), d_nan, nan_rep.size(), cudaMemcpyDeviceToHost, st));
    ABFIT_CUDA(cudaStreamSynchronize(st));
    if (nan_reps_out)
        for (int p = 0; p < n_probs; ++p) {
            int32_t n = 0;
            for (int k = 0; k < n_boot; ++k) n += nan_rep[(size_t)p * n_boot + k];
            nan_reps_out[p] = n;
        }
    if (analysis_out && !dev_stats)
        for (int p = 0; p < n_probs; ++p) abfit_analyze(rows_out + (size_t)p * n_boot * 7, n_boot, analysis_out + (size_t)p * 32);
    return 0;
}

static int site_boot_impl(abfit_ctx *ctx, bool device_inputs, const abfit_problem *probs, int32_t n_probs,
                          const int32_t *pairs, const uint8_t *status, const double *posterior_max, const double *meth_lvl,
                          int32_t S, int64_t L, const int64_t *seg, double thr, int64_t block_sites, const abfit_fit *best,
                          int32_t n_boot, uint64_t seed, uint64_t first_problem_id, const uint64_t *problem_ids,
                          int32_t max_iters, double sd_tol, uint32_t flags, double *rows_out, abfit_fit *fits_out,
                          double *analysis_out, double *dstar_out, int32_t *nan_reps_out)
{
    // every refusal that needs no device comes first
    if (block_sites < 1 || block_sites >= ((int64_t)1 << 31)) {
        set_error("site bootstrap: block_sites must lie in [1, 2^31)");
        return ABFIT_ERR_ARG;
    }
    if (!probs || n_probs <= 0 || !pairs || !seg || !best || !rows_out || n_boot <= 0 || max_iters < 0 || !status ||
        !posterior_max || !meth_lvl || S < 2 || S > 65535 || L < 0) {
        set_error("site bootstrap: missing or out-of-range argument");
        return ABFIT_ERR_ARG;
    }
    if (seg[0] < 0 || seg[n_probs] > L) {
        set_error("site bootstrap: seg_offsets outside [0, L]");
        return ABFIT_ERR_ARG;
    }
    std::vector<long long> blk_off((size_t)n_probs + 1, 0);
    std::vector<int64_t> bseg;
    for (int p = 0; p < n_probs; ++p) {
        const int64_t len = seg[p + 1] - seg[p];
        if (len <= 0) {
            set_error("site bootstrap: window " + std::to_string(p) + " has no sites");
            return ABFIT_ERR_ARG;
        }
        const int64_t nb = (len + block_sites - 1) / block_sites;
        if (nb > INT32_MAX) {
            set_error("site bootstrap: window " + std::to_string(p) + " has 2^31 blocks or more");
            return ABFIT_ERR_ARG;
        }
        for (int64_t k = 0; k < nb; ++k) bseg.push_back(seg[p] + k * block_sites);
        blk_off[p + 1] = blk_off[p] + nb;
    }
    bseg.push_back(seg[n_probs]);
    const int64_t n_blk = blk_off[n_probs];
    if (n_blk > INT32_MAX) {
        set_error("site bootstrap: 2^31 blocks or more in one call");
        return ABFIT_ERR_ARG;
    }
    const int64_t P = (int64_t)S * (S - 1) / 2;
    int64_t total_pairs = 0;
    int32_t max_rows = 0;
    for (int p = 0; p < n_probs; ++p) {
        if (probs[p].n_pairs <= 0) {
            set_error("site bootstrap: problem " + std::to_string(p) + " has no pedigree rows");
            return ABFIT_ERR_ARG;
        }
        total_pairs += probs[p].n_pairs;
        max_rows = std::max(max_rows, probs[p].n_pairs);
    }
    std::vector<int32_t> row_pair((size_t)total_pairs);
    for (int64_t r = 0; r < total_pairs; ++r) {
        int64_t i = pairs[2 * r], j = pairs[2 * r + 1];
        if (i < 0 || j < 0 || i >= S || j >= S || i == j) {
            set_error("site bootstrap: pedigree row " + std::to_string(r) + " names no pair of the S samples");
            return ABFIT_ERR_ARG;
        }
        if (i > j) std::swap(i, j);
        row_pair[(size_t)r] = (int32_t)(i * S - i * (i + 1) / 2 + (j - i - 1));  // pair order (0,1),(0,2)...
    }
    if (!ctx) {
        set_error("site bootstrap: no context");
        return ABFIT_ERR_ARG;
    }
    ABFIT_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    // the pedigrees are compiled (and refused) before the partial sums are computed
    abfit_batch *b = nullptr;
    if (int rc = workspace(ctx, probs, n_probs, &b)) return rc;

    // device memory: the partials stay resident; the divergence's u64 outputs are produced a chunk of blocks at a time
    const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(n_blk, ((int64_t)256 << 20) / (P * 24)));
    const size_t n_in = device_inputs ? 0 : (size_t)S * (size_t)L * 17;
    const size_t need = (size_t)n_blk * P * 8 + (size_t)chunk * (P * 24 + S * 16) + (size_t)n_blk * n_boot * 4 +
                        (size_t)total_pairs * n_boot * 8 + n_in + (size_t)S * (size_t)L * 3 / 8 + ((size_t)64 << 20);
    {
        size_t fr = 0, tot = 0;
        ABFIT_CUDA(cudaMemGetInfo(&fr, &tot));
        if (need > fr) {
            set_error("site bootstrap: " + std::to_string(n_blk) + " blocks x " + std::to_string(P) +
                      " pairs need about " + std::to_string(need >> 20) + " MiB of device memory, " +
                      std::to_string(fr >> 20) + " MiB are free");
            return ABFIT_ERR_TOO_LARGE;
        }
    }
    DevBuf<uint2> d_part;
    if (int rc = d_part.ensure((size_t)n_blk * P)) return rc;
    {
        DevBuf<uint8_t> in_status;
        DevBuf<double> in_post, in_meth;
        if (!device_inputs && L > 0) {
            const size_t n = (size_t)S * (size_t)L;
            if (int rc = in_status.ensure(n)) return rc;
            if (int rc = in_post.ensure(n)) return rc;
            if (int rc = in_meth.ensure(n)) return rc;
            ABFIT_CUDA(cudaMemcpyAsync(in_status.p, status, n, cudaMemcpyHostToDevice, st));
            ABFIT_CUDA(cudaMemcpyAsync(in_post.p, posterior_max, n * 8, cudaMemcpyHostToDevice, st));
            ABFIT_CUDA(cudaMemcpyAsync(in_meth.p, meth_lvl, n * 8, cudaMemcpyHostToDevice, st));
            status = in_status.p;
            posterior_max = in_post.p;
            meth_lvl = in_meth.p;
        }
        DevBuf<double> t_D, t_ms;
        DevBuf<unsigned long long> t_diff, t_cnt;
        DevBuf<long long> t_nv;
        if (int rc = t_D.ensure((size_t)chunk * P)) return rc;
        if (int rc = t_diff.ensure((size_t)chunk * P)) return rc;
        if (int rc = t_cnt.ensure((size_t)chunk * P)) return rc;
        if (int rc = t_ms.ensure((size_t)chunk * S)) return rc;
        if (int rc = t_nv.ensure((size_t)chunk * S)) return rc;
        // the fused / two-pass choice is made once for the whole block list, as one abfit_divergence call would
        const int long_windows = div_long_windows(bseg.data(), (int)n_blk) ? 1 : 0;
        for (int64_t c0 = 0; c0 < n_blk; c0 += chunk) {
            const int W = (int)std::min<int64_t>(chunk, n_blk - c0);
            int launches = 0;
            if (int rc = run_divergence(st, status, posterior_max, meth_lvl, S, L, bseg.data() + c0, W, thr, t_D.p, t_diff.p,
                                        t_cnt.p, t_ms.p, t_nv.p, nullptr, &launches, nullptr, &ctx->div_arena, long_windows))
                return rc;
            if (int rc = launch_siteboot_pack(st, t_diff.p, t_cnt.p, (int64_t)W * P, d_part.p + (size_t)c0 * P)) return rc;
        }
        ABFIT_CUDA(cudaStreamSynchronize(st));  // the temporaries are freed at the end of this scope
    }

    std::vector<SiteBootItem> ditems;
    {
        int64_t off = 0;
        for (int p = 0; p < n_probs; ++p) {
            const int np = probs[p].n_pairs;
            for (int r0 = 0; r0 < np; r0 += SB_THREADS) {
                SiteBootItem it{};
                it.prob = p;
                it.r0 = r0;
                it.n_rows = std::min(SB_THREADS, np - r0);
                it.n_pairs = np;
                it.pair_off = off;
                it.blk0 = blk_off[p];
                it.n_blk = (int32_t)(blk_off[p + 1] - blk_off[p]);
                ditems.push_back(it);
            }
            off += np;
        }
    }
    DevBuf<SiteBootItem> d_ditems;
    DevBuf<long long> d_blk_off;
    DevBuf<int32_t> d_row_pair;
    DevBuf<uint32_t> d_counts;
    DevBuf<double> d_dstar;
    DevBuf<uint8_t> d_nan;
    if (int rc = d_ditems.ensure(ditems.size())) return rc;
    if (int rc = d_blk_off.ensure(blk_off.size())) return rc;
    if (int rc = d_row_pair.ensure(row_pair.size())) return rc;
    if (int rc = d_counts.ensure((size_t)n_blk * n_boot)) return rc;
    if (int rc = d_dstar.ensure((size_t)total_pairs * n_boot)) return rc;
    if (int rc = d_nan.ensure((size_t)n_probs * n_boot)) return rc;
    const unsigned long long *d_ids = nullptr;
    if (problem_ids) {
        if (int rc = b->d_ids.ensure(n_probs)) return rc;
        ABFIT_CUDA(cudaMemcpyAsync(b->d_ids.p, problem_ids, (size_t)n_probs * 8, cudaMemcpyHostToDevice, st));
        d_ids = b->d_ids.p;
    }
    ABFIT_CUDA(cudaMemcpyAsync(d_ditems.p, ditems.data(), ditems.size() * sizeof(SiteBootItem), cudaMemcpyHostToDevice, st));
    ABFIT_CUDA(cudaMemcpyAsync(d_blk_off.p, blk_off.data(), blk_off.size() * 8, cudaMemcpyHostToDevice, st));
    ABFIT_CUDA(cudaMemcpyAsync(d_row_pair.p, row_pair.data(), row_pair.size() * 4, cudaMemcpyHostToDevice, st));
    ABFIT_CUDA(cudaMemsetAsync(d_counts.p, 0, (size_t)n_blk * n_boot * 4, st));
    ABFIT_CUDA(cudaMemsetAsync(d_nan.p, 0, (size_t)n_probs * n_boot, st));
    if (int rc = launch_siteboot_counts(st, seed, first_problem_id, d_ids, d_blk_off.p, n_probs, n_boot, n_blk, d_counts.p)) return rc;
    if (int rc = launch_siteboot_dstar(st, d_ditems.p, (int)ditems.size(), n_boot, d_part.p, P, d_counts.p, d_row_pair.p,
                                       d_dstar.p, d_nan.p))
        return rc;
    return refit_given_dstar(ctx, b, n_probs, best, n_boot, seed, first_problem_id, d_ids, d_dstar.p, d_nan.p, total_pairs,
                             max_iters, sd_tol, flags, rows_out, fits_out, analysis_out, dstar_out, nan_reps_out);
}

int abfit_site_boot_batch(abfit_ctx *ctx, const abfit_problem *probs, int32_t n_probs, const int32_t *pairs,
                          const uint8_t *status, const double *posterior_max, const double *meth_lvl, int32_t S, int64_t L,
                          const int64_t *seg_offsets, double thr, int64_t block_sites, const abfit_fit *best,
                          int32_t n_boot, uint64_t seed, uint64_t first_problem_id, const uint64_t *problem_ids,
                          int32_t max_iters, double sd_tol, uint32_t flags, double *rows_out, abfit_fit *fits_out,
                          double *analysis_out, double *dstar_out, int32_t *nan_reps_out)
{
    return site_boot_impl(ctx, false, probs, n_probs, pairs, status, posterior_max, meth_lvl, S, L, seg_offsets, thr,
                          block_sites, best, n_boot, seed, first_problem_id, problem_ids, max_iters, sd_tol, flags, rows_out,
                          fits_out, analysis_out, dstar_out, nan_reps_out);
}

int abfit_site_boot_batch_device(abfit_ctx *ctx, const abfit_problem *probs, int32_t n_probs, const int32_t *pairs,
                                 const uint8_t *d_status, const double *d_posterior_max, const double *d_meth_lvl, int32_t S,
                                 int64_t L, const int64_t *seg_offsets, double thr, int64_t block_sites,
                                 const abfit_fit *best, int32_t n_boot, uint64_t seed, uint64_t first_problem_id,
                                 const uint64_t *problem_ids, int32_t max_iters, double sd_tol, uint32_t flags,
                                 double *rows_out, abfit_fit *fits_out, double *analysis_out, double *dstar_out,
                                 int32_t *nan_reps_out)
{
    return site_boot_impl(ctx, true, probs, n_probs, pairs, d_status, d_posterior_max, d_meth_lvl, S, L, seg_offsets, thr,
                          block_sites, best, n_boot, seed, first_problem_id, problem_ids, max_iters, sd_tol, flags, rows_out,
                          fits_out, analysis_out, dstar_out, nan_reps_out);
}

// ---------------------------------------------------------------------------------------
// parametric bootstrap: replicates simulated from every window's fitted model and counted to exact per-row sums in one
// kernel (k_psim_counts) -> D* = D_sim + theta3 (k_psim_dstar) -> the site bootstrap's refit of the given D*
// ---------------------------------------------------------------------------------------
void abfit_gen_param_boot_seeds(uint64_t seed, uint64_t problem_key, int32_t n_boot, uint64_t *seeds_out)
{
    if (!seeds_out) return;
    for (int32_t b = 0; b < n_boot; ++b) seeds_out[b] = param_boot_seed(seed, problem_key, (uint64_t)b);
}

int abfit_param_boot_batch(abfit_ctx *ctx, const abfit_sim_tree *tree, const abfit_problem *probs, int32_t n_probs,
                           const int64_t *n_sites, const double *missing, double thr, const abfit_fit *best, int32_t n_boot,
                           uint64_t seed, uint64_t first_problem_id, const uint64_t *problem_ids, int32_t max_iters,
                           double sd_tol, uint32_t flags, double *rows_out, abfit_fit *fits_out, double *analysis_out,
                           double *dstar_out, double *lse_star_out, double *gof_p_out, int32_t *window_status_out,
                           int32_t *nan_reps_out)
{
    auto refuse = [](int rc, const std::string &m) {
        set_error("parametric bootstrap: " + m);
        return rc;
    };
    // every refusal that needs no device comes first
    if (!tree || !probs || n_probs <= 0 || !n_sites || !best || !rows_out || n_boot <= 0 || max_iters < 0)
        return refuse(ABFIT_ERR_ARG, "missing or out-of-range argument");
    if (n_boot > 65535) return refuse(ABFIT_ERR_TOO_LARGE, "at most 65535 replicates per call");
    int32_t n_nodes = 0, S = 0, R = 0;
    abfit_sim_tree_info(tree, &n_nodes, &S, &R);
    if (R <= 0) return refuse(ABFIT_ERR_ARG, "the forest has no pair of sampled nodes in one tree");
    if (S > PSIM_MAX_S)
        return refuse(ABFIT_ERR_TOO_LARGE, std::to_string(S) + " sampled nodes, at most " + std::to_string(PSIM_MAX_S));
    std::vector<double> tp((size_t)R * 5);
    abfit_sim_tree_pairs(tree, tp.data(), R);
    for (int p = 0; p < n_probs; ++p) {
        if (probs[p].n_pairs != R || !probs[p].pedigree)
            return refuse(ABFIT_ERR_ARG, "problem " + std::to_string(p) + " has " + std::to_string(probs[p].n_pairs) +
                                             " pedigree rows, the forest " + std::to_string(R));
        for (int r = 0; r < R; ++r)
            for (int c = 0; c < 3; ++c)
                if (!(probs[p].pedigree[(size_t)r * 4 + c] == tp[(size_t)r * 5 + 2 + c]))
                    return refuse(ABFIT_ERR_ARG, "problem " + std::to_string(p) + ", pedigree row " + std::to_string(r) +
                                                     ": (t0, t1, t2) differ from the forest's pair rows");
        if (n_sites[p] <= 0) return refuse(ABFIT_ERR_ARG, "window " + std::to_string(p) + " has no sites");
        if (n_sites[p] >= ((int64_t)1 << 31))
            return refuse(ABFIT_ERR_TOO_LARGE, "window " + std::to_string(p) + " has 2^31 sites or more");
        if (missing)
            for (int s = 0; s < S; ++s) {
                const double m = missing[(size_t)p * S + s];
                if (!(m >= 0.0 && m <= 1.0))
                    return refuse(ABFIT_ERR_ARG, "window " + std::to_string(p) + ", sample " + std::to_string(s) +
                                                     ": missing rate outside [0, 1]");
            }
    }
    if (!ctx) return refuse(ABFIT_ERR_ARG, "no context");
    const uint64_t smem = psim_smem_bytes(n_nodes, S, R);
    if (smem > (uint64_t)ctx->smem_optin)
        return refuse(ABFIT_ERR_TOO_LARGE, std::to_string(n_nodes) + " nodes, " + std::to_string(S) + " samples and " +
                                               std::to_string(R) + " rows need " + std::to_string(smem) +
                                               " B of shared memory per block, " + std::to_string(ctx->smem_optin) +
                                               " B are available");
    // windows whose fitted model cannot be simulated get status 1 and no launch
    auto in01 = [](double x) { return x >= 0.0 && x <= 1.0; };
    std::vector<int32_t> valid;
    std::vector<int32_t> wstat(n_probs, 0);
    for (int p = 0; p < n_probs; ++p) {
        const double *th = best[p].theta;
        const bool ok = in01(th[0]) && in01(th[1]) && in01(th[2]) && in01(probs[p].p0uu) && std::isfinite(th[3]);
        wstat[p] = ok ? 0 : 1;
        if (ok) valid.push_back(p);
    }
    const int nv = (int)valid.size();
    // host tables: walk, per-window thresholds and missing rates, tile items
    std::vector<int32_t> parent_pos, node_id, row_pos, row_ij(R);
    sim_walk(tree, parent_pos, node_id, row_pos);
    for (int r = 0; r < R; ++r) row_ij[r] = (int32_t)tp[(size_t)r * 5] | ((int32_t)tp[(size_t)r * 5 + 1] << 16);
    std::vector<double> thr6((size_t)nv * n_nodes * 6), miss((size_t)nv * S, 0.0), theta3(nv);
    std::vector<unsigned long long> keys(nv);
    std::vector<abfit_problem> vprobs(nv);
    std::vector<abfit_fit> vbest(nv);
    std::vector<PsimItem> items;
    for (int q = 0; q < nv; ++q) {
        const int p = valid[q];
        const abfit_sim_params prm{best[p].theta[0], best[p].theta[1], best[p].theta[2], probs[p].p0uu, 0.0, 0};
        if (int rc = sim_thresholds_walk(tree, &prm, thr6.data() + (size_t)q * n_nodes * 6)) return rc;
        if (missing) std::copy(missing + (size_t)p * S, missing + (size_t)(p + 1) * S, miss.begin() + (size_t)q * S);
        theta3[q] = best[p].theta[3];
        keys[q] = problem_ids ? problem_ids[p] : first_problem_id + (uint64_t)p;
        vprobs[q] = probs[p];
        vbest[q] = best[p];
        const int64_t tiles = (n_sites[p] + PSIM_TILE - 1) / PSIM_TILE;
        for (int64_t t0 = 0; t0 < tiles; t0 += PSIM_MAX_TILES)
            items.push_back(PsimItem{q, (int32_t)std::min<int64_t>(PSIM_MAX_TILES, tiles - t0), t0, n_sites[p]});
    }
    if (items.size() > (size_t)INT32_MAX) return refuse(ABFIT_ERR_TOO_LARGE, "2^31 tiles or more in one call");
    const int64_t total_rows = (int64_t)nv * R;
    // results of the windows that run: straight into the caller's arrays when every window runs, else compacted
    const bool all = nv == n_probs;
    std::vector<double> c_rows, c_an, c_dstar;
    std::vector<abfit_fit> c_fits;
    std::vector<int32_t> c_nan(nv);
    if (!all) {
        c_rows.resize((size_t)nv * n_boot * 7);
        if (analysis_out) c_an.resize((size_t)nv * 32);
        if (dstar_out) c_dstar.resize((size_t)total_rows * n_boot);
    }
    if (!fits_out || !all) c_fits.resize((size_t)nv * n_boot);
    abfit_fit *fits = all && fits_out ? fits_out : c_fits.data();
    if (nv > 0) {
        ABFIT_CUDA(cudaSetDevice(ctx->device));
        cudaStream_t st = ctx->stream;
        abfit_batch *b = nullptr;
        if (int rc = workspace(ctx, vprobs.data(), nv, &b)) return rc;
        const size_t need = (size_t)total_rows * n_boot * 8 + (size_t)nv * n_boot * (7 * 8 + sizeof(abfit_fit) + 16 * 8 + 8 * 8 + 1) +
                            thr6.size() * 8 + miss.size() * 8 + items.size() * sizeof(PsimItem) +
                            (size_t)b->hp.max_pairs * 32 * 8 * (size_t)(4 * ctx->prop.multiProcessorCount + 1) + ((size_t)64 << 20);
        size_t fr = 0, tot = 0;
        ABFIT_CUDA(cudaMemGetInfo(&fr, &tot));
        if (need > fr)
            return refuse(ABFIT_ERR_TOO_LARGE, std::to_string(nv) + " windows x " + std::to_string(n_boot) + " replicates x " +
                                                   std::to_string(R) + " rows need about " + std::to_string(need >> 20) +
                                                   " MiB of device memory, " + std::to_string(fr >> 20) + " MiB are free");
        DevBuf<PsimItem> d_items;
        DevBuf<double> d_thr6, d_miss, d_theta3;
        DevBuf<int32_t> d_parent, d_node, d_rowpos, d_rowij;
        DevBuf<unsigned long long> d_keys, d_sums;
        DevBuf<uint8_t> d_nan;
        if (int rc = d_items.ensure(items.size())) return rc;
        if (int rc = d_thr6.ensure(thr6.size())) return rc;
        if (int rc = d_miss.ensure(miss.size())) return rc;
        if (int rc = d_theta3.ensure(nv)) return rc;
        if (int rc = d_parent.ensure(n_nodes)) return rc;
        if (int rc = d_node.ensure(n_nodes)) return rc;
        if (int rc = d_rowpos.ensure(S)) return rc;
        if (int rc = d_rowij.ensure(R)) return rc;
        if (int rc = d_keys.ensure(nv)) return rc;
        if (int rc = d_sums.ensure((size_t)total_rows * n_boot)) return rc;
        if (int rc = d_nan.ensure((size_t)nv * n_boot)) return rc;
        ABFIT_CUDA(cudaMemcpyAsync(d_items.p, items.data(), items.size() * sizeof(PsimItem), cudaMemcpyHostToDevice, st));
        ABFIT_CUDA(cudaMemcpyAsync(d_thr6.p, thr6.data(), thr6.size() * 8, cudaMemcpyHostToDevice, st));
        ABFIT_CUDA(cudaMemcpyAsync(d_miss.p, miss.data(), miss.size() * 8, cudaMemcpyHostToDevice, st));
        ABFIT_CUDA(cudaMemcpyAsync(d_theta3.p, theta3.data(), (size_t)nv * 8, cudaMemcpyHostToDevice, st));
        ABFIT_CUDA(cudaMemcpyAsync(d_parent.p, parent_pos.data(), (size_t)n_nodes * 4, cudaMemcpyHostToDevice, st));
        ABFIT_CUDA(cudaMemcpyAsync(d_node.p, node_id.data(), (size_t)n_nodes * 4, cudaMemcpyHostToDevice, st));
        ABFIT_CUDA(cudaMemcpyAsync(d_rowpos.p, row_pos.data(), (size_t)S * 4, cudaMemcpyHostToDevice, st));
        ABFIT_CUDA(cudaMemcpyAsync(d_rowij.p, row_ij.data(), (size_t)R * 4, cudaMemcpyHostToDevice, st));
        ABFIT_CUDA(cudaMemcpyAsync(d_keys.p, keys.data(), (size_t)nv * 8, cudaMemcpyHostToDevice, st));
        ABFIT_CUDA(cudaMemsetAsync(d_sums.p, 0, (size_t)total_rows * n_boot * 8, st));
        ABFIT_CUDA(cudaMemsetAsync(d_nan.p, 0, (size_t)nv * n_boot, st));
        if (int rc = launch_psim_counts(st, d_items.p, (int)items.size(), d_thr6.p, d_parent.p, d_node.p, n_nodes, d_rowpos.p,
                                        d_miss.p, S, d_rowij.p, R, thr, seed, d_keys.p, n_boot, d_sums.p))
            return rc;
        if (int rc = launch_psim_dstar(st, d_sums.p, total_rows * n_boot, R, n_boot, d_theta3.p, d_nan.p)) return rc;
        if (int rc = refit_given_dstar(ctx, b, nv, vbest.data(), n_boot, seed, 0, d_keys.p,
                                       reinterpret_cast<const double *>(d_sums.p), d_nan.p, total_rows, max_iters, sd_tol, flags,
                                       all ? rows_out : c_rows.data(), fits, all ? analysis_out : (analysis_out ? c_an.data() : nullptr),
                                       all ? dstar_out : (dstar_out ? c_dstar.data() : nullptr), c_nan.data()))
            return rc;
    }
    // scatter the windows that ran; the others get NaN
    const double qnan = std::nan("");
    for (int p = 0, q = 0; p < n_probs; ++p) {
        const bool ran = wstat[p] == 0;
        if (!all) {
            double *ro = rows_out + (size_t)p * n_boot * 7;
            if (ran) std::copy(c_rows.begin() + (size_t)q * n_boot * 7, c_rows.begin() + (size_t)(q + 1) * n_boot * 7, ro);
            else std::fill(ro, ro + (size_t)n_boot * 7, qnan);
            if (analysis_out) {
                double *ao = analysis_out + (size_t)p * 32;
                if (ran) std::copy(c_an.begin() + (size_t)q * 32, c_an.begin() + (size_t)(q + 1) * 32, ao);
                else std::fill(ao, ao + 32, qnan);
            }
            if (dstar_out) {
                double *d = dstar_out + (size_t)p * R * n_boot;
                if (ran) std::copy(c_dstar.begin() + (size_t)q * R * n_boot, c_dstar.begin() + (size_t)(q + 1) * R * n_boot, d);
                else std::fill(d, d + (size_t)R * n_boot, qnan);
            }
            if (fits_out)
                for (int k = 0; k < n_boot; ++k) {
                    abfit_fit &f = fits_out[(size_t)p * n_boot + k];
                    if (ran) {
                        f = c_fits[(size_t)q * n_boot + k];
                        continue;
                    }
                    f.theta[0] = f.theta[1] = f.theta[2] = f.theta[3] = f.cost = f.lse = qnan;
                    f.iters = f.evals = 0;
                    f.status = ABFIT_FIT_NAN;
                    f.start_id = k;
                }
        }
        int32_t fitted = 0, ge = 0;
        for (int k = 0; k < n_boot; ++k) {
            const double l = ran ? fits[(size_t)q * n_boot + k].lse : qnan;
            if (lse_star_out) lse_star_out[(size_t)p * n_boot + k] = l;
            if (ran && fits[(size_t)q * n_boot + k].status != ABFIT_FIT_NAN) {
                ++fitted;
                ge += l >= best[p].lse ? 1 : 0;
            }
        }
        if (gof_p_out) gof_p_out[p] = ran ? (1.0 + (double)ge) / (1.0 + (double)fitted) : qnan;
        if (nan_reps_out) nan_reps_out[p] = ran ? c_nan[q] : 0;
        if (window_status_out) window_status_out[p] = wstat[p];
        if (ran) ++q;
    }
    return 0;
}

int abfit_simulate(abfit_ctx *ctx, const abfit_sim_tree *tree, const abfit_sim_params *params, int64_t first_site, int64_t L,
                   uint8_t *status, double *posterior_max, double *meth_lvl)
{
    if (!ctx) return ABFIT_ERR_ARG;
    ABFIT_CUDA(cudaSetDevice(ctx->device));
    return run_simulate(ctx->stream, ctx->prop.multiProcessorCount, tree, params, first_site, L, status, posterior_max, meth_lvl,
                        false, nullptr);
}

int abfit_simulate_device(abfit_ctx *ctx, const abfit_sim_tree *tree, const abfit_sim_params *params, int64_t first_site,
                          int64_t L, uint8_t *d_status, double *d_posterior_max, double *d_meth_lvl, float *kernel_ms)
{
    if (!ctx) return ABFIT_ERR_ARG;
    ABFIT_CUDA(cudaSetDevice(ctx->device));
    return run_simulate(ctx->stream, ctx->prop.multiProcessorCount, tree, params, first_site, L, d_status, d_posterior_max,
                        d_meth_lvl, true, kernel_ms);
}

// ---------------------------------------------------------------------------------------
// bootstrap statistics (src/analysis.rs:50-98) — O(n_boot) host post-processing
// ---------------------------------------------------------------------------------------
int abfit_analyze(const double *rows, int32_t n, double out[32])
{
    if (!rows || n <= 0 || !out) return ABFIT_ERR_ARG;
    std::vector<double> col(n);
    const int src[8] = {0, 1, -1, 2, 3, 4, 5, 6};
    for (int f = 0; f < 8; ++f) {
        double sum = 0.0;
        if (src[f] < 0) {
            // beta/alpha is an owned contiguous array in the reference: ndarray sums it with its
            // 8-accumulator unrolled fold; strided column views are folded sequentially
            for (int i = 0; i < n; ++i) col[i] = rows[7 * (size_t)i + 1] / rows[7 * (size_t)i];
            double p[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            int i = 0;
            for (; n - i >= 8; i += 8)
                for (int k = 0; k < 8; ++k) p[k] += col[i + k];
            sum += p[0] + p[4];
            sum += p[1] + p[5];
            sum += p[2] + p[6];
            sum += p[3] + p[7];
            for (; i < n; ++i) sum += col[i];
        } else {
            for (int i = 0; i < n; ++i) {
                col[i] = rows[7 * (size_t)i + src[f]];
                sum += col[i];
            }
        }
        out[f] = sum / (double)n;
        // std(ddof = 1): Welford with mul_add, as ndarray 0.15 `var`
        double mean = 0.0, ssq = 0.0;
        for (int i = 0; i < n; ++i) {
            const double delta = col[i] - mean;
            mean = mean + delta / (double)(i + 1);
            ssq = std::fma(col[i] - mean, delta, ssq);
        }
        out[8 + f] = std::sqrt(ssq / ((double)n - 1.0));
        // quantiles 0.025 / 0.975, ndarray-stats `Linear`
        std::sort(col.begin(), col.end());
        const double qs[2] = {0.025, 0.975};
        for (int k = 0; k < 2; ++k) {
            const double pos = (double)(n - 1) * qs[k];
            const double lo = std::floor(pos), hi = std::ceil(pos);
            const double a = col[(size_t)lo], b2 = col[(size_t)hi];
            out[16 + 2 * f + k] = a + (b2 - a) * (pos - std::trunc(pos));
        }
    }
    return 0;
}

}  // extern "C"
