#!/usr/bin/env python3
"""bench.py — ABneutral fits/sec on the C4 workload (BASELINE.json configs[3]).

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --steps K --warmup W    (CPU arm: the oracle port of the reference)
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   (also writes what the last timed step computed)

A *step* is one pass of the hot path over one batch of synthetic windows: for every window,
`n_starts` Nelder-Mead fits from random simplices (ab_neutral::run), best-of-starts, then `n_boot`
bootstrap refits (boot_model::run).  One fit = one NM run to termination.

Scaling is STRONG, as BASELINE.json configs[3] is written: `--windows` (10 000) windows in total, sharded over the
N ranks by window (`multi.window_shard`), no data-path collective.  The weak-scaling figure (10 000 windows per
GPU) is reported beside it as `weak` when N > 1.

Printed JSON (one line, rank 0):
  value      fits/s with all inputs already resident in HBM (kernels only, CUDA events on the library stream)
  e2e        fits/s through the host-buffer C-ABI call abfit_alphabeta_batch (= alphabeta::run per window): pinned
             host inputs copied H2D and results D2H inside the timed region, incl. compiling the pedigrees, the
             draw of the bootstrap vary-vertices that depends on the fit result, and the bootstrap statistics
  roofline   dominant kernel (multi-start NM) against the FP64 (DFMA) peak measured in the same run;
             achieved = executed objective evaluations x algorithmic FLOPs per evaluation / kernel time;
             pipe_frac = executed FP64 instructions / the pipe's instruction rate (the ceiling of `frac` under the
             bit-exact arithmetic contract is frac_ceiling = flops / (2 x fp64 instructions))
  cpu_baseline  oracle port of the reference ("literal work": per-pair matrix_power, no early exit, the sort_by
             whose comparator re-evaluates divergence()) on all host cores, bounded sample of the same workload
  other_configs  c2 (BASELINE configs[0..1]), c5 (configs[4]: observed divergence of 200 samples x 5 M sites
             site-sharded over the ranks + the 1000-start fit of the 19 900-pair pedigree) and
             divergence_roofline (HBM roofline of the divergence reduction: 17 S L + 24 P algorithmic bytes)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)
SEED = 0xAB0B200
DUMP_BYTES = 32_000_000  # --dump-outputs writes at most this many bytes of arrays
GOLDEN_PED = os.path.join(ROOT, "tests", "golden", "pedigree.txt")
METRIC = "ABneutral fits/sec (window x start x boot, f64)"


# ---------------------------------------------------------------------------------------------
# synthetic C4 windows (SURVEY.md §8d): the 351-row time structure of data/pedigree.txt,
# D = c + dt(alpha,beta,w) + N(0, 5e-4), clipped at 0
# ---------------------------------------------------------------------------------------------
def load_shape():
    rows = []
    for line in open(GOLDEN_PED).read().split("\n")[1:]:
        if line:
            rows.append([float(x) for x in line.split(" ")[:4]])
    return np.array(rows)


def synth_windows(W, first_window, shape):
    """returns pedigrees [W, N, 4] and p0uu [W]; generator only (numpy), not the product path.  Window w of a run is
    the same whatever the sharding: the generator is keyed per block of 64 windows."""
    N = len(shape)
    peds = np.empty((W, N, 4))
    p0 = np.empty(W)
    BLK = 64
    w = first_window
    while w < first_window + W:
        blk = w // BLK
        pb, ub = _synth_block(blk, BLK, shape)
        lo = w - blk * BLK
        n = min(BLK - lo, first_window + W - w)
        peds[w - first_window:w - first_window + n] = pb[lo:lo + n]
        p0[w - first_window:w - first_window + n] = ub[lo:lo + n]
        w += n
    return peds, p0


def _synth_block(block, W, shape):
    rng = np.random.default_rng([SEED, block])
    N = len(shape)
    a = 10 ** rng.uniform(-5, -3.3, W)
    b = 10 ** rng.uniform(-4, -2.3, W)
    w = rng.uniform(0, 0.1, W)
    c = rng.uniform(0, 0.005, W)
    p0uu = rng.uniform(0.6, 0.95, W)
    G = np.empty((W, 3, 3))
    G[:, 0, 0] = (1 - a) ** 2; G[:, 0, 1] = 2 * (1 - a) * a; G[:, 0, 2] = a ** 2
    G[:, 1, 0] = 0.25 * (b + 1 - a) ** 2; G[:, 1, 1] = 0.5 * (b + 1 - a) * (a + 1 - b); G[:, 1, 2] = 0.25 * (a + 1 - b) ** 2
    G[:, 2, 0] = b ** 2; G[:, 2, 1] = 2 * (1 - b) * b; G[:, 2, 2] = (1 - b) ** 2
    tmax = int(shape[:, :3].max())
    P = [np.broadcast_to(np.eye(3), (W, 3, 3)).copy()]
    for _ in range(tmax):
        P.append(P[-1] @ G)
    sv0 = np.stack([p0uu, w * (1 - p0uu), (1 - w) * (1 - p0uu)], axis=1)
    tri = shape[:, :3].astype(int)
    uniq, inv = np.unique(tri, axis=0, return_inverse=True)
    dt_u = np.empty((W, len(uniq)))
    for u, (t0, t1, t2) in enumerate(uniq):
        s = np.einsum("wi,wij->wj", sv0, P[t0])
        A, B = P[t1 - t0], P[t2 - t0]
        d = 0.5 * (A[:, :, 0] * B[:, :, 1] + A[:, :, 1] * B[:, :, 0] + A[:, :, 1] * B[:, :, 2] + A[:, :, 2] * B[:, :, 1]) \
            + (A[:, :, 0] * B[:, :, 2] + A[:, :, 2] * B[:, :, 0])
        dt_u[:, u] = np.einsum("wk,wk->w", s, d)
    D = np.maximum(c[:, None] + dt_u[:, inv.ravel()] + rng.normal(0, 5e-4, (W, N)), 0.0)
    peds = np.empty((W, N, 4))
    peds[:, :, :3] = shape[None, :, :3]
    peds[:, :, 3] = D
    return peds, p0uu


# ---------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i",
                 str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); smax.append(float(r[2])); power.append(float(r[3]))
            except ValueError:
                continue
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference, all host threads, bounded sample.  Inputs come from the pure-Python
# twin of the seeded generators (oracle/gen_py.py, pinned bit for bit against libabfit's in tests/test_abi.py), so
# this arm never touches the product library, and they are drawn BEFORE the clock starts.
# ---------------------------------------------------------------------------------------------
def cpu_reference_sample(shape, n_starts_sample, n_boot_sample, literal=True, threads=None, window=0, balance=True):
    """times ab_neutral::run + boot_model::run of ONE synthetic window on the host cores.
    literal=True: the reference's own work (per-pair matrix_power, pedigree clone per start, all max_iters on
    stalled starts, best-of-starts through the sort_by whose comparator re-evaluates divergence() twice)."""
    from oracle import abref_py as o
    from oracle import gen_py as g

    o.build()
    threads = threads or o.hw_threads()
    peds, p0uu = synth_windows(1, window, shape)
    ped, u = peds[0], float(p0uu[0])
    pb = o.Problem(ped, u, u, 1.0)
    sx = g.gen_start_simplices(SEED, window, n_starts_sample, float(ped[:, 3].max()))
    idx = g.gen_resample_idx(SEED, window, n_boot_sample, len(ped))
    # (the vary vertices depend on the fit result: Model::vary is drawn inside the timed region, as in the reference)
    flags = o.LITERAL_SORT if literal else (o.FAST_DIVERGENCE | o.EARLY_EXIT_ON_STALL)
    if literal and balance and n_starts_sample < 1000:
        # A stalled start runs all 10 000 iterations (~20 000 evaluations against a median of ~850).  Over the 1000 starts
        # of a real window rayon's work stealing hides those behind the rest; a bounded sample would instead wait for the
        # one that happens to be handed out last.  So the sample's starts are handed out longest first (lengths from the
        # minimal-work port, before the clock starts) — the balance the reference reaches on a whole window.
        _, _, quick, _, _ = o.ab_neutral(pb, sx, max_iters=10000, flags=o.FAST_DIVERGENCE | o.EARLY_EXIT_ON_STALL, n_threads=threads)
        length = np.where(quick["status"] == 3, 1 << 30, quick["evals"].astype(np.int64))
        sx = np.ascontiguousarray(sx[np.argsort(-length, kind="stable")])
    t0 = time.perf_counter()
    rc, best, allr, pred, resid = o.ab_neutral(pb, sx, max_iters=10000, flags=flags, n_threads=threads)
    vary = g.gen_vary_vertices(SEED, window, n_boot_sample, best["theta"])
    rc2, rows, fits = o.boot_model(pb, best["theta"], pred, resid, idx, vary, max_iters=1000, flags=flags,
                                   n_threads=threads)
    dt = time.perf_counter() - t0
    assert rc == 0 and rc2 == 0
    return (n_starts_sample + n_boot_sample) / dt, dt, threads


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    shape = load_shape()
    from oracle import abref_py as o

    o.build()
    threads = o.hw_threads()
    # bounded sample, sized from the step count: literal reference work costs ~0.85 core-seconds per fit (measured:
    # one full window, 1100 fits, 112 s on 8 cores) and a stalled start alone runs its 10 000 iterations for ~8 s on
    # one core, so a SHORT sample is slower per fit than the reference really is (one stalled start is the whole
    # step); the steps get as many starts as ~2.5 minutes of host time allow, up to the full window.
    n_steps = max(1, args.warmup + args.steps)
    ns = int(min(args.starts, max(4 * threads, threads * 150.0 / (n_steps * 0.85 * 1.1))))
    nb = max(2, ns * args.boots // args.starts)
    vals = []
    for i in range(args.warmup + args.steps):
        v, dt, _ = cpu_reference_sample(shape, ns, nb, literal=True, threads=threads, window=i)
        if i >= args.warmup:
            vals.append((v, dt))
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([dt for _, dt in vals]) * 1e3)
    full = None
    if ns >= args.starts:
        full = {"fits_per_s": value, "seconds": ms / 1e3, "sample": "every timed step is one full window"}
    elif not args.no_full_window:
        # one whole window exactly as BASELINE configs[3] sizes it (1000 starts + 100 replicates): the reference's
        # real rate (stalled starts amortised over 1000 starts; serial sort_by tail of n log n comparisons)
        v, dt, _ = cpu_reference_sample(shape, args.starts, args.boots, literal=True, threads=threads, window=10 ** 6)
        full = {"fits_per_s": v, "seconds": dt, "sample": f"1 window x ({args.starts} starts + {args.boots} replicates), once"}
    sample = (f"1 synthetic C4 window x ({ns} starts + {nb} bootstrap replicates) per step, literal reference work "
              "(per-pair matrix_power, pedigree clone per start, sort_by comparator re-evaluating divergence twice); "
              "inputs drawn before the clock starts by oracle/gen_py.py; the process maps oracle/libabref.so only; the "
              "sample's starts are handed to the threads longest first (a stalled start runs 10 000 iterations: rayon hides "
              "those behind the other 999 starts of a whole window, a short sample handed out in index order would wait "
              "for them and UNDERSTATE the reference); cpu_baseline.full_window is the rate on a whole window")
    line = {
        "impl": "reference", "metric": METRIC, "value": value,
        "unit": "fits/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, shape),
        "cpu_baseline": {"value": value, "unit": "fits/s", "cores": threads, "kind": "port", "sample": sample,
                         "full_window": full},
        "e2e": {"value": value, "unit": "fits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "C restatement of alphabeta-rs (oracle/abref.c), not the Rust binary: no cargo/rustc in this image",
    }
    print(json.dumps(line))


def workload_config(args, shape):
    return {"workload": "C4 synthetic gbM metaprofile (BASELINE.json configs[3]): windows sharded over the GPUs",
            "windows_total": args.windows, "n_starts": args.starts, "n_boot": args.boots,
            "pairs_per_window": int(len(shape)), "distinct_triples": 10, "tmax": 32, "max_iters_fit": 10000,
            "max_iters_boot": 1000, "fits_per_window": args.starts + args.boots,
            "l2": "inputs (start simplices + resample indices, GBs) are far larger than the 126 MB L2"}


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def small_case_c2(ab, ctx, n_starts=1000, n_boot=1000):
    """BASELINE.json configs[0..1] on the GPU: the repo's example pedigree (data/nodelist.txt + edgelist.txt,
    6 pairs, tests/golden/pedigree_generated.txt) fitted from 1000 starts, then 1000 bootstrap replicates —
    one abfit_alphabeta_batch call from host buffers.  Latency-bound by construction (2000 fits), so it is
    reported as wall time, not as a roofline fraction.  (Parity of exactly this configuration against the oracle:
    tests/test_gpu_parity.py::test_c1_c2_default_counts_bitwise.)"""
    ped = np.loadtxt(os.path.join(ROOT, "tests", "golden", "pedigree_generated.txt"), skiprows=1)
    p0uu = 0.6554051647850442
    prob = [ab.Problem(ped, p0uu, p0uu, 1.0)]
    sx = ab.gen_start_simplices(SEED, 0, n_starts, float(ped[:, 3].max()))[None]
    idx = ab.gen_resample_idx(SEED, 0, n_boot, len(ped)).ravel()
    ctx.alphabeta_batch(prob, sx, idx, SEED)  # warm
    t0 = time.perf_counter()
    out = ctx.alphabeta_batch(prob, sx, idx, SEED)
    dt = time.perf_counter() - t0
    b = out["best"][0]
    return {"workload": "data/nodelist.txt pedigree (6 pairs): 1000 starts + 1000 bootstrap replicates, one call",
            "wall_ms": 1e3 * dt, "fits_per_s": (n_starts + n_boot) / dt,
            "best": {"alpha": float(b["theta"][0]), "beta": float(b["theta"][1]), "lse": float(b["lse"])}}


def suffstats_experiment(ab, ctx, probs, sx, n_windows=2000, idx=None, n_boot=0, first=0):
    """EXPERIMENT, never the default and never part of `value` (VERDICT round 1, item 9): the multi-start kernel with
    the objective evaluated from per-triple sufficient statistics (ABFIT_EXPERIMENT_SUFFSTATS=1; O(distinct triples)
    per evaluation instead of O(pairs); regrouped sum, so NOT bit-identical).  Same windows, same start simplices, both
    ways; the experiment's best-of-starts is checked at north_star's tolerances against the exact path: exact RSS at
    its best theta within 1e-9 relative, alpha / beta within 1e-6."""
    Ws = min(n_windows, len(probs))
    P, S = probs[:Ws], np.ascontiguousarray(sx[:Ws])
    NS = S.shape[1]
    res, ms = {}, {}
    old = {k: os.environ.get(k) for k in ("ABFIT_EXPERIMENT_SUFFSTATS", "ABFIT_JIT")}
    try:
        os.environ["ABFIT_JIT"] = "1"
        for mode in ("0", "1"):
            os.environ["ABFIT_EXPERIMENT_SUFFSTATS"] = mode
            b = ctx.batch(P)
            b.upload_starts(S)
            b.run_fit()
            t = []
            for _ in range(3):
                b.run_fit()
                t.append(b.timing()["fit_ms"])
            res[mode], ms[mode] = b.download_fit(), float(np.median(t))
            b.close()
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    be, bs = res["0"].best, res["1"].best
    boot = None
    if idx is not None and n_boot > 0:
        # mode 2: the bootstrap refits too, from the exact best models on both sides
        try:
            N = P[0].n_pairs
            I = np.ascontiguousarray(idx[:Ws]).reshape(-1)
            vary = np.stack([ab.gen_vary_vertices(SEED, first + i, n_boot, be[i]["theta"]) for i in range(Ws)])
            rows, bms = {}, {}
            os.environ["ABFIT_JIT"] = "1"
            for mode in ("0", "2"):
                os.environ["ABFIT_EXPERIMENT_SUFFSTATS"] = mode
                b = ctx.batch(P)
                b.upload_boot(I, vary, best=be, pred=res["0"].pred, resid=res["0"].resid)
                b.run_boot()
                t = []
                for _ in range(3):
                    b.run_boot()
                    t.append(b.timing()["boot_ms"])
                rows[mode], bms[mode] = b.download_boot()[0], float(np.median(t))
                b.close()
            r2 = np.abs(rows["2"][:, :, :2] - rows["0"][:, :, :2]) / np.maximum(np.abs(rows["0"][:, :, :2]), 1e-300)
            boot = {"replicates": n_boot, "bootstrap_ms_exact": bms["0"], "bootstrap_ms_experiment": bms["2"],
                    "speedup": bms["0"] / bms["2"], "replicates_within_1e-6": float(np.mean((r2 <= 1e-6).all(axis=2))),
                    "replicates_bit_identical": float(np.mean((rows["2"][:, :, :4] == rows["0"][:, :, :4]).all(axis=2)))}
        except Exception as e:
            boot = {"error": str(e)}
        finally:
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
    _, lse_at = ctx.cost_batch(P, bs["theta"], np.arange(Ws, dtype=np.int32))
    rel = lambda a, b: np.abs(a - b) / np.maximum(np.abs(b), 1e-300)
    d_rss, d_a, d_b = rel(lse_at, be["lse"]), rel(bs["theta"][:, 0], be["theta"][:, 0]), rel(bs["theta"][:, 1], be["theta"][:, 1])
    ok = (d_rss <= 1e-9) & (d_a <= 1e-6) & (d_b <= 1e-6)
    return {"what": "multi-start objective from per-triple sufficient statistics, ABFIT_EXPERIMENT_SUFFSTATS=1: an experiment, "
                    "never the default, not in `value` (not bit-identical to the reference's sequential sum)",
            "windows": Ws, "starts": NS, "multi_start_ms_exact": ms["0"], "multi_start_ms_experiment": ms["1"],
            "multi_start_Mfits_per_s_exact": Ws * NS / ms["0"] / 1e3, "multi_start_Mfits_per_s_experiment": Ws * NS / ms["1"] / 1e3,
            "speedup": ms["0"] / ms["1"], "windows_within_tolerance": int(ok.sum()),
            "tolerance": "exact RSS at the experiment's best theta within 1e-9 relative of the exact path's, alpha and beta within 1e-6",
            "max_rel_diff": {"rss": float(d_rss.max()), "alpha": float(d_a.max()), "beta": float(d_b.max())},
            "same_winning_start": float(np.mean(be["start_id"] == bs["start_id"])),
            "bootstrap_mode_2": boot}


def c5_times(lineages=10, generations=20):
    """time structure of the C5 pedigree: `lineages` lines sampled at generations 1..`generations` from one founder"""
    samples = [(l, g) for l in range(lineages) for g in range(1, generations + 1)]
    rows = []
    for i in range(len(samples)):
        for j in range(i + 1, len(samples)):
            (l1, g1), (l2, g2) = samples[i], samples[j]
            rows.append([min(g1, g2) if l1 == l2 else 0, g1, g2, 0.0])
    return np.array(rows, dtype=np.float64)


def large_case_c5(ab, multi, ctx, torch, dist, rank, world, local, L, n_starts, hbm_gbs, hbm_src):
    """BASELINE.json configs[4]: 200 simulated methylomes x L CG sites -> observed divergence of all 19 900 pairs +
    p0uu (site axis sharded over the ranks, exact integer partial sums added up), then the ABneutral fit of that one
    pedigree from `n_starts` starts (start ids sharded over the ranks, winners compared by the reference's rule).
    Returns (c5, divergence_roofline) on rank 0."""
    dev = torch.device("cuda", local)
    lineages, generations = 10, 20
    S = lineages * generations
    P = S * (S - 1) // 2
    first, count = multi.site_shard(L, rank, world)
    g = torch.Generator(device=dev)
    g.manual_seed(1000 + rank)
    founder = (torch.rand(count, device=dev, generator=g) < 0.25).to(torch.uint8) * 2
    status = torch.empty((S, count), dtype=torch.uint8, device=dev)
    for l in range(lineages):
        cur = founder.clone()
        for t in range(generations):
            r = torch.rand(count, device=dev, generator=g)
            cur = torch.where((cur == 0) & (r < 2e-4), torch.full_like(cur, 2),
                              torch.where((cur == 2) & (r < 1e-3), torch.zeros_like(cur), cur))
            status[l * generations + t] = cur
    post = torch.empty((S, count), dtype=torch.float64, device=dev)
    meth = torch.empty((S, count), dtype=torch.float64, device=dev)
    for s in range(S):  # row by row: no (S, L) temporaries beside the 17 bytes per sample-site of the inputs
        u = torch.rand(count, device=dev, generator=g, dtype=torch.float64)
        post[s] = torch.where(torch.rand(count, device=dev, generator=g) < 0.9, torch.full_like(u, 0.9999), u * 0.49 + 0.5)
        meth[s] = (status[s].to(torch.float64) * 0.5 +
                   0.05 * torch.randn(count, device=dev, generator=g, dtype=torch.float64)).clamp_(0, 1)
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def vmax(x):
        if world == 1:
            return np.asarray(x, dtype=np.float64)
        t = torch.tensor(x, device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.cpu().numpy()

    ctx.dmatrix_device(status.data_ptr(), post.data_ptr(), meth.data_ptr(), S, count)  # warm-up
    reps = 5
    pk = pr = wall = 0.0
    for _ in range(reps):
        barrier()
        t0 = time.perf_counter()
        out = ctx.dmatrix_device(status.data_ptr(), post.data_ptr(), meth.data_ptr(), S, count)
        wall += time.perf_counter() - t0
        pk += out["kernel_ms"][0]
        pr += out["kernel_ms"][1]
    pk_ms, pr_ms, call_ms = vmax([pk / reps, pr / reps, 1e3 * wall / reps])
    # exact integer partial sums -> D is independent of the number of GPUs (src/pedigree.rs:257)
    diff = torch.from_numpy(out["diff"][0].astype(np.int64)).to(dev)
    cnt = torch.from_numpy(out["cnt"][0].astype(np.int64)).to(dev)
    nvalid = torch.from_numpy(np.asarray(out["nvalid"][0], dtype=np.int64)).to(dev)
    methsum = torch.from_numpy(np.asarray(out["methsum"][0], dtype=np.float64)).to(dev)
    if world > 1:
        dist.all_reduce(diff)
        dist.all_reduce(cnt)
        dist.all_reduce(nvalid)
        parts = [torch.empty_like(methsum) for _ in range(world)]
        dist.all_gather(parts, methsum)
        methsum = parts[0].clone()
        for p in parts[1:]:  # f64 partials added in rank order on every rank: same bits everywhere
            methsum = methsum + p
    D, p0uu, _, _ = multi.combine_site_shards([diff.cpu().numpy().astype(np.uint64)], [cnt.cpu().numpy().astype(np.uint64)],
                                              [methsum.cpu().numpy()], [nvalid.cpu().numpy()])
    del status, post, meth
    torch.cuda.empty_cache()
    ped = c5_times(lineages, generations)
    ped[:, 3] = D
    p0uu = float(p0uu)

    sx_all = ab.gen_start_simplices(SEED, 0, n_starts, float(np.nanmax(D)))
    s0, sc = multi.start_shard(n_starts, rank, world)
    bt = ctx.batch([ab.Problem(ped, p0uu, p0uu, 1.0)])
    fl = bt.flops_per_eval(0)
    bt.upload_starts(np.ascontiguousarray(sx_all[s0:s0 + sc])[None])
    bt.run_fit()  # warm-up
    barrier()
    t0 = time.perf_counter()
    bt.run_fit()
    res = bt.download_fit(want_all=True)
    fit_wall = time.perf_counter() - t0
    tm = bt.timing()
    fit_ms, fit_call_ms = vmax([tm["fit_ms"], 1e3 * fit_wall])
    rec = res.best[:1].copy()
    cands, firsts = rec, np.array([s0], dtype=np.int64)
    evals_max = int(res.all[0]["evals"].max())
    if world > 1:
        raw = torch.from_numpy(rec.view(np.uint8).copy()).to(dev)
        allraw = [torch.empty_like(raw) for _ in range(world)]
        dist.all_gather(allraw, raw)
        cands = np.concatenate([r.cpu().numpy().view(ab.FIT_DTYPE) for r in allraw])
        fs = torch.tensor([s0], device=dev, dtype=torch.int64)
        allfs = [torch.empty_like(fs) for _ in range(world)]
        dist.all_gather(allfs, fs)
        firsts = np.array([int(f.item()) for f in allfs], dtype=np.int64)
        evals_max = int(vmax([float(evals_max)])[0])
    win, best = multi.best_of_shards(cands, firsts)
    bt.close()
    c5_experiment = None
    if world == 1:
        # EXPERIMENT, never the default (DESIGN.md §2.13): the same fit with the objective from per-triple sufficient
        # statistics — O(distinct triples) per evaluation instead of the sequential sum over 19 900 pairs that bounds
        # the exact fit; checked at north_star's tolerances against the exact result above
        old_env = os.environ.get("ABFIT_EXPERIMENT_SUFFSTATS")
        try:
            os.environ["ABFIT_EXPERIMENT_SUFFSTATS"] = "1"
            be = ctx.batch([ab.Problem(ped, p0uu, p0uu, 1.0)])
            be.upload_starts(np.ascontiguousarray(sx_all)[None])
            be.run_fit()
            be.run_fit()
            ems = be.timing()["fit_ms"]
            eres = be.download_fit()
            be.close()
            _, lse_at = ctx.cost_batch([ab.Problem(ped, p0uu, p0uu, 1.0)], eres.best["theta"], np.zeros(1, dtype=np.int32))
            rel = lambda a, b: abs(a - b) / max(abs(b), 1e-300)
            c5_experiment = {
                "what": "ABFIT_EXPERIMENT_SUFFSTATS=1 (not bit-identical, never the default): objective from per-triple statistics",
                "fit_kernel_ms": float(ems), "speedup": float(fit_ms / ems) if ems > 0 else None,
                "rss_rel_diff": float(rel(lse_at[0], best["lse"])), "alpha_rel_diff": float(rel(eres.best["theta"][0, 0], best["theta"][0])),
                "beta_rel_diff": float(rel(eres.best["theta"][0, 1], best["theta"][1])),
                "within_tolerance": bool(rel(lse_at[0], best["lse"]) <= 1e-9 and rel(eres.best["theta"][0, 0], best["theta"][0]) <= 1e-6
                                         and rel(eres.best["theta"][0, 1], best["theta"][1]) <= 1e-6)}
        except Exception as e:
            c5_experiment = {"error": str(e)}
        finally:
            if old_env is None:
                os.environ.pop("ABFIT_EXPERIMENT_SUFFSTATS", None)
            else:
                os.environ["ABFIT_EXPERIMENT_SUFFSTATS"] = old_env
    if rank != 0:
        return None, None
    alg_bytes = 17.0 * S * L + 24.0 * P
    peak = hbm_gbs * world
    c5 = {"workload": f"C5 (BASELINE configs[4]): {S} samples x {L} CG sites ({P} pairs) site-sharded over {world} GPU(s), "
                      f"then one ABneutral fit of the {P}-pair pedigree from {n_starts} starts (start ids sharded)",
          "divergence_call_ms": float(call_ms), "pack_kernel_ms": float(pk_ms), "pair_kernel_ms": float(pr_ms),
          "fit_kernel_ms": float(fit_ms), "fit_call_ms": float(fit_call_ms), "fit_flops_per_eval": fl["flops"],
          "fit_longest_start_evals": evals_max,
          "fit_note": "warp-per-fit kernels; the fit lasts as long as its longest start (sequential pair sum, one dependent "
                      "DADD per pair), so sharding the starts does not shorten it: effectively a 1-GPU fit at any N",
          "p0uu": p0uu, "best": {"alpha": float(best["theta"][0]), "beta": float(best["theta"][1]),
                                 "lse": float(best["lse"]), "start_id": int(best["start_id"]), "rank": int(win)},
          "experiment_suffstats": c5_experiment}
    kern_ms = float(pk_ms + pr_ms)
    fused = out["launches"] <= 4  # k_fused + the three finalisation kernels (the two-pass path has >= 5 launches)
    droof = {"bound": "hbm", "kernels": "k_fused (bulk-copy packer warps + all-pairs popcount warps in one persistent "
             "kernel) + finalisation" if fused else "k_pack + k_pairs (+ finalisation)", "fused": bool(fused),
             "algorithmic_bytes": alg_bytes,
             "bytes_formula": "17 S L + 24 P (SURVEY.md §8d): posteriorMax f64 + rc.meth.lvl f64 + status u8 read once, "
                              "D / diff / cnt written once", "S": S, "L": L, "P": P, "n_gpus": world,
             "pack_kernel_ms": float(pk_ms), "pair_kernel_ms": float(pr_ms),
             "achieved": alg_bytes / (kern_ms * 1e-3) / 1e9 if kern_ms > 0 else None, "peak": peak, "unit": "GB/s",
             "frac": alg_bytes / (kern_ms * 1e-3) / 1e9 / peak if kern_ms > 0 else None,
             "pack_frac": 17.0 * S * L / (pk_ms * 1e-3) / 1e9 / peak if pk_ms > 0 else None,
             "peak_source": hbm_src + (f" x {world} GPUs" if world > 1 else ""),
             "note": ("per-rank kernel times (CUDA events inside the library), max over ranks; pack_kernel_ms = k_fused (streams the "
                      "17 B per sample-site once; the bit-planes stay in shared memory), pair_kernel_ms = finalisation" if fused else
                      "per-rank kernel times (CUDA events inside the library), max over ranks; k_pack is HBM-bound, "
                      "k_pairs is bound by the POPC pipe (3 x popc64 per pair and 64 sites)")}
    return c5, droof


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (burst copy bandwidth, driver-written)"
        except Exception:
            pass
    return 6650.0, "fallback of B200_PROFILING.md (MEASURED_PEAKS.json absent)"


def make_inputs(ab, torch, W, first, NS, NB, shape, pool):
    N = len(shape)
    peds, p0uu = synth_windows(W, first, shape)
    probs = [ab.Problem(peds[i], float(p0uu[i]), float(p0uu[i]), 1.0) for i in range(W)]
    sx_t = torch.empty((W, NS, 5, 4), dtype=torch.float64, pin_memory=True)
    idx_t = torch.empty((W, NB, N), dtype=torch.int32, pin_memory=True)
    sx, idx = sx_t.numpy(), idx_t.numpy()
    maxd = peds[:, :, 3].max(axis=1)

    def gen_w(i):
        sx[i] = ab.gen_start_simplices(SEED, first + i, NS, float(maxd[i]))
        idx[i] = ab.gen_resample_idx(SEED, first + i, NB, N)

    list(pool.map(gen_w, range(W)))
    return peds, probs, sx_t, idx_t


def dump_outputs(out_dir, fit, rows, first, n_pairs):
    """--dump-outputs: the arrays the timed path hands back (Batch.download_fit + download_boot), as float64 .npy files,
    for a fixed seeded sample of windows that stays under DUMP_BYTES (every window when they fit).  The inputs depend on
    the arguments only, so two builds of the project run with the same arguments can be compared file by file."""
    W, NB = len(fit.best), rows.shape[1]
    per_window = 8 * (len(fit.best.dtype.names) + 3 + 2 + 2 * n_pairs + 7 * NB)  # theta holds 4; + window, status
    n = min(W, max(1, DUMP_BYTES // per_window))
    win = np.sort(np.random.default_rng([SEED, W]).choice(W, n, replace=False))
    out = {"window": first + win, "status": fit.status[win], "pred": fit.pred.reshape(W, n_pairs)[win],
           "resid": fit.resid.reshape(W, n_pairs)[win], "boot_rows": rows[win]}
    for f in fit.best.dtype.names:
        out["best_" + f] = fit.best[f][win]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--windows", type=int, default=10000, help="windows in TOTAL per step (sharded over the GPUs)")
    ap.add_argument("--starts", type=int, default=1000)
    ap.add_argument("--boots", type=int, default=100)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the weak-scaling side measurement")
    ap.add_argument("--no-c5", action="store_true", help="skip other_configs.c5 / divergence_roofline")
    ap.add_argument("--no-experiments", action="store_true", help="skip the flagged experiments reported beside the contract line")
    ap.add_argument("--c5-sites", type=int, default=5_000_000)
    ap.add_argument("--no-full-window", action="store_true", help="reference arm: skip the one full 1000 + 100 window")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the fits and bootstrap rows of the last timed step to DIR/<name>.npy (one GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1):
        ap.error("--dump-outputs needs the GPU arm on one GPU")

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    from __graft_entry__ import _load_product

    ab = _load_product()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus or world == 1

    NS, NB = args.starts, args.boots
    shape = load_shape()
    N = len(shape)
    from alphabeta_rs_b200 import multi

    first, W = multi.window_shard(args.windows, rank, world)  # STRONG scaling: the windows of one job, sharded
    ctx = ab.Context(local)
    fp64_peak = ctx.measure_fp64_peak()  # TFLOP/s, DFMA = 2 FLOP
    pool = ThreadPoolExecutor(max_workers=max(4, min(32, (os.cpu_count() or 8) // max(1, world))))

    # ---- inputs: host-generated from seeds (north_star), staged in PINNED host memory ----------
    peds, probs, sx_t, idx_t = make_inputs(ab, torch, W, first, NS, NB, shape, pool)
    sx, idx = sx_t.numpy(), idx_t.numpy()
    vary = np.empty((W, NB, 4, 4))

    def gen_vary(best_theta):
        def one(i):
            vary[i] = ab.gen_vary_vertices(SEED, first + i, NB, best_theta[i])
        list(pool.map(one, range(W)))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if world == 1:
            return float(x)
        tt = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    def allsum(x):
        if world == 1:
            return float(x)
        tt = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        return float(tt.item())

    def resident_run(batch, n_warm, n_steps, sample_clocks, pipelined=True):
        """everything in HBM before the timed region; returns per-rank totals.  pipelined: fit -> select -> bootstrap
        as one pipelined pass over sub-batches of windows (abfit_batch_run_pipelined: what abfit_alphabeta_batch does);
        else the two kernels one after the other, each timed on its own (roofline of the dominant kernel)."""
        def step():
            if pipelined:
                batch.run_pipelined()
            else:
                batch.run_fit()
                batch.run_boot()

        for _ in range(n_warm):
            step()
        ctx.sync()
        sampler = ClockSampler(local) if sample_clocks else None
        barrier()
        if sampler:
            sampler.start()
        ctx.timer_start()
        acc = {"fit_ms": 0.0, "select_ms": 0.0, "boot_ms": 0.0, "evals_fit": 0, "evals_boot": 0, "launches": 0}
        for _ in range(n_steps):
            step()
            # per-kernel CUDA events recorded by the library on its own stream (timing() waits for this step's events)
            t = batch.timing()
            for k in acc:
                acc[k] += t[k]
        acc["total_ms"] = ctx.timer_stop()
        barrier()
        acc["clocks"] = sampler.stop() if sampler else None
        return acc

    fits_per_step = args.windows * (NS + NB)
    batch = ctx.batch(probs)
    fl = batch.flops_per_eval(0)
    batch.upload_starts(sx)
    batch.run_fit()
    res = batch.download_fit()
    gen_vary(res.best["theta"])
    batch.upload_boot(idx, vary)
    batch.run_boot()
    batch.sync()
    r = resident_run(batch, max(0, args.warmup - 1), args.steps, True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, batch.download_fit(), batch.download_boot()[0], first, N)
    clocks = r["clocks"]
    t_max = allmax(r["total_ms"])
    value = fits_per_step * args.steps / (t_max * 1e-3)
    launches = r["launches"]
    n_pipes = batch.pipes()
    # the dominant kernel on its own: the same batch, multi-start and bootstrap launched one after the other (in the
    # pipelined pass above the sub-batches' kernels overlap, so a launch has no duration of its own there)
    rsteps = max(1, min(args.steps, 5))
    rr = resident_run(batch, 1, rsteps, False, pipelined=False)
    fit_ms, boot_ms = rr["fit_ms"], rr["boot_ms"]
    evals_fit, evals_boot = rr["evals_fit"], rr["evals_boot"]
    seq_ms = allmax(rr["total_ms"]) / rsteps

    # ---- end-to-end: host buffers through the one-shot C-ABI calls ------------------------------
    best_t = torch.zeros((W, 64), dtype=torch.uint8, pin_memory=True)
    best_h = best_t.numpy().view(ab.FIT_DTYPE).reshape(W)
    pred_t = torch.empty(W * N, dtype=torch.float64, pin_memory=True)
    resid_t = torch.empty(W * N, dtype=torch.float64, pin_memory=True)
    rows_t = torch.empty((W, NB, 7), dtype=torch.float64, pin_memory=True)
    status_h = np.zeros(W, dtype=np.int32)
    analysis_h = np.empty((W, 32))
    packed = ab._pack_problems(probs)

    def e2e_step():
        # abfit_alphabeta_batch = alphabeta::run for every window: fit, draw of the vary vertices from the
        # best-of-starts, bootstrap, statistics; host buffers in, host buffers out
        ctx.alphabeta_batch(probs, sx, idx, SEED, first_problem_id=first, best=best_h, pred=pred_t.numpy(),
                            resid=resid_t.numpy(), status=status_h, rows=rows_t.numpy(), analysis=analysis_h, packed=packed)

    h2d = allsum(sx.nbytes + idx.nbytes + peds.nbytes)
    d2h = allsum(best_h.nbytes + 2 * pred_t.numpy().nbytes + rows_t.numpy().nbytes + status_h.nbytes)
    e2e_step()  # warm
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    ctx.sync()
    e2e_s = allmax(time.perf_counter() - t0)
    e2e_value = fits_per_step * args.steps / e2e_s

    # ---- roofline of the dominant kernel (this rank's launches; every rank runs the same shape) ------------------
    achieved = evals_fit * fl["flops"] / (fit_ms * 1e-3) / 1e12  # TFLOP/s, algorithmic
    instr_rate = fp64_peak * 1e12 / 2.0                            # FP64 lane-instructions per second at the DFMA peak
    # DRAM bytes of one multi-start launch at the default 1-GPU configuration, from an ncu capture of this command
    # (profiles/: start simplices in, fit records out; the kernel never re-reads HBM).  Other shapes were not captured.
    # profiles/r02v_dram_fit_kernels_w10000.csv: abfit_jit_fit_starts_v2, first captured launch (algorithmic: 160 B of
    # start simplex in + 64 B of fit record out per fit = 2.24 GB)
    traffic = 1753669888 + 705587200 if (W, NS, NB) == (10000, 1000, 100) else None
    roofline = {"bound": "fp64", "kernel": "k_fit_starts (multi-start Nelder-Mead)", "achieved": achieved, "peak": fp64_peak,
                "unit": "TFLOP/s", "frac": achieved / fp64_peak,
                "pipe_frac": evals_fit * fl["fp64_instr"] / (fit_ms * 1e-3) / instr_rate,
                "frac_ceiling": fl["flops"] / (2.0 * fl["fp64_instr"]),
                "pipe_note": "pipe_frac = FP64 instructions executed (evaluations x program-derived count per evaluation) / "
                             "(0.5 warp-instructions per clock and SM sub-partition = the DFMA peak's instruction rate); "
                             "only the 3x3 products may be FMAs (bit-exact contract), so frac <= frac_ceiling x pipe_frac",
                "fp64_instr_per_eval": fl["fp64_instr"],
                "traffic": traffic, "traffic_unit": "bytes per launch (dram read + write, ncu)",
                "bound_note": "FP64 vector pipe (BASELINE.json: % FP64 peak); no tensor cores, HBM traffic is 2.5 GB per 1.66 s launch",
                "peak_source": "DFMA micro-benchmark in this run (MEASURED_PEAKS.json has no FP64 figure; nominal 37.2)",
                "flops_per_eval": fl["flops"], "evals_per_launch": evals_fit / rsteps,
                "kernel_ms": fit_ms / rsteps, "kernel_share_of_step": fit_ms / rr["total_ms"],
                "boot_kernel_ms": boot_ms / rsteps,
                "measured_over": f"{rsteps} un-pipelined steps right after the timed region (one multi-start launch + one "
                                 f"bootstrap launch per step, {seq_ms:.1f} ms per step); the timed region runs the same "
                                 f"kernels as {n_pipes} overlapping sub-batches",
                "specialised_kernels": bool(batch.uses_specialised_kernels()),
                "boot_achieved": evals_boot * fl["flops"] / (boot_ms * 1e-3) / 1e12 if boot_ms > 0 else None,
                "windows_this_rank": W}
    batch.close()

    # ---- weak-scaling figure beside the headline (N > 1): 10 000 windows per GPU ---------------------------------
    weak = None
    if world > 1 and not args.no_weak:
        del sx_t, idx_t, sx, idx
        Ww = args.windows
        wfirst = args.windows + rank * Ww
        wpeds, wprobs, wsx_t, widx_t = make_inputs(ab, torch, Ww, wfirst, NS, NB, shape, pool)
        wb = ctx.batch(wprobs)
        wb.upload_starts(wsx_t.numpy())
        wb.run_fit()
        wres = wb.download_fit()
        wvary = np.stack(list(pool.map(lambda i: ab.gen_vary_vertices(SEED, wfirst + i, NB, wres.best["theta"][i]), range(Ww))))
        wb.upload_boot(widx_t.numpy(), wvary)
        wb.run_boot()
        wb.sync()
        wsteps = max(1, min(3, args.steps))
        wr = resident_run(wb, 1, wsteps, False)
        wt = allmax(wr["total_ms"])
        weak = {"value": world * Ww * (NS + NB) * wsteps / (wt * 1e-3), "unit": "fits/s", "windows_per_gpu": Ww,
                "steps": wsteps, "ms_per_step": wt / wsteps, "note": "inputs resident, same kernels; every rank fits its own 10 000 windows"}
        wb.close()
        del wsx_t, widx_t

    # ---- CPU baseline beside it (rank 0, N=1 only) ---------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import abref_py as o

        threads = o.hw_threads()
        ns = max(8, 8 * threads)
        nb = max(2, ns // 10)
        v, dt, _ = cpu_reference_sample(shape, ns, nb, literal=True, threads=threads)
        v2, dt2, _ = cpu_reference_sample(shape, 16 * ns, 16 * nb, literal=False, threads=threads)
        cpu = {"value": v, "unit": "fits/s", "cores": threads, "kind": "port",
               "sample": f"1 C4 window x ({ns} starts + {nb} boots), literal reference work incl. the re-evaluating sort_by, {dt:.1f} s "
                         "(starts handed to the threads longest first; a sample this short is still bounded by one stalled start, "
                         "10 000 iterations: the whole-window rate is `bench.py --impl reference`'s cpu_baseline.full_window)",
               "minimal_work_value": v2,
               "minimal_work_note": "same port with the power table + stall early-exit the GPU path uses "
                                    f"({16 * ns} starts + {16 * nb} boots, {dt2:.1f} s): separates algorithmic "
                                    "from hardware speed-up"}

    # ---- other BASELINE configs, reported beside the headline (outside every timed region) -------------
    aux = {}
    if rank == 0:
        try:
            aux["c2"] = small_case_c2(ab, ctx)
        except Exception as e:  # never let a side measurement break the contract line
            aux["c2"] = {"error": str(e)}
    if not args.no_c5:
        hbm, hbm_src = hbm_peak()
        try:
            c5, droof = large_case_c5(ab, multi, ctx, torch, dist, rank, world, local, args.c5_sites, 1000, hbm, hbm_src)
            if rank == 0:
                aux["c5"], aux["divergence_roofline"] = c5, droof
        except Exception as e:
            if world > 1:
                raise  # a rank that drops out of the collectives would hang the others
            aux["c5"] = {"error": str(e)}

    experiments = {}
    if rank == 0 and world == 1 and not args.no_experiments:
        try:
            experiments["suffstats"] = suffstats_experiment(ab, ctx, probs, sx, idx=idx, n_boot=NB, first=first)
        except Exception as e:
            experiments["suffstats"] = {"error": str(e)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "fits/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_max / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, shape),
            "e2e": {"value": e2e_value, "unit": "fits/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
            "evals_per_fit": {"starts": evals_fit / (rsteps * W * NS), "boots": evals_boot / (rsteps * W * NB)},
            "pipelined_sub_batches": n_pipes,
            "weak": weak, "other_configs": aux, "experiments": experiments,
        }
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
