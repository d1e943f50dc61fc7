"""Calibration and timing of the site-block bootstrap (DESIGN.md §9).

    python3 tools/siteboot_calibration.py --out profiles/r04_siteboot_calibration.json [--replicates 32] [--skip-timing]

Calibration: R design_study replicates of a design simulated with known alpha and beta (iid sites) give the true
sampling spread of the fitted rates (their across-replicate sd).  Against it, for the residual bootstrap and for the
site-block bootstrap at each block size: the median over replicates of the bootstrap sd, and the share of replicates
whose 95 % bootstrap interval covers the true rate.  Designs: the R-original pedigree (13 samples, 78 pairs, 500 000
sites) and eight lines sampled at generations 1-5 (40 samples, 780 pairs, 200 000 sites).

Timing: the three phases of one abfit_site_boot_batch_device call — per-block partial sums (the observed-divergence
kernels and k_siteboot_pack), D* (k_siteboot_counts, k_siteboot_dstar) and the refit (k_fit_boot / k_fit_wide) — as
device kernel time from torch.profiler, at the C5 shape (200 samples x 5 M sites, one window, 100 replicates, 5000-site
blocks) and the metaprofile shape (10 000 windows x 1000 sites, 27 samples, 100 replicates, 50-site blocks), beside the
card's name and power limit.  The best model handed to the bootstrap is the simulated truth (the timing is of the
bootstrap, not of the multi-start fit)."""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALPHA, BETA = 3e-3, 6e-3


def load_product():
    name = "alphabeta_rs_b200"
    if name in sys.modules:
        return sys.modules[name]
    pkg = os.path.join(ROOT, "alphabeta-rs_b200")
    spec = importlib.util.spec_from_file_location(name, os.path.join(pkg, "__init__.py"), submodule_search_locations=[pkg])
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def summarise(res):
    th, an = res["theta"], res["analysis"]
    ok = res["status"] == 0
    out = {"n_ok": int(ok.sum())}
    for f, (name, truth) in enumerate((("alpha", ALPHA), ("beta", BETA))):
        out[name] = {"across_replicate_sd": float(np.std(th[ok, f], ddof=1)),
                     "median_bootstrap_sd": float(np.nanmedian(an[ok, 8 + f])),
                     "ci95_coverage": float(np.mean((an[ok, 16 + 2 * f] <= truth) & (truth <= an[ok, 17 + 2 * f])))}
        out[name]["ratio"] = out[name]["median_bootstrap_sd"] / out[name]["across_replicate_sd"]
    return out


def calibration(ab, ctx, R):
    designs = {
        "R-original (13 samples, 78 pairs, 500 000 sites)": (
            ab.SimTree.from_files(os.path.join(ROOT, "tests", "golden", "desired_output", "nodelist.fn"),
                                  os.path.join(ROOT, "tests", "golden", "desired_output", "edgelist.fn")), 500_000, (1, 100, 10_000)),
        # block_sites = 1 here would need 200 000 x 32 blocks x 780 pairs x 8 B = 40 GB of partials
        "8 lines x generations 1-5 (40 samples, 780 pairs, 200 000 sites)": (
            ab.SimTree.lines(8, range(1, 6)), 200_000, (100, 10_000)),
    }
    out = {}
    for name, (tree, L, sizes) in designs.items():
        kw = dict(L=L, n_replicates=R, n_starts=32, n_boot=100, seed=13)
        row = {}
        t = time.time()
        row["residual"] = summarise(ab.design_study([ctx], tree, ALPHA, BETA, **kw))
        row["residual"]["wall_s"] = time.time() - t
        for bs in sizes:
            t = time.time()
            row[f"sites_{bs}"] = summarise(ab.design_study([ctx], tree, ALPHA, BETA, bootstrap="sites", block_sites=bs, **kw))
            row[f"sites_{bs}"]["wall_s"] = time.time() - t
        out[name] = row
        print(name, json.dumps(row, indent=1), flush=True)
    return out


PHASES = {"partials": ("k_pack", "k_pairs", "k_fused", "k_finalize", "k_p0uu", "k_siteboot_pack"),
          "dstar": ("k_siteboot_counts", "k_siteboot_dstar"),
          "refit": ("k_fit_boot", "k_fit_wide", "k_gen_vary", "k_analyze")}


def timed_call(ab, ctx, tree, n_windows, win_len, block_sites, n_boot, seed):
    import torch
    from torch.profiler import ProfilerActivity, profile

    S, L = tree.n_samples, n_windows * win_len
    dev = torch.device("cuda", ctx.device)
    st = torch.empty((S, L), dtype=torch.uint8, device=dev)
    po = torch.empty((S, L), dtype=torch.float64, device=dev)
    me = torch.empty((S, L), dtype=torch.float64, device=dev)
    torch.cuda.synchronize(dev)
    ctx.simulate_device(tree, st.data_ptr(), po.data_ptr(), me.data_ptr(), ALPHA, BETA, L=L, seed=seed, missing_rate=0.05)
    seg = np.arange(n_windows + 1, dtype=np.int64) * win_len
    dm = ctx.dmatrix_device(st.data_ptr(), po.data_ptr(), me.data_ptr(), S, L, seg_offsets=seg)
    probs = [ab.Problem(tree.pedigree(dm["D"][w]), float(dm["p0uu"][w]), float(dm["p0uu"][w]), 1.0) for w in range(n_windows)]
    best = np.zeros(n_windows, dtype=ab.FIT_DTYPE)
    best["theta"] = (ALPHA, BETA, 0.5, 0.0)
    pairs = np.tile(tree.pairs(), (n_windows, 1))
    args = (probs, pairs, st.data_ptr(), po.data_ptr(), me.data_ptr(), S, L, seg, best, n_boot, seed, block_sites)
    ctx.site_bootstrap_device(*args)  # warm-up: module loads, allocations
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        t = time.time()
        res = ctx.site_bootstrap_device(*args)
        wall = time.time() - t
    ms = {k: 0.0 for k in PHASES}
    other = 0.0
    for e in prof.key_averages():
        d = getattr(e, "device_time_total", None)
        d = e.cuda_time_total if d is None else d
        ph = next((k for k, names in PHASES.items() if any(n in e.key for n in names)), None)
        if ph:
            ms[ph] += d / 1000.0
        elif "emcpy" not in e.key and "emset" not in e.key:
            other += d / 1000.0
    return {"samples": S, "pairs": tree.n_pairs, "windows": n_windows, "sites_per_window": win_len, "block_sites": block_sites,
            "n_boot": n_boot, "kernel_ms": ms, "other_kernel_ms": other, "wall_ms": wall * 1000.0,
            "nan_replicates": int(res["nan_reps"].sum())}


def timing(ab, ctx):
    out = {}
    out["C5: 200 x 5 M sites, 1 window, 100 replicates, 5000-site blocks"] = timed_call(
        ab, ctx, ab.SimTree.lines(20, range(1, 11)), 1, 5_000_000, 5000, 100, 21)
    print(json.dumps(out, indent=1), flush=True)
    out["metaprofile: 10 000 windows x 1000 sites, 27 samples, 100 replicates, 50-site blocks"] = timed_call(
        ab, ctx, ab.SimTree.lines(3, range(1, 10)), 10_000, 1000, 50, 100, 22)
    print(json.dumps(out, indent=1), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--replicates", type=int, default=32)
    ap.add_argument("--skip-timing", action="store_true")
    ap.add_argument("--skip-calibration", action="store_true")
    a = ap.parse_args()
    ab = load_product()
    ctx = ab.Context(0)
    try:
        result = {"card": card(), "truth": {"alpha": ALPHA, "beta": BETA}}
        if not a.skip_timing:
            result["timing"] = timing(ab, ctx)
        if not a.skip_calibration:
            result["calibration"] = calibration(ab, ctx, a.replicates)
    finally:
        ctx.close()
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print("written", a.out)


if __name__ == "__main__":
    main()
