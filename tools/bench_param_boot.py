"""Time the parametric bootstrap (abfit_param_boot_batch) on one GPU: simulate-and-count (k_psim_counts + k_psim_dstar)
and the refit, and compare the fused simulate-and-count with the materialising route (abfit_simulate_device into
[S][L] site arrays, then abfit_divergence_device) in the same run, alternating the two.

    python3 tools/bench_param_boot.py [--shape c5|metaprofile|both] [--rounds 2] [--out results.json]

Shapes:
  c5           one window, 200 samples (the 201-node C5 tree, 20 lines x generations 1..10) x 5 M sites, 100 replicates
  metaprofile  10 000 windows x 1000 sites, 27 samples (3 lines x generations 1..9, 351 pairs), 100 replicates
Device times are the sums of kernel durations recorded by torch.profiler (CUDA activities).  The materialising route
runs one simulation per replicate over all windows' sites with one model (the fused call simulates every window from
its own model; the bytes and the pair work are the same).  The card's name and power limit are printed with the
numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import load_product  # noqa: E402

ALPHA, BETA = 3e-3, 6e-3


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def kernel_ms(prof, names):
    """device time (ms) of the kernels whose names contain one of `names`, and of all kernels"""
    sel = tot = 0.0
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        tot += us
        if any(n in e.name for n in names):
            sel += us
    return sel / 1e3, tot / 1e3


def profiled(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, prof, (time.perf_counter() - t0) * 1e3


def run_shape(ab, ctx, name, rounds):
    import torch

    if name == "c5":
        tree, n_win, L = ab.SimTree.lines(20, range(1, 11)), 1, 5_000_000
    else:
        tree, n_win, L = ab.SimTree.lines(3, range(1, 10)), 10_000, 1000
    n_boot, S, R = 100, tree.n_samples, tree.n_pairs
    p0, w = ab.sim_equilibrium(ALPHA, BETA)
    ped = np.column_stack([tree.pairs()[:, 2:5], np.full(R, 0.05)])
    probs = [ab.Problem(ped, p0, p0, 1.0)] * n_win
    best = np.zeros(n_win, dtype=ab.FIT_DTYPE)
    best["theta"] = (ALPHA, BETA, w, 0.0)
    miss = np.full((n_win, S), 0.05)
    dev = torch.device("cuda", 0)
    st = torch.empty((S, n_win * L), dtype=torch.uint8, device=dev)
    po = torch.empty((S, n_win * L), dtype=torch.float64, device=dev)
    me = torch.empty((S, n_win * L), dtype=torch.float64, device=dev)
    seg = np.arange(n_win + 1, dtype=np.int64) * L
    torch.cuda.synchronize()

    def fused():
        return ctx.parametric_bootstrap(tree, probs, [L] * n_win, miss, best, n_boot, 7)

    def materialising():
        for b, s in enumerate(ab.gen_param_boot_seeds(7, 0, n_boot)):
            ctx.simulate_device(tree, st.data_ptr(), po.data_ptr(), me.data_ptr(), ALPHA, BETA, w, p0, L=n_win * L,
                                seed=int(s), missing_rate=0.05)
            ctx.dmatrix_device(st.data_ptr(), po.data_ptr(), me.data_ptr(), S, n_win * L, seg_offsets=seg)

    # warm-up of every kernel and shape the timed rounds use
    ctx.parametric_bootstrap(tree, probs[:1], [min(L, 100_000)], miss[:1], best[:1], 2, 1, max_iters=5)
    ctx.simulate_device(tree, st.data_ptr(), po.data_ptr(), me.data_ptr(), ALPHA, BETA, w, p0, L=n_win * L, seed=1)
    ctx.dmatrix_device(st.data_ptr(), po.data_ptr(), me.data_ptr(), S, n_win * L, seg_offsets=seg)
    out = []
    for r in range(rounds):
        res, prof, wall = profiled(fused)
        simc, tot = kernel_ms(prof, ("k_psim_counts", "k_psim_dstar"))
        _, prof2, wall2 = profiled(materialising)
        _, mat = kernel_ms(prof2, ("",))
        row = {"shape": name, "round": r, "windows": n_win, "sites": L, "samples": S, "rows": R, "replicates": n_boot,
               "fused_sim_count_ms": simc, "fused_refit_and_rest_ms": tot - simc, "fused_call_wall_ms": wall,
               "materialising_sim_count_ms": mat, "materialising_wall_ms": wall2,
               "nan_reps": int(res["nan_reps"].sum()), "gof_p_median": float(np.nanmedian(res["gof_p"]))}
        print(json.dumps(row), flush=True)
        out.append(row)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="both", choices=["c5", "metaprofile", "both"])
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ab = load_product()
    ctx = ab.Context(0)
    info = {"card": card()}
    print(json.dumps(info), flush=True)
    rows = []
    for s in (["c5", "metaprofile"] if a.shape == "both" else [a.shape]):
        rows += run_shape(ab, ctx, s, a.rounds)
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump({"device": info, "rows": rows}, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
