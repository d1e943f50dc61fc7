"""Throughput of the ABneutral simulator (abfit_simulate_device) on the C5 time structure: 10 lines x 20 generations
below one founder, 200 sampled methylomes of 5 M sites, outputs in device memory (17 bytes per sample-site, 17 GB).

Reports the simulation kernel's time and output bandwidth, the bandwidth of plain store kernels writing the same bytes
(torch fill_ of the three output arrays, measured in the same run: the HBM store rate the simulator is compared with),
and the time of the simulate + observed-divergence chain (abfit_simulate_device then abfit_divergence_device, no host
round trip of the site tables).

    python tools/bench_simulate.py [--sites 5000000] [--reps 5] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=5_000_000)
    ap.add_argument("--lines", type=int, default=10)
    ap.add_argument("--generations", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--alpha", type=float, default=1e-3)
    ap.add_argument("--beta", type=float, default=2e-3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    from __graft_entry__ import _load_product

    ab = _load_product()
    ctx = ab.Context(0)
    tree = ab.SimTree.lines(a.lines, range(1, a.generations + 1))
    S, L = tree.n_samples, a.sites
    out_bytes = S * L * 17
    dev = torch.device("cuda", 0)
    status = torch.empty((S, L), dtype=torch.uint8, device=dev)
    post = torch.empty((S, L), dtype=torch.float64, device=dev)
    meth = torch.empty((S, L), dtype=torch.float64, device=dev)
    ptrs = (status.data_ptr(), post.data_ptr(), meth.data_ptr())

    def simulate(seed):
        return ctx.simulate_device(tree, *ptrs, a.alpha, a.beta, L=L, seed=seed)

    def store_ms():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        status.fill_(1)
        post.fill_(1.0)
        meth.fill_(0.5)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    # warm-up of every shape (outputs are 17 GB: far beyond L2, every pass goes to HBM)
    simulate(0)
    store_ms()
    ctx.dmatrix_device(*ptrs, S, L)
    sim, store, chain = [], [], []
    for r in range(a.reps):  # alternated, so that both see the same conditions
        sim.append(simulate(r + 1))
        store.append(store_ms())
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        simulate(100 + r)
        dm = ctx.dmatrix_device(*ptrs, S, L)
        chain.append((time.perf_counter() - t0) * 1e3)
    sim_ms, store_med, chain_ms = float(np.median(sim)), float(np.median(store)), float(np.median(chain))
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split("\n")[0]
    except Exception as e:  # the measurement stands without it; say so
        smi = f"unavailable ({e})"
    res = {
        "tool": "bench_simulate",
        "device": torch.cuda.get_device_name(0),
        "nvidia_smi_name_power_limit_max_sm_clock": smi,
        "design": f"{a.lines} lines x {a.generations} generations below one founder",
        "n_nodes": tree.n_nodes, "n_samples": S, "n_pairs": tree.n_pairs, "sites": L,
        "alpha": a.alpha, "beta": a.beta, "reps": a.reps,
        "output_bytes": out_bytes,
        "simulate_kernel_ms": sim_ms, "simulate_kernel_ms_all": sim,
        "simulate_output_GBps": out_bytes / (sim_ms * 1e-3) / 1e9,
        "store_kernels_ms": store_med, "store_kernels_ms_all": store,
        "store_GBps": out_bytes / (store_med * 1e-3) / 1e9,
        "fraction_of_store_bandwidth": store_med / sim_ms,
        "simulate_plus_dmatrix_ms": chain_ms, "simulate_plus_dmatrix_ms_all": chain,
        "dmatrix_kernel_ms": list(dm["kernel_ms"]),
        "mean_D": float(np.mean(dm["D"])),
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
