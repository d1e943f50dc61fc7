"""Observed divergence of many genomic regions over resident site arrays (abfit_region_divergence_device) against the
route the library offered before it: gather every region's sites into a new [S][sum len] array, then one
abfit_divergence_device call with a window per region.

Shape: S samples x 5.5 M sites simulated on the device (5.5 M is an assumed Arabidopsis CG count: 135 Mb at ~41 CG per
kb).  Regions are index-range tiles of 407 sites (10 kb at that density):
  * overlap:     13 500 tiles at a step of 41 sites (10 kb tiles at a 1 kb step over the first ~13.5 Mb; every site in
                 ten tiles),
  * disjoint:    13 500 tiles at a step of 407 sites (10 kb tiles over the whole genome).
Default widths 27 and 200 (C5) samples.  The gather runs on the device (torch index_select, timed with CUDA events
together with the divergence kernels); at --host-samples width it is also run from the host (numpy gather, then
abfit_divergence, which copies the gathered arrays to the device), timed on the host clock.  The outputs of both routes
are compared bit for bit.  Bytes: the inputs each route reads and writes, from the shapes (17 bytes per sample-site of
status, posteriorMax and meth_lvl; methsum re-reads 16 bytes per sample-site of every region).

    python tools/bench_regions.py [--samples 27,200] [--sites 5500000] [--reps 3] [--host-samples 27] [--out r.json]
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

TILE, STEP_OVERLAP, N_TILES = 407, 41, 13_500


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", default="27,200")
    ap.add_argument("--sites", type=int, default=5_500_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--host-samples", type=int, default=27)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    from __graft_entry__ import _load_product

    ab = _load_product()
    ctx = ab.Context(0)
    dev = torch.device("cuda", 0)
    L = a.sites
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split("\n")[0]
    except Exception as e:  # the measurement stands without it; say so
        smi = f"unavailable ({e})"
    results = []
    for S in [int(s) for s in a.samples.split(",")]:
        n_lines = 10 if S % 10 == 0 else 1
        tree = ab.SimTree.lines(n_lines, range(1, S // n_lines + 1))
        assert tree.n_samples == S
        st = torch.empty((S, L), dtype=torch.uint8, device=dev)
        po = torch.empty((S, L), dtype=torch.float64, device=dev)
        me = torch.empty((S, L), dtype=torch.float64, device=dev)
        torch.cuda.synchronize()
        ctx.simulate_device(tree, st.data_ptr(), po.data_ptr(), me.data_ptr(), 1e-3, 2e-3, L=L, seed=3, missing_rate=0.05)
        for case, step in (("overlap", STEP_OVERLAP), ("disjoint", TILE)):
            lo = np.arange(N_TILES, dtype=np.int64) * step
            keep = lo + TILE <= L
            lo = lo[keep]
            hi = lo + TILE
            W = len(lo)
            idx = torch.from_numpy(np.concatenate([np.arange(x, y) for x, y in zip(lo, hi)])).to(dev)
            seg = np.arange(W + 1, dtype=np.int64) * TILE
            union = int(hi[-1] - lo[0])  # step <= TILE: the tiles cover one contiguous range

            def regions():
                return ctx.region_divergence_device(st.data_ptr(), po.data_ptr(), me.data_ptr(), S, L, lo, hi)

            def gathered():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                gs, gp, gm = st.index_select(1, idx), po.index_select(1, idx), me.index_select(1, idx)
                e1.record()
                e1.synchronize()
                out = ctx.dmatrix_device(gs.data_ptr(), gp.data_ptr(), gm.data_ptr(), S, int(idx.numel()), seg_offsets=seg)
                g_ms = e0.elapsed_time(e1)
                del gs, gp, gm
                return out, g_ms

            regions()  # warm-up of both routes (the inputs, 17 B per sample-site, are far beyond L2)
            gathered()
            reg_ms, gat_ms, gat_div_ms = [], [], []
            for _ in range(a.reps):  # alternated, so that both see the same conditions
                r = regions()
                reg_ms.append(r["kernel_ms"])
                g, g_ms = gathered()
                gat_ms.append(g_ms + sum(g["kernel_ms"]))
                gat_div_ms.append(sum(g["kernel_ms"]))
            same = all(np.array_equal(np.asarray(r[k]).view(np.uint64), np.asarray(g[k]).view(np.uint64))
                       for k in ("D", "diff", "cnt", "p0uu", "methsum", "nvalid"))
            tot = W * TILE
            res = {
                "samples": S, "sites": L, "case": case, "regions": W, "region_sites": TILE, "step_sites": step,
                "sites_in_regions": tot, "sites_covered": union,
                "region_divergence_device_ms": float(np.median(reg_ms)), "region_divergence_device_ms_all": reg_ms,
                "gather_plus_divergence_device_ms": float(np.median(gat_ms)), "gather_plus_divergence_device_ms_all": gat_ms,
                "divergence_of_gathered_ms": float(np.median(gat_div_ms)),
                "outputs_bit_identical": bool(same),
                "bytes_regions": S * (17 * union + 16 * tot),
                "bytes_gather_route": S * (17 * tot * 3 + 16 * tot),
            }
            if S <= a.host_samples:
                hs, hp, hm = st.cpu().numpy(), po.cpu().numpy(), me.cpu().numpy()
                hidx = idx.cpu().numpy()
                t_host = []
                for _ in range(a.reps):
                    t0 = time.perf_counter()
                    h = ctx.dmatrix(hs[:, hidx], hp[:, hidx], hm[:, hidx], seg_offsets=seg)
                    t_host.append((time.perf_counter() - t0) * 1e3)
                t_reg = []
                for _ in range(a.reps):
                    t0 = time.perf_counter()
                    hr = ctx.region_divergence(hs, hp, hm, lo, hi)
                    t_reg.append((time.perf_counter() - t0) * 1e3)
                res["host_gather_plus_divergence_ms"] = float(np.median(t_host))
                res["host_region_divergence_ms"] = float(np.median(t_reg))
                res["host_outputs_bit_identical"] = bool(np.array_equal(h["D"].view(np.uint64), hr["D"].view(np.uint64)) and
                                                         np.array_equal(h["methsum"].view(np.uint64), hr["methsum"].view(np.uint64)))
                del hs, hp, hm
            print(json.dumps(res), flush=True)
            results.append(res)
            del idx
        del st, po, me
        torch.cuda.empty_cache()
    out = {"tool": "bench_regions", "device": torch.cuda.get_device_name(0),
           "nvidia_smi_name_power_limit_max_sm_clock": smi, "reps": a.reps, "results": results}
    print(json.dumps(out))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
