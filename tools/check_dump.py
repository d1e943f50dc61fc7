#!/usr/bin/env python3
"""Check a `bench.py --dump-outputs DIR` directory against the oracle.

    python3 tools/check_dump.py DIR [--starts 1000 --boots 100 --sample K]

A dumped window's inputs depend only on its index: its pedigree comes from bench.synth_windows, its start simplices,
resample indices and vary vertices from oracle/gen_py.py keyed by bench.SEED and the window index.  So every dumped
window can be refitted by the oracle (multi-start fit, then the bootstrap from the oracle's own best model) without
the product library, and its best record, pred, resid, status and bootstrap rows compared bit for bit.  K of the
dumped windows are checked (a seeded sample; all of them with --sample 0).  Prints one line per window and a summary;
the exit status is 1 if any window differs."""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BEST_FIELDS = ("theta", "cost", "lse", "iters", "evals", "status", "start_id")
ERR_NAN = -4  # ABFIT_ERR_NAN (include/abfit.h)


def _bits_equal(a, b):
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def oracle_window(o, shape, window, starts, boots, threads):
    """the oracle's fit and bootstrap of synthetic C4 window `window` -> dict(rc, best, all, pred, resid, rows, fits)
    (rows and fits None when the oracle refuses the window)"""
    import bench
    from oracle import gen_py as g

    peds, p0uu = bench.synth_windows(1, window, shape)
    ped, u = peds[0], float(p0uu[0])
    pb = o.Problem(ped, u, u, 1.0)
    flags = o.FAST_DIVERGENCE | o.EARLY_EXIT_ON_STALL
    sx = g.gen_start_simplices(bench.SEED, window, starts, float(ped[:, 3].max()))
    rc, best, allr, pred, resid = o.ab_neutral(pb, sx, flags=flags, n_threads=threads)
    rows = fits = None
    if rc == 0:
        idx = g.gen_resample_idx(bench.SEED, window, boots, len(ped))
        vary = g.gen_vary_vertices(bench.SEED, window, boots, best["theta"])
        rc2, rows, fits = o.boot_model(pb, best["theta"], pred, resid, idx, vary, flags=flags, n_threads=threads)
        assert rc2 == 0, (window, rc2)
    return {"rc": rc, "best": best, "all": allr, "pred": pred, "resid": resid, "rows": rows, "fits": fits}


def check(dump_dir, starts=1000, boots=100, sample=8, threads=None, out=sys.stdout):
    """checks `sample` dumped windows (all with 0) against the oracle; returns {window: [names of arrays that differ]}"""
    import bench
    from oracle import abref_py as o

    o.build()
    threads = threads or o.hw_threads()
    d = {f[:-4]: np.load(os.path.join(dump_dir, f)) for f in os.listdir(dump_dir) if f.endswith(".npy")}
    windows = d["window"].astype(np.int64)
    rows_at = np.arange(len(windows))
    if sample and sample < len(windows):
        rows_at = np.sort(np.random.default_rng([bench.SEED, len(windows)]).choice(len(windows), sample, replace=False))
    if d["boot_rows"].shape[1] != boots:
        raise ValueError(f"the dump holds {d['boot_rows'].shape[1]} bootstrap replicates per window, not {boots}")
    shape = bench.load_shape()
    diffs = {}
    for k in rows_at:
        w = int(windows[k])
        r = oracle_window(o, shape, w, starts, boots, threads)
        rc, best, pred, resid, rows = r["rc"], r["best"], r["pred"], r["resid"], r["rows"]
        # a window the oracle refuses (NaN in its pedigree) has the library's window status ABFIT_ERR_NAN
        bad = [] if _bits_equal(d["status"][k], 0 if rc == 0 else ERR_NAN if rc == o.ERR_NAN else rc) else ["status"]
        if rc == 0:
            bad += [f"best_{f}" for f in BEST_FIELDS if not _bits_equal(d["best_" + f][k], best[f])]
            bad += [n for n, ref in (("pred", pred), ("resid", resid), ("boot_rows", rows)) if not _bits_equal(d[n][k], ref)]
        diffs[w] = bad
        print(f"window {w}: " + ("identical to the oracle" if not bad else "DIFFERS in " + ", ".join(bad)), file=out,
              flush=True)
    n_ok = sum(1 for b in diffs.values() if not b)
    print(f"{n_ok} of {len(diffs)} windows identical to the oracle ({len(windows)} windows in the dump)", file=out)
    return diffs


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("dir")
    ap.add_argument("--starts", type=int, default=1000)
    ap.add_argument("--boots", type=int, default=100)
    ap.add_argument("--sample", type=int, default=8, help="windows to check (0: every dumped window)")
    args = ap.parse_args()
    diffs = check(args.dir, args.starts, args.boots, args.sample)
    return 1 if any(diffs.values()) else 0


if __name__ == "__main__":
    sys.exit(main())
