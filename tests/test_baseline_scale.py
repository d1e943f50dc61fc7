"""The benchmark's configuration at full size, against the oracle.

BASELINE configs[3] is 10 000 windows x (1000 starts + 100 bootstrap replicates) of the 351-pair C4 pedigree.  Only at
this size do the default kernels cut guided work items of 256 fits, does the multi-start kernel of
abfit_alphabeta_batch wait on the upload of 1.6 GB of pinned start simplices, and are the continuous-scheduling
kernels relaunched step after step on one resident batch.  The inputs are built as bench.py builds them.

* R0, the reference route, is bench.py's preparation of its resident batch: upload_starts -> run_fit ->
  download_fit(want_all) -> host vary vertices -> upload_boot -> run_boot -> download_boot(want_fits).  Sampled
  windows are compared with the oracle: every start record, best, pred, resid, bootstrap rows and replicate fits.
* R1-R9 are the other routes (repeated pipelined steps, the end-to-end call with pinned, pageable or device-drawn
  inputs, the interpreter kernels, one rank's shard, NaN windows, a second call on the same context).  Each is
  compared with R0 byte for byte over all 10 000 windows.
"""
import importlib.util
import os
import re
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

W, NS, NB = 10000, 1000, 100
# first and last windows, and both sides of the first upload-chunk boundaries (256 windows per chunk)
EDGE_WINDOWS = (0, 1, 255, 256, 511, 512, 4999, 5000, 9998, 9999)
FIELDS = ("theta", "cost", "lse", "iters", "evals", "status", "start_id")
BOOT_FIELDS = ("theta", "cost", "iters", "evals", "status", "start_id")  # the oracle's bootstrap fits carry no lse
V2_KERNELS = {"abfit_jit_fit_starts_v2", "abfit_jit_fit_boot_gather_v2"}
DEV_KNOBS = ("ABFIT_JIT", "ABFIT_JIT_MIN_FITS", "ABFIT_DEV_NWARPS", "ABFIT_DEV_XGLOBAL", "ABFIT_DEV_BIG", "ABFIT_DEV_WIDE",
             "ABFIT_DEV_BOOT_XGLOBAL", "ABFIT_DEV_BOOT_TILE", "ABFIT_DEV_CHUNK", "ABFIT_DEV_PIPES", "ABFIT_DEV_SCHED",
             "ABFIT_DEV_NO_UPLOAD_WATCH", "ABFIT_DEV_HOST_STATS", "ABFIT_EXPERIMENT_SUFFSTATS", "ABFIT_DEV_VERBOSE")


def _load_tool(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "tools", name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


check_dump = _load_tool("check_dump")


def sampled_windows():
    rest = np.setdiff1d(np.arange(W), EDGE_WINDOWS)
    return sorted(EDGE_WINDOWS) + sorted(int(w) for w in np.random.default_rng(20261022).choice(rest, 14, replace=False))


# ---------------------------------------------------------------------------------------------
# comparisons
# ---------------------------------------------------------------------------------------------
def per_window(a, n):
    return np.ascontiguousarray(a).view(np.uint8).reshape(n, -1)


def same_bytes(got, ref, what, n=W, skip=()):
    """byte for byte, window by window (axis 0 holds n windows); names the first windows that differ"""
    g, r = per_window(got, n), per_window(ref, n)
    assert g.shape == r.shape, (what, g.shape, r.shape)
    bad = np.flatnonzero((g != r).any(axis=1))
    bad = bad[~np.isin(bad, skip)]
    assert bad.size == 0, f"{what}: {bad.size} windows differ, the first ones {bad[:8].tolist()}"


def same_route(got, ref, what, keys=("best", "pred", "resid", "status", "rows"), n=W, skip=()):
    for k in keys:
        same_bytes(got[k], ref[k], f"{what} {k}", n, skip)


def same_fields(got, ref, fields, what):
    for f in fields:
        g, r = np.ascontiguousarray(got[f]), np.ascontiguousarray(ref[f])
        assert g.shape == r.shape and np.array_equal(g.view(np.uint8), r.view(np.uint8)), (what, f)


def same_bits(got, ref, what):
    g, r = np.ascontiguousarray(got, dtype=np.float64), np.ascontiguousarray(ref, dtype=np.float64)
    assert g.shape == r.shape and np.array_equal(g.view(np.uint64), r.view(np.uint64)), what


def check_against_oracle(res, window, ref, what, row=None, fits=True, all_records=True):
    """res: a route's outputs; `row` is the window's position in them (default: `window`)"""
    p = window if row is None else row
    assert ref["rc"] == 0 and res["status"][p] == 0, (what, window)
    if all_records:
        same_fields(res["all"][p], ref["all"], FIELDS, (what, "start records", window))
    same_fields(res["best"][p], ref["best"], FIELDS, (what, "best", window))
    N = len(ref["pred"])
    same_bits(res["pred"][p * N:(p + 1) * N], ref["pred"], (what, "pred", window))
    same_bits(res["resid"][p * N:(p + 1) * N], ref["resid"], (what, "resid", window))
    same_bits(res["rows"][p], ref["rows"], (what, "bootstrap rows", window))
    if fits:
        same_fields(res["fits"][p], ref["fits"], BOOT_FIELDS, (what, "replicate fits", window))


# ---------------------------------------------------------------------------------------------
# fixtures: inputs, the oracle, the reference route R0
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", autouse=True)
def _env(tmp_path_factory):
    """the defaults, and one JIT cache for the module (the specialised kernels are compiled once)"""
    with pytest.MonkeyPatch.context() as mp:
        for k in DEV_KNOBS:
            mp.delenv(k, raising=False)
        mp.setenv("ABFIT_CACHE_DIR", str(tmp_path_factory.mktemp("jit-cache")))
        yield


@pytest.fixture(scope="module")
def torch():
    import torch

    return torch


@pytest.fixture(scope="module")
def bench():
    import bench

    return bench


@pytest.fixture(scope="module")
def pool():
    with ThreadPoolExecutor(max_workers=max(4, min(32, os.cpu_count() or 8))) as p:
        yield p


@pytest.fixture(scope="module")
def inputs(ab, torch, bench, pool):
    """bench.make_inputs: pinned start simplices and resample indices, keyed by bench.SEED and the window index"""
    peds, probs, sx_t, idx_t = bench.make_inputs(ab, torch, W, 0, NS, NB, bench.load_shape(), pool)
    return {"peds": peds, "probs": probs, "sx_t": sx_t, "idx_t": idx_t, "sx": sx_t.numpy(), "idx": idx_t.numpy()}


def oracle_windows(bench, oracle, windows):
    shape = bench.load_shape()
    threads = os.cpu_count() or 8
    t0 = time.perf_counter()
    ref = {w: check_dump.oracle_window(oracle, shape, w, NS, NB, threads) for w in windows}
    print(f"\noracle: {len(windows)} windows x ({NS} starts + {NB} replicates) in {time.perf_counter() - t0:.1f} s "
          f"on {threads} threads")
    return ref


@pytest.fixture(scope="module")
def oracle_ref(bench, oracle):
    return oracle_windows(bench, oracle, sampled_windows())


def gen_vary(ab, bench, pool, best_theta, first=0):
    vary = np.empty((len(best_theta), NB, 4, 4))

    def one(i):
        vary[i] = ab.gen_vary_vertices(bench.SEED, first + i, NB, best_theta[i])

    list(pool.map(one, range(len(best_theta))))
    return vary


def resident(ab, bench, pool, ctx, inputs, vary=None):
    """bench.py's preparation of its resident batch; returns the batch, its outputs and its evaluation counters"""
    batch = ctx.batch(inputs["probs"])
    batch.upload_starts(inputs["sx"])
    batch.run_fit()
    fit = batch.download_fit(want_all=True)
    if vary is None:
        vary = gen_vary(ab, bench, pool, fit.best["theta"])
    batch.upload_boot(inputs["idx"], vary)
    batch.run_boot()
    rows, fits = batch.download_boot(want_fits=True)
    out = {"best": fit.best, "all": fit.all, "pred": fit.pred, "resid": fit.resid, "status": fit.status, "rows": rows,
           "fits": fits, "vary": vary, "timing": batch.timing()}
    return batch, out


@pytest.fixture(scope="module")
def r0(ab, bench, pool, ctx, inputs):
    batch, out = resident(ab, bench, pool, ctx, inputs)
    out["batch"] = batch
    yield out
    batch.close()


def e2e(ab, torch, bench, ctx, probs, sx, idx, first=0, packed=None):
    """ctx.alphabeta_batch as bench.py's e2e_step calls it: pinned outputs, packed problems"""
    n, N = len(probs), probs[0].n_pairs
    best_t = torch.zeros((n, 64), dtype=torch.uint8, pin_memory=True)
    pred_t = torch.empty(n * N, dtype=torch.float64, pin_memory=True)
    resid_t = torch.empty(n * N, dtype=torch.float64, pin_memory=True)
    rows_t = torch.empty((n, NB, 7), dtype=torch.float64, pin_memory=True)
    best = best_t.numpy().view(ab.FIT_DTYPE).reshape(n)
    status, analysis = np.zeros(n, dtype=np.int32), np.empty((n, 32))
    ctx.alphabeta_batch(probs, sx, idx, bench.SEED, first_problem_id=first, best=best, pred=pred_t.numpy(),
                        resid=resid_t.numpy(), status=status, rows=rows_t.numpy(), analysis=analysis,
                        packed=ab._pack_problems(probs) if packed is None else packed)
    return {"best": best.copy(), "pred": pred_t.numpy().copy(), "resid": resid_t.numpy().copy(), "status": status,
            "rows": rows_t.numpy().copy(), "analysis": analysis}


def verbose(monkeypatch, capfd, fn, **env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv("ABFIT_DEV_VERBOSE", "1")
    capfd.readouterr()
    r = fn()
    err = capfd.readouterr().err
    monkeypatch.delenv("ABFIT_DEV_VERBOSE")
    for k in env:
        monkeypatch.delenv(k)
    return r, err


def kernels_named(err):
    return set(re.findall(r"\[abfit\] ((?:k|abfit_jit)_\w+)", err))


WATCH_LINE = "the multi-start kernel watches the upload"


# ---------------------------------------------------------------------------------------------
# R0 against the oracle
# ---------------------------------------------------------------------------------------------
def test_r0_is_the_benchmark_path_and_counts_its_evaluations(r0):
    batch = r0["batch"]
    assert batch.uses_specialised_kernels()
    assert np.all(r0["status"] == 0)
    # bench.py's roofline divides evals_fit by the multi-start kernel's time
    assert r0["timing"]["evals_fit"] == int(r0["all"]["evals"].astype(np.int64).sum())
    assert r0["timing"]["evals_boot"] == int(r0["fits"]["evals"].astype(np.int64).sum())


def test_r0_against_the_oracle(r0, oracle_ref):
    for w, ref in oracle_ref.items():
        check_against_oracle(r0, w, ref, "R0")


# ---------------------------------------------------------------------------------------------
# R1: the resident batch after bench.py's warm-up and timed steps
# ---------------------------------------------------------------------------------------------
def test_r1_repeated_pipelined_steps(ab, bench, r0, tmp_path):
    batch = r0["batch"]
    for _ in range(2 + 3):
        batch.run_pipelined()
        assert batch.pipes() == 1
    t = batch.timing()
    fit = batch.download_fit(want_all=True)
    rows, fits = batch.download_boot(want_fits=True)
    r1 = {"best": fit.best, "all": fit.all, "pred": fit.pred, "resid": fit.resid, "status": fit.status, "rows": rows,
          "fits": fits}
    same_route(r1, r0, "R1", keys=("best", "all", "pred", "resid", "status", "rows", "fits"))
    assert t["evals_fit"] == r0["timing"]["evals_fit"] and t["evals_boot"] == r0["timing"]["evals_boot"]
    # bench.py --dump-outputs of this step, checked against the oracle by tools/check_dump.py
    bench.dump_outputs(str(tmp_path), fit, rows, 0, r0["pred"].size // W)
    diffs = check_dump.check(str(tmp_path), NS, NB, sample=4)
    assert len(diffs) == 4 and not any(diffs.values()), diffs


# ---------------------------------------------------------------------------------------------
# R2-R5: the end-to-end call
# ---------------------------------------------------------------------------------------------
def test_r2_end_to_end_pinned(ab, torch, bench, ctx, inputs, r0, oracle, oracle_ref, monkeypatch, capfd):
    probs, packed = inputs["probs"], ab._pack_problems(inputs["probs"])
    r2, err = verbose(monkeypatch, capfd, lambda: e2e(ab, torch, bench, ctx, probs, inputs["sx"], inputs["idx"],
                                                      packed=packed))
    assert kernels_named(err) == V2_KERNELS, err
    assert WATCH_LINE in err, err
    same_route(r2, r0, "R2")
    for w in range(W):
        assert np.array_equal(r2["analysis"][w], ab.analyze(r2["rows"][w]), equal_nan=True), ("analysis", w)
    for w, ref in oracle_ref.items():
        same_bits(r2["analysis"][w], oracle.analyze(ref["rows"]), ("R2 analysis against the oracle", w))
    # whether a warp had to wait for the upload depends on timing: reported, not asserted
    m = re.search(r"alphabeta_batch: enqueue kernels\s+([\d.]+) ms", err)
    dst = torch.empty(inputs["sx_t"].shape, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dst.copy_(inputs["sx_t"], non_blocking=True)
    torch.cuda.synchronize()
    copy_ms = 1e3 * (time.perf_counter() - t0)
    del dst
    print(f"\nR2: enqueue kernels {m.group(1) if m else '?'} ms; torch pinned copy of the "
          f"{inputs['sx'].nbytes / 1e9:.2f} GB of start simplices {copy_ms:.1f} ms")


def test_r3_without_the_upload_watch(ab, torch, bench, ctx, inputs, r0, monkeypatch, capfd):
    r3, err = verbose(monkeypatch, capfd, lambda: e2e(ab, torch, bench, ctx, inputs["probs"], inputs["sx"], inputs["idx"]),
                      ABFIT_DEV_NO_UPLOAD_WATCH="1")
    assert WATCH_LINE not in err, err
    assert kernels_named(err) == V2_KERNELS, err
    same_route(r3, r0, "R3")


def test_r4_pageable_inputs(ab, torch, bench, ctx, inputs, r0):
    sx, idx = np.array(inputs["sx"]), np.array(inputs["idx"])  # pageable copies
    same_route(e2e(ab, torch, bench, ctx, inputs["probs"], sx, idx), r0, "R4")


def test_r5_resample_indices_drawn_on_the_device(ab, torch, bench, ctx, inputs, r0):
    same_route(e2e(ab, torch, bench, ctx, inputs["probs"], inputs["sx"], NB), r0, "R5")


# ---------------------------------------------------------------------------------------------
# R6-R9
# ---------------------------------------------------------------------------------------------
def test_r6_interpreter_kernels(ab, bench, pool, ctx, inputs, r0, monkeypatch):
    monkeypatch.setenv("ABFIT_JIT", "0")
    batch, r6 = resident(ab, bench, pool, ctx, inputs, vary=r0["vary"])
    try:
        assert not batch.uses_specialised_kernels()
    finally:
        batch.close()
    same_route(r6, r0, "R6", keys=("best", "all", "pred", "resid", "status", "rows", "fits"))


def test_r7_one_rank_of_eight(ab, torch, bench, ctx, inputs, r0):
    from alphabeta_rs_b200 import multi

    lo, n = multi.window_shard(W, 3, 8)
    assert (lo, n) == (3750, 1250)
    hi, N = lo + n, r0["pred"].size // W
    r7 = e2e(ab, torch, bench, ctx, inputs["probs"][lo:hi], inputs["sx"][lo:hi], inputs["idx"][lo:hi], first=lo)
    ref = {"best": r0["best"][lo:hi], "pred": r0["pred"][lo * N:hi * N], "resid": r0["resid"][lo * N:hi * N],
           "status": r0["status"][lo:hi], "rows": r0["rows"][lo:hi]}
    same_route(r7, ref, "R7", n=n)


def test_r8_nan_windows(ab, torch, bench, ctx, inputs, r0):
    nan_w = [256, 257, 5000]
    probs = list(inputs["probs"])
    for w in nan_w:
        ped = inputs["peds"][w].copy()
        ped[:, 3] = np.nan
        probs[w] = ab.Problem(ped, probs[w].p0uu, probs[w].eqp, probs[w].eqp_weight)
    r8 = e2e(ab, torch, bench, ctx, probs, inputs["sx"], inputs["idx"])
    assert np.all(r8["status"][nan_w] == ab.ERR_NAN) and np.all(r8["best"]["status"][nan_w] == ab.FIT_NAN)
    same_route(r8, r0, "R8", skip=nan_w)


def test_r9_second_call_on_the_same_context(ab, torch, bench, pool, ctx, inputs, oracle):
    """the second of two same-shape calls on one context: its multi-start kernel must not read the upload counter
    before the reset of the previous call's count has landed"""
    peds2, probs2, sx2_t, idx2_t = bench.make_inputs(ab, torch, W, W, NS, NB, bench.load_shape(), pool)
    e2e(ab, torch, bench, ctx, inputs["probs"], inputs["sx"], inputs["idx"])
    r9 = e2e(ab, torch, bench, ctx, probs2, sx2_t.numpy(), idx2_t.numpy(), first=W)
    fresh = ab.Context(0)
    try:
        ref = e2e(ab, torch, bench, fresh, probs2, sx2_t.numpy(), idx2_t.numpy(), first=W)
    finally:
        fresh.close()
    same_route(r9, ref, "R9")
    same_bytes(r9["analysis"], ref["analysis"], "R9 analysis")
    sample = [0, 256, 5000, 9999]
    sample += [int(w) for w in np.random.default_rng(9).choice(np.setdiff1d(np.arange(W), sample), 2, replace=False)]
    for w, o in oracle_windows(bench, oracle, [W + w for w in sample]).items():
        check_against_oracle(r9, w, o, "R9", row=w - W, fits=False, all_records=False)
        same_bits(r9["analysis"][w - W], oracle.analyze(o["rows"]), ("R9 analysis against the oracle", w))
