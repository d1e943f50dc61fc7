"""The fit path at every launch shape the planner picks and at the optimiser's edges, against the oracle.

* Shape pins (CPU): the host planner (abfit_plan.cu, abfit_jit.cu), built for the CPU in tests/host_emul, puts each
  pedigree below where its test claims, so a moved threshold cannot silently turn a case into a different one.
* Launch shapes (GPU): each pinned case runs with the default planner, under ABFIT_DEV_VERBOSE=1, which names the
  kernels it launches; every start record, the best-of-starts, pred / resid, the bootstrap rows and fits and the
  device-side analysis are compared bit for bit with the oracle.
* Optimiser edges (CPU and GPU): sd_tol and max_iters special cases, degenerate and +-inf / NaN simplices, costs of
  -inf (a very negative penalty weight), tied LSEs across lanes, warps and work items, windows with some or all
  starts NaN, on every fit and bootstrap kernel family, and through the device headers built for the CPU.
"""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

from conftest import GOLDEN
from test_host_emul import emul, random_pedigree  # noqa: F401  (emul is a fixture)

SEED = 0xF17ED6E
EPS = 2.220446049250313e-16
NT = os.cpu_count() or 4
SMEM_CAP = 227 * 1024  # opt-in shared memory per block of a B200, the cap emul_launch_shape plans with
FIELDS = ("theta", "cost", "lse", "iters", "evals", "status", "start_id")
BOOT_FIELDS = ("theta", "cost", "iters", "evals", "status", "start_id")  # the oracle's bootstrap fits carry no lse


# ---------------------------------------------------------------------------------------------
# pedigrees
# ---------------------------------------------------------------------------------------------
# ten (t0, t1, t2) triples of a lineage design: many lines, few generations
TRIP10 = [(0, 1, 1), (0, 1, 2), (0, 2, 2), (0, 2, 3), (0, 3, 5), (0, 4, 4), (0, 1, 6), (0, 6, 6), (0, 7, 7), (0, 8, 8)]


def ped10(n_pairs, seed=0):
    rng = np.random.default_rng(seed)
    return np.array([[*TRIP10[i % 10], rng.uniform(0.01, 0.3)] for i in range(n_pairs)], dtype=np.float64)


_ALL_TRIPLES = None


def distinct_triples(k, seed=1):
    """k pairs with k distinct triples 0 <= t0 <= t1 <= t2 <= 127"""
    global _ALL_TRIPLES
    if _ALL_TRIPLES is None:
        _ALL_TRIPLES = np.array([(t0, a, b) for t0 in range(128) for a in range(t0, 128) for b in range(a, 128)],
                                dtype=np.float64)
    rng = np.random.default_rng(seed)
    t = _ALL_TRIPLES[rng.choice(len(_ALL_TRIPLES), k, replace=False)]
    return np.ascontiguousarray(np.concatenate([t, rng.uniform(0.01, 0.3, (k, 1))], axis=1))


def lane_slots(m):
    """128 + 9 + m per-lane values: (0, a, a) for every a (one dt slot each), G^2 stored once, m triples (0, 2, b)"""
    t = [(0, a, a) for a in range(128)] + [(0, 2, b) for b in range(3, 3 + m)]
    rng = np.random.default_rng(m)
    return np.array([[*x, rng.uniform(0.01, 0.3)] for x in t], dtype=np.float64)


def ped351():
    from oracle import abref_py
    return abref_py.load_pedigree_file(os.path.join(GOLDEN, "pedigree.txt"))


# ---------------------------------------------------------------------------------------------
# host planner (tests/host_emul)
# ---------------------------------------------------------------------------------------------
SHAPE_KEYS = ("n_warps", "d_shared", "x_global", "big", "wide", "boot_x_global", "smem_fit", "smem_wide", "smem_boot_gather",
              "n_items")


def emul_shape(emul, ab, probs, fits_per_prob):
    arr = ab._pack_problems(probs)
    out = (C.c_int64 * 10)()
    rc = emul.emul_launch_shape(arr, len(probs), fits_per_prob, out)
    return rc, dict(zip(SHAPE_KEYS, [int(v) for v in out]))


def emul_stats(emul, ab, prob):
    arr = ab._pack_problems([prob])
    out = (C.c_int32 * 6)()
    rc = emul.emul_plan_stats(arr, out)
    return rc, dict(zip(("n_lane", "n_ops", "_", "tmax", "n_trip", "smem_1warp"), [int(v) for v in out]))


# ---------------------------------------------------------------------------------------------
# the cases: (problems, starts, replicates, max_iters fit / boot, environment, planner pin, kernels named)
# ---------------------------------------------------------------------------------------------
def _small():
    return (ped351(), 0.8)


CASES = {
    # the bootstrap index tile just fits (a quarter of the cap); the multi-start kernel keeps D and the vertices on chip
    "boot_index_tile_2000_pairs": dict(
        probs=lambda: [(ped10(2000), 0.7)], starts=64, boot=24, mi=(2000, 300),
        pin=dict(n_warps=1, d_shared=1, x_global=0, big=0, wide=0, smem_boot_gather=53696),
        kernels=["k_fit_starts<D_SHARED=1,X_GLOBAL=0,BIG=0>", "k_fit_boot_gather:"]),
    # a few more pairs: the tile no longer fits, the replicates' D* columns are stored
    "stored_dstar_2400_pairs": dict(
        probs=lambda: [(ped10(2400), 0.7)], starts=64, boot=24, mi=(2000, 300),
        pin=dict(n_warps=1, d_shared=1, x_global=1, big=0, wide=0, smem_boot_gather=0),
        kernels=["k_fit_starts<D_SHARED=1,X_GLOBAL=1,BIG=0>", "k_fit_boot<BIG=0>"]),
    # the same pedigree over 150 windows: enough fits for 3-warp multi-start blocks (windows 0, 75, 149 are checked)
    "stored_dstar_2400_pairs_150_windows": dict(
        probs=lambda: [(ped10(2400, seed=w), 0.7) for w in range(150)], starts=256, boot=8, mi=(300, 100),
        check=(0, 75, 149),
        pin=dict(n_warps=3, d_shared=1, x_global=0, big=0, wide=0, smem_boot_gather=0),
        kernels=["k_fit_starts<D_SHARED=1,X_GLOBAL=0,BIG=0>: 300 blocks x 3 warps", "k_fit_boot<BIG=0>"]),
    # D no longer fits next to the lane state: broadcast from L1/L2, vertices in global scratch
    "d_global_x_global_8191_pairs": dict(
        probs=lambda: [(ped10(8191), 0.7)], starts=48, boot=16, mi=(600, 200),
        pin=dict(n_warps=1, d_shared=0, x_global=1, big=0, wide=0, smem_boot_gather=0),
        kernels=["k_fit_starts<D_SHARED=0,X_GLOBAL=1,BIG=0>", "k_fit_boot<BIG=0>"]),
    "d_global_x_global_8192_pairs": dict(
        probs=lambda: [(ped10(8192), 0.7)], starts=48, boot=16, mi=(600, 200),
        pin=dict(n_warps=1, d_shared=0, x_global=1, big=0, wide=0, smem_boot_gather=0),
        kernels=["k_fit_starts<D_SHARED=0,X_GLOBAL=1,BIG=0>", "k_fit_boot<BIG=0>"]),
    "d_global_x_global_12000_pairs": dict(
        probs=lambda: [(ped10(12000), 0.7)], starts=40, boot=12, mi=(400, 150),
        pin=dict(n_warps=1, d_shared=0, x_global=1, big=0, wide=0, smem_boot_gather=0),
        kernels=["k_fit_starts<D_SHARED=0,X_GLOBAL=1,BIG=0>", "k_fit_boot<BIG=0>"]),
    # the pair offsets alone take 120 KB: the vertices come back into shared memory
    "d_global_x_shared_30000_pairs": dict(
        probs=lambda: [(ped10(30000), 0.7)], starts=32, boot=8, mi=(300, 100),
        pin=dict(n_warps=1, d_shared=0, x_global=0, big=0, wide=0, smem_boot_gather=0),
        kernels=["k_fit_starts<D_SHARED=0,X_GLOBAL=0,BIG=0>", "k_fit_boot<BIG=0>"]),
    # 100 random triples up to t = 127: per-lane state of one warp 112 bytes below the cap
    "tmax127_100_triples_one_warp": dict(
        probs=lambda: [(distinct_triples(100, seed=22), 0.6)], starts=64, boot=16, mi=(1000, 300),
        pin=dict(n_warps=1, d_shared=1, x_global=0, big=0, wide=0, smem_boot_gather=0, smem_fit=SMEM_CAP - 112),
        kernels=["k_fit_starts<D_SHARED=1,X_GLOBAL=0,BIG=0>", "k_fit_boot<BIG=0>"]),
    # the specialised kernels' limits (ABFIT_JIT=1 asks for them; jit_eligible still decides)
    "jit_1024_pairs": dict(
        probs=lambda: [(ped10(1024), 0.7)], starts=64, boot=24, mi=(2000, 300), env={"ABFIT_JIT": "1"},
        pin=dict(big=0, wide=0), n_lane=28,
        kernels=["abfit_jit_fit_starts", "abfit_jit_fit_boot_gather"], absent=["interpreter kernels"]),
    "jit_1025_pairs": dict(
        probs=lambda: [(ped10(1025), 0.7)], starts=64, boot=24, mi=(2000, 300), env={"ABFIT_JIT": "1"},
        pin=dict(big=0, wide=0), n_lane=28,
        kernels=["interpreter kernels: too many pairs", "k_fit_starts<", "k_fit_boot_gather:"], absent=["abfit_jit_"]),
    "jit_160_slots": dict(
        probs=lambda: [(lane_slots(23), 0.7)], starts=64, boot=24, mi=(1000, 300), env={"ABFIT_JIT": "1"},
        pin=dict(big=0, wide=0), n_lane=160,
        kernels=["abfit_jit_fit_starts", "abfit_jit_fit_boot_gather"], absent=["interpreter kernels"]),
    "jit_161_slots": dict(
        probs=lambda: [(lane_slots(24), 0.7)], starts=64, boot=24, mi=(1000, 300), env={"ABFIT_JIT": "1"},
        pin=dict(big=0, wide=0), n_lane=161,
        kernels=["interpreter kernels: too many per-lane values", "k_fit_starts<", "k_fit_boot_gather:"],
        absent=["abfit_jit_"]),
    # warp-per-fit at its shared-memory limit; the small pedigree of the batch runs on the same kernels
    "warp_per_fit_17000_triples_mixed": dict(
        probs=lambda: [_small(), (distinct_triples(17000), 0.7)], starts=32, boot=8, mi=(300, 100),
        pin=dict(big=1, wide=1, smem_wide=223456),
        kernels=["k_fit_wide<starts>", "k_fit_wide<boot>"], absent=["k_fit_starts<"]),
    # too large for warp-per-fit: lane-per-fit with everything in global scratch, for the small pedigree too
    "big_lane_per_fit_20000_triples_mixed": dict(
        probs=lambda: [_small(), (distinct_triples(20000), 0.7)], starts=32, boot=8, mi=(300, 100),
        pin=dict(big=1, wide=0, d_shared=0, x_global=1),
        kernels=["k_fit_starts<D_SHARED=0,X_GLOBAL=1,BIG=1>", "k_fit_boot<BIG=1>"], absent=["k_fit_wide"]),
}


def case_problems(ab, name):
    c = CASES[name]
    return [ab.Problem(p, u, u, 1.0) for p, u in c["probs"]()]


@pytest.mark.parametrize("name", list(CASES))
def test_planner_puts_each_case_where_it_claims(emul, ab, name):
    c = CASES[name]
    probs = case_problems(ab, name)
    rc, sh = emul_shape(emul, ab, probs, c["starts"])
    assert rc == 0, (name, rc)
    for k, v in c["pin"].items():
        assert sh[k] == v, (name, k, sh)
    if "n_lane" in c:
        assert emul_stats(emul, ab, probs[0])[1]["n_lane"] == c["n_lane"]
    assert sh["smem_fit"] <= SMEM_CAP and sh["smem_wide"] <= SMEM_CAP and sh["smem_boot_gather"] <= SMEM_CAP // 4


def test_planner_boundaries(emul, ab):
    """the thresholds the cases sit next to"""
    mk = lambda p: ab.Problem(p, 0.7, 0.7, 1.0)  # noqa: E731
    # index tile: 2000 pairs fit, the 10-triple pedigrees from 2400 pairs on do not
    assert emul_shape(emul, ab, [mk(ped10(2000))], 64)[1]["smem_boot_gather"] > 0
    assert emul_shape(emul, ab, [mk(ped10(2400))], 64)[1]["smem_boot_gather"] == 0
    # specialised kernels: limits of jit_eligible (JIT_MAX_PAIRS, JIT_MAX_SLOTS)
    assert [emul_stats(emul, ab, mk(lane_slots(m)))[1]["n_lane"] for m in (23, 24)] == [160, 161]
    # t <= 127: warp-per-fit up to ~17 700 distinct triples (per-warp tables), BIG lane-per-fit up to ~22 500 (the
    # program in shared memory), then refused
    shapes = [emul_shape(emul, ab, [mk(distinct_triples(k))], 1000) for k in (17700, 17800, 22500, 22600)]
    assert [rc for rc, _ in shapes] == [0, 0, 0, ab.ERR_TOO_LARGE]
    assert [(sh["big"], sh["wide"]) for _, sh in shapes[:3]] == [(1, 1), (1, 0), (1, 0)]


def test_too_large_refusals_on_the_host(emul, ab):
    """> ~22 500 triples: the program does not fit in shared memory (launch shape); n_lane >= 0xfff0: the
    pedigree compiler refuses before any shape is chosen"""
    p = ab.Problem(distinct_triples(26000), 0.7, 0.7, 1.0)
    assert emul_stats(emul, ab, p)[0] == 0 and emul_shape(emul, ab, [p], 32)[0] == -5
    q = ab.Problem(distinct_triples(66000), 0.7, 0.7, 1.0)
    assert emul_stats(emul, ab, q)[0] == -5 and emul_shape(emul, ab, [q], 32)[0] == -5


# ---------------------------------------------------------------------------------------------
# oracle (cached: the same inputs are checked against several kernel families)
# ---------------------------------------------------------------------------------------------
_cache = {}


def _key(*parts):
    h = hashlib.sha1()
    for x in parts:
        h.update(np.ascontiguousarray(x).tobytes() if isinstance(x, np.ndarray) else repr(x).encode())
    return h.hexdigest()


def oracle_fit(oracle, prob, sx, max_iters, sd_tol):
    k = _key("fit", prob.pedigree, prob.p0uu, prob.eqp, prob.eqp_weight, sx, max_iters, sd_tol)
    if k not in _cache:
        pb = oracle.Problem(prob.pedigree, prob.p0uu, prob.eqp, prob.eqp_weight)
        _cache[k] = oracle.ab_neutral(pb, sx, max_iters=max_iters, sd_tol=sd_tol,
                                      flags=oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, n_threads=NT)
    return _cache[k]


def oracle_boot(oracle, prob, theta, pred, resid, idx, vary, max_iters, sd_tol):
    k = _key("boot", prob.pedigree, prob.p0uu, prob.eqp, prob.eqp_weight, theta, pred, resid, idx, vary, max_iters, sd_tol)
    if k not in _cache:
        pb = oracle.Problem(prob.pedigree, prob.p0uu, prob.eqp, prob.eqp_weight)
        _cache[k] = oracle.boot_model(pb, theta, pred, resid, idx, vary, max_iters=max_iters, sd_tol=sd_tol,
                                      flags=oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, n_threads=NT)
    return _cache[k]


def same(a, b, fields, what):
    for f in fields:
        assert np.array_equal(a[f], b[f], equal_nan=True), (what, f, a[f], b[f])


def run_and_check(ab, ctx, oracle, probs, sx, n_boot, mi_fit, mi_boot, sd_tol=EPS, check=None):
    """fit_batch (every start record), boot_batch (rows and fits) and alphabeta_batch (the fused chain with the
    device-side analysis), all against the oracle; returns the fit result"""
    res = ctx.fit_batch(probs, sx, max_iters=mi_fit, sd_tol=sd_tol)
    check = range(len(probs)) if check is None else check
    offs = np.concatenate([[0], np.cumsum([p.n_pairs for p in probs])])
    good = []
    for i in check:
        o, n = offs[i], probs[i].n_pairs
        rc, best, allr, pred, resid = oracle_fit(oracle, probs[i], sx[i], mi_fit, sd_tol)
        same(res.all[i], allr, FIELDS, ("window", i))
        if rc == 0:
            assert res.status[i] == 0, i
            same(res.best[i], best, FIELDS, ("best", i))
            assert np.array_equal(res.pred[o:o + n], pred) and np.array_equal(res.resid[o:o + n], resid), i
            good.append(i)
        else:
            assert rc == oracle.ERR_NAN and res.status[i] == ab.ERR_NAN, i
    if not n_boot:
        return res
    idx = [ab.gen_resample_idx(SEED, i, n_boot, p.n_pairs) for i, p in enumerate(probs)]
    vary = np.stack([ab.gen_vary_vertices(SEED, i, n_boot, res.best[i]["theta"]) for i in range(len(probs))])
    idx_flat = np.concatenate([x.ravel() for x in idx])
    rows, fits = ctx.boot_batch(probs, res.best, res.pred, res.resid, idx_flat, vary, max_iters=mi_boot, sd_tol=sd_tol)
    out = ctx.alphabeta_batch(probs, sx, idx_flat, SEED, max_iters_fit=mi_fit, max_iters_boot=mi_boot, sd_tol=sd_tol)
    assert np.array_equal(out["status"], res.status)
    same(out["best"], res.best, FIELDS, "alphabeta best")
    assert np.array_equal(out["pred"], res.pred) and np.array_equal(out["resid"], res.resid)
    for i in good:
        o, n = offs[i], probs[i].n_pairs
        orc, orows, ofits = oracle_boot(oracle, probs[i], res.best[i]["theta"], res.pred[o:o + n], res.resid[o:o + n],
                                        idx[i], vary[i], mi_boot, sd_tol)
        assert orc == 0
        assert np.array_equal(rows[i], orows, equal_nan=True), ("rows", i)
        same(fits[i], ofits, BOOT_FIELDS, ("boot fits", i))
        assert np.array_equal(out["rows"][i], orows, equal_nan=True), ("alphabeta rows", i)
        assert np.array_equal(out["analysis"][i], oracle.analyze(orows), equal_nan=True), ("analysis", i)
    return res


def starts_for(ab, probs, n_starts):
    return np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p.pedigree[:, 3].max())) for i, p in enumerate(probs)])


def verbose_run(monkeypatch, capfd, env, fn):
    for k in ("ABFIT_DEV_NWARPS", "ABFIT_DEV_XGLOBAL", "ABFIT_DEV_BIG", "ABFIT_DEV_WIDE", "ABFIT_DEV_BOOT_XGLOBAL",
              "ABFIT_DEV_BOOT_TILE", "ABFIT_DEV_CHUNK", "ABFIT_JIT"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv("ABFIT_DEV_VERBOSE", "1")
    capfd.readouterr()
    r = fn()
    return r, capfd.readouterr().err


@pytest.fixture(autouse=True)
def _jit_cache(tmp_path, monkeypatch):
    monkeypatch.setenv("ABFIT_CACHE_DIR", str(tmp_path / "jit-cache"))


@pytest.mark.gpu
def test_device_shared_memory_is_what_the_pins_assume():
    import torch

    prop = torch.cuda.get_device_properties(0)
    assert prop.shared_memory_per_block_optin == SMEM_CAP
    assert prop.shared_memory_per_multiprocessor == 228 * 1024


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_launch_shape_against_oracle(ab, ctx, oracle, monkeypatch, capfd, name):
    c = CASES[name]
    probs = case_problems(ab, name)
    sx = starts_for(ab, probs, c["starts"])
    _, err = verbose_run(monkeypatch, capfd, c.get("env", {}),
                         lambda: run_and_check(ab, ctx, oracle, probs, sx, c["boot"], *c["mi"], check=c.get("check")))
    for k in c["kernels"]:
        assert k in err, (k, err)
    for k in c.get("absent", []):
        assert k not in err, (k, err)


@pytest.mark.gpu
@pytest.mark.parametrize("style", ["lineage", "sibling", "any"])
@pytest.mark.parametrize("family", ["interpreter", "specialised", "warp_per_fit", "big"])
def test_tmax127_programs_on_every_kernel(ab, ctx, oracle, monkeypatch, capfd, style, family):
    """the random time structures of the host-emulation tests (identity operands, G itself, stored powers, deferred
    d-vectors), at t up to 127, on the GPU"""
    rng = np.random.default_rng(["lineage", "sibling", "any"].index(style) + 127)

    def ped(n):
        p = random_pedigree(rng, n, 127, style)
        p[:, :3] = np.minimum(p[:, :3], 127)  # "sibling" steps up to two generations past tmax
        return p

    # 12 pairs: at most 160 per-lane values, so the specialised kernels take it (they take one program per batch);
    # 60 pairs: lane-per-fit interpreter kernels by default
    probs = [ab.Problem(ped(12), 0.75, 0.75, 1.0)]
    if family != "specialised":
        probs.append(ab.Problem(ped(60), 0.6, 0.6, 1.3))
    sx = starts_for(ab, probs, 40)
    env = FAMILY_ENV[family][0]
    names = {"interpreter": ["k_fit_starts<", "BIG=0>: ", "k_fit_boot<BIG=0>"],
             "specialised": ["abfit_jit_fit_starts", "abfit_jit_fit_boot_gather"],
             "warp_per_fit": ["k_fit_wide<starts>", "k_fit_wide<boot>"],
             "big": ["BIG=1>: ", "k_fit_boot<BIG=1>"]}[family]
    _, err = verbose_run(monkeypatch, capfd, env, lambda: run_and_check(ab, ctx, oracle, probs, sx, 12, 1500, 300))
    for k in names:
        assert k in err, (k, err)


@pytest.mark.gpu
def test_too_large_pedigrees_are_refused_without_a_launch(ab, ctx, oracle, monkeypatch, capfd):
    for ped in (distinct_triples(26000), distinct_triples(66000)):
        probs = [ab.Problem(ped, 0.7, 0.7, 1.0)]
        sx = starts_for(ab, probs, 4)
        with pytest.raises(ab.AbfitError) as e:
            verbose_run(monkeypatch, capfd, {}, lambda: ctx.fit_batch(probs, sx, max_iters=10))
        assert e.value.code == ab.ERR_TOO_LARGE
        assert "k_fit" not in capfd.readouterr().err
    # the context is still usable
    probs = [ab.Problem(ped10(300), 0.7, 0.7, 1.0)]
    run_and_check(ab, ctx, oracle, probs, starts_for(ab, probs, 40), 8, 2000, 300)


# ---------------------------------------------------------------------------------------------
# optimiser and selection edges
# ---------------------------------------------------------------------------------------------
SD_TOLS = [0.0, -1.0, float("nan"), float("inf"), 1e-300, 5e-324, 1e-3, 1e200]
MAX_ITERS = [0, 1, 2, 7]
SETTINGS = [(EPS, 300)] + [(s, 300) for s in SD_TOLS] + [(EPS, m) for m in MAX_ITERS]
SETTING_IDS = ["default"] + [f"sd_tol={s!r}" for s in SD_TOLS] + [f"max_iters={m}" for m in MAX_ITERS]
TIES = (3, 35, 40, 257)  # lanes 3, 3, 8, 1; rounds 0, 1, 1, 8 of a one-warp block; different warps / items otherwise
N_EDGE = 264
NAN_STARTS = (5, 40, 41)

# ABFIT_JIT=0: once the specialised kernels of a program are loaded (or cached on disk) the library uses them for
# every later batch of that program, so the interpreter families ask for the interpreter
FAMILY_ENV = {
    "interpreter": ({"ABFIT_JIT": "0"}, ["k_fit_starts<", "BIG=0>", "k_fit_boot_gather:"]),
    "specialised": ({"ABFIT_JIT": "1"}, ["abfit_jit_fit_starts", "abfit_jit_fit_boot_gather"]),
    "big": ({"ABFIT_JIT": "0", "ABFIT_DEV_BIG": "1", "ABFIT_DEV_WIDE": "0"}, ["BIG=1>: ", "k_fit_boot<BIG=1>"]),
    "warp_per_fit": ({"ABFIT_JIT": "0", "ABFIT_DEV_WIDE": "1"}, ["k_fit_wide<starts>", "k_fit_wide<boot>"]),
    "stored_dstar": ({"ABFIT_JIT": "0", "ABFIT_DEV_BOOT_TILE": "1"}, ["k_fit_starts<", "k_fit_boot<BIG=0>"]),
}


def edge_windows(ab, oracle):
    """six windows on one time structure (one pedigree program, so the specialised kernels take the batch too):
    0 plain starts with a tied best at TIES; 1, 2 penalty weights -1e308 (every cost -inf) and -1e300 (some);
    3 degenerate simplices and +-inf / NaN vertices behind a finite vertex 0; 4 NaN vertex 0 at NAN_STARTS only;
    5 NaN vertex 0 everywhere"""
    if "edge" in _cache:
        return _cache["edge"]
    ped = ped351()
    u = 0.8
    probs = [ab.Problem(ped, u, u, 1.0), ab.Problem(ped, u, 0.7, -1e308), ab.Problem(ped, u, 0.7, -1e300),
             ab.Problem(ped, u, u, 1.0), ab.Problem(ped, u, u, 1.0), ab.Problem(ped, 0.7, 0.7, 1.0)]
    sx = starts_for(ab, probs, N_EDGE).copy()
    # ties: copies of window 0's best simplex; its own slot gets the worst one
    rc, best, allr, _, _ = oracle_fit(oracle, probs[0], sx[0], 300, EPS)
    assert rc == 0
    b, w = int(best["start_id"]), int(np.argmax(allr["lse"]))
    orig = sx[0].copy()
    for t in TIES:
        sx[0, t] = orig[b]
    if b not in TIES:
        sx[0, b] = orig[w]
    s3 = sx[3]
    for k in range(N_EDGE):
        kind = k % 5
        if kind == 0:
            s3[k, 1:] = s3[k, 0]  # five identical vertices
        elif kind == 1:
            s3[k, 2, 0] = np.inf
        elif kind == 2:
            s3[k, 3, 2] = -np.inf
        elif kind == 3:
            s3[k, 4] = np.nan
        else:
            s3[k, 1, 1] = -np.inf
            s3[k, 4, 0] = np.inf
    for k in NAN_STARTS:
        sx[4, k, 0, 0:2] = 0.0 if k != 41 else [np.inf, 1e-3]  # alpha = beta = 0 -> 0/0; alpha = inf
    sx[5, :, 0, 0:2] = 0.0
    _cache["edge"] = (probs, sx)
    return probs, sx


@pytest.mark.gpu
@pytest.mark.parametrize("setting", SETTINGS, ids=SETTING_IDS)
@pytest.mark.parametrize("family", list(FAMILY_ENV))
def test_optimiser_edges_on_every_kernel_family(ab, ctx, oracle, monkeypatch, capfd, family, setting):
    sd_tol, mi = setting
    probs, sx = edge_windows(ab, oracle)
    env, names = FAMILY_ENV[family]
    res, err = verbose_run(monkeypatch, capfd, env, lambda: run_and_check(ab, ctx, oracle, probs, sx, 16, mi, mi, sd_tol))
    for k in names:
        assert k in err, (k, err)
    assert [int(s) for s in res.status] == [0, 0, 0, 0, ab.ERR_NAN, ab.ERR_NAN]
    if setting == (EPS, 300):
        assert res.best[0]["start_id"] == TIES[0]
        assert len({res.all[0][t]["lse"] for t in TIES}) == 1
        assert np.all(res.all[1]["status"] == ab.TERM_TARGET_COST)
        assert np.any(res.all[2]["status"] == ab.TERM_TARGET_COST)
    if sd_tol == EPS:  # the -inf stop comes after the sd and max_iters tests, never before
        assert np.all(res.all[1]["iters"] == 0) and np.all(res.all[1]["evals"] == 5)
    ok = np.setdiff1d(np.arange(N_EDGE), NAN_STARTS)
    assert np.all(res.all[4]["status"][list(NAN_STARTS)] == ab.FIT_NAN) and np.all(res.all[4]["status"][ok] >= 0)
    assert np.all(res.all[5]["status"] == ab.FIT_NAN) and res.best[5]["status"] == ab.FIT_NAN
    assert np.array_equal(res.all[5]["theta"], sx[5][:, 0], equal_nan=True) and np.all(np.isnan(res.all[5]["cost"]))


# ---- the same edges through the device headers built for the CPU ------------------------------
def emul_run(emul, ab, prob, sx, max_iters, sd_tol, dstar=None, wide=False):
    arr = ab._pack_problems([prob])
    sx = np.ascontiguousarray(sx, dtype=np.float64)
    n = sx.size // 20
    out = np.zeros(n, dtype=ab.FIT_DTYPE)
    dp = None if dstar is None else np.ascontiguousarray(dstar, dtype=np.float64).ctypes.data_as(C.c_void_p)
    rc = (emul.emul_fit_wide if wide else emul.emul_fit)(arr, sx.ctypes.data_as(C.c_void_p), n, dp, max_iters,
                                                         C.c_double(sd_tol), 0, out.ctypes.data_as(C.c_void_p))
    assert rc == 0, rc
    return out


CPU_STARTS = {1: range(6), 2: range(6), 3: range(10), 4: (0, 1) + NAN_STARTS, 5: (0, 1)}


@pytest.mark.parametrize("wide", [False, True], ids=["lane", "warp"])
@pytest.mark.parametrize("setting", SETTINGS, ids=SETTING_IDS)
def test_optimiser_edges_through_the_device_headers(emul, ab, oracle, setting, wide):
    """the Nelder-Mead state machine of abfit_nm.cuh as every fit kernel drives it, against abref_nelder_mead"""
    sd_tol, mi = setting
    probs, sx = edge_windows(ab, oracle)
    for w, starts in CPU_STARTS.items():
        pb = oracle.Problem(probs[w].pedigree, probs[w].p0uu, probs[w].eqp, probs[w].eqp_weight)
        sel = sx[w][list(starts)]
        g = emul_run(emul, ab, probs[w], sel, mi, sd_tol, wide=wide)
        for j in range(len(sel)):
            o = oracle.nelder_mead(pb, sel[j], max_iters=mi, sd_tol=sd_tol,
                                   flags=oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL)
            same(g[j], o, ("theta", "cost", "iters", "evals", "status"), (w, starts[j]))
        if w == 1 and sd_tol == EPS:  # every cost -inf: stopped before the first iteration (max_iters = 0 first)
            assert np.all(g["status"] == (ab.TERM_TARGET_COST if mi > 0 else ab.TERM_MAX_ITERS))
            assert np.all(g["iters"] == 0) and np.all(g["evals"] == 5)
        if w == 5:
            assert np.all(g["status"] == ab.FIT_NAN) and np.array_equal(g["theta"], sel[:, 0], equal_nan=True)


@pytest.mark.parametrize("weight", [-1e308, -1e300])
def test_minus_inf_costs_in_the_bootstrap_through_the_device_headers(emul, ab, oracle, weight):
    ped = ped351()
    u = 0.8
    plain = ab.Problem(ped, u, u, 1.0)
    sx = starts_for(ab, [plain], 16)[0]
    rc, best, _, pred, resid = oracle_fit(oracle, plain, sx, 2000, EPS)
    assert rc == 0
    n_boot = 10
    idx = ab.gen_resample_idx(SEED, 0, n_boot, len(ped))
    vary = ab.gen_vary_vertices(SEED, 0, n_boot, best["theta"])
    simplices = np.concatenate([np.broadcast_to(best["theta"], (n_boot, 1, 4)), vary], axis=1)
    prob = ab.Problem(ped, u, 0.7, weight)
    orc, rows, ofits = oracle.boot_model(oracle.Problem(ped, u, 0.7, weight), best["theta"], pred, resid, idx, vary,
                                         max_iters=300, flags=oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL)
    assert orc == 0 and np.any(ofits["status"] == ab.TERM_TARGET_COST)
    for wide in (False, True):
        g = emul_run(emul, ab, prob, simplices, 300, EPS, dstar=pred[None, :] + resid[idx], wide=wide)
        same(g, ofits, ("theta", "cost", "iters", "evals", "status"), ("boot", wide))


def test_oracle_nan_record_is_vertex_zero(oracle):
    """a start whose vertex 0 costs NaN: the oracle reports that vertex with a NaN cost, as the kernels do"""
    pb = oracle.Problem(ped351(), 0.8, 0.8, 1.0)
    sx = np.array([[0.0, 0.0, 0.05, 0.01], [1e-4, 1e-4, 0.05, 0.01], [2e-4, 1e-4, 0.05, 0.01], [1e-4, 3e-4, 0.04, 0.01],
                   [1e-4, 1e-4, 0.05, 0.02]])
    f = oracle.nelder_mead(pb, sx, max_iters=50)
    assert f["status"] == oracle.ERR_NAN and np.array_equal(f["theta"], sx[0]) and np.isnan(f["cost"])
