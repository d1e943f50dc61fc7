"""Parity tests proper: the CUDA path, called through the C ABI, against the CPU oracle on the
same seeded inputs.  Integer / index work and — because the kernels keep the reference's
operation order — all f64 results are compared BIT FOR BIT; the north-star tolerances
(divergence 1e-12, RSS 1e-9, alpha/beta 1e-6 relative) are asserted as well."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, resolve_golden

pytestmark = pytest.mark.gpu

SEED = 0xAB0B200


def rel(a, b):
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))


@pytest.fixture(scope="module")
def ped351(oracle):
    return oracle.load_pedigree_file(os.path.join(GOLDEN, "pedigree.txt"))


@pytest.fixture(scope="module")
def ped78(oracle):
    ped, p0uu, _ = oracle.build_pedigree(os.path.join(GOLDEN, "desired_output", "nodelist.fn"),
                                         os.path.join(GOLDEN, "desired_output", "edgelist.fn"), 0.99, resolve_golden)
    return ped, p0uu


def synth_problem(rng, ped_shape, n_keep=None):
    """C4-style synthetic window: D = c + dt(alpha,beta,w) + noise on the time structure of a real pedigree"""
    from oracle import abref_py as o

    ped = ped_shape.copy()
    if n_keep:
        ped = ped[np.sort(rng.choice(len(ped), n_keep, replace=False))]
    a, b = 10 ** rng.uniform(-5, -3.3), 10 ** rng.uniform(-4, -2.3)
    w, c = rng.uniform(0, 0.1), rng.uniform(0, 0.005)
    p0uu = rng.uniform(0.6, 0.95)
    pb = o.Problem(ped, p0uu, p0uu, 1.0)
    dt, _ = o.divergence(pb, a, b, w, o.FAST_DIVERGENCE)
    ped[:, 3] = np.maximum(c + dt + rng.normal(0, 5e-4, len(ped)), 0.0)
    return ped, p0uu


# ---------------------------------------------------------------------------------------------
# objective
# ---------------------------------------------------------------------------------------------
def test_cost_kat_exact(ab, ctx, ped351):
    """src/structs.rs:233 through the GPU"""
    pb = ab.Problem(ped351, 0.75, 0.5, 0.7)
    assert pb.cost([0.0001179555, 0.0001180614, 0.03693534, 0.003023981], ctx) == 0.0006700888539608879


def test_divergence_same_as_r(ab, ctx, oracle, ped351):
    """src/divergence.rs:139-161 through the GPU; and == oracle bit for bit"""
    r = np.array([float(x) for x in open(os.path.join(GOLDEN, "divergence.txt")).read().split("\n")])
    dt, puu = ctx.divergence(ab.Problem(ped351, 0.75, 0.5, 0.7), [3.974271e-09, 1.519045e-07, 0.06892953, 0.0])
    assert np.max(np.abs(dt - r)) <= 1e-4 and rel(dt, r) < 1e-12
    want, want_puu = oracle.divergence(oracle.Problem(ped351, 0.75, 0.5, 0.7), 3.974271e-09, 1.519045e-07, 0.06892953)
    assert np.array_equal(dt, want) and puu == want_puu


def test_cost_batch_matches_oracle_bitwise(ab, ctx, oracle, ped351, ped78):
    rng = np.random.default_rng(1)
    peds = [(ped351, 0.75), ped78, (np.loadtxt(os.path.join(GOLDEN, "pedigree_generated.txt"), skiprows=1), 0.655)]
    probs = [ab.Problem(p, u, u, 1.0) for p, u in peds]
    oprobs = [oracle.Problem(p, u, u, 1.0) for p, u in peds]
    B = 301  # ragged: not a multiple of 32, interleaved problems
    pot = rng.integers(0, 3, B).astype(np.int32)
    theta = np.stack([10 ** rng.uniform(-9, -2, B), 10 ** rng.uniform(-9, -2, B), rng.uniform(0, 0.1, B),
                      rng.uniform(0, 0.02, B)], axis=1)
    theta[5] = [-1e-4, 2e-3, -0.3, 0.01]  # the reference has no bounds: negative parameters are legal
    theta[6] = [0.0, 0.0, 0.0, 0.0]       # alpha + beta = 0 -> 0/0 in p_uu_est -> NaN cost
    cost, lse = ctx.cost_batch(probs, theta, pot)
    for i in range(B):
        wc = oracle.cost(oprobs[pot[i]], theta[i])
        wl = oracle.lse(oprobs[pot[i]], theta[i])
        assert (cost[i] == wc) or (np.isnan(cost[i]) and np.isnan(wc)), i
        assert lse[i] == wl, i
    assert np.isnan(cost[6]) and np.isfinite(lse[6])


def test_time_validation(ab, ctx):
    ped = np.array([[2.0, 1.0, 3.0, 0.1]])  # t1 < t0: the reference would take the matrix-inverse path
    with pytest.raises(ab.AbfitError) as e:
        ctx.cost_batch([ab.Problem(ped, 0.7, 0.7, 1.0)], np.zeros((1, 4)))
    assert e.value.code == ab.ERR_TIME
    # `as i8` truncation (src/divergence.rs:52): 3.9 -> 3
    ped2 = np.array([[0.0, 3.9, 5.2, 0.1], [0.0, 3.0, 5.0, 0.1]])
    c, _ = ctx.cost_batch([ab.Problem(ped2[:1], 0.7, 0.7, 1.0), ab.Problem(ped2[1:], 0.7, 0.7, 1.0)],
                          np.array([[1e-4, 1e-3, 0.05, 0.0]] * 2), np.array([0, 1], dtype=np.int32))
    assert c[0] == c[1]


# ---------------------------------------------------------------------------------------------
# multi-start fit
# ---------------------------------------------------------------------------------------------
def check_fit_against_oracle(ab, oracle, res, p, pb_o, sx, max_iters, flags_o, off, n):
    rc, best, allr, pred, resid = oracle.ab_neutral(pb_o, sx, max_iters=max_iters, flags=flags_o, n_threads=8)
    assert rc == 0
    g = res.all[p]
    for f in ("theta", "cost", "lse", "iters", "evals", "status", "start_id"):
        assert np.array_equal(g[f], allr[f]), f
    gb = res.best[p]
    assert gb["start_id"] == best["start_id"] and np.array_equal(gb["theta"], best["theta"])
    assert np.array_equal(res.pred[off:off + n], pred) and np.array_equal(res.resid[off:off + n], resid)
    # north-star tolerances (implied by the above)
    assert abs(gb["lse"] - best["lse"]) <= 1e-9 * best["lse"]
    assert rel(gb["theta"][:2], best["theta"][:2]) <= 1e-6


def test_fit_c1_real_pedigrees_bitwise(ab, ctx, oracle, ped78):
    """C1: data/nodelist.txt (N=6) and desired_output (N=78) fits, all starts bit-identical to the oracle"""
    ped6, p6, _ = oracle.build_pedigree(os.path.join(GOLDEN, "nodelist.txt"), os.path.join(GOLDEN, "edgelist.txt"), 0.99,
                                        resolve_golden)
    cases = [(ped6, p6), ped78]
    n_starts = 100
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    res = ctx.fit_batch(probs, sx, max_iters=10000)
    assert np.all(res.status == 0)
    off = 0
    for i, (p, u) in enumerate(cases):
        check_fit_against_oracle(ab, oracle, res, i, oracle.Problem(p, u, u, 1.0), sx[i], 10000,
                                 oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, off, len(p))
        off += len(p)
    # R original within 10 % (src/macros.rs:25-34)
    assert abs(res.best[1]["theta"][0] - 5.7985750419976e-05) < 0.1 * 5.7985750419976e-05
    assert abs(res.best[1]["theta"][1] - 0.00655710970515347) < 0.1 * 0.00655710970515347


def test_c1_c2_default_counts_bitwise(ab, ctx, oracle, ped78):
    """BASELINE configs[0..1] at their own sizes: the repo's example pedigree (6 pairs) and the desired_output one
    (78 pairs), 1000 starts (the `alphabeta` default, src/arguments.rs:98-99) and 1000 bootstrap replicates, every
    start and every replicate bit-identical to the oracle"""
    ped6, p6, _ = oracle.build_pedigree(os.path.join(GOLDEN, "nodelist.txt"), os.path.join(GOLDEN, "edgelist.txt"), 0.99,
                                        resolve_golden)
    cases = [(ped6, p6), ped78]
    n_starts = n_boot = 1000
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    idx = np.concatenate([ab.gen_resample_idx(SEED, i, n_boot, len(p)).ravel() for i, (p, u) in enumerate(cases)])
    out = ctx.alphabeta_batch(probs, sx, idx, SEED)
    res = ctx.fit_batch(probs, sx, max_iters=10000)
    assert np.all(res.status == 0) and np.array_equal(out["best"]["theta"], res.best["theta"])
    flags = oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL
    off = 0
    for i, (p, u) in enumerate(cases):
        n = len(p)
        check_fit_against_oracle(ab, oracle, res, i, oracle.Problem(p, u, u, 1.0), sx[i], 10000, flags, off, n)
        vary = ab.gen_vary_vertices(SEED, i, n_boot, res.best[i]["theta"])
        rc, orows, _ = oracle.boot_model(oracle.Problem(p, u, u, 1.0), res.best[i]["theta"], res.pred[off:off + n],
                                         res.resid[off:off + n], idx[off * n_boot:(off + n) * n_boot].reshape(n_boot, n),
                                         vary, max_iters=1000, flags=flags, n_threads=8)
        assert rc == 0 and np.array_equal(out["rows"][i], orows)
        assert np.array_equal(out["analysis"][i], oracle.analyze(orows), equal_nan=True)
        off += n
    # R original within 10 % (src/macros.rs:25-34)
    assert abs(res.best[1]["theta"][0] - 5.7985750419976e-05) < 0.1 * 5.7985750419976e-05
    assert abs(res.best[1]["theta"][1] - 0.00655710970515347) < 0.1 * 0.00655710970515347


@pytest.mark.parametrize("n_starts,n_boot", [(1, 1), (33, 31), (97, 100), (257, 7)])
def test_ragged_start_and_replicate_counts(ab, ctx, oracle, ped78, ped351, n_starts, n_boot):
    """start / replicate counts that do not fill warps, queues or hand-off groups evenly; three different pedigrees
    in one batch; every start and every bootstrap row bit-identical to the oracle"""
    rng = np.random.default_rng(100 * n_starts + n_boot)
    cases = [ped78, synth_problem(rng, ped351), synth_problem(rng, ped351, n_keep=37)]
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    res = ctx.fit_batch(probs, sx, max_iters=10000)
    idx = np.concatenate([ab.gen_resample_idx(SEED, i, n_boot, len(p)).ravel() for i, (p, u) in enumerate(cases)])
    vary = np.stack([ab.gen_vary_vertices(SEED, i, n_boot, res.best[i]["theta"]) for i in range(len(cases))])
    rows, fits = ctx.boot_batch(probs, res.best, res.pred, res.resid, idx, vary, max_iters=1000)
    off = 0
    flags = oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL
    for i, (p, u) in enumerate(cases):
        n = len(p)
        check_fit_against_oracle(ab, oracle, res, i, oracle.Problem(p, u, u, 1.0), sx[i], 10000, flags, off, n)
        rc, orows, ofits = oracle.boot_model(oracle.Problem(p, u, u, 1.0), res.best[i]["theta"], res.pred[off:off + n],
                                             res.resid[off:off + n], idx[off * n_boot:(off + n) * n_boot].reshape(n_boot, n),
                                             vary[i], max_iters=1000, flags=flags, n_threads=8)
        assert rc == 0 and np.array_equal(rows[i], orows)
        assert np.array_equal(fits[i]["evals"], ofits["evals"])
        off += n


def test_fit_synthetic_windows_bitwise(ab, ctx, oracle, ped351):
    """C4-shaped windows (N=351, U=10, Tmax=32) + ragged ones; every start of every window bit-identical"""
    rng = np.random.default_rng(42)
    cases = [synth_problem(rng, ped351) for _ in range(3)] + [synth_problem(rng, ped351, n_keep=k) for k in (1, 33, 200)]
    n_starts = 70  # not a multiple of 32
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    res = ctx.fit_batch(probs, sx, max_iters=10000)
    off = 0
    stalled = 0
    for i, (p, u) in enumerate(cases):
        check_fit_against_oracle(ab, oracle, res, i, oracle.Problem(p, u, u, 1.0), sx[i], 10000,
                                 oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, off, len(p))
        off += len(p)
        stalled += int(np.sum(res.all[i]["status"] == ab.TERM_STALLED))
    assert stalled > 0  # the argmin-0.8.1 stall case is exercised


def test_fit_flag_variants_bitwise(ab, ctx, oracle, ped351):
    """no-early-exit (burn max_iters like the reference) and shrink-on-failed-contraction"""
    rng = np.random.default_rng(3)
    p, u = synth_problem(rng, ped351, n_keep=60)
    sx = ab.gen_start_simplices(SEED, 77, 40, float(p[:, 3].max()))
    for fl_g, fl_o, mi in ((ab.NO_EARLY_EXIT_ON_STALL, 0, 600),
                           (ab.SHRINK_ON_FAILED_CONTRACTION, oracle.SHRINK_ON_FAILED_CONTRACTION, 10000)):
        res = ctx.fit_batch([ab.Problem(p, u, u, 1.0)], sx[None], max_iters=mi, flags=fl_g)
        check_fit_against_oracle(ab, oracle, res, 0, oracle.Problem(p, u, u, 1.0), sx, mi,
                                 fl_o | oracle.FAST_DIVERGENCE, 0, len(p))


def test_fit_nan_window_is_flagged(ab, ctx, oracle, ped351):
    """empty window -> NaN divergence: the reference panics (src/ab_neutral.rs:28); we flag that window only"""
    rng = np.random.default_rng(5)
    good, u = synth_problem(rng, ped351, n_keep=20)
    bad = good.copy()
    bad[3, 3] = np.nan
    sx = np.stack([ab.gen_start_simplices(SEED, i, 32, 0.02) for i in range(2)])
    res = ctx.fit_batch([ab.Problem(bad, u, u, 1.0), ab.Problem(good, u, u, 1.0)], sx)
    assert res.status[0] == ab.ERR_NAN and res.status[1] == 0
    assert res.best[0]["status"] == ab.FIT_NAN and np.isfinite(res.best[1]["lse"])


# ---------------------------------------------------------------------------------------------
# bootstrap
# ---------------------------------------------------------------------------------------------
def test_boot_c2_bitwise(ab, ctx, oracle, ped78, ped351):
    """C2: boot_model on the real 78-pair pedigree and a synthetic 351-pair window; rows bit-identical"""
    rng = np.random.default_rng(8)
    cases = [ped78, synth_problem(rng, ped351)]
    n_starts, n_boot = 64, 75
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    res = ctx.fit_batch(probs, sx)
    idx = np.concatenate([ab.gen_resample_idx(SEED, i, n_boot, len(p)).ravel() for i, (p, u) in enumerate(cases)])
    vary = np.stack([ab.gen_vary_vertices(SEED, i, n_boot, res.best[i]["theta"]) for i in range(len(cases))])
    rows, fits = ctx.boot_batch(probs, res.best, res.pred, res.resid, idx, vary, max_iters=1000)
    off = 0
    for i, (p, u) in enumerate(cases):
        n = len(p)
        rc, orows, ofits = oracle.boot_model(oracle.Problem(p, u, u, 1.0), res.best[i]["theta"], res.pred[off:off + n],
                                             res.resid[off:off + n], idx[off * n_boot:(off + n) * n_boot].reshape(n_boot, n),
                                             vary[i], max_iters=1000,
                                             flags=oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, n_threads=8)
        assert rc == 0
        assert np.array_equal(rows[i], orows)
        for f in ("theta", "cost", "iters", "evals", "status"):
            assert np.array_equal(fits[i][f], ofits[f]), f
        assert np.array_equal(ab.analyze(rows[i]), oracle.analyze(orows))
        off += n


def test_staged_batch_equals_one_shot(ab, ctx, ped351):
    """upload / run / download (device-resident) gives the same bytes as the host-buffer calls"""
    rng = np.random.default_rng(13)
    cases = [synth_problem(rng, ped351, n_keep=50) for _ in range(4)]
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    sx = np.stack([ab.gen_start_simplices(SEED, i, 48, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    one = ctx.fit_batch(probs, sx)
    b = ctx.batch(probs)
    b.upload_starts(sx)
    b.run_fit()
    st = b.download_fit(want_all=True)
    assert st.best.tobytes() == one.best.tobytes() and st.all.tobytes() == one.all.tobytes()
    assert np.array_equal(st.pred, one.pred) and np.array_equal(st.resid, one.resid)
    n_boot = 40
    idx = np.concatenate([ab.gen_resample_idx(SEED, i, n_boot, 50).ravel() for i in range(4)])
    vary = np.stack([ab.gen_vary_vertices(SEED, i, n_boot, one.best[i]["theta"]) for i in range(4)])
    rows1, _ = ctx.boot_batch(probs, one.best, one.pred, one.resid, idx, vary)
    b.upload_boot(idx, vary)  # best / pred / resid stay on the device
    b.run_boot()
    rows2, _ = b.download_boot()
    assert np.array_equal(rows1, rows2)
    t = b.timing()
    assert t["fit_ms"] > 0 and t["boot_ms"] > 0 and t["launches"] == 3
    assert t["evals_fit"] == int(one.all["evals"].sum())
    b.close()


# ---------------------------------------------------------------------------------------------
# observed divergence
# ---------------------------------------------------------------------------------------------
def test_dmatrix_real_files_exact(ab, ctx, oracle):
    """C1 inputs: D, integer sums, valid-site counts and p0uu bit-exact (data/pedigree_generated.txt)"""
    _, p0, info = oracle.build_pedigree(os.path.join(GOLDEN, "nodelist.txt"), os.path.join(GOLDEN, "edgelist.txt"), 0.99,
                                        resolve_golden)
    out = ctx.dmatrix(info["status"], info["post"], info["meth"], 0.99)
    want = np.loadtxt(os.path.join(GOLDEN, "pedigree_generated.txt"), skiprows=1)[:, 3]
    assert np.array_equal(out["D"][0], want)
    assert [int(x) for x in out["diff"][0]] == [54, 240, 3, 169, 50, 269]
    assert [int(x) for x in out["cnt"][0]] == [247, 260, 276, 333, 271, 295]
    assert list(out["nvalid"][0]) == [309, 378, 428, 346]
    assert out["p0uu"][0] == p0


def synth_methylomes(rng, S, L):
    status = rng.choice(np.array([0, 1, 2], dtype=np.uint8), size=(S, L), p=[0.75, 0.05, 0.20])
    post = np.where(rng.random((S, L)) < 0.9, 0.9999, rng.uniform(0.5, 0.99, (S, L)))
    meth = np.clip(status / 2.0 + rng.normal(0, 0.05, (S, L)), 0, 1)
    return status, post, meth


def test_dmatrix_windows_exact(ab, ctx, oracle):
    """windowed variant: ragged and EMPTY segments, tails that are not multiples of 64"""
    rng = np.random.default_rng(21)
    S, L = 9, 5000
    status, post, meth = synth_methylomes(rng, S, L)
    seg = np.array([0, 1, 1, 64, 129, 700, 700, 4097, 5000], dtype=np.int64)
    out = ctx.dmatrix(status, post, meth, 0.99, seg)
    for w in range(len(seg) - 1):
        a, b = seg[w], seg[w + 1]
        D, diff, cnt = oracle.dmatrix(status[:, a:b], post[:, a:b], 0.99)
        assert np.array_equal(out["diff"][w], diff) and np.array_equal(out["cnt"][w], cnt)
        assert np.array_equal(out["D"][w], D, equal_nan=True)
        if b > a:
            p0, rc, nv = oracle.p0uu(post[:, a:b], meth[:, a:b], 0.99)
            assert np.array_equal(out["nvalid"][w], nv)
            assert (out["p0uu"][w] == p0) or (np.isnan(p0) and np.isnan(out["p0uu"][w]))


def test_dmatrix_large_blocked(ab, ctx, oracle):
    """a window longer than 65536 sites uses the blocked tree for methsum: integers exact, p0uu 1e-12"""
    rng = np.random.default_rng(22)
    S, L = 6, 300_001
    status, post, meth = synth_methylomes(rng, S, L)
    out = ctx.dmatrix(status, post, meth, 0.99)
    D, diff, cnt = oracle.dmatrix(status, post, 0.99)
    assert np.array_equal(out["diff"][0], diff) and np.array_equal(out["cnt"][0], cnt) and np.array_equal(out["D"][0], D)
    p0, rc, nv = oracle.p0uu(post, meth, 0.99)
    assert np.array_equal(out["nvalid"][0], nv)
    assert abs(out["p0uu"][0] - p0) <= 1e-12 * abs(p0)
    # sharding the site axis (one shard per GPU) and adding the integer partials is exact
    cut = 123_457
    a = ctx.dmatrix(status[:, :cut], post[:, :cut], meth[:, :cut], 0.99)
    b = ctx.dmatrix(status[:, cut:], post[:, cut:], meth[:, cut:], 0.99)
    assert np.array_equal(a["diff"] + b["diff"], out["diff"]) and np.array_equal(a["cnt"] + b["cnt"], out["cnt"])
    assert np.array_equal(a["nvalid"] + b["nvalid"], out["nvalid"])


@pytest.mark.parametrize("S,L,segs", [(2, 130, None), (3, 64, None), (5, 1, None), (210, 40_000, None),
                                      (37, 5_000, [0, 0, 63, 64, 700, 700, 4_999, 5_000]),
                                      (5, 2_600_000, [0, 1_300_000, 2_600_000])])
def test_dmatrix_pair_tiles_shapes(ab, ctx, oracle, S, L, segs):
    """the register-tiled pair pass: sample counts that are not multiples of the 4 x 4 tile, more tiles than one
    pass of the block covers (210 samples -> 1431 tiles), items of several hundred words that flush their packed
    counters, windows of 0 / 1 / 63 / 64 sites"""
    rng = np.random.default_rng(1000 * S + L)
    status, post, meth = synth_methylomes(rng, S, L)
    if segs is None:
        out = ctx.dmatrix(status, post, meth, 0.99)
        D, diff, cnt = oracle.dmatrix(status, post, 0.99)
        assert np.array_equal(out["diff"][0], diff) and np.array_equal(out["cnt"][0], cnt)
        assert np.array_equal(out["D"][0], D, equal_nan=True)
    else:
        out = ctx.dmatrix(status, post, meth, 0.99, seg_offsets=segs)
        for w in range(len(segs) - 1):
            a, b = segs[w], segs[w + 1]
            D, diff, cnt = oracle.dmatrix(status[:, a:b], post[:, a:b], 0.99)
            assert np.array_equal(out["diff"][w], diff) and np.array_equal(out["cnt"][w], cnt), w
            assert np.array_equal(out["D"][w], D, equal_nan=True), w


# ---------------------------------------------------------------------------------------------
# C3: metaprofile windows -> observed divergence per window -> fit, all windows in one batch
# ---------------------------------------------------------------------------------------------
def test_metaprofile_chain_windows_to_fits(ab, ctx, oracle):
    """data/methylome (4 samples x 500 CG sites, bp 6-1807 of chr 1-5, C, M) with a synthetic annotation whose genes
    overlap those sites (the shipped annotation.bed starts at bp 23 121, so every real window is empty —
    see test_windows.py).  Site -> window placement (host), per-window pairwise divergence + p0uu
    (abfit_divergence with segment offsets) and the multi-start fits of all non-empty windows in ONE batch,
    against the oracle doing the reference's per-window loop (src/cli/metaprofile.rs:50-72)."""
    ped6, p6, info = oracle.build_pedigree(os.path.join(GOLDEN, "nodelist.txt"), os.path.join(GOLDEN, "edgelist.txt"), 0.99,
                                           resolve_golden)
    status, post, meth = info["status"], info["post"], info["meth"]
    S, L = status.shape
    # the four files list the same CG positions: read them once for the placement
    sites = []
    for line in open(os.path.join(GOLDEN, "methylome", "G0.txt")).read().split("\n")[1:]:
        s = oracle.parse_methylome_line(line)
        if s is not None:
            sites.append((oracle.chromosome_id(str(s["chromosome"])), s["start"], s["end"],
                          {"+": 1, "-": -1, "*": 0}[s["strand"]]))
    assert len(sites) == L
    genes = [(1, 300, 700, -1), (1, 250, 800, 1), (2, 1200, 1600, 1), (2, 1250, 1650, -1), (3, 600, 900, 0),
             (4, 1200, 1550, -1), (4, 1150, 1600, 1), (5, 300, 900, 0), (257, 200, 900, 1), (257, 150, 950, -1),
             (256, 200, 600, -1), (256, 150, 650, 1)]  # overlapping genes, both strands, unknown strand, chr C and M
    kw = dict(window_size=10, window_step=5, cutoff=200, max_gene_length=100, absolute=False)
    dist, asite, awin = ab.place_sites(genes, sites, **kw)
    want_dist, want_assign = oracle.extract_windows(genes, sites, **kw)
    assert dist.tolist() == want_dist and list(zip(asite.tolist(), awin.tolist())) == want_assign
    n_win = len(dist)
    order, seg = ab.segments_from_assignments(asite, awin, n_win)
    assert np.array_equal(np.diff(seg), dist)
    out = ctx.dmatrix(status[:, order], post[:, order], meth[:, order], 0.99, seg_offsets=seg)

    keep, probs, oprobs = [], [], []
    for w in range(n_win):
        cols = order[seg[w]:seg[w + 1]]
        D, diff, cnt = oracle.dmatrix(status[:, cols], post[:, cols], 0.99)
        assert np.array_equal(out["diff"][w], diff) and np.array_equal(out["cnt"][w], cnt)
        assert np.array_equal(out["D"][w], D, equal_nan=True)
        if len(cols) and not np.isnan(D).any():
            want_p0 = oracle.p0uu(post[:, cols], meth[:, cols], 0.99)[0]
            assert out["p0uu"][w] == want_p0
            if D.max() > 0:
                ped = ped6.copy()
                ped[:, 3] = D  # same nodes and edges in every window (src/setup.rs:35-72): only D changes
                keep.append(w)
                probs.append(ab.Problem(ped, want_p0, want_p0, 1.0))
                oprobs.append(oracle.Problem(ped, want_p0, want_p0, 1.0))
    assert len(keep) >= 20
    n_starts = 40
    sx = np.stack([ab.gen_start_simplices(SEED, w, n_starts, float(p.pedigree[:, 3].max())) for w, p in zip(keep, probs)])
    res = ctx.fit_batch(probs, sx, max_iters=10000)
    off = 0
    for i, w in enumerate(keep):
        check_fit_against_oracle(ab, oracle, res, i, oprobs[i], sx[i], 10000,
                                 oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, off, 6)
        off += 6


def test_alphabeta_batch_equals_fit_then_boot(ab, ctx, oracle, ped351, ped78):
    """the combined call (alphabeta::run per window, overlapped uploads) against the two separate calls and the oracle"""
    rng = np.random.default_rng(21)
    cases = [synth_problem(rng, ped351) for _ in range(3)] + [ped78]
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    n_starts, n_boot, first_id = 48, 20, 1000
    sx = np.stack([ab.gen_start_simplices(SEED, first_id + i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    idx = np.concatenate([ab.gen_resample_idx(SEED, first_id + i, n_boot, len(p)).ravel() for i, (p, u) in enumerate(cases)])
    out = ctx.alphabeta_batch(probs, sx, idx, SEED, first_problem_id=first_id)
    res = ctx.fit_batch(probs, sx, max_iters=10000)
    assert np.array_equal(out["best"]["theta"], res.best["theta"]) and np.array_equal(out["pred"], res.pred)
    assert np.array_equal(out["resid"], res.resid) and np.all(out["status"] == 0)
    vary = np.stack([ab.gen_vary_vertices(SEED, first_id + i, n_boot, res.best[i]["theta"]) for i in range(len(cases))])
    rows, _ = ctx.boot_batch(probs, res.best, res.pred, res.resid, idx, vary)
    assert np.array_equal(out["rows"], rows)
    off = 0
    for i, (p, u) in enumerate(cases):
        n = len(p)
        flags = oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL
        rc, orows, _ = oracle.boot_model(oracle.Problem(p, u, u, 1.0), res.best[i]["theta"], res.pred[off:off + n],
                                         res.resid[off:off + n], idx[off * n_boot:(off + n) * n_boot].reshape(n_boot, n),
                                         vary[i], flags=flags, n_threads=4)
        assert rc == 0 and np.array_equal(out["rows"][i], orows)
        assert np.array_equal(out["analysis"][i], oracle.analyze(orows), equal_nan=True)
        off += n


# ---------------------------------------------------------------------------------------------
# large pedigrees: per-lane state in global scratch (carve_big)
# ---------------------------------------------------------------------------------------------
def c5_pedigree(rng, lineages=10, generations=20):
    """C5 shape: `lineages` independent lines sampled at generations 1..`generations` from a common G0"""
    samples = [(l, g) for l in range(lineages) for g in range(1, generations + 1)]
    rows = []
    for i in range(len(samples)):
        for j in range(i + 1, len(samples)):
            (l1, g1), (l2, g2) = samples[i], samples[j]
            rows.append([min(g1, g2) if l1 == l2 else 0, g1, g2, 0.0])
    ped = np.array(rows, dtype=np.float64)
    return ped


def test_big_variant_is_bit_identical_on_small_problems(ab, ctx, oracle, ped351, monkeypatch):
    """the global-scratch kernels forced onto the C4 pedigree give the same bits as the shared-memory ones"""
    rng = np.random.default_rng(9)
    cases = [synth_problem(rng, ped351) for _ in range(2)]
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    n_starts, n_boot = 300, 40
    sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    idx = np.concatenate([ab.gen_resample_idx(SEED, i, n_boot, len(p)).ravel() for i, (p, u) in enumerate(cases)])
    ref = ctx.alphabeta_batch(probs, sx, idx, SEED)
    monkeypatch.setenv("ABFIT_DEV_BIG", "1")
    monkeypatch.setenv("ABFIT_DEV_WIDE", "0")  # the lane-per-fit global-scratch kernels, not the warp-per-fit ones
    big = ctx.alphabeta_batch(probs, sx, idx, SEED)
    for k in ("pred", "resid", "rows", "status"):
        assert np.array_equal(ref[k], big[k], equal_nan=True), k
    assert np.array_equal(ref["best"]["theta"], big["best"]["theta"])
    theta = np.stack([10 ** rng.uniform(-6, -2, 50), 10 ** rng.uniform(-6, -2, 50), rng.uniform(0, 0.1, 50), rng.uniform(0, 0.01, 50)], axis=1)
    pot = rng.integers(0, 2, 50).astype(np.int32)
    c_big, l_big = ctx.cost_batch(probs, theta, pot)
    monkeypatch.delenv("ABFIT_DEV_BIG")
    monkeypatch.delenv("ABFIT_DEV_WIDE")
    c_ref, l_ref = ctx.cost_batch(probs, theta, pot)
    assert np.array_equal(c_big, c_ref) and np.array_equal(l_big, l_ref)
    for i in range(50):
        pb_o = oracle.Problem(cases[pot[i]][0], cases[pot[i]][1], cases[pot[i]][1], 1.0)
        assert c_big[i] == oracle.cost(pb_o, theta[i]) and l_big[i] == oracle.lse(pb_o, theta[i]), i


def test_c5_large_pedigree_fit(ab, ctx, oracle):
    """BASELINE configs[4]: 200 samples -> 19 900 pairs, 590 distinct (t0,t1,t2) triples, 836 doubles of model state
    per lane: does not fit in shared memory.  The Nelder-Mead kernels run warp-per-fit (abfit_wide.cuh), cost /
    divergence / selection through the global-scratch lane-per-fit variant; all bit-exact against the oracle"""
    rng = np.random.default_rng(17)
    ped = c5_pedigree(rng)
    assert ped.shape == (19900, 4)
    a, b, w, c, p0 = 2e-4, 1e-3, 0.04, 0.002, 0.75
    pb_o = oracle.Problem(ped, p0, p0, 1.0)
    dt, _ = oracle.divergence(pb_o, a, b, w, oracle.FAST_DIVERGENCE)
    ped[:, 3] = np.maximum(c + dt + rng.normal(0, 5e-4, len(ped)), 0.0)
    prob = ab.Problem(ped, p0, p0, 1.0)
    theta = np.array([[a, b, w, c], [3e-4, 2e-3, 0.01, 0.0], [-1e-4, 1e-3, 0.2, 0.01]])
    cost, lse = ctx.cost_batch([prob], theta)
    for i in range(len(theta)):
        assert cost[i] == oracle.cost(oracle.Problem(ped, p0, p0, 1.0), theta[i])
    dtg, _ = ctx.divergence(prob, theta[0])
    assert np.array_equal(dtg, dt)
    n_starts = 40
    sx = ab.gen_start_simplices(SEED, 0, n_starts, float(ped[:, 3].max()))
    res = ctx.fit_batch([prob], sx[None], max_iters=10000)
    assert res.status[0] == 0
    check_fit_against_oracle(ab, oracle, res, 0, oracle.Problem(ped, p0, p0, 1.0), sx, 10000,
                             oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, 0, len(ped))
    assert 0.5 * a < res.best[0]["theta"][0] < 2 * a and 0.5 * b < res.best[0]["theta"][1] < 2 * b
    # bootstrap of the same pedigree (warp-per-fit, D* rows materialised per replicate)
    n_boot = 6
    idx = ab.gen_resample_idx(SEED, 0, n_boot, len(ped))
    vary = ab.gen_vary_vertices(SEED, 0, n_boot, res.best[0]["theta"])[None]
    rows, fits = ctx.boot_batch([prob], res.best, res.pred, res.resid, idx.ravel(), vary, max_iters=1000)
    rc, orows, ofits = oracle.boot_model(oracle.Problem(ped, p0, p0, 1.0), res.best[0]["theta"], res.pred, res.resid,
                                         idx, vary[0], max_iters=1000,
                                         flags=oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, n_threads=8)
    assert rc == 0 and np.array_equal(rows[0], orows)
    for f in ("theta", "cost", "iters", "evals", "status"):
        assert np.array_equal(fits[0][f], ofits[f]), f


@pytest.mark.parametrize("L", [20_000, 70_001])
def test_c5_chain_methylomes_to_fit(ab, ctx, oracle, L):
    """BASELINE configs[4] end to end at a reduced site count: 200 simulated methylomes (10 lineages x 20 generations
    from one founder) -> observed divergence of all 19 900 pairs + p0uu on the GPU -> pedigree -> ABneutral fit with
    the warp-per-fit kernels; every stage against the oracle on the same inputs.  L = 70 001 is a window longer than
    65 536 sites: the GPU's p0uu comes from the blocked sum (<= 1e-12 from the oracle's sequential one), and the two
    CHAINS are compared — oracle p0uu -> oracle fit against GPU p0uu -> GPU fit — at the north-star tolerances."""
    rng = np.random.default_rng(2024)
    lineages, generations = 10, 20
    founder = rng.choice(np.array([0, 2], dtype=np.uint8), size=L, p=[0.7, 0.3])
    rows = []
    for _ in range(lineages):
        cur = founder.copy()
        for _g in range(generations):
            r = rng.random(L)
            cur = np.where((cur == 0) & (r < 4e-3), 2, np.where((cur == 2) & (r < 1.5e-2), 0, cur)).astype(np.uint8)
            rows.append(cur.copy())
    status = np.stack(rows)
    S = len(status)
    post = np.where(rng.random((S, L)) < 0.9, 0.9999, rng.uniform(0.5, 0.99, (S, L)))
    meth = np.clip(status / 2.0 + rng.normal(0, 0.05, (S, L)), 0, 1)
    out = ctx.dmatrix(status, post, meth, 0.99)
    D, diff, cnt = oracle.dmatrix(status, post, 0.99)
    assert np.array_equal(out["diff"][0], diff) and np.array_equal(out["cnt"][0], cnt) and np.array_equal(out["D"][0], D)
    p0, _, _ = oracle.p0uu(post, meth, 0.99)
    assert abs(out["p0uu"][0] - p0) <= 1e-12 * abs(p0)
    ped = c5_pedigree(rng, lineages, generations)
    ped[:, 3] = out["D"][0]
    p0uu = float(out["p0uu"][0])
    n_starts = 12
    sx = ab.gen_start_simplices(SEED, 0, n_starts, float(ped[:, 3].max()))
    res = ctx.fit_batch([ab.Problem(ped, p0uu, p0uu, 1.0)], sx[None], max_iters=10000)
    assert res.status[0] == 0
    check_fit_against_oracle(ab, oracle, res, 0, oracle.Problem(ped, p0uu, p0uu, 1.0), sx, 10000,
                             oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, 0, len(ped))
    # the simulated rates are recovered to within a factor of two
    a, b = res.best[0]["theta"][:2]
    assert 2e-3 < a < 8e-3 and 7e-3 < b < 3e-2, (a, b)
    # chain against chain: the oracle side uses ITS OWN p0uu (p_uu0 and eqp of the objective) and its own D
    ped_o = ped.copy()
    ped_o[:, 3] = D
    rc, obest, _, opred, _ = oracle.ab_neutral(oracle.Problem(ped_o, p0, p0, 1.0), sx, max_iters=10000,
                                               flags=oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, n_threads=8)
    assert rc == 0
    gb = res.best[0]
    assert abs(gb["lse"] - obest["lse"]) <= 1e-9 * obest["lse"]              # best-fit RSS
    assert rel(gb["theta"][:2], obest["theta"][:2]) <= 1e-6                  # fitted alpha, beta
    assert rel(res.pred, opred) <= 1e-5  # predictions follow theta (alpha, beta within 1e-6): not a north-star tolerance
    if L <= 65_536:
        assert out["p0uu"][0] == p0 and np.array_equal(gb["theta"], obest["theta"])


# ---------------------------------------------------------------------------------------------
# C4 at BASELINE.json's full size, through size-independent properties
# ---------------------------------------------------------------------------------------------
def test_c4_full_size_properties(ab, ctx, oracle, ped351):
    """10 000 windows x (1000 starts + 100 bootstrap replicates) in one abfit_alphabeta_batch call (11 M fits).
    Too large for the oracle, so: (1) every window fits; (2) sharding invariance — a slice of the windows run on its
    own gives the same bits (what multi-GPU sharding relies on); (3) the oracle's best of the first 16 starts of a
    few windows can never beat the GPU's best of 1000, and is reproduced exactly when the winner is among them;
    (4) the bootstrap rows are internally consistent (equilibrium columns recomputed from alpha, beta)."""
    import bench

    W, NS, NB = 10000, 1000, 100
    shape = bench.load_shape()
    peds, p0uu = bench.synth_windows(W, 0, shape)
    N = peds.shape[1]
    probs = [ab.Problem(peds[i], float(p0uu[i]), float(p0uu[i]), 1.0) for i in range(W)]
    sx = np.empty((W, NS, 5, 4))
    idx = np.empty((W, NB, N), dtype=np.int32)
    from concurrent.futures import ThreadPoolExecutor

    def gen(i):
        sx[i] = ab.gen_start_simplices(SEED, i, NS, float(peds[i, :, 3].max()))
        idx[i] = ab.gen_resample_idx(SEED, i, NB, N)

    with ThreadPoolExecutor(16) as ex:
        list(ex.map(gen, range(W)))
    out = ctx.alphabeta_batch(probs, sx, idx, SEED)
    assert np.all(out["status"] == 0) and np.all(out["best"]["status"] > 0)
    assert np.all(np.isfinite(out["rows"])) and np.all(np.isfinite(out["analysis"][:, :16]))
    # (2) a slice on its own
    lo, hi = 4321, 4337
    sub = ctx.alphabeta_batch(probs[lo:hi], sx[lo:hi], idx[lo:hi], SEED, first_problem_id=lo)
    assert np.array_equal(sub["best"]["theta"], out["best"]["theta"][lo:hi])
    assert np.array_equal(sub["best"]["start_id"], out["best"]["start_id"][lo:hi])
    assert np.array_equal(sub["rows"], out["rows"][lo:hi]) and np.array_equal(sub["pred"], out["pred"][lo * N:hi * N])
    # (3) oracle on the first 16 starts of three windows
    for w in (0, 777, 9999):
        rc, best, _, _, _ = oracle.ab_neutral(oracle.Problem(peds[w], p0uu[w], p0uu[w], 1.0), sx[w, :16],
                                              flags=oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, n_threads=8)
        assert rc == 0 and out["best"][w]["lse"] <= best["lse"]
        if out["best"][w]["start_id"] < 16:
            assert np.array_equal(out["best"][w]["theta"], best["theta"])
    # (4) est_mm / est_um / est_uu columns (src/structs.rs:146-158) from the fitted alpha, beta
    a, b = out["rows"][..., 0], out["rows"][..., 1]
    den = (a + b) * ((a + b - 1.0) ** 2 - 2.0)
    assert np.allclose(out["rows"][..., 4], a * ((1 - a) ** 2 - (1 - b) ** 2 - 1.0) / den, rtol=1e-12, atol=0)
    assert np.allclose(out["rows"][..., 6], b * ((1 - b) ** 2 - (1 - a) ** 2 - 1.0) / den, rtol=1e-12, atol=0)
    assert np.allclose(out["rows"][..., 4:7].sum(axis=-1), 1.0, atol=1e-9)


@pytest.mark.parametrize("env", [{"ABFIT_DEV_NWARPS": "4"}, {"ABFIT_DEV_NWARPS": "2"}, {"ABFIT_DEV_NWARPS": "1"},
                                 {"ABFIT_DEV_XGLOBAL": "1"}, {"ABFIT_DEV_BOOT_TILE": "1"}, {"ABFIT_DEV_CHUNK": "40"},
                                 {"ABFIT_DEV_BIG": "1", "ABFIT_DEV_WIDE": "0"}, {"ABFIT_DEV_WIDE": "1"},
                                 {"ABFIT_DEV_BOOT_XGLOBAL": "0"}, {"ABFIT_DEV_BOOT_XGLOBAL": "1"}])
def test_kernel_variants_are_bit_identical(ab, ctx, ped351, ped78, monkeypatch, env):
    """every launch shape the library can choose (warps per block, queue chunking with tail hand-off, simplex vertices
    in shared / global memory, stored-D* / index-tile bootstrap, global-scratch lane state, warp-per-fit) returns the
    same bits"""
    rng = np.random.default_rng(33)
    ped6 = np.loadtxt(os.path.join(GOLDEN, "pedigree_generated.txt"), skiprows=1)
    # different pedigrees in one batch: 351 pairs (two share a program), 78 pairs, 6 pairs (shorter than one chunk)
    cases = [synth_problem(rng, ped351) for _ in range(2)] + [ped78, (ped6, 0.655), synth_problem(rng, ped351, n_keep=200)]
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    n_starts, n_boot = 400, 48
    sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    idx = np.concatenate([ab.gen_resample_idx(SEED, i, n_boot, len(p)).ravel() for i, (p, u) in enumerate(cases)])
    ref = ctx.alphabeta_batch(probs, sx, idx, SEED)
    ref_all = ctx.fit_batch(probs, sx).all
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    got = ctx.alphabeta_batch(probs, sx, idx, SEED)
    got_all = ctx.fit_batch(probs, sx).all
    for k in ("pred", "resid", "rows", "status", "analysis"):
        assert np.array_equal(ref[k], got[k], equal_nan=True), k
    for f in ("theta", "cost", "lse", "iters", "evals", "status", "start_id"):
        assert np.array_equal(ref_all[f], got_all[f]), f


@pytest.mark.parametrize("n_starts", [33, 61, 97])
def test_tail_handoff_stress(ab, ctx, oracle, ped351, monkeypatch, n_starts):
    """the lock-free tail hand-off (mailbox word, CAS, targeted offers) at the shapes that maximise it: 3-warp blocks
    whose queue holds 33-97 starts, i.e. it is drained almost at once and every warp thins out; 60 repetitions, all
    fit records compared bit for bit each time (a lost or duplicated lane state changes them or hangs the launch)"""
    rng = np.random.default_rng(7000 + n_starts)
    cases = [synth_problem(rng, ped351) for _ in range(6)]
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    monkeypatch.setenv("ABFIT_DEV_NWARPS", "1")   # one warp per block: no hand-off, the reference bits
    ref = ctx.fit_batch(probs, sx, max_iters=10000).all
    flags = oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL
    rc, _, allr, _, _ = oracle.ab_neutral(oracle.Problem(cases[0][0], cases[0][1], cases[0][1], 1.0), sx[0], max_iters=10000,
                                          flags=flags, n_threads=8)
    assert rc == 0 and np.array_equal(ref[0]["theta"], allr["theta"]) and np.array_equal(ref[0]["evals"], allr["evals"])
    monkeypatch.setenv("ABFIT_DEV_NWARPS", "3")
    monkeypatch.setenv("ABFIT_DEV_CHUNK", str(n_starts))
    b = ctx.batch(probs)
    b.upload_starts(sx)
    for rep in range(60):
        b.run_fit()
        got = b.download_fit(want_all=True).all
        assert got.tobytes() == ref.tobytes(), rep
    b.close()


@pytest.mark.parametrize("env", [{}, {"ABFIT_DEV_BOOT_TILE": "1"}, {"ABFIT_DEV_WIDE": "1"},
                                 {"ABFIT_DEV_BIG": "1", "ABFIT_DEV_WIDE": "0"}])
def test_resample_index_out_of_range_is_an_error_in_every_boot_kernel(ab, ctx, ped351, monkeypatch, env):
    """contract of abfit_boot_batch: a resample index outside [0, n_pairs) -> ABFIT_ERR_ARG, whichever bootstrap kernel
    the planner picks (index tile, stored D* tile, warp-per-fit, global-scratch lane state); never an out-of-bounds read"""
    rng = np.random.default_rng(77)
    p, u = synth_problem(rng, ped351, n_keep=90)
    prob = [ab.Problem(p, u, u, 1.0)]
    sx = ab.gen_start_simplices(SEED, 0, 32, float(p[:, 3].max()))[None]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    res = ctx.fit_batch(prob, sx)
    n_boot = 40
    idx = ab.gen_resample_idx(SEED, 0, n_boot, len(p))
    vary = ab.gen_vary_vertices(SEED, 0, n_boot, res.best[0]["theta"])[None]
    rows, _ = ctx.boot_batch(prob, res.best, res.pred, res.resid, idx.ravel(), vary)
    assert np.all(np.isfinite(rows))
    for bad in (len(p), -1, 2 ** 30):
        idx2 = idx.copy()
        idx2[17, 5] = bad
        with pytest.raises(ab.AbfitError) as e:
            ctx.boot_batch(prob, res.best, res.pred, res.resid, idx2.ravel(), vary)
        assert e.value.code == ab.ERR_ARG


def test_resample_index_check_large_pedigree(ab, ctx):
    """same contract on a pedigree with more than 8191 pairs (u16 index tile not applicable)"""
    rng = np.random.default_rng(78)
    ped = c5_pedigree(rng, lineages=10, generations=13)  # 130 samples -> 8385 pairs
    assert len(ped) > 8191
    ped[:, 3] = 0.002 + 1e-4 * ped[:, 1] + 1e-4 * ped[:, 2] + rng.normal(0, 1e-4, len(ped))
    prob = [ab.Problem(ped, 0.8, 0.8, 1.0)]
    sx = ab.gen_start_simplices(SEED, 0, 4, float(ped[:, 3].max()))[None]
    res = ctx.fit_batch(prob, sx, max_iters=200)
    n_boot = 3
    idx = ab.gen_resample_idx(SEED, 0, n_boot, len(ped))
    vary = ab.gen_vary_vertices(SEED, 0, n_boot, res.best[0]["theta"])[None]
    rows, _ = ctx.boot_batch(prob, res.best, res.pred, res.resid, idx.ravel(), vary, max_iters=50)
    assert np.all(np.isfinite(rows))
    idx[1, 8000] = len(ped)
    with pytest.raises(ab.AbfitError) as e:
        ctx.boot_batch(prob, res.best, res.pred, res.resid, idx.ravel(), vary, max_iters=50)
    assert e.value.code == ab.ERR_ARG


@pytest.mark.parametrize("env", [{}, {"ABFIT_DEV_CHUNK": "40"}, {"ABFIT_DEV_CHUNK": "7"}, {"ABFIT_DEV_PIPES": "2"},
                                 {"ABFIT_DEV_JIT_ROLL": "0"}, {"ABFIT_DEV_JIT_ROLL": "3", "ABFIT_DEV_CHUNK": "40"},
                                 {"ABFIT_DEV_PIPES": "5", "ABFIT_DEV_CHUNK": "40"}, {"ABFIT_DEV_JIT_WARPS": "2"},
                                 {"ABFIT_DEV_JIT_WARPS": "3", "ABFIT_DEV_CHUNK": "7", "ABFIT_DEV_PIPES": "2"},
                                 {"ABFIT_DEV_SCHED": "1", "ABFIT_DEV_NWARPS": "3", "ABFIT_DEV_CHUNK": "150"},
                                 {"ABFIT_DEV_SCHED": "1", "ABFIT_DEV_NWARPS": "4"}, {"ABFIT_DEV_SCHED": "1"},
                                 {"ABFIT_DEV_FIT_WARPS": "4"}, {"ABFIT_DEV_FIT_WARPS": "1"}, {"ABFIT_DEV_FIT_WARPS": "4", "ABFIT_DEV_CHUNK": "7"},
                                 {"ABFIT_DEV_FIT_WARPS": "3", "ABFIT_DEV_CHUNK": "40", "ABFIT_DEV_PIPES": "2"},
                                 {"ABFIT_DEV_FIT_WARPS": "6", "ABFIT_DEV_CHUNK": "150"}])
def test_specialised_kernels_are_bit_identical(ab, ctx, oracle, ped351, ped78, monkeypatch, env):
    """run-time specialised kernels (csrc/abfit_jit.cu: the batch's one micro-op program compiled to straight-line
    code by NVRTC) against the interpreter kernels and the oracle: every start, every bootstrap row, same bits.
    Default = continuous lane scheduling (persistent warps, two window slots per warp; small chunks force constant
    slot switching and waiting for stragglers); ABFIT_DEV_SCHED=1 = the block-per-item bodies on the specialised
    objective (one-warp blocks, 3-warp blocks with queue + tail hand-off, 4-warp blocks)"""
    rng = np.random.default_rng(55)
    for shape_ped, n_keep in ((ped351, None), (ped351, 123), (ped78[0], None)):
        base, u0 = synth_problem(rng, shape_ped, n_keep=n_keep)
        cases = []
        for _ in range(5):  # same time structure (one program), different D and p0uu: a metaprofile's windows
            p = base.copy()
            p[:, 3] = np.maximum(base[:, 3] * rng.uniform(0.7, 1.3) + rng.normal(0, 3e-4, len(base)), 0.0)
            cases.append((p, float(rng.uniform(0.6, 0.95))))
        probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
        n_starts, n_boot = 300, 40
        sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
        idx = np.concatenate([ab.gen_resample_idx(SEED, i, n_boot, len(p)).ravel() for i, (p, u) in enumerate(cases)])
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        monkeypatch.setenv("ABFIT_JIT", "0")
        ref = ctx.alphabeta_batch(probs, sx, idx, SEED)
        b0 = ctx.batch(probs)
        b0.upload_starts(sx)
        assert not b0.uses_specialised_kernels()
        b0.run_fit()
        ref_all = b0.download_fit(want_all=True).all
        b0.close()
        monkeypatch.setenv("ABFIT_JIT", "1")
        got = ctx.alphabeta_batch(probs, sx, idx, SEED)
        b1 = ctx.batch(probs)
        b1.upload_starts(sx)
        assert b1.uses_specialised_kernels(), ab.jit_last_error()
        b1.run_fit()
        got_all = b1.download_fit(want_all=True).all
        b1.close()
        for k in ("pred", "resid", "rows", "status", "analysis"):
            assert np.array_equal(ref[k], got[k], equal_nan=True), k
        assert got_all.tobytes() == ref_all.tobytes()
        p, u = cases[2]
        rc, best, allr, pred, resid = oracle.ab_neutral(oracle.Problem(p, u, u, 1.0), sx[2], max_iters=10000,
                                                        flags=oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, n_threads=8)
        assert rc == 0
        for f in ("theta", "cost", "lse", "iters", "evals", "status", "start_id"):
            assert np.array_equal(got_all[2][f], allr[f]), f
        monkeypatch.delenv("ABFIT_JIT")


@pytest.mark.parametrize("fit_warps,n_starts,chunk", [(4, 500, None), (4, 97, "33"), (6, 300, "40"), (2, 64, "7")])
def test_drain_merging_stress(ab, ctx, ped351, monkeypatch, fit_warps, n_starts, chunk):
    """drain merging of the multi-start kernel (ABFIT_DEV_FIT_WARPS: blocks of several independent warps whose
    emptiest warp hands its running fits to a sibling once the item cursor is dry, abfit_fitkernels.cuh): 40
    repetitions per shape, every fit record compared bit for bit with the one-warp-block kernel each time (a lost,
    duplicated or mixed-up lane state changes them or hangs the launch)"""
    rng = np.random.default_rng(8100 + n_starts)
    base, _ = synth_problem(rng, ped351)
    cases = []
    for _ in range(8):
        p = base.copy()
        p[:, 3] = np.maximum(base[:, 3] * rng.uniform(0.7, 1.3) + rng.normal(0, 3e-4, len(base)), 0.0)
        cases.append((p, float(rng.uniform(0.6, 0.95))))
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    monkeypatch.setenv("ABFIT_JIT", "1")
    monkeypatch.setenv("ABFIT_DEV_FIT_WARPS", "1")
    b = ctx.batch(probs)
    b.upload_starts(sx)
    assert b.uses_specialised_kernels(), ab.jit_last_error()
    b.run_fit()
    ref = b.download_fit(want_all=True).all
    b.close()
    monkeypatch.setenv("ABFIT_DEV_FIT_WARPS", str(fit_warps))
    if chunk:
        monkeypatch.setenv("ABFIT_DEV_CHUNK", chunk)
    b = ctx.batch(probs)
    b.upload_starts(sx)
    assert b.uses_specialised_kernels(), ab.jit_last_error()
    for rep in range(40):
        b.run_fit()
        got = b.download_fit(want_all=True).all
        assert got.tobytes() == ref.tobytes(), rep
    b.close()


@pytest.mark.parametrize("n_starts,n_boot", [(1, 1), (33, 31), (97, 100), (257, 7)])
def test_specialised_kernels_ragged_counts(ab, ctx, oracle, ped351, monkeypatch, n_starts, n_boot):
    """continuous lane scheduling with start / replicate counts that fill neither warps nor items; three windows of
    one program; every start and every bootstrap row bit-identical to the oracle"""
    rng = np.random.default_rng(900 + n_starts)
    base, _ = synth_problem(rng, ped351, n_keep=77)
    cases = []
    for _ in range(3):
        p = base.copy()
        p[:, 3] = np.maximum(base[:, 3] * rng.uniform(0.7, 1.3) + rng.normal(0, 3e-4, len(base)), 0.0)
        cases.append((p, float(rng.uniform(0.6, 0.95))))
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    idx = np.concatenate([ab.gen_resample_idx(SEED, i, n_boot, len(p)).ravel() for i, (p, u) in enumerate(cases)])
    monkeypatch.setenv("ABFIT_JIT", "1")
    b = ctx.batch(probs)
    b.upload_starts(sx)
    assert b.uses_specialised_kernels(), ab.jit_last_error()
    b.run_fit()
    res = b.download_fit(want_all=True)
    vary = np.stack([ab.gen_vary_vertices(SEED, i, n_boot, res.best[i]["theta"]) for i in range(len(cases))])
    b.upload_boot(idx, vary)
    b.run_boot()
    rows, fits = b.download_boot(want_fits=True)
    b.close()
    flags = oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL
    off = 0
    for i, (p, u) in enumerate(cases):
        n = len(p)
        check_fit_against_oracle(ab, oracle, res, i, oracle.Problem(p, u, u, 1.0), sx[i], 10000, flags, off, n)
        rc, orows, ofits = oracle.boot_model(oracle.Problem(p, u, u, 1.0), res.best[i]["theta"], res.pred[off:off + n],
                                             res.resid[off:off + n], idx[off * n_boot:(off + n) * n_boot].reshape(n_boot, n),
                                             vary[i], max_iters=1000, flags=flags, n_threads=8)
        assert rc == 0 and np.array_equal(rows[i], orows)
        assert np.array_equal(fits[i]["evals"], ofits["evals"])
        off += n
    # an out-of-range resample index is reported by the specialised bootstrap kernel too
    if n_boot > 1:
        bad = idx.copy()
        bad[5] = len(cases[0][0])
        b = ctx.batch(probs)
        b.upload_starts(sx)
        b.run_fit()
        b.upload_boot(bad, vary)
        b.run_boot()
        with pytest.raises(ab.AbfitError) as e:
            b.download_boot()
        assert e.value.code == ab.ERR_ARG
        b.close()


def test_pipelined_pass_equals_fit_then_boot(ab, ctx, ped351, monkeypatch):
    """abfit_batch_run_pipelined (sub-batches of windows as overlapping fit -> select -> bootstrap chains on their own
    streams) gives the bytes of run_fit followed by run_boot; repeated, because the overlap is scheduling-dependent"""
    rng = np.random.default_rng(57)
    base, _ = synth_problem(rng, ped351, n_keep=101)
    cases = []
    for _ in range(9):
        p = base.copy()
        p[:, 3] = np.maximum(base[:, 3] * rng.uniform(0.7, 1.3) + rng.normal(0, 3e-4, len(base)), 0.0)
        cases.append((p, float(rng.uniform(0.6, 0.95))))
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    n_starts, n_boot = 150, 37
    sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    idx = np.concatenate([ab.gen_resample_idx(SEED, i, n_boot, len(p)).ravel() for i, (p, u) in enumerate(cases)])
    monkeypatch.setenv("ABFIT_JIT", "1")
    monkeypatch.setenv("ABFIT_DEV_PIPES", "4")
    b = ctx.batch(probs)
    b.upload_starts(sx)
    b.run_fit()
    res = b.download_fit(want_all=True)
    vary = np.stack([ab.gen_vary_vertices(SEED, i, n_boot, res.best[i]["theta"]) for i in range(len(cases))])
    b.upload_boot(idx, vary)
    b.run_boot()
    rows, fits = b.download_boot(want_fits=True)
    t_seq = b.timing()
    for rep in range(5):
        b.run_pipelined()
        assert b.pipes() == 4
        res2 = b.download_fit(want_all=True)
        rows2, fits2 = b.download_boot(want_fits=True)
        assert res2.all.tobytes() == res.all.tobytes() and res2.best.tobytes() == res.best.tobytes(), rep
        assert np.array_equal(res2.pred, res.pred) and np.array_equal(res2.resid, res.resid)
        assert rows2.tobytes() == rows.tobytes() and fits2.tobytes() == fits.tobytes(), rep
        t = b.timing()
        assert t["evals_fit"] == t_seq["evals_fit"] and t["evals_boot"] == t_seq["evals_boot"] and t["launches"] == 12
    b.close()
    # the one-shot call takes the same pipelined path (vary vertices drawn on the device per sub-batch)
    out = ctx.alphabeta_batch(probs, sx, idx, SEED)
    assert np.array_equal(out["rows"], rows) and np.array_equal(out["best"]["theta"], res.best["theta"])


def test_specialised_kernels_mixed_batch_falls_back_to_interpreter(ab, ctx, ped351, ped78, monkeypatch):
    """a batch that mixes pedigree programs is not specialised (one kernel per program would be needed); same API"""
    rng = np.random.default_rng(56)
    cases = [synth_problem(rng, ped351), ped78]
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    sx = np.stack([ab.gen_start_simplices(SEED, i, 64, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    monkeypatch.setenv("ABFIT_JIT", "1")
    b = ctx.batch(probs)
    b.upload_starts(sx)
    assert not b.uses_specialised_kernels()
    b.run_fit()
    assert np.all(b.download_fit().status == 0)
    b.close()


# ---------------------------------------------------------------------------------------------
# multi-GPU inside the product: one context + host thread per device, windows (or sites) sharded
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx_pool(ab):
    """one context per visible device; on a one-GPU box three contexts on device 0 (the sharding, threading and
    gathering logic is the same, only the devices coincide)"""
    n = ab.device_count()
    devs = list(range(n)) if n >= 2 else [0, 0, 0]
    pool = [ab.Context(d) for d in devs]
    yield pool
    for c in pool:
        c.close()


def test_multi_device_alphabeta_equals_single_device(ab, ctx, ctx_pool, ped351, ped78):
    """abfit_alphabeta_batch_multi (windows sharded over the contexts, ragged pedigrees so the shards' offsets into
    the concatenated arrays differ) returns the single-device bytes; and with per-window generator keys a window's
    result does not change when another window is dropped from the batch"""
    rng = np.random.default_rng(71)
    cases = [synth_problem(rng, ped351, n_keep=k) for k in (60, 60, 33, 90, 60, 17, 45)]
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    ids = np.array([3, 4, 9, 10, 11, 40, 41], dtype=np.uint64)  # window ids with gaps (empty windows were dropped)
    n_starts, n_boot = 64, 24
    sx = np.stack([ab.gen_start_simplices(SEED, int(i), n_starts, float(p[:, 3].max())) for i, (p, u) in zip(ids, cases)])
    idx = np.concatenate([ab.gen_resample_idx(SEED, int(i), n_boot, len(p)).ravel() for i, (p, u) in zip(ids, cases)])
    one = ab.alphabeta_batch_multi([ctx], probs, sx, idx, SEED, problem_ids=ids)
    many = ab.alphabeta_batch_multi(ctx_pool, probs, sx, idx, SEED, problem_ids=ids)
    for k in ("best", "pred", "resid", "status", "rows", "analysis"):
        assert one[k].tobytes() == many[k].tobytes(), k
    # consecutive keys: the single-context entry point gives the same bytes
    idx2 = np.concatenate([ab.gen_resample_idx(SEED, 100 + i, n_boot, len(p)).ravel() for i, (p, u) in enumerate(cases)])
    sx2 = np.stack([ab.gen_start_simplices(SEED, 100 + i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    a = ctx.alphabeta_batch(probs, sx2, idx2, SEED, first_problem_id=100)
    b = ab.alphabeta_batch_multi(ctx_pool, probs, sx2, idx2, SEED, first_problem_id=100)
    for k in ("best", "pred", "resid", "status", "rows", "analysis"):
        assert a[k].tobytes() == b[k].tobytes(), k
    # drop window 2: everybody else keeps its results (ADVICE r1: vary vertices used to be keyed by batch position)
    keep = [0, 1, 3, 4, 5, 6]
    offs = np.concatenate([[0], np.cumsum([len(p) for p, u in cases])])
    idx_k = np.concatenate([idx[offs[i] * n_boot:offs[i + 1] * n_boot] for i in keep])
    sub = ab.alphabeta_batch_multi(ctx_pool, [probs[i] for i in keep], sx[keep], idx_k, SEED, problem_ids=ids[keep])
    assert np.array_equal(sub["rows"], many["rows"][keep]) and np.array_equal(sub["best"]["theta"], many["best"]["theta"][keep])


def test_resample_indices_drawn_on_the_device(ab, ctx, ctx_pool, ped351, ped78):
    """abfit_alphabeta_batch / _multi with resample_idx = NULL: the indices are drawn on the device (k_gen_resample) and
    are the numbers abfit_gen_resample_idx returns — every output equals, byte for byte, the call that is handed the
    host-generated indices; ragged pedigrees, consecutive keys with an offset, per-window keys, several contexts"""
    rng = np.random.default_rng(73)
    cases = [synth_problem(rng, ped351, n_keep=k) for k in (60, 33, 90, 17)] + [synth_problem(rng, ped78[0]), synth_problem(rng, ped351)]
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    n_starts, n_boot = 64, 37
    keys = ("best", "pred", "resid", "status", "rows", "analysis")
    sx = np.stack([ab.gen_start_simplices(SEED, 7 + i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    idx = np.concatenate([ab.gen_resample_idx(SEED, 7 + i, n_boot, len(p)).ravel() for i, (p, u) in enumerate(cases)])
    host = ctx.alphabeta_batch(probs, sx, idx, SEED, first_problem_id=7)
    dev = ctx.alphabeta_batch(probs, sx, n_boot, SEED, first_problem_id=7)
    for k in keys:
        assert host[k].tobytes() == dev[k].tobytes(), k
    ids = np.array([3, 4, 9, 10, 40, 41], dtype=np.uint64)
    idx2 = np.concatenate([ab.gen_resample_idx(SEED, int(i), n_boot, len(p)).ravel() for i, (p, u) in zip(ids, cases)])
    host2 = ab.alphabeta_batch_multi(ctx_pool, probs, sx, idx2, SEED, problem_ids=ids)
    dev2 = ab.alphabeta_batch_multi(ctx_pool, probs, sx, n_boot, SEED, problem_ids=ids)
    for k in keys:
        assert host2[k].tobytes() == dev2[k].tobytes(), k
    assert host["rows"].tobytes() != host2["rows"].tobytes()  # (the keys matter)


def test_multi_device_divergence(ab, ctx, ctx_pool, oracle):
    """abfit_divergence_multi: window-sharded = single device bit for bit; site-sharded whole methylomes: integer sums
    and D exact, p0uu within 1e-12 (north_star)"""
    rng = np.random.default_rng(72)
    S, L = 11, 40_000
    status, post, meth = synth_methylomes(rng, S, L)
    seg = np.array([0, 100, 100, 1000, 7777, 7778, 20000, 39999, 40000], dtype=np.int64)
    one = ctx.dmatrix(status, post, meth, 0.99, seg)
    many = ab.dmatrix_multi(ctx_pool, status, post, meth, 0.99, seg)
    for k in ("diff", "cnt", "nvalid"):
        assert np.array_equal(one[k], many[k]), k
    for k in ("D", "p0uu", "methsum"):
        assert np.array_equal(one[k], many[k], equal_nan=True), k
    whole1 = ctx.dmatrix(status, post, meth, 0.99)
    whole = ab.dmatrix_multi(ctx_pool, status, post, meth, 0.99)
    D, diff, cnt = oracle.dmatrix(status, post, 0.99)
    assert np.array_equal(whole["diff"][0], diff) and np.array_equal(whole["cnt"][0], cnt) and np.array_equal(whole["D"][0], D)
    assert np.array_equal(whole["nvalid"], whole1["nvalid"])
    p0 = oracle.p0uu(post, meth, 0.99)[0]
    assert abs(whole["p0uu"][0] - p0) <= 1e-12 * abs(p0)


@pytest.mark.parametrize("chunks", ["2", "5", "16"])
def test_dmatrix_overlapped_chunks(ab, ctx, oracle, monkeypatch, chunks):
    """the pack pass and the pair pass overlapped chunk by chunk on two streams (run_divergence): same integers, same D,
    same per-sample sums as the back-to-back passes and as the oracle — whole methylomes and windowed"""
    rng = np.random.default_rng(300 + int(chunks))
    S, L = 23, 330_007
    status, post, meth = synth_methylomes(rng, S, L)
    monkeypatch.setenv("ABFIT_DEV_DIV_FUSED", "0")  # the two-kernel path (whole methylomes of <= 200 samples take k_fused by default)
    monkeypatch.setenv("ABFIT_DEV_DIV_CHUNKS", "1")
    ref = ctx.dmatrix(status, post, meth, 0.99)
    seg = np.array([0, 5, 64_000, 64_001, 200_000, 200_000, 330_000, 330_007], dtype=np.int64)
    ref_w = ctx.dmatrix(status, post, meth, 0.99, seg)
    monkeypatch.setenv("ABFIT_DEV_DIV_CHUNKS", chunks)
    for rep in range(3):
        got = ctx.dmatrix(status, post, meth, 0.99)
        got_w = ctx.dmatrix(status, post, meth, 0.99, seg)
        for k in ("diff", "cnt", "nvalid"):
            assert np.array_equal(ref[k], got[k]) and np.array_equal(ref_w[k], got_w[k]), (k, rep)
        for k in ("D", "p0uu", "methsum"):
            assert np.array_equal(ref[k], got[k], equal_nan=True) and np.array_equal(ref_w[k], got_w[k], equal_nan=True), (k, rep)
    D, diff, cnt = oracle.dmatrix(status, post, 0.99)
    assert np.array_equal(got["diff"][0], diff) and np.array_equal(got["cnt"][0], cnt) and np.array_equal(got["D"][0], D)
    monkeypatch.delenv("ABFIT_DEV_DIV_CHUNKS")
    big = ctx.dmatrix(np.tile(status, (1, 2)), np.tile(post, (1, 2)), np.tile(meth, (1, 2)), 0.99)  # default: chunked (> 8192 words)
    assert np.array_equal(big["diff"][0], 2 * diff) and np.array_equal(big["cnt"][0], 2 * cnt)


@pytest.mark.parametrize("S,L,seg", [(23, 330_007, None), (2, 70_001, None), (5, 65_537, None), (200, 140_000, None),
                                     (37, 400_000, [3, 399_990]), (4, 1_000_003, [65, 1_000_003]), (9, 66_000, [1, 66_000])])
def test_dmatrix_fused_kernel(ab, ctx, oracle, monkeypatch, S, L, seg):
    """k_fused (bulk-copy packer warps + all-pairs popcount warps in one persistent kernel, whole methylomes): integers
    and D exact against the oracle and against the two-kernel path, per-sample sums within 1e-12 (its own fixed
    blocking), run-to-run identical; odd L (rows that are not 16-byte aligned), windows that start and end inside the
    rows, partial last words and groups, more packer warps than samples"""
    rng = np.random.default_rng(7000 + S + L)
    status, post, meth = synth_methylomes(rng, S, L)
    a, b = (0, L) if seg is None else seg
    import torch
    d_st, d_po, d_me = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (status, post, meth))
    run = lambda: ctx.dmatrix_device(d_st.data_ptr(), d_po.data_ptr(), d_me.data_ptr(), S, L, 0.99, seg_offsets=seg)
    monkeypatch.setenv("ABFIT_DEV_DIV_FUSED", "0")
    ref = run()
    assert ref["launches"] > 4
    monkeypatch.setenv("ABFIT_DEV_DIV_FUSED", "1")
    got = [run() for _ in range(3)]
    D, diff, cnt = oracle.dmatrix(status[:, a:b], post[:, a:b], 0.99)
    p0, rc, nv = oracle.p0uu(post[:, a:b], meth[:, a:b], 0.99)
    for g in got:
        assert g["launches"] <= 4, "the fused path did not run"
        assert np.array_equal(g["diff"][0], diff) and np.array_equal(g["cnt"][0], cnt) and np.array_equal(g["D"][0], D)
        assert np.array_equal(g["diff"], ref["diff"]) and np.array_equal(g["cnt"], ref["cnt"])
        assert np.array_equal(g["nvalid"][0], nv) and np.array_equal(g["nvalid"], ref["nvalid"])
        assert abs(g["p0uu"][0] - p0) <= 1e-12 * abs(p0)
        assert np.allclose(g["methsum"], ref["methsum"], rtol=1e-12, atol=0)
        for k in ("methsum", "p0uu"):
            assert np.array_equal(g[k], got[0][k]), k


def test_dmatrix_fused_kernel_stress(ab, ctx, oracle, monkeypatch):
    """k_fused again and again on shapes that maximise the hand-offs of its protocol — 1 to 3 groups per CTA (stage
    barriers reused or not), 8 k + 1 samples (uneven packer warps), every ring-slot parity — each run bit-compared
    with the first and the first with the oracle (no race detector on this pool: repetition instead)"""
    import torch
    rng = np.random.default_rng(99)
    monkeypatch.setenv("ABFIT_DEV_DIV_FUSED", "1")
    for S, L in [(9, 148 * 512 + 65_536 + 17), (17, 3 * 148 * 512 + 1), (64, 70_000), (33, 200_003)]:
        status, post, meth = synth_methylomes(rng, S, L)
        d_st, d_po, d_me = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (status, post, meth))
        first = None
        for rep in range(25):
            got = ctx.dmatrix_device(d_st.data_ptr(), d_po.data_ptr(), d_me.data_ptr(), S, L, 0.99)
            assert got["launches"] <= 4
            if first is None:
                first = got
                D, diff, cnt = oracle.dmatrix(status, post, 0.99)
                assert np.array_equal(got["diff"][0], diff) and np.array_equal(got["cnt"][0], cnt) and np.array_equal(got["D"][0], D)
            else:
                for k in ("diff", "cnt", "nvalid", "methsum", "p0uu", "D"):
                    assert np.array_equal(got[k], first[k], equal_nan=True), (S, L, rep, k)


def test_suffstats_experiment_within_tolerance(ab, ctx, oracle, ped351, ped78, monkeypatch):
    """EXPERIMENT (ABFIT_EXPERIMENT_SUFFSTATS=1, never the default): multi-start objective from per-triple sufficient
    statistics.  Not bit-identical by construction; what is asserted is north_star's tolerance against the exact path
    (= the oracle, bit for bit): exact RSS at the experiment's best theta within 1e-9 relative, alpha / beta within
    1e-6 — on the R-original 351-pair pedigree (C1's data), the 78-pair example pedigree and C4-style synthetic
    windows; and that the flag really switches the objective (costs differ in the last bits somewhere)."""
    rng = np.random.default_rng(2024)
    groups = [[(ped351, 0.75)], [ped78], [synth_problem(rng, ped351) for _ in range(24)]]
    monkeypatch.setenv("ABFIT_JIT", "1")
    any_diff = False
    for cases in groups:
        probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
        n_starts = 1000 if len(cases) == 1 else 300
        sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
        res = {}
        for mode in ("0", "1"):
            monkeypatch.setenv("ABFIT_EXPERIMENT_SUFFSTATS", mode)
            b = ctx.batch(probs)
            b.upload_starts(sx)
            assert b.uses_specialised_kernels()
            b.run_fit()
            res[mode] = b.download_fit(want_all=True)
            b.close()
        monkeypatch.delenv("ABFIT_EXPERIMENT_SUFFSTATS")
        exact, suff = res["0"], res["1"]
        _, lse_at = ctx.cost_batch(probs, suff.best["theta"], np.arange(len(probs), dtype=np.int32))
        for i in range(len(probs)):
            assert abs(lse_at[i] - exact.best["lse"][i]) <= 1e-9 * abs(exact.best["lse"][i]), i
            for k in (0, 1):
                assert abs(suff.best["theta"][i, k] - exact.best["theta"][i, k]) <= 1e-6 * abs(exact.best["theta"][i, k]), (i, k)
        any_diff |= not np.array_equal(exact.all["cost"], suff.all["cost"])
    assert any_diff


@pytest.mark.parametrize("n_boot", [2, 7, 8, 100, 1000])
def test_device_statistics_equal_host_statistics(ab, ctx, ped351, ped78, monkeypatch, n_boot):
    """abfit_alphabeta_batch computes RawAnalysis::analyze (src/analysis.rs:50-98) on the device behind the bootstrap
    kernel: bit-identical to the host's abfit_analyze on the rows it returns (means incl. the 8-accumulator fold of
    beta / alpha, Welford standard deviations, linear quantiles), for replicate counts around the fold width and
    the quantile positions"""
    rng = np.random.default_rng(700 + n_boot)
    cases = [synth_problem(rng, ped351, n_keep=60) for _ in range(5)] + [ped78]
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    n_starts = 40
    sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    idx = np.concatenate([ab.gen_resample_idx(SEED, i, n_boot, len(p)).ravel() for i, (p, u) in enumerate(cases)])
    out = ctx.alphabeta_batch(probs, sx, idx, SEED)
    for i in range(len(probs)):
        want = ab.analyze(out["rows"][i])
        assert np.array_equal(out["analysis"][i], want, equal_nan=True), i
    monkeypatch.setenv("ABFIT_DEV_HOST_STATS", "1")
    host = ctx.alphabeta_batch(probs, sx, idx, SEED)
    assert np.array_equal(host["analysis"], out["analysis"], equal_nan=True) and np.array_equal(host["rows"], out["rows"])


def test_dmatrix_fused_kernel_several_long_windows(ab, ctx, oracle, monkeypatch):
    """a few windows of more than 65 536 sites each (chromosomes): k_fused once per window; integers and D exact per
    window against the oracle and the two-pass path, per-sample sums within 1e-12; one short window in the list sends
    the whole call to the two-pass path"""
    import torch
    rng = np.random.default_rng(31)
    S, L = 12, 300_000
    status, post, meth = synth_methylomes(rng, S, L)
    d_st, d_po, d_me = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (status, post, meth))
    seg = [0, 70_001, 170_002, 300_000]
    run = lambda sg: ctx.dmatrix_device(d_st.data_ptr(), d_po.data_ptr(), d_me.data_ptr(), S, L, 0.99, seg_offsets=sg)
    monkeypatch.setenv("ABFIT_DEV_DIV_FUSED", "0")
    ref = run(seg)
    monkeypatch.delenv("ABFIT_DEV_DIV_FUSED")
    got = run(seg)
    assert got["launches"] == 12 and ref["launches"] < 12  # 3 x (k_fused + 3 finalisation kernels)
    for w in range(3):
        a, b = seg[w], seg[w + 1]
        D, diff, cnt = oracle.dmatrix(status[:, a:b], post[:, a:b], 0.99)
        assert np.array_equal(got["diff"][w], diff) and np.array_equal(got["cnt"][w], cnt) and np.array_equal(got["D"][w], D)
        p0, rc, nv = oracle.p0uu(post[:, a:b], meth[:, a:b], 0.99)
        assert np.array_equal(got["nvalid"][w], nv) and abs(got["p0uu"][w] - p0) <= 1e-12 * abs(p0)
    assert np.array_equal(got["diff"], ref["diff"]) and np.allclose(got["methsum"], ref["methsum"], rtol=1e-12, atol=0)
    mixed = run([0, 70_001, 70_500, 300_000])
    assert mixed["launches"] < 12
    D, diff, cnt = oracle.dmatrix(status[:, 70_001:70_500], post[:, 70_001:70_500], 0.99)
    assert np.array_equal(mixed["diff"][1], diff) and np.array_equal(mixed["cnt"][1], cnt)


def test_c5_full_size_divergence_properties(ab, ctx, oracle):
    """BASELINE configs[4] at its full size — 200 samples x 5 000 000 sites, 19 900 pairs, 17 GB streamed by k_fused —
    through size-independent properties: the integer sums of two site ranges add up exactly to those of the whole
    (any cut; here one that is not a multiple of 64), a 6-sample x 20 000-site corner equals the oracle bit for bit,
    sample order is respected (swapping two samples permutes the pair sums), and the call is repeatable bit for bit"""
    import torch
    S, L = 200, 5_000_000
    dev = torch.device("cuda", 0)
    if torch.cuda.mem_get_info(dev)[0] < 40e9:
        pytest.skip("needs 40 GB of free device memory")
    g = torch.Generator(device=dev)
    g.manual_seed(55)
    status = (torch.rand((S, L), device=dev, generator=g) * 3).to(torch.uint8).clamp_(max=2)
    post = torch.empty((S, L), dtype=torch.float64, device=dev)
    meth = torch.empty((S, L), dtype=torch.float64, device=dev)
    for s in range(S):  # row by row: no (S, L) temporaries
        u = torch.rand(L, device=dev, generator=g, dtype=torch.float64)
        post[s] = torch.where(torch.rand(L, device=dev, generator=g) < 0.9, torch.full_like(u, 0.9999), u * 0.49 + 0.5)
        meth[s] = torch.rand(L, device=dev, generator=g, dtype=torch.float64)
    torch.cuda.synchronize()  # the library's stream does not wait for torch's: the inputs must be complete first
    run = lambda seg=None: ctx.dmatrix_device(status.data_ptr(), post.data_ptr(), meth.data_ptr(), S, L, 0.99, seg_offsets=seg)
    whole = run()
    assert whole["launches"] <= 4  # the fused kernel
    again = run()
    for k in ("diff", "cnt", "nvalid", "methsum", "p0uu", "D"):
        assert np.array_equal(whole[k], again[k]), k
    parts = run([0, 1_234_567, L])
    assert np.array_equal(parts["diff"].sum(axis=0), whole["diff"][0]) and np.array_equal(parts["cnt"].sum(axis=0), whole["cnt"][0])
    assert np.array_equal(parts["nvalid"].sum(axis=0), whole["nvalid"][0])
    assert np.array_equal(whole["D"][0], whole["diff"][0] / (2.0 * whole["cnt"][0]))  # src/pedigree.rs:257
    # a corner of the data against the oracle
    s6, l6 = 6, 20_000
    sub = ctx.dmatrix(status[:s6, :l6].cpu().numpy(), post[:s6, :l6].cpu().numpy(), meth[:s6, :l6].cpu().numpy(), 0.99)
    D, diff, cnt = oracle.dmatrix(status[:s6, :l6].cpu().numpy(), post[:s6, :l6].cpu().numpy(), 0.99)
    assert np.array_equal(sub["diff"][0], diff) and np.array_equal(sub["cnt"][0], cnt) and np.array_equal(sub["D"][0], D)
    # pair (0, 1) of the whole = pair (0, 1) of the first two rows alone (nothing leaks between samples)
    two = ctx.dmatrix_device(status.data_ptr(), post.data_ptr(), meth.data_ptr(), 2, L, 0.99)
    assert two["diff"][0][0] == whole["diff"][0][0] and two["cnt"][0][0] == whole["cnt"][0][0]
    assert two["nvalid"][0][0] == whole["nvalid"][0][0] and two["nvalid"][0][1] == whole["nvalid"][0][1]


def test_suffstats_experiment_large_pedigree(ab, ctx, oracle, monkeypatch):
    """the same EXPERIMENT on the warp-per-fit kernels (pedigrees with thousands of pairs, C5's family): objective
    from per-triple statistics instead of the sequential sum over every pair; best-of-starts against the exact path at
    north_star's tolerances (exact RSS at the experiment's best theta within 1e-9, alpha / beta within 1e-6)"""
    import bench
    rng = np.random.default_rng(77)
    ped = bench.c5_times(6, 12)  # 72 samples, 2556 pairs
    th = np.array([2.3e-4, 8.1e-4, 0.04, 0.002])
    p0uu = 0.74
    dt, _ = ctx.divergence(ab.Problem(np.column_stack([ped[:, :3], np.zeros(len(ped))]), p0uu, p0uu, 1.0), th)
    ped[:, 3] = np.maximum(th[3] + dt + rng.normal(0, 4e-4, len(ped)), 0.0)
    prob = [ab.Problem(ped, p0uu, p0uu, 1.0)]
    n_starts = 96
    sx = ab.gen_start_simplices(SEED, 0, n_starts, float(ped[:, 3].max()))[None]
    monkeypatch.setenv("ABFIT_DEV_WIDE", "1")
    res = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("ABFIT_EXPERIMENT_SUFFSTATS", mode)
        b = ctx.batch(prob)
        b.upload_starts(sx)
        b.run_fit()
        res[mode] = (b.download_fit(want_all=True), b.timing()["fit_ms"])
        b.close()
    monkeypatch.delenv("ABFIT_EXPERIMENT_SUFFSTATS")
    (exact, ms_exact), (suff, ms_suff) = res["0"], res["1"]
    _, lse_at = ctx.cost_batch(prob, suff.best["theta"], np.zeros(1, dtype=np.int32))
    assert abs(lse_at[0] - exact.best["lse"][0]) <= 1e-9 * abs(exact.best["lse"][0])
    for k in (0, 1):
        assert abs(suff.best["theta"][0, k] - exact.best["theta"][0, k]) <= 1e-6 * abs(exact.best["theta"][0, k]), k
    assert not np.array_equal(exact.all["cost"], suff.all["cost"])  # the flag did switch the objective
    assert ms_suff < ms_exact


def test_suffstats_experiment_bootstrap(ab, ctx, ped351, monkeypatch):
    """EXPERIMENT, mode 2 (ABFIT_EXPERIMENT_SUFFSTATS=2): the bootstrap refits from per-replicate per-triple statistics.
    Same best models, resamples and vary vertices on both sides; nearly every replicate ends bit-identical, all but a
    few within 1e-6 in alpha / beta (a replicate whose trajectory parts may stop elsewhere: it is an experiment)"""
    rng = np.random.default_rng(4242)
    cases = [synth_problem(rng, ped351) for _ in range(16)]
    probs = [ab.Problem(p, u, u, 1.0) for p, u in cases]
    n_starts, n_boot = 120, 100
    sx = np.stack([ab.gen_start_simplices(SEED, i, n_starts, float(p[:, 3].max())) for i, (p, u) in enumerate(cases)])
    idx = np.concatenate([ab.gen_resample_idx(SEED, i, n_boot, len(p)).ravel() for i, (p, u) in enumerate(cases)])
    monkeypatch.setenv("ABFIT_JIT", "1")
    b = ctx.batch(probs)
    b.upload_starts(sx)
    b.run_fit()
    res = b.download_fit()
    vary = np.stack([ab.gen_vary_vertices(SEED, i, n_boot, res.best[i]["theta"]) for i in range(len(cases))])
    b.upload_boot(idx, vary)
    b.run_boot()
    rows_e, _ = b.download_boot()
    b.close()
    monkeypatch.setenv("ABFIT_EXPERIMENT_SUFFSTATS", "2")
    b = ctx.batch(probs)
    b.upload_boot(idx, vary, best=res.best, pred=res.pred, resid=res.resid)
    b.run_boot()
    rows_s, _ = b.download_boot()
    b.close()
    rel = np.abs(rows_s[:, :, :2] - rows_e[:, :, :2]) / np.abs(rows_e[:, :, :2])
    assert np.mean((rel <= 1e-6).all(axis=2)) >= 0.99
    assert np.mean((rows_s[:, :, :4] == rows_e[:, :, :4]).all(axis=2)) >= 0.9
