"""The site-block bootstrap (abfit_site_boot_batch): every window's sites are cut into blocks of block_sites consecutive
sites, every replicate draws as many blocks as the window has, with replacement, and its pair divergences are rebuilt
exactly from per-block integer sums, then refitted like the residual bootstrap's replicates.

* CPU: the generator (stream 5) against a Python twin and its invariants; an exact numpy reference of the per-block
  partial sums and of D* (one-hot masks, int64 sums, diff / (2.0 * cnt)) against the oracle's abref_dmatrix; the
  refusals that need no device.
* GPU: dstar_out equals the reference bit for bit (small pedigrees, the golden 4- and 13-sample designs, simulated C5
  at 200 x 1 M sites, unequal and one-site windows, block_sites >= L_w and = 1); the refits equal the oracle bit for bit
  on the stored-tile and the warp-per-fit kernels (named under ABFIT_DEV_VERBOSE); analysis_out = abfit_analyze(rows);
  zero-count replicates; generator keys; host = device entry point; calibration against the across-replicate spread."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN

M64 = (1 << 64) - 1
DBL_EPSILON = 2.220446049250313e-16


# ---------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------
def _mix64(z):
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def py_counts(seed, key, n_boot, n_blocks):
    """multiplicities of the site-block draws, restated from the generator's definition (stream 5)"""
    out = np.zeros((n_boot, n_blocks), dtype=np.uint32)
    h0 = _mix64(_mix64(seed ^ ((5 * 0xD1342543DE82EF95) & M64)) ^ key)
    for b in range(n_boot):
        h1 = _mix64(h0 ^ b)
        for d in range(n_blocks):
            u = (_mix64(h1 ^ d) >> 11) * (1.0 / 9007199254740992.0)
            out[b, min(int(u * n_blocks), n_blocks - 1)] += 1
    return out


def block_bounds(seg, block_sites):
    """per window: the site offsets of its blocks (last block = remainder)"""
    return [np.append(np.arange(seg[p], seg[p + 1], block_sites), seg[p + 1]) for p in range(len(seg) - 1)]


def ref_partials(status, post, thr, lo, hi):
    """(diff, cnt) int64 [P] of sites [lo, hi): one-hot masks, exact integer sums"""
    S = status.shape[0]
    V = (post[:, lo:hi] >= thr).astype(np.int64)
    O = [(V * (status[:, lo:hi] == x)).astype(np.int64) for x in range(3)]
    cnt = V @ V.T
    diff = sum(abs(x - y) * (O[x] @ O[y].T) for x in range(3) for y in range(3) if x != y)
    iu = np.triu_indices(S, 1)
    return diff[iu], cnt[iu]


def pair_index(pairs, S):
    i, j = np.minimum(pairs[:, 0], pairs[:, 1]).astype(np.int64), np.maximum(pairs[:, 0], pairs[:, 1]).astype(np.int64)
    return i * S - i * (i + 1) // 2 + (j - i - 1)


def ref_dstar(status, post, thr, seg, block_sites, pairs_per_window, counts_per_window):
    """D* [n_boot, n_pairs] per window and the NaN replicates, from the numpy partials and the given counts"""
    S = status.shape[0]
    out, nan_reps = [], []
    for p, bb in enumerate(block_bounds(seg, block_sites)):
        parts = [ref_partials(status, post, thr, bb[k], bb[k + 1]) for k in range(len(bb) - 1)]
        dif = np.stack([d for d, _ in parts])
        cnt = np.stack([c for _, c in parts])
        cw = counts_per_window[p].astype(np.int64)
        sd, sc = cw @ dif, cw @ cnt
        j = pair_index(pairs_per_window[p], S)
        with np.errstate(divide="ignore", invalid="ignore"):
            D = sd[:, j].astype(np.float64) / (2.0 * sc[:, j].astype(np.float64))
        out.append(D)
        nan_reps.append(int((sc[:, j] == 0).any(axis=1).sum()))
    return out, np.array(nan_reps)


def adversarial_sites(rng, S, L, thr=0.99):
    status = rng.integers(0, 3, (S, L)).astype(np.uint8)
    post = np.where(rng.random((S, L)) < 0.85, 0.9999, 0.5)
    post[rng.random((S, L)) < 0.05] = np.nan
    post[rng.random((S, L)) < 0.05] = thr  # thr-equal: valid
    return status, post, rng.random((S, L))


# ---------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed,key,n_blocks", [(0, 0, 1), (7, 3, 10), (0xAB0B200, 12345, 97), (2**63 + 5, 2**40, 1000)])
def test_site_boot_counts_are_pinned(ab, seed, key, n_blocks):
    c = ab.gen_site_boot_counts(seed, key, 12, n_blocks)
    assert np.array_equal(c, py_counts(seed, key, 12, n_blocks))
    assert np.all(c.sum(axis=1) == n_blocks)
    # a prefix of replicates does not change with n_boot
    assert np.array_equal(ab.gen_site_boot_counts(seed, key, 5, n_blocks), c[:5])
    if n_blocks > 1:
        assert not np.array_equal(c, ab.gen_site_boot_counts(seed, key + 1, 12, n_blocks))


def test_site_boot_counts_pinned_values(ab):
    assert ab.gen_site_boot_counts(7, 3, 2, 10).tolist() == py_counts(7, 3, 2, 10).tolist()
    assert ab.gen_site_boot_counts(7, 3, 1, 1).tolist() == [[1]]


@pytest.mark.parametrize("case", ["random", "adversarial"])
@pytest.mark.parametrize("block_sites", [1, 17, 64, 250, 10_000])
def test_reference_partials_match_oracle(oracle, case, block_sites):
    rng = np.random.default_rng(block_sites)
    S, L = 6, 600
    if case == "random":
        status = rng.integers(0, 3, (S, L)).astype(np.uint8)
        post = np.where(rng.random((S, L)) < 0.9, 0.9999, 0.6)
    else:
        status, post, _ = adversarial_sites(rng, S, L)
    seg = np.array([0, 1, 200, 451, 600])  # a one-site window, unequal lengths, short last blocks
    for bb in block_bounds(seg, block_sites):
        for k in range(len(bb) - 1):
            d, c = ref_partials(status, post, 0.99, bb[k], bb[k + 1])
            _, od, oc = oracle.dmatrix(status[:, bb[k]:bb[k + 1]], post[:, bb[k]:bb[k + 1]], 0.99)
            assert np.array_equal(d.astype(np.uint64), od) and np.array_equal(c.astype(np.uint64), oc)
    # every block drawn once: D* is the window's observed D
    iu = np.triu_indices(S, 1)
    pairs = np.column_stack(iu)
    nb = [len(bb) - 1 for bb in block_bounds(seg, block_sites)]
    dstar, _ = ref_dstar(status, post, 0.99, seg, block_sites, [pairs] * 4, [np.ones((1, n), np.uint32) for n in nb])
    for p in range(4):
        D, _, _ = oracle.dmatrix(status[:, seg[p]:seg[p + 1]], post[:, seg[p]:seg[p + 1]], 0.99)
        assert np.array_equal(dstar[p][0], D, equal_nan=True)


def _call_site_boot(ab, ctx_h, probs, pairs, status, post, meth, seg, block_sites, best, n_boot=4):
    S, L = status.shape
    rows = np.empty((len(probs), n_boot, 7))
    return ab._lib.abfit_site_boot_batch(ctx_h, ab._pack_problems(probs), len(probs), ab._ptr(pairs), ab._ptr(status),
                                         ab._ptr(post), ab._ptr(meth), S, L, ab._ptr(seg), 0.99, block_sites, ab._ptr(best),
                                         n_boot, 1, 0, None, 100, DBL_EPSILON, 0, ab._ptr(rows), None, None, None, None)


def test_refusals_before_any_device_work(ab):
    rng = np.random.default_rng(0)
    S, L = 4, 100
    status = rng.integers(0, 3, (S, L)).astype(np.uint8)
    post, meth = np.ones((S, L)), np.zeros((S, L))
    ped = np.array([[0, 1, 1, 0.1]] * 6)
    pairs = np.ascontiguousarray(np.column_stack(np.triu_indices(S, 1)), dtype=np.int32)
    probs = [ab.Problem(ped, 0.7, 0.7, 1.0)] * 2
    best = np.zeros(2, dtype=ab.FIT_DTYPE)
    pairs2 = np.ascontiguousarray(np.concatenate([pairs, pairs]))
    seg = np.array([0, 50, 100], dtype=np.int64)
    for bs, msg in ((0, "block_sites"), (-3, "block_sites"), (2**31, "block_sites")):
        assert _call_site_boot(ab, None, probs, pairs2, status, post, meth, seg, bs, best) == -1
        assert msg in ab._lib.abfit_last_error().decode()
    empty = np.array([0, 50, 50], dtype=np.int64)
    assert _call_site_boot(ab, None, probs, pairs2, status, post, meth, empty, 10, best) == -1
    assert "window 1 has no sites" in ab._lib.abfit_last_error().decode()
    bad = pairs2.copy()
    bad[7] = (2, 2)
    assert _call_site_boot(ab, None, probs, bad, status, post, meth, seg, 10, best) == -1
    assert "pedigree row 7" in ab._lib.abfit_last_error().decode()
    bad[7] = (0, S)
    assert _call_site_boot(ab, None, probs, bad, status, post, meth, seg, 10, best) == -1


# ---------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------
def sim_sites(ab, ctx, tree, L, seed, missing=0.0, alpha=3e-3, beta=6e-3):
    return ctx.simulate(tree, alpha, beta, L=L, seed=seed, missing_rate=missing)


def observed_problems(ab, ctx, tree, status, post, meth, seg, thr=0.99):
    dm = ctx.dmatrix(status, post, meth, thr, seg_offsets=seg)
    return [ab.Problem(tree.pedigree(dm["D"][w]), float(dm["p0uu"][w]), float(dm["p0uu"][w]), 1.0)
            for w in range(len(seg) - 1)], dm


def fit_best(ab, ctx, probs, seed=11, n_starts=16, max_iters=3000):
    def max_div(d):
        d = d[~np.isnan(d)]
        return float(d.max()) if d.size else 0.1

    sx = np.stack([ab.gen_start_simplices(seed, p, n_starts, max_div(pb.pedigree[:, 3])) for p, pb in enumerate(probs)])
    return ctx.fit_batch(probs, sx, max_iters=max_iters, want_all=False).best


def check_dstar(ab, res, tree, status, post, seg, block_sites, n_boot, seed, keys):
    pr = tree.pairs()[:, :2].astype(np.int64)
    bb = block_bounds(seg, block_sites)
    counts = [ab.gen_site_boot_counts(seed, int(k), n_boot, len(b) - 1) for k, b in zip(keys, bb)]
    want, nan_reps = ref_dstar(status, post, 0.99, seg, block_sites, [pr] * (len(seg) - 1), counts)
    got = res["dstar"].reshape(len(seg) - 1, n_boot, len(pr))
    for p in range(len(seg) - 1):
        assert np.array_equal(got[p].view(np.uint64), want[p].view(np.uint64)), p
    assert np.array_equal(res["nan_reps"], nan_reps)
    return want


def golden_tree(ab, name):
    if name == "golden4":
        return ab.SimTree.from_files(os.path.join(GOLDEN, "nodelist.txt"), os.path.join(GOLDEN, "edgelist.txt"))
    return ab.SimTree.from_files(os.path.join(GOLDEN, "desired_output", "nodelist.fn"),
                                 os.path.join(GOLDEN, "desired_output", "edgelist.fn"))


@pytest.mark.gpu
@pytest.mark.parametrize("tree_name", ["lines3", "golden4", "golden13"])
@pytest.mark.parametrize("block_sites", [1, 7, 100, 5000])
def test_dstar_equals_reference(ab, ctx, tree_name, block_sites):
    tree = ab.SimTree.lines(3, [1, 2]) if tree_name == "lines3" else golden_tree(ab, tree_name)
    status, post, meth = sim_sites(ab, ctx, tree, 3001, seed=5, missing=0.2)
    seg = np.array([0, 1, 900, 2100, 3001], dtype=np.int64)  # a one-site window, unequal lengths
    probs, dm = observed_problems(ab, ctx, tree, status, post, meth, seg)
    best = fit_best(ab, ctx, probs, max_iters=500)
    n_boot = 19
    res = ctx.site_bootstrap(probs, np.tile(tree.pairs(), (4, 1)), status, post, meth, seg, best, n_boot, 3, block_sites,
                             max_iters=50)
    want = check_dstar(ab, res, tree, status, post, seg, block_sites, n_boot, 3, range(4))
    for p in range(4):
        if block_sites >= seg[p + 1] - seg[p]:  # one block: every replicate is the observed column
            assert np.array_equal(want[p], np.tile(probs[p].pedigree[:, 3], (n_boot, 1)), equal_nan=True)
        bad = np.isnan(want[p]).any(axis=1)
        assert np.all(np.isnan(res["rows"][p][bad])) and np.all(res["fits"]["status"][p][bad] == -1)


@pytest.mark.gpu
def test_dstar_c5_one_million_sites(ab, ctx):
    """200 samples x 1 M sites, 1000-site blocks: all 19 900 pairs of every replicate, against the exact reference on
    the GPU (torch one-hot products per block); the refit is cut short, only D* is checked here"""
    import torch

    tree = ab.SimTree.lines(20, range(1, 11))
    assert tree.n_samples == 200
    L, bs, n_boot = 1_000_000, 1000, 4
    dev = torch.device("cuda", 0)
    st = torch.empty((200, L), dtype=torch.uint8, device=dev)
    po = torch.empty((200, L), dtype=torch.float64, device=dev)
    me = torch.empty((200, L), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    ctx.simulate_device(tree, st.data_ptr(), po.data_ptr(), me.data_ptr(), 3e-3, 6e-3, L=L, seed=9, missing_rate=0.05)
    seg = np.array([0, L], dtype=np.int64)
    dm = ctx.dmatrix_device(st.data_ptr(), po.data_ptr(), me.data_ptr(), 200, L, seg_offsets=seg)
    prob = ab.Problem(tree.pedigree(dm["D"][0]), float(dm["p0uu"][0]), float(dm["p0uu"][0]), 1.0)
    best = np.zeros(1, dtype=ab.FIT_DTYPE)
    best[0]["theta"] = (3e-3, 6e-3, 0.5, 0.0)
    res = ctx.site_bootstrap_device([prob], tree.pairs(), st.data_ptr(), po.data_ptr(), me.data_ptr(), 200, L, seg, best,
                                    n_boot, 21, bs, max_iters=2)
    n_blk = L // bs
    V = po >= 0.99
    O = [(V & (st == x)).to(torch.float64) for x in range(3)]
    Vf = V.to(torch.float64)
    # float64 products of integers below 2^53: exact
    dif = torch.empty((n_blk, 200, 200), dtype=torch.float64, device=dev)
    cnt = torch.empty_like(dif)
    for k in range(n_blk):
        s = slice(k * bs, (k + 1) * bs)
        cnt[k] = Vf[:, s] @ Vf[:, s].T
        dif[k] = sum(abs(x - y) * (O[x][:, s] @ O[y][:, s].T) for x in range(3) for y in range(3) if x != y)
    counts = torch.as_tensor(ab.gen_site_boot_counts(21, 0, n_boot, n_blk).astype(np.float64), device=dev)
    sd = torch.einsum("bk,kij->bij", counts, dif)
    sc = torch.einsum("bk,kij->bij", counts, cnt)
    pr = tree.pairs()[:, :2].astype(np.int64)
    i, j = torch.as_tensor(pr[:, 0], device=dev), torch.as_tensor(pr[:, 1], device=dev)
    assert bool((sd == sd.round()).all()) and float(sd.max()) < 2.0 ** 53
    want = (sd[:, i, j] / (2.0 * sc[:, i, j])).cpu().numpy()
    assert np.array_equal(res["dstar"].reshape(n_boot, -1).view(np.uint64), want.view(np.uint64))


def oracle_rows(oracle, prob, best_theta, dstar, vary, max_iters=1000):
    """the oracle's bootstrap refit of one replicate whose D column is dstar: boot_model with pred = D*, resid = 0 and
    every index 0 (D*_i + 0.0 = D*_i)"""
    n = len(dstar)
    op = oracle.Problem(prob.pedigree, prob.p0uu, prob.eqp, prob.eqp_weight)
    flags = oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL
    return oracle.boot_model(op, best_theta, dstar, np.zeros(n), np.zeros(n, np.int32), vary, max_iters=max_iters,
                             flags=flags)


def check_refits(ab, oracle, probs, best, res, n_boot, seed, keys, check_reps=None, max_iters=1000):
    total = 0
    for p, pb in enumerate(probs):
        n = pb.n_pairs
        ds = res["dstar"][total * n_boot:(total + n) * n_boot].reshape(n_boot, n)
        total += n
        vary = ab.gen_vary_vertices(seed, int(keys[p]), n_boot, best[p]["theta"])
        for b in (range(n_boot) if check_reps is None else check_reps):
            if np.isnan(ds[b]).any():
                continue
            rc, orows, ofits = oracle_rows(oracle, pb, best[p]["theta"], ds[b], vary[b:b + 1], max_iters)
            assert rc == 0
            assert np.array_equal(res["rows"][p, b].view(np.uint64), orows[0].view(np.uint64)), (p, b)
            f = res["fits"][p, b]
            for k in ("theta", "cost", "iters", "evals", "status"):  # the oracle's bootstrap fits carry no lse
                assert np.asarray(f[k]).tobytes() == np.asarray(ofits[0][k]).tobytes(), (p, b, k)
            assert f["start_id"] == b


def run_verbose(monkeypatch, capfd, env, fn):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv("ABFIT_DEV_VERBOSE", "1")
    capfd.readouterr()
    r = fn()
    return r, capfd.readouterr().err


@pytest.mark.gpu
def test_refits_stored_tile_equal_oracle(ab, ctx, oracle, monkeypatch, capfd):
    tree = golden_tree(ab, "golden13")
    status, post, meth = sim_sites(ab, ctx, tree, 40_000, seed=2)
    seg = np.array([0, 15_000, 40_000], dtype=np.int64)
    probs, _ = observed_problems(ab, ctx, tree, status, post, meth, seg)
    best = fit_best(ab, ctx, probs)
    n_boot = 24
    res, err = run_verbose(monkeypatch, capfd, {}, lambda: ctx.site_bootstrap(
        probs, np.tile(tree.pairs(), (2, 1)), status, post, meth, seg, best, n_boot, 17, 250, first_problem_id=40))
    assert "k_fit_boot<BIG=0,DGIVEN=1>" in err and "k_siteboot_dstar" in err
    check_refits(ab, oracle, probs, best, res, n_boot, 17, [40, 41])
    for p in range(2):
        assert np.array_equal(res["analysis"][p].view(np.uint64), ab.analyze(res["rows"][p]).view(np.uint64))


@pytest.mark.gpu
def test_refits_warp_per_fit_equal_oracle(ab, ctx, oracle, monkeypatch, capfd):
    """the warp-per-fit mapping (forced on with ABFIT_DEV_WIDE=1, as for the residual bootstrap) on the C5 pedigree"""
    tree = ab.SimTree.lines(20, range(1, 11))
    status, post, meth = sim_sites(ab, ctx, tree, 20_000, seed=4)
    seg = np.array([0, 20_000], dtype=np.int64)
    probs, _ = observed_problems(ab, ctx, tree, status, post, meth, seg)
    best = np.zeros(1, dtype=ab.FIT_DTYPE)
    best[0]["theta"] = (3e-3, 6e-3, 0.4, 0.01)
    n_boot = 3
    res, err = run_verbose(monkeypatch, capfd, {"ABFIT_DEV_WIDE": "1"}, lambda: ctx.site_bootstrap(
        probs, tree.pairs(), status, post, meth, seg, best, n_boot, 8, 2000, max_iters=1000))
    assert "k_fit_wide<boot,DGIVEN=1>" in err
    check_refits(ab, oracle, probs, best, res, n_boot, 8, [0])


@pytest.mark.gpu
def test_zero_count_replicates_are_not_fitted(ab, ctx, oracle):
    tree = ab.SimTree.lines(2, [1, 2])
    S = tree.n_samples
    status, post, meth = sim_sites(ab, ctx, tree, 1000, seed=6)
    post = post.copy()
    post[0, 100:] = 0.0  # sample 0 has valid sites in block 0 only (100-site blocks)
    seg = np.array([0, 1000], dtype=np.int64)
    probs, _ = observed_problems(ab, ctx, tree, status, post, meth, seg)
    best = fit_best(ab, ctx, probs)
    n_boot = 40
    res = ctx.site_bootstrap(probs, tree.pairs(), status, post, meth, seg, best, n_boot, 12, 100, max_iters=200)
    counts = ab.gen_site_boot_counts(12, 0, n_boot, 10)
    bad = counts[:, 0] == 0
    assert 0 < bad.sum() < n_boot
    assert res["nan_reps"][0] == bad.sum()
    assert np.all(np.isnan(res["rows"][0][bad])) and not np.isnan(res["rows"][0][~bad]).any()
    f = res["fits"][0]
    assert np.all(f["status"][bad] == -1) and np.all(f["iters"][bad] == 0) and np.all(f["start_id"] == np.arange(n_boot))
    check_dstar(ab, res, tree, status, post, seg, 100, n_boot, 12, [0])
    check_refits(ab, oracle, probs, best, res, n_boot, 12, [0], max_iters=200)
    # the context still works
    again = ctx.site_bootstrap(probs, tree.pairs(), status, post, meth, seg, best, n_boot, 12, 100, max_iters=200)
    assert np.array_equal(again["rows"].view(np.uint64), res["rows"].view(np.uint64))


@pytest.mark.gpu
def test_keys_and_device_entry_point(ab, ctx):
    import torch

    tree = golden_tree(ab, "golden13")
    status, post, meth = sim_sites(ab, ctx, tree, 9000, seed=8)
    seg = np.array([0, 3000, 6000, 9000], dtype=np.int64)
    probs, _ = observed_problems(ab, ctx, tree, status, post, meth, seg)
    best = fit_best(ab, ctx, probs)
    pairs = tree.pairs()
    n_boot = 16
    kw = dict(max_iters=300)
    full = ctx.site_bootstrap(probs, np.tile(pairs, (3, 1)), status, post, meth, seg, best, n_boot, 5, 64,
                              problem_ids=[70, 71, 72], **kw)
    one = ctx.site_bootstrap(probs[1:2], pairs, status[:, 3000:6000], post[:, 3000:6000], meth[:, 3000:6000],
                             np.array([0, 3000]), best[1:2], n_boot, 5, 64, problem_ids=[71], **kw)
    assert np.array_equal(one["rows"][0].view(np.uint64), full["rows"][1].view(np.uint64))
    tail = ctx.site_bootstrap(probs[1:], np.tile(pairs, (2, 1)), status, post, meth, np.array([0, 3000, 6000, 9000])[1:],
                              best[1:], n_boot, 5, 64, first_problem_id=71, **kw)
    assert np.array_equal(tail["rows"].view(np.uint64), full["rows"][1:].view(np.uint64))
    dev = torch.device("cuda", 0)
    ts, tp, tm = (torch.as_tensor(a, device=dev).contiguous() for a in (status, post, meth))
    torch.cuda.synchronize()
    d = ctx.site_bootstrap_device(probs, np.tile(pairs, (3, 1)), ts.data_ptr(), tp.data_ptr(), tm.data_ptr(),
                                  status.shape[0], status.shape[1], seg, best, n_boot, 5, 64, problem_ids=[70, 71, 72], **kw)
    for k in ("rows", "analysis", "dstar"):
        assert np.array_equal(d[k].view(np.uint64), full[k].view(np.uint64)), k
    assert np.array_equal(d["fits"].view(np.uint8), full["fits"].view(np.uint8))


@pytest.mark.gpu
def test_too_large_partials_are_refused(ab, ctx):
    """200 samples x 1.2 M one-site blocks: 191 GB of partials, refused before any launch; the context works after"""
    import torch

    tree = ab.SimTree.lines(20, range(1, 11))
    L = 1_200_000
    dev = torch.device("cuda", 0)
    st = torch.zeros((200, L), dtype=torch.uint8, device=dev)
    po = torch.ones((200, L), dtype=torch.float64, device=dev)
    me = torch.zeros((200, L), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    prob = ab.Problem(tree.pedigree(np.full(19900, 0.1)), 0.7, 0.7, 1.0)
    best = np.zeros(1, dtype=ab.FIT_DTYPE)
    with pytest.raises(ab.AbfitError) as e:
        ctx.site_bootstrap_device([prob], tree.pairs(), st.data_ptr(), po.data_ptr(), me.data_ptr(), 200, L,
                                  np.array([0, L]), best, 2, 5, 1)
    assert e.value.code == -5
    del st, po, me
    small = ab.SimTree.lines(3, [1, 2])
    status, post, meth = sim_sites(ab, ctx, small, 2000, seed=1)
    seg = np.array([0, 2000], dtype=np.int64)
    probs, _ = observed_problems(ab, ctx, small, status, post, meth, seg)
    r = ctx.site_bootstrap(probs, small.pairs(), status, post, meth, seg, fit_best(ab, ctx, probs), 8, 5, 1, max_iters=100)
    assert r["rows"].shape == (1, 8, 7) and not np.isnan(r["rows"]).any()


@pytest.mark.gpu
def test_calibration_on_iid_sites(ab, ctx):
    """R = 32 replicates of the R-original design at 500 000 iid sites, 100-site blocks: the median site-bootstrap sd
    of alpha and of beta lies within a factor 2 of the across-replicate sd of the fitted values"""
    tree = golden_tree(ab, "golden13")
    res = ab.design_study([ctx], tree, 3e-3, 6e-3, L=500_000, n_replicates=32, n_starts=32, n_boot=100, seed=13,
                          bootstrap="sites", block_sites=100)
    assert np.all(res["status"] == 0)
    for f in (0, 1):
        true_sd = np.std(res["theta"][:, f], ddof=1)
        boot_sd = np.median(res["analysis"][:, 8 + f])
        print(f"field {f}: across-replicate sd {true_sd:.3e}, median site-bootstrap sd {boot_sd:.3e}")
        assert 0.5 < boot_sd / true_sd < 2.0


# ---------------------------------------------------------------------------------------------
# command-line tools
# ---------------------------------------------------------------------------------------------
def golden_sites(ab, cwd, nodelist, edgelist):
    """the [S, L] site arrays of the golden methylomes, read as the tools read them, and the pedigree's (i, j) rows"""
    files, pairs = ab.pedigree_graph(nodelist, edgelist)
    parsed = [ab.parse_methylome_buffer(open(os.path.join(cwd, f), "rb").read()) for f in files]
    assert len({len(q["status"]) for q in parsed}) == 1
    return (np.stack([q["status"] for q in parsed]), np.stack([q["posteriormax"] for q in parsed]),
            np.stack([q["meth_lvl"] for q in parsed]), pairs)


def _golden_cwd(tmp_path):
    os.makedirs(os.path.join(tmp_path, "data"))
    os.symlink(os.path.join(GOLDEN, "methylome"), os.path.join(tmp_path, "data", "methylome"))
    return str(tmp_path)


@pytest.mark.gpu
def test_alphabeta_cli_site_bootstrap_equals_library(ab, ctx, tmp_path):
    """`alphabeta --site-bootstrap 50` on the golden 4-sample methylomes: raw.npy and analysis.txt are the library's fit +
    site bootstrap on the same seed, and the library's D* on these real methylomes equals the exact reference"""
    import subprocess
    from conftest import ROOT

    cwd = _golden_cwd(tmp_path)
    out = os.path.join(cwd, "out")
    os.makedirs(out)
    nl, el = os.path.join(GOLDEN, "nodelist.txt"), os.path.join(GOLDEN, "edgelist.txt")
    n, seed, bs = 40, 99, 50
    r = subprocess.run([os.path.join(ROOT, "alphabeta-rs_b200", "alphabeta"), "-n", nl, "-e", el, "-i", str(n), "-o", out,
                        "--seed", str(seed), "--site-bootstrap", str(bs)], cwd=cwd, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    old = os.getcwd()
    os.chdir(cwd)
    try:
        ped, p0uu, _ = ab.build_pedigree(ctx, nl, el, 0.99)
        status, post, meth, pairs = golden_sites(ab, cwd, nl, el)
    finally:
        os.chdir(old)
    prob = ab.Problem(ped, p0uu, p0uu, 1.0)
    best = ctx.fit_batch([prob], ab.gen_start_simplices(seed, 0, n, float(ped[:, 3].max()))[None], max_iters=10000,
                         want_all=False).best
    L = status.shape[1]
    res = ctx.site_bootstrap([prob], pairs, status, post, meth, [0, L], best, n, seed, bs)
    assert np.array_equal(np.load(os.path.join(out, "raw.npy")).view(np.uint64), res["rows"][0].view(np.uint64))
    ab.write_analysis(os.path.join(cwd, "lib_analysis.txt"), res["analysis"][0])
    assert open(os.path.join(out, "analysis.txt")).read() == open(os.path.join(cwd, "lib_analysis.txt")).read()
    check_dstar(ab, {"dstar": res["dstar"], "nan_reps": res["nan_reps"]}, _Pairs(pairs), status, post,
                np.array([0, L]), bs, n, seed, [0])


class _Pairs:
    """the pairs() of a pedigree read from files, for check_dstar"""

    def __init__(self, pairs):
        self._p = pairs

    def pairs(self):
        return self._p


GENES = [(1, 300, 700, "-"), (1, 250, 800, "+"), (2, 1200, 1600, "+"), (2, 1250, 1650, "-"), (3, 600, 900, "*"),
         (4, 1200, 1550, "-"), (4, 1150, 1600, "+"), (5, 300, 900, "*"), ("C", 200, 900, "+"), ("C", 150, 950, "-"),
         ("M", 200, 600, "-"), ("M", 150, 650, "+")]


def _metaprofile(tmp_path, meth_dir, extra, n_it=24, seed=777):
    import subprocess
    from conftest import ROOT

    ann = os.path.join(tmp_path, "ann.bed")
    open(ann, "w").write("".join(f"{c}\t{s}\t{e}\tg{i}\tgbM\t{sd}\n" for i, (c, s, e, sd) in enumerate(GENES)))
    out = os.path.join(tmp_path, "out")
    os.makedirs(out, exist_ok=True)
    return out, subprocess.run([os.path.join(ROOT, "alphabeta-rs_b200", "metaprofile"), "-m", meth_dir, "-g", ann, "-w", "10",
                                "-s", "5", "-c", "200", "-o", out, "--name", "sb", "--iterations", str(n_it), "--seed", str(seed),
                                *extra, "alphabeta", "--nodes", os.path.join(GOLDEN, "nodelist.txt"), "--edges",
                                os.path.join(GOLDEN, "edgelist.txt")], capture_output=True, text=True, timeout=300)


def test_metaprofile_site_bootstrap_refusals(oracle, tmp_path):
    """refused before any device work: several devices, and a window whose samples list different numbers of sites"""
    out, r = _metaprofile(tmp_path, os.path.join(GOLDEN, "methylome"), ["--devices", "0-1", "--site-bootstrap", "5"])
    assert r.returncode == 2 and "--site-bootstrap runs on one device" in r.stderr
    meth_dir = os.path.join(tmp_path, "methylome")
    os.makedirs(meth_dir)
    for name in sorted(os.listdir(os.path.join(GOLDEN, "methylome"))):
        lines = open(os.path.join(GOLDEN, "methylome", name)).read().split("\n")
        if name == "G1_2.txt":
            cg = [i for i, l in enumerate(lines) if oracle.parse_methylome_line(l) is not None]
            lines = [l for i, l in enumerate(lines) if i != cg[len(cg) // 3]]
        open(os.path.join(meth_dir, name), "w").write("\n".join(lines))
    out, r = _metaprofile(tmp_path, meth_dir, ["--site-bootstrap", "5", "--device", "99"])
    assert r.returncode == 1 and "list different numbers of sites" in r.stdout, r.stdout + r.stderr
    assert "Error: --site-bootstrap: the samples of window" in r.stdout


@pytest.mark.gpu
def test_metaprofile_cli_site_bootstrap_equals_per_window_library(ab, ctx, oracle, tmp_path):
    """`metaprofile ... --site-bootstrap 3 alphabeta`: every window's bootstrap rows equal the library's fit + site
    bootstrap of that window's sites alone, keyed by the window's position"""
    n_it, seed, bs = 24, 777, 3
    out, r = _metaprofile(tmp_path, os.path.join(GOLDEN, "methylome"), ["--site-bootstrap", str(bs)], n_it, seed)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = np.load(os.path.join(out, "raw.npy"))  # [iteration][column][window]
    ped6, _, info = oracle.build_pedigree(os.path.join(GOLDEN, "nodelist.txt"), os.path.join(GOLDEN, "edgelist.txt"), 0.99,
                                          __import__("conftest").resolve_golden)
    _, pairs = ab.pedigree_graph(os.path.join(GOLDEN, "nodelist.txt"), os.path.join(GOLDEN, "edgelist.txt"))
    strand = {"+": 1, "-": -1, "*": 0}
    og = [(oracle.chromosome_id(str(c)), s, e, strand[sd]) for c, s, e, sd in GENES]
    per_sample = []
    for node in info["nodes"]:
        path = os.path.join(GOLDEN, "methylome", os.path.basename(__import__("conftest").resolve_golden(node["file"])))
        sites, st, po, me = [], [], [], []
        for line in open(path).read().split("\n")[1:]:
            q = oracle.parse_methylome_line(line)
            if q is not None:
                sites.append((oracle.chromosome_id(str(q["chromosome"])), q["start"], q["end"], strand[q["strand"]]))
                st.append(q["status"]); po.append(q["posteriormax"]); me.append(q["meth_lvl"])
        d, assign = oracle.extract_windows(og, sites, window_size=10, window_step=5, cutoff=200)
        per_sample.append((d, assign, np.array(st, dtype=np.uint8), np.array(po), np.array(me)))
    f, checked = 0, 0
    for w in range(len(per_sample[0][0])):
        cols = [[si for si, ww in ps[1] if ww == w] for ps in per_sample]
        if not any(cols):
            continue
        assert len({len(c) for c in cols}) == 1
        status = np.stack([ps[2][c] for ps, c in zip(per_sample, cols)])
        post = np.stack([ps[3][c] for ps, c in zip(per_sample, cols)])
        meth = np.stack([ps[4][c] for ps, c in zip(per_sample, cols)])
        D, _, _ = oracle.dmatrix(status, post, 0.99)
        p0 = oracle.p0uu(post, meth, 0.99)[0]
        if np.isnan(D).any() or np.isnan(p0):
            continue
        ped = ped6.copy()
        ped[:, 3] = D
        prob = ab.Problem(ped, p0, p0, 1.0)
        sx = ab.gen_start_simplices(seed, w, n_it, float(D.max()))[None]
        best = ctx.fit_batch([prob], sx, max_iters=10000, want_all=False).best
        if best[0]["status"] < 0:
            continue
        res = ctx.site_bootstrap([prob], pairs, status, post, meth, [0, status.shape[1]], best, n_it, seed, bs,
                                 problem_ids=[w])
        assert np.array_equal(raw[:, :, f].view(np.uint64), res["rows"][0].view(np.uint64)), w
        f += 1
        checked += 1
    assert checked >= 3 and f == raw.shape[2]
