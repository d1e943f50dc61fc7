"""The observed divergence (abfit_divergence and its device / multi-device variants) against an exact reference that
shares no code with the kernels: one-hot status masks and float64 matrix products instead of the kernels' thermometer
bit-planes and popcounts, exactly rounded sums instead of the kernels' summation trees.

* integers (diff, cnt, nvalid) and D = diff / (2 cnt) are compared bit for bit on every path;
* methsum is compared bit for bit where the exact sum is representable (meth levels k / 1024) and otherwise against a
  bound derived from the summation tree of the path that produced it; p0uu is checked bit for bit as the reference's
  sequential formula (src/pedigree.rs:179-183) applied to the kernel's own methsum / nvalid;
* at full scale (200 x 5 M sites: every one of the 19 900 pairs), at the packed 16-bit counters' limit, on NaN / inf /
  threshold-equal / subnormal / signed-zero inputs, at the shape boundaries of the kernel choice, on unaligned device
  pointers, and across devices (window-sharded = one device, byte for byte)."""
import math
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, resolve_golden

SITE_CHUNK = 1 << 20   # sites per matrix product: every partial sum is an integer below 2^53
EXACT_MAX = 65536      # windows up to this many sites sum meth_lvl sequentially (abfit_divergence.cu)
U = 2.0 ** -53         # unit roundoff of float64


# ---------------------------------------------------------------------------------------------
# the exact reference
# ---------------------------------------------------------------------------------------------
def ref_pairs(status, post, thr):
    """(diff, cnt) [P] uint64 for the pairs i < j in row-major order, exactly.  status / post: numpy arrays or torch
    tensors (any device).  V = post >= thr, O_x = V & (status == x); cnt = V V^T, diff = sum_{x,y} |x - y| O_x O_y^T as
    float64 matrix products over chunks of at most 2^20 sites (each product is an exact integer), chunks added as int64."""
    is_np = isinstance(status, np.ndarray)
    S, L = status.shape
    if is_np:
        f64, i64 = (lambda m: m.astype(np.float64)), (lambda m: m.astype(np.int64))
        cnt, diff = np.zeros((S, S), np.int64), np.zeros((S, S), np.int64)
    else:
        import torch
        f64, i64 = (lambda m: m.to(torch.float64)), (lambda m: m.to(torch.int64))
        cnt = torch.zeros((S, S), dtype=torch.int64, device=status.device)
        diff = torch.zeros((S, S), dtype=torch.int64, device=status.device)
    for a in range(0, L, SITE_CHUNK):
        st, V = status[:, a:a + SITE_CHUNK], post[:, a:a + SITE_CHUNK] >= thr
        O = [f64(V & (st == x)) for x in range(3)]
        Vf = f64(V)
        c = Vf @ Vf.T
        d = sum(abs(x - y) * (O[x] @ O[y].T) for x in range(3) for y in range(3) if x != y)
        for m in (c, d):
            assert bool((m == m.round()).all()) and bool((m >= 0).all())
        cnt += i64(c)
        diff += i64(d)
    if not is_np:
        cnt, diff = cnt.cpu().numpy(), diff.cpu().numpy()
    iu = np.triu_indices(S, 1)
    return diff[iu].astype(np.uint64), cnt[iu].astype(np.uint64)


def ref_D(diff, cnt):
    with np.errstate(divide="ignore", invalid="ignore"):
        return diff.astype(np.float64) / (2.0 * cnt.astype(np.float64))  # src/pedigree.rs:257 (0/0 -> NaN)


def exact_sum(x):
    """the exactly rounded sum of x (IEEE semantics for NaN / inf: NaN if any NaN or both infinities)"""
    x = np.asarray(x, dtype=np.float64)
    if np.isnan(x).any() or (np.isposinf(x).any() and np.isneginf(x).any()):
        return math.nan
    if np.isinf(x).any():
        return float(x[np.isinf(x)][0])
    return math.fsum(x)


def ref_samples(post, meth, thr):
    """per sample: nvalid, the exact methsum and sum |meth| over the valid sites (numpy)"""
    V = post >= thr
    nv = V.sum(axis=1).astype(np.int64)
    ms = np.array([exact_sum(meth[s][V[s]]) for s in range(len(post))])
    ab = np.array([exact_sum(np.abs(meth[s][V[s]])) for s in range(len(post))])
    return nv, ms, ab


def seq_sum(x):
    """sequential sum in site order (the reference's own fold, src/pedigree.rs:171-172)"""
    with np.errstate(invalid="ignore"):
        return float(np.cumsum(x)[-1]) + 0.0 if len(x) else 0.0   # + 0.0: the fold starts at +0.0


def ref_p0uu(methsum, nvalid):
    """src/pedigree.rs:179-183: sum over samples, in sample order, of 1 - methsum / nvalid, over S"""
    acc = np.float64(0.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        for m, n in zip(methsum, nvalid):
            acc += np.float64(1.0) - np.float64(m) / np.float64(n)
        return float(acc / np.float64(len(methsum)))


def same(a, b):
    """bit for bit, NaN = NaN"""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=a.dtype.kind == "f")


def ceil_div(a, b):
    return -(-a // b)


def gamma(h):
    return h * U / (1 - h * U)


def sum_depth(path, n, n_ctx=3):
    """the most roundings any term of a window of n sites goes through in `path`'s meth_lvl sum (a term added to 0.0
    counts as one rounding too): |sum - exact| <= gamma(depth) * sum |x| (recursive summation in any tree)
      exact : one sequential pass                                    n
      pack  : 128 sites per lane and 64-word block, 5 shuffle levels, blocks added in order
      fused : 16 sites per lane and 512-site group, 5 shuffle levels, per thread ceil(groups / 256) groups, 8 tree levels
      site  : a site-sharded call: one of the above on each device's share of whole words, then the n_ctx device
              sums added in order"""
    words = ceil_div(n, 64)
    if path == "site":
        share = ceil_div(words, n_ctx) * 64
        return max(sum_depth("pack", share), sum_depth("fused", share)) + n_ctx
    if path == "exact" or n <= EXACT_MAX:
        return n
    if path == "pack":
        return 128 + 5 + ceil_div(words, 64)
    return 16 + 5 + ceil_div(ceil_div(words, 8), 256) + 8


def check_window(got, w, status, post, meth, thr, path, bitwise_sums=False, n_ctx=3):
    """window w of a dmatrix() result against the reference on the window's [S][n] arrays"""
    diff, cnt = ref_pairs(status, post, thr)
    assert same(got["diff"][w], diff), "diff"
    assert same(got["cnt"][w], cnt), "cnt"
    assert same(got["D"][w], ref_D(diff, cnt)), "D"
    nv, ms, ab = ref_samples(post, meth, thr)
    assert same(got["nvalid"][w], nv), "nvalid"
    check_methsum(got["methsum"][w], ms, ab, post, meth, thr, path, bitwise_sums, n_ctx)
    assert same(got["p0uu"][w], ref_p0uu(got["methsum"][w], got["nvalid"][w])), "p0uu"


def check_methsum(got, ms, ab, post, meth, thr, path, bitwise=False, n_ctx=3):
    n = post.shape[1]
    for s in range(len(ms)):
        if bitwise:
            assert same(got[s], ms[s]), ("methsum", s, got[s], ms[s])
        elif not np.isfinite(ms[s]):
            assert same(got[s], ms[s]), ("methsum", s, got[s], ms[s])
        else:
            bound = (gamma(sum_depth(path, n, n_ctx)) + U) * ab[s] * (1 + 4 * U)
            assert abs(got[s] - ms[s]) <= bound, ("methsum", s, got[s], ms[s], bound)
        if path == "exact" or (n <= EXACT_MAX and path != "site"):
            assert same(got[s], seq_sum(meth[s][post[s] >= thr])), ("methsum not the sequential sum", s)


def synth(rng, S, L, dyadic=False):
    status = rng.choice(np.array([0, 1, 2], dtype=np.uint8), size=(S, L), p=[0.6, 0.1, 0.3])
    post = np.where(rng.random((S, L)) < 0.85, 0.9999, rng.uniform(0.5, 0.995, (S, L)))
    meth = rng.integers(0, 1025, (S, L)) / 1024.0 if dyadic else rng.random((S, L))
    return status, post, meth


# ---------------------------------------------------------------------------------------------
# CPU: the reference equals the oracle (after which it may judge the kernels)
# ---------------------------------------------------------------------------------------------
def adversarial(rng, S, L):
    status, post, meth = synth(rng, S, L)
    thr = 0.99
    specials = [np.nan, np.inf, -np.inf, thr, np.nextafter(thr, -np.inf), 5e-324, -0.0, 0.0, 1.0]
    k = rng.random((S, L)) < 0.3
    post[k] = rng.choice(specials, k.sum())
    mk = rng.random((S, L)) < 0.02
    meth[mk] = rng.choice([np.nan, np.inf, -np.inf, -0.0, 5e-324], mk.sum())
    return status, post, meth


@pytest.mark.parametrize("thr", [0.99, 0.0, 1.0, np.inf, -np.inf, np.nan, 5e-324, -0.0])
def test_reference_equals_oracle(oracle, thr):
    rng = np.random.default_rng(11)
    cases = [synth(rng, 7, 3001), adversarial(rng, 9, 2049), adversarial(rng, 2, 1), adversarial(rng, 1, 100)]
    # all sites valid and maximal distances: alternating rows of 0 and 2
    st = np.zeros((4, 700), np.uint8)
    st[1::2] = 2
    cases.append((st, np.ones((4, 700)), st / 2.0))
    for status, post, meth in cases:
        D, diff, cnt = oracle.dmatrix(status, post, thr)
        rd, rc = ref_pairs(status, post, thr)
        assert same(rd, diff) and same(rc, cnt) and same(ref_D(rd, rc), D)
        p0, rcs, nv = oracle.p0uu(post, meth, thr)
        rnv, _, _ = ref_samples(post, meth, thr)
        assert same(rnv, nv)
        seq = [seq_sum(meth[s][post[s] >= thr]) for s in range(len(post))]
        with np.errstate(divide="ignore", invalid="ignore"):
            assert same(np.array(seq) / nv.astype(np.float64), rcs)
        assert same(ref_p0uu(seq, nv), p0)


# ---------------------------------------------------------------------------------------------
# GPU
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


def to_dev(*xs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in xs]


def device_run(ctx, status, post, meth, thr, seg=None):
    d = to_dev(status, post, meth)
    S, L = status.shape
    return ctx.dmatrix_device(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), S, L, thr, seg_offsets=seg)


def edge_inputs(rng, S, L, thr):
    """posteriors at NaN, +-inf, thr, just below thr, subnormal, +-0.0; meth NaN / inf on filtered and on valid sites"""
    status, post, meth = synth(rng, S, L)
    specials = [np.nan, np.inf, -np.inf, 5e-324, -5e-324, 0.0, -0.0, 1.0]
    if np.isfinite(thr):
        specials += [thr, np.nextafter(thr, -np.inf)]
    k = rng.random((S, L)) < 0.2
    post[k] = rng.choice(specials, k.sum())
    with np.errstate(invalid="ignore"):
        invalid = ~(post >= thr)
    # NaN / inf meth on filtered sites everywhere: they must never reach methsum
    f = invalid & (rng.random((S, L)) < 0.5)
    meth[f] = rng.choice([np.nan, np.inf, -np.inf], f.sum())
    # on valid sites: sample 1 gets one NaN, sample 2 one +inf, sample 3 +inf and -inf
    for s, vals in ((1, [np.nan]), (2, [np.inf]), (3, [np.inf, -np.inf])):
        idx = np.flatnonzero(~invalid[s])
        if len(idx) >= len(vals):
            meth[s, rng.choice(idx, len(vals), replace=False)] = vals
    return status, post, meth


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [0.99, 0.0, 1.0, np.inf, -np.inf, np.nan])
def test_edge_inputs_every_path(ab, ctx, ctx_pool, monkeypatch, thr):
    """edge posteriors, thresholds and meth values through every path: exact short windows, long two-pass (back to back
    and chunk-overlapped), k_fused, dmatrix_device, window- and site-sharded dmatrix_multi"""
    rng = np.random.default_rng(404)
    S, L = 9, 70_001
    status, post, meth = edge_inputs(rng, S, L, thr)
    seg = [0, 1000, 5000, 5001, 70_001]   # every window <= 65 536 sites: the exact path
    runs = {}
    runs["fused"] = (device_run(ctx, status, post, meth, thr), "fused")
    assert runs["fused"][0]["launches"] <= 4, "k_fused did not run"
    runs["host_fused"] = (ctx.dmatrix(status, post, meth, thr), "fused")
    monkeypatch.setenv("ABFIT_DEV_DIV_FUSED", "0")
    for chunks in ("1", "2", "5"):
        monkeypatch.setenv("ABFIT_DEV_DIV_CHUNKS", chunks)
        runs["pack" + chunks] = (ctx.dmatrix(status, post, meth, thr), "pack")
    monkeypatch.delenv("ABFIT_DEV_DIV_CHUNKS")
    runs["device_pack"] = (device_run(ctx, status, post, meth, thr), "pack")
    monkeypatch.delenv("ABFIT_DEV_DIV_FUSED")
    runs["site_sharded"] = (ab.dmatrix_multi(ctx_pool, status, post, meth, thr), "site")
    for name, (got, path) in runs.items():
        try:
            check_window(got, 0, status, post, meth, thr, path, n_ctx=len(ctx_pool))
        except AssertionError as e:
            raise AssertionError(f"{name}: {e}") from e
    win = ctx.dmatrix(status, post, meth, thr, seg)
    many = ab.dmatrix_multi(ctx_pool, status, post, meth, thr, seg)
    for w in range(len(seg) - 1):
        a, b = seg[w], seg[w + 1]
        check_window(win, w, status[:, a:b], post[:, a:b], meth[:, a:b], thr, "exact")
    for k in ("D", "diff", "cnt", "nvalid", "methsum", "p0uu"):
        assert win[k].tobytes() == many[k].tobytes(), k


@pytest.mark.gpu
def test_dyadic_sums_are_exact_on_every_path(ab, ctx, ctx_pool, monkeypatch):
    """meth levels k / 1024: every partial sum of every tree is exact, so methsum and p0uu equal the exact reference
    bit for bit whatever the path"""
    rng = np.random.default_rng(8)
    S, L = 13, 200_003
    status, post, meth = synth(rng, S, L, dyadic=True)
    got = [ctx.dmatrix(status, post, meth, 0.99), ab.dmatrix_multi(ctx_pool, status, post, meth, 0.99)]
    monkeypatch.setenv("ABFIT_DEV_DIV_FUSED", "0")
    got.append(ctx.dmatrix(status, post, meth, 0.99))
    for g in got:
        check_window(g, 0, status, post, meth, 0.99, "site", bitwise_sums=True)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["fused", "pack", "site"])
def test_non_dyadic_sums_within_the_tree_bound(ab, ctx, ctx_pool, monkeypatch, path):
    """23 x 330 007 sites of U(0, 1) meth levels: methsum within gamma(depth) sum|x| of the exactly rounded sum, depth
    from the path's summation tree (sum_depth); integers and D exact"""
    rng = np.random.default_rng(330)
    S, L = 23, 330_007
    status, post, meth = synth(rng, S, L)
    if path == "site":
        got = ab.dmatrix_multi(ctx_pool, status, post, meth, 0.99)
    else:
        monkeypatch.setenv("ABFIT_DEV_DIV_FUSED", "1" if path == "fused" else "0")
        got = device_run(ctx, status, post, meth, 0.99)
        assert (got["launches"] <= 4) == (path == "fused")
    check_window(got, 0, status, post, meth, 0.99, path, n_ctx=len(ctx_pool))


# ---------------------------------------------------------------------------------------------
# the packed 16-bit counters at their limit
# ---------------------------------------------------------------------------------------------
def alternating(S, L):
    """all sites valid, rows alternately all 0 and all 2: diff = 2 per site for pairs of unlike rows"""
    status = np.zeros((S, L), np.uint8)
    status[1::2] = 2
    return status, np.ones((S, L)), status / 2.0


def check_alternating(got, w, S, n):
    i, j = np.triu_indices(S, 1)
    unlike = (i % 2) != (j % 2)
    assert same(got["cnt"][w], np.full(len(i), n, np.uint64)), "cnt"
    assert same(got["diff"][w], np.where(unlike, 2 * n, 0).astype(np.uint64)), "diff"
    assert same(got["D"][w], np.where(unlike, 1.0, 0.0)), "D"
    assert same(got["nvalid"][w], np.full(S, n, np.int64))
    assert same(got["methsum"][w], np.where(np.arange(S) % 2 == 1, float(n), 0.0))
    assert same(got["p0uu"][w], ref_p0uu(got["methsum"][w], got["nvalid"][w]))


@pytest.mark.gpu
def test_counter_extremes_two_pass(ab, ctx):
    """pair items of the two-pass path hold at most 256 words (16 384 sites); windows of k * 16 384 and k * 16 384 +- 1
    sites, enough of them that the items reach 256 words, starting inside the rows"""
    S = 6
    lens = [16_384 * k + d for k in (1, 2, 3) for d in (-1, 0, 1)] * 17
    seg = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64) + 5
    L = int(seg[-1]) + 3
    status, post, meth = alternating(S, L)
    got = ctx.dmatrix(status, post, meth, 0.99, seg)
    for w, n in enumerate(lens):
        check_alternating(got, w, S, n)


@pytest.mark.gpu
@pytest.mark.parametrize("grid", ["1", "3"])
def test_counter_extremes_fused(ab, ctx, monkeypatch, grid):
    """k_fused flushes its packed counters every 32 groups (16 384 sites); with one or three CTAs every CTA runs
    through several full flush periods (staggered by the CTA index); whole rows and windows inside the rows"""
    S = 7
    monkeypatch.setenv("ABFIT_DEV_DIV_FUSED_GRID", grid)
    for n in (5 * 16_384 - 1, 5 * 16_384, 5 * 16_384 + 1, 9 * 16_384):
        status, post, meth = alternating(S, n + 40)
        whole = device_run(ctx, status[:, :n], post[:, :n], meth[:, :n], 0.99)
        inside = device_run(ctx, status, post, meth, 0.99, seg=[17, 17 + n])
        for got in (whole, inside):
            assert got["launches"] <= 4
            check_alternating(got, 0, S, n)


# ---------------------------------------------------------------------------------------------
# shape boundaries
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_one_sample(ab, ctx, ctx_pool):
    """S = 1: no pairs; nvalid, methsum and p0uu alone are defined"""
    rng = np.random.default_rng(1)
    for L in (1, 1000, 70_001):
        status, post, meth = synth(rng, 1, L)
        for got, path in ((ctx.dmatrix(status, post, meth, 0.99), "pack"), (device_run(ctx, status, post, meth, 0.99), "pack"),
                          (ab.dmatrix_multi(ctx_pool, status, post, meth, 0.99), "site"),
                          (ab.dmatrix_multi(ctx_pool, status, post, meth, 0.99, [0, L]), "pack")):
            assert got["D"].shape == (1, 0) and got["diff"].shape == (1, 0)
            check_window(got, 0, status, post, meth, 0.99, path, n_ctx=len(ctx_pool))


@pytest.mark.gpu
@pytest.mark.parametrize("S", [2, 200, 201])
def test_sample_counts_around_the_fused_limit(ab, ctx, S):
    """k_fused takes up to 200 samples; 201 is the first that takes the two-pass path"""
    rng = np.random.default_rng(S)
    L = 70_001
    status, post, meth = synth(rng, S, L)
    got = device_run(ctx, status, post, meth, 0.99)
    assert (got["launches"] <= 4) == (S <= 200)
    diff, cnt = ref_pairs(*to_dev(status, post), 0.99)
    assert same(got["diff"][0], diff) and same(got["cnt"][0], cnt) and same(got["D"][0], ref_D(diff, cnt))
    nv, ms, ab_ = ref_samples(post, meth, 0.99)
    assert same(got["nvalid"][0], nv)
    check_methsum(got["methsum"][0], ms, ab_, post, meth, 0.99, "fused" if S <= 200 else "pack")
    assert same(got["p0uu"][0], ref_p0uu(got["methsum"][0], got["nvalid"][0]))


@pytest.mark.gpu
def test_largest_sample_count_of_the_pair_kernel(ab, ctx):
    """the pair kernel stages Sp x 24 bytes per word in at most 200 KiB of shared memory: S = 8528 is the largest S it
    takes (Sp = 8530), S = 8529 (Sp = 8534) is refused with ABFIT_ERR_TOO_LARGE"""
    rng = np.random.default_rng(8528)
    S, L = 8528, 200
    status, post, meth = synth(rng, S, L)
    got = ctx.dmatrix(status, post, meth, 0.99)
    diff, cnt = ref_pairs(*to_dev(status, post), 0.99)
    assert same(got["diff"][0], diff) and same(got["cnt"][0], cnt) and same(got["D"][0], ref_D(diff, cnt))
    nv, ms, ab_ = ref_samples(post, meth, 0.99)
    assert same(got["nvalid"][0], nv)
    check_methsum(got["methsum"][0], ms, ab_, post, meth, 0.99, "exact")
    status, post, meth = synth(rng, S + 1, L)
    with pytest.raises(ab.AbfitError) as e:
        ctx.dmatrix(status, post, meth, 0.99)
    assert e.value.code == ab.ERR_TOO_LARGE
    small = synth(rng, 3, 100)   # the context is still usable
    assert same(ctx.dmatrix(*small, 0.99)["cnt"][0], ref_pairs(small[0], small[1], 0.99)[1])


@pytest.mark.gpu
def test_windows_around_the_exact_limit(ab, ctx):
    """65 536 sites: the sequential (reference-order) sum; 65 537: a blocked tree, k_fused alone, the two-pass path
    beside a short window"""
    rng = np.random.default_rng(65536)
    S = 5
    status, post, meth = synth(rng, S, 65_536 + 65_537)
    cases = [([0, 65_536], ["exact"]), ([65_536, 131_073], ["fused"]), ([0, 65_536, 131_073], ["exact", "pack"])]
    for seg, paths in cases:
        got = device_run(ctx, status, post, meth, 0.99, seg)
        assert (got["launches"] == 4 * len(paths)) == (paths == ["fused"])
        for w, path in enumerate(paths):
            a, b = seg[w], seg[w + 1]
            check_window(got, w, status[:, a:b], post[:, a:b], meth[:, a:b], 0.99, path)


@pytest.mark.gpu
@pytest.mark.parametrize("W", [64, 65])
def test_64_and_65_long_windows(ab, ctx, W):
    """k_fused runs once per window for up to 64 long windows; 65 take the two-pass path"""
    rng = np.random.default_rng(W)
    S, n = 4, 66_000
    status, post, meth = synth(rng, S, W * n + 3)
    seg = [3 + w * n for w in range(W + 1)]
    got = device_run(ctx, status, post, meth, 0.99, seg)
    path = "fused" if W <= 64 else "pack"
    assert (got["launches"] == 4 * W) == (W <= 64)
    for w in range(W):
        a, b = seg[w], seg[w + 1]
        check_window(got, w, status[:, a:b], post[:, a:b], meth[:, a:b], 0.99, path)


@pytest.mark.gpu
@pytest.mark.parametrize("fused", ["1", "0"])
def test_unaligned_device_pointers(ab, ctx, monkeypatch, fused):
    """dmatrix_device on views inside larger allocations: f64 arrays 8 bytes and u8 arrays 1, 7 and 15 bytes past a
    16-byte boundary (k_fused rounds its bulk copies from the base pointers), even and odd L"""
    import torch
    monkeypatch.setenv("ABFIT_DEV_DIV_FUSED", fused)
    rng = np.random.default_rng(15)
    S = 5
    for L in (70_000, 70_001):
        status, post, meth = synth(rng, S, L)
        n = S * L
        for o8, o1 in ((1, 1), (0, 7), (1, 15), (1, 0)):
            bst = torch.zeros(n + 32, dtype=torch.uint8, device="cuda")
            bpo = torch.zeros(n + 4, dtype=torch.float64, device="cuda")
            bme = torch.zeros(n + 4, dtype=torch.float64, device="cuda")
            assert bst.data_ptr() % 16 == 0 and bpo.data_ptr() % 16 == 0 and bme.data_ptr() % 16 == 0
            st, po, me = bst[o1:o1 + n], bpo[o8:o8 + n], bme[o8:o8 + n]
            st.copy_(torch.from_numpy(status.ravel()))
            po.copy_(torch.from_numpy(post.ravel()))
            me.copy_(torch.from_numpy(meth.ravel()))
            torch.cuda.synchronize()
            got = ctx.dmatrix_device(st.data_ptr(), po.data_ptr(), me.data_ptr(), S, L, 0.99)
            assert (got["launches"] <= 4) == (fused == "1")
            check_window(got, 0, status, post, meth, 0.99, "fused" if fused == "1" else "pack")


# ---------------------------------------------------------------------------------------------
# several devices = one device
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("lens", [[70_001, 70_001, 500], [66_000] * 65, [67_000] * 100, [1, 70_000, 64, 65_537, 3000, 80_000, 0, 65_536],
                                  [200_000]], ids=["two_long_one_short", "65_long", "100_long", "mixed", "one_window"])
def test_window_sharded_equals_one_device(ab, ctx, ctx_pool, lens):
    """dmatrix_multi with seg_offsets returns ctx.dmatrix's bytes for every output: every shard sums meth_lvl in the
    tree one device picks for the whole window list, and a single window stays on one device"""
    rng = np.random.default_rng(len(lens))
    S = 3 if len(lens) > 64 else 6
    seg = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64) + 2
    status, post, meth = synth(rng, S, int(seg[-1]) + 1)
    one = ctx.dmatrix(status, post, meth, 0.99, seg)
    many = ab.dmatrix_multi(ctx_pool, status, post, meth, 0.99, seg)
    for k in ("D", "diff", "cnt", "nvalid", "methsum", "p0uu"):
        assert one[k].tobytes() == many[k].tobytes(), k
    for w in (0, len(lens) - 1):
        a, b = seg[w], seg[w + 1]
        path = "fused" if len(lens) <= 64 and min(lens) > EXACT_MAX else "pack"
        check_window(one, w, status[:, a:b], post[:, a:b], meth[:, a:b], 0.99, path)


# ---------------------------------------------------------------------------------------------
# full scale: BASELINE configs[4], 200 samples x 5 000 000 sites, all 19 900 pairs
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def c5(ab):
    import torch
    S, L = 200, 5_000_000
    dev = torch.device("cuda", 0)
    if torch.cuda.mem_get_info(dev)[0] < 40e9:
        pytest.skip("needs 40 GB of free device memory")
    g = torch.Generator(device=dev)
    g.manual_seed(5)
    status = (torch.rand((S, L), device=dev, generator=g) * 3).to(torch.uint8).clamp_(max=2)
    post = torch.empty((S, L), dtype=torch.float64, device=dev)
    kmeth = torch.empty((S, L), dtype=torch.int16, device=dev)
    for s in range(S):  # row by row: no (S, L) temporaries
        u = torch.rand(L, device=dev, generator=g, dtype=torch.float64)
        post[s] = torch.where(torch.rand(L, device=dev, generator=g) < 0.9, torch.full_like(u, 0.9999), u * 0.49 + 0.5)
        kmeth[s] = torch.randint(0, 1025, (L,), device=dev, generator=g, dtype=torch.int16)
    meth = torch.empty((S, L), dtype=torch.float64, device=dev)
    for s in range(S):
        meth[s] = kmeth[s].to(torch.float64) / 1024.0
    diff, cnt = ref_pairs(status, post, 0.99)
    V = post >= 0.99
    nvalid = V.sum(dim=1).cpu().numpy().astype(np.int64)
    ksum = torch.zeros(S, dtype=torch.int64, device=dev)
    for s in range(S):
        ksum[s] = torch.where(V[s], kmeth[s].to(torch.int64), 0).sum()
    del V, kmeth
    methsum = ksum.cpu().numpy().astype(np.float64) / 1024.0   # exact: the integer sums are below 2^53
    torch.cuda.synchronize()  # the library's stream does not wait for torch's: the inputs must be complete first
    yield {"S": S, "L": L, "status": status, "post": post, "meth": meth, "diff": diff, "cnt": cnt, "nvalid": nvalid,
           "methsum": methsum}
    torch.cuda.empty_cache()


def check_c5(got, c):
    assert same(got["diff"][0], c["diff"]) and same(got["cnt"][0], c["cnt"])
    assert same(got["D"][0], ref_D(c["diff"], c["cnt"]))
    assert same(got["nvalid"][0], c["nvalid"]) and same(got["methsum"][0], c["methsum"])
    assert same(got["p0uu"][0], ref_p0uu(c["methsum"], c["nvalid"]))


@pytest.mark.gpu
@pytest.mark.parametrize("fused", ["1", "0"])
def test_c5_full_size_against_the_exact_reference(ab, ctx, c5, monkeypatch, fused):
    """k_fused (default) and the two-pass path on all 19 900 pairs: integers and D exact, methsum / p0uu bit for bit"""
    monkeypatch.setenv("ABFIT_DEV_DIV_FUSED", fused)
    got = ctx.dmatrix_device(c5["status"].data_ptr(), c5["post"].data_ptr(), c5["meth"].data_ptr(), c5["S"], c5["L"], 0.99)
    assert (got["launches"] <= 4) == (fused == "1")
    check_c5(got, c5)


@pytest.mark.gpu
def test_c5_full_size_site_sharded(ab, ctx_pool, c5):
    """the site-sharded dmatrix_multi (host arrays, 17 GB) on all 19 900 pairs"""
    if os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_AVPHYS_PAGES") < 64e9:
        pytest.skip("needs 64 GB of free host memory")
    host = [c5[k].cpu().numpy() for k in ("status", "post", "meth")]
    got = ab.dmatrix_multi(ctx_pool, *host, 0.99)
    check_c5(got, c5)


# ---------------------------------------------------------------------------------------------
# NaN / inf posteriors end to end: methylome files -> abfit_pedigree_build and the alphabeta CLI
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_nan_posteriors_end_to_end(ab, ctx, oracle, monkeypatch, tmp_path):
    """the example methylomes with posteriorMax nan / inf / -inf / NaN on some CG lines and rc.meth.lvl nan / inf on
    some filtered lines: pedigree and p0uu of abfit_pedigree_build and of the alphabeta CLI equal the oracle's"""
    mdir = os.path.join(tmp_path, "data", "methylome")
    os.makedirs(mdir)
    words = ["nan", "inf", "-inf", "NaN", "0.99", "infinity"]
    n_changed = 0
    for i, name in enumerate(sorted(os.listdir(os.path.join(GOLDEN, "methylome")))):
        lines = open(os.path.join(GOLDEN, "methylome", name)).read().split("\n")
        for k in range(1, len(lines)):
            f = lines[k].split("\t")
            if len(f) < 10 or f[3] != "CG":
                continue
            if (k + i) % 9 == 0:
                f[6] = words[(k // 9) % len(words)]
                n_changed += 1
            elif (k + i) % 13 == 0:
                f[6], f[8] = "0.5", ["nan", "inf", "-inf"][k % 3]   # filtered: its meth level must not count
            lines[k] = "\t".join(f)
        open(os.path.join(mdir, name), "w").write("\n".join(lines))
    assert n_changed > 20
    monkeypatch.chdir(tmp_path)
    nodes, edges = os.path.join(GOLDEN, "nodelist.txt"), os.path.join(GOLDEN, "edgelist.txt")
    ped, p0uu, _ = ab.build_pedigree(ctx, nodes, edges, 0.99)
    want, want_p0, _ = oracle.build_pedigree(nodes, edges, 0.99, lambda p: os.path.join(tmp_path, p[2:]))
    assert same(ped, want) and same(p0uu, want_p0) and np.isfinite(p0uu)
    clean, clean_p0, _ = oracle.build_pedigree(nodes, edges, 0.99, resolve_golden)
    assert not same(ped, clean) and p0uu != clean_p0   # the edits did change the inputs
    out = os.path.join(tmp_path, "out")
    os.makedirs(out)
    exe = os.path.join(ROOT, "alphabeta-rs_b200", "alphabeta")
    r = subprocess.run([exe, "-n", nodes, "-e", edges, "-i", "20", "-o", out, "--seed", "7"], cwd=tmp_path, capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    ab.write_pedigree(os.path.join(tmp_path, "want.txt"), want)
    assert open(os.path.join(out, "pedigree.txt"), "rb").read() == open(os.path.join(tmp_path, "want.txt"), "rb").read()
    assert "Observed steady state methylation %s\n" % oracle.rust_f64(1.0 - want_p0) in r.stdout


# ---------------------------------------------------------------------------------------------
# metaprofile on several devices, windows of more than 65 536 sites
# ---------------------------------------------------------------------------------------------
def write_long_gene_methylomes(rng, mdir, names, gene_len):
    """one gene on chromosome 1 covered by a CG line at every one of its positions and none outside it: with -w 10 -s 5
    the 19 first gene windows gather ~gene_len / 10 sites each, the last one half as many, the flank windows none"""
    header = ("seqnames\tstart\tstrand\tcontext\tcounts.methylated\tcounts.total\tposteriorMax\tstatus\trc.meth.lvl\t"
              "context.trinucleotide\n")
    pos = np.arange(1000, 1000 + gene_len)
    for name in names:
        n = len(pos)
        st = rng.choice(np.array(["U", "I", "M"]), n, p=[0.6, 0.1, 0.3])
        post = np.where(rng.random(n) < 0.9, "0.9999", np.char.mod("%.4f", rng.uniform(0.5, 0.99, n)))
        lvl = np.char.mod("%.4f", rng.random(n))
        cols = [np.full(n, "1"), pos.astype(str), np.full(n, "+"), np.full(n, "CG"), np.full(n, "0"), np.full(n, "0"), post, st, lvl,
                np.full(n, "CGA")]
        lines = cols[0]
        for c in cols[1:]:
            lines = np.char.add(np.char.add(lines, "\t"), c)
        open(os.path.join(mdir, name), "w").write(header + "\n".join(lines.tolist()) + "\n")


@pytest.mark.gpu
def test_metaprofile_devices_long_windows(ab, tmp_path):
    """`metaprofile --devices` on 19 windows of more than 65 536 sites and one of 35 000 gives the one-device
    results.txt / raw.npy byte for byte (one device takes the two-pass path for the whole window list; so must every
    shard, also those that hold only long windows)"""
    rng = np.random.default_rng(70_000)
    mdir = os.path.join(tmp_path, "methylome")
    os.makedirs(mdir)
    write_long_gene_methylomes(rng, mdir, ["G0.txt", "G1_2.txt", "G4_2.txt", "G4_8.txt"], gene_len=700_000)
    ann = os.path.join(tmp_path, "ann.bed")
    open(ann, "w").write("1\t1000\t701000\tg0\tgbM\t+\n")
    exe = os.path.join(ROOT, "alphabeta-rs_b200", "metaprofile")
    nd = ab.device_count()
    outs = {}
    for devs in ("0", f"0-{nd - 1}" if nd >= 2 else "0,0,0"):
        out = os.path.join(tmp_path, "out_" + devs)
        os.makedirs(out)
        r = subprocess.run([exe, "-m", mdir, "-g", ann, "-w", "10", "-s", "5", "-c", "200", "-o", out, "--name", "long",
                            "--iterations", "20", "--seed", "5", "--devices", devs, "alphabeta",
                            "--nodes", os.path.join(GOLDEN, "nodelist.txt"), "--edges", os.path.join(GOLDEN, "edgelist.txt")],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        outs[devs] = out
    one, many = outs.values()
    dist = [int(x) for x in open(os.path.join(one, "distribution_G0.txt")).read().split()]
    long = [d > EXACT_MAX for d in dist if d > 0]
    assert len(long) == 20 and sum(long) == 19, dist
    for fn in ("results.txt", "raw.npy"):
        assert open(os.path.join(one, fn), "rb").read() == open(os.path.join(many, fn), "rb").read(), fn
