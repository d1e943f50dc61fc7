"""Epimutation rates in arbitrary genomic regions: BED lines -> site ranges (abfit_parse_region_line,
abfit_region_ranges), the exact per-region observed divergence (abfit_region_divergence) and the `regions` tool.

* CPU: the BED line parser; region_ranges against numpy.searchsorted on random multi-chromosome site lists and its
  refusals; the tool's refusals that come before any device work.
* GPU: every output of every region equals abfit_divergence on the single window {lo, hi} bit for bit (heavy overlap,
  nesting, repeats, empty, one-site and > 65 536-site regions; thr-equal and NaN posteriors; status >= 3; S = 2; 200
  samples x 1 M simulated sites); host = device entry point; permuted regions give permuted outputs; the out-of-memory
  refusal; the tool against the library pipeline, over three contexts, with --site-bootstrap, and on known rates."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

TOOL = os.path.join(ROOT, "alphabeta-rs_b200", "regions")
KEYS = ("D", "diff", "cnt", "p0uu", "methsum", "nvalid")


# ---------------------------------------------------------------------------------------------
# CPU: parser and ranges
# ---------------------------------------------------------------------------------------------
def test_parse_region_line(ab):
    for line in ("", "   ", "\r", "# comment", "#chrom\tstart\tend", "track name=dmr", "browser position chr1:1-100"):
        assert ab.parse_region_line(line) is None, line
    assert ab.parse_region_line("1\t100\t200") == (1, 100, 200)
    assert ab.parse_region_line("chr2\t0\t5\tname") == (2, 0, 5)
    assert ab.parse_region_line("chr3 7 9 name 0") == (3, 7, 9)
    assert ab.parse_region_line("4\t1\t2\tg\t0\t+\r\n") == (4, 1, 2)
    assert ab.parse_region_line("chrM\t0\t1") == (256, 0, 1)
    assert ab.parse_region_line("C\t5\t5") == (257, 5, 5)
    assert ab.parse_region_line("chr255\t0\t4294967295") == (255, 0, 4294967295)
    for line in ("chrom\tstart\tend", "1\t100", "1", "1\tx\t5", "1\t5\t-1", "1\t-3\t5", "1\t1.5\t5", "1\t0\t4294967296",
                 "chr256\t0\t1", "Mt\t0\t1", "1\t10\t9"):
        with pytest.raises(ab.AbfitError) as e:
            ab.parse_region_line(line)
        assert e.value.code < 0, line
    with pytest.raises(ab.AbfitError, match="end < start"):
        ab.parse_region_line("1\t10\t9")


def random_sites(ab, rng, chroms, per_chrom):
    parts = []
    for c in chroms:
        pos = np.sort(rng.integers(1, 5000, per_chrom))
        s = np.zeros(per_chrom, dtype=ab.SITE_DTYPE)
        s["chromosome"], s["start"], s["end"] = c, pos, pos
        parts.append(s)
    return np.concatenate(parts)


def ref_ranges(sites, chrom, start0, end):
    """numpy reference: the sites at 1-based positions start0 + 1 .. end of the region's chromosome"""
    lo, hi = np.zeros(len(chrom), dtype=np.int64), np.zeros(len(chrom), dtype=np.int64)
    for w, (c, a, b) in enumerate(zip(chrom, start0, end)):
        idx = np.flatnonzero(sites["chromosome"] == c)
        if idx.size == 0:
            continue
        pos = sites["start"][idx].astype(np.int64)
        lo[w] = idx[0] + np.searchsorted(pos, a, "right")
        hi[w] = idx[0] + np.searchsorted(pos, b, "right")
    return lo, hi


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_region_ranges_against_searchsorted(ab, seed):
    rng = np.random.default_rng(seed)
    sites = random_sites(ab, rng, [3, 1, 257, 2], 400)  # chromosomes in file order, not sorted; duplicates allowed
    pos = sites["start"].astype(np.int64)
    chrom, start0, end = [], [], []

    def add(c, a, b):
        chrom.append(c), start0.append(a), end.append(b)

    for c in (1, 2, 3, 257):
        cp = pos[sites["chromosome"] == c]
        add(c, 0, int(cp.min()) - 1)              # before the first site
        add(c, int(cp.max()) + 5, int(cp.max()) + 50)  # after the last
        add(c, 0, 10_000)                         # the whole chromosome
        for _ in range(200):
            a = int(rng.integers(0, 5200))
            b = a + int(rng.integers(0, 300))
            add(c, a, b)
            add(c, a, b)                          # identical
            add(c, a + 1, max(a + 1, b - 1))      # nested
            add(c, b, b + 7)                      # touching
            add(c, a, a)                          # zero length
        k = int(rng.integers(1, len(cp) - 1))
        add(c, int(cp[k]) - 1, int(cp[k]))        # exactly one position
        add(c, int(cp[k]), int(cp[k]) + 1)
    for c in (4, 256, 0):                         # chromosomes without sites
        add(c, 0, 100)
    lo, hi = ab.region_ranges(sites, chrom, start0, end)
    rlo, rhi = ref_ranges(sites, np.array(chrom), np.array(start0), np.array(end))
    assert np.array_equal(lo, rlo) and np.array_equal(hi, rhi)
    assert np.all(lo[-3:] == 0) and np.all(hi[-3:] == 0)
    # many regions (the multi-threaded path) give the same ranges
    big = np.tile(np.arange(len(chrom)), 100)
    blo, bhi = ab.region_ranges(sites, np.array(chrom)[big], np.array(start0)[big], np.array(end)[big])
    assert np.array_equal(blo, lo[big]) and np.array_equal(bhi, hi[big])


def test_region_ranges_refusals(ab):
    rng = np.random.default_rng(5)
    sites = random_sites(ab, rng, [1, 2, 3], 50)
    split = np.concatenate([sites[:20], sites[60:], sites[20:60]])  # chromosome 1 split in two runs
    with pytest.raises(ab.AbfitError, match=r"chromosome 1 appears again at site 110"):
        ab.region_ranges(split, [1], [0], [10])
    unsorted = sites.copy()
    unsorted["start"][70], unsorted["start"][71] = 4000, 3  # chromosome 2, sites 70 and 71
    with pytest.raises(ab.AbfitError, match=r"positions decrease on chromosome 2 at site 71"):
        ab.region_ranges(unsorted, [1], [0], [10])
    with pytest.raises(ab.AbfitError, match="end < start"):
        ab.region_ranges(sites, [1], [10], [9])
    with pytest.raises(ValueError):
        ab.region_ranges(sites, [1, 2], [0], [10])


# ---------------------------------------------------------------------------------------------
# GPU: exact per-region divergence
# ---------------------------------------------------------------------------------------------
def device_inputs(status, post, meth):
    import torch

    dev = torch.device("cuda", 0)
    t = (torch.from_numpy(np.ascontiguousarray(status)).to(dev), torch.from_numpy(np.ascontiguousarray(post)).to(dev),
         torch.from_numpy(np.ascontiguousarray(meth)).to(dev))
    torch.cuda.synchronize()
    return t


def check_regions(ctx, tensors, S, L, lo, hi, thr, out, which=None):
    """every (chosen) region's outputs equal dmatrix_device on the window {lo, hi} bit for bit"""
    st, po, me = tensors
    for w in range(len(lo)) if which is None else which:
        ref = ctx.dmatrix_device(st.data_ptr(), po.data_ptr(), me.data_ptr(), S, L, thr, seg_offsets=[lo[w], hi[w]])
        for k in KEYS:
            assert np.array_equal(out[k][w].view(np.uint64) if out[k].dtype == np.float64 else out[k][w],
                                  ref[k][0].view(np.uint64) if ref[k].dtype == np.float64 else ref[k][0]), (k, w, lo[w], hi[w])


def adversarial(rng, S, L, thr):
    status = rng.integers(0, 6, (S, L)).astype(np.uint8)  # values >= 3 count as 2
    post = np.where(rng.random((S, L)) < 0.85, 0.999, 0.5)
    post[rng.random((S, L)) < 0.05] = thr
    post[rng.random((S, L)) < 0.02] = np.nan
    meth = rng.random((S, L))
    meth[post < thr] = np.nan  # never read
    return status, post, meth


def region_set(rng, L):
    lo, hi = [], []
    for a in range(1000, 60_000, 100):  # 1000-site tiles at step 100
        lo.append(a), hi.append(a + 1000)
    for _ in range(150):
        a = int(rng.integers(0, L - 3000))
        b = a + int(rng.integers(0, 3000))
        lo += [a, a, a + 7, b, a]
        hi += [b, b, max(a + 7, b - 5), b, a + 1]  # repeat, nested, empty, one site
    lo += [0, L, 5000, 3, 10, L - 70_000]
    hi += [0, L, 5000 + 65_536, 3 + 65_537, L, L]  # empty at both ends, exactly EXACT_MAX, just above, long ones
    return np.array(lo, dtype=np.int64), np.array(hi, dtype=np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("S", [2, 7, 37])
def test_region_divergence_equals_single_windows(ab, ctx, S):
    rng = np.random.default_rng(S)
    L, thr = 200_000, 0.99
    status, post, meth = adversarial(rng, S, L, thr)
    lo, hi = region_set(rng, L)
    out = ctx.region_divergence(status, post, meth, lo, hi, thr)
    tensors = device_inputs(status, post, meth)
    which = sorted(set(rng.choice(len(lo), 300, replace=False).tolist()) | set(range(len(lo) - 6, len(lo))))
    check_regions(ctx, tensors, S, L, lo, hi, thr, out, which)
    assert np.isnan(out["D"][len(lo) - 6]).all() and np.isnan(out["p0uu"][len(lo) - 6])
    assert (out["cnt"][len(lo) - 6] == 0).all() and (out["nvalid"][len(lo) - 6] == 0).all()
    assert (out["methsum"][len(lo) - 6] == 0).all()
    # the device entry point gives the same bits; a permutation of the regions permutes the outputs
    dev = ctx.region_divergence_device(*(t.data_ptr() for t in tensors), S, L, lo, hi, thr)
    for k in KEYS:
        assert np.array_equal(dev[k].view(np.uint64) if dev[k].dtype == np.float64 else dev[k],
                              out[k].view(np.uint64) if out[k].dtype == np.float64 else out[k]), k
    assert dev["kernel_ms"] > 0 and dev["launches"] > 0
    perm = rng.permutation(len(lo))
    pout = ctx.region_divergence(status, post, meth, lo[perm], hi[perm], thr)
    for k in KEYS:
        a, b = pout[k], out[k][perm]
        assert np.array_equal(a.view(np.uint64) if a.dtype == np.float64 else a, b.view(np.uint64) if b.dtype == np.float64 else b), k


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [0.99, 0.0, float("nan"), float("inf")])
def test_thresholds_and_one_sample(ab, ctx, thr):
    rng = np.random.default_rng(3)
    L = 20_000
    for S in (1, 2, 5):
        status, post, meth = adversarial(rng, S, L, 0.99)
        lo = np.array([0, 100, 100, 5, 19_999, 0, 7], dtype=np.int64)
        hi = np.array([L, 300, 300, 5, L, 1, 7_000], dtype=np.int64)
        out = ctx.region_divergence(status, post, meth, lo, hi, thr)
        check_regions(ctx, device_inputs(status, post, meth), S, L, lo, hi, thr, out)


@pytest.mark.gpu
def test_c5_width_one_million_sites(ab, ctx):
    """200 simulated samples x 1 M sites, 10 000-site tiles at step 1000 plus long regions"""
    import torch

    tree = ab.SimTree.lines(20, range(1, 11))
    S, L = tree.n_samples, 1_000_000
    dev = torch.device("cuda", 0)
    st = torch.empty((S, L), dtype=torch.uint8, device=dev)
    po = torch.empty((S, L), dtype=torch.float64, device=dev)
    me = torch.empty((S, L), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    ctx.simulate_device(tree, st.data_ptr(), po.data_ptr(), me.data_ptr(), 3e-3, 6e-3, L=L, seed=17, missing_rate=0.1)
    a = np.arange(0, L - 10_000 + 1, 1000)
    lo = np.concatenate([a, [0, 250_000, 17]]).astype(np.int64)
    hi = np.concatenate([a + 10_000, [L, 250_000 + 65_537, 17]]).astype(np.int64)
    out = ctx.region_divergence_device(st.data_ptr(), po.data_ptr(), me.data_ptr(), S, L, lo, hi)
    which = list(range(0, len(a), 97)) + list(range(len(lo) - 3, len(lo)))
    check_regions(ctx, (st, po, me), S, L, lo, hi, 0.99, out, which)
    assert not np.isnan(out["D"][:len(a)]).any()


@pytest.mark.gpu
def test_too_large_is_refused(ab, ctx):
    """400 000 regions x 19 900 pairs: 191 GB of outputs, refused before any launch; the context works after"""
    import torch

    S, L, W = 200, 1000, 400_000
    dev = torch.device("cuda", 0)
    st = torch.zeros((S, L), dtype=torch.uint8, device=dev)
    po = torch.ones((S, L), dtype=torch.float64, device=dev)
    me = torch.zeros((S, L), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    lo = np.zeros(W, dtype=np.int64)
    hi = np.full(W, 10, dtype=np.int64)
    rc = ab._lib.abfit_region_divergence_device(ctx._h, C.c_void_p(st.data_ptr()), C.c_void_p(po.data_ptr()),
                                                C.c_void_p(me.data_ptr()), S, L, lo.ctypes.data_as(C.c_void_p),
                                                hi.ctypes.data_as(C.c_void_p), W, 0.99, None, None, None, None, None, None,
                                                None, None)
    assert rc == -5 and "MiB of device memory" in ab._lib.abfit_last_error().decode()
    out = ctx.region_divergence_device(st.data_ptr(), po.data_ptr(), me.data_ptr(), S, L, [0, 3], [10, 900])
    assert np.array_equal(out["cnt"][0], np.full(S * (S - 1) // 2, 10, dtype=np.uint64))
    with pytest.raises(ab.AbfitError):
        ctx.region_divergence_device(st.data_ptr(), po.data_ptr(), me.data_ptr(), S, L, [5], [4])
    with pytest.raises(ab.AbfitError):
        ctx.region_divergence_device(st.data_ptr(), po.data_ptr(), me.data_ptr(), S, L, [0], [L + 1])


# ---------------------------------------------------------------------------------------------
# the `regions` tool
# ---------------------------------------------------------------------------------------------
NL, EL = os.path.join(GOLDEN, "nodelist.txt"), os.path.join(GOLDEN, "edgelist.txt")
BED = ("track name=test\n"
       "1\t100\t700\tr_a\n"
       "1\t400\t1200\tr_b\tx\t+\n"
       "chr2\t0\t3000\tchr2_all\n"
       "2\t500\t500\tempty\n"
       "# a comment\n"
       "4\t0\t100000\n"
       "9\t0\t10\tno_chromosome\n"
       "C\t0\t5000\tchloroplast\n"
       "3\t1\t2\tone_position\n")


def sorted_golden(ab, tmp_path, mutate=None):
    """the golden methylomes with their lines sorted by (chromosome, position): every sample lists the same sequence"""
    d = os.path.join(tmp_path, "data", "methylome")
    os.makedirs(d)
    for name in sorted(os.listdir(os.path.join(GOLDEN, "methylome"))):
        lines = open(os.path.join(GOLDEN, "methylome", name)).read().split("\n")
        head, body = lines[0], [l for l in lines[1:] if l.strip()]
        body.sort(key=lambda l: (ab.parse_region_line(l.split("\t")[0] + "\t0\t0")[0], int(l.split("\t")[1])))
        if mutate:
            body = mutate(name, body)
        open(os.path.join(d, name), "w").write("\n".join([head] + body) + "\n")
    open(os.path.join(tmp_path, "r.bed"), "w").write(BED)
    os.makedirs(os.path.join(tmp_path, "out"), exist_ok=True)
    return str(tmp_path)


def run_tool(cwd, *extra, out="out"):
    return subprocess.run([TOOL, "-n", NL, "-e", EL, "-r", "r.bed", "-o", out, *extra], cwd=cwd, capture_output=True,
                          text=True, timeout=600)


def test_tool_refusals(ab, tmp_path):
    """refused before any device work: samples listing different sites, sites not grouped by chromosome, bad BED lines,
    --site-bootstrap with several devices"""
    cwd = os.path.join(tmp_path, "a")
    os.makedirs(os.path.join(cwd, "data"))
    os.symlink(os.path.join(GOLDEN, "methylome"), os.path.join(cwd, "data", "methylome"))
    open(os.path.join(cwd, "r.bed"), "w").write(BED)
    os.makedirs(os.path.join(cwd, "out"))
    r = run_tool(cwd, "--device", "99")  # the golden files list the chromosomes in different orders
    assert r.returncode == 1 and "G1_2.txt differs from the first sample at line" in r.stdout, r.stdout + r.stderr
    # every sample moves its first chromosome-1 site to the end: same sequence, chromosome 1 in two runs
    def move_first_site(name, body):
        k = next(i for i, l in enumerate(body) if ab.parse_methylome_line(l) is not None)
        return body[:k] + body[k + 1:] + body[k:k + 1]

    cwd = sorted_golden(ab, os.path.join(tmp_path, "b"), move_first_site)
    r = run_tool(cwd, "--device", "99")
    assert r.returncode == 1 and "chromosome 1 appears again" in r.stdout, r.stdout + r.stderr
    cwd = sorted_golden(ab, os.path.join(tmp_path, "c"))
    open(os.path.join(cwd, "r.bed"), "a").write("1\t50\t10\n")
    r = run_tool(cwd, "--device", "99")
    assert r.returncode == 1 and "r.bed line 11" in r.stdout and "end < start" in r.stdout, r.stdout
    r = run_tool(cwd, "--devices", "0-1", "--site-bootstrap", "5")
    assert r.returncode == 2 and "--site-bootstrap runs on one device" in r.stderr


def read_tsv(path):
    lines = open(path).read().rstrip("\n").split("\n")
    return lines[0].split("\t"), [l.split("\t") for l in lines[1:]]


def library_regions(ab, ctx, cwd, seed, n):
    """the pipeline the tool replaces: each region's sites gathered, abfit_divergence on them alone, then
    abfit_alphabeta_batch keyed by the region's line index"""
    files, pairs = ab.pedigree_graph(NL, EL)
    parsed = [ab.parse_methylome_buffer(open(os.path.join(cwd, f), "rb").read()) for f in files]
    sites = parsed[0]["sites"]
    status = np.stack([q["status"] for q in parsed])
    post = np.stack([q["posteriormax"] for q in parsed])
    meth = np.stack([q["meth_lvl"] for q in parsed])
    regs = []
    for ln, line in enumerate(BED.split("\n")):
        r = ab.parse_region_line(line)
        if r is not None:
            regs.append((ln, line.split()[3] if len(line.split()) > 3 else ".", *r))
    lo, hi = ab.region_ranges(sites, [r[2] for r in regs], [r[3] for r in regs], [r[4] for r in regs])
    S = status.shape[0]
    res = []
    for (ln, name, c, a, b), l, h in zip(regs, lo, hi):
        if h == l:
            res.append((ln, name, l, h, None, "no sites"))
            continue
        g = ctx.dmatrix(status[:, l:h], post[:, l:h], meth[:, l:h])
        i, j = pairs[:, 0].astype(np.int64), pairs[:, 1].astype(np.int64)
        D = g["D"][0][i * S - i * (i + 1) // 2 + (j - i - 1)]
        p0 = float(g["p0uu"][0])
        if np.isnan(D).any():
            res.append((ln, name, l, h, p0, "pair without valid sites"))
            continue
        ped = np.column_stack([pairs[:, 2:5], D])
        prob = ab.Problem(ped, p0, p0, 1.0)
        sx = ab.gen_start_simplices(seed, ln, n, float(D.max()))[None]
        r = ctx.alphabeta_batch([prob], sx, n, seed, first_problem_id=ln)
        res.append((ln, name, l, h, p0, r, (status[:, l:h], post[:, l:h], meth[:, l:h], prob, pairs)))
    return res


@pytest.mark.gpu
def test_tool_equals_library_pipeline(ab, ctx, tmp_path):
    seed, n = 21, 24
    cwd = sorted_golden(ab, tmp_path)
    r = run_tool(cwd, "-i", str(n), "--seed", str(seed))
    assert r.returncode == 0, r.stdout + r.stderr
    head, rows = read_tsv(os.path.join(cwd, "out", "regions.tsv"))
    assert head[:6] == ["name", "chromosome", "start", "end", "sites", "p0uu"] and head[-1] == "status"
    raw = np.load(os.path.join(cwd, "out", "raw.npy"))
    lib = library_regions(ab, ctx, cwd, seed, n)
    assert len(rows) == len(lib) == 8
    f = 0
    for row, q in zip(rows, lib):
        assert row[0] == q[1] and int(row[4]) == q[3] - q[2]
        if q[4] is None:
            assert row[-1] == "no sites" and all(v == "NaN" for v in row[5:-1])
            continue
        assert row[5] == ab.format_f64(q[4])
        if isinstance(q[5], str):
            assert row[-1] == q[5]
            continue
        res = q[5]
        if res["status"][0] != 0:
            assert row[-1] == "fit failed"
            continue
        best, an = res["best"][0], res["analysis"][0]
        want = [*best["theta"], an[8], an[16], an[17], an[9], an[18], an[19]]
        assert row[6:16] == [ab.format_f64(v) for v in want] and row[-1] == "ok"
        assert np.array_equal(raw[f].view(np.uint64), res["rows"][0].view(np.uint64))
        f += 1
    assert f == raw.shape[0] >= 4
    # three contexts on device 0: byte-identical files
    os.makedirs(os.path.join(cwd, "out3"))
    r = run_tool(cwd, "-i", str(n), "--seed", str(seed), "--devices", "0,0,0", out="out3")
    assert r.returncode == 0, r.stdout + r.stderr
    for name in ("regions.tsv", "raw.npy"):
        assert open(os.path.join(cwd, "out", name), "rb").read() == open(os.path.join(cwd, "out3", name), "rb").read()
    # --site-bootstrap: abfit_site_boot_batch on the gathered regions
    os.makedirs(os.path.join(cwd, "outsb"))
    r = run_tool(cwd, "-i", str(n), "--seed", str(seed), "--site-bootstrap", "7", out="outsb")
    assert r.returncode == 0, r.stdout + r.stderr
    _, srows = read_tsv(os.path.join(cwd, "outsb", "regions.tsv"))
    sraw = np.load(os.path.join(cwd, "outsb", "raw.npy"))
    fitted = [q for q in lib if not isinstance(q[5], str) and q[4] is not None]
    probs = [q[6][3] for q in fitted]
    seg = np.concatenate([[0], np.cumsum([q[3] - q[2] for q in fitted])])
    cat = [np.concatenate([q[6][k] for q in fitted], axis=1) for k in range(3)]
    sx = np.stack([ab.gen_start_simplices(seed, q[0], n, float(q[6][3].pedigree[:, 3].max())) for q in fitted])
    best = ctx.fit_batch(probs, sx, max_iters=10000, want_all=False)
    pairs = np.concatenate([q[6][4][:, :2] for q in fitted]).astype(np.int32)
    sb = ctx.site_bootstrap(probs, pairs, *cat, seg, best.best, n, seed, 7, problem_ids=[q[0] for q in fitted])
    f = 0
    for k, q in enumerate(fitted):
        if best.status[k] != 0:
            continue
        row = next(rw for rw, qq in zip(srows, lib) if qq[0] == q[0])
        an = sb["analysis"][k]
        assert row[6:16] == [ab.format_f64(v) for v in [*best.best[k]["theta"], an[8], an[16], an[17], an[9], an[18], an[19]]]
        assert np.array_equal(sraw[f].view(np.uint64), sb["rows"][k].view(np.uint64))
        f += 1
    assert f == sraw.shape[0]


def lines_pedigree(d, n_lines=4, gens=(2, 4, 8, 12)):
    """nodelist / edgelist of a founder (sampled) and n_lines lines sampled at the given generations"""
    nodes, edges = ["filename,node,gen,meth", "x,F,0,Y"], ["from\tto\tgendiff"]
    for l in range(n_lines):
        prev, pg = "F", 0
        for g in gens:
            nodes.append(f"x,L{l}_{g},{g},Y")
            edges.append(f"{prev}\tL{l}_{g}\t{g - pg}")
            prev, pg = f"L{l}_{g}", g
    open(os.path.join(d, "nodes.txt"), "w").write("\n".join(nodes) + "\n")
    open(os.path.join(d, "edges.txt"), "w").write("\n".join(edges) + "\n")


@pytest.mark.gpu
def test_tool_recovers_known_rates(ab, ctx, tmp_path):
    """simulated methylomes with known alpha and beta (17 samples), 20 tiles of 10 000 sites: the median fitted rates
    lie within 10 % of the truth"""
    alpha, beta, L = 3e-3, 6e-3, 200_000
    d = str(tmp_path)
    lines_pedigree(d)
    sim = os.path.join(d, "sim")
    r = subprocess.run([os.path.join(ROOT, "alphabeta-rs_b200", "simulate"), "-n", "nodes.txt", "-e", "edges.txt", "-o", sim,
                        "--alpha", str(alpha), "--beta", str(beta), "--sites", str(L), "--seed", "5"], cwd=d,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    files, _ = ab.pedigree_graph(os.path.join(sim, "nodelist.txt"), os.path.join(sim, "edgelist.txt"))
    first = ab.parse_methylome_buffer(open(files[0], "rb").read())["sites"]
    assert len(first) == L and np.all(first["chromosome"] == first["chromosome"][0])
    tiles = np.linspace(0, L, 21).astype(np.int64)
    pos = first["start"].astype(np.int64)
    bed = "".join(f"{first['chromosome'][0]}\t{pos[a] - 1}\t{pos[b - 1]}\ttile{k}\n"
                  for k, (a, b) in enumerate(zip(tiles[:-1], tiles[1:])))
    open(os.path.join(sim, "tiles.bed"), "w").write(bed)
    out = os.path.join(sim, "out")
    os.makedirs(out)
    r = subprocess.run([TOOL, "-n", "nodelist.txt", "-e", "edgelist.txt", "-r", "tiles.bed", "-o", out, "-i", "16"], cwd=sim,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    _, rows = read_tsv(os.path.join(out, "regions.tsv"))
    assert len(rows) == 20 and all(rw[-1] == "ok" for rw in rows) and all(int(rw[4]) == L // 20 for rw in rows)
    a = np.median([float(rw[6]) for rw in rows])
    b = np.median([float(rw[7]) for rw in rows])
    print(f"median alpha {a:.4e} (true {alpha}), beta {b:.4e} (true {beta})")
    assert abs(a / alpha - 1) < 0.1 and abs(b / beta - 1) < 0.1
