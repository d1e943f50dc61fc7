"""Simulated methylomes under ABneutral (abfit_sim_tree_* / abfit_simulate*, SimTree, Context.simulate, design_study,
the `simulate` CLI).

CPU: the forest and its pedigree rows against the pedigree builder, the draw table against the oracle, and the model's
statistics (observed D against dt1t2) on oracle-simulated data.  GPU: the kernel bit for bit against the oracle, its
invariances (host / device outputs, site ranges, contexts), the Monte-Carlo check of dt1t2 at scale, recovery of alpha
and beta by the fit, and the CLI round trip through `alphabeta`."""
import math
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

PKG = os.path.join(ROOT, "alphabeta-rs_b200")
SIM = os.path.join(PKG, "simulate")
ALPHABETA = os.path.join(PKG, "alphabeta")


@pytest.fixture(scope="module")
def sim_oracle():
    """the simulation's CPU oracle (oracle/abref_sim.c)"""
    from oracle import abref_sim_py

    abref_sim_py.build()
    return abref_sim_py


def lines_tree(n_lines, n_gens):
    """one unsampled founder at generation 0, n_lines lines sampled at generations 1..n_gens"""
    parent, gen, smp = [-1], [0], [0]
    for _ in range(n_lines):
        prev = 0
        for g in range(1, n_gens + 1):
            parent.append(prev)
            gen.append(g)
            smp.append(1)
            prev = len(gen) - 1
    return np.array(parent, np.int32), np.array(gen, np.int32), np.array(smp, np.uint8)


def golden_files(name):
    if name == "golden":
        return os.path.join(GOLDEN, "nodelist.txt"), os.path.join(GOLDEN, "edgelist.txt")
    return os.path.join(GOLDEN, "desired_output", "nodelist.fn"), os.path.join(GOLDEN, "desired_output", "edgelist.fn")


def arrays_of_files(nodelist, edgelist):
    """(parent, generation, sampled) of the files, with the oracle's parsers"""
    from oracle import abref_py as o

    nodes = o.parse_nodelist(open(nodelist).read())
    pos = {n["id"]: k for k, n in enumerate(nodes)}
    parent = np.full(len(nodes), -1, np.int32)
    for a, b in o.parse_edgelist(open(edgelist).read(), nodes):
        parent[pos[b["id"]]] = pos[a["id"]]
    return parent, np.array([n["generation"] for n in nodes], np.int32), np.array([n["meth"] for n in nodes], np.uint8)


def two_root_forest():
    """two trees; the second root sits at generation 3; a generation-0 edge (delta = 0) in each"""
    parent = [-1, 0, 1, 1, 2, 3, -1, 6, 7, 7, 8]
    gen = [0, 1, 1, 4, 6, 5, 3, 3, 5, 7, 9]
    smp = [1, 1, 0, 1, 1, 1, 0, 1, 1, 1, 1]
    return np.array(parent, np.int32), np.array(gen, np.int32), np.array(smp, np.uint8)


def big_forest(n_lines=25, n_gens=20):
    """more nodes than a block keeps in shared memory (global-scratch variant of the kernel)"""
    return lines_tree(n_lines, n_gens)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("files", ["golden", "desired_output"])
def test_tree_pairs_equal_pedigree_graph(ab, sim_oracle, files):
    nl, el = golden_files(files)
    t = ab.SimTree.from_files(nl, el)
    _, pairs = ab.pedigree_graph(nl, el)
    got = t.pairs()
    assert got.shape == pairs.shape and np.array_equal(got, pairs)
    # the same forest from arrays, and the oracle's numpy restatement
    par, gen, smp = arrays_of_files(nl, el)
    assert np.array_equal(ab.SimTree(par, gen, smp).pairs(), pairs)
    assert np.array_equal(sim_oracle.sim_pairs(par, gen, smp), pairs)
    if files == "desired_output":
        assert (t.n_samples, t.n_pairs) == (13, 78)


def test_random_forests_pairs_match_oracle(ab, sim_oracle):
    rng = np.random.default_rng(5)
    for _ in range(30):
        n = int(rng.integers(1, 40))
        parent = np.full(n, -1, np.int32)
        gen = np.zeros(n, np.int32)
        for v in range(n):
            if v and rng.random() < 0.85:
                parent[v] = rng.integers(0, v)
                gen[v] = gen[parent[v]] + rng.integers(0, 4)
            else:
                gen[v] = rng.integers(0, 5)
        smp = (rng.random(n) < 0.6).astype(np.uint8)
        assert np.array_equal(ab.SimTree(parent, gen, smp).pairs(), sim_oracle.sim_pairs(parent, gen, smp))


def _write(tmp_path, nodes, edges):
    nl, el = tmp_path / "nodelist.txt", tmp_path / "edgelist.txt"
    nl.write_text("filename,node,gen,meth\n" + "".join(f"-,{n},{g},{m}\n" for n, g, m in nodes))
    el.write_text("from to\n" + "".join(f"{a} {b}\n" for a, b in edges))
    return str(nl), str(el)


@pytest.mark.parametrize("case", ["two_parents", "cycle", "reversed", "gen128", "unknown"])
def test_bad_pedigrees_are_refused(ab, tmp_path, case):
    nodes = [("a", 0, "Y"), ("b", 1, "Y"), ("c", 1, "Y")]
    edges = [("a", "b"), ("a", "c")]
    want = {"two_parents": "two parents", "cycle": "cycle", "reversed": "back in time", "gen128": "outside 0..127",
            "unknown": "not in the nodelist"}[case]
    if case == "two_parents":
        edges.append(("b", "c"))
    elif case == "cycle":
        nodes = [("a", 1, "Y"), ("b", 1, "Y"), ("c", 1, "Y")]
        edges = [("a", "b"), ("b", "c"), ("c", "a")]
    elif case == "reversed":
        edges = [("b", "a"), ("a", "c")]
    elif case == "gen128":
        nodes[2] = ("c", 128, "Y")
    elif case == "unknown":
        edges.append(("a", "zz"))
    with pytest.raises(ab.AbfitError) as e:
        ab.SimTree.from_files(*_write(tmp_path, nodes, edges))
    assert e.value.code == ab.ERR_ARG and want in str(e.value), str(e.value)


def test_bad_arrays_are_refused(ab):
    for parent, gen in (([-1, 2, 1], [0, 1, 1]),   # cycle 1 <-> 2
                        ([-1, 0], [2, 1]),          # generation decreases
                        ([-1, 0], [0, 128]),        # outside the i8 time range
                        ([-1, 5], [0, 1])):         # parent is not a node
        with pytest.raises(ab.AbfitError) as e:
            ab.SimTree(parent, gen, [1] * len(parent))
        assert e.value.code == ab.ERR_ARG
    t = ab.SimTree([-1, 0], [0, 1], [1, 1])
    for bad in ({"alpha": 1.5}, {"beta": -0.1}, {"alpha": math.nan}, {"weight": 2.0}, {"p0uu": math.nan}):
        kw = dict(alpha=0.01, beta=0.01, weight=0.5, p0uu=0.5)
        kw.update(bad)
        with pytest.raises(ab.AbfitError) as e:
            t.thresholds(**kw)
        assert e.value.code == ab.ERR_ARG


@pytest.mark.parametrize("alpha,beta,weight,p0uu", [(1e-2, 2e-2, 0.3, 0.6), (3e-4, 7e-4, None, None), (0.2, 0.05, 0.0, 1.0),
                                                    (0.0, 0.0, 1.0, 0.0), (1.0, 1.0, 0.5, 0.5)])
def test_thresholds_match_oracle(ab, sim_oracle, alpha, beta, weight, p0uu):
    if weight is None:
        p0uu, weight = ab.sim_equilibrium(alpha, beta)
    # roots at generations 0..127 and one child per delta 0..127
    gen = np.concatenate([np.arange(128), np.arange(128)]).astype(np.int32)
    parent = np.concatenate([np.full(128, -1), np.zeros(128)]).astype(np.int32)
    t = ab.SimTree(parent, gen, np.ones(256, np.uint8))
    got = t.thresholds(alpha, beta, weight, p0uu)
    want = sim_oracle.sim_thresholds(parent, gen, alpha, beta, weight, p0uu)
    assert got.tobytes() == want.tobytes()
    c0, c1 = got[:, 0::2], got[:, 1::2]
    eps = 1e-14  # rows of G^delta sum to 1 up to rounding
    assert np.all(c0 >= 0) and np.all(c1 - c0 >= -eps) and np.all(c1 <= 1 + eps) and np.all(c0 <= 1 + eps)
    # delta = 0: the child copies the parent's state
    assert np.array_equal(got[128], [1, 1, 0, 1, 0, 0])


def test_equilibrium(ab, oracle):
    p, w = ab.sim_equilibrium(1e-3, 4e-3)
    assert p == oracle.lib().abref_p_uu_est(1e-3, 4e-3)
    pm, pu = oracle.lib().abref_p_mm_est(1e-3, 4e-3), oracle.lib().abref_p_um_est(1e-3, 4e-3)
    assert w == pu / (pu + pm)
    with pytest.raises(ab.AbfitError):
        ab.sim_equilibrium(0.0, 0.0)


def test_oracle_observed_divergence_matches_model(oracle, sim_oracle):
    """4 lines x 8 generations, L = 200 000: every pair's observed D lies within 6 sqrt(dt1t2 / L) of dt1t2 (a site's
    |s_i - s_j| / 2 lies in [0, 1], so its variance is at most its mean); with 20 % missingness per sample-site a pair
    keeps 0.64 L sites on average"""
    alpha, beta, L = 1.2e-2, 2.5e-2, 200_000
    parent, gen, smp = lines_tree(4, 8)
    p0, w = oracle.lib().abref_p_uu_est(alpha, beta), None
    pm, pu = oracle.lib().abref_p_mm_est(alpha, beta), oracle.lib().abref_p_um_est(alpha, beta)
    w = pu / (pu + pm)
    pairs = sim_oracle.sim_pairs(parent, gen, smp)
    status, post, _ = sim_oracle.simulate(parent, gen, smp, alpha, beta, w, p0, L, seed=17)
    D, _, cnt = oracle.dmatrix(status, post, 0.99)
    S = int(smp.sum())
    i, j = pairs[:, 0].astype(int), pairs[:, 1].astype(int)
    idx = i * S - i * (i + 1) // 2 + (j - i - 1)
    ped = np.column_stack([pairs[:, 2:5], D[idx]])
    dt, _ = oracle.divergence(oracle.Problem(ped, p0, p0, 1.0), alpha, beta, w)
    assert len(pairs) == 32 * 31 // 2 and np.all(cnt == L)
    z = np.abs(D[idx] - dt) / np.sqrt(dt / L)
    assert z.max() < 6, z.max()
    assert 0.5 < z.mean() < 1.1  # not only inside the band but of the size sampling noise has

    status, post, _ = sim_oracle.simulate(parent, gen, smp, alpha, beta, w, p0, L, seed=18, missing_rate=0.2)
    _, _, cnt = oracle.dmatrix(status, post, 0.99)
    sd = math.sqrt(L * 0.64 * 0.36)
    assert np.all(np.abs(cnt.astype(np.float64) - 0.64 * L) < 6 * sd)


def test_simulate_cli_arguments():
    assert os.path.exists(SIM), "build() compiles the simulate CLI"
    r = subprocess.run([SIM, "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--alpha" in r.stdout and "--sites" in r.stdout
    nl, el = golden_files("desired_output")
    base = ["-n", nl, "-e", el, "-o", "/nonexistent-dir-for-sure/out"]
    for args, msg in (([], "required"), (base + ["--beta", "0.01", "--sites", "10"], "--alpha"),
                      (base + ["--alpha", "0.01", "--beta", "0.01"], "--sites"),
                      (base + ["--alpha", "x", "--beta", "0.01", "--sites", "10"], "invalid number"),
                      (base + ["--alpha", "0.01", "--beta", "0.01", "--sites", "-3"], "positive integer"),
                      (base + ["--alpha", "2", "--beta", "0.01", "--sites", "10", "--weight", "0.5", "--p0uu", "0.5"], "[0, 1]"),
                      (base + ["--bogus"], "unexpected argument"),
                      (["-n", nl, "-e", "/nonexistent.txt", "-o", "x", "--alpha", "0.01", "--beta", "0.01", "--sites", "5"],
                       "cannot read")):
        r = subprocess.run([SIM] + args, capture_output=True, text=True)
        assert r.returncode != 0 and msg in r.stderr, (args, r.stderr)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _equilibrium(oracle, alpha, beta):
    pm, pu = oracle.lib().abref_p_mm_est(alpha, beta), oracle.lib().abref_p_um_est(alpha, beta)
    return oracle.lib().abref_p_uu_est(alpha, beta), pu / (pu + pm)


CASES = {
    "tile_remainder": (lambda: lines_tree(2, 5), dict(alpha=0.05, beta=0.08, weight=0.4, p0uu=0.5), 1000, 0.0),
    "missing": (lambda: lines_tree(3, 4), dict(alpha=0.02, beta=0.03, weight=0.6, p0uu=0.3), 3000, 0.3),
    "two_roots_delta0": (two_root_forest, dict(alpha=0.1, beta=0.2, weight=0.5, p0uu=0.4), 2049, 0.1),
    "c5_shape": (lambda: lines_tree(10, 20), dict(alpha=0.01, beta=0.02, weight=0.5, p0uu=0.6), 2000, 0.05),
    "global_scratch": (big_forest, dict(alpha=0.03, beta=0.01, weight=0.2, p0uu=0.7), 1500, 0.1),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_kernel_matches_oracle(ab, sim_oracle, ctx, case):
    mk, prm, L, miss = CASES[case]
    parent, gen, smp = mk()
    if case == "global_scratch":
        assert len(parent) > 400  # more node states than a block keeps in shared memory
    t = ab.SimTree(parent, gen, smp)
    got = ctx.simulate(t, L=L, seed=99, missing_rate=miss, first_site=12345, **prm)
    want = sim_oracle.simulate(parent, gen, smp, L=L, seed=99, missing_rate=miss, first_site=12345, **prm)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
    if miss > 0:
        assert 0 < np.mean(got[1] == 0.5) < 2 * miss


@pytest.mark.gpu
def test_simulation_invariances(ab, ctx):
    import torch

    parent, gen, smp = lines_tree(6, 12)
    t = ab.SimTree(parent, gen, smp)
    kw = dict(alpha=0.01, beta=0.03, seed=7, missing_rate=0.1)
    L = 100_003
    one = ctx.simulate(t, L=L, **kw)
    # device outputs
    S = t.n_samples
    d = [torch.empty((S, L), dtype=dt, device="cuda:0") for dt in (torch.uint8, torch.float64, torch.float64)]
    ms = ctx.simulate_device(t, *(x.data_ptr() for x in d), L=L, **kw)
    assert ms > 0
    for g, w in zip(d, one):
        assert np.array_equal(g.cpu().numpy(), w)
    # two calls with first_site
    a = ctx.simulate(t, L=40_000, **kw)
    b = ctx.simulate(t, L=L - 40_000, first_site=40_000, **kw)
    for x, y, w in zip(a, b, one):
        assert np.array_equal(np.concatenate([x, y], axis=1), w)
    # two contexts, one half each
    c2 = ab.Context(0)
    try:
        b2 = c2.simulate(t, L=L - 40_000, first_site=40_000, **kw)
    finally:
        c2.close()
    for x, y in zip(b, b2):
        assert np.array_equal(x, y)


@pytest.mark.gpu
def test_observed_divergence_matches_model_at_scale(ab, oracle, ctx):
    """C5 time structure (10 lines x 20 generations below one founder: 200 samples, 19 900 pairs) at L = 4 M: every
    pair's D from abfit_divergence lies within 6 sqrt(dt1t2 / L) of abfit_model_divergence"""
    import torch

    alpha, beta, L = 1e-2, 2e-2, 4_000_000
    t = ab.SimTree(*lines_tree(10, 20))
    S = t.n_samples
    p0, w = ab.sim_equilibrium(alpha, beta)
    d = [torch.empty((S, L), dtype=dt, device="cuda:0") for dt in (torch.uint8, torch.float64, torch.float64)]
    ctx.simulate_device(t, *(x.data_ptr() for x in d), alpha, beta, L=L, seed=2024)
    out = ctx.dmatrix_device(*(x.data_ptr() for x in d), S, L)
    del d
    ped = t.pedigree(out["D"][0])
    assert ped.shape == (19900, 4)
    dt, _ = ctx.divergence(ab.Problem(ped, p0, p0, 1.0), [alpha, beta, w, 0.0])
    z = np.abs(ped[:, 3] - dt) / np.sqrt(dt / L)
    assert z.max() < 6, z.max()
    assert 0.5 < z.mean() < 1.1


@pytest.mark.gpu
def test_design_study_recovers_rates(ab, ctx):
    """R = 8 replicates on the R-original design (two lines from one G0 founder, 13 sampled nodes, 78 pairs),
    alpha = 3e-3, beta = 6e-3, L = 500 000 sites: every fit converges and the medians of alpha and beta lie within 10 %
    of the truth (src/macros.rs:25-34).  Observed median relative errors (one B200): alpha 0.03 %, beta 0.03 %, far
    inside half the tolerance."""
    nl, el = golden_files("desired_output")
    t = ab.SimTree.from_files(nl, el)
    alpha, beta = 3e-3, 6e-3
    res = ab.design_study([ctx], t, alpha, beta, L=500_000, n_replicates=8, n_starts=32, n_boot=16, seed=3)
    assert np.all(res["status"] == 0)
    ea = abs(np.median(res["theta"][:, 0]) / alpha - 1)
    eb = abs(np.median(res["theta"][:, 1]) / beta - 1)
    print(f"design_study: median relative error alpha {ea:.4f}, beta {eb:.4f}")
    assert ea < 0.1 and eb < 0.1
    assert res["analysis"].shape == (8, 32)


@pytest.mark.gpu
def test_cli_round_trip_through_alphabeta(ab, ctx, tmp_path):
    nl, el = golden_files("desired_output")
    out, fit = tmp_path / "sim", tmp_path / "fit"
    fit.mkdir()
    kw = dict(alpha=4e-3, beta=8e-3, L=3000, seed=11, missing_rate=0.05)
    r = subprocess.run([SIM, "-n", nl, "-e", el, "--alpha", "0.004", "--beta", "0.008", "--sites", "3000", "--seed", "11",
                        "--missing-rate", "0.05", "-o", str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert (out / "truth.txt").read_text().startswith("alpha\t0.004\nbeta\t0.008\n")
    r = subprocess.run([ALPHABETA, "-n", str(out / "nodelist.txt"), "-e", str(out / "edgelist.txt"), "-o", str(fit),
                        "-i", "50"], capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Model:" in r.stdout and (fit / "analysis.txt").exists()
    t = ab.SimTree.from_files(nl, el)
    status, post, meth = ctx.simulate(t, **kw)
    want = t.pedigree(ctx.dmatrix(status, post, meth, 0.99)["D"][0])
    got = np.array([[float(x) for x in line.split("\t")] for line in (fit / "pedigree.txt").read_text().split("\n")[1:] if line])
    assert got.shape == want.shape and np.array_equal(got, want)
