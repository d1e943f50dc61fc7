"""Pins the CPU oracle against every golden vector the reference ships for the hot path
(SURVEY.md §8c).  CPU only."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, resolve_golden


@pytest.fixture(scope="module")
def ped351(oracle):
    return oracle.load_pedigree_file(os.path.join(GOLDEN, "pedigree.txt"))


def test_manifest_intact():
    import hashlib

    man = json.load(open(os.path.join(GOLDEN, "MANIFEST.json")))
    for rel, sha in man.items():
        if rel.startswith("_"):
            continue
        assert hashlib.sha256(open(os.path.join(GOLDEN, rel), "rb").read()).hexdigest() == sha, rel


def test_cost_kat_exact(oracle, ped351):
    """src/structs.rs:225-240: Problem::default() at Model::default() == 0.0006700888539608879 (assert_eq!)"""
    assert ped351.shape == (351, 4)
    pb = oracle.Problem(ped351, p_uu=0.75, eqp=0.5, eqp_weight=0.7, p_mm=0.25, p_um=0.0)
    theta = [0.0001179555, 0.0001180614, 0.03693534, 0.003023981]
    for flags in (0, oracle.FAST_DIVERGENCE):
        assert oracle.cost(pb, theta, flags) == 0.0006700888539608879


def test_divergence_same_as_r(oracle, ped351):
    """src/divergence.rs:139-161: dt1t2 equals the R output within 1e-4 abs (assert_close!) and is_normal()"""
    r = np.array([float(x) for x in open(os.path.join(GOLDEN, "divergence.txt")).read().split("\n")])
    pb = oracle.Problem(ped351, p_uu=0.75, eqp=0.5, eqp_weight=0.7, p_mm=0.25)
    for flags in (0, oracle.FAST_DIVERGENCE):
        dt, _ = oracle.divergence(pb, 3.974271e-09, 1.519045e-07, 0.06892953, flags)
        assert len(dt) == len(r) == 351
        assert np.all(np.isfinite(dt)) and np.all(np.abs(dt) >= np.finfo(float).tiny)
        assert np.max(np.abs(dt - r)) <= 1e-4
        assert np.max(np.abs(dt - r) / r) < 1e-13  # in fact agrees to rounding
    a, _ = oracle.divergence(pb, 3.974271e-09, 1.519045e-07, 0.06892953, 0)
    b, _ = oracle.divergence(pb, 3.974271e-09, 1.519045e-07, 0.06892953, oracle.FAST_DIVERGENCE)
    assert np.array_equal(a, b)  # power table == per-pair recomputation, bit for bit


def test_matrix_power_properties(oracle):
    """src/divergence.rs:130-137,164-209"""
    G = oracle.genmatrix(3.974271e-09, 1.519045e-07)
    assert np.array_equal(oracle.matrix_power(G, 0), np.eye(3))
    assert np.array_equal(oracle.matrix_power(G, 1), G)
    P5 = oracle.matrix_power(G, 5)
    for k in range(3):
        e = np.zeros(3)
        e[k] = 1.0
        assert np.allclose(e @ P5, P5[k], rtol=0, atol=0)
    assert np.allclose(P5, np.linalg.matrix_power(G, 5), rtol=1e-14)
    assert np.allclose(G.sum(axis=1), 1.0, rtol=1e-15)


def test_steady_state_todo_value(oracle):
    """src/divergence.rs:123-127 (TODO in the reference): steady_state(3.974271e-09,1.519045e-07) ~ 0.9745041
    is the R value for Pr(UU); check the closed forms are a probability vector instead."""
    a, b = 3.974271e-09, 1.519045e-07
    lib = oracle.lib()
    s = lib.abref_p_uu_est(a, b) + lib.abref_p_um_est(a, b) + lib.abref_p_mm_est(a, b)
    assert abs(s - 1.0) < 1e-12
    assert abs(lib.abref_p_uu_est(a, b) - 0.9745041) < 1e-6
    assert abs(lib.abref_steady_state(a, b) - (lib.abref_p_mm_est(a, b) + 0.5 * lib.abref_p_um_est(a, b))) == 0.0


def test_build_pedigree_generated_exact(oracle):
    """src/pedigree.rs:345-358: the checked-in data/pedigree_generated.txt is the reference's own output
    (17 significant digits): 6 rows, bit-exact."""
    ped, p0uu, info = oracle.build_pedigree(os.path.join(GOLDEN, "nodelist.txt"), os.path.join(GOLDEN, "edgelist.txt"),
                                            0.99, resolve_golden)
    want = np.loadtxt(os.path.join(GOLDEN, "pedigree_generated.txt"), skiprows=1)
    assert ped.shape == (6, 4)
    assert np.array_equal(ped, want)
    assert info["status"].shape == (4, 500)  # src/methylation_site.rs:565-593: 500 CG sites per file
    assert list(info["nvalid"]) == [309, 378, 428, 346]
    assert [int(x) for x in info["diff"]] == [54, 240, 3, 169, 50, 269]
    assert [int(x) for x in info["cnt"]] == [247, 260, 276, 333, 271, 295]
    # unpinned by the reference (assert disabled, src/pedigree.rs:356-357).  The survey's numpy probe
    # (pairwise summation) gave ...0442; the reference sums sequentially (Iterator::sum) -> ...0447
    assert p0uu == 0.6554051647850447 and abs(p0uu - 0.6554051647850442) < 1e-14


def test_desired_output_pedigree(oracle):
    """data/desired_output (R original, 13 samples): 78 rows, D rounded to 5 decimals."""
    ped, p0uu, info = oracle.build_pedigree(os.path.join(GOLDEN, "desired_output", "nodelist.fn"),
                                            os.path.join(GOLDEN, "desired_output", "edgelist.fn"), 0.99, resolve_golden)
    want = oracle.load_pedigree_file(
        os.path.join(GOLDEN, "desired_output", "pedigree-pdata_epimutation_rate_estimation_window_gene_0.txt"))
    assert ped.shape == want.shape == (78, 4)
    assert np.array_equal(ped[:, :3], want[:, :3])
    assert np.max(np.abs(ped[:, 3] - want[:, 3])) < 1e-5
    assert info["status"].shape == (13, 744)  # header + 744 CG rows (no trailing newline)
    r_p0uu = float(open(os.path.join(GOLDEN, "desired_output", "p0uu_in_epimutation_rate_estimation_window_gene_0.txt")).read())
    assert abs(p0uu - r_p0uu) < 1e-3  # R computes it differently; the reference's own assert is disabled


def test_desired_output_fit_within_10_percent(ab, oracle):
    """The reference's intended end-to-end criterion (src/alphabeta.rs:81-140, macros.rs:25-34): alpha and beta
    within 10 % of the R fit.  Starts come from the product's seeded generator."""
    ped, p0uu, _ = oracle.build_pedigree(os.path.join(GOLDEN, "desired_output", "nodelist.fn"),
                                         os.path.join(GOLDEN, "desired_output", "edgelist.fn"), 0.99, resolve_golden)
    pb = oracle.Problem(ped, p0uu, p0uu, 1.0)
    sx = ab.gen_start_simplices(0xAB0B200, 0, 96, float(ped[:, 3].max()))
    rc, best, allr, pred, resid = oracle.ab_neutral(
        pb, sx, flags=oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, n_threads=8)
    assert rc == 0
    r_alpha, r_beta = 5.7985750419976e-05, 0.00655710970515347
    assert abs(best["theta"][0] - r_alpha) < 0.1 * r_alpha
    assert abs(best["theta"][1] - r_beta) < 0.1 * r_beta
    assert abs(best["lse"] - 5.28198e-05) < 1e-8  # survey probe of the restated algorithm
    assert np.allclose(pred + resid, ped[:, 3], rtol=0, atol=1e-18)


def test_restated_optimiser_ends_in_a_minimum_an_independent_optimiser_confirms(ab, oracle):
    """argmin 0.8.1 is not in /root/reference, so the Nelder-Mead restatement cannot be pinned on its source.  What
    can be checked independently: the point it returns for the R-original pedigree is a local minimum of the
    reference's objective (src/structs.rs:191-217) — scipy's own Nelder-Mead and Powell, started from it with
    tight tolerances, cannot lower the cost by more than 1e-9 relative and stay within 1e-4 relative in alpha, beta
    (the valley is flat: points 1e-6 apart in alpha have costs that differ in the last bits only)."""
    from scipy.optimize import minimize

    ped, p0uu, _ = oracle.build_pedigree(os.path.join(GOLDEN, "desired_output", "nodelist.fn"),
                                         os.path.join(GOLDEN, "desired_output", "edgelist.fn"), 0.99, resolve_golden)
    pb = oracle.Problem(ped, p0uu, p0uu, 1.0)
    sx = ab.gen_start_simplices(0xAB0B200, 0, 96, float(ped[:, 3].max()))
    rc, best, *_ = oracle.ab_neutral(pb, sx, flags=oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, n_threads=8)
    assert rc == 0
    x0, f0 = best["theta"].copy(), float(best["cost"])
    f = lambda x: oracle.cost(pb, np.asarray(x, dtype=np.float64))
    assert f(x0) == f0
    for method, opts in (("Nelder-Mead", dict(xatol=1e-14, fatol=1e-18, maxiter=4000, maxfev=8000)),
                         ("Powell", dict(xtol=1e-12, ftol=1e-16, maxiter=200))):
        r = minimize(f, x0, method=method, options=opts)
        assert r.fun >= f0 * (1 - 1e-9), (method, r.fun, f0)
        assert abs(r.x[0] - x0[0]) <= 1e-4 * abs(x0[0]) and abs(r.x[1] - x0[1]) <= 1e-4 * abs(x0[1]), (method, r.x, x0)


def test_work_saving_modes_are_result_identical(ab, oracle, ped351):
    """literal reference work == power table == early exit on stall (bit for bit), incl. a stalled start"""
    pb = oracle.Problem(ped351, 0.75, 0.75, 1.0)
    sx = ab.gen_start_simplices(7, 3, 24, float(ped351[:, 3].max()))
    lit = [oracle.nelder_mead(pb, s, 1500, flags=0) for s in sx[:6]]
    fast = [oracle.nelder_mead(pb, s, 1500, flags=oracle.FAST_DIVERGENCE) for s in sx]
    early = [oracle.nelder_mead(pb, s, 1500, flags=oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL) for s in sx]
    for a, b in zip(lit, fast):
        assert a.tobytes() == b.tobytes()
    n_stalled = 0
    for a, b in zip(fast, early):
        assert np.array_equal(a["theta"], b["theta"]) and a["cost"] == b["cost"] and a["iters"] == b["iters"]
        if b["status"] == oracle.TERM_STALLED:
            n_stalled += 1
            assert a["status"] == oracle.TERM_MAX_ITERS and b["evals"] < a["evals"]
        else:
            assert a["status"] == b["status"] and a["evals"] == b["evals"]
    assert n_stalled >= 1


def test_sanity_anchor_small_pedigree(ab, oracle):
    """SURVEY §8c item 7 (ours): fit of pedigree_generated.txt, LSE ~ 0.138178820"""
    ped = np.loadtxt(os.path.join(GOLDEN, "pedigree_generated.txt"), skiprows=1)
    pb = oracle.Problem(ped, 0.6554051647850447, 0.6554051647850447, 1.0)
    sx = ab.gen_start_simplices(0xAB0B200, 0, 200, float(ped[:, 3].max()))
    rc, best, *_ = oracle.ab_neutral(pb, sx, flags=oracle.FAST_DIVERGENCE | oracle.EARLY_EXIT_ON_STALL, n_threads=8)
    assert rc == 0
    assert abs(best["lse"] - 0.138178820) < 1e-6


def test_dmatrix_edge_cases(oracle):
    """empty overlap -> NaN (0/0), all-equal -> 0, max distance -> 1; a site is kept when post_i >= thr && post_j >= thr
    (src/pedigree.rs:249-251): a NaN posterior drops it, as it does from p0uu, and thr = NaN keeps none"""
    st = np.array([[0, 1, 2, 2, 0], [2, 1, 0, 2, 2], [0, 0, 0, 0, 0]], dtype=np.uint8)
    po = np.array([[1, 1, 1, 0.5, np.nan], [1, 1, 1, 1, 1], [0.1, 0.1, 0.1, 0.1, 0.1]])
    D, diff, cnt = oracle.dmatrix(st, po, 0.99)
    assert diff[0] == 4 and cnt[0] == 3 and D[0] == 4 / 6
    assert np.isnan(D[1]) and np.isnan(D[2]) and cnt[1] == 0
    _, _, nv = oracle.p0uu(po, po, 0.99)
    assert nv[0] == 3
    D, diff, cnt = oracle.dmatrix(st, np.ones_like(po), np.nan)
    assert (cnt == 0).all() and np.isnan(D).all()
    assert (oracle.p0uu(po, po, np.nan)[2] == 0).all()


def test_analyze_matches_numpy(oracle):
    rng = np.random.default_rng(5)
    rows = np.abs(rng.normal(1.0, 0.1, (257, 7)))
    out = oracle.analyze(rows)
    cols = [rows[:, 0], rows[:, 1], rows[:, 1] / rows[:, 0], rows[:, 2], rows[:, 3], rows[:, 4], rows[:, 5], rows[:, 6]]
    for f, c in enumerate(cols):
        assert abs(out[f] - c.mean()) < 1e-14
        assert abs(out[8 + f] - c.std(ddof=1)) < 1e-14
        lo, hi = np.quantile(c, [0.025, 0.975])
        assert abs(out[16 + 2 * f] - lo) < 1e-14 and abs(out[17 + 2 * f] - hi) < 1e-14
