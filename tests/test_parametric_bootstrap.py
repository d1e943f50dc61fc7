"""The parametric bootstrap and goodness-of-fit test of ABneutral fits (abfit_param_boot_batch): every replicate is a data
set simulated from the window's fitted model with the observed design, counted to exact pair sums on the GPU without
materialising its sites (k_psim_counts), refitted, and the observed LSE is ranked among the replicates' LSEs.

* CPU: the stream-6 seeds; the kernel's tile body (csrc/abfit_psim.cuh) built for the CPU against the oracle's
  simulation (abref_simulate, one run per sample's missing rate) and abref_dmatrix, integers exactly; the refusals
  before any device work.
* GPU: dstar_out equals the materialising route (abfit_simulate, abfit_divergence, + theta3) bit for bit; the refits
  equal the oracle on the stored-tile and warp-per-fit mappings; lse_star equals abfit_cost_batch; gof_p and
  analysis_out; windows that cannot be simulated; window keys; the memory refusal; the alphabeta tool; calibration under
  the model and power against a violation of it."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from test_simulate import arrays_of_files, golden_files, lines_tree, two_root_forest
from test_site_bootstrap import _golden_cwd, check_refits, golden_sites, run_verbose

M64 = (1 << 64) - 1
DBL_EPSILON = 2.220446049250313e-16
SMEM_OPTIN = 227 * 1024  # dynamic shared memory a block may opt in to on the B200


def _mix64(z):
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def py_seeds(seed, key, n_boot):
    """the replicate seeds restated from the generator's definition (stream 6)"""
    h = _mix64(_mix64(seed ^ ((6 * 0xD1342543DE82EF95) & M64)) ^ key)
    return np.array([_mix64(h ^ b) for b in range(n_boot)], dtype=np.uint64)


@pytest.fixture(scope="module")
def emul():
    """tests/host_emul/emul_psim.cpp built for the CPU into a per-user temporary directory keyed by the sources"""
    src = os.path.join(ROOT, "tests", "host_emul", "emul_psim.cpp")
    hdrs = [os.path.join(ROOT, "alphabeta-rs_b200", "csrc", f) for f in ("abfit_psim.cuh", "abfit_rng.h")]
    h = hashlib.sha256()
    for f in [src] + hdrs:
        h.update(open(f, "rb").read())
    out_dir = os.path.join(tempfile.gettempdir(), f"abfit_emul_psim_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    lib = os.path.join(out_dir, f"libemul_psim_{h.hexdigest()[:16]}.so")
    if not os.path.exists(lib):
        tmp = f"{lib}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CXX", "g++"), "-O1", "-std=c++17", "-ffp-contract=off", "-fno-fast-math",
                               "-shared", "-fPIC", "-o", tmp, src])
        os.replace(tmp, lib)
    e = C.CDLL(lib)
    e.emul_psim_counts.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_uint64,
                                   C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    e.emul_param_boot_seed.restype = C.c_uint64
    e.emul_param_boot_seed.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64]
    e.emul_psim_smem_bytes.restype = C.c_uint64
    e.emul_psim_smem_bytes.argtypes = [C.c_int, C.c_int, C.c_int]
    return e


@pytest.fixture(scope="module")
def sim_oracle():
    from oracle import abref_sim_py

    abref_sim_py.build()
    return abref_sim_py


def oracle_simulate_rates(sim_oracle, parent, gen, smp, alpha, beta, weight, p0uu, rates, L, seed):
    """the oracle's simulation with one missing rate per sample.  Every draw is keyed by (seed, node, site), so row s of
    abref_simulate with missing_rate = rates[s] is row s of the per-sample-rate simulation: one oracle run per distinct
    rate, each contributing the rows of that rate"""
    S = int(smp.sum())
    status, post, meth = np.empty((S, L), dtype=np.uint8), np.empty((S, L)), np.empty((S, L))
    for rate in np.unique(rates):
        rows = np.flatnonzero(rates == rate)
        st, po, me = sim_oracle.simulate(parent, gen, smp, alpha, beta, weight, p0uu, L, seed, missing_rate=float(rate))
        status[rows], post[rows], meth[rows] = st[rows], po[rows], me[rows]
    return status, post, meth


def row_ij(pairs):
    return np.ascontiguousarray(pairs[:, 0].astype(np.int32) | (pairs[:, 1].astype(np.int32) << 16))


def pair_idx(pairs, S):
    i, j = pairs[:, 0].astype(np.int64), pairs[:, 1].astype(np.int64)
    return i * S - i * (i + 1) // 2 + (j - i - 1)


def tree_arrays(name):
    if name == "golden4":
        return arrays_of_files(*golden_files("golden"))
    if name == "golden13":
        return arrays_of_files(*golden_files("desired_output"))
    if name == "forest":
        return two_root_forest()
    return lines_tree(3, 2)


# ---------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed,key", [(0, 0), (7, 3), (0xAB0B200, 12345), (2**63 + 5, 2**40)])
def test_param_boot_seeds_are_pinned(ab, emul, seed, key):
    s = ab.gen_param_boot_seeds(seed, key, 9)
    assert np.array_equal(s, py_seeds(seed, key, 9))
    assert all(emul.emul_param_boot_seed(seed, key, b) == int(s[b]) for b in range(9))
    assert np.array_equal(ab.gen_param_boot_seeds(seed, key, 4), s[:4])
    assert len(set(s.tolist())) == 9 and not np.array_equal(s, ab.gen_param_boot_seeds(seed, key + 1, 9))


def test_param_boot_seed_pinned_value(ab):
    assert int(ab.gen_param_boot_seeds(0xAB0B200, 0, 1)[0]) == int(py_seeds(0xAB0B200, 0, 1)[0])
    assert int(py_seeds(1, 2, 1)[0]) == _mix64(_mix64(_mix64(1 ^ ((6 * 0xD1342543DE82EF95) & M64)) ^ 2) ^ 0)


@pytest.mark.parametrize("tree_name", ["lines3", "golden4", "golden13", "forest"])
@pytest.mark.parametrize("L,missing", [(1, "none"), (255, "uniform"), (257, "per_sample"), (16384 + 300, "per_sample"),
                                       (20000, "uniform")])
def test_tile_body_equals_oracle(ab, oracle, emul, sim_oracle, tree_name, L, missing):
    """the header's walk, bits and popcounts, run with the kernel's tiles and flush points (one-site windows, partial
    tiles, a flush after 64 tiles), equal the oracle's simulation + abref_dmatrix in the integers"""
    parent, gen, smp = tree_arrays(tree_name)
    S = int(smp.sum())
    pairs = sim_oracle.sim_pairs(parent, gen, smp)
    R = len(pairs)
    rng = np.random.default_rng(L + S)
    rates = {"none": np.zeros(S), "uniform": np.full(S, 0.3), "per_sample": rng.uniform(0, 0.6, S)}[missing]
    if missing == "per_sample":
        rates[0] = 0.0
        rates[-1] = 1.0
    alpha, beta, weight, p0uu = 3e-3, 6e-3, 0.4, 0.6
    thr_node = sim_oracle.sim_thresholds(parent, gen, alpha, beta, weight, p0uu)
    seed = int(ab.gen_param_boot_seeds(77, 5, 1)[0])
    for thr in (0.99, 0.5):
        diff, cnt = np.empty(R, np.uint64), np.empty(R, np.uint64)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        ij = row_ij(pairs)
        assert emul.emul_psim_counts(len(parent), p(parent), p(smp), p(thr_node), p(rates), thr, seed, L, R, p(ij), p(diff),
                                     p(cnt)) == 0
        status, post, _ = oracle_simulate_rates(sim_oracle, parent, gen, smp, alpha, beta, weight, p0uu, rates, L, seed)
        _, od, oc = oracle.dmatrix(status, post, thr)
        k = pair_idx(pairs, S)
        assert np.array_equal(diff, od[k]) and np.array_equal(cnt, oc[k]), (thr, tree_name)


def _call(ab, ctx_h, tree, probs, n_sites, missing=None, best=None, n_boot=4):
    n = len(probs)
    best = np.zeros(n, dtype=ab.FIT_DTYPE) if best is None else best
    rows = np.empty((n, n_boot, 7))
    ns = np.ascontiguousarray(n_sites, dtype=np.int64)
    ms = None if missing is None else np.ascontiguousarray(missing, dtype=np.float64)
    return ab._lib.abfit_param_boot_batch(ctx_h, tree._h, ab._pack_problems(probs), n, ab._ptr(ns), ab._ptr(ms), 0.99,
                                          ab._ptr(best), n_boot, 1, 0, None, 100, DBL_EPSILON, 0, ab._ptr(rows), None, None,
                                          None, None, None, None, None)


def test_refusals_before_any_device_work(ab):
    tree = ab.SimTree.lines(3, [1, 2])
    S, R = tree.n_samples, tree.n_pairs
    ped = np.column_stack([tree.pairs()[:, 2:5], np.full(R, 0.05)])
    probs = [ab.Problem(ped, 0.7, 0.7, 1.0)] * 2
    err = lambda: ab._lib.abfit_last_error().decode()
    bad = ped.copy()
    bad[3, 1] += 1
    assert _call(ab, None, tree, [probs[0], ab.Problem(bad, 0.7, 0.7, 1.0)], [10, 10]) == -1
    assert "problem 1, pedigree row 3" in err()
    assert _call(ab, None, tree, [ab.Problem(ped[:-1], 0.7, 0.7, 1.0)], [10]) == -1 and "pedigree rows" in err()
    for ns in ([10, 0], [10, -5]):
        assert _call(ab, None, tree, probs, ns) == -1 and "window 1 has no sites" in err()
    assert _call(ab, None, tree, probs, [10, 2**31]) == -5 and "2^31" in err()
    for m in (1.5, -0.1, np.nan):
        miss = np.zeros((2, S))
        miss[1, 2] = m
        assert _call(ab, None, tree, probs, [10, 10], miss) == -1 and "window 1, sample 2" in err()
    assert _call(ab, None, tree, probs, [10, 10], n_boot=70000) == -5
    big = ab.SimTree.lines(201, [1])  # 201 samples (a star of founder + 201 children)
    bped = np.column_stack([big.pairs()[:, 2:5], np.full(big.n_pairs, 0.05)])
    assert _call(ab, None, big, [ab.Problem(bped, 0.7, 0.7, 1.0)], [10]) == -5 and "at most 200" in err()
    with pytest.raises(ValueError):
        ab.Context.parametric_bootstrap(None, tree, probs, [10], None, np.zeros(2, ab.FIT_DTYPE), 4, 1)
    with pytest.raises(ValueError):
        ab.Context.parametric_bootstrap(None, tree, probs, [10, 10], np.zeros((2, S + 1)), np.zeros(2, ab.FIT_DTYPE), 4, 1)


def test_shared_memory_limit_is_the_kernel_layout(emul):
    """the host refuses a forest exactly when the kernel's shared-memory layout exceeds a block's opt-in limit"""
    assert emul.emul_psim_smem_bytes(201, 200, 19900) == 8 * 201 + 8 * 200 + 96 * 200 + 4 * 19900 + 256 * 201
    n = max_accepted_nodes(emul)
    assert emul.emul_psim_smem_bytes(n, 200, 19900) <= SMEM_OPTIN < emul.emul_psim_smem_bytes(n + 1, 200, 19900)


def max_accepted_nodes(emul, S=200, R=19900):
    n = 1
    while emul.emul_psim_smem_bytes(n + 1, S, R) <= SMEM_OPTIN:
        n += 1
    return n


def _cli(args, cwd):
    return subprocess.run([os.path.join(ROOT, "alphabeta-rs_b200", "alphabeta")] + args, cwd=cwd, capture_output=True,
                          text=True, timeout=300)


def test_alphabeta_cli_refusals(tmp_path):
    nl, el = os.path.join(GOLDEN, "nodelist.txt"), os.path.join(GOLDEN, "edgelist.txt")
    r = _cli(["-n", nl, "-e", el, "-o", str(tmp_path), "--site-bootstrap", "5", "--parametric-bootstrap", "3"], str(tmp_path))
    assert r.returncode == 2 and "cannot be used together" in r.stderr
    r = _cli(["-n", nl, "-e", el, "-o", str(tmp_path), "--parametric-bootstrap", "0"], str(tmp_path))
    assert r.returncode == 2
    # a node with two parents is not a forest: refused, naming the node, before any device work
    edges = open(el).read().rstrip("\n") + "\n1_8\t2_2\t0\n"
    bad = tmp_path / "edgelist.txt"
    bad.write_text(edges)
    r = _cli(["-n", nl, "-e", str(bad), "-o", str(tmp_path), "--parametric-bootstrap", "3", "--device", "999"], str(tmp_path))
    assert r.returncode == 1 and "node 2_2 has two parents" in r.stdout, r.stdout + r.stderr


# ---------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------
def fitted_best(ab, theta, lse=0.0):
    best = np.zeros(len(theta), dtype=ab.FIT_DTYPE)
    best["theta"] = theta
    best["lse"] = lse
    return best


def problems_of(ab, tree, D, p0uu):
    ped = np.column_stack([tree.pairs()[:, 2:5], D])
    return ab.Problem(ped, p0uu, p0uu, 1.0)


def materialised_dstar(ab, ctx, tree, theta, p0uu, L, rate, seed, key, n_boot, thr=0.99):
    """abfit_simulate then abfit_divergence, + theta3, for every replicate of one window"""
    pr = tree.pairs()
    k = pair_idx(pr, tree.n_samples)
    out = np.empty((n_boot, len(pr)))
    for b, s in enumerate(ab.gen_param_boot_seeds(seed, key, n_boot)):
        st, po, me = ctx.simulate(tree, theta[0], theta[1], theta[2], p0uu, L=L, seed=int(s), missing_rate=rate)
        out[b] = ctx.dmatrix(st, po, me, thr)["D"][0][k] + theta[3]
    return out


def sim_tree(ab, name):
    if name == "lines3":
        return ab.SimTree.lines(3, [1, 2])
    return ab.SimTree(*tree_arrays(name))


@pytest.mark.gpu
@pytest.mark.parametrize("tree_name", ["lines3", "golden4", "golden13", "forest"])
def test_dstar_equals_materialising_route(ab, ctx, tree_name):
    tree = sim_tree(ab, tree_name)
    R = tree.n_pairs
    n_sites = [1, 255, 16384 + 257, 4000]  # a one-site window, partial tiles, two blocks of tiles
    rates = [0.0, 0.2, 0.05, 0.5]
    theta = np.array([[3e-3, 6e-3, 0.4, 0.0], [1e-2, 2e-3, 0.9, 0.01], [2e-4, 5e-4, 0.1, -0.003], [0.2, 0.3, 0.5, 1e-3]])
    p0 = [0.6, 0.3, 0.9, 0.5]
    probs = [problems_of(ab, tree, np.full(R, 0.05), p0[p]) for p in range(4)]
    n_boot = 5
    res = ctx.parametric_bootstrap(tree, probs, n_sites, np.repeat(np.array(rates)[:, None], tree.n_samples, 1),
                                   fitted_best(ab, theta), n_boot, 31, problem_ids=[9, 3, 2**40, 0], max_iters=2)
    assert np.all(res["window_status"] == 0)
    for p, key in enumerate([9, 3, 2**40, 0]):
        want = materialised_dstar(ab, ctx, tree, theta[p], p0[p], n_sites[p], rates[p], 31, key, n_boot)
        assert np.array_equal(res["dstar"][p].view(np.uint64), want.view(np.uint64)), p
        assert res["nan_reps"][p] == int(np.isnan(want).any(axis=1).sum())


@pytest.mark.gpu
def test_dstar_per_sample_missing_equals_oracle(ab, ctx, oracle, sim_oracle):
    parent, gen, smp = tree_arrays("golden13")
    tree = ab.SimTree(parent, gen, smp)
    S, R, L = tree.n_samples, tree.n_pairs, 3000
    rates = np.linspace(0.0, 0.9, S)
    theta = np.array([[3e-3, 6e-3, 0.4, 0.002]])
    res = ctx.parametric_bootstrap(tree, [problems_of(ab, tree, np.full(R, 0.05), 0.7)], [L], rates[None],
                                   fitted_best(ab, theta), 3, 5, first_problem_id=12, max_iters=2)
    k = pair_idx(tree.pairs(), S)
    for b, s in enumerate(ab.gen_param_boot_seeds(5, 12, 3)):
        st, po, _ = oracle_simulate_rates(sim_oracle, parent, gen, smp, 3e-3, 6e-3, 0.4, 0.7, rates, L, int(s))
        D, _, _ = oracle.dmatrix(st, po, 0.99)
        assert np.array_equal(res["dstar"][0][b].view(np.uint64), (D[k] + 0.002).view(np.uint64)), b


def c5_tree(ab, extra_nodes=0):
    """the 201-node C5 tree (20 lines x generations 1..10, 200 samples), with unsampled leaves under the founder"""
    parent, gen, smp = lines_tree(20, 10)
    parent = np.concatenate([parent, np.zeros(extra_nodes, np.int32)])
    gen = np.concatenate([gen, np.ones(extra_nodes, np.int32)])
    smp = np.concatenate([smp, np.zeros(extra_nodes, np.uint8)])
    return ab.SimTree(parent, gen, smp)


def materialised_dstar_device(ab, ctx, tree, theta, p0uu, L, rate, seed, key, n_boot):
    import torch

    S = tree.n_samples
    dev = torch.device("cuda", 0)
    st = torch.empty((S, L), dtype=torch.uint8, device=dev)
    po = torch.empty((S, L), dtype=torch.float64, device=dev)
    me = torch.empty((S, L), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    k = pair_idx(tree.pairs(), S)
    out = np.empty((n_boot, tree.n_pairs))
    for b, s in enumerate(ab.gen_param_boot_seeds(seed, key, n_boot)):
        ctx.simulate_device(tree, st.data_ptr(), po.data_ptr(), me.data_ptr(), theta[0], theta[1], theta[2], p0uu, L=L,
                            seed=int(s), missing_rate=rate)
        D = ctx.dmatrix_device(st.data_ptr(), po.data_ptr(), me.data_ptr(), S, L, seg_offsets=np.array([0, L]))["D"][0]
        out[b] = D[k] + theta[3]
    return out


@pytest.mark.gpu
def test_dstar_c5_200_samples_200k_sites(ab, ctx):
    tree = c5_tree(ab)
    assert tree.n_nodes == 201 and tree.n_samples == 200 and tree.n_pairs == 19900
    L, n_boot = 200_000, 2
    theta = np.array([[3e-3, 6e-3, 0.45, 0.004]])
    prob = problems_of(ab, tree, np.full(19900, 0.05), 0.65)
    res = ctx.parametric_bootstrap(tree, [prob], [L], np.full((1, 200), 0.05), fitted_best(ab, theta), n_boot, 3,
                                   max_iters=1)
    want = materialised_dstar_device(ab, ctx, tree, theta[0], 0.65, L, 0.05, 3, 0, n_boot)
    assert np.array_equal(res["dstar"][0].view(np.uint64), want.view(np.uint64))


@pytest.mark.gpu
def test_largest_accepted_tree(ab, ctx, emul):
    n = max_accepted_nodes(emul)
    tree = c5_tree(ab, n - 201)
    assert tree.n_nodes == n
    L, n_boot = 3000, 2
    theta = np.array([[3e-3, 6e-3, 0.45, 0.0]])
    prob = problems_of(ab, tree, np.full(19900, 0.05), 0.65)
    res = ctx.parametric_bootstrap(tree, [prob], [L], None, fitted_best(ab, theta), n_boot, 4, max_iters=1)
    want = materialised_dstar_device(ab, ctx, tree, theta[0], 0.65, L, 0.0, 4, 0, n_boot)
    assert np.array_equal(res["dstar"][0].view(np.uint64), want.view(np.uint64))
    with pytest.raises(ab.AbfitError) as e:
        ctx.parametric_bootstrap(c5_tree(ab, n - 200), [prob], [L], None, fitted_best(ab, theta), n_boot, 4, max_iters=1)
    assert e.value.code == -5 and "shared memory" in str(e.value)


def observed_fit(ab, ctx, tree, L, seed, alpha=3e-3, beta=6e-3, n_windows=2, missing=0.0, n_starts=16):
    """n_windows simulated windows of L sites, their problems (true p0uu) and best fits"""
    p0, w = ab.sim_equilibrium(alpha, beta)
    st, po, me = ctx.simulate(tree, alpha, beta, L=n_windows * L, seed=seed, missing_rate=missing)
    seg = np.arange(n_windows + 1, dtype=np.int64) * L
    dm = ctx.dmatrix(st, po, me, 0.99, seg_offsets=seg)
    probs = [ab.Problem(tree.pedigree(dm["D"][p]), p0, p0, 1.0) for p in range(n_windows)]
    sx = np.stack([ab.gen_start_simplices(seed, p, n_starts, float(np.nanmax(pb.pedigree[:, 3]))) for p, pb in enumerate(probs)])
    best = ctx.fit_batch(probs, sx, max_iters=3000, want_all=False).best
    return probs, best


def check_lse_and_p(ab, ctx, probs, best, res, n_boot):
    for p, pb in enumerate(probs):
        f = res["fits"][p]
        ok = f["status"] != -1
        for b in np.flatnonzero(ok):
            ped = pb.pedigree.copy()
            ped[:, 3] = res["dstar"][p][b]
            _, lse = ctx.cost_batch([ab.Problem(ped, pb.p0uu, pb.eqp, pb.eqp_weight)], f["theta"][b][None])
            assert res["lse_star"][p][b].tobytes() == lse[0].tobytes() == f["lse"][b].tobytes(), (p, b)
        assert np.all(np.isnan(res["lse_star"][p][~ok]))
        want = (1 + np.sum(res["lse_star"][p][ok] >= best[p]["lse"])) / (1 + ok.sum())
        assert res["gof_p"][p] == want
        assert np.array_equal(res["analysis"][p].view(np.uint64), ab.analyze(res["rows"][p]).view(np.uint64))


@pytest.mark.gpu
def test_refits_stored_tile_equal_oracle(ab, ctx, oracle, monkeypatch, capfd):
    tree = ab.SimTree(*tree_arrays("golden13"))
    probs, best = observed_fit(ab, ctx, tree, 20_000, seed=2)
    n_boot = 24
    res, err = run_verbose(monkeypatch, capfd, {}, lambda: ctx.parametric_bootstrap(
        tree, probs, [20_000, 7_000], np.full((2, tree.n_samples), 0.1), best, n_boot, 17, first_problem_id=40))
    assert "k_fit_boot<BIG=0,DGIVEN=1>" in err and "k_psim_counts" in err
    flat = {"rows": res["rows"], "fits": res["fits"], "dstar": res["dstar"].reshape(-1)}
    check_refits(ab, oracle, probs, best, flat, n_boot, 17, [40, 41])
    check_lse_and_p(ab, ctx, probs, best, res, n_boot)


@pytest.mark.gpu
def test_refits_warp_per_fit_equal_oracle(ab, ctx, oracle, monkeypatch, capfd):
    tree = c5_tree(ab)
    theta = np.array([[3e-3, 6e-3, 0.4, 0.01]])
    prob = problems_of(ab, tree, np.full(19900, 0.05), 0.65)
    best = fitted_best(ab, theta, lse=1e-3)
    n_boot = 3
    res, err = run_verbose(monkeypatch, capfd, {"ABFIT_DEV_WIDE": "1"}, lambda: ctx.parametric_bootstrap(
        tree, [prob], [20_000], None, best, n_boot, 8, max_iters=1000))
    assert "k_fit_wide<boot,DGIVEN=1>" in err
    flat = {"rows": res["rows"], "fits": res["fits"], "dstar": res["dstar"].reshape(-1)}
    check_refits(ab, oracle, [prob], best, flat, n_boot, 8, [0])
    check_lse_and_p(ab, ctx, [prob], best, res, n_boot)


@pytest.mark.gpu
def test_windows_that_cannot_be_simulated_and_keys(ab, ctx):
    """status-1 windows get NaN and no launch, and leave the other windows as they are; a window's replicates depend on
    its key alone, not on the call's other windows"""
    tree = ab.SimTree(*tree_arrays("golden4"))
    probs, best = observed_fit(ab, ctx, tree, 5000, seed=3, n_windows=3)
    n_boot, kw = 12, dict(max_iters=300)
    ids = [70, 71, 72]
    full = ctx.parametric_bootstrap(tree, probs, [5000] * 3, None, best, n_boot, 5, problem_ids=ids, **kw)
    assert np.all(full["window_status"] == 0)
    for bad_theta, bad_p0 in (((-1e-4, 6e-3, 0.4, 0.0), None), ((3e-3, 1.5, 0.4, 0.0), None),
                              ((3e-3, 6e-3, np.nan, 0.0), None), ((3e-3, 6e-3, 0.4, np.inf), None), (None, 1.2)):
        b2 = best.copy()
        p2 = list(probs)
        if bad_theta is not None:
            b2[1]["theta"] = bad_theta
        else:
            p2[1] = ab.Problem(probs[1].pedigree, bad_p0, bad_p0, 1.0)
        r = ctx.parametric_bootstrap(tree, p2, [5000] * 3, None, b2, n_boot, 5, problem_ids=ids, **kw)
        assert r["window_status"].tolist() == [0, 1, 0]
        for k in ("rows", "dstar", "lse_star", "analysis"):
            assert np.all(np.isnan(r[k][1])), k
            assert np.array_equal(r[k][[0, 2]].view(np.uint64), full[k][[0, 2]].view(np.uint64)), k
        assert np.isnan(r["gof_p"][1]) and np.array_equal(r["gof_p"][[0, 2]], full["gof_p"][[0, 2]])
        assert np.all(r["fits"]["status"][1] == -1) and r["nan_reps"][1] == 0
    one = ctx.parametric_bootstrap(tree, probs[1:2], [5000], None, best[1:2], n_boot, 5, problem_ids=[71], **kw)
    tail = ctx.parametric_bootstrap(tree, probs[1:], [5000] * 2, None, best[1:], n_boot, 5, first_problem_id=71, **kw)
    for k in ("rows", "dstar", "lse_star", "gof_p"):
        assert np.array_equal(one[k][0].view(np.uint64), full[k][1].view(np.uint64)), k
        assert np.array_equal(tail[k].view(np.uint64), full[k][1:].view(np.uint64)), k


@pytest.mark.gpu
def test_zero_count_replicates(ab, ctx):
    """every site missing in one sample: every replicate has a cnt = 0 row, none is fitted"""
    tree = ab.SimTree.lines(2, [1, 2])
    S, R = tree.n_samples, tree.n_pairs
    miss = np.zeros((1, S))
    miss[0, 1] = 1.0
    res = ctx.parametric_bootstrap(tree, [problems_of(ab, tree, np.full(R, 0.05), 0.7)], [500], miss,
                                   fitted_best(ab, np.array([[3e-3, 6e-3, 0.4, 0.0]])), 6, 2, max_iters=50)
    assert res["nan_reps"][0] == 6 and np.all(np.isnan(res["rows"])) and np.all(res["fits"]["status"] == -1)
    assert np.isnan(res["lse_star"]).all() and res["gof_p"][0] == 1.0


@pytest.mark.gpu
def test_too_large_is_refused(ab, ctx):
    """40 windows x 65 535 replicates x 19 900 rows of D*: 417 GB, refused before any launch; the context works after"""
    tree = c5_tree(ab)
    prob = problems_of(ab, tree, np.full(19900, 0.05), 0.65)
    best = fitted_best(ab, np.tile([3e-3, 6e-3, 0.4, 0.0], (40, 1)))
    assert _call(ab, ctx._h, tree, [prob] * 40, [1000] * 40, best=best, n_boot=65535) == -5
    assert "device memory" in ab._lib.abfit_last_error().decode()
    small = ab.SimTree.lines(3, [1, 2])
    probs, best = observed_fit(ab, ctx, small, 2000, seed=1, n_windows=1)
    r = ctx.parametric_bootstrap(small, probs, [2000], None, best, 8, 5, max_iters=100)
    assert r["rows"].shape == (1, 8, 7) and not np.isnan(r["rows"]).any()


def _library_run(ab, ctx, cwd, nl, el, n, n_boot, seed):
    """what `alphabeta --parametric-bootstrap` computes, through the library: fit, per-sample missing rates of the
    methylomes read as the tool reads them, parametric bootstrap on the forest of the same files"""
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
    missing = 1.0 - (post >= 0.99).sum(axis=1) / L
    return best, ctx.parametric_bootstrap(ab.SimTree.from_files(nl, el), [prob], [L], missing[None], best, n_boot, seed)


@pytest.mark.gpu
def test_alphabeta_cli_parametric_bootstrap_equals_library(ab, ctx, tmp_path):
    """simulated methylomes of the golden 13-sample design (the `simulate` tool): raw.npy, analysis.txt and
    goodness_of_fit.txt of `alphabeta --parametric-bootstrap 30` are the library's"""
    from test_simulate import SIM

    sim = tmp_path / "sim"
    nl0, el0 = golden_files("desired_output")
    r = subprocess.run([SIM, "-n", nl0, "-e", el0, "--alpha", "0.004", "--beta", "0.008", "--sites", "20000", "--seed", "11",
                        "--missing-rate", "0.05", "-o", str(sim)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = tmp_path / "out"
    out.mkdir()
    nl, el = str(sim / "nodelist.txt"), str(sim / "edgelist.txt")
    n, n_boot, seed = 40, 30, 99
    r = _cli(["-n", nl, "-e", el, "-i", str(n), "-o", str(out), "--seed", str(seed), "--parametric-bootstrap", str(n_boot)],
             str(tmp_path))
    assert r.returncode == 0, r.stdout + r.stderr
    best, res = _library_run(ab, ctx, str(tmp_path), nl, el, n, n_boot, seed)
    assert res["window_status"][0] == 0
    assert np.array_equal(np.load(str(out / "raw.npy")).view(np.uint64), res["rows"][0].view(np.uint64))
    ab.write_analysis(str(tmp_path / "lib_analysis.txt"), res["analysis"][0])
    assert (out / "analysis.txt").read_text() == (tmp_path / "lib_analysis.txt").read_text()
    fitted = int((res["fits"]["status"][0] != -1).sum())
    want = (f"observed_lse\t{ab.format_f64(best[0]['lse'])}\np\t{ab.format_f64(res['gof_p'][0])}\n"
            f"replicates_fitted\t{fitted}\nnan_replicates\t{res['nan_reps'][0]}\n")
    assert (out / "goodness_of_fit.txt").read_text() == want
    assert (out / "bootstrap.png").stat().st_size > 0


@pytest.mark.gpu
def test_alphabeta_cli_refuses_a_fit_it_cannot_simulate(ab, ctx, tmp_path):
    """the golden 4-sample methylomes fit a weight outside [0, 1]: the library gives the window status 1, the tool an
    error"""
    cwd = _golden_cwd(tmp_path)
    nl, el = os.path.join(GOLDEN, "nodelist.txt"), os.path.join(GOLDEN, "edgelist.txt")
    r = _cli(["-n", nl, "-e", el, "-i", "40", "-o", cwd, "--seed", "99", "--parametric-bootstrap", "30"], cwd)
    _, res = _library_run(ab, ctx, cwd, nl, el, 40, 30, 99)
    assert res["window_status"][0] == 1 and np.isnan(res["gof_p"][0])
    assert r.returncode == 1 and "cannot be simulated" in r.stdout, r.stdout + r.stderr


def _gof_rates(ab, ctx, violate, n_windows, seed):
    """fraction of windows with p < 0.05 on golden13 (the R-original design), 500 000 sites per window, 100 replicates:
    data simulated from ABneutral, or (violate) half the sites at alpha, beta and half at 10 alpha, 10 beta"""
    import torch

    tree = ab.SimTree(*tree_arrays("golden13"))
    S, L, alpha, beta = tree.n_samples, 500_000, 3e-3, 6e-3
    dev = torch.device("cuda", 0)
    st = torch.empty((S, n_windows * L), dtype=torch.uint8, device=dev)
    po = torch.empty((S, n_windows * L), dtype=torch.float64, device=dev)
    me = torch.empty((S, n_windows * L), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    p0, w = ab.sim_equilibrium(alpha, beta)
    if violate:  # window w = [L/2 sites at (alpha, beta) | L/2 sites at (10 alpha, 10 beta)]
        h = L // 2
        parts = []
        for k, (a, b) in enumerate(((alpha, beta), (10 * alpha, 10 * beta))):
            s2 = torch.empty((S, n_windows * h), dtype=torch.uint8, device=dev)
            p2 = torch.empty((S, n_windows * h), dtype=torch.float64, device=dev)
            m2 = torch.empty((S, n_windows * h), dtype=torch.float64, device=dev)
            torch.cuda.synchronize()
            ctx.simulate_device(tree, s2.data_ptr(), p2.data_ptr(), m2.data_ptr(), a, b, w, p0, L=n_windows * h,
                                seed=seed + k)
            parts.append((s2.view(S, n_windows, h), p2.view(S, n_windows, h), m2.view(S, n_windows, h)))
        st.view(S, n_windows, L).copy_(torch.cat([parts[0][0], parts[1][0]], 2))
        po.view(S, n_windows, L).copy_(torch.cat([parts[0][1], parts[1][1]], 2))
        me.view(S, n_windows, L).copy_(torch.cat([parts[0][2], parts[1][2]], 2))
        del parts
        torch.cuda.synchronize()
    else:
        ctx.simulate_device(tree, st.data_ptr(), po.data_ptr(), me.data_ptr(), alpha, beta, w, p0, L=n_windows * L, seed=seed)
    seg = np.arange(n_windows + 1, dtype=np.int64) * L
    dm = ctx.dmatrix_device(st.data_ptr(), po.data_ptr(), me.data_ptr(), S, n_windows * L, seg_offsets=seg)
    del st, po, me
    probs = [ab.Problem(tree.pedigree(dm["D"][p]), p0, p0, 1.0) for p in range(n_windows)]
    sx = np.stack([ab.gen_start_simplices(seed, p, 32, float(pb.pedigree[:, 3].max())) for p, pb in enumerate(probs)])
    best = ctx.fit_batch(probs, sx, max_iters=10000, want_all=False).best
    res = ctx.parametric_bootstrap(tree, probs, [L] * n_windows, None, best, 100, seed)
    ok = res["window_status"] == 0
    return float(np.mean(res["gof_p"][ok] < 0.05)), int(ok.sum()), res


@pytest.mark.gpu
def test_calibration_under_the_model(ab, ctx):
    rate, n_ok, res = _gof_rates(ab, ctx, False, 64, 101)
    print(f"ABneutral data: {rate:.3f} of {n_ok} windows have p < 0.05; p quartiles "
          f"{np.nanpercentile(res['gof_p'], [25, 50, 75])}")
    assert n_ok == 64 and rate <= 0.15


@pytest.mark.gpu
def test_power_against_mixed_rates(ab, ctx):
    rate, n_ok, res = _gof_rates(ab, ctx, True, 32, 202)
    print(f"mixed-rate data: {rate:.3f} of {n_ok} windows have p < 0.05; p quartiles "
          f"{np.nanpercentile(res['gof_p'], [25, 50, 75])}")
    assert n_ok >= 16 and rate > 0.5
