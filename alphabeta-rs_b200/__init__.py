"""abfit-b200 — Python binding (ctypes) of libabfit, the sm_100a implementation of the
alphabeta-rs model-fitting hot path.

This module is plumbing for tests and bench.py: it loads the in-tree ``libabfit.so`` and
exposes the C ABI of ``include/abfit.h`` with numpy arrays, under names that mirror the
reference's Rust interface (``ab_neutral_run`` = ``ab_neutral::run`` src/ab_neutral.rs:13,
``boot_model_run`` = ``boot_model::run`` src/boot_model.rs:17, ``Problem.cost`` =
``CostFunction::cost`` src/structs.rs:194, ``divergence`` = src/divergence.rs:33,
``dmatrix`` = ``DMatrix::from`` src/pedigree.rs:214).

There is no CPU fallback anywhere in the product path: if the CUDA library is missing the
import fails, and without a CUDA device every compute call raises ``AbfitError``.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import weakref
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libabfit.so")

DBL_EPSILON = 2.220446049250313e-16

# flags (include/abfit.h)
SHRINK_ON_FAILED_CONTRACTION = 1
NO_EARLY_EXIT_ON_STALL = 2

TERM_SD, TERM_MAX_ITERS, TERM_STALLED, FIT_NAN = 1, 2, 3, -1
ERR_ARG, ERR_CUDA, ERR_TIME, ERR_NAN, ERR_TOO_LARGE, ERR_STATE = -1, -2, -3, -4, -5, -6


class AbfitError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"abfit error {code}: {msg}")
        self.code = code


class _Problem(C.Structure):
    _fields_ = [
        ("pedigree", C.POINTER(C.c_double)),
        ("n_pairs", C.c_int32),
        ("p0uu", C.c_double),
        ("eqp", C.c_double),
        ("eqp_weight", C.c_double),
    ]


FIT_DTYPE = np.dtype(
    [
        ("theta", "<f8", (4,)),
        ("cost", "<f8"),
        ("lse", "<f8"),
        ("iters", "<i4"),
        ("evals", "<i4"),
        ("status", "<i4"),
        ("start_id", "<i4"),
    ],
    align=True,
)
assert FIT_DTYPE.itemsize == 64


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found — build it first (python -c 'import __graft_entry__ as g; g.build()' "
            "or make -C alphabeta-rs_b200). abfit-b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, u32, u64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_double
    PP = C.POINTER(_Problem)
    sig = {
        "abfit_last_error": (C.c_char_p, []),
        "abfit_version": (C.c_char_p, []),
        "abfit_ctx_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
        "abfit_ctx_destroy": (None, [vp]),
        "abfit_ctx_info": (C.c_int, [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i64)]),
        "abfit_measure_fp64_peak": (C.c_int, [vp, C.POINTER(dbl)]),
        "abfit_ctx_timer_start": (C.c_int, [vp]),
        "abfit_ctx_timer_stop": (C.c_int, [vp, C.POINTER(C.c_float)]),
        "abfit_ctx_sync": (C.c_int, [vp]),
        "abfit_gen_start_simplices": (None, [u64, u64, i32, dbl, vp]),
        "abfit_gen_vary_vertices": (None, [u64, u64, i32, vp, vp]),
        "abfit_gen_resample_idx": (None, [u64, u64, i32, i32, vp]),
        "abfit_gen_vary_vertices_batch": (None, [u64, u64, i32, i32, vp, vp]),
        "abfit_device_count": (C.c_int, []),
        "abfit_alphabeta_batch_multi": (C.c_int, [vp, i32, vp, i32, i32, vp, i32, vp, u64, u64, vp, i32, i32, dbl, u32, vp, vp, vp, vp, vp, vp]),
        "abfit_divergence_multi": (C.c_int, [vp, i32, vp, vp, vp, i32, i64, vp, i32, dbl, vp, vp, vp, vp, vp, vp]),
        "abfit_alphabeta_batch": (C.c_int, [vp, PP, i32, i32, vp, i32, vp, u64, u64, i32, i32, dbl, u32, vp, vp, vp, vp, vp, vp]),
        "abfit_cost_batch": (C.c_int, [vp, PP, i32, vp, vp, i32, vp, vp]),
        "abfit_model_divergence": (C.c_int, [vp, PP, vp, vp, vp]),
        "abfit_fit_batch": (C.c_int, [vp, PP, i32, i32, vp, i32, dbl, u32, vp, vp, vp, vp, vp]),
        "abfit_boot_batch": (C.c_int, [vp, PP, i32, vp, vp, vp, i32, vp, vp, i32, dbl, u32, vp, vp]),
        "abfit_divergence": (C.c_int, [vp, vp, vp, vp, i32, i64, vp, i32, dbl, vp, vp, vp, vp, vp, vp]),
        "abfit_divergence_device": (C.c_int, [vp, vp, vp, vp, i32, i64, vp, i32, dbl, vp, vp, vp, vp, vp, vp, vp, vp]),
        "abfit_batch_create": (C.c_int, [vp, PP, i32, C.POINTER(vp)]),
        "abfit_batch_destroy": (None, [vp]),
        "abfit_batch_upload_starts": (C.c_int, [vp, i32, vp]),
        "abfit_batch_run_fit": (C.c_int, [vp, i32, dbl, u32]),
        "abfit_batch_download_fit": (C.c_int, [vp, vp, vp, vp, vp, vp]),
        "abfit_batch_upload_boot": (C.c_int, [vp, i32, vp, vp, vp, vp, vp]),
        "abfit_batch_run_boot": (C.c_int, [vp, i32, dbl, u32]),
        "abfit_batch_download_boot": (C.c_int, [vp, vp, vp]),
        "abfit_batch_run_pipelined": (C.c_int, [vp, i32, i32, dbl, u32]),
        "abfit_batch_pipes": (C.c_int, [vp]),
        "abfit_batch_sync": (C.c_int, [vp]),
        "abfit_batch_timing": (C.c_int, [vp, vp, vp, C.POINTER(i32)]),
        "abfit_batch_flops_per_eval": (C.c_int, [vp, i32, C.POINTER(dbl), C.POINTER(i32), C.POINTER(i32)]),
        "abfit_batch_fp64_instr_per_eval": (C.c_int, [vp, i32, C.POINTER(dbl)]),
        "abfit_batch_uses_specialised_kernels": (C.c_int, [vp]),
        "abfit_jit_dump": (C.c_int, [vp, C.c_char_p, C.c_char_p, C.POINTER(dbl)]),
        "abfit_jit_last_error": (C.c_char_p, []),
        "abfit_analyze": (C.c_int, [vp, i32, vp]),
        "abfit_parse_methylome_line": (C.c_int, [C.c_char_p, i32, vp, vp, vp, vp]),
        "abfit_parse_methylome_buffer": (C.c_int, [C.c_char_p, i64, i32, i32, i64, vp, vp, vp, vp, vp, vp, vp]),
        "abfit_pedigree_build": (C.c_int, [vp, C.c_char_p, C.c_char_p, dbl, C.POINTER(vp)]),
        "abfit_pedigree_info": (C.c_int, [vp, vp, vp, vp, vp]),
        "abfit_pedigree_graph": (C.c_int, [C.c_char_p, C.c_char_p, vp, C.c_char_p, i32, vp, vp, i32]),
        "abfit_parse_annotation_line": (C.c_int, [C.c_char_p, i32, vp]),
        "abfit_pedigree_rows": (vp, [vp]),
        "abfit_pedigree_warnings": (C.c_char_p, [vp]),
        "abfit_pedigree_free": (None, [vp]),
        "abfit_format_f64": (C.c_int, [dbl, C.c_char_p, i32]),
        "abfit_steady_state": (dbl, [dbl, dbl]),
        "abfit_write_pedigree": (C.c_int, [C.c_char_p, vp, i32]),
        "abfit_write_analysis": (C.c_int, [C.c_char_p, vp]),
        "abfit_format_analysis": (C.c_int, [vp, C.c_char_p, i32]),
        "abfit_write_npy_f64": (C.c_int, [C.c_char_p, vp, i32, vp]),
        "abfit_write_metaprofile_results": (C.c_int, [C.c_char_p, C.c_char_p, i32, vp, vp, vp, vp, vp]),
        "abfit_plot_metaplot": (C.c_int, [C.c_char_p, i32, vp, vp, vp, vp, vp, vp]),
        "abfit_plot_bootstrap": (C.c_int, [C.c_char_p, vp, vp, i32]),
        "abfit_window_counts": (C.c_int, [vp, vp]),
        "abfit_place_sites": (C.c_int, [vp, i32, vp, i64, vp, vp, vp, i64, vp, vp]),
        "abfit_sim_tree_build": (C.c_int, [C.c_char_p, C.c_char_p, C.POINTER(vp)]),
        "abfit_sim_tree_from_arrays": (C.c_int, [i32, vp, vp, vp, C.POINTER(vp)]),
        "abfit_sim_tree_info": (C.c_int, [vp, vp, vp, vp]),
        "abfit_sim_tree_pairs": (C.c_int, [vp, vp, i32]),
        "abfit_sim_tree_thresholds": (C.c_int, [vp, vp, vp]),
        "abfit_sim_tree_free": (None, [vp]),
        "abfit_sim_equilibrium": (C.c_int, [dbl, dbl, C.POINTER(dbl), C.POINTER(dbl)]),
        "abfit_simulate": (C.c_int, [vp, vp, vp, i64, i64, vp, vp, vp]),
        "abfit_simulate_device": (C.c_int, [vp, vp, vp, i64, i64, vp, vp, vp, C.POINTER(C.c_float)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = _load()
EXPORTED_SYMBOLS = (
    "abfit_last_error abfit_version abfit_ctx_create abfit_ctx_destroy abfit_ctx_info abfit_measure_fp64_peak "
    "abfit_ctx_timer_start abfit_ctx_timer_stop abfit_ctx_sync "
    "abfit_gen_start_simplices abfit_gen_vary_vertices abfit_gen_vary_vertices_batch abfit_gen_resample_idx "
    "abfit_alphabeta_batch abfit_cost_batch "
    "abfit_device_count abfit_model_divergence abfit_fit_batch abfit_boot_batch abfit_alphabeta_batch_multi abfit_divergence abfit_divergence_multi abfit_divergence_device abfit_batch_create "
    "abfit_batch_destroy abfit_batch_upload_starts abfit_batch_run_fit abfit_batch_download_fit "
    "abfit_batch_upload_boot abfit_batch_run_boot abfit_batch_download_boot abfit_batch_run_pipelined abfit_batch_pipes abfit_batch_sync "
    "abfit_batch_timing abfit_batch_flops_per_eval abfit_batch_fp64_instr_per_eval abfit_batch_uses_specialised_kernels abfit_jit_dump abfit_jit_last_error abfit_analyze abfit_window_counts abfit_place_sites "
    "abfit_parse_methylome_line abfit_parse_methylome_buffer abfit_parse_annotation_line abfit_pedigree_graph abfit_pedigree_build abfit_pedigree_info abfit_pedigree_rows abfit_pedigree_warnings "
    "abfit_pedigree_free abfit_format_f64 abfit_steady_state abfit_write_pedigree abfit_write_analysis abfit_format_analysis "
    "abfit_write_npy_f64 abfit_write_metaprofile_results abfit_plot_metaplot abfit_plot_bootstrap "
    "abfit_sim_tree_build abfit_sim_tree_from_arrays abfit_sim_tree_info abfit_sim_tree_pairs abfit_sim_tree_thresholds "
    "abfit_sim_tree_free abfit_sim_equilibrium abfit_simulate abfit_simulate_device"
).split()


def _check(rc: int) -> None:
    if rc != 0:
        raise AbfitError(rc, (_lib.abfit_last_error() or b"").decode())


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f64(a, shape=None) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


def version() -> str:
    return _lib.abfit_version().decode()


# ---------------------------------------------------------------------------------------------
# input generators (host, seeded; the same arrays feed the oracle and the GPU)
# ---------------------------------------------------------------------------------------------
def gen_start_simplices(seed: int, problem_id: int, n_starts: int, max_divergence: float) -> np.ndarray:
    """5 x Model::new per start (src/structs.rs:78-96, src/ab_neutral.rs:49-55) -> [n_starts,5,4]."""
    out = np.empty((n_starts, 5, 4), dtype=np.float64)
    _lib.abfit_gen_start_simplices(seed, problem_id, n_starts, float(max_divergence), _ptr(out))
    return out


def gen_vary_vertices(seed: int, problem_id: int, n_boot: int, best_theta) -> np.ndarray:
    """4 x Model::vary per replicate (src/structs.rs:100-128, src/boot_model.rs:71-74) -> [n_boot,4,4]."""
    th = _f64(best_theta, (4,))
    out = np.empty((n_boot, 4, 4), dtype=np.float64)
    _lib.abfit_gen_vary_vertices(seed, problem_id, n_boot, _ptr(th), _ptr(out))
    return out


def gen_resample_idx(seed: int, problem_id: int, n_boot: int, n_pairs: int) -> np.ndarray:
    """residual resampling with replacement (src/boot_model.rs:43-48) -> int32 [n_boot,n_pairs]."""
    out = np.empty((n_boot, n_pairs), dtype=np.int32)
    _lib.abfit_gen_resample_idx(seed, problem_id, n_boot, n_pairs, _ptr(out))
    return out


# ---------------------------------------------------------------------------------------------
# problems
# ---------------------------------------------------------------------------------------------
@dataclass
class Problem:
    """`Problem` of src/structs.rs:12-19. pedigree: [n_pairs,4] rows (t0,t1,t2,D)."""

    pedigree: np.ndarray
    p0uu: float
    eqp: float
    eqp_weight: float

    def __post_init__(self):
        self.pedigree = _f64(self.pedigree)
        if self.pedigree.ndim != 2 or self.pedigree.shape[1] != 4:
            raise ValueError("pedigree must be [n_pairs, 4]")

    @property
    def n_pairs(self) -> int:
        return int(self.pedigree.shape[0])

    def cost(self, theta, ctx: "Context") -> float:
        """CostFunction::cost (src/structs.rs:194-216) evaluated on the GPU."""
        c, _ = ctx.cost_batch([self], np.asarray(theta, dtype=np.float64).reshape(1, 4))
        return float(c[0])


def _pack_problems(probs: Sequence[Problem]):
    arr = (_Problem * len(probs))()
    for i, p in enumerate(probs):
        arr[i].pedigree = p.pedigree.ctypes.data_as(C.POINTER(C.c_double))
        arr[i].n_pairs = p.n_pairs
        arr[i].p0uu = p.p0uu
        arr[i].eqp = p.eqp
        arr[i].eqp_weight = p.eqp_weight
    return arr


def jit_last_error() -> str:
    return (_lib.abfit_jit_last_error() or b"").decode()


def jit_dump(prob: "Problem", source_path: Optional[str] = None, cubin_path: Optional[str] = None) -> float:
    """abfit_jit_dump: the CUDA C++ source specialised for this pedigree (and its sm_100a cubin); returns the NVRTC
    compile time in seconds (0 when the cubin came from the disk cache).  Needs no GPU."""
    arr = _pack_problems([prob])
    secs = C.c_double()
    _check(_lib.abfit_jit_dump(arr, None if source_path is None else source_path.encode(),
                               None if cubin_path is None else cubin_path.encode(), C.byref(secs)))
    return secs.value


def device_count() -> int:
    return int(_lib.abfit_device_count())


def alphabeta_batch_multi(ctxs: Sequence["Context"], probs, simplices, resample_idx, seed, first_problem_id=0,
                          problem_ids=None, max_iters_fit=10000, max_iters_boot=1000, sd_tol=DBL_EPSILON, flags=0):
    """abfit_alphabeta_batch_multi: alphabeta::run for every window, windows sharded over the contexts' GPUs (one host
    thread per device, no collective) -> the dict Context.alphabeta_batch returns, in window order."""
    n_probs = len(probs)
    simplices = _f64(simplices)
    n_starts = simplices.size // (n_probs * 20)
    total = sum(p.n_pairs for p in probs)
    if isinstance(resample_idx, (int, np.integer)):  # a replicate count: the indices are drawn on the device
        idx, n_boot = None, int(resample_idx)
    else:
        idx = np.ascontiguousarray(resample_idx, dtype=np.int32)
        n_boot = idx.size // total
    best = np.zeros(n_probs, dtype=FIT_DTYPE)
    pred, resid = np.empty(total), np.empty(total)
    status = np.zeros(n_probs, dtype=np.int32)
    rows, analysis = np.empty((n_probs, n_boot, 7)), np.empty((n_probs, 32))
    ids = None if problem_ids is None else np.ascontiguousarray(problem_ids, dtype=np.uint64)
    hs = (C.c_void_p * len(ctxs))(*[c._h for c in ctxs])
    _check(_lib.abfit_alphabeta_batch_multi(hs, len(ctxs), _pack_problems(probs), n_probs, n_starts, _ptr(simplices), n_boot,
                                            _ptr(idx), seed, first_problem_id, _ptr(ids), max_iters_fit, max_iters_boot, sd_tol,
                                            flags, _ptr(best), _ptr(pred), _ptr(resid), _ptr(status), _ptr(rows), _ptr(analysis)))
    return {"best": best, "pred": pred, "resid": resid, "status": status, "rows": rows, "analysis": analysis}


def dmatrix_multi(ctxs: Sequence["Context"], status, posterior_max, meth_lvl, thr=0.99, seg_offsets=None):
    """abfit_divergence_multi: windows (or, for one window, the site axis) sharded over the contexts' GPUs"""
    status = np.ascontiguousarray(status, dtype=np.uint8)
    post, meth = _f64(posterior_max), _f64(meth_lvl)
    S, L = status.shape
    seg = None if seg_offsets is None else np.ascontiguousarray(seg_offsets, dtype=np.int64)
    W = 1 if seg is None else len(seg) - 1
    P = S * (S - 1) // 2
    D = np.empty((W, P))
    diff, cnt = np.empty((W, P), dtype=np.uint64), np.empty((W, P), dtype=np.uint64)
    p0uu, methsum, nvalid = np.empty(W), np.empty((W, S)), np.empty((W, S), dtype=np.int64)
    hs = (C.c_void_p * len(ctxs))(*[c._h for c in ctxs])
    _check(_lib.abfit_divergence_multi(hs, len(ctxs), _ptr(status), _ptr(post), _ptr(meth), S, L, _ptr(seg), W, thr, _ptr(D),
                                       _ptr(diff), _ptr(cnt), _ptr(p0uu), _ptr(methsum), _ptr(nvalid)))
    return {"D": D, "diff": diff, "cnt": cnt, "p0uu": p0uu, "methsum": methsum, "nvalid": nvalid}


@dataclass
class FitResult:
    best: np.ndarray  # FIT_DTYPE [n_probs]
    all: Optional[np.ndarray]  # FIT_DTYPE [n_probs, n_starts]
    pred: np.ndarray  # concatenated [sum n_pairs]
    resid: np.ndarray
    status: np.ndarray  # int32 [n_probs]


_live_contexts = weakref.WeakSet()


@atexit.register
def _close_all():
    # release device objects while the CUDA runtime is still loaded (not from __del__ during interpreter teardown)
    for c in list(_live_contexts):
        try:
            c.close()
        except Exception:
            pass


class Context:
    """One CUDA device + stream (abfit_ctx)."""

    def __init__(self, device: int = 0):
        h = C.c_void_p()
        _check(_lib.abfit_ctx_create(device, C.byref(h)))
        self._h = h
        self.device = device
        self._batches = weakref.WeakSet()
        _live_contexts.add(self)

    def close(self):
        """destroys the batches created on this context first (they hold device buffers and a pointer to it)"""
        if getattr(self, "_h", None):
            for b in list(self._batches):
                b.close()
            _lib.abfit_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self):
        sm, khz, mem = C.c_int32(), C.c_int32(), C.c_int64()
        _check(_lib.abfit_ctx_info(self._h, C.byref(sm), C.byref(khz), C.byref(mem)))
        return {"sm_count": sm.value, "sm_clock_khz": khz.value, "mem_bytes": mem.value}

    def timer_start(self):
        _check(_lib.abfit_ctx_timer_start(self._h))

    def timer_stop(self) -> float:
        ms = C.c_float()
        _check(_lib.abfit_ctx_timer_stop(self._h, C.byref(ms)))
        return ms.value

    def sync(self):
        _check(_lib.abfit_ctx_sync(self._h))

    def measure_fp64_peak(self) -> float:
        v = C.c_double()
        _check(_lib.abfit_measure_fp64_peak(self._h, C.byref(v)))
        return v.value

    # -- objective ---------------------------------------------------------------------------
    def cost_batch(self, probs: Sequence[Problem], theta, prob_of_theta=None):
        theta = _f64(theta).reshape(-1, 4)
        B = theta.shape[0]
        pot = None if prob_of_theta is None else np.ascontiguousarray(prob_of_theta, dtype=np.int32)
        cost = np.empty(B)
        lse = np.empty(B)
        arr = _pack_problems(probs)
        _check(_lib.abfit_cost_batch(self._h, arr, len(probs), _ptr(pot), _ptr(theta), B, _ptr(cost), _ptr(lse)))
        return cost, lse

    def divergence(self, prob: Problem, theta):
        """divergence() of src/divergence.rs:33-94 -> (dt1t2 [n_pairs], p_uu)."""
        th = _f64(theta, (4,))
        dt = np.empty(prob.n_pairs)
        puu = C.c_double()
        arr = _pack_problems([prob])
        _check(_lib.abfit_model_divergence(self._h, arr, _ptr(th), _ptr(dt), C.cast(C.byref(puu), C.c_void_p)))
        return dt, puu.value

    # -- ab_neutral::run, batched over windows --------------------------------------------------
    def fit_batch(self, probs: Sequence[Problem], simplices, max_iters=10000, sd_tol=DBL_EPSILON, flags=0,
                  want_all=True) -> FitResult:
        simplices = _f64(simplices)
        n_probs = len(probs)
        n_starts = simplices.size // (n_probs * 20)
        assert simplices.size == n_probs * n_starts * 20
        best = np.zeros(n_probs, dtype=FIT_DTYPE)
        allr = np.zeros((n_probs, n_starts), dtype=FIT_DTYPE) if want_all else None
        total = sum(p.n_pairs for p in probs)
        pred, resid = np.empty(total), np.empty(total)
        status = np.zeros(n_probs, dtype=np.int32)
        arr = _pack_problems(probs)
        _check(
            _lib.abfit_fit_batch(self._h, arr, n_probs, n_starts, _ptr(simplices), max_iters, sd_tol, flags,
                                 _ptr(best), _ptr(allr), _ptr(pred), _ptr(resid), _ptr(status))
        )
        return FitResult(best, allr, pred, resid, status)

    def fit_batch_into(self, probs, simplices, best, pred, resid, status, max_iters=10000, sd_tol=DBL_EPSILON,
                       flags=0, packed=None):
        """abfit_fit_batch writing into caller-owned (e.g. pinned) arrays; no per-start records."""
        n_probs = len(probs)
        n_starts = simplices.size // (n_probs * 20)
        arr = packed if packed is not None else _pack_problems(probs)
        _check(
            _lib.abfit_fit_batch(self._h, arr, n_probs, n_starts, _ptr(simplices), max_iters, sd_tol, flags,
                                 _ptr(best), None, _ptr(pred), _ptr(resid), _ptr(status))
        )

    def boot_batch_into(self, probs, best, pred, resid, resample_idx, vary_vertices, rows, max_iters=1000,
                        sd_tol=DBL_EPSILON, flags=0, packed=None):
        n_probs = len(probs)
        n_boot = vary_vertices.size // (n_probs * 16)
        arr = packed if packed is not None else _pack_problems(probs)
        _check(
            _lib.abfit_boot_batch(self._h, arr, n_probs, _ptr(best), _ptr(pred), _ptr(resid), n_boot,
                                  _ptr(resample_idx), _ptr(vary_vertices), max_iters, sd_tol, flags, _ptr(rows), None)
        )

    # -- alphabeta::run (fit + bootstrap), batched over windows -----------------------------------
    def alphabeta_batch(self, probs, simplices, resample_idx, seed, first_problem_id=0, max_iters_fit=10000,
                        max_iters_boot=1000, sd_tol=DBL_EPSILON, flags=0, best=None, pred=None, resid=None, status=None,
                        rows=None, analysis=None, packed=None):
        """alphabeta::run (src/alphabeta.rs:23-59) for every window in one call -> dict(best, pred, resid, status, rows,
        analysis).  Output arrays may be passed in (e.g. pinned)."""
        n_probs = len(probs)
        simplices = _f64(simplices)
        n_starts = simplices.size // (n_probs * 20)
        total = sum(p.n_pairs for p in probs)
        if isinstance(resample_idx, (int, np.integer)):  # a replicate count: the indices are drawn on the device
            idx, n_boot = None, int(resample_idx)       # (the numbers of gen_resample_idx(seed, window key, ...))
        else:
            idx = np.ascontiguousarray(resample_idx, dtype=np.int32)
            n_boot = idx.size // total
        best = np.zeros(n_probs, dtype=FIT_DTYPE) if best is None else best
        pred = np.empty(total) if pred is None else pred
        resid = np.empty(total) if resid is None else resid
        status = np.zeros(n_probs, dtype=np.int32) if status is None else status
        rows = np.empty((n_probs, n_boot, 7)) if rows is None else rows
        analysis = np.empty((n_probs, 32)) if analysis is None else analysis
        arr = packed if packed is not None else _pack_problems(probs)
        _check(
            _lib.abfit_alphabeta_batch(self._h, arr, n_probs, n_starts, _ptr(simplices), n_boot, _ptr(idx), seed,
                                       first_problem_id, max_iters_fit, max_iters_boot, sd_tol, flags, _ptr(best),
                                       _ptr(pred), _ptr(resid), _ptr(status), _ptr(rows), _ptr(analysis))
        )
        return {"best": best, "pred": pred, "resid": resid, "status": status, "rows": rows, "analysis": analysis}

    # -- boot_model::run, batched over windows ---------------------------------------------------
    def boot_batch(self, probs: Sequence[Problem], best, pred, resid, resample_idx, vary_vertices, max_iters=1000,
                   sd_tol=DBL_EPSILON, flags=0):
        n_probs = len(probs)
        best = np.ascontiguousarray(best, dtype=FIT_DTYPE).reshape(n_probs)
        pred, resid = _f64(pred), _f64(resid)
        vary = _f64(vary_vertices)
        n_boot = vary.size // (n_probs * 16)
        idx = np.ascontiguousarray(resample_idx, dtype=np.int32)
        rows = np.empty((n_probs, n_boot, 7))
        fits = np.zeros((n_probs, n_boot), dtype=FIT_DTYPE)
        arr = _pack_problems(probs)
        _check(
            _lib.abfit_boot_batch(self._h, arr, n_probs, _ptr(best), _ptr(pred), _ptr(resid), n_boot, _ptr(idx),
                                  _ptr(vary), max_iters, sd_tol, flags, _ptr(rows), _ptr(fits))
        )
        return rows, fits

    # -- DMatrix::from + p0uu ------------------------------------------------------------------
    def dmatrix(self, status, posterior_max, meth_lvl, thr=0.99, seg_offsets=None):
        status = np.ascontiguousarray(status, dtype=np.uint8)
        S, L = status.shape
        post, meth = _f64(posterior_max, (S, L)), _f64(meth_lvl, (S, L))
        seg = None if seg_offsets is None else np.ascontiguousarray(seg_offsets, dtype=np.int64)
        W = 1 if seg is None else len(seg) - 1
        P = S * (S - 1) // 2
        D = np.empty((W, P))
        diff = np.empty((W, P), dtype=np.uint64)
        cnt = np.empty((W, P), dtype=np.uint64)
        p0uu = np.empty(W)
        methsum = np.empty((W, S))
        nvalid = np.empty((W, S), dtype=np.int64)
        _check(
            _lib.abfit_divergence(self._h, _ptr(status), _ptr(post), _ptr(meth), S, L, _ptr(seg), W, thr, _ptr(D),
                                  _ptr(diff), _ptr(cnt), _ptr(p0uu), _ptr(methsum), _ptr(nvalid))
        )
        return {"D": D, "diff": diff, "cnt": cnt, "p0uu": p0uu, "methsum": methsum, "nvalid": nvalid}

    def dmatrix_device(self, d_status: int, d_post: int, d_meth: int, S: int, L: int, thr=0.99, seg_offsets=None):
        """abfit_divergence_device: the three [S][L] inputs are DEVICE pointers (ints); returns the dmatrix() dict plus
        kernel_ms = (pack pass, pair pass) and launches"""
        seg = None if seg_offsets is None else np.ascontiguousarray(seg_offsets, dtype=np.int64)
        W = 1 if seg is None else len(seg) - 1
        P = S * (S - 1) // 2
        D = np.empty((W, P))
        diff = np.empty((W, P), dtype=np.uint64)
        cnt = np.empty((W, P), dtype=np.uint64)
        p0uu = np.empty(W)
        methsum = np.empty((W, S))
        nvalid = np.empty((W, S), dtype=np.int64)
        ms = (C.c_float * 2)()
        launches = C.c_int32()
        _check(
            _lib.abfit_divergence_device(self._h, C.c_void_p(d_status), C.c_void_p(d_post), C.c_void_p(d_meth), S, L,
                                         _ptr(seg), W, thr, _ptr(D), _ptr(diff), _ptr(cnt), _ptr(p0uu), _ptr(methsum),
                                         _ptr(nvalid), C.cast(ms, C.c_void_p), C.cast(C.byref(launches), C.c_void_p))
        )
        return {"D": D, "diff": diff, "cnt": cnt, "p0uu": p0uu, "methsum": methsum, "nvalid": nvalid,
                "kernel_ms": (ms[0], ms[1]), "launches": launches.value}

    def batch(self, probs: Sequence[Problem]) -> "Batch":
        return Batch(self, probs)

    # -- simulated methylomes (ABneutral on a pedigree forest) -----------------------------------
    def simulate(self, tree: "SimTree", alpha, beta, weight=None, p0uu=None, *, L: int, seed: int, missing_rate=0.0,
                 first_site=0):
        """sites [first_site, first_site + L) of every sampled node -> (status u8, posterior_max, meth_lvl), each
        [n_samples, L], the inputs of dmatrix().  weight / p0uu default to the steady state (sim_equilibrium)."""
        prm = _sim_params(alpha, beta, weight, p0uu, missing_rate, seed)
        S = tree.n_samples
        status, post, meth = np.empty((S, L), dtype=np.uint8), np.empty((S, L)), np.empty((S, L))
        _check(_lib.abfit_simulate(self._h, tree._h, C.byref(prm), first_site, L, _ptr(status), _ptr(post), _ptr(meth)))
        return status, post, meth

    def simulate_device(self, tree: "SimTree", d_status: int, d_post: int, d_meth: int, alpha, beta, weight=None, p0uu=None,
                        *, L: int, seed: int, missing_rate=0.0, first_site=0) -> float:
        """simulate() into DEVICE arrays [n_samples][L] (raw pointers, e.g. torch tensors' data_ptr()) of this context's
        device; returns when they are written.  -> device time of the simulation kernel (ms)"""
        prm = _sim_params(alpha, beta, weight, p0uu, missing_rate, seed)
        ms = C.c_float()
        _check(_lib.abfit_simulate_device(self._h, tree._h, C.byref(prm), first_site, L, C.c_void_p(d_status),
                                          C.c_void_p(d_post), C.c_void_p(d_meth), C.byref(ms)))
        return ms.value


class Batch:
    """Device-resident batch of windows (abfit_batch): upload / run / download are separate so
    callers can keep inputs in HBM (bench.py times run_* alone and the whole sequence)."""

    def __init__(self, ctx: Context, probs: Sequence[Problem]):
        self.ctx = ctx
        self.probs = list(probs)
        self.n_probs = len(self.probs)
        self.total_pairs = sum(p.n_pairs for p in self.probs)
        arr = _pack_problems(self.probs)
        h = C.c_void_p()
        _check(_lib.abfit_batch_create(ctx._h, arr, self.n_probs, C.byref(h)))
        self._h = h
        ctx._batches.add(self)
        self.n_starts = 0
        self.n_boot = 0

    def close(self):
        if getattr(self, "_h", None) and getattr(self.ctx, "_h", None):
            _lib.abfit_batch_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload_starts(self, simplices: np.ndarray):
        assert simplices.dtype == np.float64 and simplices.flags.c_contiguous
        self.n_starts = simplices.size // (self.n_probs * 20)
        _check(_lib.abfit_batch_upload_starts(self._h, self.n_starts, _ptr(simplices)))

    def upload_starts_ptr(self, n_starts: int, host_ptr: int):
        self.n_starts = n_starts
        _check(_lib.abfit_batch_upload_starts(self._h, n_starts, C.c_void_p(host_ptr)))

    def run_fit(self, max_iters=10000, sd_tol=DBL_EPSILON, flags=0):
        _check(_lib.abfit_batch_run_fit(self._h, max_iters, sd_tol, flags))

    def download_fit(self, want_all=False, best=None, pred=None, resid=None, status=None) -> FitResult:
        best = np.zeros(self.n_probs, dtype=FIT_DTYPE) if best is None else best
        allr = np.zeros((self.n_probs, self.n_starts), dtype=FIT_DTYPE) if want_all else None
        pred = np.empty(self.total_pairs) if pred is None else pred
        resid = np.empty(self.total_pairs) if resid is None else resid
        status = np.zeros(self.n_probs, dtype=np.int32) if status is None else status
        _check(_lib.abfit_batch_download_fit(self._h, _ptr(best), _ptr(allr), _ptr(pred), _ptr(resid), _ptr(status)))
        return FitResult(best, allr, pred, resid, status)

    def upload_boot(self, resample_idx: np.ndarray, vary_vertices: np.ndarray, best=None, pred=None, resid=None):
        assert resample_idx.dtype == np.int32 and resample_idx.flags.c_contiguous
        assert vary_vertices.dtype == np.float64 and vary_vertices.flags.c_contiguous
        self.n_boot = vary_vertices.size // (self.n_probs * 16)
        if best is not None:
            best = np.ascontiguousarray(best, dtype=FIT_DTYPE)
            pred, resid = _f64(pred), _f64(resid)
        self._keep = (best, pred, resid)
        _check(
            _lib.abfit_batch_upload_boot(self._h, self.n_boot, _ptr(best), _ptr(pred), _ptr(resid),
                                         _ptr(resample_idx), _ptr(vary_vertices))
        )

    def run_boot(self, max_iters=1000, sd_tol=DBL_EPSILON, flags=0):
        _check(_lib.abfit_batch_run_boot(self._h, max_iters, sd_tol, flags))

    def run_pipelined(self, max_iters_fit=10000, max_iters_boot=1000, sd_tol=DBL_EPSILON, flags=0):
        """run_fit + run_boot as one pipelined pass over sub-batches of windows (abfit_batch_run_pipelined)"""
        _check(_lib.abfit_batch_run_pipelined(self._h, max_iters_fit, max_iters_boot, sd_tol, flags))

    def pipes(self) -> int:
        return int(_lib.abfit_batch_pipes(self._h))

    def download_boot(self, want_fits=False, rows=None):
        rows = np.empty((self.n_probs, self.n_boot, 7)) if rows is None else rows
        fits = np.zeros((self.n_probs, self.n_boot), dtype=FIT_DTYPE) if want_fits else None
        _check(_lib.abfit_batch_download_boot(self._h, _ptr(rows), _ptr(fits)))
        return rows, fits

    def sync(self):
        _check(_lib.abfit_batch_sync(self._h))

    def timing(self):
        ms = (C.c_float * 3)()
        ev = (C.c_int64 * 2)()
        launches = C.c_int32()
        _check(_lib.abfit_batch_timing(self._h, C.cast(ms, C.c_void_p), C.cast(ev, C.c_void_p), C.byref(launches)))
        return {"fit_ms": ms[0], "select_ms": ms[1], "boot_ms": ms[2], "evals_fit": ev[0], "evals_boot": ev[1],
                "launches": launches.value}

    def uses_specialised_kernels(self) -> bool:
        return bool(_lib.abfit_batch_uses_specialised_kernels(self._h))

    def flops_per_eval(self, p: int = 0):
        f, u, t = C.c_double(), C.c_int32(), C.c_int32()
        _check(_lib.abfit_batch_flops_per_eval(self._h, p, C.byref(f), C.byref(u), C.byref(t)))
        n = C.c_double()
        _check(_lib.abfit_batch_fp64_instr_per_eval(self._h, p, C.byref(n)))
        return {"flops": f.value, "n_triples": u.value, "tmax": t.value, "fp64_instr": n.value}


# ---------------------------------------------------------------------------------------------
# reference-shaped convenience wrappers (single window)
# ---------------------------------------------------------------------------------------------
def ab_neutral_run(ctx: Context, pedigree, p0uu, eqp, eqp_weight, n_starts, seed=0xAB0B200, problem_id=0,
                   simplices=None, max_iters=10000, flags=0):
    """ab_neutral::run (src/ab_neutral.rs:13-142) -> (model theta[4], predicted divergence, residuals, FitResult)."""
    prob = Problem(pedigree, p0uu, eqp, eqp_weight)
    if simplices is None:
        simplices = gen_start_simplices(seed, problem_id, n_starts, float(np.max(prob.pedigree[:, 3])))
    res = ctx.fit_batch([prob], simplices, max_iters=max_iters, flags=flags)
    if res.status[0] != 0:
        raise AbfitError(int(res.status[0]), "NaN in pedigree or fit (the reference panics here)")
    return res.best[0]["theta"].copy(), res.pred, res.resid, res


def boot_model_run(ctx: Context, pedigree, best_fit, pred, resid, p0uu, eqp, eqp_weight, n_boot, seed=0xAB0B200,
                   problem_id=0, resample_idx=None, vary_vertices=None, max_iters=1000, flags=0):
    """boot_model::run (src/boot_model.rs:17-115) -> (analysis[32], raw rows [n_boot,7])."""
    prob = Problem(pedigree, p0uu, eqp, eqp_weight)
    best = np.ascontiguousarray(best_fit, dtype=FIT_DTYPE).reshape(1)
    if resample_idx is None:
        resample_idx = gen_resample_idx(seed, problem_id, n_boot, prob.n_pairs)
    if vary_vertices is None:
        vary_vertices = gen_vary_vertices(seed, problem_id, n_boot, best[0]["theta"])
    rows, _ = ctx.boot_batch([prob], best, pred, resid, resample_idx, vary_vertices, max_iters=max_iters, flags=flags)
    return analyze(rows[0]), rows[0]


def analyze(rows) -> np.ndarray:
    """RawAnalysis::analyze (src/analysis.rs:50-98): 8 means, 8 sds, 8 (q.025,q.975) pairs."""
    rows = _f64(rows).reshape(-1, 7)
    out = np.empty(32)
    _check(_lib.abfit_analyze(_ptr(rows), rows.shape[0], _ptr(out)))
    return out


# ---------------------------------------------------------------------------------------------
# site -> window assignment (host side of the metaprofile path)
# ---------------------------------------------------------------------------------------------
GENE_DTYPE = np.dtype([("chromosome", "<i4"), ("start", "<u4"), ("end", "<u4"), ("strand", "<i4")])
SITE_DTYPE = GENE_DTYPE  # same layout: chromosome, start, end, strand (+1 / -1 / 0 = '*')


class _WindowArgs(C.Structure):
    _fields_ = [("window_size", C.c_uint32), ("window_step", C.c_uint32), ("cutoff", C.c_uint32),
                ("max_gene_length", C.c_uint32), ("absolute", C.c_int32), ("cutoff_gene_length", C.c_int32)]


def _window_args(window_size, window_step, cutoff, max_gene_length, absolute, cutoff_gene_length):
    return _WindowArgs(window_size, window_step, cutoff, max_gene_length, int(bool(absolute)), int(bool(cutoff_gene_length)))


def window_counts(window_size=5, window_step=0, cutoff=2048, max_gene_length=100, absolute=False,
                  cutoff_gene_length=False):
    """Windows::new (src/windows.rs:28-44) -> (n_upstream, n_gene, n_downstream)"""
    a = _window_args(window_size, window_step, cutoff, max_gene_length, absolute, cutoff_gene_length)
    out = (C.c_int32 * 3)()
    _check(_lib.abfit_window_counts(C.byref(a), out))
    return tuple(out)


def place_sites(genes, sites, window_size=5, window_step=0, cutoff=2048, max_gene_length=100, absolute=False,
                cutoff_gene_length=False, want_assignments=True):
    """Windows::extract's placement loop + Windows::distribution (src/windows.rs:158-165,331-337,
    src/methylation_site.rs:368-490) -> (distribution int32 [n_up+n_gene+n_down], assign_site int64, assign_window int32)"""
    genes = np.ascontiguousarray(genes, dtype=GENE_DTYPE)
    sites = np.ascontiguousarray(sites, dtype=SITE_DTYPE)
    a = _window_args(window_size, window_step, cutoff, max_gene_length, absolute, cutoff_gene_length)
    n = sum(window_counts(window_size, window_step, cutoff, max_gene_length, absolute, cutoff_gene_length))
    dist = np.zeros(n, dtype=np.int32)
    n_assign = C.c_int64()
    _check(_lib.abfit_place_sites(_ptr(genes), len(genes), _ptr(sites), len(sites), C.byref(a), _ptr(dist),
                                  C.byref(n_assign), 0, None, None))
    if not want_assignments:
        return dist, None, None
    cap = n_assign.value
    asite = np.empty(cap, dtype=np.int64)
    awin = np.empty(cap, dtype=np.int32)
    _check(_lib.abfit_place_sites(_ptr(genes), len(genes), _ptr(sites), len(sites), C.byref(a), _ptr(dist),
                                  C.byref(n_assign), cap, _ptr(asite), _ptr(awin)))
    return dist, asite, awin


def segments_from_assignments(assign_site, assign_window, n_windows):
    """(site, window) hits -> (gather order int64 [n_hits], seg_offsets int64 [n_windows+1]): sites of window w are
    order[seg_offsets[w]:seg_offsets[w+1]], in file order (the order Windows::save writes them, src/windows.rs:259-285).
    Gathering status / posteriorMax / rc.meth.lvl columns with `order` gives the [S][L] arrays abfit_divergence takes
    with `seg_offsets` — every window of a metaprofile in one call instead of one directory per window."""
    assign_site = np.asarray(assign_site, dtype=np.int64)
    assign_window = np.asarray(assign_window, dtype=np.int64)
    perm = np.argsort(assign_window, kind="stable")
    counts = np.bincount(assign_window, minlength=n_windows).astype(np.int64)
    seg = np.zeros(n_windows + 1, dtype=np.int64)
    np.cumsum(counts, out=seg[1:])
    return assign_site[perm], seg


# ---------------------------------------------------------------------------------------------
# result files (byte-for-byte the reference's formats)
# ---------------------------------------------------------------------------------------------
def format_f64(v: float) -> str:
    """f64 as Rust's `{}` prints it"""
    buf = C.create_string_buffer(512)
    n = _lib.abfit_format_f64(float(v), buf, 512)
    if n < 0:
        raise AbfitError(n, "format_f64")
    return buf.value.decode()


def steady_state(alpha: float, beta: float) -> float:
    """steady_state (src/alphabeta.rs:71-79)"""
    return _lib.abfit_steady_state(float(alpha), float(beta))


def write_pedigree(path: str, pedigree) -> None:
    """Pedigree::to_file (src/pedigree.rs:81-90)"""
    ped = _f64(pedigree).reshape(-1, 4)
    _check(_lib.abfit_write_pedigree(os.fsencode(path), _ptr(ped), ped.shape[0]))


def write_analysis(path: str, analysis) -> None:
    """Analysis::to_file (src/analysis.rs:102-144) from analyze()'s 32 values"""
    a = _f64(analysis, (32,))
    _check(_lib.abfit_write_analysis(os.fsencode(path), _ptr(a)))


def format_analysis(analysis) -> str:
    a = _f64(analysis, (32,))
    buf = C.create_string_buffer(8192)
    n = _lib.abfit_format_analysis(_ptr(a), buf, 8192)
    if n < 0:
        raise AbfitError(n, "format_analysis")
    return buf.value.decode()


def write_npy(path: str, array) -> None:
    """write_npy of raw.npy (src/cli/alphabeta.rs:34-35)"""
    a = _f64(array)
    shape = np.asarray(a.shape, dtype=np.int64)
    _check(_lib.abfit_write_npy_f64(os.fsencode(path), _ptr(a), a.ndim, _ptr(shape)))


def write_metaprofile_results(path: str, run_name: str, cg_count, region, best, analysis, obs_steady_state) -> None:
    """results.txt of `metaprofile ... alphabeta` (src/cli/metaprofile.rs:74-99)"""
    cg = np.ascontiguousarray(cg_count, dtype=np.int32)
    rg = np.ascontiguousarray(region, dtype=np.int32)
    best = np.ascontiguousarray(best, dtype=FIT_DTYPE)
    an = _f64(analysis).reshape(-1, 32)
    obs = _f64(obs_steady_state)
    _check(_lib.abfit_write_metaprofile_results(os.fsencode(path), run_name.encode(), len(cg), _ptr(cg), _ptr(rg), _ptr(best),
                                                _ptr(an), _ptr(obs)))


def plot_metaplot(path: str, alpha, beta, ci_alpha=None, ci_beta=None) -> None:
    """metaplot.png (src/plot.rs:6-82): alpha / beta per window, ci_* = (lo[n], hi[n]) 95 % bands"""
    a, b = _f64(alpha), _f64(beta)
    cal, cah = (None, None) if ci_alpha is None else (_f64(ci_alpha[0], a.shape), _f64(ci_alpha[1], a.shape))
    cbl, cbh = (None, None) if ci_beta is None else (_f64(ci_beta[0], a.shape), _f64(ci_beta[1], a.shape))
    _check(_lib.abfit_plot_metaplot(os.fsencode(path), len(a), _ptr(a), _ptr(b), _ptr(cal), _ptr(cah), _ptr(cbl), _ptr(cbh)))


def plot_bootstrap(path: str, alphas, betas) -> None:
    """bootstrap.png (src/plot.rs:84-137): box plots of the bootstrap alphas and betas"""
    a = _f64(alphas)
    b = _f64(betas, a.shape)
    _check(_lib.abfit_plot_bootstrap(os.fsencode(path), _ptr(a), _ptr(b), len(a)))


# ---------------------------------------------------------------------------------------------
# input files
# ---------------------------------------------------------------------------------------------
def parse_methylome_line(line: str, invert_strand: bool = False):
    """MethylationSite::from_methylome_file_line (src/methylation_site.rs:146-362) -> dict or None"""
    site = np.zeros(1, dtype=SITE_DTYPE)
    post, lvl, status = C.c_double(), C.c_double(), C.c_int32()
    rc = _lib.abfit_parse_methylome_line(line.encode(), int(invert_strand), _ptr(site), C.cast(C.byref(post), C.c_void_p),
                                         C.cast(C.byref(status), C.c_void_p), C.cast(C.byref(lvl), C.c_void_p))
    if rc == 1:
        return None
    _check(rc)
    return {"chromosome": int(site[0]["chromosome"]), "start": int(site[0]["start"]), "end": int(site[0]["end"]),
            "strand": int(site[0]["strand"]), "posteriormax": post.value, "status": status.value, "meth_lvl": lvl.value}


def parse_methylome_buffer(data: bytes, invert_strand: bool = False, skip_first_line: bool = False, want_lines: bool = False):
    """abfit_parse_methylome_buffer: every line of a methylome file image that parses as a site, in file order ->
    dict of arrays (sites: SITE_DTYPE, posteriormax, status, meth_lvl[, line_off, line_len])"""
    cap = data.count(b"\n") + 1
    sites = np.zeros(cap, dtype=SITE_DTYPE)
    post, lvl = np.zeros(cap), np.zeros(cap)
    status = np.zeros(cap, dtype=np.uint8)
    off = np.zeros(cap if want_lines else 0, dtype=np.int64)
    ln = np.zeros(cap if want_lines else 0, dtype=np.int32)
    n = C.c_int64()
    _check(_lib.abfit_parse_methylome_buffer(data, len(data), int(invert_strand), int(skip_first_line), cap, _ptr(sites), _ptr(post),
                                             _ptr(status), _ptr(lvl), _ptr(off) if want_lines else None,
                                             _ptr(ln) if want_lines else None, C.cast(C.byref(n), C.c_void_p)))
    k = n.value
    out = {"sites": sites[:k], "posteriormax": post[:k], "status": status[:k], "meth_lvl": lvl[:k]}
    if want_lines:
        out["line_off"], out["line_len"] = off[:k], ln[:k]
    return out


def build_pedigree(ctx: Context, nodelist: str, edgelist: str, posterior_max_filter: float = 0.99):
    """Pedigree::build (src/pedigree.rs:92-193): (pedigree [n,4], p0uu, info dict).  File names inside the nodelist are
    relative to the current directory, as in the reference."""
    h = C.c_void_p()
    _check(_lib.abfit_pedigree_build(ctx._h, os.fsencode(nodelist), os.fsencode(edgelist), posterior_max_filter, C.byref(h)))
    try:
        n, p0, ns, nl = C.c_int32(), C.c_double(), C.c_int32(), C.c_int64()
        _check(_lib.abfit_pedigree_info(h, C.cast(C.byref(n), C.c_void_p), C.cast(C.byref(p0), C.c_void_p),
                                        C.cast(C.byref(ns), C.c_void_p), C.cast(C.byref(nl), C.c_void_p)))
        rows = np.ctypeslib.as_array(C.cast(_lib.abfit_pedigree_rows(h), C.POINTER(C.c_double)), shape=(max(n.value, 1), 4))[:n.value].copy() \
            if n.value else np.zeros((0, 4))
        warn = (_lib.abfit_pedigree_warnings(h) or b"").decode()
    finally:
        _lib.abfit_pedigree_free(h)
    return rows, p0.value, {"n_samples": ns.value, "n_sites": nl.value, "warnings": warn}


def parse_annotation_line(line: str, invert_strand: bool = False):
    """Gene::from_annotation_file_line (src/genes.rs:166-216) -> (chromosome, start, end, strand) or None"""
    g = np.zeros(1, dtype=GENE_DTYPE)
    rc = _lib.abfit_parse_annotation_line(line.encode(), int(invert_strand), _ptr(g))
    if rc == 1:
        return None
    _check(rc)
    return (int(g[0]["chromosome"]), int(g[0]["start"]), int(g[0]["end"]), int(g[0]["strand"]))


def pedigree_graph(nodelist: str, edgelist: str):
    """nodelist + edgelist -> (measured files [S], pairs float64 [n_pairs, 5] = i, j, t0, t1, t2)"""
    ns, npairs = C.c_int32(), C.c_int32()
    files = C.create_string_buffer(1 << 20)
    pairs = np.zeros((1 << 16, 5))
    _check(_lib.abfit_pedigree_graph(os.fsencode(nodelist), os.fsencode(edgelist), C.cast(C.byref(ns), C.c_void_p), files,
                                     1 << 20, C.cast(C.byref(npairs), C.c_void_p), _ptr(pairs), 1 << 16))
    return files.value.decode().split("\n")[:-1], pairs[:npairs.value].copy()


# ---------------------------------------------------------------------------------------------
# simulated methylomes: ABneutral run forward on a pedigree forest (include/abfit.h), and design studies
# ---------------------------------------------------------------------------------------------
class _SimParams(C.Structure):
    _fields_ = [("alpha", C.c_double), ("beta", C.c_double), ("weight", C.c_double), ("p0uu", C.c_double),
                ("missing_rate", C.c_double), ("seed", C.c_uint64)]


def sim_equilibrium(alpha: float, beta: float):
    """founders at the model's steady state -> (p0uu, weight): p0uu = p_uu_est(alpha, beta), weight = p_um / (p_um +
    p_mm) (src/alphabeta.rs:62-79).  With p0uu = p_uu_est the fit's penalty target eqp = p0uu agrees with the truth."""
    p, w = C.c_double(), C.c_double()
    _check(_lib.abfit_sim_equilibrium(float(alpha), float(beta), C.byref(p), C.byref(w)))
    return p.value, w.value


def _sim_params(alpha, beta, weight, p0uu, missing_rate, seed) -> _SimParams:
    if weight is None or p0uu is None:
        p_eq, w_eq = sim_equilibrium(alpha, beta)
        weight = w_eq if weight is None else weight
        p0uu = p_eq if p0uu is None else p0uu
    return _SimParams(float(alpha), float(beta), float(weight), float(p0uu), float(missing_rate), int(seed))


class SimTree:
    """A pedigree forest to simulate on (abfit_sim_tree).  SimTree(parent, generation, sampled): parent[v] = -1 for a
    root; SimTree.from_files(nodelist, edgelist): the files of `alphabeta`.  Sampled nodes give the output rows in node
    order; pairs() are their pedigree rows (i, j, t0, t1, t2), the order and values pedigree_graph() gives."""

    def __init__(self, parent, generation, sampled, _handle=None):
        h = _handle
        if h is None:
            par = np.ascontiguousarray(parent, dtype=np.int32)
            gen = np.ascontiguousarray(generation, dtype=np.int32)
            smp = np.ascontiguousarray(sampled, dtype=np.uint8)
            if not (par.ndim == gen.ndim == smp.ndim == 1 and len(par) == len(gen) == len(smp)):
                raise ValueError("parent, generation and sampled must be 1-D arrays of one length")
            h = C.c_void_p()
            _check(_lib.abfit_sim_tree_from_arrays(len(par), _ptr(par), _ptr(gen), _ptr(smp), C.byref(h)))
        self._h = h
        n, s, p = C.c_int32(), C.c_int32(), C.c_int32()
        _check(_lib.abfit_sim_tree_info(h, C.byref(n), C.byref(s), C.byref(p)))
        self.n_nodes, self.n_samples, self.n_pairs = n.value, s.value, p.value

    @classmethod
    def from_files(cls, nodelist: str, edgelist: str) -> "SimTree":
        h = C.c_void_p()
        _check(_lib.abfit_sim_tree_build(os.fsencode(nodelist), os.fsencode(edgelist), C.byref(h)))
        return cls(None, None, None, _handle=h)

    @classmethod
    def lines(cls, n_lines: int, generations, sample_founder: bool = False) -> "SimTree":
        """n_lines lines descending from one founder at generation 0, each sampled at the given generations (e.g. 8
        lines x generations 1..20); unsampled generations in between are not nodes (an edge spans the gap)"""
        gens = sorted(int(g) for g in generations)
        parent, gen, smp = [-1], [0], [1 if sample_founder else 0]
        for _ in range(n_lines):
            prev = 0
            for g in gens:
                parent.append(prev)
                gen.append(g)
                smp.append(1)
                prev = len(gen) - 1
        return cls(parent, gen, smp)

    def pairs(self) -> np.ndarray:
        out = np.empty((max(self.n_pairs, 1), 5))
        _check(_lib.abfit_sim_tree_pairs(self._h, _ptr(out), self.n_pairs))
        return out[:self.n_pairs]

    def thresholds(self, alpha, beta, weight=None, p0uu=None) -> np.ndarray:
        """the per-node draw table [n_nodes, 6] (include/abfit.h, abfit_sim_tree_thresholds)"""
        prm = _sim_params(alpha, beta, weight, p0uu, 0.0, 0)
        out = np.empty((self.n_nodes, 6))
        _check(_lib.abfit_sim_tree_thresholds(self._h, C.byref(prm), _ptr(out)))
        return out

    def pedigree(self, D) -> np.ndarray:
        """[n_pairs, 4] rows (t0, t1, t2, D) from a dmatrix() D row (pair order (0,1),(0,2)..)"""
        pr = self.pairs()
        i, j = pr[:, 0].astype(np.int64), pr[:, 1].astype(np.int64)
        S = self.n_samples
        idx = i * S - i * (i + 1) // 2 + (j - i - 1)
        return np.column_stack([pr[:, 2:5], np.asarray(D)[idx]])

    def close(self):
        if getattr(self, "_h", None):
            _lib.abfit_sim_tree_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def design_study(ctxs, tree: SimTree, alpha, beta, weight=None, p0uu=None, *, L: int, n_replicates: int, n_starts=64,
                 n_boot=100, seed=0, missing_rate=0.0, thr=0.99, use_true_p0uu=True, max_iters_fit=10000,
                 max_iters_boot=1000):
    """How tightly does a design determine alpha and beta?  Simulates n_replicates independent data sets of L sites on
    `tree` and fits every one with alphabeta::run (multi-start fit + bootstrap):
      1. one simulation of n_replicates * L sites into device memory of ctxs[0] (replicate r = sites [r L, (r+1) L));
      2. one observed-divergence call with a window per replicate (dmatrix_device);
      3. one problem per replicate from tree.pairs();
      4. one batched fit (alphabeta_batch, or alphabeta_batch_multi over all contexts); all windows share one pedigree
         time structure, so the batch runs on the specialised kernels when it is large enough.
    use_true_p0uu: the problems' p0uu (and penalty target) is the simulated founder Pr(UU); otherwise the one the
    pipeline estimates from meth_lvl, mean over samples of 1 - mean(meth_lvl) = P(UU) + P(UM) / 2 (the reference's
    estimator, src/pedigree.rs:159-183), which is not P(UU).
    Device memory: 17 bytes per sample-site of n_samples x n_replicates x L.
    -> dict(theta [R,4] best alpha, beta, weight, intercept; status [R] fit status (0 = ok); analysis [R,32]
    (abfit_analyze of the bootstrap); D [R,n_pairs]; p0uu [R] used; truth dict)"""
    import torch

    ctxs = list(ctxs) if isinstance(ctxs, (list, tuple)) else [ctxs]
    prm = _sim_params(alpha, beta, weight, p0uu, missing_rate, seed)
    R, S = int(n_replicates), tree.n_samples
    if R <= 0 or L <= 0 or S < 2 or tree.n_pairs == 0:
        raise ValueError("design_study needs n_replicates > 0, L > 0 and a tree with sampled pairs")
    dev = torch.device("cuda", ctxs[0].device)
    status = torch.empty((S, R * L), dtype=torch.uint8, device=dev)
    post = torch.empty((S, R * L), dtype=torch.float64, device=dev)
    meth = torch.empty((S, R * L), dtype=torch.float64, device=dev)
    torch.cuda.synchronize(dev)
    ctxs[0].simulate_device(tree, status.data_ptr(), post.data_ptr(), meth.data_ptr(), prm.alpha, prm.beta, prm.weight,
                            prm.p0uu, L=R * L, seed=seed, missing_rate=missing_rate)
    seg = np.arange(R + 1, dtype=np.int64) * L
    dm = ctxs[0].dmatrix_device(status.data_ptr(), post.data_ptr(), meth.data_ptr(), S, R * L, thr=thr, seg_offsets=seg)
    del status, post, meth
    p0 = np.full(R, prm.p0uu) if use_true_p0uu else dm["p0uu"]
    probs = [Problem(tree.pedigree(dm["D"][r]), float(p0[r]), float(p0[r]), 1.0) for r in range(R)]
    sx = np.stack([gen_start_simplices(seed, r, n_starts, float(pb.pedigree[:, 3].max())) for r, pb in enumerate(probs)])
    if len(ctxs) > 1:
        res = alphabeta_batch_multi(ctxs, probs, sx, n_boot, seed, max_iters_fit=max_iters_fit, max_iters_boot=max_iters_boot)
    else:
        res = ctxs[0].alphabeta_batch(probs, sx, n_boot, seed, max_iters_fit=max_iters_fit, max_iters_boot=max_iters_boot)
    return {"theta": res["best"]["theta"].copy(), "status": res["status"], "analysis": res["analysis"],
            "D": np.stack([pb.pedigree[:, 3] for pb in probs]), "p0uu": p0,
            "truth": {"alpha": prm.alpha, "beta": prm.beta, "weight": prm.weight, "p0uu": prm.p0uu,
                      "missing_rate": prm.missing_rate, "seed": int(seed)}}
