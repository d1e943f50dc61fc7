"""ctypes wrapper of the CPU oracle of the ABneutral methylome simulation (oracle/abref_sim.c, linked with abref.c) and
a numpy restatement of the forest's pedigree rows.

TEST INFRASTRUCTURE ONLY — see oracle/abref.h.  The library is compiled on first use into a per-user temporary
directory (keyed by the sources' contents), so the tree itself is never written."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = [os.path.join(HERE, f) for f in ("abref.c", "abref_sim.c")]
_lib = None


def build() -> str:
    h = hashlib.sha256()
    for f in _SRC + [os.path.join(HERE, "abref.h")]:
        h.update(open(f, "rb").read())
    out_dir = os.path.join(tempfile.gettempdir(), f"abref_sim_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    lib = os.path.join(out_dir, f"libabref_sim_{h.hexdigest()[:16]}.so")
    if not os.path.exists(lib):
        tmp = f"{lib}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-std=c11", "-ffp-contract=off", "-fno-fast-math",
                               "-fPIC", "-pthread", "-shared", "-o", tmp] + _SRC + ["-lm"])
        os.replace(tmp, lib)
    return lib


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _forest_arrays(parent, generation, sampled):
    return (np.ascontiguousarray(parent, dtype=np.int32), np.ascontiguousarray(generation, dtype=np.int32),
            np.ascontiguousarray(sampled, dtype=np.uint8))


def sim_pairs(parent, generation, sampled):
    """pedigree rows (i, j, t0, t1, t2) of the sampled nodes of a forest, i < j in node order, pairs of different trees
    left out; t0 = generation of the most recent common ancestor (= the smallest generation on the path, since
    generations do not decrease from parent to child).  Rejects what is not a forest with non-decreasing generations."""
    parent, gen, sampled = _forest_arrays(parent, generation, sampled)
    n = len(parent)
    anc = []
    for v in range(n):
        chain, u = [v], int(parent[v])
        while u >= 0:
            if len(chain) > n:
                raise ValueError("cycle")
            if not (0 <= u < n) or gen[u] > gen[chain[-1]]:
                raise ValueError("parent out of range or generation decreases")
            chain.append(u)
            u = int(parent[u])
        anc.append(chain)
    if np.any(gen < 0) or np.any(gen > 127):
        raise ValueError("generation outside 0..127")
    meas = [v for v in range(n) if sampled[v]]
    out = []
    for a in range(len(meas)):
        sa = set(anc[meas[a]])
        for b in range(a + 1, len(meas)):
            lca = next((u for u in anc[meas[b]] if u in sa), None)
            if lca is not None:
                out.append((a, b, float(gen[lca]), float(gen[meas[a]]), float(gen[meas[b]])))
    return np.array(out, dtype=np.float64).reshape(-1, 5)


def sim_thresholds(parent, generation, alpha, beta, weight, p0uu):
    parent, gen, _ = _forest_arrays(parent, generation, np.zeros(len(parent)))
    out = np.empty((len(parent), 6))
    lib().abref_sim_thresholds(len(parent), _p(parent), _p(gen), C.c_double(alpha), C.c_double(beta), C.c_double(weight),
                               C.c_double(p0uu), _p(out))
    return out


def simulate(parent, generation, sampled, alpha, beta, weight, p0uu, L, seed, missing_rate=0.0, first_site=0):
    """-> (status u8, posterior_max, meth_lvl), each [n_sampled, L]"""
    parent, gen, sampled = _forest_arrays(parent, generation, sampled)
    S = int(sampled.astype(bool).sum())
    status, post, meth = np.empty((S, L), dtype=np.uint8), np.empty((S, L)), np.empty((S, L))
    lib().abref_simulate(len(parent), _p(parent), _p(gen), _p(sampled), C.c_double(alpha), C.c_double(beta),
                         C.c_double(weight), C.c_double(p0uu), C.c_double(missing_rate), C.c_uint64(seed),
                         C.c_int64(first_site), C.c_int64(L), _p(status), _p(post), _p(meth))
    return status, post, meth
