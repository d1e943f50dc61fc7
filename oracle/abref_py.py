"""ctypes wrapper of the CPU oracle (oracle/libabref.so) plus a Python restatement of the
reference's input side (nodelist / edgelist / methylome parsing and the pedigree graph).

TEST INFRASTRUCTURE ONLY — see oracle/abref.h.  Imported by tests/, by the smoke check in
__graft_entry__.py and by bench.py's cpu_baseline / --impl reference legs; never by the
product package.
"""
from __future__ import annotations

import ctypes as C
import heapq
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libabref.so")

SHRINK_ON_FAILED_CONTRACTION, EARLY_EXIT_ON_STALL, FAST_DIVERGENCE, LITERAL_SORT = 1, 2, 4, 8
TERM_SD, TERM_MAX_ITERS, TERM_STALLED, TERM_TARGET_COST, ERR_NAN, ERR_TIME = 1, 2, 3, 4, -1, -2
DBL_EPSILON = 2.220446049250313e-16


def build(force: bool = False) -> str:
    src = [os.path.join(HERE, f) for f in ("abref.c", "abref.h", "Makefile")]
    if force or not os.path.exists(LIB) or any(os.path.getmtime(s) > os.path.getmtime(LIB) for s in src):
        subprocess.check_call(["make", "-C", HERE, "-s", "-B", "libabref.so"])
    return LIB


class _Problem(C.Structure):
    _fields_ = [("ped", C.POINTER(C.c_double)), ("n", C.c_int32), ("p_mm", C.c_double), ("p_um", C.c_double),
                ("p_uu", C.c_double), ("eqp", C.c_double), ("eqp_weight", C.c_double)]


FIT_DTYPE = np.dtype([("theta", "<f8", (4,)), ("cost", "<f8"), ("lse", "<f8"), ("iters", "<i4"), ("evals", "<i4"),
                      ("status", "<i4"), ("start_id", "<i4")], align=True)

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        l = C.CDLL(LIB)
        l.abref_cost.restype = C.c_double
        l.abref_lse.restype = C.c_double
        for n in ("abref_p_uu_est", "abref_p_mm_est", "abref_p_um_est", "abref_steady_state"):
            getattr(l, n).restype = C.c_double
            getattr(l, n).argtypes = [C.c_double, C.c_double]
        l.abref_p0uu.restype = C.c_double
        _lib = l
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Problem:
    """src/structs.rs:12-19; p_mm = 1 - p_uu, p_um = 0 as in src/ab_neutral.rs:23-24 unless given."""

    def __init__(self, pedigree, p_uu, eqp, eqp_weight, p_mm=None, p_um=0.0):
        self.ped = np.ascontiguousarray(pedigree, dtype=np.float64)
        self.n = self.ped.shape[0]
        self.p_uu = float(p_uu)
        self.p_mm = float(1.0 - p_uu if p_mm is None else p_mm)
        self.p_um = float(p_um)
        self.eqp, self.eqp_weight = float(eqp), float(eqp_weight)
        self.c = _Problem(self.ped.ctypes.data_as(C.POINTER(C.c_double)), self.n, self.p_mm, self.p_um, self.p_uu,
                          self.eqp, self.eqp_weight)


def genmatrix(a, b):
    G = np.empty(9)
    lib().abref_genmatrix(C.c_double(a), C.c_double(b), _p(G))
    return G.reshape(3, 3)


def matrix_power(M, p):
    M = np.ascontiguousarray(M, dtype=np.float64)
    out = np.empty(9)
    lib().abref_matrix_power(_p(M), int(p), _p(out))
    return out.reshape(3, 3)


def divergence(pb: Problem, alpha, beta, weight, flags=0):
    dt = np.empty(pb.n)
    puu = C.c_double()
    rc = lib().abref_divergence(_p(pb.ped), pb.n, C.c_double(pb.p_mm), C.c_double(pb.p_um), C.c_double(pb.p_uu),
                                C.c_double(alpha), C.c_double(beta), C.c_double(weight), flags, _p(dt), C.byref(puu))
    if rc:
        raise ValueError(f"abref_divergence rc={rc}")
    return dt, puu.value


def cost(pb: Problem, theta, flags=0) -> float:
    th = np.ascontiguousarray(theta, dtype=np.float64)
    return lib().abref_cost(C.byref(pb.c), _p(th), flags)


def lse(pb: Problem, theta, flags=0) -> float:
    th = np.ascontiguousarray(theta, dtype=np.float64)
    return lib().abref_lse(C.byref(pb.c), _p(th), flags)


def nelder_mead(pb: Problem, simplex, max_iters=10000, sd_tol=DBL_EPSILON, flags=0):
    sx = np.ascontiguousarray(simplex, dtype=np.float64).reshape(20)
    out = np.zeros(1, dtype=FIT_DTYPE)
    lib().abref_nelder_mead(C.byref(pb.c), _p(sx), max_iters, C.c_double(sd_tol), flags, _p(out))
    return out[0]


def ab_neutral(pb: Problem, simplices, max_iters=10000, sd_tol=DBL_EPSILON, flags=0, n_threads=1):
    sx = np.ascontiguousarray(simplices, dtype=np.float64)
    n_starts = sx.size // 20
    best = np.zeros(1, dtype=FIT_DTYPE)
    allr = np.zeros(n_starts, dtype=FIT_DTYPE)
    pred, resid = np.empty(pb.n), np.empty(pb.n)
    rc = lib().abref_ab_neutral(C.byref(pb.c), n_starts, _p(sx), max_iters, C.c_double(sd_tol), flags, n_threads,
                                _p(best), _p(allr), _p(pred), _p(resid))
    return rc, best[0], allr, pred, resid


def boot_model(pb: Problem, best_theta, pred, resid, resample_idx, vary, max_iters=1000, sd_tol=DBL_EPSILON, flags=0,
               n_threads=1):
    th = np.ascontiguousarray(best_theta, dtype=np.float64)
    pred = np.ascontiguousarray(pred, dtype=np.float64)
    resid = np.ascontiguousarray(resid, dtype=np.float64)
    idx = np.ascontiguousarray(resample_idx, dtype=np.int32)
    vary = np.ascontiguousarray(vary, dtype=np.float64)
    n_boot = vary.size // 16
    rows = np.empty((n_boot, 7))
    fits = np.zeros(n_boot, dtype=FIT_DTYPE)
    rc = lib().abref_boot_model(C.byref(pb.c), _p(th), _p(pred), _p(resid), n_boot, _p(idx), _p(vary), max_iters,
                                C.c_double(sd_tol), flags, n_threads, _p(rows), _p(fits))
    return rc, rows, fits


def dmatrix(status, post, thr):
    status = np.ascontiguousarray(status, dtype=np.uint8)
    post = np.ascontiguousarray(post, dtype=np.float64)
    S, L = status.shape
    P = S * (S - 1) // 2
    D = np.empty(P)
    diff = np.empty(P, dtype=np.uint64)
    cnt = np.empty(P, dtype=np.uint64)
    lib().abref_dmatrix(_p(status), _p(post), S, C.c_int64(L), C.c_double(thr), _p(D), _p(diff), _p(cnt))
    return D, diff, cnt


def p0uu(post, meth, thr):
    post = np.ascontiguousarray(post, dtype=np.float64)
    meth = np.ascontiguousarray(meth, dtype=np.float64)
    S, L = post.shape
    rc = np.empty(S)
    nv = np.empty(S, dtype=np.int64)
    v = lib().abref_p0uu(_p(post), _p(meth), S, C.c_int64(L), C.c_double(thr), _p(rc), _p(nv))
    return v, rc, nv


def analyze(rows):
    rows = np.ascontiguousarray(rows, dtype=np.float64).reshape(-1, 7)
    out = np.empty(32)
    lib().abref_analyze(_p(rows), rows.shape[0], _p(out))
    return out


def hw_threads() -> int:
    return lib().abref_hw_threads()


# ---------------------------------------------------------------------------------------------
# input side, restated in Python (small inputs only)
# ---------------------------------------------------------------------------------------------
def _parse_chromosome(s: str):
    """src/methylation_site.rs:55-68"""
    while s.startswith("chr"):
        s = s[3:]
    if s == "M":
        return "M"
    if s == "C":
        return "C"
    if s.isascii() and s.isdigit() or (s.startswith("+") and s[1:].isdigit()):
        v = int(s)
        if 0 <= v <= 255:
            return v
    raise ValueError("chromosome")


def _u32(s: str) -> int:
    if not (s.isascii() and (s.isdigit() or (s.startswith("+") and s[1:].isdigit()))):
        raise ValueError("u32")
    v = int(s)
    if v > 0xFFFFFFFF:
        raise ValueError("u32")
    return v


_F64_RE = None


def _f64_rust(s: str) -> float:
    """<f64 as FromStr>::from_str: no surrounding whitespace, no underscores, no hex; inf / infinity / nan in any case"""
    global _F64_RE
    import re

    if _F64_RE is None:
        _F64_RE = re.compile(r"^[+-]?((\d+\.?\d*|\.\d+)([eE][+-]?\d+)?|(?i:inf|infinity|nan))$")
    if not (s.isascii() and _F64_RE.match(s)):
        raise ValueError("f64")
    return float(s)


def _status(s: str) -> int:
    """src/methylation_site.rs:101-115,130-136: U=0, I=1, M=2; anything else parses as U"""
    if not s:
        raise ValueError("status")
    return {"M": 2, "I": 1, "U": 0}.get(s[0], 0)


def parse_methylome_line(line: str, invert_strand: bool = False):
    """MethylationSite::from_methylome_file_line (src/methylation_site.rs:146-362), CG formats.
    Returns dict(chromosome,start,end,strand,posteriormax,status,meth_lvl) or None."""
    f = line.split("\t")

    def mk(chrom, start, end, strand, post, status, lvl, cm, ct):
        return {
            "chromosome": _parse_chromosome(chrom), "start": start, "end": end,
            "strand": ("+" if ((strand == "+") ^ invert_strand) else "-"),
            "count_methylated": _u32(cm), "count_total": _u32(ct),
            "posteriormax": _f64_rust(post), "status": _status(status), "meth_lvl": _f64_rust(lvl), "original": line,
        }

    # `location.parse::<u32>()? + 1` (src/methylation_site.rs:166,210): a release build wraps at u32::MAX
    try:
        if len(f) == 9 and f[3] == "CG":
            return mk(f[0], _u32(f[1]), (_u32(f[1]) + 1) & 0xFFFFFFFF, f[2], f[6], f[7], f[8], f[4], f[5])
    except ValueError:
        pass
    try:
        if len(f) == 10 and f[3] == "CG":
            return mk(f[0], _u32(f[1]), (_u32(f[1]) + 1) & 0xFFFFFFFF, f[2], f[6], f[7], f[8], f[4], f[5])
    except ValueError:
        pass
    try:
        if len(f) == 11 and f[3] == "CG":
            return mk(f[0], _u32(f[1]), _u32(f[2]), f[5], f[8], f[9], f[10], f[6], f[7])
    except ValueError:
        pass
    g = line.replace("\t", " ").split(" ")
    try:
        if len(g) == 4:  # chromatin-state / bedGraph / heterogeneity formats: strand unknown, posteriormax 0
            return {"chromosome": _parse_chromosome(g[0]), "start": _u32(g[1]), "end": _u32(g[2]), "strand": "*",
                    "count_methylated": 0, "count_total": 0, "posteriormax": 0.0, "status": 0, "meth_lvl": 0.0,
                    "original": line}
    except ValueError:
        pass
    return None


def read_methylome(path: str):
    """sites of one sample as arrays (status u8, posteriormax f64, meth_lvl f64), file order
    (src/pedigree.rs:141-157)."""
    st, po, me = [], [], []
    with open(path) as fh:
        for line in fh.read().split("\n"):
            if line.endswith("\r"):
                line = line[:-1]
            s = parse_methylome_line(line)
            if s is None:
                continue
            st.append(s["status"])
            po.append(s["posteriormax"])
            me.append(s["meth_lvl"])
    return np.array(st, dtype=np.uint8), np.array(po), np.array(me)


def parse_nodelist(text: str):
    """src/pedigree.rs:99-116: id = line index after the header (blank lines count)."""
    nodes = []
    lines = text.replace("\r", "\n").split("\n")[1:]
    for i, line in enumerate(lines):
        e = line.replace(",", "\t").replace(" ", "\t").split("\t")
        if len(e) < 4:
            continue
        try:
            gen = _u32(e[2])
        except ValueError:
            continue
        nodes.append({"id": i, "file": e[0], "name": e[1], "generation": gen, "meth": e[3] == "Y"})
    return nodes


def parse_edgelist(text: str, nodes):
    """src/pedigree.rs:123-135"""
    byname = {}
    for n in nodes:
        byname.setdefault(n["name"], n)
    edges = []
    for line in text.replace("\r", "\n").split("\n")[1:]:
        e = line.replace(",", "\t").replace(" ", "\t").split("\t")
        if len(e) < 2 or e[0] not in byname or e[1] not in byname:
            continue
        edges.append((byname[e[0]], byname[e[1]]))
    return edges


def pedigree_pairs(meas, edges):
    """DMatrix::convert (src/pedigree.rs:264-337) without the divergences: for every pair i < j of measured nodes that
    the edge graph connects, (i, j, t0, t1, t2) with t0 = the smallest generation on the shortest path (edge weight =
    |generation difference|), in pair order."""
    # graph: undirected, weight = |generation difference| (src/pedigree.rs:265-277)
    adj = {}
    gen_of = {}
    for a, b in edges:
        w = abs(a["generation"] - b["generation"])
        adj.setdefault(a["id"], []).append((b["id"], w))
        adj.setdefault(b["id"], []).append((a["id"], w))
        gen_of.setdefault(a["id"], a["generation"])
        gen_of.setdefault(b["id"], b["generation"])

    def shortest(src, dst):
        dist = {src: 0}
        prev = {}
        pq = [(0, src)]
        while pq:
            d, u = heapq.heappop(pq)
            if u == dst:
                path = [u]
                while u in prev:
                    u = prev[u]
                    path.append(u)
                return d, path
            if d > dist.get(u, 1 << 60):
                continue
            for v, w in adj.get(u, []):
                nd = d + w
                if nd < dist.get(v, 1 << 60):
                    dist[v] = nd
                    prev[v] = u
                    heapq.heappush(pq, (nd, v))
        return None

    out = []
    S = len(meas)
    for i in range(S):
        for j in range(i + 1, S):
            r = shortest(meas[i]["id"], meas[j]["id"]) if meas[i]["id"] in adj or meas[i]["id"] == meas[j]["id"] else None
            if r is not None:
                dist, path = r
                t0 = float(min(gen_of[n] for n in path))
                t1, t2 = float(meas[i]["generation"]), float(meas[j]["generation"])
                assert float(dist) == t1 - t0 + t2 - t0
                out.append((i, j, t0, t1, t2))
    return out


def build_pedigree(nodelist_path: str, edgelist_path: str, thr: float, resolve=lambda p: p):
    """Pedigree::build (src/pedigree.rs:92-193) + DMatrix::convert (:264-337).
    Returns (pedigree [n,4], p0uu, dict with the per-sample arrays)."""
    nodes = parse_nodelist(open(nodelist_path).read())
    if not nodes:
        raise ValueError("No nodes could be parsed from the nodelist")
    edges = parse_edgelist(open(edgelist_path).read(), nodes)
    meas = [n for n in nodes if n["meth"]]
    data = [read_methylome(resolve(n["file"])) for n in meas]
    lens = {len(d[0]) for d in data}
    S = len(meas)
    if len(lens) == 1:
        status = np.stack([d[0] for d in data])
        post = np.stack([d[1] for d in data])
        meth = np.stack([d[2] for d in data])
        D, diff, cnt = dmatrix(status, post, thr)
        p0, rc, nv = p0uu(post, meth, thr)
    else:
        raise NotImplementedError("ragged site lists: the reference sets D = 0 for such pairs")
    rows = [[t0, t1, t2, D[i * S - i * (i + 1) // 2 + (j - i - 1)]] for i, j, t0, t1, t2 in pedigree_pairs(meas, edges)]
    ped = np.array(rows, dtype=np.float64).reshape(-1, 4)
    return ped, p0, {"status": status, "post": post, "meth": meth, "D": D, "diff": diff, "cnt": cnt, "rc": rc,
                     "nvalid": nv, "nodes": meas}


def load_pedigree_file(path: str) -> np.ndarray:
    """Pedigree::from_file (src/pedigree.rs:62-79): header skipped, space separated."""
    rows = []
    for line in open(path).read().split("\n")[1:]:
        if not line:
            continue
        rows.append([float(x) for x in line.split(" ")[:4]])
    return np.array(rows, dtype=np.float64)


# ---------------------------------------------------------------------------------------------
# site -> window assignment: literal Python restatement (small cases only; pure-Python loops)
#   Gene::from_annotation_file_line   src/genes.rs:166-216
#   Genome / GenesByStrand            src/genes.rs:24-57,127-163
#   is_in_gene / find_gene / place_in_windows   src/methylation_site.rs:368-490
#   Windows::new / extract loop / distribution  src/windows.rs:28-44,331-337,158-165
# genes / sites are tuples (chromosome, start, end, strand) with strand +1 / -1 / 0 ('*').
# ---------------------------------------------------------------------------------------------
U32 = 0xFFFFFFFF


def _strand_of(s: str):
    return {"+": 1, "-": -1, "*": 0}.get(s)


def _strand_eq(a: int, b: int) -> bool:  # src/genes.rs:88-96: Unknown equals anything
    return not ((a > 0 and b < 0) or (a < 0 and b > 0))


def chromosome_id(s: str):
    """Chromosome::try_from (src/methylation_site.rs:57-68) -> Numbered(n) = n, M = 256, C = 257, else None"""
    try:
        c = _parse_chromosome(s)
    except ValueError:
        return None
    return {"M": 256, "C": 257}.get(c, c)


def parse_annotation_line(line: str, invert: bool = False):
    """src/genes.rs:166-216: `chr start end name annotation strand` or `chr start end width strand name`"""
    parts = line.replace("\t", " ").split(" ")
    if len(parts) != 6:
        return None
    if _strand_of(parts[5]) is not None:
        c, st, en, strand = parts[0], parts[1], parts[2], parts[5]
    elif _strand_of(parts[4]) is not None:
        c, st, en, strand = parts[0], parts[1], parts[2], parts[4]
    else:
        return None
    cid = chromosome_id(c)
    try:
        a, b = _u32(st), _u32(en)
    except ValueError:
        return None
    if cid is None:
        return None
    sd = _strand_of(strand)
    return (cid, a, b, -sd if invert else sd)


def window_counts(window_size, window_step, cutoff, max_gene_length, absolute):
    step = window_step or window_size  # src/extract.rs:26-28
    gene = (max_gene_length // step) if absolute else (100 // step)
    updown = (cutoff // step) if absolute else (100 // step)
    return updown, gene, updown


def _gene_cutoff(g, cutoff, cutoff_gene_length):
    return ((g[2] - g[1]) & U32) if cutoff_gene_length else cutoff


def is_in_gene(site, g, cutoff, cutoff_gene_length=False):
    c = _gene_cutoff(g, cutoff, cutoff_gene_length)
    return (site[0] == g[0] and g[1] <= ((site[1] + c) & U32) and site[2] <= ((g[2] + c) & U32)
            and _strand_eq(site[3], g[3]))


def build_genome(genes):
    genome = {}
    for g in genes:
        l = genome.setdefault(g[0], {"sense": [], "antisense": [], "combined": []})
        l["combined"].append(g)
        if g[3] > 0:
            l["sense"].append(g)
        if g[3] < 0:
            l["antisense"].append(g)
    for l in genome.values():
        for k in l:
            l[k].sort(key=lambda g: g[1])  # list.sort is stable, like Vec::sort_by
    return genome


def find_gene(site, genome, cutoff, cutoff_gene_length=False):
    chrom = genome.get(site[0])
    if chrom is None:
        return None
    strand = chrom["sense"] if site[3] > 0 else chrom["antisense"] if site[3] < 0 else chrom["combined"]
    # slice::binary_search_by_key, Rust 1.52..1.81
    size = len(strand)
    left, right = 0, size
    idx = None
    while left < right:
        mid = left + size // 2
        key = (strand[mid][2] + _gene_cutoff(strand[mid], cutoff, cutoff_gene_length)) & U32
        if key < site[1]:
            left = mid + 1
        elif key > site[1]:
            right = mid
        else:
            idx = mid
            break
        size = right - left
    if idx is None:
        idx = left
    if len(strand) < idx + 1:
        return None
    g = strand[idx]
    return g if is_in_gene(site, g, cutoff, cutoff_gene_length) else None


def place_in_windows(site, g, counts, window_size, window_step, cutoff, absolute):
    """returns [(region, window index)] with region 0/1/2 = upstream/gene/downstream"""
    E = 0.1
    step = float(window_step or window_size)
    size = float(window_size)
    location, start, end = float(site[1]), float(g[1]), float(g[2])
    cut = float(cutoff)
    length = end - start
    antisense = site[3] < 0  # Unknown is treated as Sense (:439-443)
    offset = (end - location) if antisense else (location - start)
    region = 0 if offset < 0.0 else 2 if offset > length else 1
    if not antisense:
        position = (location - start + cut, location - start, location - end)[region]
    else:
        position = (end - location + cut, end - location, start - location)[region]
    if not absolute:
        try:
            position = position / length if region == 1 else position / cut
        except ZeroDivisionError:
            position = float("nan") if position == 0 else float("inf") * (1 if position > 0 else -1)
        position *= 100.0
    hits = []
    for i in range(counts[region]):
        lower = i * step - E
        upper = lower + size + E
        if position >= lower and position <= upper:
            hits.append((region, i))
    return hits


def extract_windows(genes, sites, window_size=5, window_step=0, cutoff=2048, max_gene_length=100, absolute=False,
                    cutoff_gene_length=False):
    """Windows::extract placement loop -> (distribution list, [(site index, flat window index)])"""
    counts = window_counts(window_size, window_step, cutoff, max_gene_length, absolute)
    base = (0, counts[0], counts[0] + counts[1])
    dist = [0] * sum(counts)
    assign = []
    genome = build_genome(genes)
    last = None
    for si, s in enumerate(sites):
        if last is None or not is_in_gene(s, last, cutoff, cutoff_gene_length):
            last = find_gene(s, genome, cutoff, cutoff_gene_length)
        if last is None:
            continue
        for region, i in place_in_windows(s, last, counts, window_size, window_step, cutoff, absolute):
            dist[base[region] + i] += 1
            assign.append((si, base[region] + i))
    return dist, assign


# ---------------------------------------------------------------------------------------------
# result files: literal restatement of the reference's writers
# ---------------------------------------------------------------------------------------------
def rust_f64(v: float) -> str:
    """`format!("{}", v)` for an f64: shortest round-trip digits (Python's repr has the same digits), positional"""
    import math
    from decimal import Decimal

    if math.isnan(v):
        return "NaN"
    if math.isinf(v):
        return "-inf" if v < 0 else "inf"
    s = format(Decimal(repr(float(v))), "f")
    if "." in s:
        s = s.rstrip("0").rstrip(".")
    if s in ("-", ""):
        s += "0"
    if v == 0 and math.copysign(1.0, v) < 0 and not s.startswith("-"):
        s = "-" + s
    return s


def pedigree_file_text(ped) -> str:
    """Pedigree::to_file (src/pedigree.rs:81-90)"""
    out = "time0\ttime1\ttime2\tD.value\n"
    for r in np.asarray(ped, dtype=np.float64).reshape(-1, 4):
        out += "\t".join(rust_f64(x) for x in r) + "\n"
    return out


def analysis_file_text(a) -> str:
    """Analysis::to_file (src/analysis.rs:102-144); a = analyze() output (8 means, 8 sds, 8 CI pairs)"""
    names = ["Alpha", "Beta", "AlphaBeta", "Weight", "Intercept", "PrMM", "PrUM", "PrUU"]
    out = "".join(f"{n}\t{rust_f64(a[i])}\n" for i, n in enumerate(names))
    out += "".join(f"SD{n}\t{rust_f64(a[8 + i])}\n" for i, n in enumerate(names))
    out += "".join(f"CI{n}\t{rust_f64(a[16 + 2 * i])}-{rust_f64(a[17 + 2 * i])}\n" for i, n in enumerate(names))
    return out


def steady_state(alpha, beta) -> float:
    return float(lib().abref_steady_state(C.c_double(alpha), C.c_double(beta)))


def metaprofile_results_text(run_name, cg_count, region, best_theta, analysis, obs) -> str:
    """src/cli/metaprofile.rs:74-99"""
    out = ("run;window;cg_count;region;alpha;beta;1/2*(alpha+beta);pred_steady_state;obs_steady_state;sd_alpha;sd_beta;"
           "ci_alpha_0.025;ci_alpha_0.975;ci_beta_0.025;ci_beta_0.975\n")
    reg = ["upstream", "gene", "downstream"]
    for i in range(len(cg_count)):
        a, b = float(best_theta[i][0]), float(best_theta[i][1])
        an = analysis[i]
        vals = [a, b, 0.5 * (a + b), steady_state(a, b), obs[i], an[8], an[9], an[16], an[17], an[18], an[19]]
        out += f"{run_name};{i};{int(cg_count[i])};{reg[region[i]]};" + ";".join(rust_f64(float(x)) for x in vals) + "\n"
    return out
