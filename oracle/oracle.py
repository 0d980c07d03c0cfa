"""oracle/oracle.py — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Python face of the CPU oracle for KOMB's hot path.  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module; nothing under komb_b200/ does.

Parity status: PINNED (see the header of komb_oracle.c and
tests/test_oracle.py): checked against fixtures produced by the reference
itself (oracle/_ref/komb2_ref, reference sources compiled unmodified against
oracle/igraph_shim) and against networkx / scipy.

Contents
  * ctypes bindings to libkomb_oracle.so (C restatement, komb_oracle.c)
  * tokenise_sam(): pure-Python restatement of the reference SAM tokeniser
    (src/graph.cpp:197-239) including the -t dependent line drop (quirk Q1)
  * canonical readers for the three komb2 output files (quirks Q4, Q7, Q9)
  * run_komb2(): run a komb2 binary (the reference build or the new drop-in)
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_LIB_PATH = _HERE / "libkomb_oracle.so"
REF_KOMB2 = _HERE / "_ref" / "komb2_ref"
REF_COREA = _HERE / "_ref" / "corea_ref"
REF_DENSEST = _HERE / "_ref" / "densest_ref"

KEY_REF32 = 0
KEY_EXACT64 = 1

_lib = None


def build() -> None:
    """Compile the C restatement (and, when /root/reference exists, the
    reference itself into oracle/_ref/)."""
    subprocess.run(["make", "-C", str(_HERE), "all"], check=True, capture_output=True)
    if Path("/root/reference/src/graph.cpp").exists():
        subprocess.run(["make", "-C", str(_HERE), "ref"], check=True, capture_output=True)


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists() or _LIB_PATH.stat().st_mtime < (_HERE / "komb_oracle.c").stat().st_mtime:
            build()
        L = ctypes.CDLL(str(_LIB_PATH))
        u32p = ctypes.POINTER(ctypes.c_uint32)
        u64p = ctypes.POINTER(ctypes.c_uint64)
        i32p = ctypes.POINTER(ctypes.c_int32)
        f64p = ctypes.POINTER(ctypes.c_double)
        L.ko_build_edges.argtypes = [u32p, u32p, ctypes.c_uint64, ctypes.POINTER(u64p), u64p, u64p, u64p]
        L.ko_build_edges.restype = ctypes.c_int
        L.ko_simplify.argtypes = [u32p, u32p, ctypes.c_uint64, ctypes.POINTER(u64p), u64p]
        L.ko_simplify.restype = ctypes.c_int
        L.ko_coreness.argtypes = [ctypes.c_uint32, u64p, ctypes.c_uint64, i32p, i32p]
        L.ko_coreness.restype = ctypes.c_int
        L.ko_corea.argtypes = [ctypes.c_uint32, i32p, i32p, ctypes.c_int, f64p]
        L.ko_corea.restype = ctypes.c_int
        L.ko_corea_ranks.argtypes = [ctypes.c_uint32, i32p, i32p, ctypes.c_int, f64p, f64p]
        L.ko_corea_ranks.restype = ctypes.c_int
        L.ko_free.argtypes = [ctypes.c_void_p]
        L.ko_free.restype = None
        _lib = L
    return _lib


def _p(a: np.ndarray, ct):
    return a.ctypes.data_as(ctypes.POINTER(ct))


def _take_u64(ptr, count: int) -> np.ndarray:
    if count == 0 or not ptr:
        if ptr:
            lib().ko_free(ctypes.cast(ptr, ctypes.c_void_p))
        return np.zeros(0, dtype=np.uint64)
    arr = np.ctypeslib.as_array(ptr, shape=(count,)).copy()
    lib().ko_free(ctypes.cast(ptr, ctypes.c_void_p))
    return arr


# ---------------------------------------------------------------------------
# stage restatements (C)
# ---------------------------------------------------------------------------

def build_edges(read_key: np.ndarray, unitig: np.ndarray):
    """Hits of both mate files (concatenated) -> (packed sorted simple edges
    u<<32|v with u<v, P pairs emitted before dedup, S distinct (read,unitig))."""
    rk = np.ascontiguousarray(read_key, dtype=np.uint32)
    ut = np.ascontiguousarray(unitig, dtype=np.uint32)
    assert rk.shape == ut.shape
    out = ctypes.POINTER(ctypes.c_uint64)()
    E = ctypes.c_uint64(); P = ctypes.c_uint64(); S = ctypes.c_uint64()
    rc = lib().ko_build_edges(_p(rk, ctypes.c_uint32), _p(ut, ctypes.c_uint32), rk.shape[0],
                              ctypes.byref(out), ctypes.byref(E), ctypes.byref(P), ctypes.byref(S))
    if rc != 0:
        raise RuntimeError(f"ko_build_edges rc={rc}")
    return _take_u64(out, E.value), P.value, S.value


def simplify(u: np.ndarray, v: np.ndarray) -> np.ndarray:
    uu = np.ascontiguousarray(u, dtype=np.uint32)
    vv = np.ascontiguousarray(v, dtype=np.uint32)
    out = ctypes.POINTER(ctypes.c_uint64)()
    E = ctypes.c_uint64()
    rc = lib().ko_simplify(_p(uu, ctypes.c_uint32), _p(vv, ctypes.c_uint32), uu.shape[0],
                           ctypes.byref(out), ctypes.byref(E))
    if rc != 0:
        raise RuntimeError(f"ko_simplify rc={rc}")
    return _take_u64(out, E.value)


def coreness(n: int, edges: np.ndarray):
    """BZ coreness + degree of the simple graph given as packed edges."""
    e = np.ascontiguousarray(edges, dtype=np.uint64)
    deg = np.zeros(n, dtype=np.int32)
    core = np.zeros(n, dtype=np.int32)
    rc = lib().ko_coreness(n, _p(e, ctypes.c_uint64), e.shape[0], _p(deg, ctypes.c_int32), _p(core, ctypes.c_int32))
    if rc != 0:
        raise RuntimeError(f"ko_coreness rc={rc}")
    return deg, core


def corea(core: np.ndarray, deg: np.ndarray, key_mode: int = KEY_REF32) -> np.ndarray:
    c = np.ascontiguousarray(core, dtype=np.int32)
    d = np.ascontiguousarray(deg, dtype=np.int32)
    n = c.shape[0]
    score = np.zeros(n, dtype=np.float64)
    rc = lib().ko_corea(n, _p(c, ctypes.c_int32), _p(d, ctypes.c_int32), key_mode, _p(score, ctypes.c_double))
    if rc != 0:
        raise RuntimeError(f"ko_corea rc={rc}")
    return score


def corea_ranks(core: np.ndarray, deg: np.ndarray, key_mode: int = KEY_REF32):
    c = np.ascontiguousarray(core, dtype=np.int32)
    d = np.ascontiguousarray(deg, dtype=np.int32)
    n = c.shape[0]
    rd = np.zeros(n, dtype=np.float64)
    rk = np.zeros(n, dtype=np.float64)
    rc = lib().ko_corea_ranks(n, _p(c, ctypes.c_int32), _p(d, ctypes.c_int32), key_mode,
                              _p(rd, ctypes.c_double), _p(rk, ctypes.c_double))
    if rc != 0:
        raise RuntimeError(f"ko_corea_ranks rc={rc}")
    return rd, rk


# Every ranking path builds its ranks as exact half-integers in FP64, so a score can differ from |ln rd - ln rk| of the
# exact ranks only by the rounding of two log() calls and one subtraction: a few ulp of ln(2^32) < 23, about 1e-14.
# A key rank off by one half at rank r moves a score by about 0.5 / r, which is 2.3e-10 even at r = 2^31.
COREA_ATOL = 6e-14


def check_corea_ranks(got: np.ndarray, rd: np.ndarray, rk: np.ndarray, atol: float = COREA_ATOL) -> None:
    """Assert that the scores `got` are |ln rd - ln rk| of the exact descending average ranks (degree ranks rd, key
    ranks rk) within `atol` absolute, and that vertices with the same rank pair have bit-identical scores."""
    got = np.asarray(got)
    assert got.dtype == np.float64 and got.shape == rd.shape == rk.shape, (got.dtype, got.shape, rd.shape, rk.shape)
    exp = np.abs(np.log(rd) - np.log(rk))
    err = np.abs(got - exp)
    bad = np.flatnonzero(~(err <= atol))          # NaN fails too
    if bad.size:
        i = int(bad[np.argmax(np.nan_to_num(err[bad], nan=np.inf))])
        raise AssertionError(f"{bad.size} CORE-A scores off by more than {atol:g}; worst at vertex {i}: got {got[i]!r}, "
                             f"expected {exp[i]!r} (degree rank {rd[i]}, key rank {rk[i]})")
    if got.size > 1:
        o = np.lexsort((rk, rd))
        same = (rd[o[1:]] == rd[o[:-1]]) & (rk[o[1:]] == rk[o[:-1]])
        bits = got.view(np.uint64)[o]
        split = np.flatnonzero(same & (bits[1:] != bits[:-1]))
        if split.size:
            a, b = int(o[split[0]]), int(o[split[0] + 1])
            raise AssertionError(f"vertices {a} and {b} share the rank pair ({rd[a]}, {rk[a]}) but score {got[a]!r} "
                                 f"and {got[b]!r}")


def check_corea(got: np.ndarray, core: np.ndarray, deg: np.ndarray, key_mode: int, ranking: bool = True) -> None:
    """The exact CORE-A check: `got` against the oracle's exact ranks (check_corea_ranks) and, with `ranking`, the
    anomaly ranking (descending score, ties by vertex id) identical to the oracle's.  Leave `ranking` off for
    random (coreness, degree) arrays: their many near-tied scores of different rank pairs order by the last bit of
    log()."""
    rd, rk = corea_ranks(core, deg, key_mode)
    check_corea_ranks(got, rd, rk)
    if ranking:
        exp = corea(core, deg, key_mode)
        assert np.array_equal(np.argsort(-got, kind="stable"), np.argsort(-exp, kind="stable")), "anomaly ranking differs"


def densest_core(core: np.ndarray, edges: np.ndarray) -> dict:
    """Checker for kombgpu_graph_densest_core: the k-core maximising edges / vertices (equal density: the larger
    block; k = smallest coreness inside the block).
    Restates the density bookkeeping of CombineCoreA::runMerge (src/CombineCoreA.h:112-145: suspiciousSum /
    numOfNodesBelong with suspiciousness == nullptr) over the nested k-cores instead of single-node removals."""
    n = int(core.shape[0])
    if n == 0 or edges.shape[0] == 0:
        return {"k": 0, "n_vertices": n, "n_edges": int(edges.shape[0]), "density": (edges.shape[0] / n) if n else 0.0}
    u, v = unpack_edges(edges)
    kmax = int(core.max())
    hv = np.bincount(core, minlength=kmax + 1).astype(np.int64)
    he = np.bincount(np.minimum(core[u], core[v]), minlength=kmax + 1).astype(np.int64)
    vk = np.cumsum(hv[::-1])[::-1]
    ek = np.cumsum(he[::-1])[::-1]
    best = None
    for k in range(kmax, -1, -1):
        if vk[k] == 0:
            continue
        d = float(ek[k]) / float(vk[k])
        if best is None or d > best["density"] or (d == best["density"] and int(vk[k]) > best["n_vertices"]):
            best = {"k": k, "n_vertices": int(vk[k]), "n_edges": int(ek[k]), "density": d}
    return best


def densest_block_bulk(n: int, edges: np.ndarray, weight=None, eps: float = 0.5) -> dict:
    """Checker for kombgpu_graph_densest_block: the greedy densest-block peel of CombineCoreA::runMerge
    (src/CombineCoreA.h:45-219) in bulk form.  f(S) = sum of weights + edges inside S, density = f(S) / |S|
    (suspiciousSum / numOfNodesBelong, :133: both halved, a unitig's row and column copy always carry the same
    priority on a symmetric adjacency); a pass removes every survivor with weight + degree inside S <= 2 (1 + eps)
    density(S); the densest S seen wins (strict >, like :134)."""
    u, v = unpack_edges(edges)
    u, v = u.astype(np.int64), v.astype(np.int64)
    w = np.zeros(n, np.float64) if weight is None else np.asarray(weight, np.float64)
    alive = np.ones(n, bool)
    deg = np.bincount(np.concatenate([u, v]), minlength=n).astype(np.int64) if n else np.zeros(0, np.int64)
    W, E, N = float(w.sum()), int(edges.shape[0]), n
    best = {"n_vertices": n, "n_edges": E, "weight_sum": W, "density": (W + E) / n if n else 0.0, "passes": 0, "member": alive.copy()}
    t = 0
    e_alive = np.ones(edges.shape[0], bool)
    while N > 0:
        rho = (W + float(E)) / float(N)
        if t == 0 or rho > best["density"]:
            best = {"n_vertices": N, "n_edges": E, "weight_sum": W, "density": rho, "member": alive.copy()}
        thr = 2.0 * (1.0 + eps) * rho
        take = alive & (w + deg.astype(np.float64) <= thr)
        assert take.any()
        alive &= ~take
        gone = e_alive & (take[u] | take[v])
        # survivors lose a neighbour for every edge towards a removed unitig
        np.subtract.at(deg, u[gone & ~take[u]], 1)
        np.subtract.at(deg, v[gone & ~take[v]], 1)
        e_alive &= ~gone
        N -= int(take.sum())
        E -= int(gone.sum())
        W -= float(w[take].sum())
        if W < 0.0 or N == 0:
            W = 0.0
        t += 1
    best["passes"] = t
    return best


def densest_block_greedy(n: int, edges: np.ndarray, weight, workdir) -> dict:
    """The reference's serial greedy (CombineCoreA::runMerge, src/CombineCoreA.h:45-219) over the reference's own
    HashIndexedMinHeap: oracle/_ref/densest_ref.  Density is in the reference's units, (2 sum w + 2 E(S)) / (rows +
    columns left)."""
    workdir = Path(workdir)
    u, v = unpack_edges(edges)
    with open(workdir / "densest_in.bin", "wb") as f:
        f.write(np.array([n, 0 if weight is None else 1], dtype=np.int32).tobytes())
        f.write(np.array([edges.shape[0]], dtype=np.int64).tobytes())
        if weight is not None:
            f.write(np.ascontiguousarray(weight, dtype=np.float64).tobytes())
        f.write(u.astype(np.int32).tobytes())
        f.write(v.astype(np.int32).tobytes())
    subprocess.run([str(REF_DENSEST), str(workdir / "densest_in.bin"), str(workdir / "densest_out.bin")], check=True)
    raw = (workdir / "densest_out.bin").read_bytes()
    density = float(np.frombuffer(raw[:8], np.float64)[0])
    nr, nc = (int(x) for x in np.frombuffer(raw[8:16], np.int32))
    ids = np.frombuffer(raw[16:], np.int32)
    return {"density": density, "rows": np.sort(ids[:nr]), "cols": np.sort(ids[nr:nr + nc])}


def densest_block_serial(n: int, edges: np.ndarray, weight=None) -> dict:
    """The serial greedy peel of CombineCoreA::runMerge (src/CombineCoreA.h:56-186) restated over a binary heap, with
    `removed` cleared (the reference reads it uninitialised, :105-109) and ties between equal priorities broken by the
    smaller id (the reference's HashIndexedMinHeap has its own tie order).  A row and a column copy of every unitig,
    priority weight + degree; the copy of least priority goes (the row on a strict <), its neighbours' other copies
    lose one; the densest remainder seen wins (strict >, :134).  Density is in the reference's units,
    (2 sum w + 2 E(S)) / (rows + columns left)."""
    import heapq
    u, v = unpack_edges(edges)
    u, v = u.astype(np.int64), v.astype(np.int64)
    w = np.zeros(n, np.float64) if weight is None else np.asarray(weight, np.float64)
    adj = [[] for _ in range(n)]
    for a, b in zip(u.tolist(), v.tolist()):
        adj[a].append(b)
        adj[b].append(a)
    prio = [[float(w[i]) + len(adj[i]) for i in range(n)] for _ in range(2)]      # [0]: rows, [1]: columns
    heaps = [[(p, i) for i, p in enumerate(prio[0])], [(p, i) for i, p in enumerate(prio[1])]]
    for h in heaps:
        heapq.heapify(h)
    removed = [bytearray(n), bytearray(n)]
    suspicious = 2.0 * float(w.sum()) + 2.0 * float(u.shape[0])

    def peek(mode):
        h = heaps[mode]
        while h and (removed[mode][h[0][1]] or h[0][0] != prio[mode][h[0][1]]):
            heapq.heappop(h)                            # stale entry: removed, or its priority was refreshed since
        return h[0] if h else None

    order, modes = [0] * (2 * n), [0] * (2 * n)
    best, best_left, left = 0.0, 0, 2 * n
    while left >= 1:
        r, c = peek(0), peek(1)
        mode = 0 if r is not None and (c is None or r[0] < c[0]) else 1
        p, node = heapq.heappop(heaps[mode])
        suspicious -= p
        left -= 1
        order[left], modes[left] = node, mode
        if left >= 1 and suspicious / left > best:
            best, best_left = suspicious / left, left
        removed[mode][node] = 1
        other = 1 - mode
        for dst in adj[node]:
            if not removed[other][dst]:
                prio[other][dst] -= 1.0
                heapq.heappush(heaps[other], (prio[other][dst], dst))
    rows = [order[i] for i in range(best_left) if modes[i] == 0]
    cols = [order[i] for i in range(best_left) if modes[i] == 1]
    return {"density": best, "rows": np.sort(np.array(rows, np.int64)), "cols": np.sort(np.array(cols, np.int64))}


def max_core_truss(n: int, edges: np.ndarray, core: np.ndarray) -> dict:
    """Kgraph::runTruss (src/graph.cpp:486-563) restated, for SMALL graphs (pure Python): the induced subgraph of the
    vertices of maximal coreness (:470-476, :502), igraph_trussness of its edges (:508; the largest k such that the edge
    lies in a k-truss, i.e. closes >= k - 2 triangles inside it; 2 without triangles) by the textbook support peel,
    and the vertices on edges of maximal trussness (:519-533).  Returns edges as (u, v) original ids, canonical order."""
    kmax = int(core.max()) if n else 0
    inside = core == kmax
    eu, ev = unpack_edges(edges)
    keep = inside[eu] & inside[ev] if edges.size else np.zeros(0, bool)
    su, sv = eu[keep].tolist(), ev[keep].tolist()
    adj = {}
    for a, b in zip(su, sv):
        adj.setdefault(a, set()).add(b)
        adj.setdefault(b, set()).add(a)
    sup = {(a, b): len(adj[a] & adj[b]) for a, b in zip(su, sv)}
    truss = {}
    k = 2
    alive = dict(sup)
    while alive:
        # peel every edge whose support is below what a (k + 1)-truss needs; what is peeled here has trussness k
        queue = [e for e, s in alive.items() if s <= k - 2]
        if not queue:
            k += 1
            continue
        while queue:
            e = queue.pop()
            if e not in alive:
                continue
            a, b = e
            del alive[e]
            truss[e] = k
            for w in adj[a] & adj[b]:
                for f in ((min(a, w), max(a, w)), (min(b, w), max(b, w))):
                    if f in alive:
                        alive[f] -= 1
                        if alive[f] <= k - 2:
                            queue.append(f)
            adj[a].discard(b)
            adj[b].discard(a)
    tr = np.array([truss[(a, b)] for a, b in zip(su, sv)], dtype=np.int32)
    tmax = int(tr.max()) if tr.size else 0
    verts = sorted({x for (a, b), t in truss.items() if t == tmax for x in (a, b)})
    return {"n_core_vertices": int(inside.sum()), "n_core_edges": len(su), "max_trussness": tmax,
            "u": np.array(su, np.uint32), "v": np.array(sv, np.uint32), "trussness": tr,
            "truss_vertices": np.array(verts, np.uint32)}


def unpack_edges(packed: np.ndarray):
    return (packed >> np.uint64(32)).astype(np.uint32), (packed & np.uint64(0xFFFFFFFF)).astype(np.uint32)


def pack_edges(u: np.ndarray, v: np.ndarray) -> np.ndarray:
    return (u.astype(np.uint64) << np.uint64(32)) | v.astype(np.uint64)


# ---------------------------------------------------------------------------
# SAM tokeniser restatement (pure Python; small inputs only)
# ---------------------------------------------------------------------------

def tokenise_sam(data: bytes, threads: int = 1):
    """Restates src/graph.cpp:197-239.  Returns [(read_key: bytes, rname: bytes)].

    The byte range is split statically over `threads` (GCC `omp for` static
    schedule: the first len % T chunks get one extra byte, :206).  A thread
    records the newline offsets inside its chunk (:208-211; thread 0 also seeds
    offset 0, :203) and processes the line starting after every recorded
    offset EXCEPT its last (:214-218) — so the line after each thread's last
    newline is parsed by nobody (quirk Q1; at T=1 only an unterminated final
    line is lost).  A line is skipped if it starts with '@' (:220); the read is
    token 0 and the unitig token 2 under strtok_r(.., "\\t") (:222-231, empty
    fields collapse); RNAME '*' is skipped (:232); key = read.substr(1,
    read.find('/')) (:235, quirk Q2).
    """
    n = len(data)
    base, extra = divmod(n, threads)
    hits = []
    start = 0
    for t in range(threads):
        size = base + (1 if t < extra else 0)
        chunk_lo, chunk_hi = start, start + size
        start = chunk_hi
        pos = [0] if t == 0 else []
        i = data.find(b"\n", chunk_lo, chunk_hi)
        while i != -1:
            pos.append(i)
            i = data.find(b"\n", i + 1, chunk_hi)
        for k in range(1, len(pos)):
            sp = pos[k - 1] + 1
            if sp == 1:
                sp = 0
            if sp >= n or data[sp:sp + 1] == b"@":
                continue
            # strtok_r is not line-bounded, but for well-formed SAM (>= 3 tab
            # separated fields per line) the first three tokens lie in the line.
            eol = data.find(b"\n", sp)
            line = data[sp:eol if eol != -1 else n]
            toks = [x for x in line.split(b"\t") if x]
            if len(toks) < 3:
                raise ValueError("malformed SAM line (undefined behaviour in the reference)")
            read, rname = toks[0], toks[2]
            if rname == b"*":
                continue
            slash = read.find(b"/")
            key = read[1:] if slash == -1 else read[1:1 + slash]
            hits.append((key, rname))
    return hits


def intern_hits(hit_lists):
    """[(key, rname)] per mate file -> (read_key u32[], unitig u32[], names):
    dense ids by first appearance (any injective numbering is equivalent:
    comparisons are by Name, quirk Q4)."""
    keys, names, name_list = {}, {}, []
    rk, ut = [], []
    for hits in hit_lists:
        for key, rname in hits:
            rk.append(keys.setdefault(key, len(keys)))
            if rname not in names:
                names[rname] = len(names)
                name_list.append(rname.decode())
            ut.append(names[rname])
    return np.array(rk, dtype=np.uint32), np.array(ut, dtype=np.uint32), name_list


def komb2_expected(sam1: bytes, sam2: bytes, threads: int = 1, key_mode: int = KEY_REF32):
    """Whole-path expectation from SAM bytes: canonical dict like read_outputs()."""
    rk, ut, names = intern_hits([tokenise_sam(sam1, threads), tokenise_sam(sam2, threads)])
    n = len(names)
    edges, _, _ = build_edges(rk, ut)
    deg, core = coreness(n, edges)
    score = corea(core, deg, key_mode)
    eu, ev = unpack_edges(edges)
    return {
        "edges": {tuple(sorted((names[a], names[b]))) for a, b in zip(eu.tolist(), ev.tolist())},
        "kcore": {names[i]: (int(core[i]), int(deg[i])) for i in range(n)},
        "score": {names[i]: float(score[i]) for i in range(n)},
    }


# ---------------------------------------------------------------------------
# komb2 output files -> canonical, Name-keyed form (quirks Q4, Q7, Q9)
# ---------------------------------------------------------------------------

def read_outputs(outdir) -> dict:
    outdir = Path(outdir)
    vid_name, kcore = {}, {}
    with open(outdir / "kcore.tsv") as f:
        header = f.readline()
        assert header == "#VID\tName\tCoreness\tDegree\n", header
        for line in f:
            vid, name, c, d = line.rstrip("\n").split("\t")
            vid_name[int(vid)] = name
            kcore[name] = (int(c), int(d))
    edges = set()
    with open(outdir / "edgelist.txt") as f:
        for line in f:
            a, b = line.split("\t")
            a, b = int(a), int(b)
            if a == b:
                continue
            edges.add(tuple(sorted((vid_name[a], vid_name[b]))))
    score, score_text = {}, {}
    with open(outdir / "CoreA_anomaly.txt") as f:
        for line in f:
            vid, s = line.rstrip("\n").split("\t")
            score[vid_name[int(vid)]] = float(s)
            score_text[vid_name[int(vid)]] = s
    return {"edges": edges, "kcore": kcore, "score": score, "score_text": score_text}


def run_komb2(binary, sam1: bytes, sam2: bytes, workdir, n_unitigs_fasta: int = 4, threads: int = 1,
              extra_env=None):
    """Run a komb2 executable (reference build or drop-in) the way KOMB.py does
    (KOMB.py:436-442).  Returns (canonical outputs, stdout)."""
    workdir = Path(workdir)
    out = workdir / "out"
    out.mkdir(parents=True, exist_ok=True)
    (workdir / "r1.sam").write_bytes(sam1)
    (workdir / "r2.sam").write_bytes(sam2)
    with open(workdir / "unitigs.fasta", "w") as f:
        for u in range(n_unitigs_fasta):
            f.write(f">{u} LN:i:8\nACGTACGT\n")
    env = dict(os.environ)
    if extra_env:
        env.update(extra_env)
    cp = subprocess.run([str(binary), "-t", str(threads), "-l", "100", "-o", str(out),
                         "-i", str(workdir / "r1.sam"), "-j", str(workdir / "r2.sam"),
                         "-u", str(workdir / "unitigs.fasta")],
                        capture_output=True, text=True, env=env)
    if cp.returncode != 0:
        raise RuntimeError(f"{binary} rc={cp.returncode}\n{cp.stdout}\n{cp.stderr}")
    return read_outputs(out), cp.stdout


def corea_reference(core: np.ndarray, deg: np.ndarray, workdir) -> np.ndarray:
    """CoreA::getAnomalyScore straight from the reference header (oracle/_ref/corea_ref)."""
    workdir = Path(workdir)
    n = int(core.shape[0])
    with open(workdir / "corea_in.bin", "wb") as f:
        f.write(np.array([n], dtype=np.int32).tobytes())
        f.write(np.ascontiguousarray(core, dtype=np.int32).tobytes())
        f.write(np.ascontiguousarray(deg, dtype=np.int32).tobytes())
    subprocess.run([str(REF_COREA), str(workdir / "corea_in.bin"), str(workdir / "corea_out.bin")], check=True)
    return np.fromfile(workdir / "corea_out.bin", dtype=np.float64)
