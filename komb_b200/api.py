"""Host-side Python face of the KOMB hot path, a thin mirror of the C ABI
(include/kombgpu.h) used by the tests and by bench.py.

The call order is the reference's (src/komb2.cpp:93-132):
    readSAM x2 + getEdgeInfo + generateGraph + igraph_create/simplify -> Context.build_graph
    runCore (igraph_degree, igraph_coreness)                         -> Graph.degree / Graph.coreness
    anomalyDetection -> CombineCoreA::run -> CoreA::getAnomalyScore   -> Graph.corea

Arrays may be numpy arrays (host pointers -> the plain entry points, copies
included) or torch CUDA tensors (device pointers -> the `_dev` entry points).
Everything is computed by the CUDA library; nothing here falls back to the CPU.
"""
from __future__ import annotations

import ctypes
from ctypes import byref, c_double, c_int32, c_uint32, c_uint64, c_void_p

import numpy as np

from . import _lib
from ._lib import KEY_EXACT64, KEY_REF32, KombGpuError, Stats  # noqa: F401


def _is_torch_cuda(x) -> bool:
    return hasattr(x, "data_ptr") and hasattr(x, "is_cuda") and x.is_cuda


def _host(x, dtype) -> np.ndarray:
    a = np.ascontiguousarray(x, dtype=dtype)
    return a


def _ptr(a: np.ndarray) -> c_void_p:
    return c_void_p(a.ctypes.data)


class Context:
    """One per process and device (kombgpu_ctx)."""

    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        h = c_void_p()
        rc = self._lib.kombgpu_ctx_create(int(device), byref(h))
        if rc != 0:
            raise KombGpuError(rc, self._lib.kombgpu_last_error(None).decode())
        self._h = h
        self.device = int(device)
        self._pinned = []

    def close(self):
        if getattr(self, "_h", None):
            for p in self._pinned:
                self._lib.kombgpu_pinned_free(self._h, p)
            self._pinned = []
            self._lib.kombgpu_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise KombGpuError(rc, self._lib.kombgpu_last_error(self._h).decode())

    def set_stream(self, cuda_stream: int | None):
        """Run on an existing CUDA stream handle; 0 / None is CUDA's legacy default stream
        (torch's default).  reset_stream() goes back to the context's private stream."""
        self._check(self._lib.kombgpu_ctx_set_stream(self._h, c_void_p(cuda_stream or 0)))

    def reset_stream(self):
        self._check(self._lib.kombgpu_ctx_reset_stream(self._h))

    def pinned_empty(self, count: int, dtype) -> np.ndarray:
        """A page-locked numpy array (freed with the context): pass it as `out=` to the getters, or fill it
        with hits, so that host<->device copies run at full PCIe rate."""
        dt = np.dtype(dtype)
        p = c_void_p()
        self._check(self._lib.kombgpu_pinned_alloc(self._h, int(count) * dt.itemsize, byref(p)))
        self._pinned.append(p)
        buf = (ctypes.c_char * (max(int(count), 0) * dt.itemsize)).from_address(p.value)
        return np.frombuffer(buf, dtype=dt, count=int(count))

    def launches(self) -> int:
        """Kernels of libkombgpu launched through this context so far."""
        n = c_uint64()
        self._check(self._lib.kombgpu_ctx_launches(self._h, byref(n)))
        return n.value

    def trim(self):
        self._check(self._lib.kombgpu_ctx_trim(self._h))

    def _pair_call(self, host_fn, dev_fn, a, b, n_vertices: int) -> "Graph":
        g = c_void_p()
        if _is_torch_cuda(a):
            import torch
            assert _is_torch_cuda(b) and a.dtype in (torch.uint32, torch.int32) and b.dtype == a.dtype
            assert a.is_contiguous() and b.is_contiguous() and a.numel() == b.numel()
            rc = dev_fn(self._h, c_void_p(a.data_ptr()), c_void_p(b.data_ptr()), a.numel(), n_vertices, byref(g))
            keep = (a, b)
        else:
            ha, hb = _host(a, np.uint32), _host(b, np.uint32)
            if ha.shape != hb.shape or ha.ndim != 1:
                raise ValueError("expected two 1-D arrays of equal length")
            rc = host_fn(self._h, _ptr(ha), _ptr(hb), ha.shape[0], n_vertices, byref(g))
            keep = None
        self._check(rc)
        return Graph(self, g, keep)

    def build_graph(self, read_key, unitig, n_vertices: int) -> "Graph":
        """Hits of both mate files (concatenated) -> simple unitig graph."""
        return self._pair_call(self._lib.kombgpu_build_graph, self._lib.kombgpu_build_graph_dev,
                               read_key, unitig, int(n_vertices))

    def analyse_hits_csr(self, read_key, unitig, n_vertices: int, key_mode: int = KEY_REF32, out: dict | None = None,
                         edge_capacity: int | None = None) -> tuple["Graph", dict]:
        """analyse_hits with the edge list in CSR form (kombgpu_analyse_hits_csr): result keys fwd_ptr (uint64[n+1])
        and v (uint32[E]) instead of u and v -- half the device-to-host bytes."""
        ha, hb = _host(read_key, np.uint32), _host(unitig, np.uint32)
        if ha.shape != hb.shape or ha.ndim != 1:
            raise ValueError("expected two 1-D arrays of equal length")
        out = out or {}
        n = int(n_vertices)
        if out.get("v") is not None:
            cap = out["v"].shape[0] if edge_capacity is None else int(edge_capacity)
            bv = out["v"]
        else:
            cap = 3 * ha.shape[0] if edge_capacity is None else int(edge_capacity)
            bv = np.empty(cap, np.uint32)
        r = {"fwd_ptr": Graph._out(out.get("fwd_ptr"), n + 1, np.uint64), "degree": Graph._out(out.get("degree"), n, np.int32),
             "coreness": Graph._out(out.get("coreness"), n, np.int32), "score": Graph._out(out.get("score"), n, np.float64)}
        g = c_void_p()
        self._check(self._lib.kombgpu_analyse_hits_csr(self._h, _ptr(ha), _ptr(hb), ha.shape[0], n, int(key_mode), cap, _ptr(r["fwd_ptr"]),
                                                       _ptr(bv), _ptr(r["degree"]), _ptr(r["coreness"]), _ptr(r["score"]), byref(g)))
        graph = Graph(self, g, None)
        r["v"] = bv[:graph.counts()[1]]
        return graph, r

    def analyse_hits(self, read_key, unitig, n_vertices: int, key_mode: int = KEY_REF32, out: dict | None = None,
                     edge_capacity: int | None = None) -> tuple["Graph", dict]:
        """Host hits in, every result on the host, one call (kombgpu_analyse_hits): the edge list starts downloading
        half-way through the build.  `out` may hold caller buffers (u, v, degree, coreness, score; e.g. pinned_empty
        arrays); u / v must hold `edge_capacity` entries (default: their length, or 3 x the number of hits when
        they are allocated here).  Returns the graph and the result arrays (u / v cut to the edge count)."""
        ha, hb = _host(read_key, np.uint32), _host(unitig, np.uint32)
        if ha.shape != hb.shape or ha.ndim != 1:
            raise ValueError("expected two 1-D arrays of equal length")
        out = out or {}
        n = int(n_vertices)
        if out.get("u") is not None:
            cap = min(out["u"].shape[0], out["v"].shape[0]) if edge_capacity is None else int(edge_capacity)
            bu, bv = out["u"], out["v"]
        else:
            cap = 3 * ha.shape[0] if edge_capacity is None else int(edge_capacity)
            bu, bv = np.empty(cap, np.uint32), np.empty(cap, np.uint32)
        r = {"degree": Graph._out(out.get("degree"), n, np.int32), "coreness": Graph._out(out.get("coreness"), n, np.int32),
             "score": Graph._out(out.get("score"), n, np.float64)}
        g = c_void_p()
        self._check(self._lib.kombgpu_analyse_hits(self._h, _ptr(ha), _ptr(hb), ha.shape[0], n, int(key_mode), cap, _ptr(bu), _ptr(bv),
                                                   _ptr(r["degree"]), _ptr(r["coreness"]), _ptr(r["score"]), byref(g)))
        graph = Graph(self, g, None)
        m = graph.counts()[1]
        r["u"], r["v"] = bu[:m], bv[:m]
        return graph, r

    def sam_parse(self, texts) -> "Hits":
        """SAM bytes of the mate files (mate 1 first) -> integer hits on the device (kombgpu_sam_parse): the GPU
        form of Kgraph::readSAM's tokeniser + interner (src/graph.cpp:197-256)."""
        texts = [bytes(t) for t in texts]
        n = len(texts)
        arr = (ctypes.c_char_p * max(n, 1))(*texts)
        sizes = (c_uint64 * max(n, 1))(*[len(t) for t in texts])
        h = c_void_p()
        self._check(self._lib.kombgpu_sam_parse(self._h, arr, sizes, n, byref(h)))
        return Hits(self, h, texts)

    def fasta(self, text: bytes) -> "Fasta":
        """Upload the bytes of a FASTA file and index its records on the device (kombgpu_fasta_load)."""
        text = bytes(text)
        h = c_void_p()
        self._check(self._lib.kombgpu_fasta_load(self._h, text, len(text), byref(h)))
        return Fasta(self, h)

    def anomalous(self, score, whisker: float = 1.5) -> dict:
        """IQR fence on CORE-A over host scores (kombgpu_anomalous): q1, q3, fence, n_selected and the member mask."""
        sc = _host(score, np.float64)
        if sc.ndim != 1:
            raise ValueError("expected a 1-D array of scores")
        member = np.zeros(sc.shape[0], np.uint8)
        q1, q3, fence, ns = c_double(), c_double(), c_double(), c_uint32()
        self._check(self._lib.kombgpu_anomalous(self._h, _ptr(sc), sc.shape[0], float(whisker), byref(q1), byref(q3), byref(fence), byref(ns),
                                                _ptr(member)))
        return {"q1": q1.value, "q3": q3.value, "fence": fence.value, "n_selected": ns.value, "member": member.astype(bool)}

    def graph_from_edges(self, u, v, n_vertices: int) -> "Graph":
        return self._pair_call(self._lib.kombgpu_graph_from_edges, self._lib.kombgpu_graph_from_edges_dev,
                               u, v, int(n_vertices))

    def graph_from_csr(self, row_ptr, col, n_vertices: int) -> "Graph":
        """Adopt a device-resident CSR (torch CUDA tensors: int64 row_ptr[n+1], int32 col)."""
        g = c_void_p()
        self._check(self._lib.kombgpu_graph_from_csr_dev(self._h, c_void_p(row_ptr.data_ptr()),
                                                         c_void_p(col.data_ptr() if col.numel() else 0), int(n_vertices), byref(g)))
        return Graph(self, g, (row_ptr, col))

    def format_corea(self, score) -> bytes:
        """CoreA_anomaly.txt ("%d\\t%f\\n" rows) from a host array of scores, formatted on the device."""
        sc = _host(score, np.float64)
        n = c_uint64()
        cap = 40 * sc.shape[0] + 16
        buf = ctypes.create_string_buffer(cap)
        self._check(self._lib.kombgpu_format_corea(self._h, _ptr(sc), sc.shape[0], buf, cap, byref(n)))
        return buf.raw[:n.value]

    def corea(self, coreness, degree, key_mode: int = KEY_REF32) -> np.ndarray:
        """CoreA::getAnomalyScore on host arrays."""
        c, d = _host(coreness, np.int32), _host(degree, np.int32)
        if c.shape != d.shape or c.ndim != 1:
            raise ValueError("expected two 1-D arrays of equal length")
        score = np.empty(c.shape[0], dtype=np.float64)
        self._check(self._lib.kombgpu_corea(self._h, _ptr(c), _ptr(d), c.shape[0], int(key_mode), _ptr(score)))
        return score


class Hits:
    """Device-resident tokenised hits of a set of SAM files (kombgpu_hits)."""

    def __init__(self, ctx: Context, handle: c_void_p, texts):
        self._ctx, self._lib, self._h, self._texts = ctx, ctx._lib, handle, texts

    def close(self):
        if getattr(self, "_h", None):
            self._lib.kombgpu_hits_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def counts(self) -> dict:
        nh, nr, nu, nl = c_uint64(), c_uint32(), c_uint32(), c_uint64()
        self._ctx._check(self._lib.kombgpu_hits_counts(self._h, byref(nh), byref(nr), byref(nu), byref(nl)))
        return {"n_hits": nh.value, "n_reads": nr.value, "n_unitigs": nu.value, "n_lines": nl.value}

    def names(self) -> list[bytes]:
        """Unitig name of every vertex, cut out of the input bytes with the spans the device reports."""
        n = self.counts()["n_unitigs"]
        f, off, ln = np.empty(n, np.uint32), np.empty(n, np.uint64), np.empty(n, np.uint32)
        self._ctx._check(self._lib.kombgpu_hits_names(self._h, _ptr(f), _ptr(off), _ptr(ln)))
        return [self._texts[int(f[i])][int(off[i]):int(off[i]) + int(ln[i])] for i in range(n)]

    def download(self) -> tuple[np.ndarray, np.ndarray]:
        n = self.counts()["n_hits"]
        rk, ut = np.empty(n, np.uint32), np.empty(n, np.uint32)
        self._ctx._check(self._lib.kombgpu_hits_download(self._h, _ptr(rk), _ptr(ut)))
        return rk, ut

    def timing(self) -> dict:
        a, b, l, r = ctypes.c_float(), ctypes.c_float(), c_uint64(), ctypes.c_int()
        self._ctx._check(self._lib.kombgpu_hits_timing(self._h, byref(a), byref(b), byref(l), byref(r)))
        return {"ms_upload": a.value, "ms_parse": b.value, "kernel_launches": l.value, "hash_rounds": r.value}

    def build_graph(self) -> "Graph":
        g = c_void_p()
        self._ctx._check(self._lib.kombgpu_build_graph_hits(self._h, byref(g)))
        return Graph(self._ctx, g, self)


class Fasta:
    """A FASTA file indexed on the device (kombgpu_fasta): join its records to a graph's vertices by name, then copy
    out the records of selected vertices."""

    def __init__(self, ctx: Context, handle: c_void_p):
        self._ctx, self._lib, self._h = ctx, ctx._lib, handle

    def close(self):
        if getattr(self, "_h", None):
            self._lib.kombgpu_fasta_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def counts(self) -> dict:
        nr, nb = c_uint32(), c_uint64()
        self._ctx._check(self._lib.kombgpu_fasta_counts(self._h, byref(nr), byref(nb)))
        return {"n_records": nr.value, "n_bytes": nb.value}

    def join(self, hits: "Hits | None" = None, names=None) -> int:
        """vertex -> record by name: the vertex names of `hits` (the device copy of the SAM text), or a host list of
        names (bytes), vertex v = names[v].  Returns the number of vertices without a record."""
        if (hits is None) == (names is None):
            raise ValueError("pass exactly one of hits= and names=")
        miss = c_uint32()
        if hits is not None:
            self._ctx._check(self._lib.kombgpu_fasta_join_hits(self._h, hits._h, byref(miss)))
        else:
            names = [bytes(x) for x in names]
            off = np.zeros(len(names) + 1, np.uint64)
            np.cumsum([len(x) for x in names], out=off[1:])
            self._ctx._check(self._lib.kombgpu_fasta_join_names(self._h, b"".join(names), _ptr(off), len(names), byref(miss)))
        return miss.value

    def extract(self, mask) -> bytes:
        """The records of the vertices with a true mask entry, verbatim, in file order (kombgpu_fasta_extract)."""
        m = np.ascontiguousarray(np.asarray(mask).astype(bool).astype(np.uint8))
        n = c_uint64()
        self._ctx._check(self._lib.kombgpu_fasta_extract(self._h, _ptr(m), m.shape[0], byref(n)))
        buf = ctypes.create_string_buffer(max(n.value, 1))
        self._ctx._check(self._lib.kombgpu_fasta_extract_fetch(self._h, buf))
        return buf.raw[:n.value]

    def timing(self) -> dict:
        up, ix, jn, ex, l = ctypes.c_float(), ctypes.c_float(), ctypes.c_float(), ctypes.c_float(), c_uint64()
        self._ctx._check(self._lib.kombgpu_fasta_timing(self._h, byref(up), byref(ix), byref(jn), byref(ex), byref(l)))
        return {"ms_upload": up.value, "ms_index": ix.value, "ms_join": jn.value, "ms_extract": ex.value, "kernel_launches": l.value}


class Graph:
    """Device-resident simple unitig graph (kombgpu_graph)."""

    def __init__(self, ctx: Context, handle: c_void_p, keepalive=None):
        self._ctx = ctx
        self._lib = ctx._lib
        self._h = handle
        self._keep = keepalive

    def close(self):
        if getattr(self, "_h", None):
            self._lib.kombgpu_graph_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def counts(self) -> tuple[int, int]:
        n, m = c_uint32(), c_uint64()
        self._ctx._check(self._lib.kombgpu_graph_counts(self._h, byref(n), byref(m)))
        return n.value, m.value

    @staticmethod
    def _out(out, count, dtype):
        if out is None:
            return np.empty(count, dtype)
        if out.dtype != np.dtype(dtype) or out.ndim != 1 or out.shape[0] < count or not out.flags.c_contiguous:
            raise ValueError(f"out= must be a contiguous 1-D {np.dtype(dtype)} array of at least {count} elements")
        return out[:count]

    def edges(self, out=None) -> tuple[np.ndarray, np.ndarray]:
        """Canonical edge list; `out=(u_buf, v_buf)` reuses caller (e.g. page-locked) buffers."""
        _, m = self.counts()
        u = self._out(out[0] if out else None, m, np.uint32)
        v = self._out(out[1] if out else None, m, np.uint32)
        self._ctx._check(self._lib.kombgpu_graph_edges(self._h, _ptr(u), _ptr(v)))
        return u, v

    def edges_csr(self, out=None) -> tuple[np.ndarray, np.ndarray]:
        """Canonical edge list in CSR form: (fwd_ptr uint64[n+1], v uint32[E]); edge i has source u where
        fwd_ptr[u] <= i < fwd_ptr[u+1] (kombgpu_graph_edges_csr)."""
        n, m = self.counts()
        fp = self._out(out[0] if out else None, n + 1, np.uint64)
        v = self._out(out[1] if out else None, m, np.uint32)
        self._ctx._check(self._lib.kombgpu_graph_edges_csr(self._h, _ptr(fp), _ptr(v)))
        return fp, v

    def edge_multiplicity(self) -> np.ndarray:
        """Pairs that collapsed into each edge of the canonical edge list (kombgpu_graph_edge_multiplicity)."""
        _, m = self.counts()
        mult = np.empty(m, np.uint32)
        self._ctx._check(self._lib.kombgpu_graph_edge_multiplicity(self._h, _ptr(mult)))
        return mult

    def csr(self) -> tuple[np.ndarray, np.ndarray]:
        n, m = self.counts()
        row_ptr, col = np.empty(n + 1, np.uint64), np.empty(2 * m, np.uint32)
        self._ctx._check(self._lib.kombgpu_graph_csr(self._h, _ptr(row_ptr), _ptr(col)))
        return row_ptr, col

    def degree(self, out=None) -> np.ndarray:
        n, _ = self.counts()
        d = self._out(out, n, np.int32)
        self._ctx._check(self._lib.kombgpu_degree(self._h, _ptr(d)))
        return d

    def coreness(self, copy: bool = True, out=None, again: bool = False):
        """igraph_coreness.  `again=True` (measurement aid, include/kombgpu_debug.h) peels once more on a graph that
        already holds its coreness."""
        n, _ = self.counts()
        if again:
            self._ctx._check(self._lib.kombgpu_debug_peel_again(self._h))
        if not copy:
            self._ctx._check(self._lib.kombgpu_coreness(self._h, None))
            return None
        c = self._out(out, n, np.int32)
        self._ctx._check(self._lib.kombgpu_coreness(self._h, _ptr(c)))
        return c

    def corea(self, key_mode: int = KEY_REF32, copy: bool = True, out=None):
        n, _ = self.counts()
        if not copy:
            self._ctx._check(self._lib.kombgpu_graph_corea(self._h, int(key_mode), None))
            return None
        s = self._out(out, n, np.float64)
        self._ctx._check(self._lib.kombgpu_graph_corea(self._h, int(key_mode), _ptr(s)))
        return s

    def results(self, key_mode: int = KEY_REF32, out: dict | None = None) -> dict:
        """Everything the komb2 host writes, in one call (kombgpu_graph_results): runs peel + CORE-A if needed;
        the edge-list download overlaps the peel.  `out` may hold caller buffers under the keys
        u, v, degree, coreness, score (e.g. Context.pinned_empty arrays)."""
        n, m = self.counts()
        out = out or {}
        r = {"u": self._out(out.get("u"), m, np.uint32), "v": self._out(out.get("v"), m, np.uint32),
             "degree": self._out(out.get("degree"), n, np.int32), "coreness": self._out(out.get("coreness"), n, np.int32),
             "score": self._out(out.get("score"), n, np.float64)}
        self._ctx._check(self._lib.kombgpu_graph_results(self._h, int(key_mode), _ptr(r["u"]), _ptr(r["v"]), _ptr(r["degree"]),
                                                         _ptr(r["coreness"]), _ptr(r["score"])))
        return r

    def results_csr(self, key_mode: int = KEY_REF32, out: dict | None = None) -> dict:
        """results() with the edge list in CSR form (fwd_ptr, v): half the download (kombgpu_graph_results_csr)."""
        n, m = self.counts()
        out = out or {}
        r = {"fwd_ptr": self._out(out.get("fwd_ptr"), n + 1, np.uint64), "v": self._out(out.get("v"), m, np.uint32),
             "degree": self._out(out.get("degree"), n, np.int32), "coreness": self._out(out.get("coreness"), n, np.int32),
             "score": self._out(out.get("score"), n, np.float64)}
        self._ctx._check(self._lib.kombgpu_graph_results_csr(self._h, int(key_mode), _ptr(r["fwd_ptr"]), _ptr(r["v"]), _ptr(r["degree"]),
                                                             _ptr(r["coreness"]), _ptr(r["score"])))
        return r

    def analyse(self, key_mode: int = KEY_REF32):
        self._ctx._check(self._lib.kombgpu_graph_analyse(self._h, int(key_mode)))

    FILE_EDGELIST, FILE_KCORE, FILE_COREA, FILE_ONION = 0, 1, 2, 3

    def format(self, which: int, hits: "Hits | None" = None) -> bytes:
        """The bytes of edgelist.txt / kcore.tsv / CoreA_anomaly.txt / onion.tsv, formatted on the device
        (kombgpu_graph_format); kcore.tsv and onion.tsv take the unitig names from the Hits the graph was built from."""
        n = c_uint64()
        self._ctx._check(self._lib.kombgpu_graph_format(self._h, int(which), hits._h if hits is not None else None, byref(n)))
        buf = ctypes.create_string_buffer(max(n.value, 1))
        self._ctx._check(self._lib.kombgpu_graph_format_fetch(self._h, int(which), buf, 0))
        return buf.raw[:n.value]

    def summary(self) -> tuple[int, float]:
        mc, ms = c_int32(), c_double()
        self._ctx._check(self._lib.kombgpu_graph_summary(self._h, byref(mc), byref(ms)))
        return mc.value, ms.value

    def densest_core(self) -> dict:
        """Densest k-core {v : coreness(v) >= k}: level, size and edges / vertices (kombgpu_graph_densest_core)."""
        k, nv, ne, d = c_int32(), c_uint32(), c_uint64(), c_double()
        self._ctx._check(self._lib.kombgpu_graph_densest_core(self._h, byref(k), byref(nv), byref(ne), byref(d)))
        return {"k": k.value, "n_vertices": nv.value, "n_edges": ne.value, "density": d.value}

    def densest_block(self, weight=None, use_scores: bool = False, eps: float = 0.5) -> dict:
        """Densest block by the bulk form of the reference's greedy peel (kombgpu_graph_densest_block): sizes, density
        f(S) / |S| with f = weights + edges inside S, passes, and the block's membership mask."""
        n, _ = self.counts()
        nv, ne, ws, d, np_ = c_uint32(), c_uint64(), c_double(), c_double(), c_uint32()
        member = np.zeros(n, np.uint8)
        wt = _host(weight, np.float64) if weight is not None else None
        if wt is not None and wt.shape != (n,):
            raise ValueError("weight must hold one value per vertex")
        self._ctx._check(self._lib.kombgpu_graph_densest_block(self._h, _ptr(wt) if wt is not None else None, int(bool(use_scores)), float(eps),
                                                               byref(nv), byref(ne), byref(ws), byref(d), byref(np_), _ptr(member)))
        return {"n_vertices": nv.value, "n_edges": ne.value, "weight_sum": ws.value, "density": d.value, "passes": np_.value,
                "member": member.astype(bool)}

    def max_core_truss(self) -> dict:
        """Maximal core + trussness of its edges (kombgpu_graph_max_core_truss, reference Kgraph::runTruss): sizes, the
        induced edges (original ids) with their trussness, and the unitigs on edges of maximal trussness."""
        nc, mc, tm, nt = c_uint32(), c_uint64(), c_int32(), c_uint32()
        self._ctx._check(self._lib.kombgpu_graph_max_core_truss(self._h, byref(nc), byref(mc), byref(tm), byref(nt)))
        u, v, tr = np.empty(mc.value, np.uint32), np.empty(mc.value, np.uint32), np.empty(mc.value, np.int32)
        self._ctx._check(self._lib.kombgpu_graph_max_core_edges(self._h, _ptr(u), _ptr(v), _ptr(tr)))
        tv = np.empty(nt.value, np.uint32)
        self._ctx._check(self._lib.kombgpu_graph_truss_vertices(self._h, _ptr(tv)))
        return {"n_core_vertices": nc.value, "n_core_edges": mc.value, "max_trussness": tm.value, "u": u, "v": v, "trussness": tr,
                "truss_vertices": tv}

    def onion(self, again: bool = False) -> dict:
        """Onion layers (kombgpu_graph_onion; networkx.onion_layers): the 1-based layer of every vertex and the number of
        layers.  `again=True` (measurement aid, include/kombgpu_debug.h) runs the decomposition once more."""
        n, _ = self.counts()
        if again:
            self._ctx._check(self._lib.kombgpu_debug_onion_again(self._h))
        layer, nl = np.empty(n, np.uint32), c_uint32()
        self._ctx._check(self._lib.kombgpu_graph_onion(self._h, _ptr(layer), byref(nl)))
        return {"layer": layer, "n_layers": nl.value}

    def onion_timing(self) -> dict:
        """What the last onion run measured (measurement aid, include/kombgpu_debug.h): kernel time from CUDA events,
        non-empty levels, steps between grid barriers, layers run by one CTA."""
        ms, lv, steps, thin = ctypes.c_float(), c_uint32(), c_uint32(), c_uint32()
        self._ctx._check(self._lib.kombgpu_debug_onion_timing(self._h, byref(ms), byref(lv), byref(steps), byref(thin)))
        return {"ms_kernel": ms.value, "levels": lv.value, "steps": steps.value, "thin_layers": thin.value}

    def anomalous(self, whisker: float = 1.5) -> dict:
        """IQR fence on the graph's own CORE-A scores (kombgpu_graph_anomalous; needs corea() first)."""
        n, _ = self.counts()
        member = np.zeros(n, np.uint8)
        q1, q3, fence, ns = c_double(), c_double(), c_double(), c_uint32()
        self._ctx._check(self._lib.kombgpu_graph_anomalous(self._h, float(whisker), byref(q1), byref(q3), byref(fence), byref(ns), _ptr(member)))
        return {"q1": q1.value, "q3": q3.value, "fence": fence.value, "n_selected": ns.value, "member": member.astype(bool)}

    def build_chunks(self) -> int:
        """Chunks the build reduced its clique pairs in: 1 for the one-shot path (measurement aid,
        include/kombgpu_debug.h)."""
        n = c_uint32()
        self._ctx._check(self._lib.kombgpu_debug_build_chunks(self._h, byref(n)))
        return n.value

    def stats(self) -> dict:
        st = Stats()
        self._ctx._check(self._lib.kombgpu_graph_stats(self._h, byref(st)))
        return st.as_dict()

    def device_arrays(self) -> dict:
        ptrs = [c_void_p() for _ in range(6)]
        self._ctx._check(self._lib.kombgpu_graph_device_arrays(self._h, *[byref(p) for p in ptrs]))
        names = ["row_ptr", "col", "edges_packed", "degree", "coreness", "score"]
        return {k: (p.value or 0) for k, p in zip(names, ptrs)}
