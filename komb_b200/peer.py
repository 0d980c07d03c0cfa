"""Python face of the peer-memory multi-GPU path (include/kombgpu.h, "multi-GPU, peer-memory path"): a thin
ctypes mirror.  All compute — partitioned build, device-driven peel over NVLink mailboxes, sharded CORE-A — is
in libkombgpu.so; Python only provides the bootstrap all-gather when the ranks are separate processes.

    one process per GPU (torchrun):   comm = Comm.from_torch(ctx)          # bootstrap over torch.distributed
    one process, a thread per GPU:    run_local(world, fn, devices=[...])  # bootstrap built into the library
    tests on a one-GPU box:           run_local(world, fn)                 # every rank on device 0 (emulation)
"""
from __future__ import annotations

import ctypes
import threading
from ctypes import byref, c_double, c_float, c_int, c_int32, c_uint32, c_uint64, c_void_p

import numpy as np

from . import _lib
from ._lib import KEY_REF32, DistStats
from .api import Context


class Comm:
    """kombgpu_comm: one rank of the peer-memory communicator."""

    def __init__(self, ctx: Context, handle: c_void_p, keep=None):
        self.ctx = ctx
        self._lib = ctx._lib
        self._h = handle
        self._keep = keep
        r, w, sd, hb = c_int(), c_int(), c_int(), c_uint64()
        ctx._check(self._lib.kombgpu_comm_info(self._h, byref(r), byref(w), byref(sd), byref(hb)))
        self.rank, self.world, self.same_device = r.value, w.value, bool(sd.value)

    @classmethod
    def create(cls, ctx: Context, rank: int, world: int, allgather, heap_bytes: int = 0) -> "Comm":
        """`allgather(data: bytes) -> list[bytes]` gathers one blob per rank, in rank order (any transport)."""
        def _cb(_user, send, recv, nbytes):
            try:
                parts = allgather(ctypes.string_at(send, nbytes))
                blob = b"".join(parts)
                if len(blob) != nbytes * world:
                    return -1
                ctypes.memmove(recv, blob, len(blob))
                return 0
            except Exception:   # the C side turns this into KOMBGPU_ESTATE
                return -1
        cb = _lib.ALLGATHER_FN(_cb)
        h = c_void_p()
        ctx._check(ctx._lib.kombgpu_comm_create(ctx._h, rank, world, cb, None, int(heap_bytes), byref(h)))
        return cls(ctx, h, keep=(cb, allgather))

    @classmethod
    def from_torch(cls, ctx: Context, heap_bytes: int = 0) -> "Comm":
        """Ranks = the processes of the initialised torch.distributed group (one GPU each)."""
        import torch.distributed as dist
        world, rank = dist.get_world_size(), dist.get_rank()

        def gather(data: bytes):
            out = [None] * world
            dist.all_gather_object(out, data)
            return out
        return cls.create(ctx, rank, world, gather, heap_bytes)

    @classmethod
    def create_local(cls, ctx: Context, rank: int, world: int, group_slot: c_void_p, heap_bytes: int = 0) -> "Comm":
        h = c_void_p()
        ctx._check(ctx._lib.kombgpu_comm_create_local(ctx._h, rank, world, byref(group_slot), int(heap_bytes), byref(h)))
        return cls(ctx, h, keep=group_slot)

    def heap_bytes(self) -> int:
        hb = c_uint64()
        self.ctx._check(self._lib.kombgpu_comm_info(self._h, None, None, None, byref(hb)))
        return hb.value

    def close(self):
        if getattr(self, "_h", None):
            self._lib.kombgpu_comm_destroy(self._h)
            self._h = None


class DistGraph:
    """kombgpu_dist_graph: this rank's share of the partitioned graph."""

    def __init__(self, comm: Comm, handle: c_void_p, keep=None):
        self.comm = comm
        self._ctx = comm.ctx
        self._lib = comm._lib
        self._h = handle
        self._keep = keep

    @classmethod
    def _build(cls, fn, comm: Comm, a, b, n_global: int) -> "DistGraph":
        assert a.is_cuda and b.is_cuda and a.is_contiguous() and b.is_contiguous() and a.numel() == b.numel()
        h = c_void_p()
        comm.ctx._check(fn(comm._h, c_void_p(a.data_ptr() if a.numel() else 0), c_void_p(b.data_ptr() if b.numel() else 0),
                           a.numel(), int(n_global), byref(h)))
        return cls(comm, h, keep=(a, b))

    @classmethod
    def from_hits(cls, comm: Comm, read_key, unitig, n_global: int) -> "DistGraph":
        """Hits of THIS rank's reads (torch CUDA int32/uint32 tensors, global unitig ids).  Collective."""
        return cls._build(comm._lib.kombgpu_dist_build_hits_dev, comm, read_key, unitig, n_global)

    @classmethod
    def from_dist_hits(cls, hits: "DistHits") -> "DistGraph":
        """The graph of the hits a DistHits routed to this rank, n_global = its n_unitigs.  Collective."""
        h = c_void_p()
        hits.comm.ctx._check(hits._lib.kombgpu_dist_build_graph_hits(hits._h, byref(h)))
        return cls(hits.comm, h, keep=hits)

    @classmethod
    def from_pairs(cls, comm: Comm, u, v, n_global: int) -> "DistGraph":
        """This rank's share of an edge list.  Collective."""
        return cls._build(comm._lib.kombgpu_dist_build_pairs_dev, comm, u, v, n_global)

    def coreness(self):
        self._ctx._check(self._lib.kombgpu_dist_coreness(self._h))

    def corea(self, key_mode: int = KEY_REF32):
        self._ctx._check(self._lib.kombgpu_dist_corea(self._h, int(key_mode)))

    def analyse(self, key_mode: int = KEY_REF32):
        self.coreness()
        self.corea(key_mode)

    def stats(self) -> dict:
        st = DistStats()
        self._ctx._check(self._lib.kombgpu_dist_graph_stats(self._h, byref(st)))
        return st.as_dict()

    def build_rounds(self) -> int:
        """Rounds the build emitted, routed and reduced the clique pairs in: 1 on the one-shot path (kombgpu_debug.h)."""
        n = c_uint32()
        self._ctx._check(self._lib.kombgpu_debug_dist_build_rounds(self._h, byref(n)))
        return n.value

    def summary(self) -> tuple[int, float]:
        mc, ms = c_int32(), c_double()
        self._ctx._check(self._lib.kombgpu_dist_graph_summary(self._h, byref(mc), byref(ms)))
        return mc.value, ms.value

    def max_core_truss(self) -> dict:
        """Maximal core of the whole graph + trussness of its edges, the dict of Graph.max_core_truss on every rank
        (kombgpu_dist_max_core_truss).  Collective."""
        nc, mc, tm, nt = c_uint32(), c_uint64(), c_int32(), c_uint32()
        self._ctx._check(self._lib.kombgpu_dist_max_core_truss(self._h, byref(nc), byref(mc), byref(tm), byref(nt)))
        u, v, tr = np.empty(mc.value, np.uint32), np.empty(mc.value, np.uint32), np.empty(mc.value, np.int32)
        self._ctx._check(self._lib.kombgpu_dist_max_core_edges(self._h, c_void_p(u.ctypes.data), c_void_p(v.ctypes.data),
                                                               c_void_p(tr.ctypes.data)))
        tv = np.empty(nt.value, np.uint32)
        self._ctx._check(self._lib.kombgpu_dist_truss_vertices(self._h, c_void_p(tv.ctypes.data)))
        return {"n_core_vertices": nc.value, "n_core_edges": mc.value, "max_trussness": tm.value, "u": u, "v": v, "trussness": tr,
                "truss_vertices": tv}

    def truss_timing(self) -> dict:
        """CUDA-event split of this rank's last max_core_truss() in ms (measurement aid, include/kombgpu_debug.h)."""
        a, b, c = c_float(), c_float(), c_float()
        self._ctx._check(self._lib.kombgpu_debug_dist_truss_timing(self._h, byref(a), byref(b), byref(c)))
        return {"ms_core_gather": a.value, "ms_slice_gather": b.value, "ms_truss": c.value}

    def densest_core(self) -> dict:
        """Densest k-core of the whole graph, the dict of Graph.densest_core on every rank (kombgpu_dist_densest_core).
        Collective."""
        k, nv, ne, d = c_int32(), c_uint32(), c_uint64(), c_double()
        self._ctx._check(self._lib.kombgpu_dist_densest_core(self._h, byref(k), byref(nv), byref(ne), byref(d)))
        return {"k": k.value, "n_vertices": nv.value, "n_edges": ne.value, "density": d.value}

    def densest_block(self, weight=None, use_scores: bool = False, eps: float = 0.5) -> dict:
        """Densest block of the whole graph by the bulk greedy peel, the dict of Graph.densest_block on every rank
        (kombgpu_dist_densest_block).  `weight` and the returned `member` are this rank's slice: unitigs
        [v_lo, v_lo + n_local).  Collective."""
        st = self.stats()
        n = st["n_local"]
        wt = np.ascontiguousarray(weight, dtype=np.float64) if weight is not None else None
        if wt is not None and wt.shape != (n,):
            raise ValueError("weight must hold one value per unitig of this rank")
        nv, ne, ws, d, np_ = c_uint32(), c_uint64(), c_double(), c_double(), c_uint32()
        member = np.zeros(n, np.uint8)
        self._ctx._check(self._lib.kombgpu_dist_densest_block(self._h, c_void_p(wt.ctypes.data) if wt is not None else None,
                                                              int(bool(use_scores)), float(eps), byref(nv), byref(ne), byref(ws),
                                                              byref(d), byref(np_), c_void_p(member.ctypes.data)))
        return {"n_vertices": nv.value, "n_edges": ne.value, "weight_sum": ws.value, "density": d.value, "passes": np_.value,
                "member": member.astype(bool), "v_lo": st["v_lo"]}

    def onion(self, again: bool = False) -> dict:
        """Onion layers over the ranks (kombgpu_dist_onion): `layer` is this rank's slice, the 1-based layer of unitigs
        [v_lo, v_lo + n_local); the slices of ranks 0, 1, ... concatenate to Graph.onion()["layer"] on one GPU, and
        `n_layers` is the number of layers of the whole graph.  The first call is collective and the result is cached;
        again=True runs it again (collective; measurement aid)."""
        n = self.stats()["n_local"]
        if again:
            self._ctx._check(self._lib.kombgpu_debug_dist_onion_again(self._h))
        layer, nl = np.empty(n, np.uint32), c_uint32()
        self._ctx._check(self._lib.kombgpu_dist_onion(self._h, c_void_p(layer.ctypes.data) if n else None, byref(nl)))
        return {"layer": layer, "n_layers": nl.value, "v_lo": self.stats()["v_lo"]}

    def onion_timing(self) -> dict:
        """What this rank's last onion run measured (measurement aid, include/kombgpu_debug.h): kernel time from CUDA
        events, non-empty levels, meetings of all ranks, walk steps run on one CTA, and the time of the by-neighbour
        layout built from rows (0.0 when the build left that layout)."""
        ms, lv, mt, so, tr = c_float(), c_uint32(), c_uint32(), c_uint32(), c_float()
        self._ctx._check(self._lib.kombgpu_debug_dist_onion_timing(self._h, byref(ms), byref(lv), byref(mt), byref(so), byref(tr)))
        return {"ms_kernel": ms.value, "levels": lv.value, "meetings": mt.value, "solo_steps": so.value, "ms_transpose": tr.value}

    FILE_EDGELIST, FILE_KCORE, FILE_COREA, FILE_ONION = 0, 1, 2, 3

    def format(self, which: int, hits: "DistHits | None" = None) -> bytes:
        """This rank's slice of edgelist.txt / kcore.tsv / CoreA_anomaly.txt / onion.tsv, formatted on its device
        (kombgpu_dist_graph_format): the slices of ranks 0, 1, ... concatenate to Graph.format on one GPU.  kcore.tsv
        and onion.tsv take the unitig names from the DistHits the graph was built from.  Local, not collective."""
        n = c_uint64()
        self._ctx._check(self._lib.kombgpu_dist_graph_format(self._h, int(which), hits._h if hits is not None else None, byref(n)))
        buf = ctypes.create_string_buffer(max(n.value, 1))
        self._ctx._check(self._lib.kombgpu_dist_graph_format_fetch(self._h, int(which), buf, 0))
        return buf.raw[:n.value]

    def anomalous(self, whisker: float = 1.5) -> dict:
        """IQR fence on the CORE-A scores of all ranks, the dict of Graph.anomalous on every rank
        (kombgpu_dist_anomalous; needs corea() first).  `member` is this rank's slice: unitigs [v_lo, v_lo + n_local).
        Collective."""
        st = self.stats()
        member = np.zeros(st["n_local"], np.uint8)
        q1, q3, fence, ns = c_double(), c_double(), c_double(), c_uint32()
        self._ctx._check(self._lib.kombgpu_dist_anomalous(self._h, float(whisker), byref(q1), byref(q3), byref(fence), byref(ns),
                                                          c_void_p(member.ctypes.data)))
        return {"q1": q1.value, "q3": q3.value, "fence": fence.value, "n_selected": ns.value, "member": member.astype(bool),
                "v_lo": st["v_lo"]}

    def results(self, out: dict | None = None) -> dict:
        """degree / coreness / score of the local unitigs [v_lo, v_lo + n_local) on the host."""
        st = self.stats()
        n = st["n_local"]
        out = out or {}
        r = {"degree": out.get("degree", np.empty(n, np.int32))[:n], "coreness": out.get("coreness", np.empty(n, np.int32))[:n],
             "score": out.get("score", np.empty(n, np.float64))[:n]}
        if any(a.shape[0] != n for a in r.values()):
            raise ValueError("out= buffers are too small for this rank's unitigs")
        self._ctx._check(self._lib.kombgpu_dist_graph_results(self._h, c_void_p(r["degree"].ctypes.data), c_void_p(r["coreness"].ctypes.data),
                                                              c_void_p(r["score"].ctypes.data)))
        r["v_lo"] = st["v_lo"]
        return r

    def edges(self, with_mult: bool = False):
        """This rank's slice of the canonical edge list (u, v[, mult])."""
        m = self.stats()["n_fwd_local"]
        u, v = np.empty(m, np.uint32), np.empty(m, np.uint32)
        mult = np.empty(m, np.uint32) if with_mult else None
        self._ctx._check(self._lib.kombgpu_dist_graph_edges(self._h, c_void_p(u.ctypes.data), c_void_p(v.ctypes.data),
                                                            c_void_p(mult.ctypes.data) if with_mult else None))
        return (u, v, mult) if with_mult else (u, v)

    def edges_csr(self, out: dict | None = None):
        """This rank's slice of the edge list as (fwd_ptr uint64[n_local+1], v uint32[n_fwd_local])."""
        st = self.stats()
        out = out or {}
        fp = out.get("fwd_ptr", np.empty(st["n_local"] + 1, np.uint64))[:st["n_local"] + 1]
        v = out.get("v", np.empty(st["n_fwd_local"], np.uint32))[:st["n_fwd_local"]]
        if fp.shape[0] != st["n_local"] + 1 or v.shape[0] != st["n_fwd_local"]:
            raise ValueError("out= buffers are too small for this rank's slice of the edge list")
        self._ctx._check(self._lib.kombgpu_dist_graph_edges_csr(self._h, c_void_p(fp.ctypes.data), c_void_p(v.ctypes.data)))
        return fp, v

    def device_arrays(self) -> dict:
        ptrs = [c_void_p() for _ in range(6)]
        self._ctx._check(self._lib.kombgpu_dist_graph_device_arrays(self._h, *[byref(p) for p in ptrs]))
        names = ["row_ptr", "col", "edges_packed", "degree", "coreness", "score"]
        return {k: (p.value or 0) for k, p in zip(names, ptrs)}

    def close(self):
        if getattr(self, "_h", None):
            self._lib.kombgpu_dist_graph_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class DistHits:
    """kombgpu_dist_hits: SAM text parsed and interned over the ranks.  This rank holds the hits of its own reads
    (global unitig ids, read ids unique over the ranks) and the names of the unitigs it owns."""

    def __init__(self, comm: Comm, handle: c_void_p, texts):
        self.comm = comm
        self._ctx = comm.ctx
        self._lib = comm._lib
        self._h = handle
        self._texts = texts

    @classmethod
    def parse(cls, comm: Comm, texts) -> "DistHits":
        """SAM bytes of the mate files (mate 1 first), the same on every rank (kombgpu_dist_sam_parse).  Collective."""
        texts = [bytes(t) for t in texts]
        n = len(texts)
        arr = (ctypes.c_char_p * max(n, 1))(*texts)
        sizes = (c_uint64 * max(n, 1))(*[len(t) for t in texts])
        h = c_void_p()
        comm.ctx._check(comm._lib.kombgpu_dist_sam_parse(comm._h, arr, sizes, n, byref(h)))
        return cls(comm, h, texts)

    def counts(self) -> dict:
        hl, hg, nr, nu, nl = c_uint64(), c_uint64(), c_uint32(), c_uint32(), c_uint64()
        self._ctx._check(self._lib.kombgpu_dist_hits_counts(self._h, byref(hl), byref(hg), byref(nr), byref(nu), byref(nl)))
        return {"n_hits_local": hl.value, "n_hits": hg.value, "n_reads": nr.value, "n_unitigs": nu.value, "n_lines": nl.value}

    def local_range(self) -> tuple[int, int]:
        """(v_lo, n_local) of this rank in the unitig-range partition (step = ceil(n_unitigs / world))."""
        n = self.counts()["n_unitigs"]
        step = -(-n // self.comm.world) if n else 1
        lo = min(n, self.comm.rank * step)
        return lo, min(n, lo + step) - lo

    def names(self) -> list[bytes]:
        """Names of the unitigs this rank owns, [v_lo, v_lo + n_local), cut out of the input bytes."""
        _, n = self.local_range()
        f, off, ln = np.empty(n, np.uint32), np.empty(n, np.uint64), np.empty(n, np.uint32)
        self._ctx._check(self._lib.kombgpu_dist_hits_names(self._h, c_void_p(f.ctypes.data), c_void_p(off.ctypes.data),
                                                           c_void_p(ln.ctypes.data)))
        return [self._texts[int(f[i])][int(off[i]):int(off[i]) + int(ln[i])] for i in range(n)]

    def hits(self) -> tuple[np.ndarray, np.ndarray]:
        """This rank's routed hits (read id, unitig id) on the host."""
        n = self.counts()["n_hits_local"]
        rk, ut = np.empty(n, np.uint32), np.empty(n, np.uint32)
        self._ctx._check(self._lib.kombgpu_dist_hits_download(self._h, c_void_p(rk.ctypes.data), c_void_p(ut.ctypes.data)))
        return rk, ut

    def timing(self) -> dict:
        a, b, c, d, r = c_float(), c_float(), c_float(), c_float(), c_int()
        self._ctx._check(self._lib.kombgpu_dist_hits_timing(self._h, byref(a), byref(b), byref(c), byref(d), byref(r)))
        return {"ms_upload": a.value, "ms_parse": b.value, "ms_intern": c.value, "ms_route": d.value, "hash_rounds": r.value}

    def close(self):
        if getattr(self, "_h", None):
            self._lib.kombgpu_dist_hits_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class DistFasta:
    """kombgpu_dist_fasta: a FASTA file indexed over the ranks, each holding its slice of the records; the mirror of
    Fasta.  join() and extract() work on this rank's vertices, and the extraction slices of ranks 0, 1, ... concatenate
    to Fasta.extract on one GPU."""

    def __init__(self, comm: Comm, handle: c_void_p):
        self.comm = comm
        self._ctx = comm.ctx
        self._lib = comm._lib
        self._h = handle

    @classmethod
    def load(cls, comm: Comm, text: bytes) -> "DistFasta":
        """The bytes of one FASTA file, the same on every rank (kombgpu_dist_fasta_load).  Collective."""
        text = bytes(text)
        h = c_void_p()
        comm.ctx._check(comm._lib.kombgpu_dist_fasta_load(comm._h, text, len(text), byref(h)))
        return cls(comm, h)

    def counts(self) -> dict:
        nl, ng, rl, bl, bh = c_uint32(), c_uint32(), c_uint32(), c_uint64(), c_uint64()
        self._ctx._check(self._lib.kombgpu_dist_fasta_counts(self._h, byref(nl), byref(ng), byref(rl), byref(bl), byref(bh)))
        return {"n_records_local": nl.value, "n_records": ng.value, "rec_lo": rl.value, "byte_lo": bl.value, "byte_hi": bh.value}

    def join(self, hits: "DistHits | None" = None, names=None) -> int:
        """vertex -> record by name for this rank's vertices: the names `hits` holds for the unitigs this rank owns, or a
        host list of this rank's names (bytes).  Returns the vertices without a record over all ranks.  Collective."""
        if (hits is None) == (names is None):
            raise ValueError("pass exactly one of hits= and names=")
        miss = c_uint32()
        if hits is not None:
            self._ctx._check(self._lib.kombgpu_dist_fasta_join_hits(self._h, hits._h, byref(miss)))
        else:
            names = [bytes(x) for x in names]
            off = np.zeros(len(names) + 1, np.uint64)
            np.cumsum([len(x) for x in names], out=off[1:])
            self._ctx._check(self._lib.kombgpu_dist_fasta_join_names(self._h, b"".join(names), c_void_p(off.ctypes.data), len(names),
                                                                     byref(miss)))
        return miss.value

    def extract(self, mask) -> bytes:
        """This rank's slice of the records of the selected vertices; `mask` covers this rank's vertices.  Collective."""
        m = np.ascontiguousarray(np.asarray(mask).astype(bool).astype(np.uint8))
        n = c_uint64()
        self._ctx._check(self._lib.kombgpu_dist_fasta_extract(self._h, c_void_p(m.ctypes.data), m.shape[0], byref(n)))
        buf = ctypes.create_string_buffer(max(n.value, 1))
        self._ctx._check(self._lib.kombgpu_dist_fasta_extract_fetch(self._h, buf))
        return buf.raw[:n.value]

    def timing(self) -> dict:
        up, ix, jn, ex, l = c_float(), c_float(), c_float(), c_float(), c_uint64()
        self._ctx._check(self._lib.kombgpu_dist_fasta_timing(self._h, byref(up), byref(ix), byref(jn), byref(ex), byref(l)))
        return {"ms_upload": up.value, "ms_index": ix.value, "ms_join": jn.value, "ms_extract": ex.value, "kernel_launches": l.value}

    def close(self):
        if getattr(self, "_h", None):
            self._lib.kombgpu_dist_fasta_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def run_local(world: int, fn, devices=None, heap_bytes: int = 0):
    """Run `fn(comm) -> result` on `world` ranks inside this process, one host thread per rank (ctypes releases the
    GIL inside the library).  devices=None puts every rank on device 0: the emulation mode for one-GPU boxes."""
    devices = list(devices) if devices is not None else [0] * world
    assert len(devices) == world
    slot = c_void_p(None)
    results, errors = [None] * world, [None] * world

    def worker(rank):
        ctx = comm = None
        try:
            ctx = Context(devices[rank])
            comm = Comm.create_local(ctx, rank, world, slot, heap_bytes)
            results[rank] = fn(comm)
        except BaseException as e:   # noqa: BLE001 - reported to the caller below
            errors[rank] = e
            if comm is not None:
                comm._lib.kombgpu_comm_abort(comm._h)   # the other ranks must not wait for this one
        finally:
            if comm is not None:
                comm.close()
            if ctx is not None:
                ctx.close()

    threads = [threading.Thread(target=worker, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for e in errors:
        if e is not None:
            raise e
    return results
