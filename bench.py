#!/usr/bin/env python
"""bench.py — throughput of the KOMB hot path (hits -> graph -> k-core -> CORE-A).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--no-configs] [--no-cpu-baseline]
                    [--dump-outputs DIR]
    (KOMB_BENCH_ONLY_CONFIG=cfg3|cfg4_eighth|cfg4|cfg5 at N > 1: run the step and only that secondary config)

One "step" = one pass of the whole hot path over one synthetic batch (BASELINE.json configs[1]: 1 M unitigs,
5 M read pairs, ~20 M hits per GPU).  N = 1 runs the single-GPU path; N > 1 (launched with torch.distributed.run,
one rank per GPU) runs the peer-memory multi-GPU path of libkombgpu (komb_b200/peer.py): the graph partitioned by
unitig-id range, ranks talking through NVLink peer memory.  Prints ONE JSON line (rank 0).  Besides the headline
workload the line carries, under `configs`, the other BASELINE configs that fit the run (cfg3 / cfg5 on one GPU;
cfg3 strong-scaled and cfg4 on N GPUs) and, under `parity`, what was checked inside this very run.
See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_UNITIGS = 1_000_000
N_READ_PAIRS = 5_000_000
SEED = 11
CPU_SAMPLE_READ_PAIRS = 312_500          # 1/16 of the workload's reads: the ONE sample both CPU legs use (~3.5 s per run)
METRIC = "hot-path hits/s (graph build + k-core peel + CORE-A), with peel edges/s and build hits/s"
DTYPE = "u32/u64 ids, f64 scores"


PEEL_KINDS = {0: "log", 1: "async", 2: "replicated"}


def workload_config(world: int) -> dict:
    """The `config` object: identical for our arm and the reference arm (the driver compares them)."""
    return {"workload": "cfg2: synthetic metagenome unitig graph, 1M unitigs, 5M read pairs (~20M hits) per GPU"
                        + ("" if world == 1 else f", x{world} GPUs (weak scaling; unitig ids scrambled, graph partitioned by unitig-id range)"),
            "n_unitigs_per_gpu": N_UNITIGS, "n_read_pairs_per_gpu": N_READ_PAIRS, "seed": SEED, "corea_key": "ref32",
            "l2": "256 MB flush between timed steps; inputs (160 MB per GPU) exceed L2"}


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.idx = device_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 8:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for nm, val in zip(names, r[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation (oracle/_ref/komb2_ref = reference sources compiled
# unmodified against oracle/igraph_shim), else the oracle port.  Runs on a bounded sample of the same workload.
# ---------------------------------------------------------------------------

def _komb2_run(binary, d: Path, outdir: Path, threads: int, env=None):
    outdir.mkdir(exist_ok=True)
    t0 = time.perf_counter()
    cp = subprocess.run([str(binary), "-t", str(threads), "-l", "100", "-o", str(outdir), "-i", str(d / "r1.sam"),
                         "-j", str(d / "r2.sam"), "-u", str(d / "u.fasta")], capture_output=True, text=True, env=env)
    wall = time.perf_counter() - t0
    if cp.returncode != 0:
        raise RuntimeError(f"{binary} failed: {cp.stderr[-400:]}")
    return cp, wall


def cpu_reference_run(n_unitigs: int, sample_read_pairs: int, seed: int, threads: int, dropin: bool = False, ctx=None) -> dict:
    from komb_b200 import synth
    from oracle import oracle
    m1, m2 = synth.metagenome_hits(n_unitigs, sample_read_pairs, seed=seed)
    n_hits = m1.n_hits + m2.n_hits
    sample = (f"{sample_read_pairs} of {N_READ_PAIRS} read pairs ({n_hits} hits) over the same "
              f"{n_unitigs} unitigs, seed {seed}")
    if oracle.REF_KOMB2.exists():
        with tempfile.TemporaryDirectory() as d:
            d = Path(d)
            (d / "r1.sam").write_bytes(synth.render_sam(m1, n_unitigs, 1, with_header=False))
            (d / "r2.sam").write_bytes(synth.render_sam(m2, n_unitigs, 2, with_header=False))
            synth.write_fasta(str(d / "u.fasta"), 4)
            cp, wall = _komb2_run(oracle.REF_KOMB2, d, d / "out", threads)
            drop = None
            tok = None
            if ctx is not None:
                # the device tokeniser (kombgpu_sam_parse) on the same SAM text: bytes in, integer hits on the device
                texts = [(d / "r1.sam").read_bytes(), (d / "r2.sam").read_bytes()]
                best = None
                for _ in range(3):
                    with ctx.sam_parse(texts) as hits:
                        c, tm = hits.counts(), hits.timing()
                        if best is None or tm["ms_parse"] < best["ms_parse"]:
                            best = dict(tm, **c)
                nbytes = sum(len(t) for t in texts)
                tok = {"sam_bytes": nbytes, "n_hits": best["n_hits"], "n_lines": best["n_lines"], "ms_upload_pageable": best["ms_upload"],
                       "ms_parse_and_intern": best["ms_parse"], "kernel_launches": best["kernel_launches"],
                       "parse_gb_per_s": nbytes / (best["ms_parse"] * 1e-3) / 1e9, "parse_hits_per_s": best["n_hits"] / (best["ms_parse"] * 1e-3),
                       "hits_equal_generator": bool(best["n_hits"] == n_hits),
                       "cpu_reading_sams_s": None}
            if dropin and (ROOT / "bin" / "komb2").exists():
                # the drop-in executable on the SAME SAM pair: like for like (text in, three files out)
                env = dict(os.environ, KOMB_TIMING="1")
                walls, ctx_s, after_s = [], [], []
                for _ in range(3):
                    cpd, w = _komb2_run(ROOT / "bin" / "komb2", d, d / "out_gpu", threads, env)
                    walls.append(w)
                    m = re.search(r"kombgpu_ctx_create \(joined\)\s+\+([0-9.]+) s \(at ([0-9.]+) s\)", cpd.stderr)
                    ctx_s.append(float(m.group(2)) if m else None)
                    ends = re.findall(r"\(at ([0-9.]+) s\)", cpd.stderr)
                    after_s.append(float(ends[-1]) - float(m.group(2)) if m and ends else None)
                # the same executable with the host tokeniser / host writers (KOMB_TOKENIZE=host): the round-1 path
                _, wall_host_tok = _komb2_run(ROOT / "bin" / "komb2", d, d / "out_gpu_host", threads, dict(env, KOMB_TOKENIZE="host"))
                # parity target is the reference at -t 1 (at -t > 1 it silently drops SAM lines: SURVEY quirk Q1)
                _, wall_t1 = _komb2_run(oracle.REF_KOMB2, d, d / "out_t1", 1)
                ref_out, our_out = oracle.read_outputs(d / "out_t1"), oracle.read_outputs(d / "out_gpu")
                same = (ref_out["kcore"] == our_out["kcore"] and ref_out["edges"] == our_out["edges"]
                        and all(abs(ref_out["score"][k] - our_out["score"][k]) <= 1e-6 * max(1.0, abs(ref_out["score"][k])) + 1e-6
                                for k in ref_out["score"]))
                drop = {"komb2_wall_s": walls, "device_ready_at_s": ctx_s, "work_after_context_s": after_s,
                        "komb2_host_tokeniser_wall_s": wall_host_tok, "komb2_ref_wall_s": wall, "komb2_ref_t1_wall_s": wall_t1,
                        "threads": threads,
                        "speedup_wall": wall / min(walls), "outputs_equal_by_name": bool(same),
                        "note": "bin/komb2 vs komb2_ref on the same SAM pair; wall clock of the whole process including CUDA context "
                                "creation (device_ready_at_s: when the context was usable; work_after_context_s: SAM text to "
                                "the three files once the device is up -- tokenised, interned and formatted on the device)"}
        stages = {m.group(1).strip(): float(m.group(2))
                  for m in re.finditer(r"Time elapsed (?:for|doing) ([^:]+): ([0-9.]+) s", cp.stdout)}
        total = stages.get("KOMB", wall)          # komb2's own end-to-end timer (komb2.cpp:141-143)
        edges = int(re.search(r"Number of edges: (\d+)", cp.stdout).group(1))
        kcore_s = stages.get("K-core decomposition")
        return {"value": n_hits / total, "unit": "hits/s", "cores": threads, "kind": "reference",
                "sample": sample + f"; komb2_ref -t {threads} from SAM text, {total:.2f} s (igraph stages are the shim's)",
                "seconds": total, "n_hits": n_hits, "n_edges": edges,
                "peel_edges_per_s": (edges / kcore_s) if kcore_s else None,
                "stage_seconds": stages, "dropin": drop,
                "tokenise": dict(tok, cpu_reading_sams_s=stages.get("reading SAMs")) if tok else None}
    # port: the C restatement (single thread)
    rk = np.concatenate([m1.read_key, m2.read_key]); ut = np.concatenate([m1.unitig, m2.unitig])
    t0 = time.perf_counter()
    edges, _, _ = oracle.build_edges(rk, ut)
    t1 = time.perf_counter()
    deg, core = oracle.coreness(n_unitigs, edges)
    t2 = time.perf_counter()
    oracle.corea(core, deg, oracle.KEY_REF32)
    t3 = time.perf_counter()
    return {"value": n_hits / (t3 - t0), "unit": "hits/s", "cores": 1, "kind": "port",
            "sample": sample + "; oracle/komb_oracle.c from integer hits (no SAM parsing)",
            "seconds": t3 - t0, "n_hits": n_hits, "n_edges": int(edges.shape[0]),
            "peel_edges_per_s": edges.shape[0] / (t2 - t1), "stage_seconds": {"build": t1 - t0, "peel": t2 - t1, "corea": t3 - t2},
            "dropin": None, "tokenise": None}


def cpu_stage_samples(core: np.ndarray, deg: np.ndarray, hbm_note: str = "") -> dict:
    """SURVEY 8(d) "CPU reference timing" for the stages komb2's own timers do not isolate: igraph's single-threaded
    create/simplify/coreness on an R-MAT sample (the BZ port: the shim's igraph_coreness is the same algorithm), and
    CoreA::getAnomalyScore straight from the reference's CoreA.h, which is O(n x distinct keys): timed at n <= 10^6 and
    extrapolated above, next to an O(n log n) restatement."""
    from oracle import oracle
    import torch
    out = {}
    n = int(core.shape[0])
    n_keys = int(np.unique(core.astype(np.int64) * n + deg).shape[0])
    t0 = time.perf_counter()
    oracle.corea(core, deg, oracle.KEY_REF32)
    t_port = time.perf_counter() - t0
    out["corea"] = {"n": n, "distinct_keys": n_keys, "port_nlogn_s": t_port, "port_vertices_per_s": n / t_port}
    if oracle.REF_COREA.exists():
        with tempfile.TemporaryDirectory() as d:
            m = min(n, 1_000_000)
            t0 = time.perf_counter()
            oracle.corea_reference(core[:m], deg[:m], d)
            t_ref = time.perf_counter() - t0
        out["corea"].update({"reference_coreA_h_n": m, "reference_coreA_h_s": t_ref, "reference_vertices_per_s": m / t_ref,
                             "reference_note": "CoreA.h fractionalRank is O(n x distinct keys): cfg3 (50 M unitigs, ~10^6 distinct "
                                               "keys) is DNF on the CPU (extrapolated: > 10^4 x this time); the O(n log n) port is the "
                                               "fair CPU number"})
    # igraph create + simplify + coreness, single thread, on an R-MAT sample of cfg3's generator (scale 22 -> 2.5 M unitigs)
    u, v = rmat_device(22, 40_000_000, 2_500_000, 42)
    uh, vh = u.cpu().numpy().view(np.uint32), v.cpu().numpy().view(np.uint32)
    del u, v
    torch.cuda.empty_cache()
    t0 = time.perf_counter()
    edges = oracle.simplify(uh, vh)
    t1 = time.perf_counter()
    oracle.coreness(2_500_000, edges)
    t2 = time.perf_counter()
    E = int(edges.shape[0])
    out["rmat_sample"] = {"workload": "R-MAT scale 22, 40 M draws over 2.5 M unitigs (cfg3's generator at 1/13 size), one thread",
                          "n_edges": E, "simplify_s": t1 - t0, "coreness_bz_s": t2 - t1, "build_edges_per_s": E / (t1 - t0),
                          "peel_edges_per_s": E / (t2 - t1)}
    return out


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    vals = []
    last = None
    for i in range(args.warmup + args.steps):
        r = cpu_reference_run(N_UNITIGS, CPU_SAMPLE_READ_PAIRS, SEED, threads)
        if i >= args.warmup:
            vals.append(r)
        last = r
    v = float(np.mean([r["value"] for r in vals])) if vals else last["value"]
    secs = float(np.mean([r["seconds"] for r in vals])) if vals else last["seconds"]
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "hits/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {k: last[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": v, "unit": "hits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "peel_edges_per_s": last.get("peel_edges_per_s"),
        "stage_seconds": last.get("stage_seconds"),
    }
    line["cpu_baseline"]["value"] = v
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------
# device-side helpers (torch is the checker here, never the path)
# ---------------------------------------------------------------------------

def dev_view(ptr: int, count: int, typestr: str, owner, device):
    import torch
    from komb_b200.distributed import _DevArray
    if count == 0 or not ptr:
        return torch.zeros(0, dtype={"<i4": torch.int32, "<i8": torch.int64, "<f8": torch.float64}[typestr], device=device)
    return torch.as_tensor(_DevArray(ptr, count, typestr, owner), device=device)


def rmat_device(scale, draws, n, seed, chunk=1 << 26):
    """R-MAT (0.57, 0.19, 0.19, 0.05) draws generated on the device, ids scrambled and folded mod n (SURVEY 8(d) cfg3)."""
    import torch
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    us, vs = [], []
    a, b, c = 0.57, 0.19, 0.19
    for s0 in range(0, draws, chunk):
        m = min(chunk, draws - s0)
        u = torch.zeros(m, dtype=torch.int64, device="cuda"); v = torch.zeros_like(u)
        for _ in range(scale):
            r = torch.rand(m, device="cuda", generator=g)
            ub = (r >= a + b).to(torch.int64)
            vb = (((r >= a) & (r < a + b)) | (r >= a + b + c)).to(torch.int64)
            u = (u << 1) | ub; v = (v << 1) | vb

        def scr(x):
            x = (x ^ (x >> 16)) & 0xFFFFFFFF; x = (x * 0x7FEB352D) & 0xFFFFFFFF
            x = (x ^ (x >> 15)) & 0xFFFFFFFF; x = (x * 0x846CA68B) & 0xFFFFFFFF
            return (x ^ (x >> 16)) & 0xFFFFFFFF
        us.append((scr(u) % n).to(torch.int32)); vs.append((scr(v) % n).to(torch.int32))
    return torch.cat(us), torch.cat(vs)


def ramp_device(levels, per, n_bg, bg_scale, bg_edges, seed):
    """cfg5: planted ramp (levels x per vertices, level j adjacent to the next c(j)) over an R-MAT background."""
    import torch
    L = levels * per
    j = torch.arange(L, dtype=torch.int64, device="cuda"); c = 1 + j // per
    us, vs = [], []
    for d in range(1, levels + 1):
        sel = j[(c >= d) & (j + d < L)]
        us.append(sel); vs.append(sel + d)
    t = torch.arange(L - (levels + 1), L, dtype=torch.int64, device="cuda")
    iu = torch.triu_indices(levels + 1, levels + 1, 1, device="cuda")
    us.append(t[iu[0]]); vs.append(t[iu[1]])
    u = torch.cat(us) + n_bg; v = torch.cat(vs) + n_bg
    if bg_edges:
        bu, bv = rmat_device(bg_scale, bg_edges, n_bg, seed)
        u = torch.cat([u, bu.to(torch.int64)]); v = torch.cat([v, bv.to(torch.int64)])
    n = n_bg + L
    a = 2654435761
    while np.gcd(a, n) != 1:
        a += 2
    f = lambda x: ((x * a + 12345) % n).to(torch.int32)   # noqa: E731 - fixed bijection: a range partition stays balanced
    return f(u), f(v), n


def cfg4_hits_device(n, r_lo, r_cnt, p, seed, chunk=1 << 25):
    """cfg4: hits of read pairs [r_lo, r_lo + r_cnt): centre ~ scrambled power law, hits at centre + Geometric(p) - 1."""
    import torch
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    a = 2654435761
    while np.gcd(a, n) != 1:
        a += 2
    ks = torch.tensor([1, 1, 2, 2, 2, 3, 3], device="cuda")
    centre = torch.empty(r_cnt, dtype=torch.int64, device="cuda")
    for s0 in range(0, r_cnt, chunk):
        m = min(chunk, r_cnt - s0)
        x = torch.rand(m, device="cuda", generator=g, dtype=torch.float64)
        c = torch.clamp((n * x * x).to(torch.int64), max=n - 1)
        centre[s0:s0 + m] = (c * a + 12345) % n
    mates = []
    for _ in range(2):
        rk_parts, ut_parts = [], []
        for s0 in range(0, r_cnt, chunk):
            m = min(chunk, r_cnt - s0)
            k = ks[torch.randint(0, 7, (m,), device="cuda", generator=g)]
            reads = torch.repeat_interleave(torch.arange(s0, s0 + m, device="cuda"), k)
            off = torch.empty(reads.numel(), device="cuda").geometric_(p, generator=g).to(torch.int64) - 1
            ut_parts.append(((centre[reads] + off) % n).to(torch.int32))
            rk_parts.append((reads + r_lo).to(torch.int32))
        mates.append((torch.cat(rk_parts), torch.cat(ut_parts)))
    return torch.cat([mates[0][0], mates[1][0]]), torch.cat([mates[0][1], mates[1][1]])


DUMP_SAMPLE = 1 << 20      # entries of one output written whole; a longer output is written as a seeded sample


def dump_outputs(out_dir: str, r: dict) -> None:
    """--dump-outputs: what the last timed step hands its caller (kombgpu_graph_results: canonical edge list, degree,
    coreness, CORE-A score) as float64 .npy files, so that two builds can be compared output for output.  An output
    longer than DUMP_SAMPLE entries is written at DUMP_SAMPLE positions drawn with a fixed seed from its length;
    vertex_index.npy / edge_index.npy hold the positions written.  counts.npy = [n_vertices, n_edges]."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)

    def positions(count: int) -> np.ndarray:
        if count <= DUMP_SAMPLE:
            return np.arange(count, dtype=np.int64)
        return np.sort(np.random.default_rng(0).choice(count, DUMP_SAMPLE, replace=False))

    n, E = r["degree"].shape[0], r["u"].shape[0]
    vi, ei = positions(n), positions(E)
    arrays = {"counts": np.array([n, E]), "vertex_index": vi, "edge_index": ei,
              "degree": r["degree"][vi], "coreness": r["coreness"][vi], "score": r["score"][vi],
              "edges_u": r["u"][ei], "edges_v": r["v"][ei]}
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", a.astype(np.float64))   # ids and counts stay below 2^53: exact in float64


def certificate_single(core, col, deg, n, chunk=1 << 27):
    import torch
    ge = torch.zeros(n, dtype=torch.int32, device="cuda"); gt = torch.zeros(n, dtype=torch.int32, device="cuda")
    row_ptr = torch.zeros(n + 1, dtype=torch.int64, device="cuda"); torch.cumsum(deg.to(torch.int64), 0, out=row_ptr[1:])
    total = int(row_ptr[-1])
    for s0 in range(0, total, chunk):
        e = torch.arange(s0, min(total, s0 + chunk), device="cuda")
        src = torch.searchsorted(row_ptr, e, right=True) - 1
        cu = core[col[s0:s0 + e.numel()].to(torch.int64)]; cs = core[src]
        ge.index_add_(0, src, (cu >= cs).to(torch.int32)); gt.index_add_(0, src, (cu > cs).to(torch.int32))
    return bool((ge >= core).all()) and bool((gt <= core).all()) and bool((core <= deg).all())


def run_config_single(ctx, name: str, hbm_gbs: float, reps: int = 2) -> dict:
    """BASELINE cfg3 / cfg5 at full size on ONE GPU: stage times from the library's own CUDA events, sizes, the
    k-core certificate on the device."""
    import torch
    import komb_b200
    t0 = time.perf_counter()
    if name == "cfg3":
        u, v = rmat_device(26, 540_000_000, 50_000_000, 42); n = 50_000_000
        desc = "R-MAT scale 26, 540 M draws folded onto 50 M unitigs, seed 42"
    else:
        u, v, n = ramp_device(5000, 40, 9_800_000, 24, 40_000_000, 7)
        desc = "deep core: ramp of 5000 levels x 40 unitigs over an R-MAT background, 10 M unitigs, ids scrambled"
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    best = None
    g = None
    for _ in range(reps):
        if g is not None:
            g.close()
        g = ctx.graph_from_edges(u, v, n)
        g.analyse(komb_b200.KEY_EXACT64)
        st = g.stats()
        if best is None or st["ms_build"] + st["ms_peel"] + st["ms_corea"] < best["ms_build"] + best["ms_peel"] + best["ms_corea"]:
            best = st
    E = best["n_edges"]
    arr = g.device_arrays()
    core = dev_view(arr["coreness"], n, "<i4", g, "cuda"); deg = dev_view(arr["degree"], n, "<i4", g, "cuda")
    col = dev_view(arr["col"], 2 * E, "<i4", g, "cuda")
    cert = certificate_single(core, col, deg, n)
    g.close()
    del u, v
    torch.cuda.empty_cache()
    ctx.trim()
    b_peel, b_build, b_corea = 24 * E + 16 * n, 16 * best["n_pairs"] + 8 * E + 8 * (n + 1), 32 * n
    total_ms = best["ms_build"] + best["ms_peel"] + best["ms_corea"]
    return {"workload": f"{name}: {desc}, 1 GPU", "n_unitigs": n, "input_pairs": best["n_pairs"], "n_edges": E,
            "max_degree": best["max_degree"], "max_coreness": best["max_coreness"], "peel_levels": best["peel_levels"],
            "ms_build": best["ms_build"], "ms_peel": best["ms_peel"], "ms_peel_kernel": best["ms_peel_kernel"], "ms_corea": best["ms_corea"],
            "ms_total": total_ms, "edges_per_s_total": E / (total_ms * 1e-3),
            "peel_edges_per_s": E / (best["ms_peel"] * 1e-3), "peel_frac_hbm": b_peel / (best["ms_peel_kernel"] * 1e-3) / 1e9 / hbm_gbs,
            "build_edges_per_s": E / (best["ms_build"] * 1e-3), "build_frac_hbm": b_build / (best["ms_build"] * 1e-3) / 1e9 / hbm_gbs,
            "corea_frac_hbm": b_corea / (best["ms_corea"] * 1e-3) / 1e9 / hbm_gbs,
            "corea_key": "exact64", "kcore_certificate_on_device": cert, "generate_s": gen_s}


# ---------------------------------------------------------------------------
# our arm, one GPU
# ---------------------------------------------------------------------------

def run_ours(args):
    import torch
    import torch.distributed as dist

    import komb_b200
    from komb_b200 import synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"      # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        return run_ours_multi(args, rank, world, local_rank)

    hbm_gbs, peak_src = load_peaks()
    ctx = komb_b200.Context(local_rank)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)      # time on the stream the kernels are launched on

    # synthetic hits (host, pinned) and a device-resident copy
    m1, m2 = synth.metagenome_hits(N_UNITIGS, N_READ_PAIRS, seed=SEED)
    rk_h = torch.from_numpy(np.concatenate([m1.read_key, m2.read_key]).view(np.int32)).pin_memory()
    ut_h = torch.from_numpy(np.concatenate([m1.unitig, m2.unitig]).view(np.int32)).pin_memory()
    rk_d = rk_h.cuda(non_blocking=True)
    ut_d = ut_h.cuda(non_blocking=True)
    n_hits = rk_h.numel()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    torch.cuda.synchronize()

    def step_device(keep=False):
        g = ctx.build_graph(rk_d, ut_d, N_UNITIGS)
        g.analyse(komb_b200.KEY_REF32)
        st = g.stats()
        if keep:
            return st, g
        g.close()
        return st

    # page-locked result buffers, allocated once (as a long-running host would)
    e_cap = int(2.2 * n_hits)
    pin = {"fwd_ptr": ctx.pinned_empty(N_UNITIGS + 1, np.uint64), "v": ctx.pinned_empty(e_cap, np.uint32),
           "core": ctx.pinned_empty(N_UNITIGS, np.int32), "deg": ctx.pinned_empty(N_UNITIGS, np.int32),
           "score": ctx.pinned_empty(N_UNITIGS, np.float64)}

    def step_e2e():
        """The call a user of the C ABI makes: host hits in (page-locked), every output the komb2 host writes to its
        three files back on the host (page-locked); the edge list travels in CSR form (offsets + targets)."""
        g, r = ctx.analyse_hits_csr(rk_h.numpy().view(np.uint32), ut_h.numpy().view(np.uint32), N_UNITIGS, komb_b200.KEY_REF32,
                                    out={"fwd_ptr": pin["fwd_ptr"], "v": pin["v"], "degree": pin["deg"], "coreness": pin["core"],
                                         "score": pin["score"]})
        st = g.stats()
        g.close()
        return st, sum(a.nbytes for a in r.values()), r

    n_warm = 1 if args.profile else max(args.warmup, 3)
    for _ in range(n_warm):
        st = step_device()
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    stats = []
    last_graph = None
    torch.cuda.synchronize()
    for i in range(args.steps):
        flush.fill_(i & 0xff)                 # L2 flush between timed iterations (outside the events)
        torch.cuda.synchronize()
        ev[i][0].record(stream)
        if args.dump_outputs and i == args.steps - 1:
            # the last step's graph outlives its timed window so that its results can be written below
            st_last, last_graph = step_device(keep=True)
            stats.append(st_last)
        else:
            stats.append(step_device())
        ev[i][1].record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    if last_graph is not None:
        dump_outputs(args.dump_outputs, last_graph.results(komb_b200.KEY_REF32))
        last_graph.close()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    ms_per_step = float(np.mean(step_ms))
    st = stats[-1]
    H, P, E, n = st["n_hits"], st["n_pairs"], st["n_edges"], st["n_vertices"]

    ms_build = float(np.mean([s["ms_build"] for s in stats]))
    ms_peel = float(np.mean([s["ms_peel"] for s in stats]))
    ms_corea = float(np.mean([s["ms_corea"] for s in stats]))
    ms_peel_kernel = float(np.mean([s["ms_peel_kernel"] for s in stats]))

    if args.profile:
        print(json.dumps({"profile_run": True, "ms_per_step": ms_per_step, "launches_per_step": st["kernel_launches"],
                          "ms_build": ms_build, "ms_peel": ms_peel, "ms_corea": ms_corea,
                          "dumped_outputs": args.dump_outputs}), flush=True)
        ctx.close()
        return

    # e2e: host buffers, copies inside the timed region
    for _ in range(2):
        step_e2e()
    torch.cuda.synchronize()
    e2e_t = []
    d2h = 0
    r_e2e = None
    for _ in range(max(2, min(args.steps, 5))):
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, d2h, r_e2e = step_e2e()
        torch.cuda.synchronize()
        e2e_t.append(time.perf_counter() - t0)
    e2e_s = float(np.mean(e2e_t))

    # parity inside this run (size-independent; the oracle comparisons live in tests/): the host results of the e2e
    # call equal the device-resident run's, and the coreness passes the k-core certificate on the device
    _, g = step_device(keep=True)
    arr = g.device_arrays()
    core_d = dev_view(arr["coreness"], n, "<i4", g, "cuda"); deg_d = dev_view(arr["degree"], n, "<i4", g, "cuda")
    col_d = dev_view(arr["col"], 2 * E, "<i4", g, "cuda"); score_d = dev_view(arr["score"], n, "<f8", g, "cuda")
    edges_d = dev_view(arr["edges_packed"], E, "<i8", g, "cuda")
    parity = {
        "e2e_host_results_equal_device_run": bool(
            np.array_equal(r_e2e["coreness"], core_d.cpu().numpy()) and np.array_equal(r_e2e["degree"], deg_d.cpu().numpy())
            and np.array_equal(r_e2e["score"], score_d.cpu().numpy())
            and np.array_equal(r_e2e["v"], (edges_d & 0xFFFFFFFF).to(torch.int32).cpu().numpy().view(np.uint32))
            and int(r_e2e["fwd_ptr"][-1]) == E),
        "kcore_certificate_on_device": certificate_single(core_d, col_d, deg_d, n),
        "degree_sum_is_2E": int(deg_d.to(torch.int64).sum()) == 2 * E,
        "checked_against_oracle_in": "tests/test_gpu_parity.py::test_cfg2_full_size (same inputs, bit-exact) and __graft_entry__.smoke()",
    }
    g.close()

    # algorithmic bytes (DESIGN.md "Roofline"): SURVEY 8(d)
    b_peel = 24 * E + 16 * n
    b_build = 8 * H + 16 * P + 8 * E + 8 * (n + 1)
    b_corea = 32 * n
    peel_gbs = b_peel / (ms_peel_kernel * 1e-3) / 1e9
    line = {
        "metric": METRIC,
        "value": H / (ms_per_step * 1e-3),
        "unit": "hits/s",
        "n_gpus": 1, "steps": args.steps, "warmup": n_warm, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": DTYPE, "data": "synthetic",
        "config": workload_config(1),
        "workload_sizes": {"n_unitigs": n, "n_read_pairs": N_READ_PAIRS, "n_hits": H, "n_pairs": P, "n_edges": E,
                           "max_coreness": st["max_coreness"], "peel_levels": st["peel_levels"]},
        "stages": {
            "build": {"ms": ms_build, "hits_per_s": H / (ms_build * 1e-3), "algorithmic_bytes": b_build,
                      "gbs": b_build / (ms_build * 1e-3) / 1e9, "frac_hbm": b_build / (ms_build * 1e-3) / 1e9 / hbm_gbs},
            "peel": {"ms": ms_peel, "edges_per_s": E / (ms_peel * 1e-3), "algorithmic_bytes": b_peel,
                     "gbs": b_peel / (ms_peel * 1e-3) / 1e9, "frac_hbm": b_peel / (ms_peel * 1e-3) / 1e9 / hbm_gbs},
            "corea": {"ms": ms_corea, "vertices_per_s": n / (ms_corea * 1e-3), "algorithmic_bytes": b_corea,
                      "gbs": b_corea / (ms_corea * 1e-3) / 1e9, "frac_hbm": b_corea / (ms_corea * 1e-3) / 1e9 / hbm_gbs},
        },
        "peel_edges_per_s": E / (ms_peel * 1e-3),
        "build_hits_per_s": H / (ms_build * 1e-3),
        "roofline": {"kernel": "peel_kernel (persistent cooperative frontier peel, warp-autonomous process phase)", "bound": "hbm",
                     "achieved": peel_gbs, "peak": hbm_gbs, "unit": "GB/s", "frac": peel_gbs / hbm_gbs,
                     "traffic": 352.1e6, "traffic_source": "dram__bytes_read+write of one peel_kernel launch, ncu --set full "
                     "(profiles/r2/r2ar_peel_kernel_raw.csv: 320.9 MB read + 31.2 MB written; the 4 MB degree array stays in L2, so DRAM traffic is below "
                     "the algorithmic bytes; the kernel is bound by its dependency depth and by L2 atomics, not by bytes)",
                     "algorithmic_bytes": b_peel, "kernel_ms": ms_peel_kernel, "peak_source": peak_src},
        "e2e": {"value": H / e2e_s, "unit": "hits/s", "h2d_bytes_per_step": 8 * H, "d2h_bytes_per_step": int(d2h),
                "ms_per_step": e2e_s * 1e3, "edge_list_form": "csr (forward offsets u64[n+1] + targets u32[E])"},
        "gpu_launches": int(sum(s["kernel_launches"] for s in stats)),
        "parity": parity,
        "clocks": clocks,
        # set when the last timed step kept its graph past its end event (--dump-outputs): not like for like with a run
        # without the flag
        "dumped_outputs": args.dump_outputs,
    }
    del rk_d, ut_d
    if not args.no_configs:
        line["configs"] = {}
        for name in ("cfg3", "cfg5"):
            try:
                line["configs"][name] = run_config_single(ctx, name, hbm_gbs)
            except Exception as e:  # a secondary workload never costs the headline line
                line["configs"][name] = {"error": f"{type(e).__name__}: {e}"}
    if not args.no_cpu_baseline:
        try:
            cb = cpu_reference_run(N_UNITIGS, CPU_SAMPLE_READ_PAIRS, SEED, os.cpu_count() or 1, dropin=True, ctx=ctx)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
            line["cpu_baseline"]["peel_edges_per_s"] = cb.get("peel_edges_per_s")
            line["cpu_baseline"]["stage_seconds"] = cb.get("stage_seconds")
            line["dropin"] = cb.get("dropin")
            line["stages"]["tokenise"] = cb.get("tokenise")
            try:
                line["cpu_baseline"]["stage_samples"] = cpu_stage_samples(np.array(r_e2e["coreness"]), np.array(r_e2e["degree"]))
            except Exception as e:
                line["cpu_baseline"]["stage_samples"] = {"error": f"{type(e).__name__}: {e}"}
        except Exception as e:  # the baseline is a reported number, never a reason to lose the GPU line
            line["cpu_baseline"] = {"value": None, "unit": "hits/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
    print(json.dumps(line), flush=True)
    ctx.close()


# ---------------------------------------------------------------------------
# our arm, N GPUs: the peer-memory path
# ---------------------------------------------------------------------------

def verify_against_single_gpu(ctx, tcomm, dg, a_d, b_d, kind: str, n_global: int, key_mode: int) -> dict:
    """Parity inside the run: gather every rank's input (NCCL, checker plumbing), run the SINGLE-GPU path of the
    library on the whole input on this GPU, and compare this rank's share of the partitioned result with it:
    edge-list slice, degree and coreness bit-exact, CORE-A within 1e-6 and the global ranking identical."""
    import torch
    import torch.distributed as dist
    a_all, b_all = tcomm.all_gather_var(a_d), tcomm.all_gather_var(b_d)
    g1 = ctx.build_graph(a_all, b_all, n_global) if kind == "hits" else ctx.graph_from_edges(a_all, b_all, n_global)
    try:
        g1.analyse(key_mode)
        n, E = g1.counts()
        arr = g1.device_arrays()
        st = dg.stats()
        lo, nl = st["v_lo"], st["n_local"]
        deg1 = dev_view(arr["degree"], n, "<i4", g1, "cuda"); core1 = dev_view(arr["coreness"], n, "<i4", g1, "cuda")
        score1 = dev_view(arr["score"], n, "<f8", g1, "cuda"); edges1 = dev_view(arr["edges_packed"], E, "<i8", g1, "cuda")
        darr = dg.device_arrays()
        deg_p = dev_view(darr["degree"], nl, "<i4", dg, "cuda"); core_p = dev_view(darr["coreness"], nl, "<i4", dg, "cuda")
        score_p = dev_view(darr["score"], nl, "<f8", dg, "cuda"); edges_p = dev_view(darr["edges_packed"], st["n_fwd_local"], "<i8", dg, "cuda")
        bounds = torch.tensor([lo << 32, (lo + nl) << 32], dtype=torch.int64, device="cuda")
        e_lo, e_hi = [int(x) for x in torch.searchsorted(edges1, bounds)]
        s1 = score1[lo:lo + nl]
        rel = float(((score_p - s1).abs() / torch.clamp(s1.abs(), min=1e-300)).max()) if nl else 0.0
        absd = float((score_p - s1).abs().max()) if nl else 0.0
        score_all = tcomm.all_gather_var(score_p.clone())
        rank_same = bool(torch.equal(torch.argsort(score_all, descending=True, stable=True), torch.argsort(score1, descending=True, stable=True)))
        flags = torch.tensor([
            int(st["n_edges_global"] == E),
            int(e_hi - e_lo == st["n_fwd_local"] and bool(torch.equal(edges1[e_lo:e_hi], edges_p))),
            int(bool(torch.equal(deg1[lo:lo + nl], deg_p))),
            int(bool(torch.equal(core1[lo:lo + nl], core_p))),
            int(absd <= 1e-12 or rel <= 1e-6),
            int(rank_same)], dtype=torch.int64, device="cuda")
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        mx = torch.tensor([rel], dtype=torch.float64, device="cuda")
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        names = ["n_edges_equal", "edge_list_slices_bit_exact", "degree_bit_exact", "coreness_bit_exact", "corea_within_1e-6", "corea_ranking_identical"]
        out = {k: bool(v) for k, v in zip(names, flags.tolist())}
        out["corea_max_rel_diff"] = float(mx.item())
        out["against"] = "the single-GPU path of libkombgpu on the gathered input, run on every GPU (itself bit-exact against the CPU oracle in tests/)"
        return out
    finally:
        g1.close()
        del a_all, b_all
        torch.cuda.empty_cache()
        ctx.trim()


def run_ours_multi(args, rank, world, local_rank):
    """N > 1: weak scaling, 1 M unitigs and 5 M read pairs PER GPU; every rank holds the hits of its own reads."""
    import torch
    import torch.distributed as dist

    import komb_b200
    from komb_b200 import synth
    from komb_b200.distributed import Comm as TorchComm, CudaEngine, analyse_partitioned
    from komb_b200.peer import Comm, DistGraph

    hbm_gbs, peak_src = load_peaks()
    ctx = komb_b200.Context(local_rank)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    comm = Comm.from_torch(ctx, heap_bytes=1 << 30)
    tcomm = TorchComm("nccl")
    n_global = N_UNITIGS * world
    m1, m2 = synth.metagenome_hits(n_global, N_READ_PAIRS, seed=SEED + rank, read_offset=rank * N_READ_PAIRS, scramble=True)
    rk_h = torch.from_numpy(np.concatenate([m1.read_key, m2.read_key]).view(np.int32)).pin_memory()
    ut_h = torch.from_numpy(np.concatenate([m1.unitig, m2.unitig]).view(np.int32)).pin_memory()
    rk_d, ut_d = rk_h.cuda(non_blocking=True), ut_h.cuda(non_blocking=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def timed(fn):
        dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        out = fn()
        b.record(stream)
        torch.cuda.synchronize()
        t = torch.tensor([a.elapsed_time(b)], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)       # device time, max over ranks
        return out, float(t.item())

    def step_device(keep=False, a=None, b=None):
        g = DistGraph.from_hits(comm, rk_d if a is None else a, ut_d if b is None else b, n_global)
        g.analyse(komb_b200.KEY_REF32)
        st = g.stats()
        if keep:
            return st, g
        g.close()
        return st

    pin = {}

    def step_e2e():
        """Host hits in, this rank's share of every output back on the host (edge-list slice in CSR form, degree,
        coreness, score) -- the same outputs as the N = 1 e2e step."""
        a = rk_h.cuda(non_blocking=True)
        b = ut_h.cuda(non_blocking=True)
        _, g = step_device(keep=True, a=a, b=b)
        r = g.results(out=pin)
        fp, v = g.edges_csr(out=pin)
        g.close()
        return r["degree"].nbytes + r["coreness"].nbytes + r["score"].nbytes + fp.nbytes + v.nbytes

    n_warm = 1 if args.profile else max(args.warmup, 3)
    for _ in range(n_warm):
        st_w = step_device()
    # page-locked result buffers, sized from the warm-up (a rank's share of the edge list depends on the id range it owns)
    n_loc = st_w["n_local"]
    pin.update({"fwd_ptr": ctx.pinned_empty(n_loc + 1, np.uint64), "v": ctx.pinned_empty(st_w["n_fwd_local"] + 1024, np.uint32),
                "coreness": ctx.pinned_empty(n_loc, np.int32), "degree": ctx.pinned_empty(n_loc, np.int32),
                "score": ctx.pinned_empty(n_loc, np.float64)})
    launches0 = ctx.launches()
    sampler = ClockSampler(local_rank)
    sampler.start()
    times, stats = [], []
    for i in range(args.steps):
        flush.fill_(i & 0xff)
        st, t = timed(step_device)
        times.append(t)
        stats.append(st)
    clocks = sampler.stop()
    launches = tcomm.all_gather_ints([ctx.launches() - launches0])[:, 0]
    ms_per_step = float(np.mean(times))
    step_e2e()
    e2e_t, d2h = [], 0
    for _ in range(max(2, min(args.steps, 3))):
        flush.fill_(1)
        dist.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        d2h = step_e2e()
        torch.cuda.synchronize(); dist.barrier()
        e2e_t.append(time.perf_counter() - t0)
    e2e_s = float(np.mean(e2e_t))

    # parity inside the run: the partitioned result against the single-GPU path on the gathered hits
    _, g = step_device(keep=True)
    parity = verify_against_single_gpu(ctx, tcomm, g, rk_d, ut_d, "hits", n_global, komb_b200.KEY_REF32)
    mc, ms = g.summary()
    g.close()

    # the NCCL path of round 1 (distributed build, CSR all-gathered, replicated peel), timed once for comparison
    nccl_ms = None
    try:
        eng = CudaEngine(ctx)
        for _ in range(2):
            analyse_partitioned(eng, tcomm, n_global, read_key=rk_d, unitig=ut_d, peel_mode="gather")
        _, nccl_ms = timed(lambda: analyse_partitioned(eng, tcomm, n_global, read_key=rk_d, unitig=ut_d, peel_mode="gather"))
    except Exception as e:   # comparison only
        nccl_ms = f"failed: {type(e).__name__}: {e}"

    def mean_max(key):
        """mean over the timed steps of this rank, then max over ranks (ms)"""
        t = torch.tensor([float(np.mean([s[key] for s in stats]))], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    ms_build, ms_peel, ms_corea = mean_max("ms_build"), mean_max("ms_peel"), mean_max("ms_corea")
    ms_route, ms_sort, ms_csr = mean_max("ms_build_route"), mean_max("ms_build_sort"), mean_max("ms_build_csr")
    tot = tcomm.all_gather_ints([rk_h.numel(), d2h, stats[-1]["n_pairs_local"], stats[-1]["n_messages_sent"], stats[-1]["n_directed_local"]])
    H, P, msgs = int(tot[:, 0].sum()), int(tot[:, 2].sum()), int(tot[:, 3].sum())
    st = stats[-1]
    E, n = st["n_edges_global"], n_global
    b_peel = 24 * E + 16 * n
    b_build = 8 * H + 16 * P + 8 * E + 8 * (n + 1)
    line = {
        "metric": METRIC, "value": H / (ms_per_step * 1e-3), "unit": "hits/s", "n_gpus": world, "steps": args.steps,
        "warmup": n_warm, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": DTYPE, "data": "synthetic",
        "config": workload_config(world),
        "workload_sizes": {"n_unitigs": n, "n_read_pairs": N_READ_PAIRS * world, "n_hits": H, "n_pairs": P, "n_edges": E,
                           "max_coreness": st["max_coreness"], "peel_levels": st["peel_levels"],
                           "directed_entries_per_rank": [int(x) for x in tot[:, 4]]},
        "parallelism": f"unitig-range partition x{world}, one process per GPU; peer-memory path of libkombgpu: pairs routed to the owner "
                       "of min(u,v) by stores into peer memory; device-driven peel, one persistent kernel per GPU ("
                       + {1: "asynchronous: a neighbour is decremented where it lives by an atomic over NVLink, a unitig that falls to the "
                             "level is pushed into its owner's pool, ranks meet once per level",
                          2: "replicated: the graph is small, every rank pulls the other ranks' rows out of peer memory and peels the whole "
                             "graph with the single-GPU kernel",
                          0: "log-based: ranks broadcast the unitigs they peel and meet once per cascade generation through flags in peer "
                             "memory"}[int(st.get("peel_async", 0))]
                       + "; chosen by the shape of the graph, KOMBGPU_DIST_PEEL overrides), sharded CORE-A; no collective library on the data "
                       "path (torch.distributed only bootstraps the cudaIpc handles)",
        "stages": {"build": {"ms": ms_build, "hits_per_s": H / (ms_build * 1e-3), "algorithmic_bytes": b_build,
                             "frac_hbm": b_build / (ms_build * 1e-3) / 1e9 / (hbm_gbs * world),
                             "route_ms": ms_route, "sort_unique_ms": ms_sort, "csr_ms": ms_csr},
                   "peel": {"ms": ms_peel, "edges_per_s": E / (ms_peel * 1e-3), "algorithmic_bytes": b_peel,
                            "frac_hbm": b_peel / (ms_peel * 1e-3) / 1e9 / (hbm_gbs * world),
                            "kind": PEEL_KINDS[int(st.get("peel_async", 0))],
                            "subrounds": st["peel_subrounds"], "solo_subrounds_rank0": st["peel_solo_subrounds"],
                            "messages": msgs, "message_bytes_over_nvlink": 4 * msgs},
                   "corea": {"ms": ms_corea, "vertices_per_s": n / (ms_corea * 1e-3)},
                   "nccl_path_round1": {"ms_per_step": nccl_ms, "what": "distributed build over NCCL all_to_all, CSR all-gathered, "
                                        "peel replicated on every GPU (the default of round 1), same input"}},
        "peel_edges_per_s": E / (ms_peel * 1e-3),
        "build_hits_per_s": H / (ms_build * 1e-3),
        "roofline": {"kernel": {1: "apeel_kernel (asynchronous partitioned peel", 0: "ppeel_kernel (log-based partitioned peel",
                                2: "peel_kernel (replicated peel of the gathered graph"}[int(st.get("peel_async", 0))]
                     + ", one persistent kernel per GPU)", "bound": "hbm",
                     "achieved": b_peel / (ms_peel * 1e-3) / 1e9, "peak": hbm_gbs * world, "unit": "GB/s",
                     "frac": b_peel / (ms_peel * 1e-3) / 1e9 / (hbm_gbs * world), "traffic": None,
                     "algorithmic_bytes": b_peel, "kernel_ms": ms_peel,
                     "peak_source": peak_src + f" x {world} GPUs (aggregate)"},
        "e2e": {"value": H / e2e_s, "unit": "hits/s", "h2d_bytes_per_step": 8 * H, "d2h_bytes_per_step": int(tot[:, 1].sum()),
                "ms_per_step": e2e_s * 1e3, "edge_list_form": "csr slices (forward offsets + targets per rank)"},
        "gpu_launches": int(launches.sum()),
        "parity": parity,
        "symmetric_heap_bytes_per_rank": comm.heap_bytes(),
        "clocks": clocks,
    }
    del rk_d, ut_d
    torch.cuda.empty_cache()
    ctx.trim()
    if not args.no_configs:
        line["configs"] = {}
        only = os.environ.get("KOMB_BENCH_ONLY_CONFIG")
        if not only:
            try:
                line["configs"]["cfg3_strong"] = run_config_multi(ctx, comm, tcomm, "cfg3", world, rank, hbm_gbs, timed)
            except Exception as e:
                line["configs"]["cfg3_strong"] = {"error": f"{type(e).__name__}: {e}"}
        for name in ([only] if only else ["cfg4_eighth"] + (["cfg4", "cfg5"] if world == 8 else [])):
            try:
                line["configs"][name] = run_config_multi(ctx, comm, tcomm, name, world, rank, hbm_gbs, timed)
            except Exception as e:
                line["configs"][name] = {"error": f"{type(e).__name__}: {e}"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    dist.barrier()
    comm.close()
    ctx.close()
    dist.destroy_process_group()


def run_config_multi(ctx, comm, tcomm, name, world, rank, hbm_gbs, timed, reps: int = 2) -> dict:
    """cfg3 strong-scaled (the 1-GPU graph split over N GPUs), cfg4 at full size (8 GPUs) and at an eighth of it
    (fits one GPU, so the partitioned result is compared with the single-GPU path: the 1-vs-N invariance check)."""
    import torch
    import komb_b200
    from komb_b200.peer import DistGraph
    t0 = time.perf_counter()
    if name == "cfg3":
        n = 50_000_000
        a, b = rmat_device(26, 540_000_000 // world, n, 42 + 1000 * rank)
        kind, key_mode, verify = "pairs", komb_b200.KEY_EXACT64, True
        desc = f"cfg3: R-MAT scale 26, 540 M draws over 50 M unitigs (every rank draws 1/{world} of them), strong scaling"
    elif name == "cfg5":
        # the 1-GPU deep-core graph, every rank takes 1/world of its pair list (the generator is deterministic)
        u, v, n = ramp_device(5000, 40, 9_800_000, 24, 40_000_000, 7)
        lo, hi = u.numel() * rank // world, u.numel() * (rank + 1) // world
        a, b = u[lo:hi].clone(), v[lo:hi].clone()
        del u, v
        torch.cuda.empty_cache()
        kind, key_mode, verify = "pairs", komb_b200.KEY_EXACT64, True
        desc = (f"cfg5: deep core: ramp of 5000 levels x 40 unitigs over an R-MAT background, 10 M unitigs, ids scrambled, "
                f"{world} GPUs (strong scaling: every rank holds 1/{world} of the pair list)")
    else:
        scale = 8 if name == "cfg4_eighth" else 1
        n, pairs_total = 100_000_000 // scale, 500_000_000 // scale
        per = pairs_total // world
        a, b = cfg4_hits_device(n, rank * per, per, 0.2, 1234 + rank)
        kind, key_mode, verify = "hits", komb_b200.KEY_REF32, name == "cfg4_eighth"
        desc = (f"{name}: {pairs_total} read pairs (~{4 * pairs_total} hits) over {n} unitigs, window p = 0.2, "
                f"{world} GPUs" + (" (1/8 of cfg4: fits one GPU, compared with the single-GPU path)" if scale == 8 else ""))
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    build = DistGraph.from_hits if kind == "hits" else DistGraph.from_pairs

    def run(keep=False):
        g = build(comm, a, b, n)
        g.analyse(key_mode)
        st = g.stats()
        if keep:
            return st, g
        g.close()
        return st
    best, best_t = None, None
    for _ in range(reps):
        st, t = timed(run)
        if best_t is None or t < best_t:
            best, best_t = st, t
    st, g = run(keep=True)
    E = st["n_edges_global"]
    darr = g.device_arrays()
    deg_p = dev_view(darr["degree"], st["n_local"], "<i4", g, "cuda"); core_p = dev_view(darr["coreness"], st["n_local"], "<i4", g, "cuda")
    sums = tcomm.all_gather_ints([int(deg_p.to(torch.int64).sum()), int((core_p > deg_p).sum()), a.numel(), st["n_pairs_local"],
                                  st["n_messages_sent"]])
    out = {"workload": desc, "n_gpus": world, "n_unitigs": n, "n_inputs": int(sums[:, 2].sum()), "n_pairs": int(sums[:, 3].sum()), "n_edges": E,
           "max_degree": st["max_degree"], "max_coreness": st["max_coreness"], "peel_levels": st["peel_levels"],
           "peel_kind": PEEL_KINDS[int(st.get("peel_async", 0))],
           "peel_subrounds": st["peel_subrounds"], "peel_messages": int(sums[:, 4].sum()),
           "ms_total_max_over_ranks": best_t, "ms_build": best["ms_build"], "ms_peel": best["ms_peel"], "ms_corea": best["ms_corea"],
           "edges_per_s_total": E / (best_t * 1e-3), "peel_edges_per_s": E / (best["ms_peel"] * 1e-3),
           "peel_frac_of_aggregate_hbm": (24 * E + 16 * n) / (best["ms_peel"] * 1e-3) / 1e9 / (hbm_gbs * world),
           "degree_sum_is_2E": int(sums[:, 0].sum()) == 2 * E, "coreness_le_degree": int(sums[:, 1].sum()) == 0,
           "generate_s": gen_s}
    if verify:
        out["parity_vs_single_gpu"] = verify_against_single_gpu(ctx, tcomm, g, a, b, kind, n, key_mode)
    g.close()
    del a, b
    torch.cuda.empty_cache()
    ctx.trim()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the secondary BASELINE configs (cfg3 / cfg4 / cfg5)")
    ap.add_argument("--profile", action="store_true",
                    help="minimal run for ncu: 1 warm-up + the timed steps only, no e2e / CPU legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float64; single-GPU path)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.gpus != 1 or args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs writes the single-GPU path's outputs: use it with --gpus 1 --impl ours, in one process")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
