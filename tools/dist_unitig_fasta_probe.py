"""The unitig FASTA over the ranks (kombgpu_dist_fasta_*, kombgpu_dist_anomalous, pfasta.cu) against the single-GPU
kombgpu_fasta_* calls, at the sizes of profiles/r3/r3a_unitig_fasta_probe.json (1 M and 50 M records), and komb2 with
KOMB_UNITIG_FASTA=anomalous under KOMB_GPU_DEVICES, this tree against a parent build.

In one run:
- single: tools/unitig_fasta_probe.py's pass on one GPU (upload, index, join, fence over host scores, extraction);
- dist: N = 1, 2, 4 ranks with every rank on GPU 0 (emulation: one PCIe link for every rank's upload, host-side
  exchanges) and, where the box has N GPUs, one GPU per rank.  Per rank the CUDA-event times of upload, index, join and
  extraction (anomalous records, then every record), which include the waits for the other ranks, and the host time of
  kombgpu_dist_anomalous on the scores of a partitioned graph with one vertex per record (it ends in a device
  synchronise); the concatenated extraction is checked against the single-GPU bytes;
- komb2: bin/komb2 on the drop-in probe's SAM pair (625 000 pairs, 1 M unitigs) with a FASTA of every unitig,
  KOMB_UNITIG_FASTA=anomalous and KOMB_GPU_DEVICES, this tree and --parent (a parent commit's bin/komb2 with its
  library beside it), alternated, --reps runs each; anomalous_unitigs.fasta must be equal.
The card's name and power limit are read in the same run.

    python tools/dist_unitig_fasta_probe.py --out profiles/r3/r3f_dist_unitig_fasta_probe.json --parent <tree>
"""
import argparse
import ctypes
import json
import os
import re
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import komb_b200  # noqa: E402
from komb_b200 import synth  # noqa: E402
from komb_b200.peer import DistFasta, DistGraph, run_local  # noqa: E402
from unitig_fasta_probe import decimal_table, hbm_peak, probe_pass, synth_fasta  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q or ["unknown"]


def graph_pairs(n, seed):
    """A ring over n vertices with n random chords: scores with ties and a tail."""
    rng = np.random.default_rng(seed)
    u = np.concatenate([np.arange(n), rng.integers(0, n, n)]).astype(np.int32)
    v = np.concatenate([(np.arange(n) + 1) % n, rng.integers(0, n, n)]).astype(np.int32)
    keep = u != v
    return u[keep], v[keep]


def single_reference(ctx, text, names, off, u, v, n):
    """The single-GPU anomalous mask of the graph and its extraction: what the ranks' slices must equal."""
    with ctx.graph_from_edges(u, v, n) as g:
        g.coreness()
        g.corea()
        anom = g.anomalous()
    h = ctypes.c_void_p()
    ctx._check(ctx._lib.kombgpu_fasta_load(ctx._h, ctypes.c_char_p(text.ctypes.data), len(text), ctypes.byref(h)))
    fa = komb_b200.Fasta(ctx, h)
    miss = ctypes.c_uint32()
    ctx._check(ctx._lib.kombgpu_fasta_join_names(fa._h, names, ctypes.c_void_p(off.ctypes.data), n, ctypes.byref(miss)))
    out = fa.extract(anom["member"])
    fa.close()
    return anom, out


def dist_pass(world, devices, text, names, off, u, v, n):
    import torch

    def body(comm):
        r = {"rank": comm.rank}
        dev = torch.device("cuda", comm.ctx.device)
        lo, hi = len(u) * comm.rank // comm.world, len(u) * (comm.rank + 1) // comm.world
        du, dv = torch.from_numpy(u[lo:hi]).to(dev), torch.from_numpy(v[lo:hi]).to(dev)
        torch.cuda.synchronize(dev)
        with DistGraph.from_pairs(comm, du, dv, n) as g:
            g.analyse()
            st = g.stats()
            t0 = time.perf_counter()
            anom = g.anomalous()
            r["ms_fence_host"] = (time.perf_counter() - t0) * 1e3
            h = ctypes.c_void_p()
            comm.ctx._check(comm._lib.kombgpu_dist_fasta_load(comm._h, ctypes.c_char_p(text.ctypes.data), len(text), ctypes.byref(h)))
            fa = DistFasta(comm, h)
            a, b = int(off[st["v_lo"]]), int(off[st["v_lo"] + st["n_local"]])
            loff = (off[st["v_lo"]:st["v_lo"] + st["n_local"] + 1] - off[st["v_lo"]]).astype(np.uint64)
            miss = ctypes.c_uint32()
            comm.ctx._check(comm._lib.kombgpu_dist_fasta_join_names(fa._h, names[a:b], ctypes.c_void_p(loff.ctypes.data), st["n_local"],
                                                                    ctypes.byref(miss)))
            assert miss.value == 0
            out = fa.extract(anom["member"])
            r.update(fa.timing())
            r["ms_extract_anomalous"] = r.pop("ms_extract")
            r["extract_anomalous_bytes"] = len(out)
            all_bytes = len(fa.extract(np.ones(st["n_local"], bool)))
            r["ms_extract_all"] = fa.timing()["ms_extract"]
            r["extract_all_bytes"] = all_bytes
            r["slice_bytes"] = fa.counts()["byte_hi"] - fa.counts()["byte_lo"]
            r["records_local"] = fa.counts()["n_records_local"]
            r["n_selected"] = anom["n_selected"]
            fa.close()
            return r, out, (anom["q1"], anom["q3"], anom["fence"])
    return run_local(world, body, devices=devices)


def probe_size(ctx, n, seed, peak, worlds, n_gpus):
    text = synth_fasta(n, seed)
    res = {"records": n, "fasta_bytes": len(text)}
    probe_pass(ctx, text, n, seed, peak)                     # warm-up
    res["single"] = probe_pass(ctx, text, n, seed, peak)
    perm = np.random.default_rng(seed + 1).permutation(n)
    names, off = decimal_table(perm)
    names, off = names.tobytes(), off.astype(np.uint64)
    u, v = graph_pairs(n, seed + 3)
    anom, exp = single_reference(ctx, text, names, off, u, v, n)
    res["single_fence"] = {k: anom[k] for k in ("q1", "q3", "fence", "n_selected")}
    res["dist"] = []
    for world in worlds:
        layouts = [("emulated", [0] * world)] + ([("distinct", list(range(world)))] if n_gpus >= world and world > 1 else [])
        for how, devices in layouts:
            for rep in range(2):   # the second run is reported: kernels loaded, heap grown
                parts = dist_pass(world, devices, text, names, off, u, v, n)
            ranks = [p[0] for p in parts]
            ok = b"".join(p[1] for p in parts) == exp and all(p[2] == (anom["q1"], anom["q3"], anom["fence"]) for p in parts)
            res["dist"].append({"world": world, "devices": how, "equal_to_single": ok, "ranks": ranks})
    if not any(d["devices"] == "distinct" for d in res["dist"]):
        res["distinct_gpus"] = "not measured (%d GPU present)" % n_gpus
    return res


def komb2_ab(parent, reps, threads, devices):
    n = 1_000_000
    m1, m2 = synth.metagenome_hits(n, 625_000, seed=11)
    trees = {"this": ROOT / "bin" / "komb2", "parent": Path(parent) / "bin" / "komb2"}
    res = {"pairs": 625_000, "unitigs": n, "KOMB_GPU_DEVICES": devices, "runs": []}
    with tempfile.TemporaryDirectory() as d:
        d = Path(d)
        (d / "r1.sam").write_bytes(synth.render_sam(m1, n, 1, with_header=False))
        (d / "r2.sam").write_bytes(synth.render_sam(m2, n, 2, with_header=False))
        (d / "u.fasta").write_bytes(synth_fasta(n, 5).tobytes())
        fastas = {}
        for k in range(2 * reps):
            which = ("this", "parent")[k % 2]
            env = dict(os.environ, KOMB_UNITIG_FASTA="anomalous", KOMB_GPU_DEVICES=devices)
            out = d / f"out{k}"
            out.mkdir()
            t0 = time.perf_counter()
            cp = subprocess.run([str(trees[which]), "-t", str(threads), "-l", "100", "-o", str(out), "-i", str(d / "r1.sam"), "-j", str(d / "r2.sam"),
                                 "-u", str(d / "u.fasta")], capture_output=True, text=True, env=env)
            wall = time.perf_counter() - t0
            ana = re.search(r"analysis \(sec\) = ([0-9.]+)", cp.stdout)
            run = {"tree": which, "rc": cp.returncode, "wall_s": round(wall, 3), "analysis_s": float(ana.group(1)) if ana else None}
            f = out / "anomalous_unitigs.fasta"
            if f.exists():
                fastas.setdefault(which, f.read_bytes())
                run["anomalous_unitigs_bytes"] = f.stat().st_size
            if cp.returncode:
                run["stderr"] = cp.stderr[-500:]
            res["runs"].append(run)
        res["fasta_equal"] = len(fastas) == 2 and fastas["this"] == fastas["parent"]
    for which in ("this", "parent"):
        w = [r["wall_s"] for r in res["runs"] if r["tree"] == which]
        res[f"median_wall_s_{which}"] = float(np.median(w))
    return res


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r3/r3f_dist_unitig_fasta_probe.json")
    ap.add_argument("--sizes", default="1000000,50000000")
    ap.add_argument("--worlds", default="1,2,4")
    ap.add_argument("--parent", default="")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--threads", type=int, default=16)
    a = ap.parse_args()
    peak, peak_src = hbm_peak()
    n_gpus = torch.cuda.device_count()
    res = {"card": card(), "gpus": n_gpus, "hbm_peak_gbs": peak, "peak_source": peak_src, "sizes": []}
    ctx = komb_b200.Context(0)
    worlds = [int(x) for x in a.worlds.split(",")]
    for k, n in enumerate(int(x) for x in a.sizes.split(",")):
        res["sizes"].append(probe_size(ctx, n, 100 + k, peak, worlds, n_gpus))
    ctx.close()
    if a.parent:
        devices = ",".join(str(d) for d in range(min(n_gpus, 4))) if n_gpus >= 2 else "0,0"
        res["komb2"] = komb2_ab(a.parent, a.reps, a.threads, devices)
    res["card_after"] = card()
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1))
    print(json.dumps({k: res[k] for k in ("card", "gpus")}))


if __name__ == "__main__":
    main()
