"""Max-core trussness and the densest k-core on the partitioned graph (pcore.cu) against the single-GPU Graph.

Workloads (bench.py's generators):
- cfg2_xN: bench.py's weak-scaled metagenome hits, 1 M unitigs and 5 M read pairs per rank, unitig ids scrambled;
- cfg3_strong: R-MAT scale 26, 540 M draws over 50 M unitigs, generated once and split into N slices;
- cfg5_reduced: the cfg5 ramp at a fifth of its depth (1000 levels x 40 unitigs over an R-MAT background of 2 M
  unitigs, 8 M draws), split into N slices.
For N = 1, 2, 4, 8 ranks, threads of one process with one GPU each (N above the GPUs present is not measured that
way; with --emulate-upto M, N <= M also runs with every rank on GPU 0, which checks the results but times host-side
exchanges, not NVLink).  Per run and rank: the maximal core's size (n_core, m_core), the max trussness, the CUDA-event
split of kombgpu_dist_max_core_truss (coreness gather, selection + slice gather, truss peel; kombgpu_debug.h), the
host time of the call and of kombgpu_dist_densest_core, and whether both results equal the single-GPU Graph's on the
same whole input bit for bit.  The single-GPU truss is timed too (host clock around kombgpu_graph_max_core_truss,
which ends in a device synchronise), twice on one graph rebuilt in between.  Each distributed run is done twice
(`reps`); the first includes module loading.  The card's name and power limit are read in the same run.

    python tools/dist_truss_probe.py --out profiles/r3/r3d_dist_truss_probe.json
"""
import argparse
import json
import subprocess
import sys
import time
from ctypes import c_int32, c_uint32, c_uint64, byref
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import torch  # noqa: E402

import bench  # noqa: E402  (the workload generators)
import komb_b200  # noqa: E402
from komb_b200 import synth  # noqa: E402
from komb_b200.peer import DistGraph, run_local  # noqa: E402

_WHOLE = {}   # name -> (n, u, v) of a strong-scaled workload
_REF = {}     # name -> the single-GPU answers on a strong-scaled workload
TRUSS_KEYS = ("n_core_vertices", "n_core_edges", "max_trussness", "u", "v", "trussness", "truss_vertices")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q or ["unknown"]


def same_truss(a, b):
    return all(np.array_equal(a[k], b[k]) and (not isinstance(a[k], np.ndarray) or a[k].dtype == b[k].dtype) for k in TRUSS_KEYS)


def workload(name, world, quick):
    """-> (kind, n, shares): shares[r] = (a, b) host arrays of rank r."""
    if name == "cfg2_xN":
        n_u, n_r = (20_000, 60_000) if quick else (bench.N_UNITIGS, bench.N_READ_PAIRS)
        shares = []
        for r in range(world):
            m1, m2 = synth.metagenome_hits(n_u * world, n_r, seed=bench.SEED + r, read_offset=r * n_r, scramble=True)
            shares.append((np.concatenate([m1.read_key, m2.read_key]), np.concatenate([m1.unitig, m2.unitig])))
        return "hits", n_u * world, shares
    if name not in _WHOLE:   # strong scaling: one whole input, split N ways
        if name == "cfg3_strong":
            scale, draws, n = (18, 2_000_000, 200_000) if quick else (26, 540_000_000, 50_000_000)
            u, v = bench.rmat_device(scale, draws, n, 42)
        else:
            u, v, n = bench.ramp_device(100, 10, 50_000, 15, 200_000, 7) if quick else bench.ramp_device(1000, 40, 2_000_000, 21, 8_000_000, 7)
        _WHOLE[name] = (n, u.cpu().numpy().view(np.uint32), v.cpu().numpy().view(np.uint32))
        del u, v
        torch.cuda.empty_cache()
    n, u, v = _WHOLE[name]
    return "pairs", n, [(u[len(u) * r // world:len(u) * (r + 1) // world], v[len(v) * r // world:len(v) * (r + 1) // world])
                        for r in range(world)]


def single_gpu(kind, n, shares):
    """The single-GPU Graph on the whole input: its truss (timed) and densest core."""
    a = np.concatenate([s[0] for s in shares])
    b = np.concatenate([s[1] for s in shares])
    ctx = komb_b200.Context(0)
    times = []
    try:
        for _ in range(2):
            with (ctx.build_graph(a, b, n) if kind == "hits" else ctx.graph_from_edges(a, b, n)) as g:
                g.coreness()
                nc, mc, tm, nt = c_uint32(), c_uint64(), c_int32(), c_uint32()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ctx._check(ctx._lib.kombgpu_graph_max_core_truss(g._h, byref(nc), byref(mc), byref(tm), byref(nt)))
                times.append((time.perf_counter() - t0) * 1e3)
                truss, dense = g.max_core_truss(), g.densest_core()
                st = g.stats()
        ctx.trim()
    finally:
        ctx.close()
    return truss, dense, {"ms_truss_host": times, "n_edges": st["n_edges"], "max_coreness": st["max_coreness"]}


def dist_run(kind, n, shares, devices, ref_truss, ref_dense):
    world = len(devices)

    def body(comm):
        a, b = shares[comm.rank]
        dev = torch.device("cuda", comm.ctx.device)
        ta = torch.from_numpy(a.view(np.int32)).to(dev)
        tb = torch.from_numpy(b.view(np.int32)).to(dev)
        torch.cuda.synchronize(dev)
        build = DistGraph.from_hits if kind == "hits" else DistGraph.from_pairs
        with build(comm, ta, tb, n) as g:
            g.coreness()
            nc, mc, tm, nt = c_uint32(), c_uint64(), c_int32(), c_uint32()
            t0 = time.perf_counter()
            g._ctx._check(g._lib.kombgpu_dist_max_core_truss(g._h, byref(nc), byref(mc), byref(tm), byref(nt)))
            ms_call = (time.perf_counter() - t0) * 1e3
            split = g.truss_timing()
            truss = g.max_core_truss()
            t0 = time.perf_counter()
            dense = g.densest_core()
            ms_dense = (time.perf_counter() - t0) * 1e3
            st = g.stats()
        return {"rank": comm.rank, "device": comm.ctx.device, "n_local": st["n_local"], "peel": bench.PEEL_KINDS.get(st["peel_async"]),
                "ms_truss_call_host": ms_call, **split, "ms_densest_call_host": ms_dense,
                "truss_equal_single_gpu": same_truss(truss, ref_truss), "densest_equal_single_gpu": dense == ref_dense}

    return run_local(world, body, devices=devices, heap_bytes=1 << 30)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--worlds", default="1,2,4,8")
    ap.add_argument("--workloads", default="cfg2_xN,cfg3_strong,cfg5_reduced")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--emulate-upto", type=int, default=0, help="also run N <= this with every rank on GPU 0")
    ap.add_argument("--quick", action="store_true", help="tiny inputs: a rehearsal of the probe itself")
    args = ap.parse_args()
    n_dev = torch.cuda.device_count()
    res = {"card": card(), "gpus_present": n_dev, "quick": args.quick, "workloads": {}}
    print(res["card"], flush=True)
    worlds = [int(w) for w in args.worlds.split(",")]
    for name in args.workloads.split(","):
        out = {}
        for world in worlds:
            placements = {}
            if world <= n_dev:
                placements["one_gpu_per_rank"] = list(range(world))
            if world > 1 and world <= args.emulate_upto:
                placements["emulated_on_gpu0"] = [0] * world
            if not placements:
                out[f"N{world}"] = f"not measured: {n_dev} GPU(s) present"
                continue
            kind, n, shares = workload(name, world, args.quick)
            if kind == "hits" or name not in _REF:
                _REF[name] = single_gpu(kind, n, shares)
            ref_truss, ref_dense, ref_info = _REF[name]
            entry = {"n_unitigs": n, "n_inputs": int(sum(len(s[0]) for s in shares)), **ref_info,
                     "n_core": ref_truss["n_core_vertices"], "m_core": ref_truss["n_core_edges"],
                     "max_trussness": ref_truss["max_trussness"], "n_truss_vertices": int(ref_truss["truss_vertices"].size),
                     "densest_core": ref_dense}
            for pl, devices in placements.items():
                entry[pl] = [dist_run(kind, n, shares, devices, ref_truss, ref_dense) for _ in range(args.reps)]
            out[f"N{world}"] = entry
            print(name, world, json.dumps(entry), flush=True)
            del shares
        res["workloads"][name] = out
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")   # after every workload
    res["card_after"] = card()
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
