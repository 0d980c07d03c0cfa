"""The densest block on the partitioned graph (kombgpu_dist_densest_block, pcore.cu) against the single-GPU Graph.

Workloads (those of tools/dist_truss_probe.py, from bench.py's generators):
- cfg2_xN: bench.py's weak-scaled metagenome hits, 1 M unitigs and 5 M read pairs per rank, unitig ids scrambled;
- cfg3_strong: R-MAT scale 26, 540 M draws over 50 M unitigs, generated once and split into N slices.
For N = 1 on one GPU, N = 2 and 4 with every rank on GPU 0 (--emulate-upto: this checks the results but times
host-side exchanges, not NVLink) and, where the box has several GPUs, N up to their number with one GPU per rank.
Two weightings at eps = 0.5: unweighted, and dyadic weights (integers(0, 8192) / 1024, every partial sum exact in
double), each rank passing its slice.  Per run and rank: the build layout, the passes, the host time of the call
(it ends in reading the member mask back, so it is synchronised) and whether every scalar and the rank's member slice
equal the single-GPU Graph.densest_block on the same whole input bit for bit.  The single-GPU call is timed on the
same input, twice per weighting after a warm-up call.  Each distributed run is done twice (`reps`); the first
includes module loading.  The card's name and power limit are read in the same run.

    python tools/dist_densest_block_probe.py --emulate-upto 4 --out profiles/r3/r3e_dist_densest_block_probe.json
"""
import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import torch  # noqa: E402

import bench  # noqa: E402
import komb_b200  # noqa: E402
from dist_truss_probe import card, workload  # noqa: E402  (the same workloads)
from komb_b200.peer import DistGraph, run_local  # noqa: E402

KEYS = ("n_vertices", "n_edges", "weight_sum", "density", "passes")
EPS = 0.5


def weights(n):
    return np.random.default_rng(3).integers(0, 8192, n).astype(np.float64) / 1024.0


def single_gpu(kind, n, shares):
    """The single-GPU Graph.densest_block on the whole input, per weighting, with its host times."""
    a = np.concatenate([s[0] for s in shares])
    b = np.concatenate([s[1] for s in shares])
    w = weights(n)
    ctx = komb_b200.Context(0)
    ref, ms = {}, {}
    try:
        with (ctx.build_graph(a, b, n) if kind == "hits" else ctx.graph_from_edges(a, b, n)) as g:
            for name, wt in (("unweighted", None), ("dyadic", w)):
                g.densest_block(weight=wt, eps=EPS)   # warm-up
                ms[name] = []
                for _ in range(2):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    ref[name] = g.densest_block(weight=wt, eps=EPS)
                    ms[name].append((time.perf_counter() - t0) * 1e3)
            st = g.stats()
        ctx.trim()
    finally:
        ctx.close()
    info = {"n_edges": st["n_edges"], "ms_single_gpu_host": ms,
            **{f"block_{k}": {k2: ref[k][k2] for k2 in KEYS} for k in ref}}
    return ref, info


def dist_run(kind, n, shares, devices, ref):
    world = len(devices)
    w = weights(n)

    def body(comm):
        a, b = shares[comm.rank]
        dev = torch.device("cuda", comm.ctx.device)
        ta = torch.from_numpy(a.view(np.int32)).to(dev)
        tb = torch.from_numpy(b.view(np.int32)).to(dev)
        torch.cuda.synchronize(dev)
        build = DistGraph.from_hits if kind == "hits" else DistGraph.from_pairs
        out = {"rank": comm.rank, "device": comm.ctx.device}
        with build(comm, ta, tb, n) as g:
            st = g.stats()
            lo, hi = st["v_lo"], st["v_lo"] + st["n_local"]
            out.update(n_local=st["n_local"], layout=bench.PEEL_KINDS.get(st["peel_async"]))
            for name, wt in (("unweighted", None), ("dyadic", w[lo:hi])):
                t0 = time.perf_counter()
                got = g.densest_block(weight=wt, eps=EPS)
                out[f"ms_call_host_{name}"] = (time.perf_counter() - t0) * 1e3
                out[f"passes_{name}"] = got["passes"]
                out[f"bit_equal_{name}"] = bool(all(got[k] == ref[name][k] for k in KEYS)
                                                and np.array_equal(got["member"], ref[name]["member"][lo:hi]))
        out["bit_equal"] = out["bit_equal_unweighted"] and out["bit_equal_dyadic"]
        return out

    return run_local(world, body, devices=devices, heap_bytes=1 << 30)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--worlds", default="1,2,4")
    ap.add_argument("--workloads", default="cfg2_xN,cfg3_strong")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--emulate-upto", type=int, default=0, help="also run N <= this with every rank on GPU 0")
    ap.add_argument("--quick", action="store_true", help="tiny inputs: a rehearsal of the probe itself")
    args = ap.parse_args()
    n_dev = torch.cuda.device_count()
    res = {"card": card(), "gpus_present": n_dev, "quick": args.quick, "eps": EPS, "workloads": {}}
    print(res["card"], flush=True)
    worlds = [int(w) for w in args.worlds.split(",")]
    refs = {}
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
            if kind == "hits" or name not in refs:   # cfg2 grows with N; cfg3 is one input
                refs[name] = single_gpu(kind, n, shares)
            ref, info = refs[name]
            entry = {"n_unitigs": n, "n_inputs": int(sum(len(s[0]) for s in shares)), **info}
            for pl, devices in placements.items():
                entry[pl] = [dist_run(kind, n, shares, devices, ref) for _ in range(args.reps)]
            out[f"N{world}"] = entry
            print(name, world, json.dumps(entry), flush=True)
            del shares
        res["workloads"][name] = out
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")   # after every workload
    res["all_bit_equal"] = all(r["bit_equal"] for wl in res["workloads"].values() for e in wl.values() if isinstance(e, dict)
                               for pl in ("one_gpu_per_rank", "emulated_on_gpu0") for rep in e.get(pl, []) for r in rep)
    res["card_after"] = card()
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
