"""Onion layers on the partitioned graph (kombgpu_dist_onion, ponion.cu) against the single-GPU onion of the same graph.

Workloads (those of tools/dist_truss_probe.py, from bench.py's generators):
- cfg2_xN: bench.py's weak-scaled metagenome hits, 1 M unitigs and 5 M read pairs per rank, unitig ids scrambled;
- cfg5_reduced: the cfg5 ramp at a fifth of its depth (1000 levels x 40 unitigs over an R-MAT background of 2 M
  unitigs, 8 M draws), as in tools/onion_probe.py, split N ways;
- cfg3_strong: R-MAT scale 26, 540 M draws over 50 M unitigs, generated once and split N ways.
For N = 1, 2, 4, 8 with one GPU per rank where the box has that many GPUs and, with --emulate-upto, N up to that many
with every rank on GPU 0 (this checks the layers but times one grid that holds every rank and meetings through one
device's memory, not NVLink).  Per run: the build layout (rows or by neighbour), the kernel's CUDA-event time (a warm-up run, then `reps`
runs through kombgpu_debug_dist_onion_again; the slowest rank of each run, then the best run), levels, meetings,
walk steps run on one CTA, the time of the by-neighbour layout built from rows when the build left rows, and whether
the ranks' layers, concatenated, equal the single-GPU Graph.onion() on the same whole input bit for bit, with the
same number of layers on every rank.  The single-GPU onion is timed in the same run, best of `reps` after a warm-up.
The card's name and power limit are read in the same run.

    python tools/dist_onion_probe.py --emulate-upto 4 --out profiles/r3/r3g_dist_onion_probe.json
"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import torch  # noqa: E402

import komb_b200  # noqa: E402
from dist_truss_probe import card, workload  # noqa: E402  (the same workloads)
from komb_b200.peer import DistGraph, run_local  # noqa: E402


def single_gpu(kind, n, shares, reps):
    a = np.concatenate([s[0] for s in shares])
    b = np.concatenate([s[1] for s in shares])
    ctx = komb_b200.Context(0)
    try:
        with (ctx.build_graph(a, b, n) if kind == "hits" else ctx.graph_from_edges(a, b, n)) as g:
            r = g.onion()
            ms = []
            for _ in range(reps):
                g.onion(again=True)
                ms.append(g.onion_timing()["ms_kernel"])
            t = g.onion_timing()
            info = {"n_edges": g.stats()["n_edges"], "n_layers": r["n_layers"], "levels": t["levels"], "steps": t["steps"],
                    "thin_layers": t["thin_layers"], "ms_kernel": ms, "ms_kernel_best": min(ms)}
        ctx.trim()
    finally:
        ctx.close()
    return r["layer"], info


def dist_run(kind, n, shares, devices, ref_layer, ref_n, reps):
    def body(comm):
        a, b = shares[comm.rank]
        dev = torch.device("cuda", comm.ctx.device)
        ta = torch.from_numpy(a.view(np.int32)).to(dev)
        tb = torch.from_numpy(b.view(np.int32)).to(dev)
        torch.cuda.synchronize(dev)
        build = DistGraph.from_hits if kind == "hits" else DistGraph.from_pairs
        with build(comm, ta, tb, n) as g:
            st = g.stats()
            lo, hi = st["v_lo"], st["v_lo"] + st["n_local"]
            r = g.onion()
            warm = g.onion_timing()
            runs = []
            for _ in range(reps):
                again = g.onion(again=True)
                assert np.array_equal(again["layer"], r["layer"])
                runs.append(g.onion_timing())
            # the build's layout: by neighbour (the log-based peel's) or rows (the asynchronous or replicated peel's),
            # which the onion transposes first
            layout = "rows" if warm["ms_transpose"] > 0 else "by_neighbour"
            return {"rank": comm.rank, "device": comm.ctx.device, "n_local": st["n_local"], "layout": layout,
                    "n_layers": r["n_layers"], "bit_equal": bool(np.array_equal(r["layer"], ref_layer[lo:hi])), "warmup": warm, "runs": runs}

    parts = run_local(len(devices), body, devices=devices, heap_bytes=1 << 30)
    per_run = [max(p["runs"][i]["ms_kernel"] for p in parts) for i in range(reps)]
    last = parts[0]["runs"][-1]
    return {"layout": parts[0]["layout"], "ms_kernel_slowest_rank": per_run, "ms_kernel_best": min(per_run),
            "levels": last["levels"], "meetings": last["meetings"], "solo_steps": [p["runs"][-1]["solo_steps"] for p in parts],
            "ms_transpose": [p["runs"][-1]["ms_transpose"] for p in parts], "n_local": [p["n_local"] for p in parts],
            "equal": bool(all(p["bit_equal"] for p in parts) and {p["n_layers"] for p in parts} == {ref_n})}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--worlds", default="1,2,4,8")
    ap.add_argument("--workloads", default="cfg2_xN,cfg5_reduced,cfg3_strong")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--emulate-upto", type=int, default=0, help="also run N <= this with every rank on GPU 0")
    ap.add_argument("--quick", action="store_true", help="tiny inputs: a rehearsal of the probe itself")
    args = ap.parse_args()
    n_dev = torch.cuda.device_count()
    res = {"card": card(), "gpus_present": n_dev, "quick": args.quick, "reps": args.reps, "workloads": {}}
    print(res["card"], flush=True)
    for name in args.workloads.split(","):
        out = {}
        for world in [int(w) for w in args.worlds.split(",")]:
            placements = {}
            if world <= n_dev:
                placements["one_gpu_per_rank"] = list(range(world))
            if 1 < world <= args.emulate_upto:
                placements["emulated_on_gpu0"] = [0] * world
            if not placements:
                continue
            kind, n, shares = workload(name, world, args.quick)
            ref_layer, single = single_gpu(kind, n, shares, args.reps)
            row = {"n_unitigs": n, "single_gpu": single}
            for where, devices in placements.items():
                row[where] = dist_run(kind, n, shares, devices, ref_layer, single["n_layers"], args.reps)
                print(name, world, where, json.dumps(row[where]), flush=True)
            out[str(world)] = row
            torch.cuda.empty_cache()
            res["workloads"][name] = out
            Path(args.out).parent.mkdir(parents=True, exist_ok=True)
            Path(args.out).write_text(json.dumps(res, indent=1) + "\n")   # after every run
    res["card_after"] = card()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
