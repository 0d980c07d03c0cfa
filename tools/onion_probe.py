"""Onion layers (onion.cu, kombgpu_graph_onion) on bench.py's workloads, next to the k-core peel on the same graph.

Workloads (bench.py's generators):
- cfg2: the metagenome hits of bench.py, 1 M unitigs and 5 M read pairs;
- cfg3: R-MAT scale 26, 540 M draws over 50 M unitigs;
- cfg5_reduced: the cfg5 ramp at a fifth of its depth (1000 levels x 40 unitigs over an R-MAT background of 2 M
  unitigs, 8 M draws), as in tools/dist_truss_probe.py.
Per workload: the number of layers and of non-empty levels, the steps between grid barriers and the layers CTA 0 ran
alone; the onion kernel's CUDA-event time, best of 5 runs after a warm-up run (kombgpu_debug_onion_again /
_timing); the same for the k-core peel (kombgpu_debug_peel_again, stats ms_peel_kernel); and whether the layers equal
the C restatement (tests/onion_ref.c) and the onion's coreness the peel's, where the restatement is run (not on cfg3,
whose edge list would take the host minutes).  The card's name and power limit are read in the same run.

    python tools/onion_probe.py --out profiles/r3/r3f_onion_probe.json
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import torch  # noqa: E402

import bench  # noqa: E402  (the workload generators)
import komb_b200  # noqa: E402
from komb_b200 import synth  # noqa: E402
from onion_ref import onion_layers  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return q.strip().splitlines() or ["unknown"]


def graph(ctx, name, quick):
    if name == "cfg2":
        n_u, n_r = (20_000, 60_000) if quick else (bench.N_UNITIGS, bench.N_READ_PAIRS)
        m1, m2 = synth.metagenome_hits(n_u, n_r, seed=bench.SEED)
        return ctx.build_graph(np.concatenate([m1.read_key, m2.read_key]), np.concatenate([m1.unitig, m2.unitig]), n_u)
    if name == "cfg3":
        scale, draws, n = (18, 2_000_000, 200_000) if quick else (26, 540_000_000, 50_000_000)
        u, v = bench.rmat_device(scale, draws, n, 42)
    else:
        u, v, n = bench.ramp_device(100, 10, 50_000, 15, 200_000, 7) if quick else bench.ramp_device(1000, 40, 2_000_000, 21, 8_000_000, 7)
    torch.cuda.synchronize()   # the library's stream does not wait for torch's
    return ctx.graph_from_edges(u, v, n)


def measure(ctx, name, quick, reps, oracle):
    with graph(ctx, name, quick) as g:
        n, m = g.counts()
        r = g.onion()
        t = [g.onion_timing()]
        for _ in range(reps):
            g.onion(again=True)
            t.append(g.onion_timing())
        core = g.coreness()
        peel = []
        for _ in range(reps):
            g.coreness(copy=False, again=True)
            peel.append(g.stats()["ms_peel_kernel"])
        out = {"n_unitigs": n, "n_edges": m, "n_layers": r["n_layers"], "levels": t[-1]["levels"], "steps": t[-1]["steps"],
               "thin_layers": t[-1]["thin_layers"], "max_coreness": int(core.max()) if n else 0,
               "onion_ms_warmup": t[0]["ms_kernel"], "onion_ms": [x["ms_kernel"] for x in t[1:]],
               "onion_ms_best": min(x["ms_kernel"] for x in t[1:]), "peel_ms": peel, "peel_ms_best": min(peel)}
        if oracle:
            u, v = g.edges()
            layer, ref_core, ref_n = onion_layers(n, u, v)
            out["oracle_layers_equal"] = bool(ref_n == r["n_layers"] and np.array_equal(layer, r["layer"]))
            out["oracle_coreness_equal"] = bool(np.array_equal(ref_core, core))
        else:
            out["oracle"] = "not run"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workloads", default="cfg2,cfg5_reduced,cfg3")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="tiny inputs: a rehearsal of the probe itself")
    args = ap.parse_args()
    ctx = komb_b200.Context(0)
    res = {"card": card(), "quick": args.quick, "workloads": {}}
    print(res["card"], flush=True)
    for name in args.workloads.split(","):
        res["workloads"][name] = measure(ctx, name, args.quick, args.reps, oracle=name != "cfg3")
        print(name, json.dumps(res["workloads"][name]), flush=True)
        torch.cuda.empty_cache()
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")   # after every workload
    res["card_after"] = card()
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
