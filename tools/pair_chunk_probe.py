"""Chunked clique-pair build on one GPU: repeat-family hit sets whose pairs exceed 2^32 (synth.repeat_family_hits).

For each workload: build time (kombgpu_stats.ms_build, host hits in, upload included), the chunk count, pairs per
second, the arena's growth over the build (cudaMemGetInfo before and after, with the context's arena trimmed before:
every block the build held at once, plus blocks it cached and could not reuse, so an upper bound on the peak), and a
kernel-time split over all chunks (emit / sort / reduce / merge) from a separate torch.profiler run.  Then an A/B at
P ~ 3.5e9 (below 2^32): the one-shot path against the default chunk forced with KOMBGPU_PAIR_CHUNK, alternated.

    python tools/pair_chunk_probe.py --out profiles/r3/r3b_pair_chunk_probe.json
"""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch  # noqa: E402

import komb_b200  # noqa: E402
from komb_b200 import synth  # noqa: E402

K_PAIR_CHUNK = (1 << 30) - (1 << 20)

WORKLOADS = {   # name -> repeat_family_hits arguments
    "P4.5e9_Esmall": dict(),
    "P9e9_Esmall": dict(reads_per_family=1500),
    "P4.5e9_E3e8": dict(n_unitigs=400_000, family_size=2000, overlap=0, n_families=150, reads_per_family=15),
}


def phase(name):
    if "emit_" in name:
        return "emit"
    if "radix" in name or "sweep" in name:
        return "sort"
    if "EdgeFlagIn" in name:
        return "reduce"
    if "unique_merge" in name or "ReadU32" in name:
        return "merge"
    return "other"


def build_once(ctx, rk, ut, n):
    ctx.trim()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    t0 = time.perf_counter()
    g = ctx.build_graph(rk, ut, n)
    wall = time.perf_counter() - t0
    free1 = torch.cuda.mem_get_info()[0]
    st = g.stats()
    r = {"n_hits": st["n_hits"], "n_pairs": st["n_pairs"], "n_edges": st["n_edges"], "n_chunks": g.build_chunks(),
         "ms_build": st["ms_build"], "s_wall": wall, "pairs_per_s": st["n_pairs"] / (st["ms_build"] * 1e-3),
         "arena_growth_gb": (free0 - free1) / 1e9}
    g.close()
    return r


def split(ctx, rk, ut, n):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        g = ctx.build_graph(rk, ut, n)
        torch.cuda.synchronize()
    g.close()
    ms = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t:
            ms[phase(ev.key)] = ms.get(phase(ev.key), 0.0) + t / 1e3
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--skip-ab", action="store_true")
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else "unknown", "workloads": {}, "ab": []}
    print(res["gpu"], flush=True)
    ctx = komb_b200.Context(0)
    os.environ.pop("KOMBGPU_PAIR_CHUNK", None)
    for name, kw in WORKLOADS.items():
        m1, m2 = synth.repeat_family_hits(**kw)
        n = kw.get("n_unitigs", 200_000)
        rk, ut = np.concatenate([m1.read_key, m2.read_key]), np.concatenate([m1.unitig, m2.unitig])
        build_once(ctx, rk, ut, n)                     # warm-up
        runs = [build_once(ctx, rk, ut, n) for _ in range(2)]
        res["workloads"][name] = {"runs": runs, "kernel_ms_by_phase": split(ctx, rk, ut, n)}
        print(name, json.dumps(res["workloads"][name]), flush=True)
    if not args.skip_ab:
        m1, m2 = synth.repeat_family_hits(reads_per_family=584)
        rk, ut = np.concatenate([m1.read_key, m2.read_key]), np.concatenate([m1.unitig, m2.unitig])
        build_once(ctx, rk, ut, 200_000)
        for arm in ["one_shot", "chunked", "one_shot", "chunked"]:
            if arm == "chunked":
                os.environ["KOMBGPU_PAIR_CHUNK"] = str(K_PAIR_CHUNK)
            else:
                os.environ.pop("KOMBGPU_PAIR_CHUNK", None)
            r = build_once(ctx, rk, ut, 200_000)
            r["arm"] = arm
            res["ab"].append(r)
            print("ab", json.dumps(r), flush=True)
        os.environ.pop("KOMBGPU_PAIR_CHUNK", None)
    ctx.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
