#!/usr/bin/env python
"""Kernel split of one bench.py step on one GPU: the cfg2 hits (bench.py's workload and seed) built into a graph, peeled
and scored once under torch.profiler, after two warm-up steps.  Prints (and with --out writes) one JSON object: every
kernel's name, launches and summed device time, largest first, and the step's stats.

    python tools/build_kernel_split.py [--root TREE] [--out FILE]

--root imports komb_b200 from another tree (a parent commit's, for a before/after split from one run).
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=str(Path(__file__).resolve().parents[1]))
    ap.add_argument("--out")
    args = ap.parse_args()
    sys.path.insert(0, str(Path(args.root).resolve()))
    import torch
    from torch.profiler import ProfilerActivity, profile

    import komb_b200
    from komb_b200 import synth

    card = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    ctx = komb_b200.Context(0)
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    m1, m2 = synth.metagenome_hits(1_000_000, 5_000_000, seed=11)
    rk = torch.from_numpy(np.concatenate([m1.read_key, m2.read_key]).view(np.int32)).cuda()
    ut = torch.from_numpy(np.concatenate([m1.unitig, m2.unitig]).view(np.int32)).cuda()

    def step():
        g = ctx.build_graph(rk, ut, 1_000_000)
        g.analyse(komb_b200.KEY_REF32)
        st = g.stats()
        g.close()
        return st

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        st = step()
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        k = kernels.setdefault(e.name, {"name": e.name, "launches": 0, "us": 0.0})
        k["launches"] += 1
        k["us"] += e.device_time if hasattr(e, "device_time") else e.cuda_time
    rows = sorted(kernels.values(), key=lambda k: -k["us"])
    out = {"root": args.root, "card": card, "stats": st, "total_us": sum(k["us"] for k in rows), "kernels": rows}
    ctx.close()
    text = json.dumps(out, indent=1)
    if args.out:
        Path(args.out).write_text(text)
    print(text)


if __name__ == "__main__":
    main()
