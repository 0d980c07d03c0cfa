"""Multi-GPU (peer-memory) build of repeat-family hit sets whose clique pairs exceed 2^32: the pairs are emitted,
routed to the owner of min(u, v), sorted and merged there in rounds (pbuild.cu, DESIGN.md §4).

Workloads (synth.repeat_family_hits through DistGraph.from_hits):
- P4.5e9_world2_range: the default instance, reads split by read range over 2 ranks: every family read lands on rank 0,
  whose own pairs exceed 2^32;
- P9e9_world3_roundrobin: reads_per_family=1500, whole reads dealt round-robin over 3 ranks: every rank's pairs stay
  below 2^32, but the owner of the low ids receives more than 2^32 of them.

Each runs with emulated ranks (every rank on device 0: the exchanges are host-side, so the route times measure host
exchanges, not NVLink) and, when the box has enough GPUs, with one GPU per rank.  Per rank: rounds, ms_build and its
route / sort / csr split, the pairs it emitted and received, and the symmetric heap's high water
(kombgpu_comm_info); per device: how much free memory the build took (cudaMemGetInfo before the ranks start and
after every rank has built, contexts and arenas still held: every block the build held at once, plus blocks it cached
and could not reuse, so an upper bound on the peak).  The card's name and power limit are read in the same run.

    python tools/dist_pair_chunk_probe.py --out profiles/r3/r3c_dist_pair_chunk_probe.json
"""
import argparse
import json
import subprocess
import sys
import threading
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch  # noqa: E402

from komb_b200 import synth  # noqa: E402
from komb_b200.peer import DistGraph, run_local  # noqa: E402

WORKLOADS = {   # name -> (repeat_family_hits arguments, world, how the reads are split)
    "P4.5e9_world2_range": (dict(), 2, "range"),
    "P9e9_world3_roundrobin": (dict(reads_per_family=1500), 3, "roundrobin"),
}
N_UNITIGS = 200_000


def share(rk, ut, rank, world, how):
    if how == "range":
        reads = int(rk.max()) + 1
        sel = (rk >= reads * rank // world) & (rk < reads * (rank + 1) // world)
    else:
        sel = rk % world == rank
    return rk[sel], ut[sel]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q or ["unknown"]


def run(rk, ut, world, how, devices):
    torch.cuda.empty_cache()
    free0 = {d: torch.cuda.mem_get_info(d)[0] for d in set(devices)}
    meet = threading.Barrier(world)
    growth = {}

    def body(comm):
        a, b = share(rk, ut, comm.rank, world, how)
        dev = torch.device("cuda", comm.ctx.device)
        ta, tb = torch.from_numpy(a.view(np.int32)).to(dev), torch.from_numpy(b.view(np.int32)).to(dev)
        torch.cuda.synchronize(dev)
        with DistGraph.from_hits(comm, ta, tb, N_UNITIGS) as g:
            st = g.stats()
            r = {"rank": comm.rank, "device": comm.ctx.device, "rounds": g.build_rounds(),
                 **{k: st[k] for k in ("ms_build", "ms_build_route", "ms_build_sort", "ms_build_csr", "n_pairs_local",
                                       "n_pairs_received", "n_fwd_local", "n_edges_global")},
                 "heap_high_water_gb": comm.heap_bytes() / 1e9}
            meet.wait()
            if comm.rank == devices.index(comm.ctx.device):   # one rank per device measures it
                torch.cuda.synchronize(dev)
                growth[comm.ctx.device] = (free0[comm.ctx.device] - torch.cuda.mem_get_info(comm.ctx.device)[0]) / 1e9
            meet.wait()
        return r

    ranks = run_local(world, body, devices=devices)
    return {"ranks": ranks, "device_growth_gb": {str(d): g for d, g in sorted(growth.items())}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    res = {"card": card(), "workloads": {}}
    print(res["card"], flush=True)
    n_dev = torch.cuda.device_count()
    for name, (kw, world, how) in WORKLOADS.items():
        m1, m2 = synth.repeat_family_hits(**kw)
        rk, ut = np.concatenate([m1.read_key, m2.read_key]), np.concatenate([m1.unitig, m2.unitig])
        out = {"world": world, "split": how}
        placements = {"emulated_one_gpu": [0] * world}
        if n_dev >= world:
            placements["one_gpu_per_rank"] = list(range(world))
        for pl, devices in placements.items():
            runs = [run(rk, ut, world, how, devices) for _ in range(2)]
            out[pl] = runs
            print(name, pl, json.dumps(runs), flush=True)
        if "one_gpu_per_rank" not in placements:
            out["one_gpu_per_rank"] = f"not measured: {n_dev} GPU(s) present"
        res["workloads"][name] = out
    res["card_after"] = card()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
