"""The three output files formatted on the device over the ranks (kombgpu_dist_graph_format, format.cu) on the cfg2 SAM
pair (synth.metagenome_hits, 1 M unitigs, 5 M read pairs, synth.render_sam with @SQ headers).

In one run:
- format: the graph parsed and built over N = 1, 2, 4 ranks (one GPU per rank where the box has them, else every rank
  on GPU 0), peeled and scored; each rank formats edgelist.txt, kcore.tsv and CoreA_anomaly.txt in turn (one rank at a
  time).  Per rank and file: bytes, and the host time of the format call up to a device synchronise, twice (the text
  is cached after the first call, so the second run builds a new graph); bytes/s over that time.  The same for
  kombgpu_graph_format on one GPU, and whether the concatenated slices equal its bytes;
- komb2: bin/komb2 with KOMB_GPU_DEVICES of N = 2, 4, 8 ranks, device output (the default) against KOMB_OUTPUT=host,
  alternated, --reps runs each, with the KOMB_TIMING marks of every run and whether the three files are identical;
- with --parse-only: only the partitioned parse of the cfg2 pair at N = 2 and 4 (per-rank CUDA-event times of the
  upload, parse, interning and routing), from the tree given by --root, so a parent tree can be measured against this
  one in the same run.
The card's name and power limit are read in the same run.

    python tools/dist_format_probe.py --out profiles/dist_format_probe.json [--quick] [--reps 3]
    python tools/dist_format_probe.py --parse-only --root <tree> --out parse.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="profiles/dist_format_probe.json")
ap.add_argument("--quick", action="store_true")
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--parse-only", action="store_true")
ap.add_argument("--root", default=str(Path(__file__).resolve().parents[1]))
args = ap.parse_args()
ROOT = Path(args.root).resolve()
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

import komb_b200  # noqa: E402
from komb_b200 import synth  # noqa: E402
from komb_b200.peer import DistGraph, DistHits, run_local  # noqa: E402

FILES = ("edgelist.txt", "kcore.tsv", "CoreA_anomaly.txt")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q or ["unknown"]


def cfg2_pair(quick):
    n_u, n_p = (20_000, 100_000) if quick else (1_000_000, 5_000_000)
    m1, m2 = synth.metagenome_hits(n_u, n_p)
    return [synth.render_sam(m1, n_u, 1), synth.render_sam(m2, n_u, 2)]


def devices_for(world, n_dev):
    return list(range(world)) if world <= n_dev else [0] * world


def timed(dev, fn):
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize(dev)   # the format's second pass is still queued when the call returns
    return r, (time.perf_counter() - t0) * 1e3


def single_format(texts):
    ctx = komb_b200.Context(0)
    runs = []
    try:
        for _ in range(2):
            with ctx.sam_parse(texts) as h, h.build_graph() as g:
                g.analyse()
                row, files = [], []
                for w in range(3):
                    n, ms = timed(0, lambda: _format_bytes(g._lib.kombgpu_graph_format, g, w, h))
                    row.append({"file": FILES[w], "bytes": n, "ms": ms, "bytes_per_s": n / (ms * 1e-3)})
                    files.append(g.format(w, h))
                runs.append(row)
    finally:
        ctx.close()
    return runs, files


def _format_bytes(fn, g, w, h):
    from ctypes import byref, c_uint64
    n = c_uint64()
    g._ctx._check(fn(g._h, w, h._h if (h is not None and w == 1) else None, byref(n)))
    return n.value


def dist_format(texts, world, devices):
    turn = threading.Lock()   # one rank formats at a time: the device synchronise covers its own work only

    def body(comm):
        runs = []
        for _ in range(2):
            with DistHits.parse(comm, texts) as h, DistGraph.from_dist_hits(h) as g:
                g.analyse()
                row, files = [], []
                for w in range(3):
                    with turn:
                        n, ms = timed(comm.ctx.device, lambda: _format_bytes(g._lib.kombgpu_dist_graph_format, g, w, h))
                    row.append({"file": FILES[w], "bytes": n, "ms": ms, "bytes_per_s": n / (ms * 1e-3) if ms else None})
                    files.append(g.format(w, h))
                runs.append(row)
        return {"runs": runs, "files": files}
    return run_local(world, body, devices=devices)


def parse_times(texts, world, devices):
    def body(comm):
        out = []
        for _ in range(3):
            torch.cuda.synchronize(comm.ctx.device)
            t0 = time.perf_counter()
            with DistHits.parse(comm, texts) as h:
                out.append({"host_ms": (time.perf_counter() - t0) * 1e3, **h.timing()})
        return out
    return run_local(world, body, devices=devices)


def komb2_runs(texts, world, devices, reps, tmp):
    d = Path(tmp)
    (d / "r1.sam").write_bytes(texts[0])
    (d / "r2.sam").write_bytes(texts[1])
    (d / "u.fasta").write_bytes(b">0\nACGT\n")
    res = {"devices": devices, "device": [], "host": []}
    for rep in range(reps):
        for mode, extra in (("device", {}), ("host", {"KOMB_OUTPUT": "host"})):
            out = d / f"out_{mode}"
            out.mkdir(exist_ok=True)
            env = {k: v for k, v in os.environ.items() if k not in ("KOMB_OUTPUT", "KOMB_TOKENIZE")}
            env.update(KOMB_GPU_DEVICES=",".join(map(str, devices)), KOMB_TIMING="1", **extra)
            t0 = time.perf_counter()
            cp = subprocess.run([str(ROOT / "bin" / "komb2"), "-t", "16", "-l", "100", "-o", str(out), "-i", str(d / "r1.sam"),
                                 "-j", str(d / "r2.sam"), "-u", str(d / "u.fasta")], env=env, capture_output=True, text=True)
            res[mode].append({"wall_s": time.perf_counter() - t0, "rc": cp.returncode,
                              "timing": [ln for ln in cp.stderr.splitlines() if ln.startswith("[komb2 timing]")],
                              "stderr_tail": cp.stderr[-300:] if cp.returncode else ""})
    res["files_identical"] = all((d / "out_device" / f).read_bytes() == (d / "out_host" / f).read_bytes() for f in FILES)
    res["file_bytes"] = {f: (d / "out_device" / f).stat().st_size for f in FILES}
    for mode in ("device", "host"):
        w = sorted(r["wall_s"] for r in res[mode])
        res[f"{mode}_wall_s_median"] = w[len(w) // 2]
    return res


def main():
    n_dev = torch.cuda.device_count()
    report = {"card": card(), "devices": n_dev, "root": str(ROOT)}
    texts = cfg2_pair(args.quick)
    report["sam_bytes"] = sum(len(t) for t in texts)
    if args.parse_only:
        report["parse"] = []
        for world in (2, 4):
            devs = devices_for(world, n_dev)
            report["parse"].append({"world": world, "devices": devs, "ranks": parse_times(texts, world, devs)})
            print(json.dumps(report["parse"][-1])[:600], flush=True)
    else:
        s_runs, s_files = single_format(texts)
        report["single"] = s_runs
        print(json.dumps({"single": s_runs[-1]}), flush=True)
        report["dist"] = []
        for world in (1, 2, 4):
            devs = devices_for(world, n_dev)
            parts = dist_format(texts, world, devs)
            row = {"world": world, "devices": devs, "ranks": [p["runs"] for p in parts],
                   "same_as_single": [b"".join(p["files"][w] for p in parts) == s_files[w] for w in range(3)]}
            report["dist"].append(row)
            print(json.dumps({"world": world, "same_as_single": row["same_as_single"], "rank0": row["ranks"][0][-1]}), flush=True)
        report["komb2"] = []
        for world in (2, 4, 8):
            devs = devices_for(world, n_dev)
            with tempfile.TemporaryDirectory() as tmp:
                r = komb2_runs(texts, world, devs, args.reps, tmp)
            report["komb2"].append({"world": world, **r})
            print(json.dumps({"world": world, "devices": devs, "device_s": r["device_wall_s_median"], "host_s": r["host_wall_s_median"],
                              "files_identical": r["files_identical"]}), flush=True)
    report["card_after"] = card()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(report, indent=1, default=str))


if __name__ == "__main__":
    main()
