"""SAM text -> hits over the GPUs of one node (kombgpu_dist_sam_parse, psam.cu) against kombgpu_sam_parse on one GPU.

In one run, on N = 1, 2, 4, 8 GPUs (those the box has; one GPU per rank):
- the SAM pair of cfg2 (synth.metagenome_hits, 1 M unitigs, 5 M read pairs, synth.render_sam with @SQ headers), parsed
  by kombgpu_sam_parse on GPU 0 and by kombgpu_dist_sam_parse on N GPUs: per-stage CUDA-event times of every rank,
  the host time of the call, GB/s of SAM text over that host time, and whether the unitig count and names (vid by vid),
  the hit and read counts and the multiset of per-read unitig lists equal the single-GPU result;
- bin/komb2 with KOMB_GPU_DEVICES=0..N-1, the default (partitioned parse) against KOMB_TOKENIZE=host: wall time of
  each and whether the three files are byte-identical;
- with --big and enough host RAM: a SAM pair with more than 2^30 lines (short records over a few keys and names),
  which kombgpu_sam_parse rejects and kombgpu_dist_sam_parse on 2 GPUs or more takes, with its time.
Each parse runs twice; the first includes module loading.  The card's name and power limit are read in the same run.

    python tools/dist_sam_probe.py --out profiles/dist_sam_probe.json [--big]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import torch  # noqa: E402

import komb_b200  # noqa: E402
from komb_b200 import synth  # noqa: E402
from komb_b200.peer import DistHits, run_local  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q or ["unknown"]


def read_signature(rk, ut):
    """Sorted (hits, sum of mixed unitig ids, sum of another mix) per read: equal for equal multisets of per-read lists."""
    if rk.size == 0:
        return np.zeros((0, 3), np.uint64)
    o = np.argsort(rk, kind="stable")
    r, u = rk[o], ut[o].astype(np.uint64)
    starts = np.flatnonzero(np.r_[True, r[1:] != r[:-1]])
    with np.errstate(over="ignore"):
        m1 = (u + np.uint64(0x9E3779B97F4A7C15)) * np.uint64(0xBF58476D1CE4E5B9)
        m2 = (u ^ np.uint64(0x94D049BB133111EB)) * np.uint64(0xD6E8FEB86659FD93)
        m1 ^= m1 >> np.uint64(31)
        m2 ^= m2 >> np.uint64(29)
    cnt = np.diff(np.r_[starts, r.size]).astype(np.uint64)
    sig = np.stack([cnt, np.add.reduceat(m1, starts), np.add.reduceat(m2, starts)], axis=1)
    return sig[np.lexsort(sig.T[::-1])]


def single(texts):
    ctx = komb_b200.Context(0)
    out = {"runs": []}
    try:
        for _ in range(2):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with ctx.sam_parse(texts) as h:
                c = h.counts()
                ms = (time.perf_counter() - t0) * 1e3
                out["runs"].append({"host_ms": ms, **h.timing()})
                last = (c, h.names(), *h.download())
    finally:
        ctx.close()
    c, names, rk, ut = last
    return out, c, names, read_signature(rk, ut)


def dist(texts, world, check):
    def body(comm):
        runs = []
        for rep in range(2):
            torch.cuda.synchronize(comm.ctx.device)
            t0 = time.perf_counter()
            with DistHits.parse(comm, texts) as h:
                c = h.counts()
                runs.append({"host_ms": (time.perf_counter() - t0) * 1e3, **h.timing()})
                if rep == 1 and check:
                    return {"runs": runs, "counts": c, "range": h.local_range(), "names": h.names(), "hits": h.hits()}
        return {"runs": runs, "counts": c}
    return run_local(world, body, devices=list(range(world)))


def cfg2_pair(quick):
    n_u, n_p = (20_000, 100_000) if quick else (1_000_000, 5_000_000)
    m1, m2 = synth.metagenome_hits(n_u, n_p)
    return [synth.render_sam(m1, n_u, 1), synth.render_sam(m2, n_u, 2)]


def komb2_runs(texts, world, tmp):
    d = Path(tmp)
    (d / "r1.sam").write_bytes(texts[0])
    (d / "r2.sam").write_bytes(texts[1])
    (d / "u.fasta").write_bytes(b">0\nACGT\n")
    res = {}
    for mode, extra in (("default", {}), ("host", {"KOMB_TOKENIZE": "host"})):
        out = d / f"out_{mode}"
        out.mkdir(exist_ok=True)
        env = dict(os.environ, KOMB_GPU_DEVICES=",".join(str(i) for i in range(world)), **extra)
        t0 = time.perf_counter()
        cp = subprocess.run([str(ROOT / "bin" / "komb2"), "-t", "16", "-l", "100", "-o", str(out), "-i", str(d / "r1.sam"),
                             "-j", str(d / "r2.sam"), "-u", str(d / "u.fasta")], env=env, capture_output=True, text=True)
        res[mode] = {"wall_s": time.perf_counter() - t0, "rc": cp.returncode, "stderr_tail": cp.stderr[-400:]}
    res["files_identical"] = all((d / "out_default" / f).read_bytes() == (d / "out_host" / f).read_bytes()
                                 for f in ("edgelist.txt", "kcore.tsv", "CoreA_anomaly.txt"))
    return res


def big_pair(n_lines):
    """Short records over 997 keys and 1009 names: more than 2^30 lines in one file, few distinct strings."""
    block = b"".join(b"%d/1\t0\tu%d\n" % (i % 997, i % 1009) for i in range(1 << 16))
    reps = -(-n_lines // (1 << 16))
    return [block * reps, b""], reps << 16


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/dist_sam_probe.json")
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--big", action="store_true")
    args = ap.parse_args()
    n_dev = torch.cuda.device_count()
    report = {"card": card(), "devices": n_dev}
    texts = cfg2_pair(args.quick)
    n_bytes = sum(len(t) for t in texts)
    report["cfg2"] = {"sam_bytes": n_bytes}
    s_runs, s_counts, s_names, s_sig = single(texts)
    s_runs["gb_per_s"] = n_bytes / (s_runs["runs"][-1]["host_ms"] * 1e-3) / 1e9
    report["cfg2"]["single"] = {**s_runs, "counts": s_counts}
    print(json.dumps({"single": report["cfg2"]["single"]}), flush=True)
    for world in [w for w in (1, 2, 4, 8) if w <= n_dev]:
        parts = dist(texts, world, check=True)
        names = [n for p in sorted(parts, key=lambda p: p["range"]) for n in p["names"]]
        sig = read_signature(np.concatenate([p["hits"][0] for p in parts]), np.concatenate([p["hits"][1] for p in parts]))
        c = parts[0]["counts"]
        host_ms = max(p["runs"][-1]["host_ms"] for p in parts)
        row = {"world": world, "host_ms": host_ms, "gb_per_s": n_bytes / (host_ms * 1e-3) / 1e9,
               "ranks": [p["runs"] for p in parts],
               "same_as_single": {"n_unitigs": c["n_unitigs"] == s_counts["n_unitigs"], "names": names == s_names,
                                  "counts": (c["n_hits"], c["n_reads"], c["n_lines"]) == (s_counts["n_hits"], s_counts["n_reads"], s_counts["n_lines"]),
                                  "per_read_unitigs": bool(sig.shape == s_sig.shape and np.array_equal(sig, s_sig))}}
        with tempfile.TemporaryDirectory() as tmp:
            row["komb2"] = komb2_runs(texts, world, tmp) if world >= 2 else None
        report["cfg2"].setdefault("dist", []).append(row)
        print(json.dumps({k: row[k] for k in ("world", "host_ms", "gb_per_s", "same_as_single", "komb2")}), flush=True)
    if args.big:
        mem = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_AVPHYS_PAGES")
        n_lines = (1 << 30) + (1 << 24)
        if mem < 64 << 30 or n_dev < 2:
            report["big"] = f"not measured: {mem >> 30} GiB free host RAM, {n_dev} GPUs"
        else:
            big, n_lines = big_pair(n_lines)
            big_rep = {"n_lines": n_lines, "sam_bytes": len(big[0])}
            ctx = komb_b200.Context(0)
            try:
                ctx.sam_parse(big).close()
                big_rep["single"] = "accepted"
            except komb_b200.KombGpuError as e:
                big_rep["single"] = f"rejected: {e}"
            finally:
                ctx.close()
            world = min(n_dev, 8)
            parts = dist(big, world, check=False)
            big_rep["dist"] = {"world": world, "host_ms": max(p["runs"][-1]["host_ms"] for p in parts), "counts": parts[0]["counts"],
                               "ranks": [p["runs"] for p in parts]}
            report["big"] = big_rep
        print(json.dumps({"big": report["big"]}), flush=True)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(report, indent=1, default=str))


if __name__ == "__main__":
    main()
