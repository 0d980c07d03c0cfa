"""Device times of the unitig FASTA path (include/kombgpu.h, unitig FASTA) at cfg2 and cfg3 sizes, and the wall-clock
cost of KOMB_UNITIG_FASTA in komb2 on the drop-in probe's SAM pair.

    python tools/unitig_fasta_probe.py [--sizes 1000000,50000000] [--komb2-pairs 625000]

Inputs are seeded synthetic FASTA files whose record names are the vertex names synth.render_sam writes (decimal ids);
sequence lengths 31 .. 20,000 (heavy-tailed), one record in ten wrapped at 60 columns.  The vertex names are joined
from a packed host table in a random vertex order.  Prints one JSON line: per size the CUDA-event times of upload,
index, join, selection (IQR fence over n random scores, score upload and mask download included) and extraction
(the anomalous records, and every record), bytes over time for index and extraction against the HBM peak bench.py
uses, and the card's name and power limit read in the same run."""
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

import komb_b200  # noqa: E402
from komb_b200 import synth  # noqa: E402


def hbm_peak():   # the same source bench.py reads
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def decimal_table(ids: np.ndarray):
    """Packed decimal strings of ids: (bytes as uint8 array, offsets[n + 1])."""
    ids = ids.astype(np.int64)
    nd = np.ones(ids.shape[0], np.int64)
    for k in range(1, 19):
        nd += ids >= 10 ** k
    off = np.zeros(ids.shape[0] + 1, np.int64)
    np.cumsum(nd, out=off[1:])
    out = np.empty(int(off[-1]), np.uint8)
    for d in range(int(nd.max())):
        m = d < nd
        out[off[:-1][m] + d] = 48 + (ids[m] // 10 ** (nd[m] - 1 - d)) % 10
    return out, off


def synth_fasta(n: int, seed: int) -> np.ndarray:
    """'>id\\n' + sequence + '\\n' for ids 0 .. n-1; every tenth record wrapped at 60 columns."""
    rng = np.random.default_rng(seed)
    length = np.minimum(31 + (rng.pareto(1.2, n) * 25).astype(np.int64), 20000)
    wrapped = (np.arange(n) % 10 == 0)
    body = length + np.where(wrapped, (length - 1) // 60, 0) + 1
    name, name_off = decimal_table(np.arange(n))
    head = (name_off[1:] - name_off[:-1]) + 2
    rec = head + body
    start = np.zeros(n + 1, np.int64)
    np.cumsum(rec, out=start[1:])
    buf = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(start[-1]), dtype=np.uint8)]
    buf[start[:-1]] = ord(">")
    nd = name_off[1:] - name_off[:-1]
    for d in range(int(nd.max())):
        m = d < nd
        buf[start[:-1][m] + 1 + d] = name[name_off[:-1][m] + d]
    buf[start[:-1] + head - 1] = 10
    buf[start[1:] - 1] = 10
    w = np.flatnonzero(wrapped & (length > 60))
    k = 1
    while w.size:
        buf[start[w] + head[w] + 61 * k - 1] = 10
        k += 1
        w = w[(length[w] - 1) // 60 >= k]
    return buf


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def probe_size(ctx, n: int, seed: int, peak: float) -> dict:
    """The whole sequence twice on the same input; the second pass is reported (kernels loaded, workspace cached), the
    first pass's index and extraction times as cold_*."""
    text = synth_fasta(n, seed)
    cold = probe_pass(ctx, text, n, seed, peak)
    r = probe_pass(ctx, text, n, seed, peak)
    r.update(cold_ms_index=cold["ms_index"], cold_ms_extract_all=cold["ms_extract_all"])
    return r


def probe_pass(ctx, text: np.ndarray, n: int, seed: int, peak: float) -> dict:
    import torch
    r = {"records": n, "fasta_bytes": len(text)}
    h = ctypes.c_void_p()   # straight from the numpy buffer: no second host copy of several GB
    ctx._check(ctx._lib.kombgpu_fasta_load(ctx._h, ctypes.c_char_p(text.ctypes.data), len(text), ctypes.byref(h)))
    fa = komb_b200.Fasta(ctx, h)
    t = fa.timing()
    r.update(ms_upload=t["ms_upload"], ms_index=t["ms_index"])
    perm = np.random.default_rng(seed + 1).permutation(n)
    names, off = decimal_table(perm)
    names, off = names.tobytes(), off.astype(np.uint64)
    miss = ctypes.c_uint32()
    ctx._check(ctx._lib.kombgpu_fasta_join_names(fa._h, names, ctypes.c_void_p(off.ctypes.data), n, ctypes.byref(miss)))
    assert miss.value == 0
    r["ms_join"] = fa.timing()["ms_join"]
    score = np.abs(np.random.default_rng(seed + 2).standard_normal(n)) ** 2
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    for _ in range(2):   # the first call warms up the sort's kernels
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        sel = ctx.anomalous(score)
        e1.record(stream)
        e1.synchronize()
    ctx.reset_stream()
    r.update(ms_select=e0.elapsed_time(e1), n_selected=sel["n_selected"])
    for what, mask in (("anomalous", sel["member"]), ("all", np.ones(n, bool))):
        out = fa.extract(mask)
        ms = fa.timing()["ms_extract"]
        r[f"ms_extract_{what}"] = ms
        r[f"extract_{what}_bytes"] = len(out)
        gbs = 2 * len(out) / (ms * 1e-3) / 1e9      # read + write of the copied records
        r[f"extract_{what}_gbs"] = gbs
        r[f"extract_{what}_frac_peak"] = gbs / peak
        del out
    index_bytes = 2 * len(text)                     # the count pass and the scan pass each read the text once
    r.update(index_bytes=index_bytes, index_gbs=index_bytes / (r["ms_index"] * 1e-3) / 1e9)
    r["index_frac_peak"] = r["index_gbs"] / peak
    r["kernel_launches"] = fa.timing()["kernel_launches"]
    fa.close()
    return r


def komb2_cost(pairs: int, threads: int) -> dict:
    """bin/komb2 on the drop-in probe's SAM pair (tests/probes/dropin_probe.py) with a FASTA of every unitig, without
    and with KOMB_UNITIG_FASTA=anomalous,truss, alternating, two runs each."""
    n = 1_000_000
    m1, m2 = synth.metagenome_hits(n, pairs, seed=11)
    res = {"pairs": pairs, "threads": threads, "runs": []}
    with tempfile.TemporaryDirectory() as d:
        d = Path(d)
        (d / "r1.sam").write_bytes(synth.render_sam(m1, n, 1, with_header=False))
        (d / "r2.sam").write_bytes(synth.render_sam(m2, n, 2, with_header=False))
        (d / "u.fasta").write_bytes(synth_fasta(n, 5).tobytes())
        for k in range(4):
            env = dict(os.environ)
            if k % 2:
                env["KOMB_UNITIG_FASTA"] = "anomalous,truss"
            out = d / f"out{k}"
            out.mkdir()
            t0 = time.perf_counter()
            cp = subprocess.run([str(ROOT / "bin" / "komb2"), "-t", str(threads), "-l", "100", "-o", str(out), "-i", str(d / "r1.sam"),
                                 "-j", str(d / "r2.sam"), "-u", str(d / "u.fasta")], capture_output=True, text=True, env=env)
            wall = time.perf_counter() - t0
            ana = re.search(r"analysis \(sec\) = ([0-9.]+)", cp.stdout)
            run = {"unitig_fasta": bool(k % 2), "rc": cp.returncode, "wall_s": round(wall, 3), "analysis_s": float(ana.group(1)) if ana else None}
            for f in ("anomalous_unitigs.fasta", "truss_unitigs.fasta"):
                if (out / f).exists():
                    run[f] = (out / f).stat().st_size
            if cp.returncode:
                run["stderr"] = cp.stderr[-500:]
            res["runs"].append(run)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000000,50000000")
    ap.add_argument("--komb2-pairs", type=int, default=625_000)
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 1)
    a = ap.parse_args()
    peak, peak_src = hbm_peak()
    ctx = komb_b200.Context(0)
    res = {"card": card(), "hbm_peak_gbs": peak, "peak_source": peak_src, "sizes": []}
    for k, n in enumerate(int(x) for x in a.sizes.split(",")):
        res["sizes"].append(probe_size(ctx, n, 100 + k, peak))
    ctx.close()
    if a.komb2_pairs:
        res["komb2"] = komb2_cost(a.komb2_pairs, a.threads)
    res["card_after"] = card()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
