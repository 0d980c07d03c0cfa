"""Time the radix sort alone (kombgpu_debug_sort_u64) on the key shapes the path sorts: sort_probe.py"""
import sys, ctypes, json
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import komb_b200
from komb_b200 import _lib
lib = _lib.load()
ctx = komb_b200.Context(0)
SHAPES = [("hits 20M (20+23 bits, reads in order)", 20_003_139, 20, 23, 1), ("pairs 33M (20+20 bits)", 32_866_974, 20, 20, 0),
          ("swapped 33M (20 bits high)", 32_850_322, 0, 20, 0), ("corea 1M (26 bits high)", 1_000_000, 0, 26, 0),
          ("pairs 540M (26+26 bits)", 540_000_000, 26, 26, 0),
          ("pairs 1.1G (20+20 bits, 64-bit status words)", 1_100_000_000, 20, 20, 0)]
for name, n, lo, hi, srt in SHAPES:
    ms, ok = ctypes.c_float(), ctypes.c_int()
    rc = lib.kombgpu_debug_sort_u64(ctx._h, n, lo, hi, srt, 3, ctypes.byref(ms), ctypes.byref(ok))
    passes = (lo + hi + 7) // 8
    gbs = passes * 16 * n / ms.value / 1e6 if rc == 0 else 0
    print(json.dumps({"shape": name, "rc": rc, "ok": ok.value, "ms": round(ms.value, 3), "passes": passes,
                      "GBs_rw_per_pass": round(gbs, 1)}), flush=True)
