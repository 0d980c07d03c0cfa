"""One sort of the 33M-pair shape (for ncu): sort_probe_one.py"""
import sys, ctypes
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import komb_b200
from komb_b200 import _lib
lib = _lib.load(); ctx = komb_b200.Context(0)
ms, ok = ctypes.c_float(), ctypes.c_int()
print(lib.kombgpu_debug_sort_u64(ctx._h, 32_866_974, 20, 20, 0, 1, ctypes.byref(ms), ctypes.byref(ok)), ms.value, ok.value)
