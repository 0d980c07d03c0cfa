"""TEST INFRASTRUCTURE: the onion decomposition restated in C (tests/onion_ref.c), compiled on first use into a
temporary directory (the tree stays untouched), and the derivation of the coreness from a layering.  It lives beside
the tests rather than in oracle/komb_oracle.c because the oracle is pinned to the reference's own outputs and is kept
as it is; this restatement is pinned to networkx instead (tests/test_onion_cpu.py)."""
from __future__ import annotations

import ctypes
import os
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np

_SRC = Path(__file__).resolve().parent / "onion_ref.c"
_lib = None
_dir = None   # the compiled library's directory, removed when the process exits


def _load():
    global _lib, _dir
    if _lib is None:
        _dir = tempfile.TemporaryDirectory(prefix="onion_ref_")
        so = os.path.join(_dir.name, "libonion_ref.so")
        cc = os.environ.get("CC") or shutil.which("cc") or shutil.which("gcc")
        subprocess.run([cc, "-O2", "-std=c11", "-shared", "-fPIC", "-Wall", "-o", so, str(_SRC)], check=True, capture_output=True)
        L = ctypes.CDLL(so)
        L.onion_ref.restype = ctypes.c_longlong
        L.onion_ref.argtypes = [ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p]
        _lib = L
    return _lib


def simple_edges(u, v) -> tuple[np.ndarray, np.ndarray]:
    """(u, v) pairs -> the simple graph's edges: loops dropped, one (min, max) pair per edge, ascending."""
    u = np.asarray(u, np.uint64)
    v = np.asarray(v, np.uint64)
    keep = u != v
    a, b = np.minimum(u[keep], v[keep]), np.maximum(u[keep], v[keep])
    key = np.unique((a << np.uint64(32)) | b)
    return (key >> np.uint64(32)).astype(np.uint32), (key & np.uint64(0xffffffff)).astype(np.uint32)


def onion_layers(n: int, u, v) -> tuple[np.ndarray, np.ndarray, int]:
    """-> (layer uint32[n], coreness int32[n], number of layers) of the simple graph on n vertices with edges (u, v)."""
    a, b = simple_edges(u, v)
    layer = np.zeros(n, np.uint32)
    core = np.zeros(n, np.int32)
    rc = _load().onion_ref(n, a.ctypes.data, b.ctypes.data, a.shape[0], layer.ctypes.data, core.ctypes.data)
    if rc < 0:
        raise MemoryError("onion_ref")
    return layer, core, int(rc)


def coreness_from_layers(n: int, u, v, layer) -> np.ndarray:
    """The coreness a layering implies: a vertex's remaining degree when its layer is removed counts its neighbours in
    the same or later layers; a layer's level is the running maximum of those degrees over the layers up to it."""
    a, b = simple_edges(u, v)
    layer = np.asarray(layer, np.int64)
    if n == 0:
        return np.zeros(0, np.int32)
    rdeg = np.zeros(n, np.int64)
    np.add.at(rdeg, a, (layer[b] >= layer[a]).astype(np.int64))
    np.add.at(rdeg, b, (layer[a] >= layer[b]).astype(np.int64))
    n_layers = int(layer.max())
    per_layer = np.zeros(n_layers + 1, np.int64)
    np.maximum.at(per_layer, layer, rdeg)
    level = np.maximum.accumulate(per_layer)
    return level[layer].astype(np.int32)
