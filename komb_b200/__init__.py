"""komb_b200 — B200-native (sm_100a) implementation of KOMB's graph-analysis hot
path: alignment hits -> unitig adjacency graph -> k-core -> CORE-A score.

`komb_b200.api` is the Python face of the C ABI in include/kombgpu.h;
`komb_b200.synth` generates the synthetic workloads of BASELINE.json.
"""
from . import synth  # noqa: F401
from ._lib import KEY_EXACT64, KEY_REF32, KombGpuError  # noqa: F401
from .api import Context, Fasta, Graph  # noqa: F401

__all__ = ["Context", "Graph", "KombGpuError", "KEY_REF32", "KEY_EXACT64", "synth"]
