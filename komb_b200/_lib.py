"""ctypes binding of komb_b200/libkombgpu.so (the C ABI in include/kombgpu.h).

There is no fallback of any kind: if the shared library is missing, or no B200
is visible when a context is created, the caller gets an exception.
"""
from __future__ import annotations

import ctypes
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_uint32, c_uint64, c_void_p
from pathlib import Path

LIB_PATH = Path(__file__).resolve().parent / "libkombgpu.so"

OK, EINVAL, ENODEV, ENOMEM, ECUDA, ESTATE, EINTERNAL = 0, -1, -2, -3, -4, -5, -6
KEY_REF32, KEY_EXACT64 = 0, 1
ERROR_NAMES = {EINVAL: "KOMBGPU_EINVAL", ENODEV: "KOMBGPU_ENODEV", ENOMEM: "KOMBGPU_ENOMEM",
               ECUDA: "KOMBGPU_ECUDA", ESTATE: "KOMBGPU_ESTATE", EINTERNAL: "KOMBGPU_EINTERNAL"}


class Stats(ctypes.Structure):
    """struct kombgpu_stats"""
    _fields_ = [
        ("n_hits", c_uint64), ("n_unique_hits", c_uint64), ("n_pairs", c_uint64), ("n_edges", c_uint64),
        ("n_vertices", c_uint32), ("max_degree", c_int32), ("max_coreness", c_int32),
        ("peel_levels", c_uint32), ("peel_rounds", c_uint32),
        ("ms_build", c_float), ("ms_peel", c_float), ("ms_corea", c_float), ("ms_peel_kernel", c_float),
        ("kernel_launches", c_uint64),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


class DistStats(ctypes.Structure):
    """struct kombgpu_dist_stats"""
    _fields_ = [
        ("n_hits_local", c_uint64), ("n_pairs_local", c_uint64), ("n_pairs_received", c_uint64), ("n_fwd_local", c_uint64),
        ("n_directed_local", c_uint64), ("n_edges_global", c_uint64), ("n_messages_sent", c_uint64), ("n_messages_recv", c_uint64),
        ("n_global", c_uint32), ("v_lo", c_uint32), ("n_local", c_uint32),
        ("max_degree", c_int32), ("max_coreness", c_int32), ("peel_levels", c_uint32), ("peel_subrounds", c_uint32),
        ("peel_solo_subrounds", c_uint32),
        ("ms_build", c_float), ("ms_peel", c_float), ("ms_corea", c_float),
        ("ms_build_route", c_float), ("ms_build_sort", c_float), ("ms_build_csr", c_float), ("peel_async", c_uint32),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


# bootstrap all-gather callback of kombgpu_comm_create
ALLGATHER_FN = ctypes.CFUNCTYPE(c_int, c_void_p, c_void_p, c_void_p, c_uint64)

# every symbol include/kombgpu.h and include/kombgpu_debug.h declare: name -> (restype, argtypes)
u32p, u64p, i32p, f64p = POINTER(c_uint32), POINTER(c_uint64), POINTER(c_int32), POINTER(c_double)
SIGNATURES = {
    "kombgpu_abi_version": (c_int, []),
    "kombgpu_debug_sort_u64": (c_int, [c_void_p, c_uint64, c_int, c_int, c_int, c_int, POINTER(c_float), POINTER(c_int)]),
    "kombgpu_ctx_create": (c_int, [c_int, POINTER(c_void_p)]),
    "kombgpu_ctx_destroy": (None, [c_void_p]),
    "kombgpu_ctx_set_stream": (c_int, [c_void_p, c_void_p]),
    "kombgpu_ctx_reset_stream": (c_int, [c_void_p]),
    "kombgpu_last_error": (c_char_p, [c_void_p]),
    "kombgpu_ctx_trim": (c_int, [c_void_p]),
    "kombgpu_ctx_launches": (c_int, [c_void_p, POINTER(c_uint64)]),
    "kombgpu_pinned_alloc": (c_int, [c_void_p, c_uint64, POINTER(c_void_p)]),
    "kombgpu_pinned_free": (c_int, [c_void_p, c_void_p]),
    "kombgpu_build_graph": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint32, POINTER(c_void_p)]),
    "kombgpu_build_graph_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint32, POINTER(c_void_p)]),
    "kombgpu_graph_from_edges": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint32, POINTER(c_void_p)]),
    "kombgpu_graph_from_edges_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint32, POINTER(c_void_p)]),
    "kombgpu_graph_from_csr_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_uint32, POINTER(c_void_p)]),
    "kombgpu_graph_destroy": (None, [c_void_p]),
    "kombgpu_graph_counts": (c_int, [c_void_p, POINTER(c_uint32), POINTER(c_uint64)]),
    "kombgpu_graph_edges": (c_int, [c_void_p, c_void_p, c_void_p]),
    "kombgpu_graph_csr": (c_int, [c_void_p, c_void_p, c_void_p]),
    "kombgpu_graph_edges_csr": (c_int, [c_void_p, c_void_p, c_void_p]),
    "kombgpu_graph_edge_multiplicity": (c_int, [c_void_p, c_void_p]),
    "kombgpu_graph_results_csr": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "kombgpu_analyse_hits_csr": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint32, c_int, c_uint64, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_void_p, POINTER(c_void_p)]),
    "kombgpu_debug_peel_again": (c_int, [c_void_p]),
    "kombgpu_debug_build_chunks": (c_int, [c_void_p, POINTER(c_uint32)]),
    "kombgpu_debug_dist_build_rounds": (c_int, [c_void_p, POINTER(c_uint32)]),
    "kombgpu_debug_dist_truss_timing": (c_int, [c_void_p, POINTER(c_float), POINTER(c_float), POINTER(c_float)]),
    "kombgpu_degree": (c_int, [c_void_p, c_void_p]),
    "kombgpu_coreness": (c_int, [c_void_p, c_void_p]),
    "kombgpu_corea": (c_int, [c_void_p, c_void_p, c_void_p, c_uint32, c_int, c_void_p]),
    "kombgpu_graph_corea": (c_int, [c_void_p, c_int, c_void_p]),
    "kombgpu_graph_summary": (c_int, [c_void_p, POINTER(c_int32), POINTER(c_double)]),
    "kombgpu_analyse_hits": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint32, c_int, c_uint64, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, POINTER(c_void_p)]),
    "kombgpu_graph_densest_core": (c_int, [c_void_p, POINTER(c_int32), POINTER(c_uint32), POINTER(c_uint64), POINTER(c_double)]),
    "kombgpu_graph_densest_block": (c_int, [c_void_p, c_void_p, c_int, c_double, POINTER(c_uint32), POINTER(c_uint64), POINTER(c_double),
                                            POINTER(c_double), POINTER(c_uint32), c_void_p]),
    "kombgpu_graph_analyse": (c_int, [c_void_p, c_int]),
    "kombgpu_graph_max_core_truss": (c_int, [c_void_p, POINTER(c_uint32), POINTER(c_uint64), POINTER(c_int32), POINTER(c_uint32)]),
    "kombgpu_graph_max_core_edges": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "kombgpu_graph_truss_vertices": (c_int, [c_void_p, c_void_p]),
    "kombgpu_graph_onion": (c_int, [c_void_p, c_void_p, POINTER(c_uint32)]),
    "kombgpu_debug_onion_again": (c_int, [c_void_p]),
    "kombgpu_debug_onion_timing": (c_int, [c_void_p, POINTER(c_float), POINTER(c_uint32), POINTER(c_uint32), POINTER(c_uint32)]),
    "kombgpu_debug_dist_onion_again": (c_int, [c_void_p]),
    "kombgpu_debug_dist_onion_timing": (c_int, [c_void_p, POINTER(c_float), POINTER(c_uint32), POINTER(c_uint32), POINTER(c_uint32),
                                                POINTER(c_float)]),
    "kombgpu_graph_results": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "kombgpu_graph_stats": (c_int, [c_void_p, POINTER(Stats)]),
    "kombgpu_graph_device_arrays": (c_int, [c_void_p] + [POINTER(c_void_p)] * 6),
    # SAM text -> hits on the device
    "kombgpu_sam_parse": (c_int, [c_void_p, POINTER(c_char_p), POINTER(c_uint64), c_int, POINTER(c_void_p)]),
    "kombgpu_hits_destroy": (None, [c_void_p]),
    "kombgpu_hits_counts": (c_int, [c_void_p, POINTER(c_uint64), POINTER(c_uint32), POINTER(c_uint32), POINTER(c_uint64)]),
    "kombgpu_hits_names": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "kombgpu_hits_download": (c_int, [c_void_p, c_void_p, c_void_p]),
    "kombgpu_hits_device_arrays": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_void_p)]),
    "kombgpu_hits_timing": (c_int, [c_void_p, POINTER(c_float), POINTER(c_float), POINTER(c_uint64), POINTER(c_int)]),
    "kombgpu_build_graph_hits": (c_int, [c_void_p, POINTER(c_void_p)]),
    # output files formatted on the device
    "kombgpu_graph_format": (c_int, [c_void_p, c_int, c_void_p, POINTER(c_uint64)]),
    "kombgpu_graph_format_fetch": (c_int, [c_void_p, c_int, c_void_p, c_int]),
    "kombgpu_graph_format_wait": (c_int, [c_void_p]),
    "kombgpu_format_corea": (c_int, [c_void_p, c_void_p, c_uint32, c_void_p, c_uint64, POINTER(c_uint64)]),
    # the unitig FASTA: index, join, anomalous selection, extraction
    "kombgpu_fasta_load": (c_int, [c_void_p, c_char_p, c_uint64, POINTER(c_void_p)]),
    "kombgpu_fasta_destroy": (None, [c_void_p]),
    "kombgpu_fasta_counts": (c_int, [c_void_p, POINTER(c_uint32), POINTER(c_uint64)]),
    "kombgpu_fasta_join_hits": (c_int, [c_void_p, c_void_p, POINTER(c_uint32)]),
    "kombgpu_fasta_join_names": (c_int, [c_void_p, c_char_p, c_void_p, c_uint32, POINTER(c_uint32)]),
    "kombgpu_fasta_extract": (c_int, [c_void_p, c_void_p, c_uint32, POINTER(c_uint64)]),
    "kombgpu_fasta_extract_fetch": (c_int, [c_void_p, c_void_p]),
    "kombgpu_fasta_timing": (c_int, [c_void_p, POINTER(c_float), POINTER(c_float), POINTER(c_float), POINTER(c_float), POINTER(c_uint64)]),
    "kombgpu_anomalous": (c_int, [c_void_p, c_void_p, c_uint32, c_double, POINTER(c_double), POINTER(c_double), POINTER(c_double),
                                  POINTER(c_uint32), c_void_p]),
    "kombgpu_graph_anomalous": (c_int, [c_void_p, c_double, POINTER(c_double), POINTER(c_double), POINTER(c_double), POINTER(c_uint32),
                                        c_void_p]),
    # multi-GPU partition interface
    "kombgpu_local_edges_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint32, POINTER(c_void_p)]),
    "kombgpu_edgeset_from_pairs_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint32, POINTER(c_void_p)]),
    "kombgpu_edgeset_counts": (c_int, [c_void_p, POINTER(c_uint64), POINTER(c_uint64), POINTER(c_uint64)]),
    "kombgpu_edgeset_route_dev": (c_int, [c_void_p, POINTER(c_uint32), c_int, c_void_p, POINTER(c_uint64)]),
    "kombgpu_edgeset_destroy": (None, [c_void_p]),
    "kombgpu_part_build_dev": (c_int, [c_void_p, c_void_p, c_uint64, c_uint32, c_uint32, c_uint32, POINTER(c_void_p)]),
    "kombgpu_part_destroy": (None, [c_void_p]),
    "kombgpu_part_counts": (c_int, [c_void_p, POINTER(c_uint32), POINTER(c_uint64), POINTER(c_int32)]),
    "kombgpu_part_device_arrays": (c_int, [c_void_p] + [POINTER(c_void_p)] * 4),
    "kombgpu_part_peel_begin": (c_int, [c_void_p]),
    "kombgpu_part_peel_scan": (c_int, [c_void_p, c_int32, POINTER(c_uint32), POINTER(c_uint32), POINTER(c_int32)]),
    "kombgpu_part_peel_process": (c_int, [c_void_p, c_int32, POINTER(c_uint32)]),
    "kombgpu_part_outbox_route_dev": (c_int, [c_void_p, POINTER(c_uint32), c_int, c_void_p, POINTER(c_uint64)]),
    "kombgpu_part_peel_apply_dev": (c_int, [c_void_p, c_int32, c_void_p, c_uint64, POINTER(c_uint32)]),
    "kombgpu_corea_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_uint32, c_int, c_void_p, POINTER(c_double)]),
    # multi-GPU, peer-memory path
    "kombgpu_comm_create": (c_int, [c_void_p, c_int, c_int, ALLGATHER_FN, c_void_p, c_uint64, POINTER(c_void_p)]),
    "kombgpu_comm_create_local": (c_int, [c_void_p, c_int, c_int, POINTER(c_void_p), c_uint64, POINTER(c_void_p)]),
    "kombgpu_comm_destroy": (None, [c_void_p]),
    "kombgpu_comm_abort": (c_int, [c_void_p]),
    "kombgpu_comm_info": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_uint64)]),
    "kombgpu_dist_build_hits_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint32, POINTER(c_void_p)]),
    "kombgpu_dist_build_pairs_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint32, POINTER(c_void_p)]),
    "kombgpu_dist_build_hits": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint32, POINTER(c_void_p)]),
    "kombgpu_dist_build_pairs": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint32, POINTER(c_void_p)]),
    "kombgpu_dist_coreness": (c_int, [c_void_p]),
    "kombgpu_dist_corea": (c_int, [c_void_p, c_int]),
    "kombgpu_dist_graph_destroy": (None, [c_void_p]),
    "kombgpu_dist_graph_stats": (c_int, [c_void_p, POINTER(DistStats)]),
    "kombgpu_dist_graph_results": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "kombgpu_dist_graph_edges": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "kombgpu_dist_graph_edges_csr": (c_int, [c_void_p, c_void_p, c_void_p]),
    "kombgpu_dist_graph_device_arrays": (c_int, [c_void_p] + [POINTER(c_void_p)] * 6),
    "kombgpu_dist_graph_summary": (c_int, [c_void_p, POINTER(c_int32), POINTER(c_double)]),
    "kombgpu_dist_max_core_truss": (c_int, [c_void_p, POINTER(c_uint32), POINTER(c_uint64), POINTER(c_int32), POINTER(c_uint32)]),
    "kombgpu_dist_max_core_edges": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "kombgpu_dist_truss_vertices": (c_int, [c_void_p, c_void_p]),
    "kombgpu_dist_densest_core": (c_int, [c_void_p, POINTER(c_int32), POINTER(c_uint32), POINTER(c_uint64), POINTER(c_double)]),
    "kombgpu_dist_densest_block": (c_int, [c_void_p, c_void_p, c_int, c_double, POINTER(c_uint32), POINTER(c_uint64), POINTER(c_double),
                                           POINTER(c_double), POINTER(c_uint32), c_void_p]),
    "kombgpu_dist_sam_parse": (c_int, [c_void_p, POINTER(c_char_p), POINTER(c_uint64), c_int, POINTER(c_void_p)]),
    "kombgpu_dist_hits_destroy": (None, [c_void_p]),
    "kombgpu_dist_hits_counts": (c_int, [c_void_p, POINTER(c_uint64), POINTER(c_uint64), POINTER(c_uint32), POINTER(c_uint32),
                                         POINTER(c_uint64)]),
    "kombgpu_dist_hits_names": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "kombgpu_dist_hits_download": (c_int, [c_void_p, c_void_p, c_void_p]),
    "kombgpu_dist_hits_device_arrays": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_void_p)]),
    "kombgpu_dist_hits_timing": (c_int, [c_void_p, POINTER(c_float), POINTER(c_float), POINTER(c_float), POINTER(c_float), POINTER(c_int)]),
    "kombgpu_dist_build_graph_hits": (c_int, [c_void_p, POINTER(c_void_p)]),
    "kombgpu_dist_graph_format": (c_int, [c_void_p, c_int, c_void_p, POINTER(c_uint64)]),
    "kombgpu_dist_graph_format_fetch": (c_int, [c_void_p, c_int, c_void_p, c_int]),
    "kombgpu_dist_graph_format_wait": (c_int, [c_void_p]),
    "kombgpu_dist_onion": (c_int, [c_void_p, c_void_p, POINTER(c_uint32)]),
    "kombgpu_dist_fasta_load": (c_int, [c_void_p, c_char_p, c_uint64, POINTER(c_void_p)]),
    "kombgpu_dist_fasta_destroy": (None, [c_void_p]),
    "kombgpu_dist_fasta_counts": (c_int, [c_void_p, POINTER(c_uint32), POINTER(c_uint32), POINTER(c_uint32), POINTER(c_uint64),
                                          POINTER(c_uint64)]),
    "kombgpu_dist_fasta_join_hits": (c_int, [c_void_p, c_void_p, POINTER(c_uint32)]),
    "kombgpu_dist_fasta_join_names": (c_int, [c_void_p, c_char_p, c_void_p, c_uint32, POINTER(c_uint32)]),
    "kombgpu_dist_fasta_extract": (c_int, [c_void_p, c_void_p, c_uint32, POINTER(c_uint64)]),
    "kombgpu_dist_fasta_extract_fetch": (c_int, [c_void_p, c_void_p]),
    "kombgpu_dist_fasta_timing": (c_int, [c_void_p, POINTER(c_float), POINTER(c_float), POINTER(c_float), POINTER(c_float),
                                          POINTER(c_uint64)]),
    "kombgpu_dist_anomalous": (c_int, [c_void_p, c_double, POINTER(c_double), POINTER(c_double), POINTER(c_double), POINTER(c_uint32),
                                       c_void_p]),
}

_lib = None


class KombGpuError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"{ERROR_NAMES.get(code, code)}: {message}")
        self.code = code


def load() -> ctypes.CDLL:
    """Load libkombgpu.so and bind every declared symbol (no CUDA call is made)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA extension is not built. Run `make` (or "
                "`python -c 'import __graft_entry__ as e; e.build()'`). There is no CPU fallback.")
        lib = ctypes.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the ABI lost a symbol
            fn.restype = res
            fn.argtypes = args
        if lib.kombgpu_abi_version() != 1:
            raise RuntimeError("libkombgpu.so ABI version mismatch")
        _lib = lib
    return _lib
