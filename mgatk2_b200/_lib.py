"""ctypes binding of libmgatk2_b200.so (include/mgatk2_b200.h). Fails loudly when the library is absent:
there is no CPU fallback for the product path."""
from __future__ import annotations

import ctypes
import os

from .batch import MgatkBatchC

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libmgatk2_b200.so")

EXPORTS = (
    "mgatk_abi_version", "mgatk_status_string", "mgatk_create", "mgatk_destroy", "mgatk_last_error",
    "mgatk_workspace_bytes", "mgatk_pileup_device", "mgatk_check_stats", "mgatk_pileup_host",
    "mgatk_filter_strand_bias_device", "mgatk_filter_strand_bias_u32_device", "mgatk_stream_begin_device", "mgatk_stream_finish_device",
    "mgatk_last_launch_count", "mgatk_last_stage_times", "mgatk_pileup_host_submit", "mgatk_pileup_host_wait",
    "mgatk_variant_stats_device", "mgatk_variant_cells_device",
    "mgatk_clone_knn_device", "mgatk_clone_snn_device", "mgatk_louvain_host", "mgatk_marker_ranks_device",
    "mgatk_deletion_scan_device",
)

N_PLANES = 11
FLAG_RAW_PILEUP = 1
FLAG_ACCUMULATE = 2
ABI_VERSION = 2


class ParamsC(ctypes.Structure):
    _fields_ = [
        ("min_baseq", ctypes.c_int32), ("min_mapq", ctypes.c_int32),
        ("min_distance_from_end", ctypes.c_int32), ("dedup_mode", ctypes.c_int32),
        ("max_strand_bias", ctypes.c_double), ("min_reads_per_cell", ctypes.c_int32),
        ("mito_length", ctypes.c_int32), ("n_cells", ctypes.c_int32), ("max_read_extent", ctypes.c_int32),
        ("flags", ctypes.c_int32),
    ]


class OutputsC(ctypes.Structure):
    _fields_ = [("planes", ctypes.c_void_p), ("cell_qc", ctypes.c_void_p), ("stats", ctypes.c_void_p),
                ("base_totals", ctypes.c_void_p), ("overflow", ctypes.c_void_p),
                ("overflow_capacity", ctypes.c_int64)]


class VariantSumsC(ctypes.Structure):
    """mgatk_variant_sums (128 bytes)."""
    _fields_ = [("sum_fwd", ctypes.c_uint64), ("sum_rev", ctypes.c_uint64), ("sum_cov", ctypes.c_uint64),
                ("sum_ff", ctypes.c_uint64), ("sum_rr", ctypes.c_uint64), ("sum_fr", ctypes.c_uint64),
                ("max_alt", ctypes.c_uint64), ("max_cov", ctypes.c_uint64),
                ("dev_sum", ctypes.c_double), ("dev_sq", ctypes.c_double),
                ("n_covered", ctypes.c_uint32), ("n_detected", ctypes.c_uint32), ("n_conf_detected", ctypes.c_uint32),
                ("n_strand", ctypes.c_uint32), ("n_over", ctypes.c_uint32 * 4), ("n_low", ctypes.c_uint32),
                ("ref", ctypes.c_int32), ("valid", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class ExtensionMissingError(RuntimeError):
    pass


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ExtensionMissingError(
            f"{LIB_PATH} is missing. The pileup path has no CPU fallback: build the CUDA library with "
            "`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc, targets sm_100a).")
    lib = ctypes.CDLL(LIB_PATH)
    missing = [s for s in EXPORTS if not hasattr(lib, s)]
    if missing:
        raise ExtensionMissingError(f"{LIB_PATH} lacks symbols {missing}")
    lib.mgatk_abi_version.restype = ctypes.c_int
    lib.mgatk_status_string.restype = ctypes.c_char_p
    lib.mgatk_status_string.argtypes = [ctypes.c_int]
    lib.mgatk_create.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int]
    lib.mgatk_destroy.argtypes = [ctypes.c_void_p]
    lib.mgatk_last_error.restype = ctypes.c_char_p
    lib.mgatk_last_error.argtypes = [ctypes.c_void_p]
    lib.mgatk_workspace_bytes.restype = ctypes.c_int64
    lib.mgatk_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32]
    lib.mgatk_pileup_device.argtypes = [ctypes.c_void_p, ctypes.POINTER(ParamsC), ctypes.POINTER(MgatkBatchC),
                                        ctypes.POINTER(OutputsC), ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]
    lib.mgatk_check_stats.argtypes = [ctypes.c_void_p]
    lib.mgatk_filter_strand_bias_device.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32,
                                                    ctypes.c_double, ctypes.c_void_p]
    lib.mgatk_filter_strand_bias_u32_device.argtypes = lib.mgatk_filter_strand_bias_device.argtypes
    lib.mgatk_pileup_host.argtypes = [ctypes.c_void_p, ctypes.POINTER(ParamsC), ctypes.POINTER(MgatkBatchC),
                                      ctypes.POINTER(OutputsC)]
    lib.mgatk_pileup_host_submit.argtypes = [ctypes.c_void_p, ctypes.POINTER(ParamsC), ctypes.POINTER(MgatkBatchC),
                                             ctypes.POINTER(OutputsC), ctypes.POINTER(ctypes.c_int64)]
    lib.mgatk_pileup_host_wait.argtypes = [ctypes.c_void_p, ctypes.c_int64]
    lib.mgatk_last_launch_count.restype = ctypes.c_int64
    lib.mgatk_last_launch_count.argtypes = [ctypes.c_void_p]
    lib.mgatk_last_stage_times.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_char_p),
                                           ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int)]
    lib.mgatk_variant_stats_device.argtypes = [ctypes.c_void_p, ctypes.POINTER(ParamsC), ctypes.POINTER(OutputsC),
                                               ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p]
    lib.mgatk_variant_cells_device.argtypes = [ctypes.c_void_p, ctypes.POINTER(ParamsC), ctypes.POINTER(OutputsC),
                                               ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p]
    lib.mgatk_clone_knn_device.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32,
                                           ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    lib.mgatk_clone_snn_device.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p,
                                           ctypes.c_void_p]
    lib.mgatk_louvain_host.argtypes = [ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_double,
                                       ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32)]
    lib.mgatk_marker_ranks_device.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32,
                                              ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p,
                                              ctypes.c_void_p]
    lib.mgatk_deletion_scan_device.argtypes = [ctypes.c_void_p, ctypes.POINTER(ParamsC), ctypes.POINTER(MgatkBatchC),
                                               ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32,
                                               ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                               ctypes.c_void_p]
    if lib.mgatk_abi_version() != ABI_VERSION:
        raise ExtensionMissingError(f"ABI mismatch: library {lib.mgatk_abi_version()}, binding {ABI_VERSION}")
    _lib = lib
    return lib
