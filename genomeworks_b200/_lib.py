"""Loader for the in-tree C-ABI library (genomeworks_b200/libgwb200.so, declared in include/gwb200.h).

There is no CPU fallback anywhere in this package: if the library is missing the import of any public
class fails loudly with the build instruction (python -c 'import __graft_entry__ as g; g.build()').
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GWB200_LIB_PATH") or os.path.join(_HERE, "libgwb200.so")  # env override: profiling builds only
_lib = None

E_INVALID_ARGUMENT = -1
E_RUNTIME = -2
E_CUDA = -3
E_BAD_ALLOC = -4


class PoaConfig(C.Structure):
    """gwb200_poa_config == cudapoa::BatchConfig (batch.hpp:60-86)."""
    _fields_ = [
        ("max_sequence_size", C.c_int32),
        ("max_consensus_size", C.c_int32),
        ("max_nodes_per_graph", C.c_int32),
        ("matrix_sequence_dimension", C.c_int32),
        ("alignment_band_width", C.c_int32),
        ("max_sequences_per_poa", C.c_int32),
        ("band_mode", C.c_int32),
        ("max_banded_pred_distance", C.c_int32),
    ]


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "genomeworks_b200: %s is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    L.gwb200_last_error.restype = C.c_char_p
    L.gwb200_version.restype = C.c_char_p
    L.gwb200_kernel_launch_count.restype = C.c_int64
    L.gwb200_poa_batch_create.argtypes = [C.POINTER(C.c_void_p), C.c_int32, C.c_void_p, C.c_int64, C.c_int8, C.POINTER(PoaConfig),
                                          C.c_int16, C.c_int16, C.c_int16]
    L.gwb200_poa_batch_destroy.argtypes = [C.c_void_p]
    L.gwb200_poa_batch_destroy.restype = None
    L.gwb200_poa_batch_add_group.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_char_p), C.c_void_p, C.POINTER(C.c_int32),
                                             C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    L.gwb200_poa_batch_add_groups_flat.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.POINTER(C.c_int32)]
    for name in ("total_poas", "max_poas", "generate", "upload", "launch", "sync", "id", "reset", "score_bytes", "resident_windows"):
        getattr(L, "gwb200_poa_batch_" + name).argtypes = [C.c_void_p]
    L.gwb200_poa_batch_get_consensus.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.gwb200_poa_batch_get_msa.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.gwb200_poa_batch_get_graphs.argtypes = [C.c_void_p] + [C.c_void_p] * 7
    L.gwb200_poa_batch_last_cells.argtypes = [C.c_void_p]
    L.gwb200_poa_batch_last_cells.restype = C.c_int64
    L.gwb200_poa_batch_last_kernel_ms.argtypes = [C.c_void_p]
    L.gwb200_poa_batch_last_kernel_ms.restype = C.c_float
    L.gwb200_poa_batch_enable_timers.argtypes = [C.c_void_p, C.c_int32]
    L.gwb200_poa_batch_get_timers.argtypes = [C.c_void_p, C.c_void_p]
    L.gwb200_device_fdividef.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    if hasattr(L, "gwb200_aligner_create"):
        L.gwb200_aligner_create.argtypes = [C.POINTER(C.c_void_p), C.c_int32, C.c_void_p, C.c_int32, C.c_int64]
        L.gwb200_aligner_destroy.argtypes = [C.c_void_p]
        L.gwb200_aligner_destroy.restype = None
        L.gwb200_aligner_add_alignment.argtypes = [C.c_void_p, C.c_int32, C.c_char_p, C.c_int32, C.c_char_p, C.c_int32, C.c_int32, C.c_int32]
        for name in ("align_all", "sync_alignments", "num_alignments", "reset", "free_temporary_device_buffers"):
            getattr(L, "gwb200_aligner_" + name).argtypes = [C.c_void_p]
        L.gwb200_aligner_reset_max_bandwidth.argtypes = [C.c_void_p, C.c_int32]
        L.gwb200_aligner_result_info.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.gwb200_aligner_result_runs.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        L.gwb200_aligner_last_cells.argtypes = [C.c_void_p]
        L.gwb200_aligner_last_cells.restype = C.c_int64
        L.gwb200_aligner_last_kernel_ms.argtypes = [C.c_void_p]
        L.gwb200_aligner_last_kernel_ms.restype = C.c_float
    if hasattr(L, "gwb200_aligner_add_alignments"):
        L.gwb200_aligner_add_alignments.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32)]
        L.gwb200_aligner_results_flat.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]
    if hasattr(L, "gwb200_global_aligner_create"):
        L.gwb200_global_aligner_create.argtypes = [C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                                   C.c_void_p, C.c_void_p, C.c_void_p]
        L.gwb200_global_aligner_destroy.argtypes = [C.c_void_p]
        L.gwb200_global_aligner_destroy.restype = None
        L.gwb200_global_aligner_add_alignment.argtypes = [C.c_void_p, C.c_char_p, C.c_int32, C.c_char_p, C.c_int32, C.c_int32, C.c_int32]
        for name in ("align_all", "sync_alignments", "num_alignments", "reset"):
            getattr(L, "gwb200_global_aligner_" + name).argtypes = [C.c_void_p]
        L.gwb200_global_aligner_result_info.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.gwb200_global_aligner_result_states.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.gwb200_global_aligner_last_cells.argtypes = [C.c_void_p]
        L.gwb200_global_aligner_last_cells.restype = C.c_int64
        L.gwb200_global_aligner_last_kernel_ms.argtypes = [C.c_void_p]
        L.gwb200_global_aligner_last_kernel_ms.restype = C.c_float
    if hasattr(L, "gwb200_extender_create"):
        L.gwb200_extender_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(C.c_int32), C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                             C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.gwb200_extender_destroy.argtypes = [C.c_void_p]
        L.gwb200_extender_destroy.restype = None
        L.gwb200_extender_extend_host.argtypes = [C.c_void_p, C.POINTER(C.c_int8), C.c_int32, C.POINTER(C.c_int8), C.c_int32, C.c_int32,
                                                  C.c_void_p, C.c_int32]
        L.gwb200_extender_extend_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                                    C.c_int32, C.c_void_p, C.c_void_p]
        for name in ("sync", "reset"):
            getattr(L, "gwb200_extender_" + name).argtypes = [C.c_void_p]
        L.gwb200_extender_num_results.argtypes = [C.c_void_p]
        L.gwb200_extender_num_results.restype = C.c_int64
        L.gwb200_extender_get_results.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
        L.gwb200_extender_get_results.restype = C.c_int64
        L.gwb200_extender_last_kernel_ms.argtypes = [C.c_void_p]
        L.gwb200_extender_last_kernel_ms.restype = C.c_float
        L.gwb200_extender_last_positions.argtypes = [C.c_void_p]
        L.gwb200_extender_last_positions.restype = C.c_int64
    _lib = L
    return L


def last_error():
    return (lib().gwb200_last_error() or b"").decode()


def check(rc):
    """Maps negative C-ABI codes to the exception class the reference API would have thrown."""
    if rc >= 0:
        return rc
    msg = last_error()
    if rc == E_INVALID_ARGUMENT:
        raise ValueError(msg)
    if rc == E_BAD_ALLOC:
        raise MemoryError(msg)
    raise RuntimeError(msg)
