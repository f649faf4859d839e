"""ctypes binding of libbbq_b200.so (include/bbq_b200.h).  Fails loudly: no CPU fallback exists.

The library is built in-tree by build_library() (nvcc, sm_100a) so it travels with the repo snapshot.
"""
from __future__ import annotations

import ctypes as C
import glob
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(_HERE, "libbbq_b200.so")
HEADER = os.path.join(_HERE, "..", "include", "bbq_b200.h")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "--fmad=false", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]
SOURCES = ["bbq_api.cu"]


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA library for sm_100a (cross-compiles without a GPU)."""
    deps = sorted(glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cuh"))) + [HEADER]
    stale = force or not os.path.exists(LIB_PATH) or any(
        os.path.getmtime(d) > os.path.getmtime(LIB_PATH) for d in deps)
    if stale:
        nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
              ["-o", LIB_PATH] + [os.path.join(CSRC, s) for s in SOURCES]
        subprocess.check_call(cmd)
    return LIB_PATH


class BbqConfig(C.Structure):
    _fields_ = [("query_bits", C.c_uint32), ("index_bits", C.c_uint32), ("similarity", C.c_uint32),
                ("iters", C.c_uint32), ("lambda_", C.c_double), ("device", C.c_int32), ("reserved", C.c_uint32)]


class BbqStats(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("last_candidates", C.c_uint64), ("last_path", C.c_uint32),
                ("last_overflow", C.c_uint32), ("last_engine", C.c_uint32), ("mma_layout", C.c_uint32),
                ("scan_launches", C.c_uint64), ("scan_ms", C.c_double),
                ("quantize_ms", C.c_double), ("select_ms", C.c_double), ("sample_ms", C.c_double),
                ("mma_n_tile", C.c_uint32), ("mma_passes", C.c_uint32), ("graph_replays", C.c_uint64)]


# every symbol include/bbq_b200.h declares: name -> (restype, argtypes)
_vp, _f32p, _u8p, _f64p, _i32p, _u32p = (C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_uint8),
                                         C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint32))
SYMBOLS = {
    "bbq_abi_version": (C.c_int, []),
    "bbq_create": (C.c_int, [C.POINTER(BbqConfig), C.POINTER(_vp)]),
    "bbq_destroy": (None, [_vp]),
    "bbq_last_error": (C.c_char_p, []),
    "bbq_last_error_pos": (None, [C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "bbq_index_build": (C.c_int, [_vp, _vp, C.c_uint64, C.c_uint32, _vp, C.POINTER(_vp)]),
    "bbq_index_build_device": (C.c_int, [_vp, _vp, C.c_uint64, C.c_uint32, _vp, C.POINTER(_vp)]),
    "bbq_index_reserve": (C.c_int, [_vp, C.c_uint64, C.c_uint32, _vp, C.POINTER(_vp)]),
    "bbq_index_append": (C.c_int, [_vp, _vp, C.c_uint64]),
    "bbq_index_append_device": (C.c_int, [_vp, _vp, C.c_uint64]),
    "bbq_centroid_accumulate": (C.c_int, [_vp, _vp, C.c_uint64, C.c_uint32, C.c_uint64, _vp]),
    "bbq_centroid_accumulate_device": (C.c_int, [_vp, _vp, C.c_uint64, C.c_uint32, C.c_uint64, _vp]),
    "bbq_centroid_finish": (C.c_int, [_vp, C.c_uint32, C.c_uint64, _vp]),
    "bbq_index_build_sharded": (C.c_int, [_vp, _vp, C.c_uint64, C.c_uint32, _vp, C.POINTER(_vp)]),
    "bbq_index_build_sharded_device": (C.c_int, [_vp, _vp, C.c_uint64, C.c_uint32, _vp, C.POINTER(_vp)]),
    "bbq_index_from_quantized": (C.c_int, [_vp, _vp, _vp, _vp, C.c_uint64, C.c_uint32, C.POINTER(_vp)]),
    "bbq_index_size": (C.c_uint64, [_vp]),
    "bbq_index_dim": (C.c_uint32, [_vp]),
    "bbq_index_centroid": (C.c_int, [_vp, _vp, C.POINTER(C.c_double)]),
    "bbq_index_export": (C.c_int, [_vp, C.c_uint64, C.c_uint64, _vp, _vp]),
    "bbq_index_set_base": (C.c_int, [_vp, C.c_uint64]),
    "bbq_index_save": (C.c_int, [_vp, C.c_char_p, C.c_char_p]),
    "bbq_index_load": (C.c_int, [_vp, C.c_char_p, C.c_char_p, C.POINTER(_vp)]),
    "bbq_index_load_rows": (C.c_int, [_vp, C.c_char_p, C.c_char_p, C.c_uint64, C.c_uint64, C.POINTER(_vp), _vp]),
    "bbq_index_write_rows": (C.c_int, [_vp, C.c_char_p, C.c_uint64, _vp]),
    "bbq_index_write_meta": (C.c_int, [_vp, C.c_char_p, C.c_uint64, _vp]),
    "bbq_index_save_sharded": (C.c_int, [_vp, C.c_char_p, C.c_char_p]),
    "bbq_index_load_sharded": (C.c_int, [_vp, C.c_char_p, C.c_char_p, C.POINTER(_vp)]),
    "bbq_index_destroy": (None, [_vp]),
    "bbq_search": (C.c_int, [_vp, _vp, C.c_uint32, C.c_int64, _vp, _vp, C.POINTER(C.c_uint32)]),
    "bbq_search_device": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, _vp, _vp, _vp]),
    "bbq_index_attach_rows": (C.c_int, [_vp, _vp]),
    "bbq_index_attach_rows_device": (C.c_int, [_vp, _vp]),
    "bbq_search_rerank": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, _vp, _vp, _vp, C.POINTER(C.c_uint32)]),
    "bbq_search_rerank_sharded": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, _vp, _vp, _vp,
                                            C.POINTER(C.c_uint32)]),
    "bbq_rerank_owned_device": (C.c_int, [_vp, _vp, C.c_uint32, _vp, C.c_uint32, _vp, _vp]),
    "bbq_merge_topk_device": (C.c_int, [_vp, _vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, _vp, _vp, _vp]),
    "bbq_debug_quantize_query": (C.c_int, [_vp, _vp, _vp, _vp]),
    "bbq_debug_qcdist": (C.c_int, [_vp, _vp, _vp]),
    "bbq_debug_qcdist_batch": (C.c_int, [_vp, _vp, C.c_uint32, _vp]),
    "bbq_comm_unique_id": (C.c_int, [_vp]),
    "bbq_comm_init": (C.c_int, [_vp, _vp, C.c_int, C.c_int]),
    "bbq_comm_destroy": (C.c_int, [_vp]),
    "bbq_comm_info": (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "bbq_search_sharded": (C.c_int, [_vp, _vp, C.c_uint32, C.c_int64, _vp, _vp, C.POINTER(C.c_uint32)]),
    "bbq_search_sharded_device": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, _vp, _vp, _vp]),
    "bbq_quantize_query": (C.c_int, [_vp, _vp, _vp, C.c_uint32, _vp, _vp]),
    "bbq_quantization_accuracy": (C.c_int, [_vp, _vp, _vp, C.c_uint64, C.c_uint32, C.c_uint64, _vp]),
    "bbq_host_alloc": (C.c_void_p, [C.c_size_t]),
    "bbq_host_free": (None, [_vp]),
    "bbq_debug_scores": (C.c_int, [_vp, _vp, _vp]),
    "bbq_get_stats": (C.c_int, [_vp, C.POINTER(BbqStats)]),
    "bbq_set_profiling": (C.c_int, [_vp, C.c_int]),
    "bbq_reset_profiling": (C.c_int, [_vp]),
    "bbq_debug_trace": (C.c_int, [_vp, _vp, C.c_uint32]),
}

_lib = None


def load():
    """dlopen the library and bind every declared symbol; raises if it is missing (never falls back)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with better-binary-quantization_b200/_native.build_library() "
                "(python -c 'import __graft_entry__ as g; g.build()').  There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the export is missing
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib
