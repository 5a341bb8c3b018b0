"""ctypes binding of libtriad_b200.so (the C ABI declared in include/triad_b200.h).

There is deliberately no fallback: if the shared library is missing or a call fails, the caller
gets an exception — nothing silently reroutes to PyTorch ops or to the CPU oracle.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p, POINTER

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libtriad_b200.so")

OK = 0
DTYPE_F32, DTYPE_BF16 = 0, 1
FWD_DEFAULT, FWD_FORCE_SIMT, FWD_FORCE_1CTA, FWD_DIVIDE_BY_T, FWD_SYNC_CHUNKS, FWD_PACK_ROWS = 0, 1, 2, 4, 8, 16
BWD_DEFAULT, BWD_GENERIC_DQ, BWD_GENERIC_DV, BWD_SMALL_BLOCKS, BWD_PACK_ROWS = 0, 1, 2, 16, 32
FWD_TEST_TRIP_WATCHDOG = 32
BWD_TEST_TRIP_WATCHDOG = 256
BWD_UNIFORM_SCALE = 128
BWD_ACCUMULATE_DV = 1024

# name -> (restype, argtypes); must list every symbol of include/triad_b200.h
SIGNATURES = {
    "triad_abi_version": (c_int, []),
    "triad_status_string": (c_char_p, [c_int]),
    "triad_last_error": (c_char_p, []),
    "triad_launch_count": (ctypes.c_longlong, []),
    "triad_device_check": (c_int, [c_int]),
    "triad_row_scale": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "triad_maxmean_fwd_workspace_bytes": (c_size_t, [c_int] * 6),
    "triad_maxmean_fwd_workspace_bytes_ex": (c_size_t, [c_int] * 7),
    "triad_maxmean_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_int, c_int, c_int, c_int, c_int, c_int,
                                  c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "triad_maxmean_fwd_status": (c_int, [c_void_p, c_void_p]),
    "triad_infonce_workspace_bytes": (c_size_t, [c_int, c_int]),
    "triad_infonce_partial": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                                      c_void_p, c_size_t, c_void_p]),
    "triad_infonce_finish": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int,
                                     c_float, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "triad_contrastive_head_workspace_bytes": (c_size_t, [c_int]),
    "triad_contrastive_head": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_size_t, c_void_p]),
    "triad_maxmean_bwd_workspace_bytes": (c_size_t, [c_int] * 6),
    "triad_maxmean_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_int, c_int, c_int, c_int, c_int, c_int,
                                  c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "triad_nonneg_workspace_bytes": (c_size_t, []),
    "triad_nonneg_chunk": (c_int, [c_void_p, c_size_t, c_int, c_void_p, c_float, c_float, c_int, c_void_p,
                                   c_void_p, c_size_t, c_void_p]),
    "triad_nonneg_fused_workspace_bytes": (c_size_t, []),
    "triad_nonneg_fused_chunk": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_float,
                                         c_void_p, ctypes.c_longlong, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "triad_maxmean_fwd_nonneg_workspace_bytes": (c_size_t, [c_int] * 5),
    "triad_maxmean_fwd_nonneg": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                         c_void_p, c_void_p, c_float, c_float, c_void_p, ctypes.c_longlong, c_void_p,
                                         c_void_p, c_size_t, c_int, c_void_p]),
    "triad_dense_grad_gemm_workspace_bytes": (c_size_t, [c_int] * 4),
    "triad_dense_grad_gemm": (c_int, [c_void_p, ctypes.c_longlong, c_int, c_int, c_void_p, c_int, c_int, c_void_p,
                                      c_void_p, c_size_t, c_void_p]),
    "triad_dense_grad_gemm_f32": (c_int, [c_void_p, ctypes.c_longlong, c_int, c_int, c_void_p, c_int, c_int, c_void_p,
                                          c_int, c_void_p, c_size_t, c_void_p]),
    "triad_pospair_workspace_bytes": (c_size_t, [c_int]),
    "triad_pospair_terms": (c_int, [c_void_p, c_int, c_void_p, c_int, c_float, c_int, c_int, c_int, c_void_p, c_void_p,
                                    c_void_p, c_size_t, c_void_p]),
    "triad_scale": (c_int, [c_void_p, c_void_p, c_size_t, c_int, c_void_p, c_void_p]),
    "triad_retrieve_workspace_bytes": (c_size_t, [c_int] * 5),
    "triad_retrieve_scores": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                                      c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "triad_quantize_e4m3": (c_int, [c_void_p, c_int, ctypes.c_longlong, c_int, c_void_p, c_void_p, c_void_p]),
    "triad_retrieve_e4m3_workspace_bytes": (c_size_t, [c_int] * 4),
    "triad_retrieve_scores_e4m3": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                           c_void_p, c_void_p, c_size_t, c_void_p]),
    "triad_ragged_plan": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "triad_ragged_pack": (c_int, [c_void_p, c_int, ctypes.c_longlong, c_int, c_void_p, ctypes.c_longlong, c_void_p,
                                  c_void_p]),
    "triad_retrieve_ragged_workspace_bytes": (c_size_t, [c_int] * 4),
    "triad_retrieve_scores_ragged": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                             c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "triad_ragged_pack_e4m3": (c_int, [c_void_p, c_int, ctypes.c_longlong, c_int, c_void_p, ctypes.c_longlong, c_void_p,
                                       c_void_p, c_void_p]),
    "triad_retrieve_scores_ragged_e4m3": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                                  c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_size_t,
                                                  c_void_p]),
    "triad_topk_workspace_bytes": (c_size_t, [c_int, c_int]),
    "triad_topk": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "triad_diag_ranks": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "triad_similarity_matrix": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                        c_void_p, c_void_p]),
    "triad_project_workspace_bytes": (c_size_t, []),
    "triad_project_tokens": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p,
                                     c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "triad_patch_compact": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "triad_project_tokens_bwd_workspace_bytes": (c_size_t, [c_int] * 3),
    "triad_project_tokens_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p,
                                         c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_size_t, c_void_p]),
    "triad_patch_expand": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
}

_lib = None


class TriadError(RuntimeError):
    def __init__(self, status: int, where: str, detail: str):
        super().__init__(f"{where} failed: status {status} ({detail})")
        self.status = status


def load() -> ctypes.CDLL:
    """Load the CUDA library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -m triad_b200.build` (or "
            "`python -c 'import __graft_entry__ as g; g.build()'`).  triad_b200 has no CPU / PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)       # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int, where: str) -> None:
    if status != OK:
        lib = load()
        msg = lib.triad_status_string(status).decode()
        last = lib.triad_last_error().decode()
        raise TriadError(status, where, f"{msg}; {last}" if last else msg)
