"""ctypes binding of the C ABI declared in ``include/flmr_maxsim.h``.

This is the stub a maintainer of the reference would add (INTEGRATION.md): plain pointers and
sizes, every call returns a status, ``flmr_last_error`` explains failures.  There is NO fallback:
if the CUDA library cannot be built/loaded the import of the product path fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

FLMR_OK = 0
FLAG_RELU = 1
CORPUS_COPY = 0
CORPUS_ADOPT = 1
DIM = 128
TOKEN_GROUP = 4
MAX_K = 128
SELECT_MAX_K = 2048


def _header_define(name: str) -> int:
    import re
    hdr = os.path.join(os.path.dirname(os.path.abspath(_build.__file__)), "..", "include", "flmr_maxsim.h")
    m = re.search(r"#define\s+%s\s+(\d+)" % name, open(hdr).read())
    return int(m.group(1))


TILE_TOKENS = _header_define("FLMR_TILE_TOKENS")

# every symbol include/flmr_maxsim.h declares (tests check the .so exports all of them)
SYMBOLS = [
    "flmr_last_error", "flmr_abi_version",
    "flmr_corpus_create", "flmr_corpus_create_plaid", "flmr_corpus_destroy",
    "flmr_corpus_plaid_builder_create", "flmr_corpus_plaid_builder_append", "flmr_corpus_plaid_builder_finish",
    "flmr_corpus_plaid_builder_destroy", "flmr_corpus_info",
    "flmr_workspace_create", "flmr_workspace_destroy", "flmr_workspace_status",
    "flmr_maxsim_scores", "flmr_maxsim_topk", "flmr_topk_merge", "flmr_topk_select", "flmr_plaid_decode",
    "flmr_maxsim_argmax", "flmr_maxsim_backward", "flmr_corpus_gather",
    "flmr_maxsim_argmax_grouped", "flmr_maxsim_backward_grouped", "flmr_ib_loss",
    "flmr_corpus_builder_create", "flmr_corpus_builder_append", "flmr_corpus_builder_append_file",
    "flmr_corpus_builder_finish", "flmr_corpus_builder_destroy",
    "flmr_comm_unique_id", "flmr_comm_create", "flmr_comm_adopt", "flmr_comm_destroy", "flmr_comm_info",
    "flmr_topk_exchange", "flmr_maxsim_topk_sharded",
    "flmr_debug_maxsim_scores_simt", "flmr_debug_set_argmax_path", "flmr_debug_set_scan_variant", "flmr_debug_build_partition", "flmr_debug_plan_passes",
    "flmr_launch_count", "flmr_set_profiling", "flmr_scan_kernel_stats",
]


class CorpusInfo(C.Structure):
    _fields_ = [
        ("n_passages", C.c_int64), ("n_tokens", C.c_int64), ("n_rows", C.c_int64),
        ("pid_base", C.c_int64), ("dim", C.c_int32), ("device", C.c_int32),
        ("n_ctas", C.c_int32), ("adopted", C.c_int32), ("n_tiles", C.c_int64),
        ("hbm_bytes", C.c_int64),
    ]


class FlmrError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("flmr_maxsim error %d: %s" % (code, msg))
        self.code = code


_lib = None


def lib() -> C.CDLL:
    """Load (building first if stale) the shared library and declare prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("FLMR_MAXSIM_LIB") or _build.build()
    L = C.CDLL(path)
    vp, i32, i64, u32 = C.c_void_p, C.c_int, C.c_int64, C.c_uint
    L.flmr_last_error.restype = C.c_char_p
    L.flmr_last_error.argtypes = []
    L.flmr_abi_version.restype = i32
    L.flmr_abi_version.argtypes = []
    L.flmr_corpus_create.argtypes = [vp, vp, i64, i32, i32, i64, u32, C.POINTER(vp)]
    L.flmr_corpus_create_plaid.argtypes = [vp, vp, vp, i64, vp, i32, vp, i64, i32, i32, i64, C.POINTER(vp)]
    L.flmr_corpus_plaid_builder_create.argtypes = [vp, i64, vp, i32, vp, i64, i32, i32, i64, C.POINTER(vp)]
    L.flmr_corpus_plaid_builder_append.argtypes = [vp, vp, vp, i64]
    L.flmr_corpus_plaid_builder_finish.argtypes = [vp, C.POINTER(vp)]
    L.flmr_corpus_plaid_builder_destroy.argtypes = [vp]
    L.flmr_corpus_destroy.argtypes = [vp]
    L.flmr_corpus_info.argtypes = [vp, C.POINTER(CorpusInfo)]
    L.flmr_workspace_create.argtypes = [vp, i32, i32, C.POINTER(vp)]
    L.flmr_workspace_destroy.argtypes = [vp]
    L.flmr_workspace_status.argtypes = [vp, C.POINTER(i32)]
    L.flmr_maxsim_scores.argtypes = [vp, vp, vp, i32, i32, u32, vp, vp]
    L.flmr_maxsim_topk.argtypes = [vp, vp, vp, i32, i32, i32, u32, vp, vp, vp]
    L.flmr_topk_merge.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, i32, vp]
    L.flmr_topk_select.argtypes = [vp, i32, i64, i32, i64, vp, vp, i32, vp]
    L.flmr_plaid_decode.argtypes = [vp, vp, i64, vp, i64, vp, i32, i32, i32, vp, i32, vp]
    L.flmr_corpus_gather.argtypes = [vp, vp, i64, i32, vp, vp, vp]
    L.flmr_maxsim_argmax.argtypes = [vp, i32, i32, vp, vp, i32, i32, vp, vp, i32, vp]
    L.flmr_maxsim_backward.argtypes = [vp, i32, i32, vp, i32, i32, vp, vp, vp, vp, i32, vp]
    L.flmr_ib_loss.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp, vp, i32, vp]
    L.flmr_maxsim_argmax_grouped.argtypes = [vp, i32, i32, vp, vp, i32, i32, vp, vp, i32, vp]
    L.flmr_maxsim_backward_grouped.argtypes = [vp, i32, i32, vp, i32, i32, vp, vp, vp, vp, i32, vp]
    L.flmr_corpus_builder_create.argtypes = [vp, i64, i32, i32, i64, C.POINTER(vp)]
    L.flmr_corpus_builder_append.argtypes = [vp, vp, i64]
    L.flmr_corpus_builder_append_file.argtypes = [vp, C.c_char_p, i64, i64]
    L.flmr_corpus_builder_finish.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_double)]
    L.flmr_corpus_builder_destroy.argtypes = [vp]
    L.flmr_comm_unique_id.argtypes = [vp]
    L.flmr_comm_create.argtypes = [vp, i32, i32, i32, C.POINTER(vp)]
    L.flmr_comm_adopt.argtypes = [vp, i32, C.POINTER(vp)]
    L.flmr_comm_destroy.argtypes = [vp]
    L.flmr_comm_info.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    L.flmr_topk_exchange.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp, vp]
    L.flmr_maxsim_topk_sharded.argtypes = [vp, vp, vp, vp, i32, i32, i32, u32, vp, vp, vp]
    L.flmr_debug_maxsim_scores_simt.argtypes = [vp, vp, i32, i32, u32, vp, vp]
    L.flmr_debug_set_argmax_path.argtypes = [i32]
    L.flmr_debug_set_scan_variant.argtypes = [i32]
    L.flmr_debug_build_partition.argtypes = [vp, i64, i32, vp, vp, vp, vp, i64, C.POINTER(i64)]
    L.flmr_debug_plan_passes.argtypes = [i32, i32, i32, vp, i32, C.POINTER(i32)]
    L.flmr_launch_count.restype = i64
    L.flmr_launch_count.argtypes = [i32]
    L.flmr_set_profiling.argtypes = [i32]
    L.flmr_scan_kernel_stats.argtypes = [C.POINTER(C.c_double), C.POINTER(i64), i32]
    for name in SYMBOLS:
        fn = getattr(L, name)
        if name not in ("flmr_last_error", "flmr_launch_count"):
            fn.restype = i32
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != FLMR_OK:
        raise FlmrError(rc, lib().flmr_last_error().decode("utf-8", "replace"))
