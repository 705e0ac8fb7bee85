"""ctypes binding of libscone_b200.so -- the C ABI declared in include/scone_b200.h.

There is no fallback: if the library is missing or a call fails, an exception is raised.
"""

from __future__ import annotations

import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))
# SCONE_B200_LIB: another build of the library (development: same-box A/B against an older build)
LIB_PATH = os.environ.get("SCONE_B200_LIB") or os.path.join(PKG, "lib", "libscone_b200.so")

QUANT = {"fp16": 0, "int8": 1, "int4": 2, "fp32": 3}
OUT_BF16, OUT_FP16, OUT_FP32 = 0, 1, 2
STATUS_TOKEN_OOR = 1
MAX_N = 7
ABI_VERSION = 200        # SCONE_B200_VERSION of include/scone_b200.h this binding was written against

E_INVALID, E_CUDA, E_VOCAB, E_NOMEM = -1, -2, -3, -4

# every symbol include/scone_b200.h declares (tests check they are all exported)
SYMBOLS = [
    "scone_version", "scone_last_error", "scone_launch_count", "scone_host_gather_rows", "scone_host_alloc", "scone_host_free",
    "scone_index_create", "scone_index_destroy", "scone_index_info", "scone_index_lookup", "scone_index_match_all", "scone_fit_vocab",
    "scone_table_layout", "scone_table_store", "scone_table_store_projected", "scone_table_gather", "scone_table_gather_packed",
    "scone_embed_forward", "scone_embed_forward_additive", "scone_embed_forward_ex", "scone_embed_gather", "scone_embed_forward_sharded", "scone_embed_mean_forward",
    "scone_pipeline_create", "scone_pipeline_submit", "scone_pipeline_follow", "scone_pipeline_wait", "scone_pipeline_destroy",
]


class IndexInfo(C.Structure):
    _fields_ = [("num_fgrams", C.c_int64), ("capacity", C.c_int64), ("bytes", C.c_int64), ("max_n", C.c_int32),
                ("len_mask", C.c_uint32), ("max_probe", C.c_int32), ("slot_bytes", C.c_int32), ("filter_bytes", C.c_int64),
                ("slot_format", C.c_int32), ("reserved", C.c_int32)]


class TableDesc(C.Structure):
    _fields_ = [("d_rows", C.c_void_p), ("row_stride", C.c_int64), ("num_rows", C.c_int64), ("quant", C.c_int32),
                ("dim", C.c_int32), ("group", C.c_int32), ("scale_offset", C.c_int32)]


class EmbedOpts(C.Structure):
    _fields_ = [("flags", C.c_uint32), ("reserved", C.c_uint32 * 3)]


EMBED_ADDITIVE, EMBED_INPUTS_STABLE = 1, 2


class SconeError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libscone_b200 error {code}: {msg}")
        self.code = code


_lib = None


def load() -> C.CDLL:
    """Load the library (once).  Raises if it has not been built -- build with `python -m scone_b200.build`."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA library has not been built (python -m scone_b200.build). "
            "scone_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int32
    L.scone_version.restype = C.c_int
    L.scone_last_error.restype = C.c_char_p
    L.scone_launch_count.restype = i64
    L.scone_index_create.argtypes = [vp, vp, i64, i32, C.c_double, vp, C.POINTER(vp)]
    L.scone_index_destroy.argtypes = [vp]
    L.scone_index_info.argtypes = [vp, C.POINTER(IndexInfo)]
    L.scone_index_lookup.argtypes = [vp, vp, i64, i64, vp, vp, vp]
    L.scone_index_match_all.argtypes = [vp, vp, i64, i64, vp, vp]
    L.scone_fit_vocab.argtypes = [vp, i64, vp, i64, i32, i64, i64, C.c_uint64, vp, vp, vp, C.POINTER(i64), C.POINTER(i64), vp]
    L.scone_table_layout.argtypes = [i32, i32, i32, i32, C.POINTER(i64), C.POINTER(i32)]
    L.scone_table_store.argtypes = [C.POINTER(TableDesc), vp, vp, i64, i64, vp]
    L.scone_table_store_projected.argtypes = [C.POINTER(TableDesc), vp, vp, i32, vp, i64, i64, vp, vp]
    L.scone_table_gather.argtypes = [C.POINTER(TableDesc), vp, i64, vp, i32, vp, vp]
    L.scone_table_gather_packed.argtypes = [C.POINTER(TableDesc), vp, i64, vp, vp, vp]
    L.scone_host_gather_rows.argtypes = [vp, i64, i64, vp, i64, vp, i32]
    L.scone_host_alloc.argtypes = [i64, i32, C.POINTER(vp), C.POINTER(vp)]
    L.scone_host_free.argtypes = [vp, i64]
    L.scone_embed_forward.argtypes = [vp, C.POINTER(TableDesc), vp, i64, vp, vp, i64, i64, vp, i32, vp, vp, vp, vp]
    L.scone_embed_forward_additive.argtypes = L.scone_embed_forward.argtypes
    L.scone_embed_forward_ex.argtypes = [vp, C.POINTER(TableDesc), vp, i64, vp, vp, i64, i64, vp, i32, vp, vp, vp, C.POINTER(EmbedOpts), vp]
    L.scone_embed_forward_sharded.argtypes = [vp, C.POINTER(TableDesc), vp, i32, i64, vp, i64, vp, vp, i64, i64, vp, i32, vp, vp, vp, vp]
    L.scone_embed_mean_forward.argtypes = [vp, C.POINTER(TableDesc), vp, i64, i64, vp, vp, i32, vp]
    L.scone_pipeline_create.argtypes = [vp, C.POINTER(TableDesc), vp, i64, vp, i64, i64, i32, i32, vp, vp, vp, vp, vp, C.POINTER(vp)]
    L.scone_pipeline_submit.argtypes = [vp, vp, C.POINTER(i32)]
    L.scone_pipeline_follow.argtypes = [vp, vp]
    L.scone_pipeline_wait.argtypes = [vp, i32]
    L.scone_pipeline_destroy.argtypes = [vp]
    L.scone_embed_gather.argtypes = [C.POINTER(TableDesc), vp, i64, vp, i64, vp, vp, i64, vp, i32, vp, vp]
    for name in SYMBOLS:
        fn = getattr(L, name)
        if name not in ("scone_version", "scone_last_error", "scone_launch_count"):
            fn.restype = C.c_int
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != 0:
        msg = load().scone_last_error().decode("utf-8", "replace")
        if rc == E_INVALID or rc == E_VOCAB:
            raise ValueError(f"libscone_b200: {msg}")
        raise SconeError(rc, msg)


def launch_count() -> int:
    return int(load().scone_launch_count())
