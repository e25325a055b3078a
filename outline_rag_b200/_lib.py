"""ctypes binding of the C-ABI in ``include/orx.h`` (``liborx.so``, built in-tree).

There is NO CPU fallback: if the shared library is missing or cannot be loaded the
import of this module raises, and every entry point needs a B200 at call time
(``orx_create`` fails with ORX_ERR_CUDA otherwise).  Loading the library and
resolving its symbols does not need a GPU (``tests/test_abi.py``).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
# The library is the in-tree build, full stop: no environment variable can swap it.  Same-box A/B measurements of an
# experimental build (`make -C csrc variant NAME=x`) select it IN PROCESS, before the first import of this package,
# by registering a module object: sys.modules["orx_lib_override"] = SimpleNamespace(LIB_PATH=...)  (bench.py --lib).
_override = getattr(sys.modules.get("orx_lib_override"), "LIB_PATH", None)
LIB_PATH = _override or os.path.join(_HERE, "liborx.so")
CSRC_DIR = os.path.join(_HERE, "csrc")

ORX_DIM = 1024
ORX_MAX_K = 128
ORX_OPT_SCAN_TIMING = 1
ORX_OPT_IMAGE_MIN_ROWS = 2
ORX_OPT_IMAGE8_MIN_ROWS = 3
ORX_IPC_HANDLE_BYTES = 64
DTYPE_F32 = 0
DTYPE_BF16 = 1

ORX_OK = 0
ORX_ERR_INVALID = -1
ORX_ERR_DIM = -2
ORX_ERR_NONFINITE = -3
ORX_ERR_CUDA = -4
ORX_ERR_CAPACITY = -5


class OrxError(RuntimeError):
    """Raised for every non-zero return of the C-ABI; ``code`` is the ORX_ERR_* value."""

    def __init__(self, code: int, message: str):
        super().__init__(f"orx error {code}: {message}")
        self.code = code
        self.message = message


class OrxValueError(OrxError, ValueError):
    """ORX_ERR_DIM / ORX_ERR_NONFINITE / ORX_ERR_INVALID: the input is at fault (pgvector
    raises `expected 1024 dimensions` / `NaN not allowed in vector` for the same inputs)."""


class OrxId(C.Structure):
    _fields_ = [("hi", C.c_uint64), ("lo", C.c_uint64)]


class OrxStats(C.Structure):
    _fields_ = [
        ("kernel_launches", C.c_uint64),
        ("searches", C.c_uint64),
        ("queries", C.c_uint64),
        ("fallback_gemv", C.c_uint64),
        ("fallback_exhaustive", C.c_uint64),
        ("rows_moved", C.c_uint64),
        ("last_scan_ms", C.c_float),
        ("last_search_ms", C.c_float),
        ("last_path", C.c_int),
        ("reserved", C.c_int),
        ("scan_launches", C.c_uint64),
        ("scan_ms_total", C.c_double),
    ]


# name -> (restype, argtypes); every symbol include/orx.h declares
_vp = C.c_void_p
SIGNATURES = {
    "orx_create": (C.c_int, [C.POINTER(_vp), C.c_int, C.c_int, C.c_uint64, C.c_int]),
    "orx_create_multi": (C.c_int, [C.POINTER(_vp), C.c_int, C.c_int, C.c_uint64, C.POINTER(C.c_int), C.c_int]),
    "orx_shard_count": (C.c_int, [_vp]),
    "orx_destroy": (None, [_vp]),
    "orx_set_stream": (C.c_int, [_vp, _vp]),
    "orx_set_option": (C.c_int, [_vp, C.c_int, C.c_int]),
    "orx_size": (C.c_uint64, [_vp]),
    "orx_capacity": (C.c_uint64, [_vp]),
    "orx_dtype": (C.c_int, [_vp]),
    "orx_mutation_count": (C.c_uint64, [_vp]),
    "orx_get_stats": (C.c_int, [_vp, C.POINTER(OrxStats)]),
    "orx_upsert": (C.c_int, [_vp, _vp, _vp, C.c_uint64, C.c_int]),
    "orx_delete": (C.c_int, [_vp, _vp, C.c_uint64, C.POINTER(C.c_uint64)]),
    "orx_contains": (C.c_int, [_vp, OrxId]),
    "orx_search": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp]),
    "orx_search_submit": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, C.POINTER(C.c_int)]),
    "orx_search_wait": (C.c_int, [_vp, C.c_int]),
    "orx_search_sharded_submit": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, C.POINTER(C.c_int)]),
    "orx_search_filtered": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp, C.c_uint64, _vp, _vp, _vp]),
    "orx_filter_create": (C.c_int, [_vp, _vp, C.c_uint64, C.POINTER(_vp)]),
    "orx_filter_destroy": (None, [_vp]),
    "orx_search_with_filter": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp]),
    "orx_search_mmr": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, _vp, _vp, _vp]),
    "orx_search_mmr_filtered": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, _vp, C.c_uint64,
                                          _vp, _vp, _vp]),
    "orx_search_mmr_with_filter": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double,
                                             _vp, _vp, _vp]),
    "orx_merge_topk": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "orx_merge_topk_strided": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, C.c_uint64, _vp, _vp, _vp]),
    "orx_export_rows": (C.c_int, [_vp, C.c_uint64, C.c_uint64, _vp, _vp]),
    "orx_import_rows": (C.c_int, [_vp, _vp, _vp, C.c_uint64]),
    "orx_shard_export": (C.c_int, [_vp, C.c_int, C.c_int, _vp]),
    "orx_shard_connect": (C.c_int, [_vp, _vp, C.c_int]),
    "orx_search_sharded": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp]),
    "orx_fetch": (C.c_int, [_vp, _vp, C.c_uint64, _vp, _vp]),
    "orx_debug_coarse_scores": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp]),
    "orx_debug_fast_scores": (C.c_int, [_vp, _vp, C.c_int, _vp]),
    "orx_debug_image_scores": (C.c_int, [_vp, _vp, C.c_int, _vp]),
    "orx_debug_image8_scores": (C.c_int, [_vp, _vp, C.c_int, _vp]),
    "orx_pgcopy_open": (C.c_int, [_vp, C.POINTER(_vp)]),
    "orx_pgcopy_open_sharded": (C.c_int, [_vp, C.c_int, C.c_int, C.POINTER(_vp)]),
    "orx_pgcopy_feed": (C.c_int, [_vp, _vp, C.c_uint64]),
    "orx_pgcopy_close": (C.c_int, [_vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "orx_parse_vector_text": (C.c_int, [C.c_char_p, C.c_uint64, _vp, C.c_int]),
    "orx_last_error": (C.c_char_p, []),
    "orx_version": (C.c_char_p, []),
}


def build(verbose: bool = False) -> str:
    """Compile ``liborx.so`` for sm_100a with the in-tree Makefile (nvcc cross-compiles
    without a GPU).  Returns the library path."""
    out = subprocess.run(["make", "-C", CSRC_DIR, "-j8"], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout)
        print(out.stderr)
    if out.returncode != 0:
        raise RuntimeError("building liborx.so failed (see output above)")
    return LIB_PATH


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `make -C {CSRC_DIR}` "
            "(or __graft_entry__.build()).  outline_rag_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the header and the library diverge
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def last_error() -> str:
    msg = lib.orx_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int) -> None:
    if rc != ORX_OK:
        cls = OrxValueError if rc in (ORX_ERR_INVALID, ORX_ERR_DIM, ORX_ERR_NONFINITE) else OrxError
        raise cls(rc, last_error())


def version() -> str:
    return lib.orx_version().decode()
