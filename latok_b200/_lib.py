"""ctypes binding of liblatok_b200.so (the C ABI in include/latok_b200.h).

This is the only place the Python package touches native code.  There is no Python or NumPy
implementation of the tokenization path in this package: if the library is missing it is built
with nvcc, and if it cannot be built or no CUDA device is present every compute call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("LATOK_B200_LIB") or PKG / "liblatok_b200.so")  # override: development builds only

OK, EINVAL, ECUDA, ENOMEM, ESTATE, EINTERNAL = range(6)
SPLITS, SPANS, FEATS, MATRIX, SPANS16 = 1, 2, 4, 8, 16
NUM_FEATURES = 25


class LatokCudaError(RuntimeError):
    """CUDA failure, missing device, or internal device-side check (maps LATOK_B200_ECUDA/EINTERNAL)."""


_lib = None


def load():
    """Load (building first if necessary) liblatok_b200.so and declare every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        from . import build as _build
        _build.build_library()
    L = C.CDLL(str(LIB_PATH))
    vp, i64, i32, u32, sz = C.c_void_p, C.c_int64, C.c_int, C.c_uint32, C.c_size_t
    P = C.POINTER
    proto = {
        "latok_b200_abi_version": (C.c_int, []),
        "latok_b200_last_error": (C.c_char_p, []),
        "latok_b200_device_count": (C.c_int, [P(C.c_int)]),
        "latok_b200_create": (C.c_int, [i32, sz, i64, P(vp)]),
        "latok_b200_destroy": (C.c_int, [vp]),
        "latok_b200_set_rules": (C.c_int, [vp, vp, i32, i32, vp, i32, i32, vp, i32, i32]),
        "latok_b200_submit": (C.c_int, [vp, vp, vp, i64, u32]),
        "latok_b200_submit_device": (C.c_int, [vp, vp, vp, i64, i64, u32]),
        "latok_b200_sizes": (C.c_int, [vp, P(i64), P(i64)]),
        "latok_b200_set_pipeline_depth": (C.c_int, [vp, i32]),
        "latok_b200_fetch": (C.c_int, [vp, i64, i64, i64, vp, vp, vp, vp, vp, vp]),
        "latok_b200_release": (C.c_int, [vp]),
        "latok_b200_in_flight": (C.c_int, [vp, P(C.c_int)]),
        "latok_b200_fetch_token_bytes": (C.c_int, [vp, i64, vp, i32]),
        "latok_b200_token_bytes_ms": (C.c_int, [vp, P(C.c_float)]),
        "latok_b200_device_results": (C.c_int, [vp, P(vp), P(vp), P(vp), P(vp), P(vp), P(vp)]),
        "latok_b200_timer_begin": (C.c_int, [vp]),
        "latok_b200_timer_end": (C.c_int, [vp, P(C.c_float)]),
        "latok_b200_launch_count": (C.c_int, [vp, P(i64)]),
        "latok_b200_last_stats": (C.c_int, [vp, P(C.c_float), P(i64)]),
        "latok_b200_reader_open": (C.c_int, [C.c_char_p, i32, P(vp)]),
        "latok_b200_reader_next": (C.c_int, [vp, i64, vp, i64, vp, P(i64)]),
        "latok_b200_reader_close": (C.c_int, [vp]),
        "latok_b200_host_alloc": (C.c_int, [P(vp), sz]),
        "latok_b200_host_free": (C.c_int, [vp]),
        "latok_b200_gen_parse_matrix": (C.c_int, [vp, vp, i64, P(i64), vp]),
        "latok_b200_gen_block_mask": (C.c_int, [vp, vp, i64, vp, i64, i64, vp]),
        "latok_b200_combine_matrix_rows": (C.c_int, [vp, vp, i64, i64, i64, i64, vp, i32, i32, vp]),
        "latok_b200_vocab_create": (C.c_int, [vp, i64, P(vp)]),
        "latok_b200_vocab_destroy": (C.c_int, [vp]),
        "latok_b200_vocab_encode": (C.c_int, [vp, vp, i32, C.c_int32, i64, vp, i32]),
        "latok_b200_vocab_size": (C.c_int, [vp, P(i64), P(i64), P(i64)]),
        "latok_b200_vocab_export": (C.c_int, [vp, i64, i64, vp, vp, vp]),
        "latok_b200_vocab_import": (C.c_int, [vp, vp, vp, vp, i64, vp]),
        "latok_b200_vocab_merge": (C.c_int, [vp, vp, vp, vp, i32]),
        "latok_b200_vocab_clear": (C.c_int, [vp]),
        "latok_b200_vocab_last_ms": (C.c_int, [vp, P(C.c_float)]),
        "latok_b200_vocab_wordpiece": (C.c_int, [vp, vp, vp, i32, i32, C.c_int32, i64, vp, P(i64), i32]),
        "latok_b200_vocab_wordpiece_fetch": (C.c_int, [vp, i64, vp, i32]),
    }
    for name, (res, args) in proto.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    if L.latok_b200_abi_version() != 2:
        raise ImportError("liblatok_b200.so ABI version mismatch; rebuild with python -m latok_b200.build")
    _lib = L
    return L


def check(rc: int):
    """Map a C status to the exception the reference raises for the same condition
    (ValueError for argument errors, latok.c:40-50,151-171,292-312; RuntimeError otherwise)."""
    if rc == OK:
        return
    msg = (load().latok_b200_last_error() or b"").decode("utf-8", "replace")
    if rc == EINVAL:
        raise ValueError(msg)
    if rc == ENOMEM:
        raise MemoryError(msg)
    if rc == ESTATE:
        raise RuntimeError(msg)
    raise LatokCudaError(msg)


def device_count() -> int:
    n = C.c_int(0)
    check(load().latok_b200_device_count(C.byref(n)))
    return n.value
