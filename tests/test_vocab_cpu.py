"""CPU-only checks of the token vocabulary's C ABI (latok_b200_vocab_*): NULL handles are rejected before any device
work, and without a GPU a Vocab fails loudly instead of counting in Python."""
import ctypes as C

import pytest

from latok_b200 import _lib


def test_null_handles_are_einval():
    L = _lib.load()
    out = C.c_void_p()
    assert L.latok_b200_vocab_create(None, 0, C.byref(out)) == _lib.EINVAL
    assert L.latok_b200_vocab_create(None, 0, None) == _lib.EINVAL
    assert L.latok_b200_vocab_destroy(None) == _lib.OK
    ids = (C.c_int32 * 4)()
    assert L.latok_b200_vocab_encode(None, None, 1, -1, 4, ids, 0) == _lib.EINVAL
    n, b = C.c_int64(0), C.c_int64(0)
    assert L.latok_b200_vocab_size(None, C.byref(n), C.byref(b), None) == _lib.EINVAL
    assert L.latok_b200_vocab_export(None, 0, 0, None, None, None) == _lib.EINVAL
    off = (C.c_int64 * 2)(0, 1)
    assert L.latok_b200_vocab_import(None, None, b"a", off, 1, None) == _lib.EINVAL
    ms = C.c_float(0)
    assert L.latok_b200_vocab_last_ms(None, C.byref(ms)) == _lib.EINVAL
    with pytest.raises(ValueError, match="NULL"):
        _lib.check(L.latok_b200_vocab_size(None, None, None, None))


def test_no_gpu_means_vocab_raises():
    if _lib.device_count() > 0:
        pytest.skip("a GPU is present")
    from latok_b200.vocab import Vocab
    with pytest.raises(_lib.LatokCudaError, match="no CPU fallback"):
        Vocab()
    with pytest.raises(_lib.LatokCudaError):
        Vocab.from_tokens(["a", "b"])
