"""CPU tests of the resident-batch entry points (tp_batch_recall, tp_batch_dendro, tp_batch_resident_bytes): the argument
checks that need no device."""
import ctypes

import pytest

from tadpole_b200 import _lib


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


def _err(lib):
    return lib.tp_last_error().decode()


def test_batch_recall_rejects_bad_selections_before_touching_a_device(lib):
    out = ctypes.c_void_p()
    one = (ctypes.c_int * 1)(0)
    rc = lib.tp_batch_recall(None, None, one, one, -1, 200, 2, 4, ctypes.byref(out))
    assert rc == _lib.TP_ERR_ARG and "nsel must not be negative" in _err(lib)
    rc = lib.tp_batch_recall(None, None, None, one, 1, 200, 2, 4, ctypes.byref(out))
    assert rc == _lib.TP_ERR_ARG and "null items / parts" in _err(lib)
    rc = lib.tp_batch_recall(None, None, one, None, 1, 200, 2, 4, ctypes.byref(out))
    assert rc == _lib.TP_ERR_ARG and "null items / parts" in _err(lib)
    rc = lib.tp_batch_recall(None, None, one, one, 1, 200, 2, 4, ctypes.byref(out))
    assert rc == _lib.TP_ERR_ARG and "null source batch" in _err(lib)
    assert not out.value


def test_batch_dendro_and_bytes_of_no_batch(lib):
    import numpy as np
    seq = np.zeros(4)
    assert lib.tp_batch_dendro(None, 0, -1, 0, _lib._dp(seq)) == _lib.TP_ERR_ARG
    assert "no such item" in _err(lib)
    assert lib.tp_batch_resident_bytes(None) == 0

