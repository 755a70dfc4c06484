"""spmv_b200_spmv_shifted without a device: a NULL handle and a handle whose create failed return -1 and leave y and
dots untouched; the Python wrapper rejects a dots argument that is not a 2-element float64 CUDA tensor."""
import types

import numpy as np
import pytest

from spmv_b200 import api


def test_null_and_failed_handles_return_an_error(libpath):
    L = api.lib()
    x, y = np.ones(4), np.full(4, 7.0)
    dots = np.full(2, 5.0)
    api.clear_error()
    assert L.spmv_b200_spmv_shifted(None, 1.0, 0.5, x.ctypes.data, 0.0, y.ctypes.data, dots.ctypes.data) == -1
    assert "NULL handle" in api.last_error()
    rowptr = np.array([1, 2, 3, 4, 5], dtype=np.int32)  # RowPtr[0] != 0: create fails, with or without a device
    h = api.spmv_create_handle_all_in_one(4, 4, rowptr, np.zeros(4, dtype=np.int32), np.ones(4), 1, api.Method_Parallel, 8)
    for args in ((x.ctypes.data, y.ctypes.data, dots.ctypes.data), (None, None, None), (x.ctypes.data, y.ctypes.data, None)):
        api.clear_error()
        assert L.spmv_b200_spmv_shifted(h, 1.0, 0.5, args[0], 0.0, args[1], args[2]) == -1
        assert "create failed" in api.last_error()
    assert (y == 7.0).all() and (dots == 5.0).all()
    api.spmv_destory_handle(h)


def test_python_wrapper_rejects_a_host_dots_array():
    unbound = types.SimpleNamespace(h=None)  # the argument check comes before any call into the library
    with pytest.raises(ValueError):
        api.Handle.spmv_shifted(unbound, 1.0, 0.5, np.ones(4), 0.0, np.zeros(4), np.zeros(2))
