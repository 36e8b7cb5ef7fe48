"""CPU-side argument checks of the prediction entry points bqb_predict_rows_device / _host and bqb_alpha_read (no GPU: the
checks come before any device call)."""
import ctypes

import numpy as np


def test_prediction_entry_points_refuse_a_null_batch():
    from bayesian_quadrature_b200 import _lib
    L = _lib.load()
    x = np.zeros(4)
    out = np.zeros(4)
    rows = (ctypes.c_int * 1)(0)
    dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    assert L.bqb_predict_rows_device(None, rows, 1, None, 0, 4, None, None, 4, None) == _lib.EINVAL
    assert L.bqb_predict_rows_device(None, None, 0, None, 0, 0, None, None, 0, None) == _lib.EINVAL
    assert L.bqb_predict_rows_host(None, rows, 1, dp(x), 0, 4, dp(out), dp(out)) == _lib.EINVAL
    assert L.bqb_predict_rows_host(None, None, 0, dp(x), 0, 4, dp(out), dp(out)) == _lib.EINVAL
    assert b"null batch" in L.bqb_last_error()
    assert L.bqb_alpha_read(None, 0, dp(out)) == _lib.EINVAL
    assert b"bad arguments" in L.bqb_last_error()
