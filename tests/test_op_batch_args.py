"""Argument refusals of ls_op_apply_batch, ls_op_batch_cols and ls_gmres_batch: returned before any CUDA call, so no
device is needed.  (The refusals that need a live operator - leading dimensions, overlaps, modes - are checked on the
device in test_gpu_apply_batch.py.)"""
import ctypes as C

import numpy as np


def test_op_apply_batch_refuses_bad_arguments(built_lib):
    from fast_solver_lippmann_schwinger_b200._lib import LS_ERR_INVALID, lib
    L = lib()
    v = np.zeros(8, complex)
    p = v.ctypes.data_as(C.c_void_p)
    for nrhs in (0, -3):
        assert L.ls_op_apply_batch(p, p, 4, p, 4, nrhs, 0, 1) == LS_ERR_INVALID
        assert b"nrhs" in L.ls_last_error()
    for h, b, y in ((None, p, p), (p, None, p), (p, p, None)):
        assert L.ls_op_apply_batch(h, b, 4, y, 4, 2, 0, 1) == LS_ERR_INVALID
        assert b"null argument" in L.ls_last_error()
    fake = np.zeros(64, np.uint8)               # zeroed memory: its handle kind is no operator's
    assert L.ls_op_apply_batch(fake.ctypes.data_as(C.c_void_p), p, 4, p, 4, 2, 0, 1) == LS_ERR_INVALID
    assert b"not an operator handle" in L.ls_last_error()


def test_op_batch_cols_refuses_bad_arguments(built_lib):
    from fast_solver_lippmann_schwinger_b200._lib import LS_ERR_INVALID, lib
    L = lib()
    c = C.c_int(-7)
    fake = np.zeros(64, np.uint8)
    assert L.ls_op_batch_cols(None, C.byref(c)) == LS_ERR_INVALID
    assert L.ls_op_batch_cols(fake.ctypes.data_as(C.c_void_p), None) == LS_ERR_INVALID
    assert b"null argument" in L.ls_last_error()
    assert L.ls_op_batch_cols(fake.ctypes.data_as(C.c_void_p), C.byref(c)) == LS_ERR_INVALID
    assert b"not an operator handle" in L.ls_last_error()
    assert c.value == -7


def test_gmres_batch_refuses_bad_arguments(built_lib):
    from fast_solver_lippmann_schwinger_b200._lib import LS_ERR_INVALID, lib
    L = lib()
    v = np.zeros(8, complex)
    p = v.ctypes.data_as(C.c_void_p)
    n64, ci = C.c_int64(), C.c_int()

    def call(k, op, nrhs, b, x, hist=None, cap=0):
        return L.ls_gmres_batch(k, op, nrhs, b, 4, x, 4, 20, 10, 1e-8, 0.0, 1, hist, cap,
                                C.byref(n64), C.byref(ci), C.byref(n64), 0)
    assert call(p, p, 0, p, p) == LS_ERR_INVALID and b"nrhs" in L.ls_last_error()
    for args in ((None, p, 2, p, p), (p, None, 2, p, p), (p, p, 2, None, p), (p, p, 2, p, None)):
        assert call(*args) == LS_ERR_INVALID
        assert b"null argument" in L.ls_last_error()
    h = np.zeros(4)
    assert call(p, p, 2, p, p, h.ctypes.data_as(C.c_void_p), -1) == LS_ERR_INVALID
    assert b"hist_cap" in L.ls_last_error()
    fake = np.zeros(64, np.uint8)               # zeroed memory: no Krylov workspace
    assert call(fake.ctypes.data_as(C.c_void_p), p, 2, p, p) == LS_ERR_INVALID
    assert b"not a Krylov workspace handle" in L.ls_last_error()
