"""Argument refusals of ls_msp_solve_batch and ls_gmres_msp_batch: returned before any CUDA call, so no device is needed."""
import ctypes as C

import numpy as np


def test_msp_solve_batch_refuses_bad_arguments(built_lib):
    from fast_solver_lippmann_schwinger_b200._lib import LS_ERR_INVALID, lib
    L = lib()
    v = np.zeros(8, complex)
    p = v.ctypes.data_as(C.c_void_p)
    for nrhs in (0, -3):
        assert L.ls_msp_solve_batch(None, p, 4, p, 4, nrhs, 0) == LS_ERR_INVALID
        assert b"nrhs" in L.ls_last_error()
    assert L.ls_msp_solve_batch(None, p, 4, p, 4, 2, 0) == LS_ERR_INVALID
    assert b"null argument" in L.ls_last_error()
    h = C.c_void_p(p.value)                     # any non-null pointer: null rhs / x are refused first
    assert L.ls_msp_solve_batch(h, None, 4, p, 4, 2, 0) == LS_ERR_INVALID
    assert L.ls_msp_solve_batch(h, p, 4, None, 4, 2, 1) == LS_ERR_INVALID
    assert b"null argument" in L.ls_last_error()


def test_gmres_msp_batch_refuses_bad_arguments(built_lib):
    from fast_solver_lippmann_schwinger_b200._lib import LS_ERR_INVALID, lib
    L = lib()
    v = np.zeros(8, complex)
    p = v.ctypes.data_as(C.c_void_p)
    n64, ci = C.c_int64(), C.c_int()

    def call(k, op, msp, nrhs, b, x):
        return L.ls_gmres_msp_batch(k, op, None, msp, nrhs, b, 4, x, 4, 20, 10, 1e-8, 0.0, 1, None, 0,
                                    C.byref(n64), C.byref(ci), C.byref(n64), 0)
    assert call(p, p, p, 0, p, p) == LS_ERR_INVALID and b"nrhs" in L.ls_last_error()
    for args in ((None, p, p, 2, p, p), (p, None, p, 2, p, p), (p, p, None, 2, p, p), (p, p, p, 2, None, p), (p, p, p, 2, p, None)):
        assert call(*args) == LS_ERR_INVALID
        assert b"null argument" in L.ls_last_error()
