"""CPU tests of LS_FLAG_EMBED's argument checks: every refusal happens before any CUDA call, so they run without a GPU.
The host arrays passed are deliberately tiny: a refusal that read them would read past their end."""
import ctypes as C

import numpy as np
import pytest

EMBED, PAD4, FORCE_GENERIC = 4, 2, 1


def _create(L, n, m, ne, me, quad, flags):
    h = C.c_void_p()
    nu = np.zeros(4)
    g = np.zeros(16, complex)
    return L.ls_op2d_create(C.byref(h), n, m, ne, me, nu.ctypes.data_as(C.c_void_p), g.ctypes.data_as(C.c_void_p),
                            1.0, quad, flags)


def test_embed_flag_combinations_refused(built_lib):
    from fast_solver_lippmann_schwinger_b200._lib import lib, FLAG_EMBED
    L = lib()
    assert FLAG_EMBED == EMBED
    # no literal 4x evaluation exists on the embedded route
    assert _create(L, 1001, 1001, 4004, 4004, 1, EMBED | PAD4) == -2
    assert b"2x padding" in L.ls_last_error()
    # two different routes asked for at once
    assert _create(L, 1001, 1001, 4004, 4004, 1, EMBED | FORCE_GENERIC) == -1
    assert b"FORCE_GENERIC" in L.ls_last_error()
    assert _create(L, 1001, 1001, 2001, 2001, 0, EMBED | FORCE_GENERIC | PAD4) == -1


@pytest.mark.parametrize("quad,n,m", [(1, 4097, 64), (1, 64, 4097), (0, 4097, 4097)])
def test_embed_size_limit_named(built_lib, quad, n, m):
    from fast_solver_lippmann_schwinger_b200._lib import lib
    L = lib()
    ne, me = (4 * n, 4 * m) if quad == 1 else (2 * n - 1, 2 * m - 1)
    assert _create(L, n, m, ne, me, quad, EMBED) == -2
    assert b"4096" in L.ls_last_error()


def test_embed_shape_checks_and_device_spectrum_limit(built_lib):
    from fast_solver_lippmann_schwinger_b200._lib import lib
    L = lib()
    assert _create(L, 1001, 1001, 4000, 4004, 1, EMBED) == -1 and b"ne = 4n" in L.ls_last_error()
    assert _create(L, 1001, 1001, 2002, 2001, 0, EMBED) == -1 and b"ne = 2n-1" in L.ls_last_error()
    h = C.c_void_p()
    nu = np.zeros(4)
    rc = L.ls_op2d_create_gv(C.byref(h), 4097, 8, nu.ctypes.data_as(C.c_void_p), 1.0, 1.0, 1.0, EMBED)
    assert rc == -2 and b"4096" in L.ls_last_error()
    rc = L.ls_op2d_create_gv(C.byref(h), 1001, 1001, nu.ctypes.data_as(C.c_void_p), 1.0, 1.0, 1.0, EMBED | PAD4)
    assert rc == -2


def test_default_still_refuses_beyond_the_general_path(built_lib):
    """Without the flag nothing changes: Greengard_Vico (1000, 4000) is still beyond the Bluestein path."""
    from fast_solver_lippmann_schwinger_b200._lib import lib
    L = lib()
    assert _create(L, 1000, 1000, 4000, 4000, 1, 0) == -2 and b"4096" in L.ls_last_error()
    assert _create(L, 1500, 700, 2999, 1399, 0, 0) == -2          # trapezoidal: ne + n - 1 = 4498


def test_python_mirror(built_lib):
    import fast_solver_lippmann_schwinger_b200 as ls
    nu = np.zeros(5 * 5)
    with pytest.raises(ls.LSUnsupported):
        ls.FastM(np.zeros((20, 20), complex), nu, 20, 20, 5, 5, 1.0, quadRule="Greengard_Vico", embed=True, pad4=True)
    with pytest.raises(ls.LSCudaError) as ei:
        ls.FastM(None, nu, 20, 20, 5, 5, 1.0, quadRule="Greengard_Vico", L=1.0, Lp=1.0, embed=True, force_generic=True)
    assert ei.value.code == -1
    from fast_solver_lippmann_schwinger_b200._lib import lib
    assert lib().ls_op2d_info(None, None, None, None, None) == -1
