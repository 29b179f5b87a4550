"""CPU tests of LS_FLAG_EMBED's argument checks on the 3-D operator: every refusal happens before any CUDA or NCCL call,
so they run without a GPU.  The host arrays passed are deliberately tiny: a refusal that read them would read past their
end."""
import ctypes as C

import numpy as np
import pytest

EMBED, PAD4, FORCE_GENERIC = 4, 2, 1


def _create(L, n, m, l, flags, gfft=True):
    h = C.c_void_p()
    nu = np.zeros(4)
    g = np.zeros(16, complex)
    gp = g.ctypes.data_as(C.c_void_p) if gfft else None
    return L.ls_op3d_create(C.byref(h), n, m, l, 4 * n, 4 * m, 4 * l, nu.ctypes.data_as(C.c_void_p), gp,
                            1.0, 1.0, 4.0, flags)


def _create_dist(L, n, l, rank, nranks, flags):
    h = C.c_void_p()
    nu = np.zeros(4)
    uid = C.create_string_buffer(b"\x01" * 128, 128)        # not a valid NCCL id: a refusal must come before NCCL
    return L.ls_op3d_create_dist(C.byref(h), n, n, l, nu.ctypes.data_as(C.c_void_p), 1.0, 1.0, 4.0, rank, nranks,
                                 uid, flags)


def test_embed_flag_combinations_refused(built_lib):
    from fast_solver_lippmann_schwinger_b200._lib import lib
    L = lib()
    assert _create(L, 48, 48, 48, EMBED | PAD4) == -2
    assert b"2x padding" in L.ls_last_error()
    assert _create(L, 48, 48, 48, EMBED | FORCE_GENERIC) == -1
    assert b"FORCE_GENERIC" in L.ls_last_error()
    assert _create(L, 48, 48, 48, EMBED | FORCE_GENERIC | PAD4) == -1
    # the reference pads (ne, ne, le): n != m is invalid on every route
    assert _create(L, 48, 40, 48, EMBED) == -1 and b"n must equal m" in L.ls_last_error()


@pytest.mark.parametrize("n,l", [(513, 64), (64, 513), (600, 600)])
def test_embed_size_limit_named(built_lib, n, l):
    from fast_solver_lippmann_schwinger_b200._lib import lib
    L = lib()
    assert _create(L, n, n, l, EMBED) == -2
    assert b"512" in L.ls_last_error()
    assert _create(L, n, n, l, EMBED, gfft=False) == -2 and b"512" in L.ls_last_error()


def test_sharded_refusals_before_nccl(built_lib):
    from fast_solver_lippmann_schwinger_b200._lib import lib
    L = lib()
    # uneven z slabs are not served: l = 50 over 4 ranks, l = 101 over 2
    assert _create_dist(L, 48, 50, 0, 4, EMBED) == -2
    assert b"divide evenly" in L.ls_last_error()
    assert _create_dist(L, 100, 101, 1, 2, EMBED) == -2 and b"divide evenly" in L.ls_last_error()
    assert _create_dist(L, 48, 48, 0, 4, EMBED | PAD4) == -2
    assert _create_dist(L, 600, 64, 0, 2, EMBED) == -2 and b"512" in L.ls_last_error()
    assert _create_dist(L, 48, 48, 0, 3, EMBED) == -1             # rank counts stay 1, 2, 4, 8


def test_default_sharded_non_power_of_two_still_refused(built_lib):
    """Without the flag nothing changes: the sharded operator serves powers of two only."""
    from fast_solver_lippmann_schwinger_b200._lib import lib
    L = lib()
    assert _create_dist(L, 96, 96, 0, 2, 0) == -2
    assert b"powers of two" in L.ls_last_error()
    assert _create(L, 900, 900, 2, 0) == -2 and b"5n - 1" in L.ls_last_error()


@pytest.mark.parametrize("bad", ["0", "-4", "", "abc", "12x", "3.5", "99999999999999999999999"])
def test_embed_chunk_slots_refused(built_lib, monkeypatch, bad):
    """LS_OP3D_EMBED_CHUNK_SLOTS (x-slots per chunk of the lag extraction) takes a positive integer; anything else is
    refused before any CUDA or NCCL call, on one GPU and sharded."""
    from fast_solver_lippmann_schwinger_b200._lib import lib
    L = lib()
    monkeypatch.setenv("LS_OP3D_EMBED_CHUNK_SLOTS", bad)
    assert _create(L, 48, 48, 48, EMBED) == -1
    assert b"LS_OP3D_EMBED_CHUNK_SLOTS" in L.ls_last_error()
    assert _create(L, 48, 48, 48, EMBED, gfft=False) == -1
    assert _create_dist(L, 48, 48, 0, 2, EMBED) == -1 and b"LS_OP3D_EMBED_CHUNK_SLOTS" in L.ls_last_error()


def test_python_mirror(built_lib):
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200 import dist as lsd
    from fast_solver_lippmann_schwinger_b200._lib import lib
    nu = np.zeros(5 * 5 * 9)
    with pytest.raises(ls.LSUnsupported):
        ls.FastM3D(None, nu, 20, 20, 36, 5, 5, 9, 1.0, L=1.0, Lp=4.0, embed=True, pad4=True)
    with pytest.raises(ls.LSUnsupported):
        ls.FastM3D(None, np.zeros(513 * 513 * 2), 2052, 2052, 8, 513, 513, 2, 1.0, L=1.0, Lp=4.0, embed=True)
    with pytest.raises(ValueError):                              # dist.slab_range: equal slabs only
        lsd.FastM3DSharded(np.zeros(4), 48, 48, 50, 1.0, 1.0, 4.0, 0, 4, b"\x01" * 128, embed=True)
    assert lib().ls_op3d_lines(None, None, None, None, None) == -1
