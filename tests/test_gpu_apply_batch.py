"""Several right-hand sides through one operator: every column of ls_op_apply_batch against ls_op2d_apply /
ls_op3d_apply of that column (bit for bit), on every route, and ls_gmres_batch against ls_gmres (Pl = Identity) run on
each right-hand side alone (bit for bit)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NRHS = [1, 2, 3, 4, 5, 8, 13]


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


@pytest.fixture(scope="module")
def ls():
    import fast_solver_lippmann_schwinger_b200 as ls
    return ls


def _check_batch(ls, M, nrhs_list, modes=(0, 1), seed=0):
    """ls_op_apply_batch with host and device pointers, ld = N + 3 and in place, against the single apply of each column"""
    from fast_solver_lippmann_schwinger_b200._lib import DeviceBuffer, check, lib
    N = M.N
    Kmax = max(nrhs_list)
    ld = N + 3
    rng = np.random.default_rng(seed)
    B = np.zeros((ld, Kmax), dtype=np.complex128, order="F")
    B[:N] = rng.standard_normal((N, Kmax)) + 1j * rng.standard_normal((N, Kmax))
    db = DeviceBuffer.from_host(B.reshape(-1, order="F"))
    dy = DeviceBuffer(B.nbytes)
    L = lib()
    for mode in modes:
        ref = np.stack([M._apply(np.ascontiguousarray(B[:N, j]), None, mode) for j in range(Kmax)], axis=1)
        for K in nrhs_list:
            Y = np.zeros((ld, K), dtype=np.complex128, order="F")
            check(L.ls_op_apply_batch(M.handle, C.c_void_p(B.ctypes.data), ld, C.c_void_p(Y.ctypes.data), ld, K, mode, 0))
            assert np.array_equal(_bits(Y[:N]), _bits(ref[:, :K])), ("host", mode, K)
            check(L.ls_op_apply_batch(M.handle, C.c_void_p(db.ptr), ld, C.c_void_p(dy.ptr), ld, K, mode, 1))
            check(L.ls_sync(M.handle))       # device pointers: the apply is enqueued on the handle's stream
            Yd = dy.to_host(count=ld * K).reshape((ld, K), order="F")
            assert np.array_equal(_bits(Yd[:N]), _bits(ref[:, :K])), ("device", mode, K)
        # in place on the device: y == b
        K = nrhs_list[-1]
        dz = DeviceBuffer.from_host(B.reshape(-1, order="F"))
        check(L.ls_op_apply_batch(M.handle, C.c_void_p(dz.ptr), ld, C.c_void_p(dz.ptr), ld, K, mode, 1))
        check(L.ls_sync(M.handle))
        Z = dz.to_host(count=ld * K).reshape((ld, K), order="F")
        assert np.array_equal(_bits(Z[:N]), _bits(ref[:, :K])), ("in place", mode, K)
    return M


def _cols(M):
    import fast_solver_lippmann_schwinger_b200 as ls
    return ls.batch_cols(M)


def _gv2d(ls, n, **kw):
    """n x n Greengard_Vico operator with the device-generated spectrum (h = 1/n, 10 points per wavelength)"""
    h = 1.0 / n
    x = -0.5 + h * np.arange(n)
    g = np.exp(-40 * x ** 2)
    nu = np.ascontiguousarray((0.3 * g[:, None] * g[None, :]).reshape(-1, order="F"))
    k = 2 * np.pi / (10 * h)
    return ls.FastM(None, nu, 4 * n, 4 * n, n, n, k, quadRule="Greengard_Vico", L=1.5 * n * h, Lp=4.0 * n * h, **kw)


@pytest.mark.parametrize("n", [64, 256, 2048, 4096])
def test_2d_fast_path_columns_equal_single_applies(ls, n):
    M = _gv2d(ls, n)
    assert M.info()["route"] == 0 and _cols(M) > 1
    _check_batch(ls, M, [2, 5] if n >= 2048 else NRHS, seed=n)


def _embedded_2d(ls, n, m, quad):
    from oracle import ls_oracle as O
    if quad == "Greengard_Vico":
        h = 1.0 / n
        x = -0.5 + h * np.arange(n)
        y = -0.5 * m / n + h * np.arange(m)
        Mo = O.buildFastConvolution(x, y, h, 2 * np.pi / (8.3 * h), O.nu_gaussian_2d, quadRule="Greengard_Vico")
    else:
        h = 1.0 / (max(n, m) - 1)
        x = -0.5 * (n - 1) * h + h * np.arange(n)
        y = -0.5 * (m - 1) * h + h * np.arange(m)
        Mo = O.buildFastConvolution(x, y, h, 1.0 / h, O.nu_gaussian_2d, quadRule="trapezoidal")
    return Mo, ls.FastM(Mo.GFFT, Mo.nu, Mo.ne, Mo.me, Mo.n, Mo.m, Mo.omega, quadRule=Mo.quadRule, embed=True)


@pytest.mark.parametrize("n,m", [(201, 201), (1001, 777)])
@pytest.mark.parametrize("quad", ["Greengard_Vico", "trapezoidal"])
def test_2d_embedded_columns_equal_single_applies(ls, n, m, quad):
    Mo, M = _embedded_2d(ls, n, m, quad)
    assert M.info()["route"] == 2 and _cols(M) > 1
    _check_batch(ls, M, NRHS, modes=(0, 1) if n == m else (0,), seed=n + m)


def test_2d_bluestein_and_pad4_go_column_by_column(ls):
    from oracle import ls_oracle as O
    Mo, _ = _embedded_2d(ls, 100, 100, "Greengard_Vico")
    Mb = ls.FastM(Mo.GFFT, Mo.nu, Mo.ne, Mo.me, 100, 100, Mo.omega, quadRule="Greengard_Vico")
    assert Mb.info()["route"] == 1 and _cols(Mb) == 1
    _check_batch(ls, Mb, NRHS, seed=1)
    x, h, k, Mo = O.pow2_problem_2d(64)
    Mp = ls.FastM(Mo.GFFT, Mo.nu, Mo.ne, Mo.me, 64, 64, Mo.omega, quadRule="Greengard_Vico", pad4=True)
    assert Mp.info()["padding_factor"] == 4 and _cols(Mp) == 1
    _check_batch(ls, Mp, NRHS, seed=2)


def _device3d(ls, n, l, **kw):
    h = 1.0 / n
    x = -0.5 + h * np.arange(n)
    z = -0.5 * l / n + h * np.arange(l)
    g = np.exp(-40 * x ** 2)
    gz = np.exp(-40 * z ** 2)
    nu = np.ascontiguousarray((0.3 * g[:, None, None] * g[None, :, None] * gz[None, None, :]).reshape(-1, order="F"))
    k = 2 * np.pi / (10 * h)
    return ls.FastM3D(None, nu, 4 * n, 4 * n, 4 * l, n, n, l, k, L=1.8 * n * h, Lp=4.0 * n * h, **kw)


@pytest.mark.parametrize("n,l,embed", [(64, 64, False), (256, 256, False), (48, 48, True), (100, 70, True)])
def test_3d_columns_equal_single_applies(ls, n, l, embed):
    M = _device3d(ls, n, l, embed=embed)
    assert M.lines()["route"] == (2 if embed else 0) and _cols(M) >= 1
    _check_batch(ls, M, [2, 5] if n >= 256 else NRHS, seed=n + l)


def test_batch_against_oracle(ls):
    from oracle import ls_oracle as O
    Mo, M = _embedded_2d(ls, 201, 201, "Greengard_Vico")
    rng = np.random.default_rng(5)
    B = rng.standard_normal((M.N, 4)) + 1j * rng.standard_normal((M.N, 4))
    Y = M * B
    for j in range(4):
        ref = O.fastconvolution(Mo, B[:, j])
        assert np.linalg.norm(Y[:, j] - ref) / np.linalg.norm(ref) <= 1e-12


def test_batch_refusals_on_a_live_handle(ls):
    from fast_solver_lippmann_schwinger_b200._lib import LS_ERR_INVALID, DeviceBuffer, lib
    L = lib()
    M = _gv2d(ls, 64)
    N = M.N
    d = DeviceBuffer(16 * (2 * N + 8))
    p, q = C.c_void_p(d.ptr), C.c_void_p(d.ptr + 16 * 4)
    assert L.ls_op_apply_batch(M.handle, p, N - 1, p, N, 2, 0, 1) == LS_ERR_INVALID      # ld < N
    assert L.ls_op_apply_batch(M.handle, p, N, q, N, 2, 0, 1) == LS_ERR_INVALID          # overlap, not in place
    assert L.ls_op_apply_batch(M.handle, p, N, p, N + 1, 2, 0, 1) == LS_ERR_INVALID      # same start, different ld
    assert L.ls_op_apply_batch(M.handle, p, N, p, N, 2, 7, 1) == LS_ERR_INVALID          # mode
    assert L.ls_op_apply_batch(M.handle, p, N, p, N, 2, 0, 9) == LS_ERR_INVALID          # memloc
    Mo, Mr = _embedded_2d(ls, 1001, 777, "Greengard_Vico")
    assert L.ls_op_apply_batch(Mr.handle, p, Mr.N, p, Mr.N, 1, 1, 1) == LS_ERR_INVALID    # FFTconvolution: square only
    with pytest.raises(ValueError):
        M * np.zeros((N + 1, 2), complex)
    with pytest.raises(ValueError):
        M * np.zeros(N + 1, complex)


def test_gmres_batch_equals_solo_runs(ls):
    """Pl = Identity: systems converging at different iterations and one at maxiter, bit for bit against ls_gmres"""
    Mo, M = _embedded_2d(ls, 201, 201, "Greengard_Vico")
    N = M.N
    rng = np.random.default_rng(11)
    B = np.empty((N, 4), complex, order="F")
    B[:, 0] = M * np.ones(N, complex)
    B[:, 1] = rng.standard_normal(N) + 1j * rng.standard_normal(N)
    B[:, 2] = 1e-3 * B[:, 1] + B[:, 0]
    B[:, 3] = rng.standard_normal(N)
    kw = dict(reltol=1e-10, restart=20, log=True)

    def solo(q, maxiter):
        x = np.zeros(N, complex)
        return ls.gmres_(x, M, np.ascontiguousarray(B[:, q]), maxiter=maxiter, **kw)
    free = [solo(q, 400)[1].iters for q in range(4)]
    assert len(set(free)) > 1, free                          # the systems converge at different iterations
    maxiter = max(free) - 1                                  # the slowest one stops at maxiter
    X = np.zeros((N, 4), complex, order="F")
    X, hs = ls.gmres_(X, M, B, Pl=None, maxiter=maxiter, **kw)
    conv = []
    for q in range(4):
        x, h = solo(q, maxiter)
        assert np.array_equal(_bits(X[:, q]), _bits(x)), q
        assert np.array_equal(_bits(hs[q]["resnorm"]), _bits(h["resnorm"])), q
        assert (hs[q].iters, hs[q].isconverged, hs[q].mvps) == (h.iters, h.isconverged, h.mvps), q
        conv.append(h.isconverged)
    assert not all(conv) and any(conv), conv


def test_gmres_batch_memory_check_before_allocation():
    """8 systems at 512^3 with restart 20: the bases alone are 8 x 21 x 2.1 GB"""
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200._lib import LS_ERR_NOMEM, DeviceBuffer, lib
    L = lib()
    M = _device3d(ls, 512, 512)
    ws = ls.KrylovWorkspace(M.N)
    d = DeviceBuffer(16 * M.N)
    n64 = np.zeros(8, np.int64)
    ci = np.zeros(8, np.int32)
    rc = L.ls_gmres_batch(ws.handle, M.handle, 8, C.c_void_p(d.ptr), 0, C.c_void_p(d.ptr), 0, 20, 10, 1e-8, 0.0, 1, None, 0,
                          C.c_void_p(n64.ctypes.data), C.c_void_p(ci.ctypes.data), C.c_void_p(n64.ctypes.data), 1)
    assert rc != 0   # ld = 0 < N
    rc = L.ls_gmres_batch(ws.handle, M.handle, 8, C.c_void_p(d.ptr), M.N, C.c_void_p(d.ptr), M.N, 20, 10, 1e-8, 0.0, 1, None, 0,
                          C.c_void_p(n64.ctypes.data), C.c_void_p(ci.ctypes.data), C.c_void_p(n64.ctypes.data), 1)
    assert rc == LS_ERR_NOMEM, L.ls_last_error()
    msg = L.ls_last_error().decode()
    assert "bytes of device memory" in msg and "free" in msg, msg
