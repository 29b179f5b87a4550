"""Several right-hand sides on the device: ls_msp_solve_batch against ls_msp_solve column by column (bit for bit), and
ls_gmres_msp_batch against ls_gmres_msp run on each right-hand side alone (bit for bit) and against the oracle's GMRES."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from test_gpu_msp import stencil9  # noqa: E402

pytestmark = pytest.mark.gpu

NRHS = [1, 2, 3, 4, 5, 8, 13]


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def _rhs(N, K, seed):
    rng = np.random.default_rng(seed)
    return np.asfortranarray(rng.standard_normal((N, K)) + 1j * rng.standard_normal((N, K)))


@pytest.fixture(scope="module")
def ls():
    import fast_solver_lippmann_schwinger_b200 as ls
    return ls


@pytest.fixture(scope="module")
def grid3d_48(ls):
    """examples/example3D.jl at 48^3 (h = 1/48, k = 1/h) with As and Msp sampled from GPU applies."""
    from oracle import ls_oracle as O
    from fast_solver_lippmann_schwinger_b200 import sparsifier as S
    n = 48
    h = 1.0 / n
    x = -0.5 + h * np.arange(n)
    k = 1.0 / h
    X, Y, Z = O.grid3d(x, x, x)
    nu = O.nu_gaussian_3d(X, Y, Z)
    span = x[-1] - x[0] + h
    Mg = ls.FastM3D(None, nu, 4 * n, 4 * n, 4 * n, n, n, n, k, L=1.5 * span, Lp=4 * span)
    As, Msp = S.sparsifying_matrices_3d(k, X, Y, Z, Mg, n, n, n, nu)
    P = ls.SparsifyingPreconditioner(Msp, As, solverType="GPU", grid=(n, n, n))
    yield dict(n=n, k=k, X=X, Y=Y, Z=Z, Mg=Mg, P=P, Msp=Msp.tocsr())
    P.destroy()


def _factor(ls, which, grid3d_48):
    if which == "3d48":
        return grid3d_48["P"].MspGPU, grid3d_48["Msp"], False
    n = int(which.split("_")[1])
    A = stencil9(n, n, seed=n)
    return ls.GPUMspFactorization(A, n, n), A.tocsr(), True


@pytest.mark.parametrize("which", ["2d_257", "2d_1024", "3d48"])
def test_batch_solve_is_the_single_solve_bit_for_bit(ls, grid3d_48, which):
    from fast_solver_lippmann_schwinger_b200._lib import MEM_DEVICE, check, lib
    F, A, own = _factor(ls, which, grid3d_48)
    N = F.N
    plan = F.plan()
    assert " cols U" in plan
    B = _rhs(N, max(NRHS), 17)
    single = np.asfortranarray(np.stack([F.solve(B[:, j]) for j in range(B.shape[1])], axis=1))
    for K in NRHS:
        X = F.solve(B[:, :K])                                                   # host pointers
        assert np.array_equal(_bits(X), _bits(single[:, :K])), (which, K)
    res = np.linalg.norm(A @ single - B, axis=0) / np.linalg.norm(B, axis=0)
    assert res.max() <= 1e-12, res.max()
    # device pointers with ld > N, then in place; every width twice (the second call replays the captured graphs)
    ld = N + 7
    for K in (3, 5, 13):
        Bp = np.zeros((ld, K), complex, order="F")
        Bp[:N] = B[:, :K]
        db = ls.DeviceBuffer.from_host(Bp.reshape(-1, order="F"))
        dx = ls.DeviceBuffer(db.nbytes)
        for _ in range(2):
            check(lib().ls_msp_solve_batch(F.handle, C.c_void_p(db.ptr), ld, C.c_void_p(dx.ptr), ld, K, MEM_DEVICE))
        F.sync()
        got = dx.to_host().reshape(ld, K, order="F")[:N]
        assert np.array_equal(_bits(got), _bits(single[:, :K])), (which, K, "device")
        check(lib().ls_msp_solve_batch(F.handle, C.c_void_p(db.ptr), ld, C.c_void_p(db.ptr), ld, K, MEM_DEVICE))
        F.sync()
        got = db.to_host().reshape(ld, K, order="F")[:N]
        assert np.array_equal(_bits(got), _bits(single[:, :K])), (which, K, "in place")
        db.free(); dx.free()
    # in place through host pointers
    H = np.asfortranarray(B[:, :8].copy())
    check(lib().ls_msp_solve_batch(F.handle, H.ctypes.data_as(C.c_void_p), N, H.ctypes.data_as(C.c_void_p), N, 8, 0))
    assert np.array_equal(_bits(H), _bits(single[:, :8]))
    if own:
        F.destroy()


@pytest.mark.parametrize("cols", ["2", "8"])
def test_other_chunk_widths_keep_the_bits(ls, cols, monkeypatch):
    """LS_MSP_BATCH_COLS: chunks of at most 2, or of up to 8 columns (the NRHS = 8 kernel), give the same columns."""
    monkeypatch.setenv("LS_MSP_BATCH_COLS", cols)
    n = 257
    F = ls.GPUMspFactorization(stencil9(n, n, seed=n), n, n)
    B = _rhs(n * n, 13, 23)
    single = np.asfortranarray(np.stack([F.solve(B[:, j]) for j in range(13)], axis=1))
    for K in (8, 13):
        assert np.array_equal(_bits(F.solve(B[:, :K])), _bits(single[:, :K])), (cols, K)
    F.destroy()


def test_a_nan_column_leaves_the_others_alone(ls):
    n = 257
    F = ls.GPUMspFactorization(stencil9(n, n, seed=3), n, n)
    N = n * n
    B = _rhs(N, 8, 5)
    clean = F.solve(B)
    Bn = B.copy(order="F")
    Bn[:, 3] = np.nan
    dirty = F.solve(Bn)
    for j in range(8):
        if j != 3:
            assert np.array_equal(_bits(dirty[:, j]), _bits(clean[:, j])), j
    assert np.isnan(dirty[:, 3]).all()
    assert np.array_equal(_bits(F.solve(B)), _bits(clean))             # no trace of the NaN in the kept work arrays
    F.destroy()


def test_batch_solve_refusals(ls):
    from fast_solver_lippmann_schwinger_b200._lib import LS_ERR_INVALID, LS_ERR_NOMEM, lib
    n = 64
    F = ls.GPUMspFactorization(stencil9(n, n, seed=1), n, n)
    N = n * n
    B = _rhs(N, 4, 1)
    p = B.ctypes.data_as(C.c_void_p)
    L = lib()
    assert L.ls_msp_solve_batch(F.handle, p, N - 1, p, N, 4, 0) == LS_ERR_INVALID
    q = C.c_void_p(p.value + 16 * N)
    assert L.ls_msp_solve_batch(F.handle, p, N, q, N, 4, 0) == LS_ERR_INVALID      # overlapping, not in place
    assert L.ls_msp_solve_batch(F.handle, p, N, p, N + 1, 2, 0) == LS_ERR_INVALID  # same start, different ld
    assert b"in place" in L.ls_last_error()
    F.destroy()


def test_lockstep_gmres_refuses_too_many_systems_before_allocating(ls):
    """60000 bases of 65 vectors of 4096 unknowns (255 GB) do not fit a B200: LS_ERR_NOMEM with the byte counts, before
    b and x are touched or anything is allocated; a small batch on the same handles works afterwards."""
    from fast_solver_lippmann_schwinger_b200._lib import LS_ERR_NOMEM, lib
    from oracle import ls_oracle as O
    n = 64
    x, h, k, Mo = O.pow2_problem_2d(n)
    N = n * n
    Mg = ls.FastM(Mo.GFFT, Mo.nu, Mo.ne, Mo.me, n, n, k, quadRule="Greengard_Vico")
    A = stencil9(n, n, seed=4)
    P = ls.SparsifyingPreconditioner(A, A, solverType="GPU", grid=(n, n))
    ws = ls.KrylovWorkspace(N)
    db = ls.DeviceBuffer(16 * N)
    n64, ci = C.c_int64(), C.c_int()
    rc = lib().ls_gmres_msp_batch(ws.handle, Mg.handle, P.As.handle, P.MspGPU.handle, 60000, C.c_void_p(db.ptr), N,
                                  C.c_void_p(db.ptr), N, 64, 10, 1e-8, 0.0, 1, None, 0, C.byref(n64), C.byref(ci),
                                  C.byref(n64), 1)
    assert rc == LS_ERR_NOMEM
    msg = lib().ls_last_error()
    assert b"60000 systems" in msg and b"bytes are free" in msg
    B = _rhs(N, 2, 3)
    X, hs = ls.gmres_(np.zeros((N, 2), complex, order="F"), Mg, B, Pl=P, log=True, maxiter=5)
    assert [h.iters for h in hs] == [5, 5]
    db.free(); ws.destroy(); P.destroy()


def _plane_waves(k, X, Y, thetas):
    return [np.exp(1j * k * (X * np.cos(t) + Y * np.sin(t))) for t in thetas]


def _compare_with_single(ls, Mg, P, B, **kw):
    """batch run of B's columns vs ls.gmres_ on each column alone: histories, counts and x bit for bit"""
    N, K = B.shape
    Xb = np.zeros((N, K), complex, order="F")
    Xb, hs = ls.gmres_(Xb, Mg, B, Pl=P, log=True, **kw)
    for q in range(K):
        xq, hq = ls.gmres_(np.zeros(N, complex), Mg, np.ascontiguousarray(B[:, q]), Pl=P, log=True, **kw)
        assert (hs[q].iters, hs[q].isconverged, hs[q].mvps) == (hq.iters, hq.isconverged, hq.mvps), q
        assert np.array_equal(_bits(hs[q]["resnorm"]), _bits(hq["resnorm"])), q
        assert np.array_equal(_bits(Xb[:, q]), _bits(xq)), q
    return Xb, hs


def test_lockstep_gmres_2d_is_each_system_alone_bit_for_bit(ls):
    from oracle import ls_oracle as O
    from oracle.gmres_is import gmres as gmres_oracle
    n = 257
    h = 1.0 / n
    x = -0.5 + h * np.arange(n)
    k = 1.0 / h
    Mo = O.buildFastConvolution(x, x, h, k, O.nu_gaussian_2d, quadRule="Greengard_Vico")
    X, Y = O.grid2d(x, x)
    D0 = O.referenceValsTrapRule()[1][0]
    cache = O.entriesSparseA(k, X, Y, D0, n, n, strict=False)
    As = O.buildSparseA(k, X, Y, D0, n, n, strict=False, _cache=cache)
    AG = O.buildSparseAG(k, X, Y, D0, n, n, strict=False, _cache=cache)
    Msp = (As + k ** 2 * (AG @ sp.diags(Mo.nu))).tocsc()
    Mg = ls.FastM(Mo.GFFT, Mo.nu, Mo.ne, Mo.me, n, n, k, quadRule="Greengard_Vico")
    P = ls.SparsifyingPreconditioner(Msp, As, solverType="GPU", grid=(n, n))
    u = _plane_waves(k, X, Y, np.linspace(0, np.pi, 4, endpoint=False))
    rhs = [-k ** 2 * O.FFTconvolution(Mo, Mo.nu * ui) for ui in u]          # examples/example.jl:76-77
    nb = np.linalg.norm(rhs[0])
    # four directions, one scaled down (reaches abstol early), one below abstol (converged at the start)
    B = np.asfortranarray(np.stack([rhs[0], 1e-4 * rhs[1], 1e-14 * rhs[2], rhs[3]], axis=1))
    abstol = 1e-9 * nb
    _, hs = _compare_with_single(ls, Mg, P, B, abstol=abstol, maxiter=200)
    iters = [h.iters for h in hs]
    assert iters[2] == 0 and hs[2].isconverged
    assert len(set(iters)) >= 3, iters                                       # systems leave at different iterations
    assert all(h.isconverged for h in hs)
    # the oracle's GMRES (SuperLU preconditioner) on the first direction
    Po = O.SparsifyingPreconditioner(Msp, As)
    _, hist_o, conv_o, mv_o = gmres_oracle(np.zeros(n * n, complex), lambda w: O.fastconvolution(Mo, w), rhs[0],
                                           Pl_ldiv=Po.solve, abstol=abstol, maxiter=200)
    assert hs[0].iters == len(hist_o) and hs[0].mvps == mv_o
    mm = min(50, len(hist_o))
    assert np.max(np.abs(hs[0]["resnorm"][:mm] - hist_o[:mm]) / hist_o[:mm]) < 1e-8
    # maxiter inside a restart cycle (restart 3, maxiter 5; with abstol deciding, direction 0 needs 6 iterations
    # even unrestarted): x of the last restart, as the single-system driver
    _, hs = _compare_with_single(ls, Mg, P, B, abstol=abstol, restart=3, maxiter=5, reltol=1e-14)
    assert hs[2].iters == 0
    assert hs[0].iters == 5 and not hs[0].isconverged, (hs[0].iters, hs[0].isconverged)
    P.destroy()


def test_lockstep_gmres_3d_is_each_system_alone_bit_for_bit(ls, grid3d_48):
    g = grid3d_48
    k, X, Y, Z = g["k"], g["X"], g["Y"], g["Z"]
    u = [np.exp(1j * k * (X * np.cos(t) + Y * np.sin(t))) for t in (0.0, 1.1, 2.3)]
    rhs = [-(g["Mg"] * ui - ui) for ui in u]                                  # example3D.jl:71-72
    B = np.asfortranarray(np.stack([rhs[0], 1e-3 * rhs[1], rhs[2]], axis=1))
    _, hs = _compare_with_single(ls, g["Mg"], g["P"], B, abstol=1e-8 * np.linalg.norm(rhs[0]), maxiter=60)
    assert all(h.isconverged for h in hs)


def test_example_py_with_four_directions(ls):
    root = os.path.dirname(HERE)
    p = subprocess.run([sys.executable, os.path.join(root, "examples", "example.py"), "--n", "201", "--nrhs", "4", "--msp", "gpu"],
                       capture_output=True, text=True, cwd=root, timeout=1800)
    assert p.returncode == 0, p.stdout + p.stderr
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("direction")]
    assert len(lines) == 4 and all("converged True" in ln for ln in lines), p.stdout
