"""GPU parity of the device-resident Msp^-1 on 3-D grids (ls_msp_factor3d): 27-point matrices against SuperLU, a grid
whose separators exceed the 48 KB staging limit against the device's own residual, the 2-D entry point as the l = 1 case
bit for bit, examples/example3D.jl:56-78 with the whole preconditioned GMRES on the device, and the memory check.

Tolerances as tests/test_gpu_msp.py: a direct solve agrees with SuperLU to 1e-10 relative, preconditioned GMRES residual
histories with the oracle to 1e-8 relative."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from util_sparse import stencil27  # noqa: E402
from test_gpu_msp import stencil9  # noqa: E402


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def shifted27(n, m, l, seed=0, classes=True):
    """Random complex 27-point matrix on the n x m x l grid, shifted on the diagonal to strict diagonal dominance: safely
    non-singular and well conditioned at every size (a fixed shift is not: the symbol of 27 random coefficients has
    zeros near some wave numbers, which the larger grids resolve)."""
    A = stencil27(n, m, l, seed=seed, classes=classes)
    shift = 1.0 + np.abs(A).sum(axis=1).max()
    A = (A + shift * sp.identity(n * m * l, format="csc")).tocsc()
    A.sort_indices()
    return A


GRIDS = [(1, 1, 1), (2, 3, 1), (3, 3, 3), (5, 6, 7), (9, 4, 3), (4, 4, 17), (12, 12, 12), (20, 20, 36), (32, 32, 32)]


@pytest.mark.parametrize("classes", [True, False])
@pytest.mark.parametrize("grid", GRIDS)
def test_msp3d_solve_matches_superlu(grid, classes):
    import fast_solver_lippmann_schwinger_b200 as ls
    n, m, l = grid
    N = n * m * l
    A = shifted27(n, m, l, seed=n + 7 * m + 31 * l, classes=classes)
    rng = np.random.default_rng(N)
    b = rng.standard_normal(N) + 1j * rng.standard_normal(N)
    F = ls.GPUMspFactorization(A, n, m, l)
    x = F.solve(b)
    x_ref = spla.splu(A).solve(b)
    assert _rel(x, x_ref) <= 1e-10
    assert np.linalg.norm(A @ x - b) / np.linalg.norm(b) <= 1e-11
    # device pointers: the first call captures the graph, the next ones replay it
    db, dx = ls.DeviceBuffer.from_host(b), ls.DeviceBuffer(b.nbytes)
    for _ in range(3):
        F.solve(db, dx)
    F.sync()
    assert np.array_equal(dx.to_host(), x)
    F.solve(db)                                             # in place
    F.sync()
    assert np.array_equal(db.to_host(), x)
    b2 = rng.standard_normal(N) + 1j * rng.standard_normal(N)    # a second right-hand side
    assert _rel(F.solve(b2), spla.splu(A).solve(b2)) <= 1e-10
    assert F.factor_bytes > 0 and F.depth >= 0
    db.free(); dx.free()
    F.destroy()


def test_msp3d_64_cubed_against_the_device_residual(monkeypatch):
    """64^3: separators of 4096 and rings of about 4160 unknowns, past the 48 KB staging limit, the upper depths on
    cuSOLVER; checked through the residual ||Msp x - b|| / ||b|| with Msp applied on the device."""
    import fast_solver_lippmann_schwinger_b200 as ls
    n = 64
    N = n ** 3
    A = shifted27(n, n, n, seed=64)
    F = ls.GPUMspFactorization(A, n, n, n)
    plan = F.plan()
    depths = [ln.split() for ln in plan.splitlines()[1:]]
    assert max(int(d[5]) for d in depths) == 4096                   # Sp of the root
    assert max(int(d[7]) for d in depths) > 3072                    # Bp past 48 KB of staged X
    assert any(d[-1] == "cusolver" for d in depths) and depths[-1][-1] == "batched"
    G = ls.GPUSparseMatrixCSC(A)
    rng = np.random.default_rng(1)
    for _ in range(2):
        b = rng.standard_normal(N) + 1j * rng.standard_normal(N)
        x = F.solve(b)
        assert np.linalg.norm(G * x - b) / np.linalg.norm(b) <= 1e-10
    db, dx = ls.DeviceBuffer.from_host(b), ls.DeviceBuffer(b.nbytes)
    for _ in range(3):
        F.solve(db, dx)
    F.sync()
    assert np.array_equal(dx.to_host(), x)
    db.free(); dx.free()
    # the first solver version (uniform batches, no staging in shared memory) on the same matrix
    monkeypatch.setenv("LS_MSP_SOLVER", "1")
    F1 = ls.GPUMspFactorization(A, n, n, n)
    assert _rel(F1.solve(b), x) <= 1e-12
    F1.destroy()
    G.destroy()
    F.destroy()


@pytest.mark.parametrize("n,m", [(1, 1), (3, 2), (9, 4), (17, 33), (40, 25), (130, 257), (201, 201)])
def test_factor3d_with_one_plane_is_the_2d_factorisation(n, m, monkeypatch):
    import fast_solver_lippmann_schwinger_b200 as ls
    monkeypatch.setenv("LS_MSP_TUNE", "0")
    A = stencil9(n, m, seed=7 * n + m)
    b = np.random.default_rng(n + m).standard_normal(n * m) + 0j
    F2 = ls.GPUMspFactorization(A, n, m)
    F3 = ls.GPUMspFactorization(A, n, m, 1)
    assert F3.plan() == F2.plan()
    assert F3.factor_bytes == F2.factor_bytes and F3.depth == F2.depth
    assert np.array_equal(F3.solve(b), F2.solve(b))
    F2.destroy(); F3.destroy()


def test_example3d_preconditioned_gmres_on_the_device():
    """gmres!(u, fastconv, rhs, precond) of examples/example3D.jl:56-78 on a 20 x 20 x 36 grid with Msp^-1 on the device
    (solverType="GPU"): the assertions of test_example3d_preconditioned_gmres_matches_oracle, no host work in the loop.
    Then with As and Msp sampled from GPU applies."""
    from oracle import ls_oracle as O
    from oracle.gmres_is import gmres as gmres_oracle
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200 import sparsifier as S
    n, l = 20, 36
    (x, z), h, k, Mo, As, Msp, Po = O.example_problem_3d(n, l)
    N = n * n * l
    X, Y, Z = O.grid3d(x, x, z)
    u_inc = np.exp(1j * k * X)
    rhs = -(Mo * u_inc - u_inc)                                   # example3D.jl:71-72
    uo, hist_o, conv_o, mv_o = gmres_oracle(np.zeros(N, complex), lambda v: Mo * v, rhs, Pl_ldiv=Po.solve)
    assert conv_o

    Mg = ls.FastM3D(Mo.GFFT, Mo.nu, Mo.ne, Mo.me, Mo.le, n, n, l, k)
    Pg = ls.SparsifyingPreconditioner(Msp, As, solverType="GPU", grid=(n, n, l))
    v = np.random.default_rng(3).standard_normal(N) + 0j
    assert _rel(Pg.solve(v), Po.solve(v)) <= 1e-9
    ug, hg = ls.gmres_(np.zeros(N, complex), Mg, rhs, Pl=Pg, log=True)
    assert hg.isconverged and hg.iters == len(hist_o)
    assert np.max(np.abs(hg["resnorm"] - hist_o) / hist_o) < 1e-8
    assert _rel(ug, uo) < 1e-7
    assert hg.msp_host_seconds == 0.0                              # nothing crossed PCIe inside the loop
    Pg.destroy()

    As_g, Msp_g = S.sparsifying_matrices_3d(k, X, Y, Z, Mg, n, n, l, Mo.nu)
    Pd = ls.SparsifyingPreconditioner(Msp_g, As_g, solverType="GPU", grid=(n, n, l))
    w = np.random.default_rng(8).standard_normal(N) + 0j
    assert _rel(Pd.solve(w), Po.solve(w)) <= 1e-7
    ud, hd = ls.gmres_(np.zeros(N, complex), Mg, rhs, Pl=Pd, log=True)
    assert hd.isconverged and np.linalg.norm(Mg * ud - rhs) / np.linalg.norm(rhs) < 1e-6
    Pd.destroy()


def test_memory_check_refuses_before_allocating():
    """A 160^3 grid (an empty pattern: colptr all ones) needs more than a B200 holds: LS_ERR_NOMEM with the byte counts
    in the message, nothing allocated; a small 3-D factorisation in the same process still works afterwards."""
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200 import _lib
    n = 160
    N = n ** 3
    colptr = np.ones(N + 1, np.int64)
    csc = (N, N, colptr, np.ones(1, np.int64), np.zeros(1, complex))
    with pytest.raises(ls.LSCudaError) as e:
        ls.GPUMspFactorization(csc, n, n, n)
    assert e.value.code == _lib.LS_ERR_NOMEM
    msg = str(e.value)
    assert "needs" in msg and "free" in msg
    need = int(msg.split(" needs ")[1].split()[0])
    assert need > 180e9
    A = shifted27(6, 5, 4, seed=2)
    F = ls.GPUMspFactorization(A, 6, 5, 4)
    b = np.ones(A.shape[0], complex)
    assert _rel(F.solve(b), spla.splu(A).solve(b)) <= 1e-10
    F.destroy()


def test_msp3d_refuses_what_it_does_not_serve():
    import fast_solver_lippmann_schwinger_b200 as ls
    n, m, l = 6, 5, 4
    A = shifted27(n, m, l, seed=4).tolil()
    A[0, 2] = 1.0                                         # two cells apart in x
    with pytest.raises(ls.LSUnsupported):
        ls.GPUMspFactorization(A.tocsc(), n, m, l)
    with pytest.raises(ValueError):
        ls.GPUMspFactorization(shifted27(n, m, l), n, m, l + 1)
    # duplicates are summed before the call: the same matrix as its canonical form
    B = shifted27(n, m, l, seed=5)
    C = B.tocoo()
    dup = sp.csc_matrix((np.concatenate([C.data, [1.0]]), (np.concatenate([C.row, [3]]), np.concatenate([C.col, [3]]))),
                        shape=B.shape)
    B2 = B.tolil()
    B2[3, 3] += 1.0
    b = np.ones(B.shape[0], complex)
    F = ls.GPUMspFactorization(dup, n, m, l)
    assert _rel(F.solve(b), spla.splu(B2.tocsc()).solve(b)) <= 1e-10
    F.destroy()
    Z = sp.csc_matrix((n * m * l, n * m * l), dtype=complex)
    with pytest.raises(ls.LSCudaError):                   # singular pivot block
        ls.GPUMspFactorization(Z, n, m, l)
