"""GPU checks of the zero-embedded 3-D route (LS_FLAG_EMBED): any n = m, l <= 512 on the power-of-two kernels of
n' = max(64, nextpow2(n)) and l', on one GPU and sharded.

Tolerances: relative L2 <= 1e-12 against the oracle and the Bluestein route, <= 1e-13 against the power-of-two fast path
and between the sharded and the single-GPU embedded applies; GMRES histories within 1e-8."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
TOL = 1e-12
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, "tests", "dist_embed_worker.py")


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _pow(n):
    p = 64
    while p < n:
        p *= 2
    return p


def _problem(n, l, k=None):
    """Greengard_Vico on x = -1/2:h:1/2-h (h = 1/n), z likewise with l points; 8.3 points per wavelength unless k is
    given (with 10, s == k falls exactly on grid frequencies whenever 0.4 n is an integer, and the reference's spectrum
    holds NaN there, Q7).  Odd n: the oracle's builder refuses the reference's unfinished odd-n branch, so the
    even-n spectrum (the one the device generates for every n) is put into the oracle's FastM3D directly."""
    from oracle import ls_oracle as O
    h = 1.0 / n
    x = -0.5 + h * np.arange(n)
    z = -0.5 * l / n + h * np.arange(l)
    k = 2 * np.pi / (8.3 * h) if k is None else k
    if n % 2 == 0:
        return h, O.buildFastConvolution3D(x, x, z, h, k, O.nu_gaussian_3d)
    X, Y, Z = O.grid3d(x, x, z)
    return h, O.FastM3D(O.gv_spectrum_3d(n, n, l, h, k), np.asarray(O.nu_gaussian_3d(X, Y, Z), dtype=np.float64),
                        4 * n, 4 * n, 4 * l, n, n, l, k)


def _nu(n, l):
    h = 1.0 / n
    x = -0.5 + h * np.arange(n)
    z = -0.5 * l / n + h * np.arange(l)
    g = np.exp(-40 * x ** 2)
    gz = np.exp(-40 * z ** 2)
    return np.ascontiguousarray((0.3 * g[:, None, None] * g[None, :, None] * gz[None, None, :]).reshape(-1, order="F"))


def _device(n, l, k, **kw):
    """Handle with the device-generated spectrum (L = 1.8, Lp = 4 in units of the x extent, as the oracle builds it)."""
    import fast_solver_lippmann_schwinger_b200 as ls
    h = 1.0 / n
    return ls.FastM3D(None, _nu(n, l), 4 * n, 4 * n, 4 * l, n, n, l, k, L=1.8 * n * h, Lp=4.0 * n * h, **kw)


@pytest.mark.parametrize("n,l", [(48, 48), (5, 9), (20, 36), (100, 37), (65, 130)])
def test_against_oracle(n, l):
    from oracle import ls_oracle as O
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200._lib import ROUTE_EMBEDDED
    # (48, 48): examples/example3D.jl as shipped, k = 1/h
    h, Mo = _problem(n, l, k=n if (n, l) == (48, 48) else None)
    Mg = ls.FastM3D(Mo.GFFT, Mo.nu, Mo.ne, Mo.me, Mo.le, n, n, l, Mo.omega, embed=True)
    assert Mg.lines() == {"route": ROUTE_EMBEDDED, "n_line": _pow(n), "m_line": _pow(n), "l_line": _pow(l)}
    N = n * n * l
    rng = np.random.default_rng(n + 7 * l)
    b = rng.standard_normal(N) + 1j * rng.standard_normal(N)
    c = rng.standard_normal(N) + 1j * rng.standard_normal(N)
    y = Mg * b
    assert Mg.launch_count() == 5
    y_ref = Mo * b
    assert _rel(y, y_ref) <= TOL
    assert _rel(y - b, y_ref - b) <= 1e-11          # the convolution part alone
    assert _rel(ls.FFTconvolution(Mg, b), O.FFTconvolution3D(Mo, b)) <= TOL
    # the second apply must not see the first one's data in the padding planes l..l'-1
    assert _rel(Mg * c, Mo * c) <= TOL
    assert np.array_equal(Mg * b, y)
    # device-generated spectrum
    Mgen = ls.FastM3D(None, Mo.nu, Mo.ne, Mo.me, Mo.le, n, n, l, Mo.omega, L=1.8 * n * h, Lp=4.0 * n * h, embed=True)
    assert Mgen.lines()["route"] == ROUTE_EMBEDDED
    assert _rel(Mgen * b, y_ref) <= TOL
    assert _rel(ls.FFTconvolution(Mgen, c), O.FFTconvolution3D(Mo, c)) <= TOL
    # device buffers, b and y aliased
    db = ls.DeviceBuffer.from_host(b)
    Mg.mul_(db, db)
    Mg.sync()
    assert np.array_equal(db.to_host(), y)


@pytest.mark.parametrize("n", [255, 301])
def test_against_bluestein(n):
    from fast_solver_lippmann_schwinger_b200._lib import ROUTE_BLUESTEIN, ROUTE_EMBEDDED
    k = 2 * np.pi / (8.3 / n)
    Mb = _device(n, n, k)
    assert Mb.lines()["route"] == ROUTE_BLUESTEIN
    rng = np.random.default_rng(n)
    b = rng.standard_normal(n ** 3) + 1j * rng.standard_normal(n ** 3)
    yb = Mb * b
    Mb.destroy()
    Me = _device(n, n, k, embed=True)
    assert Me.lines() == {"route": ROUTE_EMBEDDED, "n_line": 512 if n > 256 else 256, "m_line": 512 if n > 256 else 256,
                          "l_line": 512 if n > 256 else 256}
    assert _rel(Me * b, yb) <= TOL


def test_512_against_the_fast_path():
    """n = l = 512 with the flag runs the fast path's kernels with the lags extracted by ZGEMM; without it the lags come
    from compact_spectrum3d's pruned FFTs."""
    from fast_solver_lippmann_schwinger_b200._lib import ROUTE_EMBEDDED, ROUTE_POW2
    n = 512
    k = 2 * np.pi / (8.3 / n)
    rng = np.random.default_rng(512)
    b = rng.standard_normal(n ** 3) + 1j * rng.standard_normal(n ** 3)
    Mf = _device(n, n, k)
    assert Mf.lines() == {"route": ROUTE_POW2, "n_line": 512, "m_line": 512, "l_line": 512}
    yf = Mf * b
    Mf.destroy()
    Me = _device(n, n, k, embed=True)
    assert Me.lines() == {"route": ROUTE_EMBEDDED, "n_line": 512, "m_line": 512, "l_line": 512}
    ye = Me * b
    assert _rel(ye, yf) <= 1e-13
    assert _rel(ye - b, yf - b) <= 1e-12


def test_511_properties():
    """511^3: too large for the oracle; linearity and reciprocity (the kernel is symmetric: (M e_a)[b] / nu[a] equals
    (M e_b)[a] / nu[b]) as in test_3d_full_size_properties."""
    n = 511
    k = 2 * np.pi / (8.3 / n)
    M = _device(n, n, k, embed=True)
    nu = _nu(n, n)
    N = n ** 3
    rng = np.random.default_rng(11)
    b = rng.standard_normal(N) + 1j * rng.standard_normal(N)
    c = rng.standard_normal(N) + 1j * rng.standard_normal(N)
    assert _rel(M * (b + 2j * c), M * b + 2j * (M * c)) <= 1e-13
    for ia, ib in (((250, 260, 255), (262, 247, 250)), ((0, 0, 0), (510, 510, 510)), ((3, 500, 17), (480, 9, 490))):
        a_idx = ia[0] + n * ia[1] + n * n * ia[2]
        b_idx = ib[0] + n * ib[1] + n * n * ib[2]
        ea = np.zeros(N, complex); ea[a_idx] = 1.0
        eb = np.zeros(N, complex); eb[b_idx] = 1.0
        ra = (M * ea)[b_idx] / nu[a_idx]
        rb = (M * eb)[a_idx] / nu[b_idx]
        assert abs(ra - rb) <= 1e-11 * abs(ra)


def test_gmres_msp_48_matches_bluestein():
    """examples/example3D.jl at n = 48 with Msp^-1 on the device (ls_msp_factor3d, ls_gmres_msp): the embedded route's
    history against the Bluestein route's over the first 50 iterations."""
    from oracle import ls_oracle as O
    import fast_solver_lippmann_schwinger_b200 as ls
    import scipy.sparse as sp
    n = 48
    h = 1.0 / n
    x = -0.5 + h * np.arange(n)
    k = 1.0 / h
    Mo = O.buildFastConvolution3D(x, x, x, h, k, O.nu_gaussian_3d)
    N = n ** 3
    X, Y, Z = O.grid3d(x, x, x)
    cache = O.entriesSparseA3D(k, X, Y, Z, Mo, n, n, n)          # As and Msp as example_problem_3d builds them
    As = O.buildSparseA3DConv(k, X, Y, Z, Mo, n, n, n, _cache=cache)
    AG = O.buildSparseAG3DConv(k, X, Y, Z, Mo, n, n, n, _cache=cache)
    Msp = (As + k ** 2 * (AG @ sp.diags(Mo.nu))).tocsc()
    u_inc = np.exp(1j * k * X)
    rhs = -(Mo * u_inc - u_inc)
    Mb = ls.FastM3D(Mo.GFFT, Mo.nu, Mo.ne, Mo.me, Mo.le, n, n, n, k)
    Me = ls.FastM3D(Mo.GFFT, Mo.nu, Mo.ne, Mo.me, Mo.le, n, n, n, k, embed=True)
    assert Mb.lines()["route"] == 1 and Me.lines()["route"] == 2
    hist = []
    for M in (Mb, Me):
        Pg = ls.SparsifyingPreconditioner(Msp, As, solverType="GPU", grid=(n, n, n))
        _, hg = ls.gmres_(np.zeros(N, complex), M, rhs, Pl=Pg, maxiter=50, log=True)
        assert hg.msp_host_seconds == 0.0
        hist.append(np.asarray(hg["resnorm"]))
        Pg.destroy()
    assert len(hist[0]) == len(hist[1]) and len(hist[0]) >= 3
    assert np.max(np.abs(hist[1] - hist[0]) / hist[0]) < 1e-8


def _gpu_count():
    try:
        out = subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True, timeout=20).stdout
        return sum(1 for line in out.splitlines() if line.startswith("GPU "))
    except Exception:
        return 0


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_embedded(world):
    """n = l = 96 on 2 / 4 / 8 GPUs (tests/dist_embed_worker.py); on 8 also 400^3."""
    if _gpu_count() < world:
        pytest.skip("needs %d GPUs" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(29660 + world), WORKER, "96"]
    env = dict(os.environ)
    env.setdefault("OMP_NUM_THREADS", "4")
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=1800, env=env, cwd=ROOT)
    assert p.returncode == 0 and "DIST_EMBED_OK" in p.stdout, p.stdout[-3000:] + p.stderr[-4000:]
