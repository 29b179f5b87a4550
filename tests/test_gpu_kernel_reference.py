"""Every line-kernel instantiation of the 2-D and 3-D applies, at full line length, against an exact reference.

The reference needs no padded FFT: for a separable spectrum G = Gx (x) Gy (x) Gz the operator factorises exactly.
Each factor gives a spatial kernel along its axis,

    Greengard_Vico  gx = ifft(ifftshift(Gx)),  Tx[i, i'] = gx[(i - i') mod ne]
    trapezoidal     gx = ifft(Gx),             Tx[i, i'] = gx[(i - i' + n - 1) mod ne]   (crop at n - 1, FastConvolution.jl:82)

and fastconvolution(M, b) = b + omega^2 vec(Tx F Ty^T) with F = reshape(nu .* b, n, m) column-major (in 3-D Tz acts along
the third axis as well); FFTconvolution is the same without b and omega^2, and without nu for Greengard_Vico (Q2).
The factors are random complex vectors: the kernel then has energy at every lag, including the lags beyond +-n that the
compact (2x) and zero-embedded routes must drop, and no symmetry hides a mirrored or misplaced spectrum.

The reference is two or three dense products per apply, cheap at 4096^2 where the reference's own 4x padded FFT is
not; it shares no code with the product or the oracle.  The CPU tests check it against the oracle on small grids and
bound its own rounding at the largest case in long double.  The GPU tests hold the convolution part of each apply to
relative L2 <= 2e-14 and worst entry <= 2e-13 x RMS, far below the 1e-12 parity bar on y = b + omega^2 G(nu b), which
b dominates.  Run with -s for the table of measured errors.
"""
import ctypes as C

import numpy as np
import pytest
import scipy.fft as sfft

# Bars on the convolution part of an apply: one forward engine transform meets 1e-14 at every line length
# (tests/test_gpu_fft_engine.py) and an apply chains about six of them plus the create-time compaction.
L2_BAR = 2e-14
WORST_BAR = 2e-13
LINES = [64, 128, 256, 512, 1024, 2048, 4096]

# (route, quadRule, n, m); the route picks the flags: compact (default), pad4 (LS_FLAG_PAD4), embed (LS_FLAG_EMBED)
_THIN = [(4096, 64), (64, 4096), (2048, 256), (256, 2048), (1024, 128), (128, 1024), (512, 512), (2048, 2048)]
CASES_2D = ([("compact", "Greengard_Vico", n, m) for n, m in _THIN + [(4096, 4096)]]
            + [("pad4", "Greengard_Vico", n, m) for n, m in _THIN]
            + [("embed", "Greengard_Vico", n, m) for n, m in [(4001, 65), (65, 4001), (33, 257), (257, 33), (200, 130),
                                                              (4001, 4001)]]
            + [("embed", "trapezoidal", n, m) for n, m in [(2047, 601), (601, 2047), (1025, 1025)]])
# (pad4, n, l); n = m (FFTconvolution pads (ne, ne, le), FastConvolution3D.jl:48)
CASES_3D = [(pad4, n, l) for pad4 in (False, True) for n, l in [(256, 64), (64, 256), (128, 128), (64, 512)]]
LARGEST_2D = ("compact", "Greengard_Vico", 4096, 4096)


def _embed_len(n):
    return max(64, 1 << (n - 1).bit_length())


def _expected_info(route, n, m):
    """FastM.info() of a 2-D case: the route and the line lengths its P1/P3 (n_line) and P2 (m_line) kernels run."""
    if route == "embed":
        return {"route": 2, "n_line": _embed_len(n), "m_line": _embed_len(m), "padding_factor": 2}
    return {"route": 0, "n_line": n, "m_line": m, "padding_factor": 4 if route == "pad4" else 2}


def _id2(case):
    route, quad, n, m = case
    return "%s-%s-%dx%d" % (route, "gv" if quad == "Greengard_Vico" else "trap", n, m)


def _id3(case):
    pad4, n, l = case
    return "%s-%dx%dx%d" % ("pad4" if pad4 else "compact", n, n, l)


def _toeplitz(g, n, off):
    """T[i, i'] = g[(i - i' + off) mod len(g)]."""
    i = np.arange(n)
    return g[(i[:, None] - i[None, :] + off) % g.shape[0]]


def _axis(G, n, quad):
    """Spatial kernel of one spectrum factor and its n x n Toeplitz matrix."""
    if quad == "Greengard_Vico":
        g = sfft.ifft(sfft.ifftshift(G))
        return g, _toeplitz(g, n, 0)
    g = sfft.ifft(G)
    return g, _toeplitz(g, n, n - 1)


def _cplx(rng, *shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


class Sep2D:
    """A separable 2-D case: spectrum factors, their Toeplitz matrices, nu and b, all seeded by the shape."""

    def __init__(self, quad, n, m, rng=None):
        rng = np.random.default_rng([n, m, 0 if quad == "Greengard_Vico" else 1]) if rng is None else rng
        self.quad, self.n, self.m = quad, n, m
        self.ne, self.me = (4 * n, 4 * m) if quad == "Greengard_Vico" else (2 * n - 1, 2 * m - 1)
        self.Gx, self.Gy = _cplx(rng, self.ne), _cplx(rng, self.me)
        self.gx, self.Tx = _axis(self.Gx, n, quad)
        self.gy, self.Ty = _axis(self.Gy, m, quad)
        self.nu = rng.standard_normal(n * m)
        self.b = _cplx(rng, n * m)

    def spectrum(self):
        """GFFT[i, j] = Gx[i] Gy[j], built column-major (the transpose of a C-order outer product): no copy on upload."""
        return np.multiply.outer(self.Gy, self.Gx).T

    def conv(self, v):
        """vec(Tx F Ty^T), F = reshape(v, n, m) column-major."""
        F = v.reshape((self.n, self.m), order="F")
        return (self.Tx @ F @ self.Ty.T).reshape(-1, order="F")

    def column(self, idx):
        """conv(e_idx): Tx[:, i] (x) Ty[:, j] for the grid point idx = i + n j."""
        i, j = idx % self.n, idx // self.n
        return np.multiply.outer(self.Ty[:, j], self.Tx[:, i]).reshape(-1)


class Sep3D:
    """A separable Greengard_Vico 3-D case on an n x n x l grid."""

    def __init__(self, n, l, rng=None):
        rng = np.random.default_rng([n, l, 3]) if rng is None else rng
        self.n, self.m, self.l = n, n, l
        self.ne, self.me, self.le = 4 * n, 4 * n, 4 * l
        self.Gx, self.Gy, self.Gz = _cplx(rng, 4 * n), _cplx(rng, 4 * n), _cplx(rng, 4 * l)
        self.Tx = _axis(self.Gx, n, "Greengard_Vico")[1]
        self.Ty = _axis(self.Gy, n, "Greengard_Vico")[1]
        self.Tz = _axis(self.Gz, l, "Greengard_Vico")[1]
        self.nu = rng.standard_normal(n * n * l)
        self.b = _cplx(rng, n * n * l)

    def spectrum(self):
        return (self.Gz[:, None, None] * self.Gy[None, :, None] * self.Gx[None, None, :]).T

    def conv(self, v):
        n, m, l = self.n, self.m, self.l
        A = (self.Tx @ v.reshape((n, m * l), order="F")).reshape((n, m, l), order="F")   # x
        A = np.matmul(self.Ty, A)                                                         # y: (m x m) on each A[a]
        A = np.matmul(A, self.Tz.T)                                                       # z
        return A.reshape(-1, order="F")

    def column(self, idx):
        n, m = self.n, self.m
        i, j, k = idx % n, (idx // n) % m, idx // (n * m)
        return np.einsum("c,b,a->cba", self.Tz[:, k], self.Ty[:, j], self.Tx[:, i]).reshape(-1)


def _errors(d, ref, y=None, at_b=()):
    """(relative L2, worst entry / RMS) of d against ref.  At the entries at_b the output y also holds b: the final
    rounding of b + conv there (at most half an ulp of y) belongs to the float64 output, not to the kernels."""
    err = np.abs(d - ref)
    for i in at_b:
        err[i] = max(0.0, err[i] - 2.0 ** -52 * abs(y[i]))
    nref = np.linalg.norm(ref)
    return float(np.linalg.norm(err) / nref), float(err.max() / (nref / np.sqrt(ref.size)))


@pytest.fixture(scope="module")
def measured():
    """Collects every (case, check, relative L2, worst / RMS) and prints the table at the end of the module."""
    rows = []
    yield rows
    if rows:
        print("\nconvolution-part errors against the separable reference (bars: L2 %.0e, worst/RMS %.0e)"
              % (L2_BAR, WORST_BAR))
        for r in rows:
            print("  %-28s %-18s L2 %.2e  worst/RMS %.2e" % r)


def _check(measured, case, what, d, ref, y=None, at_b=()):
    l2, worst = _errors(d, ref, y, at_b)
    measured.append((case, what, l2, worst))
    assert l2 <= L2_BAR and worst <= WORST_BAR, "%s %s: relative L2 %.2e, worst/RMS %.2e" % (case, what, l2, worst)


def _omega(b, conv):
    """omega with ||omega^2 conv(nu b)|| = ||b||: neither part of y = b + omega^2 conv dominates."""
    return float(np.sqrt(np.linalg.norm(b) / np.linalg.norm(conv)))


# --------------------------------------------------------------------------------------------------------------------
# CPU: the reference itself
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("quad,n,m", [("Greengard_Vico", 16, 8), ("Greengard_Vico", 12, 12), ("trapezoidal", 9, 13),
                                      ("trapezoidal", 11, 11)])
def test_separable_reference_matches_oracle_2d(quad, n, m):
    from oracle import ls_oracle as O
    f = Sep2D(quad, n, m)
    Mo = O.FastM(f.spectrum(), f.nu, f.ne, f.me, n, m, 1.7, quadRule=quad)
    conv = f.conv(f.nu * f.b)
    yo = O.fastconvolution(Mo, f.b)
    assert np.linalg.norm(1.7 ** 2 * conv - (yo - f.b)) <= 1e-14 * np.linalg.norm(yo - f.b)
    if n == m:
        ref = f.conv(f.b if quad == "Greengard_Vico" else f.nu * f.b)
        co = O.FFTconvolution(Mo, f.b)
        assert np.linalg.norm(ref - co) <= 1e-14 * np.linalg.norm(co)
    e = np.zeros(n * m, complex)
    e[n * m - 1] = 1.0
    col = (O.fastconvolution(Mo, e) - e) / (1.7 ** 2 * f.nu[-1])
    assert np.linalg.norm(f.column(n * m - 1) - col) <= 1e-14 * np.linalg.norm(col)


def test_separable_reference_matches_oracle_3d():
    from oracle import ls_oracle as O
    f = Sep3D(8, 16)
    Mo = O.FastM3D(f.spectrum(), f.nu, f.ne, f.me, f.le, f.n, f.m, f.l, 0.9)
    yo = Mo * f.b
    assert np.linalg.norm(0.9 ** 2 * f.conv(f.nu * f.b) - (yo - f.b)) <= 1e-14 * np.linalg.norm(yo - f.b)
    co = O.FFTconvolution3D(Mo, f.b)
    assert np.linalg.norm(f.conv(f.b) - co) <= 1e-14 * np.linalg.norm(co)
    N = f.n * f.m * f.l
    e = np.zeros(N, complex)
    e[N - 1] = 1.0
    col = O.FFTconvolution3D(Mo, e)
    assert np.linalg.norm(f.column(N - 1) - col) <= 1e-14 * np.linalg.norm(col)


def _two_pi_ld():
    return np.longdouble(2) * np.arccos(np.longdouble(-1))


@pytest.mark.parametrize("case", [LARGEST_2D, ("embed", "trapezoidal", 2047, 601)], ids=_id2)
def test_reference_kernel_against_longdouble_dft(case):
    """gx, gy of the largest cases at 16 random lags against the inverse DFT summed in long double, with the angle
    reduced exactly in integers: the reference's float64 FFT is good to 1e-15 of the kernel's RMS on the power-of-two
    lengths.  The trapezoidal lengths 2n - 1 are odd (4093 is prime) and the FFT runs Bluestein there: 1.4e-15 was the
    worst of 64 lags at 4093, 1201 and 2049, so those are held to 2e-15, still a tenth of the GPU bar."""
    route, quad, n, m = case
    bar = 1e-15 if quad == "Greengard_Vico" else 2e-15
    f = Sep2D(quad, n, m)
    rng = np.random.default_rng(7)
    for G, g, size in ((f.Gx, f.gx, n), (f.Gy, f.gy, m)):
        ne = G.shape[0]
        freq = np.arange(ne, dtype=np.int64) - (ne // 2 if quad == "Greengard_Vico" else 0)   # centred for GV
        lags = np.concatenate([[0, size - 1, ne - size + 1], rng.choice(ne, 13, replace=False)])
        Gl = G.astype(np.clongdouble)
        rms = np.linalg.norm(g) / np.sqrt(ne)
        for d in lags:
            ang = _two_pi_ld() * ((freq * int(d)) % ne).astype(np.longdouble) / np.longdouble(ne)
            ref = np.sum(Gl * (np.cos(ang) + 1j * np.sin(ang))) / np.longdouble(ne)
            assert abs(complex(g[d] - ref)) <= bar * rms, (quad, ne, d)


def test_reference_rows_against_longdouble():
    """8 output rows of Tx F Ty^T at 4096^2 (the float64 products the GPU test uses) against the same products in long
    double: the reference's rounding is below 1e-15 of the RMS of its output in the L2 sense the GPU tests' 2e-14 bar
    uses.  Entry by entry, two 4096-term sums reach a few ulps: 1.9e-15 x RMS was measured (6e-16 in L2), held to 1e-14,
    a twentieth of the GPU tests' worst-entry bar."""
    route, quad, n, m = LARGEST_2D
    f = Sep2D(quad, n, m)
    F = (f.nu * f.b).reshape((n, m), order="F")
    ref = f.conv(f.nu * f.b).reshape((n, m), order="F")
    rms = np.linalg.norm(ref) / np.sqrt(ref.size)
    rows = np.array([0, 1, n // 2, n - 1] + list(np.random.default_rng(11).choice(np.arange(2, n - 1), 4, replace=False)))
    R = (f.Tx[rows].astype(np.clongdouble) @ F.astype(np.clongdouble)) @ f.Ty.T.astype(np.clongdouble)
    err = np.abs(ref[rows] - R).astype(np.float64)
    assert np.sqrt(np.mean(err ** 2)) <= 1e-15 * rms
    assert err.max() <= 1e-14 * rms


def test_cases_cover_every_line_length():
    """Every line kernel at every line length is launched by one of the cases below: the n side (P1/P3) and the m side
    (P2) of each 2-D route, and the x/y and z lines of both 3-D paddings."""
    for route in ("compact", "pad4", "embed"):
        info = [_expected_info(r, n, m) for r, q, n, m in CASES_2D if r == route]
        assert {i["n_line"] for i in info} == set(LINES), route
        assert {i["m_line"] for i in info} == set(LINES), route
    assert _expected_info("embed", 4001, 65) == {"route": 2, "n_line": 4096, "m_line": 128, "padding_factor": 2}
    assert _expected_info("embed", 1025, 1025)["n_line"] == 2048          # the worst embedding, ln = 2n - 2
    assert _expected_info("pad4", 64, 4096) == {"route": 0, "n_line": 64, "m_line": 4096, "padding_factor": 4}
    for pad4 in (False, True):
        assert {n for p, n, l in CASES_3D if p == pad4} == {64, 128, 256}
        assert {l for p, n, l in CASES_3D if p == pad4} == {64, 128, 256, 512}
    assert all(16 * (4 * n) ** 2 * 4 * l <= 4.3e9 for p, n, l in CASES_3D)    # host spectra at most 4.3 GB


# --------------------------------------------------------------------------------------------------------------------
# GPU: 2-D
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES_2D, ids=_id2)
def test_2d_apply_against_separable_reference(case, measured):
    import fast_solver_lippmann_schwinger_b200 as ls
    route, quad, n, m = case
    name = _id2(case)
    f = Sep2D(quad, n, m)
    N = n * m
    conv = f.conv(f.nu * f.b)
    omega = _omega(f.b, conv)
    G = f.spectrum()
    M = ls.FastM(G, f.nu, f.ne, f.me, n, m, omega, quadRule=quad, pad4=route == "pad4", embed=route == "embed")
    del G
    try:
        assert M.info() == _expected_info(route, n, m)
        y = M * f.b
        _check(measured, name, "random b", y - f.b, omega ** 2 * conv)
        del conv
        assert np.array_equal(M * f.b, y)                        # same handle, same input: same bits
        if route == "compact" and n == m == 4096:
            db = ls.DeviceBuffer.from_host(f.b)
            M.mul_(db, db)
            M.sync()
            assert np.array_equal(db.to_host(), y)
            db.free()
        del y
        for idx in (0, N - 1):                                   # the extreme lags +-(n-1), +-(m-1) in isolation
            e = np.zeros(N, complex)
            e[idx] = 1.0
            ye = M * e
            _check(measured, name, "impulse %d" % idx, ye - e, omega ** 2 * f.nu[idx] * f.column(idx), ye, (idx,))
        if n == m:
            ref = f.conv(f.b if quad == "Greengard_Vico" else f.nu * f.b)   # Q2: no nu for Greengard_Vico
            _check(measured, name, "FFTconvolution", ls.FFTconvolution(M, f.b), ref)
    finally:
        M.destroy()


# --------------------------------------------------------------------------------------------------------------------
# GPU: 3-D
# --------------------------------------------------------------------------------------------------------------------
def _padding_3d(M):
    from fast_solver_lippmann_schwinger_b200 import _lib
    pf, cx, ex = C.c_int(), C.c_int(), C.c_int()
    _lib.check(_lib.lib().ls_op3d_info(M.handle, C.byref(pf), C.byref(cx), C.byref(ex)))
    return pf.value


def _check_3d(measured, name, M, f, omega):
    N = f.n * f.m * f.l
    y = M * f.b
    _check(measured, name, "random b", y - f.b, omega ** 2 * f.conv(f.nu * f.b))
    assert np.array_equal(M * f.b, y)
    for idx in (0, N - 1):
        e = np.zeros(N, complex)
        e[idx] = 1.0
        ye = M * e
        _check(measured, name, "impulse %d" % idx, ye - e, omega ** 2 * f.nu[idx] * f.column(idx), ye, (idx,))
    from fast_solver_lippmann_schwinger_b200 import FFTconvolution
    _check(measured, name, "FFTconvolution", FFTconvolution(M, f.b), f.conv(f.b))
    return y


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES_3D, ids=_id3)
def test_3d_apply_against_separable_reference(case, measured):
    import fast_solver_lippmann_schwinger_b200 as ls
    pad4, n, l = case
    f = Sep3D(n, l)
    omega = _omega(f.b, f.conv(f.nu * f.b))
    G = f.spectrum()
    M = ls.FastM3D(G, f.nu, f.ne, f.me, f.le, n, n, l, omega, pad4=pad4)
    del G
    try:
        assert _padding_3d(M) == (4 if pad4 else 2)
        _check_3d(measured, _id3(case), M, f, omega)
    finally:
        M.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("n,l,chunks", [(64, 128, 2), (64, 128, 8), (128, 64, 4)])
def test_3d_setup_chunks_give_the_same_handle(n, l, chunks, monkeypatch, measured):
    """LS_OP3D_SETUP_CHUNKS splits the compact spectrum's set-up into x-slot chunks (taken by itself only when the 4x
    slab exceeds 20 GB, at 512^3 on one GPU).  Each line's arithmetic is the same: bit-identical applies, for the host
    spectrum and for the device-generated one (k_fill_g3d at the chunk's x-slot offset)."""
    import fast_solver_lippmann_schwinger_b200 as ls
    f = Sep3D(n, l)
    omega = _omega(f.b, f.conv(f.nu * f.b))
    G = f.spectrum()
    h = 1.0 / n
    gv = dict(L=1.8 * n * h, Lp=4.0 * n * h)
    k = 2 * np.pi / (10 * h)
    out = {}
    for c in (None, chunks):
        if c is None:
            monkeypatch.delenv("LS_OP3D_SETUP_CHUNKS", raising=False)
        else:
            monkeypatch.setenv("LS_OP3D_SETUP_CHUNKS", str(c))
        A = ls.FastM3D(G, f.nu, f.ne, f.me, f.le, n, n, l, omega)
        D = ls.FastM3D(None, f.nu, f.ne, f.me, f.le, n, n, l, k, **gv)
        try:
            assert _padding_3d(A) == 2 and _padding_3d(D) == 2
            if c is None:
                out[c] = (A * f.b, ls.FFTconvolution(A, f.b), D * f.b, ls.FFTconvolution(D, f.b))
            else:
                y = _check_3d(measured, "%dx%dx%d-C%d" % (n, n, l, c), A, f, omega)
                out[c] = (y, ls.FFTconvolution(A, f.b), D * f.b, ls.FFTconvolution(D, f.b))
        finally:
            A.destroy()
            D.destroy()
    for a, b in zip(out[None], out[chunks]):
        assert np.array_equal(a, b)


@pytest.mark.gpu
def test_3d_setup_chunks_refuses_what_the_slab_cannot_hold(monkeypatch):
    """C = 32 at n = 64 leaves 256 / 64 = 4 x-slots per half chunk (< 8): refused, not clamped; C = 16 is the largest
    that n = 64 takes, and a count that is not a power of two is refused too."""
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200._lib import LS_ERR_INVALID
    n = 64
    h = 1.0 / n
    nu = np.random.default_rng(2).standard_normal(n ** 3)
    args = (nu, 4 * n, 4 * n, 4 * n, n, n, n, 2 * np.pi / (10 * h))
    gv = dict(L=1.8 * n * h, Lp=4.0 * n * h)
    for bad in ("32", "3", "0"):
        monkeypatch.setenv("LS_OP3D_SETUP_CHUNKS", bad)
        with pytest.raises(ls.LSCudaError) as ei:
            ls.FastM3D(None, *args, **gv)
        assert ei.value.code == LS_ERR_INVALID and "LS_OP3D_SETUP_CHUNKS" in str(ei.value), bad
    monkeypatch.setenv("LS_OP3D_SETUP_CHUNKS", "16")
    M = ls.FastM3D(None, *args, **gv)
    M.destroy()
