"""Host mirror of the preconditioner and GMRES interface of the reference, on libls_cuda.so.

    reference (Julia)                                          here
    ---------------------------------------------------------  ----------------------------------
    As * b  (SparseMatrixCSC * Vector)                         GPUSparseMatrixCSC(As) * b
      preconditioner.jl:138,142,159,163
    SparseBLAS.cscmv!(transa, a, descr, A, x, beta, y)         cscmv_(transa, a, descr, A, x, beta, y)
      sparseblas.jl:14-25
    SparsifyingPreconditioner(Msp, As; solverType)  :27-58     SparsifyingPreconditioner(Msp, As, solverType=)
    M \\ b  :132-145,  ldiv!(M, b)  :147-170                     M.solve(b), M.ldiv_(b)
    gmres!(x, A, b; Pl, log, restart, maxiter, reltol, ...)    gmres_(x, A, b, Pl=, log=, ...)
      IterativeSolvers.jl (un-vendored), examples/example.jl:85

    lu(Msp)  (MspInv, preconditioner.jl:35)                    GPUMspFactorization(Msp, n, m[, l])  [solverType="GPU"]

The sparse direct solve `MspInv \\ .` (UMFPACK / MKL PARDISO upstream) has two routes here (SURVEY.md H1):
solverType="GPU" factorises Msp on the device (ls_msp_factor / ls_msp_factor3d: nested dissection, 2-D 9-point and
3-D 27-point matrices) so the
whole preconditioned GMRES loop runs without PCIe traffic; solverType="UMFPACK" keeps it on the host with the
caller - scipy's SuperLU plays UMFPACK's part and is reached through the ls_solve_cb callback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import CDouble, DeviceBuffer, LSCudaError, SOLVE_CB, check, lib, ptr
from .operators import _Handle, _as_c128


def _julia_csc(A):
    """(nrows, ncols, colptr, rowval, nzval) in Julia's 1-based SparseMatrixCSC layout."""
    if isinstance(A, tuple):
        nrows, ncols, colptr, rowval, nzval = A
        return (int(nrows), int(ncols), np.ascontiguousarray(colptr, dtype=np.int64),
                np.ascontiguousarray(rowval, dtype=np.int64), np.ascontiguousarray(nzval, dtype=np.complex128))
    A = A.tocsc()
    A.sort_indices()
    return (A.shape[0], A.shape[1], A.indptr.astype(np.int64) + 1, A.indices.astype(np.int64) + 1,
            np.ascontiguousarray(A.data, dtype=np.complex128))


class GPUSparseMatrixCSC(_Handle):
    """A SparseMatrixCSC{ComplexF64,Int64} resident on the GPU (CSR/int32 internally)."""

    def __init__(self, A):
        super().__init__()
        nrows, ncols, colptr, rowval, nzval = _julia_csc(A)
        if colptr.shape[0] != ncols + 1:
            raise ValueError("colptr must have ncols+1 entries")
        self.shape = (nrows, ncols)
        self.nnz = int(colptr[-1] - 1)
        check(lib().ls_spm_create(C.byref(self._h), nrows, ncols, ptr(colptr), ptr(rowval), ptr(nzval)))
        fmt, ncl = C.c_int(), C.c_int()
        check(lib().ls_spm_info(self.handle, None, None, None, C.byref(fmt), C.byref(ncl)))
        self.format = "stencil" if fmt.value == 1 else "csr"      # device storage chosen at create time
        self.nclasses = int(ncl.value)

    def mv(self, x, y=None, alpha=1.0, beta=0.0):
        """y <- alpha*A*x + beta*y  (cscmv! with transa='N')."""
        if isinstance(x, DeviceBuffer):
            if not isinstance(y, DeviceBuffer):
                raise TypeError("device x needs a device y")
            check(lib().ls_spm_mv(self.handle, CDouble.of(alpha), ptr(x), CDouble.of(beta), ptr(y), _lib.MEM_DEVICE))
            return y
        x = _as_c128(x, self.shape[1], "x")
        if y is None:
            if beta != 0:
                raise ValueError("beta != 0 needs y")
            y = np.empty(self.shape[0], dtype=np.complex128)
        elif not (isinstance(y, np.ndarray) and y.dtype == np.complex128 and y.shape == (self.shape[0],)
                  and y.flags.c_contiguous):
            raise ValueError("DimensionMismatch: y must be a contiguous complex128 vector of length %d" % self.shape[0])
        check(lib().ls_spm_mv(self.handle, CDouble.of(alpha), ptr(x), CDouble.of(beta), ptr(y), _lib.MEM_HOST))
        return y

    def __mul__(self, x):
        return self.mv(x)

    __matmul__ = __mul__


def cscmv_(transa, alpha, matdescra, A: GPUSparseMatrixCSC, x, beta, y):
    """``SparseBLAS.cscmv!`` (sparseblas.jl:14-25) - only the reference's own use is served:
    transa='N', general matrix ("GXXF"), preconditioner.jl:194,237."""
    if transa != "N":
        raise _lib.LSUnsupported(_lib.LS_ERR_UNSUPPORTED, "cscmv!: only transa='N' is used by the reference")
    if not matdescra.startswith("G"):
        raise _lib.LSUnsupported(_lib.LS_ERR_UNSUPPORTED, "cscmv!: only general matrices ('GXXF')")
    if len(x) != A.shape[1]:
        raise ValueError("DimensionMismatch: Matrix with %d columns multiplied with vector of length %d" % (A.shape[1], len(x)))
    if len(y) != A.shape[0]:
        raise ValueError("DimensionMismatch: Vector of length %d added to vector of length %d" % (A.shape[0], len(y)))
    return A.mv(x, y, alpha=alpha, beta=beta)


class GPUMspFactorization(_Handle):
    """``lu(Msp)`` (preconditioner.jl:35) on the GPU: nested-dissection factorisation of the 9-point matrix Msp of
    the n x m grid (ls_msp_factor), or with ``l`` of the 27-point matrix of the n x m x l grid (ls_msp_factor3d,
    examples/example3D.jl:56-61).  ``solve(b)`` = ``MspInv \\ b`` on host arrays or DeviceBuffers.  A scipy matrix is
    canonicalised first (duplicates summed, indices sorted; the caller's matrix is not modified)."""

    def __init__(self, Msp, n, m, l=None):
        super().__init__()
        if not isinstance(Msp, tuple):
            Msp = Msp.tocsc(copy=True)
            Msp.sum_duplicates()
            Msp.sort_indices()
        nrows, ncols, colptr, rowval, nzval = _julia_csc(Msp)
        self.n, self.m = int(n), int(m)
        self.l = 1 if l is None else int(l)
        N = self.n * self.m * self.l
        if nrows != ncols or nrows != N:
            raise ValueError("DimensionMismatch: Msp is %d x %d, the grid has %d unknowns" % (nrows, ncols, N))
        self.N = nrows
        if l is None:
            check(lib().ls_msp_factor(C.byref(self._h), self.n, self.m, ptr(colptr), ptr(rowval), ptr(nzval)))
        else:
            check(lib().ls_msp_factor3d(C.byref(self._h), self.n, self.m, self.l, ptr(colptr), ptr(rowval), ptr(nzval)))
        fb, dep, sec = C.c_int64(), C.c_int(), C.c_double()
        check(lib().ls_msp_info(self.handle, C.byref(fb), C.byref(dep), C.byref(sec)))
        self.factor_bytes, self.depth, self.factor_seconds = int(fb.value), int(dep.value), float(sec.value)

    def plan(self):
        """Text description of the solve plan (ls_msp_plan): solver version and, per dissection depth, the block sizes and
        the kernel geometry of the three sweeps."""
        buf = C.create_string_buffer(16384)
        check(lib().ls_msp_plan(self.handle, buf, len(buf)))
        return buf.value.decode()

    def solve(self, b, out=None):
        if isinstance(b, DeviceBuffer):
            out = b if out is None else out
            check(lib().ls_msp_solve(self.handle, ptr(b), ptr(out), _lib.MEM_DEVICE))
            return out
        b = _as_c128(b, self.N, "b")
        out = np.empty(self.N, dtype=np.complex128) if out is None else out
        check(lib().ls_msp_solve(self.handle, ptr(b), ptr(out), _lib.MEM_HOST))
        return out


class SparsifyingPreconditioner:
    """``struct SparsifyingPreconditioner`` (preconditioner.jl:27-58).

    As lives on the GPU.  MspInv is the host sparse LU (solverType "UMFPACK" / "MKLPARDISO" as upstream; SuperLU
    here) or, with solverType="GPU" and the grid size (n, m) or (n, m, l), the device factorisation (no host work
    inside gmres!).
    """

    def __init__(self, Msp, As, solverType="UMFPACK", grid=None):
        import scipy.sparse.linalg as spla
        if solverType not in ("UMFPACK", "MKLPARDISO", "GPU"):
            raise ValueError("unknown solverType %r" % (solverType,))
        self.solverType = solverType
        self.Msp = Msp.tocsc()
        self.As_host = As
        self.As = GPUSparseMatrixCSC(As)
        self.N = self.Msp.shape[0]
        self.MspGPU = None
        if solverType == "GPU":
            if grid is None:
                raise ValueError("solverType='GPU' needs grid=(n, m) or (n, m, l)")
            self.MspGPU = GPUMspFactorization(self.Msp, *grid)
            self.MspInv = self.MspGPU
            self._cb = C.cast(None, SOLVE_CB)
            return
        self.MspInv = spla.splu(self.Msp)          # lu(Msp), preconditioner.jl:35

        def _cb(user, vptr, n):
            try:
                buf = (C.c_double * (2 * n)).from_address(vptr)
                v = np.frombuffer(buf, dtype=np.complex128)
                v[:] = self.MspInv.solve(v)
                return 0
            except Exception:      # never let an exception cross the C ABI
                return 1
        self._cb = SOLVE_CB(_cb)

    def solve(self, b):
        """``M \\ b``  preconditioner.jl:132-145."""
        return self.MspInv.solve(self.As * b)

    def destroy(self):
        self.As.destroy()
        if self.MspGPU is not None:
            self.MspGPU.destroy()

    def ldiv_(self, b):
        """``ldiv!(M, b)``  preconditioner.jl:147-166 (in place)."""
        b[:] = self.solve(b)
        return b


class ConvergenceHistory:
    """The part of IterativeSolvers.ConvergenceHistory the reference reads (example.jl:86-87)."""

    def __init__(self, resnorm, iters, isconverged, mvps, restart):
        self.data = {"resnorm": resnorm}
        self.iters = iters
        self.isconverged = isconverged
        self.mvps = mvps
        self.restart = restart

    def __getitem__(self, key):
        return self.data[key if isinstance(key, str) else str(key)]

    @property
    def residuals(self):          # the older `info[2].residuals` spelling, example3D.jl:79
        return self.data["resnorm"]


class KrylovWorkspace(_Handle):
    """Reduction buffers + resident Krylov basis for vectors of length n."""

    def __init__(self, n):
        super().__init__()
        self.n = int(n)
        check(lib().ls_krylov_create(C.byref(self._h), self.n))

    def dot(self, x: DeviceBuffer, y: DeviceBuffer):
        r = CDouble()
        check(lib().ls_zdotc(self.handle, ptr(x), ptr(y), C.byref(r)))
        return complex(r.re, r.im)

    def norm(self, x: DeviceBuffer):
        r = C.c_double()
        check(lib().ls_dznrm2(self.handle, ptr(x), C.byref(r)))
        return float(r.value)

    def axpy(self, alpha, x: DeviceBuffer, y: DeviceBuffer):
        check(lib().ls_zaxpy(self.handle, CDouble.of(alpha), ptr(x), ptr(y)))

    def scal(self, alpha, x: DeviceBuffer):
        check(lib().ls_zscal(self.handle, CDouble.of(alpha), ptr(x)))

    def mgs_step(self, V: DeviceBuffer, ldv, k, w):
        """orthogonalize_and_normalize!(V[:,1:k], w, h): returns h (k+1 values).  ``w`` is a
        DeviceBuffer or a raw device address (a column of V)."""
        h = np.empty(k + 1, dtype=np.complex128)
        check(lib().ls_mgs_step(self.handle, ptr(V), ldv, k, ptr(w), ptr(h)))
        return h


ORTH_METHODS = {"ModifiedGramSchmidt": 0, "ClassicalGramSchmidt": 1, "DGKS": 2}


def gmres_(x, A, b, Pl=None, abstol=0.0, reltol=None, restart=None, maxiter=None, log=False,
           initially_zero=False, workspace=None, orth_meth="ModifiedGramSchmidt"):
    """``gmres!(x, A, b; Pl, abstol, reltol, restart, maxiter, log, initially_zero)``.

    A is a GPU operator (FastM / FastM3D); Pl is None (Identity) or a SparsifyingPreconditioner.
    x is updated in place (numpy array or DeviceBuffer).  Returns x, or (x, history) with log=True.
    """
    N = A.size(1)
    reltol = float(np.sqrt(np.finfo(np.float64).eps)) if reltol is None else float(reltol)
    restart = min(20, N) if restart is None else int(restart)
    maxiter = getattr(A, "N_global", N) if maxiter is None else max(int(maxiter), 0)
    ws = workspace if workspace is not None else KrylovWorkspace(N)
    if orth_meth not in ORTH_METHODS:
        raise ValueError("orth_meth must be one of %s" % sorted(ORTH_METHODS))
    check(lib().ls_krylov_set_orth(ws.handle, ORTH_METHODS[orth_meth]))
    dev = isinstance(x, DeviceBuffer)
    if dev != isinstance(b, DeviceBuffer):
        raise TypeError("x and b must both be DeviceBuffer or both numpy arrays")
    if not dev:
        b = _as_c128(b, N, "b")
        if not (isinstance(x, np.ndarray) and x.dtype == np.complex128 and x.shape == (N,) and x.flags.c_contiguous):
            raise ValueError("DimensionMismatch: x must be a contiguous complex128 vector of length %d" % N)
    cap = maxiter if maxiter < 1_000_000 else 1_000_000
    hist = np.zeros(max(cap, 1), dtype=np.float64)
    niter, conv, mv = C.c_int64(), C.c_int(), C.c_int64()
    as_h = Pl.As.handle if (Pl is not None and Pl.As is not None) else None
    memloc = _lib.MEM_DEVICE if dev else _lib.MEM_HOST
    if Pl is not None and getattr(Pl, "MspGPU", None) is not None:
        check(lib().ls_gmres_msp(ws.handle, A.handle, as_h, Pl.MspGPU.handle, ptr(b), ptr(x), restart, maxiter, reltol,
                                 float(abstol), 1 if initially_zero else 0, ptr(hist), cap, C.byref(niter), C.byref(conv),
                                 C.byref(mv), memloc))
    else:
        cb = Pl._cb if Pl is not None else C.cast(None, SOLVE_CB)
        check(lib().ls_gmres(ws.handle, A.handle, as_h, cb, None, ptr(b), ptr(x), restart, maxiter, reltol, float(abstol),
                             1 if initially_zero else 0, ptr(hist), cap, C.byref(niter), C.byref(conv), C.byref(mv), memloc))
    if not log:
        return x
    n = min(int(niter.value), cap)
    h = ConvergenceHistory(hist[:n].copy(), int(niter.value), bool(conv.value), int(mv.value), restart)
    sec = C.c_double()
    check(lib().ls_krylov_last_precond_host_seconds(ws.handle, C.byref(sec)))
    h.msp_host_seconds = float(sec.value)      # D2H + host Msp solve + H2D inside the loop (0 with solverType="GPU")
    return x, h
