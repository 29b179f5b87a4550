"""Host-side mirror of the reference's operator objects, backed by libls_cuda.so.

The reference is Julia and Julia is not installed in this image, so this module plays the
role of ``julia/LSCuda.jl`` (the same C-ABI calls through ctypes instead of ccall) and keeps
the reference's names and argument meaning:

    reference (Julia)                               here
    ----------------------------------------------  ---------------------------------------
    struct FastM(GFFT,nu,ne,me,n,m,k; quadRule)     FastM(GFFT, nu, ne, me, n, m, k, quadRule=)
      FastConvolution.jl:11-27
    M * b, fastconvolution(M, b)      :43-107       M * b, fastconvolution(M, b)
    mul!(Y, M, b)                     :50-54        M.mul_(Y, b)   /  mul_(Y, M, b)
    size(M, dim), size(M), eltype(M)  :31-41        M.size(dim), M.size(), M.eltype()
    FFTconvolution(M, b)              :110-154      FFTconvolution(M, b)

Arrays are numpy complex128 vectors in the reference's column-major grid order (x fastest),
or DeviceBuffer objects for callers that keep their vectors on the GPU.  There is no CPU
fallback: every method ends in a kernel launch inside libls_cuda.so or raises.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import DeviceBuffer, LSCudaError, check, lib, ptr


class _Handle:
    """Owns an ls_handle; freed like a Julia finalizer would."""

    def __init__(self):
        self._h = C.c_void_p()

    @property
    def handle(self):
        if not self._h:
            raise LSCudaError(_lib.LS_ERR_INVALID, "operator handle already destroyed")
        return self._h

    def destroy(self):
        if self._h:
            lib().ls_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass

    def sync(self):
        check(lib().ls_sync(self.handle))

    def timer_start(self):
        check(lib().ls_timer_start(self.handle))

    def timer_stop(self):
        ms = C.c_float()
        check(lib().ls_timer_stop(self.handle, C.byref(ms)))
        return float(ms.value)

    def profile_enable(self, on=True):
        check(lib().ls_profile_enable(self.handle, 1 if on else 0))

    def profile_read(self, nphase=8):
        ms = (C.c_double * nphase)()
        cnt = (C.c_int64 * nphase)()
        check(lib().ls_profile_read(self.handle, ms, cnt, nphase))
        return [float(x) for x in ms], [int(x) for x in cnt]

    def launch_count(self):
        c = C.c_int64()
        check(lib().ls_launch_count(self.handle, C.byref(c)))
        return int(c.value)


def _as_c128(b, N, name="b"):
    b = np.asarray(b)
    if b.dtype != np.complex128:
        # the reference's methods are typed AbstractArray{Complex{Float64},1}; anything else is a MethodError
        raise TypeError("%s must be complex128 (Julia: Array{Complex{Float64},1}), got %s" % (name, b.dtype))
    if b.ndim != 1 or b.shape[0] != N:
        raise ValueError("DimensionMismatch: %s has shape %s, operator needs (%d,)" % (name, b.shape, N))
    return np.ascontiguousarray(b)


def _apply_cols(M, B, out, mode):
    """The columns of an (N, K) complex128 array through one ls_op_apply_batch (each column with the bits of the single
    apply of it); out, when given, is an (N, K) complex128 array that receives them."""
    if B.dtype != np.complex128:
        raise TypeError("b must be complex128 (Julia: Array{Complex{Float64},2}), got %s" % B.dtype)
    if B.shape[0] != M.N or B.shape[1] < 1:
        raise ValueError("DimensionMismatch: b has shape %s, operator needs (%d, K)" % (B.shape, M.N))
    K = B.shape[1]
    Bf = np.asfortranarray(B)
    if out is None:
        out = np.empty((M.N, K), dtype=np.complex128, order="F")
    elif not (isinstance(out, np.ndarray) and out.dtype == np.complex128 and out.shape == B.shape):
        raise ValueError("DimensionMismatch: Y must be a complex128 array of shape %s" % (B.shape,))
    Y = out if out.flags.f_contiguous else np.empty((M.N, K), dtype=np.complex128, order="F")
    check(lib().ls_op_apply_batch(M.handle, ptr(Bf), M.N, ptr(Y), M.N, K, mode, _lib.MEM_HOST))
    if Y is not out:
        out[...] = Y
    return out


def apply_batch(M, b, y, nrhs, ldb=None, ldy=None, mode=_lib.APPLY_FASTCONVOLUTION):
    """ls_op_apply_batch on device memory: b and y are DeviceBuffers holding nrhs columns of M's N unknowns, column j at
    j*ldb (j*ldy) elements (default N); y may be b for an in-place apply."""
    if not (isinstance(b, DeviceBuffer) and isinstance(y, DeviceBuffer)):
        raise TypeError("b and y must be DeviceBuffers (numpy arrays go through M * B)")
    N = M.N
    ldb = N if ldb is None else int(ldb)
    ldy = N if ldy is None else int(ldy)
    check(lib().ls_op_apply_batch(M.handle, ptr(b), ldb, ptr(y), ldy, int(nrhs), mode, _lib.MEM_DEVICE))
    return y


def batch_cols(M):
    """ls_op_batch_cols: the columns M applies per multi-column launch (1: column by column)."""
    c = C.c_int()
    check(lib().ls_op_batch_cols(M.handle, C.byref(c)))
    return int(c.value)


class FastM(_Handle):
    """``struct FastM`` (FastConvolution.jl:11-27) with the apply on the GPU.

    GFFT is given exactly as the reference holds it: (ne, me) complex128, for
    Greengard_Vico in centred wave-number order (the fftshift/ifftshift of :94/:98 is folded
    into a one-time device permutation).

    ``embed=True`` (LS_FLAG_EMBED) serves any grid with n, m <= 4096 in both quadratures on the
    power-of-two kernels of n' = max(64, nextpow2(n)), the grid zero-embedded; ``info()`` tells
    which route a handle runs.
    """

    def __init__(self, GFFT, nu, ne, me, n, m, k, quadRule="trapezoidal", force_generic=False, pad4=False, L=None, Lp=None,
                 embed=False):
        super().__init__()
        self.ne, self.me, self.n, self.m = int(ne), int(me), int(n), int(m)
        self.omega = float(k)
        self.quadRule = quadRule
        if quadRule not in _lib.QUADRULES:
            raise ValueError("unknown quadRule %r" % (quadRule,))
        flags = ((_lib.FLAG_FORCE_GENERIC if force_generic else 0) | (_lib.FLAG_PAD4 if pad4 else 0)
                 | (_lib.FLAG_EMBED if embed else 0))
        if GFFT is None:
            # Greengard_Vico spectrum Gtruncated2D(L, k, S) evaluated on the device (FastConvolution.jl:185-231)
            if quadRule != "Greengard_Vico" or L is None or Lp is None:
                raise ValueError("GFFT=None needs quadRule='Greengard_Vico' and the truncation parameters L, Lp")
            if (self.ne, self.me) != (4 * self.n, 4 * self.m):
                raise ValueError("DimensionMismatch: Greengard_Vico pads to (4n, 4m)")
            nu = np.ascontiguousarray(np.asarray(nu, dtype=np.float64).reshape(-1))
            if nu.shape[0] != self.n * self.m:
                raise ValueError("DimensionMismatch: nu has %d entries, expected %d" % (nu.shape[0], self.n * self.m))
            self.N = self.n * self.m
            check(lib().ls_op2d_create_gv(C.byref(self._h), self.n, self.m, ptr(nu), self.omega, float(L), float(Lp), flags))
            return
        GFFT = np.asarray(GFFT)
        if GFFT.shape != (self.ne, self.me):
            raise ValueError("DimensionMismatch: GFFT is %s, expected (%d, %d)" % (GFFT.shape, self.ne, self.me))
        nu = np.ascontiguousarray(np.asarray(nu, dtype=np.float64).reshape(-1))
        if nu.shape[0] != self.n * self.m:
            raise ValueError("DimensionMismatch: nu has %d entries, expected %d" % (nu.shape[0], self.n * self.m))
        self.N = self.n * self.m
        g = np.asfortranarray(GFFT.astype(np.complex128, copy=False))   # column-major, as Julia stores it
        check(lib().ls_op2d_create(C.byref(self._h), self.n, self.m, self.ne, self.me, ptr(nu),
                                   C.c_void_p(g.ctypes.data), self.omega, _lib.QUADRULES[quadRule], flags))

    def info(self):
        """ls_op2d_info: route (_lib.ROUTE_POW2 / ROUTE_BLUESTEIN / ROUTE_EMBEDDED), the line lengths the kernels run
        and the padding factor of the spectrum the applies use."""
        route, pf = C.c_int(), C.c_int()
        nl, ml = C.c_int64(), C.c_int64()
        check(lib().ls_op2d_info(self.handle, C.byref(route), C.byref(nl), C.byref(ml), C.byref(pf)))
        return {"route": int(route.value), "n_line": int(nl.value), "m_line": int(ml.value), "padding_factor": int(pf.value)}

    # size / eltype, FastConvolution.jl:31-41 (Q1: size(M) is a tuple of tuples upstream)
    def size(self, dim=None):
        if dim is not None:
            return self.N
        return ((self.N,), (self.N,))

    def eltype(self):
        return np.dtype(np.complex128)

    def _apply(self, b, out, mode):
        if isinstance(b, DeviceBuffer) or isinstance(out, DeviceBuffer):
            if not (isinstance(b, DeviceBuffer) and isinstance(out, DeviceBuffer)):
                raise TypeError("b and out must both be DeviceBuffer or both numpy arrays")
            check(lib().ls_op2d_apply(self.handle, ptr(b), ptr(out), mode, _lib.MEM_DEVICE))
            return out
        if isinstance(b, np.ndarray) and b.ndim == 2:
            return _apply_cols(self, b, out, mode)
        b = _as_c128(b, self.N)
        if out is None:
            out = np.empty(self.N, dtype=np.complex128)
        check(lib().ls_op2d_apply(self.handle, ptr(b), ptr(out), mode, _lib.MEM_HOST))
        return out

    def __mul__(self, b):
        """``*(M::FastM, b)`` FastConvolution.jl:43-48."""
        return fastconvolution(self, b)

    __matmul__ = __mul__

    def mul_(self, Y, b):
        """``LinearAlgebra.mul!(Y, M, b)`` FastConvolution.jl:50-54 (Y[:] = M*b)."""
        if isinstance(Y, DeviceBuffer) or (isinstance(b, np.ndarray) and b.ndim == 2):
            return self._apply(b, Y, _lib.APPLY_FASTCONVOLUTION)
        if not (isinstance(Y, np.ndarray) and Y.dtype == np.complex128 and Y.shape == (self.N,)):
            raise ValueError("DimensionMismatch: Y must be a complex128 vector of length %d" % self.N)
        if Y.flags.c_contiguous:
            return self._apply(b, Y, _lib.APPLY_FASTCONVOLUTION)
        Y[:] = self._apply(b, None, _lib.APPLY_FASTCONVOLUTION)   # strided views of the Krylov basis
        return Y


class FastM3D(_Handle):
    """``struct FastM3D`` (FastConvolution3D.jl:7-26) with the apply on the GPU.

    ``GFFT`` is the (ne, me, le) centred spectrum as the reference holds it, or ``None`` together
    with the Greengard-Vico parameters ``L`` and ``Lp`` (FastConvolution3D.jl:72-73) to have
    Gtruncated3D evaluated on the device (the only practical way at 256^3 and above).
    The reference defines only ``*`` for this type (Q4); ``mul_``, ``size`` and ``eltype`` are
    added so that gmres! (which needs them) takes the operator.

    ``embed=True`` (LS_FLAG_EMBED) serves any n = m, l <= 512 on the power-of-two kernels of
    n' = max(64, nextpow2(n)) and l' likewise, the grid zero-embedded; ``lines()`` tells which
    route a handle runs.
    """

    def __init__(self, GFFT, nu, ne, me, le, n, m, l, k, quadRule="Greengard_Vico", L=None, Lp=None, pad4=False,
                 embed=False):
        super().__init__()
        self.ne, self.me, self.le, self.n, self.m, self.l = (int(v) for v in (ne, me, le, n, m, l))
        self.omega = float(k)
        self.quadRule = quadRule
        if quadRule != "Greengard_Vico":
            raise ValueError("FastM3D only knows quadRule='Greengard_Vico' (FastConvolution3D.jl:70)")
        nu = np.ascontiguousarray(np.asarray(nu, dtype=np.float64).reshape(-1))
        self.N = self.n * self.m * self.l
        if nu.shape[0] != self.N:
            raise ValueError("DimensionMismatch: nu has %d entries, expected %d" % (nu.shape[0], self.N))
        if GFFT is None:
            if L is None or Lp is None:
                raise ValueError("pass GFFT, or L and Lp to generate the Greengard-Vico spectrum on the device")
            gp = None
        else:
            GFFT = np.asarray(GFFT)
            if GFFT.shape != (self.ne, self.me, self.le):
                raise ValueError("DimensionMismatch: GFFT is %s, expected %s" % (GFFT.shape, (self.ne, self.me, self.le)))
            g = np.asfortranarray(GFFT.astype(np.complex128, copy=False))
            gp = C.c_void_p(g.ctypes.data)
        check(lib().ls_op3d_create(C.byref(self._h), self.n, self.m, self.l, self.ne, self.me, self.le, ptr(nu), gp,
                                   self.omega, float(L or 0.0), float(Lp or 0.0),
                                   (_lib.FLAG_PAD4 if pad4 else 0) | (_lib.FLAG_EMBED if embed else 0)))

    def lines(self):
        """ls_op3d_lines: route (_lib.ROUTE_POW2 / ROUTE_BLUESTEIN / ROUTE_EMBEDDED) and the line lengths the
        kernels run along x, y and z."""
        route = C.c_int()
        nl, ml, ll = C.c_int64(), C.c_int64(), C.c_int64()
        check(lib().ls_op3d_lines(self.handle, C.byref(route), C.byref(nl), C.byref(ml), C.byref(ll)))
        return {"route": int(route.value), "n_line": int(nl.value), "m_line": int(ml.value), "l_line": int(ll.value)}

    def size(self, dim=None):
        if dim is not None:
            return self.N
        return ((self.N,), (self.N,))

    def eltype(self):
        return np.dtype(np.complex128)

    def _apply(self, b, out, mode):
        if isinstance(b, DeviceBuffer) or isinstance(out, DeviceBuffer):
            if not (isinstance(b, DeviceBuffer) and isinstance(out, DeviceBuffer)):
                raise TypeError("b and out must both be DeviceBuffer or both numpy arrays")
            check(lib().ls_op3d_apply(self.handle, ptr(b), ptr(out), mode, _lib.MEM_DEVICE))
            return out
        if isinstance(b, np.ndarray) and b.ndim == 2:
            return _apply_cols(self, b, out, mode)
        b = _as_c128(b, self.N)
        if out is None:
            out = np.empty(self.N, dtype=np.complex128)
        check(lib().ls_op3d_apply(self.handle, ptr(b), ptr(out), mode, _lib.MEM_HOST))
        return out

    def __mul__(self, b):
        """``*(M::FastM3D, b)`` FastConvolution3D.jl:31-37."""
        return self._apply(b, None, _lib.APPLY_FASTCONVOLUTION)

    __matmul__ = __mul__

    def mul_(self, Y, b):
        if isinstance(b, np.ndarray) and b.ndim == 2:
            return self._apply(b, Y, _lib.APPLY_FASTCONVOLUTION)
        if isinstance(Y, DeviceBuffer) or (isinstance(Y, np.ndarray) and Y.flags.c_contiguous and Y.dtype == np.complex128
                                           and Y.shape == (self.N,)):
            return self._apply(b, Y, _lib.APPLY_FASTCONVOLUTION)
        Y[:] = self._apply(b, None, _lib.APPLY_FASTCONVOLUTION)
        return Y


def fastconvolution(M: FastM, b, out=None):
    """``fastconvolution(M, b)`` FastConvolution.jl:58-107:  b + omega^2 G (nu .* b)."""
    return M._apply(b, out, _lib.APPLY_FASTCONVOLUTION)


def FFTconvolution(M, b, out=None):
    """``FFTconvolution(M, b)`` FastConvolution.jl:110-154 / FastConvolution3D.jl:39-63.

    Reference semantics kept: no omega^2, no ``b +``; the Greengard_Vico branch does not
    apply nu (Q2) and pads/crops square (Q3).
    """
    return M._apply(b, out, _lib.APPLY_FFTCONVOLUTION)


def mul_(Y, M, b):
    """``mul!(Y, M, b)``."""
    return M.mul_(Y, b)
