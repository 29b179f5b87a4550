"""ctypes binding of libls_cuda.so (include/ls_cuda.h).

The product path has no CPU fallback: if the library is missing or a call fails, an
exception is raised.  Nothing here imports ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os
import re

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LS_CUDA_LIB") or os.path.join(HERE, "lib", "libls_cuda.so")     # LS_CUDA_LIB: another build of the same library
HEADER_PATH = os.path.join(os.path.dirname(HERE), "include", "ls_cuda.h")

LS_OK = 0
LS_ERR_INVALID, LS_ERR_UNSUPPORTED, LS_ERR_CUDA, LS_ERR_NOMEM, LS_ERR_NCCL, LS_ERR_CALLBACK = -1, -2, -3, -4, -5, -6
MEM_HOST, MEM_DEVICE = 0, 1
QUAD_TRAPEZOIDAL, QUAD_GREENGARD_VICO = 0, 1
APPLY_FASTCONVOLUTION, APPLY_FFTCONVOLUTION = 0, 1

QUADRULES = {"trapezoidal": QUAD_TRAPEZOIDAL, "Greengard_Vico": QUAD_GREENGARD_VICO}


class CDouble(C.Structure):
    _fields_ = [("re", C.c_double), ("im", C.c_double)]

    @classmethod
    def of(cls, z):
        z = complex(z)
        return cls(z.real, z.imag)


# typedef int (*ls_solve_cb)(void* user, ls_cdouble* v_inout, int64_t n)
SOLVE_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64)


class LSCudaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libls_cuda error %d: %s" % (code, msg))
        self.code = code


class LSUnsupported(LSCudaError):
    pass


_lib = None


def declared_symbols():
    """Every function name declared in include/ls_cuda.h."""
    with open(HEADER_PATH) as fh:
        text = fh.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ls_[a-z0-9_]+)\s*\(", text)))


def lib():
    """Loads libls_cuda.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LSCudaError(LS_ERR_INVALID,
                          "libls_cuda.so not built (run `python -m fast_solver_lippmann_schwinger_b200.build`); "
                          "there is no CPU fallback")
    L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    vp, i64, dbl, ci = C.c_void_p, C.c_int64, C.c_double, C.c_int
    sig = {
        "ls_version": (ci, []),
        "ls_last_error": (C.c_char_p, []),
        "ls_device_count": (ci, [C.POINTER(ci)]),
        "ls_set_device": (ci, [ci]),
        "ls_dev_alloc": (ci, [C.POINTER(vp), C.c_size_t]),
        "ls_dev_free": (ci, [vp]),
        "ls_memcpy_h2d": (ci, [vp, vp, C.c_size_t]),
        "ls_memcpy_d2h": (ci, [vp, vp, C.c_size_t]),
        "ls_host_alloc_pinned": (ci, [C.POINTER(vp), C.c_size_t]),
        "ls_host_free_pinned": (ci, [vp]),
        "ls_op2d_create": (ci, [C.POINTER(vp), i64, i64, i64, i64, vp, vp, dbl, ci, ci]),
        "ls_op2d_create_gv": (ci, [C.POINTER(vp), i64, i64, vp, dbl, dbl, dbl, ci]),
        "ls_op2d_apply": (ci, [vp, vp, vp, ci, ci]),
        "ls_op3d_create": (ci, [C.POINTER(vp), i64, i64, i64, i64, i64, i64, vp, vp, dbl, dbl, dbl, ci]),
        "ls_op3d_apply": (ci, [vp, vp, vp, ci, ci]),
        "ls_op3d_info": (ci, [vp, C.POINTER(ci), C.POINTER(ci), C.POINTER(ci)]),
        "ls_nccl_unique_id": (ci, [vp]),
        "ls_op3d_create_dist": (ci, [C.POINTER(vp), i64, i64, i64, vp, dbl, dbl, dbl, ci, ci, vp, ci]),
        "ls_op_size": (ci, [vp, C.POINTER(i64)]),
        "ls_spm_create": (ci, [C.POINTER(vp), i64, i64, vp, vp, vp]),
        "ls_spm_create_dist": (ci, [C.POINTER(vp), vp, i64, i64, vp, vp, vp]),
        "ls_spm_mv": (ci, [vp, CDouble, vp, CDouble, vp, ci]),
        "ls_spm_info": (ci, [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), C.POINTER(ci), C.POINTER(ci)]),
        "ls_krylov_create": (ci, [C.POINTER(vp), i64]),
        "ls_krylov_set_orth": (ci, [vp, ci]),
        "ls_zdotc": (ci, [vp, vp, vp, C.POINTER(CDouble)]),
        "ls_dznrm2": (ci, [vp, vp, C.POINTER(dbl)]),
        "ls_zaxpy": (ci, [vp, CDouble, vp, vp]),
        "ls_zscal": (ci, [vp, CDouble, vp]),
        "ls_mgs_step": (ci, [vp, vp, i64, ci, vp, vp]),
        "ls_gmres": (ci, [vp, vp, vp, SOLVE_CB, vp, vp, vp, ci, i64, dbl, dbl, ci, vp, i64,
                          C.POINTER(i64), C.POINTER(ci), C.POINTER(i64), ci]),
        "ls_msp_factor": (ci, [C.POINTER(vp), i64, i64, vp, vp, vp]),
        "ls_msp_factor3d": (ci, [C.POINTER(vp), i64, i64, i64, vp, vp, vp]),
        "ls_msp_solve": (ci, [vp, vp, vp, ci]),
        "ls_msp_info": (ci, [vp, C.POINTER(i64), C.POINTER(ci), C.POINTER(dbl)]),
        "ls_msp_plan": (ci, [vp, C.c_char_p, i64]),
        "ls_gmres_msp": (ci, [vp, vp, vp, vp, vp, vp, ci, i64, dbl, dbl, ci, vp, i64,
                              C.POINTER(i64), C.POINTER(ci), C.POINTER(i64), ci]),
        "ls_krylov_last_precond_host_seconds": (ci, [vp, C.POINTER(dbl)]),
        "ls_sample_rows": (ci, [vp, vp, vp, ci, vp, i64]),
        "ls_gram": (ci, [vp, vp, i64, ci, vp]),
        "ls_gather_rows": (ci, [vp, vp, i64, ci, vp, ci, vp]),
        "ls_destroy": (ci, [vp]),
        "ls_sync": (ci, [vp]),
        "ls_timer_start": (ci, [vp]),
        "ls_timer_stop": (ci, [vp, C.POINTER(C.c_float)]),
        "ls_launch_count": (ci, [vp, C.POINTER(i64)]),
        "ls_profile_enable": (ci, [vp, ci]),
        "ls_profile_read": (ci, [vp, C.POINTER(dbl), C.POINTER(i64), ci]),
        "ls_test_fft_lines": (ci, [i64, i64, vp, vp, ci]),
        "ls_test_device_peaks": (ci, [C.POINTER(dbl), C.POINTER(dbl), C.POINTER(dbl)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    L._signatures = sig
    _lib = L
    return L


def check(rc):
    if rc == LS_OK:
        return
    msg = lib().ls_last_error().decode("utf-8", "replace")
    if rc == LS_ERR_UNSUPPORTED:
        raise LSUnsupported(rc, msg)
    raise LSCudaError(rc, msg)


def ptr(a):
    """Raw pointer of a numpy array, a DeviceBuffer, an int address, or None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    if isinstance(a, DeviceBuffer):
        return C.c_void_p(a.ptr)
    return C.c_void_p(int(a))


class DeviceBuffer:
    """A raw device allocation owned by Python (Krylov vectors, bench inputs)."""

    def __init__(self, nbytes):
        p = C.c_void_p()
        check(lib().ls_dev_alloc(C.byref(p), nbytes))
        self.ptr = p.value
        self.nbytes = nbytes

    @classmethod
    def from_host(cls, arr):
        arr = np.ascontiguousarray(arr)
        buf = cls(arr.nbytes)
        check(lib().ls_memcpy_h2d(C.c_void_p(buf.ptr), ptr(arr), arr.nbytes))
        return buf

    def to_host(self, dtype=np.complex128, count=None):
        dtype = np.dtype(dtype)
        count = self.nbytes // dtype.itemsize if count is None else count
        out = np.empty(count, dtype=dtype)
        check(lib().ls_memcpy_d2h(ptr(out), C.c_void_p(self.ptr), count * dtype.itemsize))
        return out

    def offset(self, nbytes):
        return self.ptr + nbytes

    def free(self):
        if self.ptr:
            lib().ls_dev_free(C.c_void_p(self.ptr))
            self.ptr = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PinnedArray:
    """numpy view over cudaMallocHost memory (for the end-to-end timed path)."""

    def __init__(self, shape, dtype=np.complex128):
        dtype = np.dtype(dtype)
        n = int(np.prod(shape))
        p = C.c_void_p()
        check(lib().ls_host_alloc_pinned(C.byref(p), n * dtype.itemsize))
        self._ptr = p.value
        buf = (C.c_char * (n * dtype.itemsize)).from_address(self._ptr)
        self.array = np.frombuffer(buf, dtype=dtype).reshape(shape)

    def free(self):
        if self._ptr:
            self.array = None
            lib().ls_host_free_pinned(C.c_void_p(self._ptr))
            self._ptr = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
