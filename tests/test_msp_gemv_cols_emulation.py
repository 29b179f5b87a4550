"""CPU check of the index logic of the multi-column Msp sweep (k_msp_gemv2_cols, csrc/msp_gemv.cuh) that serves
ls_msp_solve_batch.

tests/msp_gemv_cols_emu.cu runs the kernel's __host__ __device__ phase functions CTA by CTA on the CPU, next to the
single-vector kernel's.  For every addressing mode of the solve, ragged node sizes and both CTA geometries (several nodes
per CTA, several CTAs per node), each column of the NRHS-column result must carry exactly the bits of the single-vector
kernel run on that column with the same LANES, whatever UNR and XS are."""
import ctypes as C
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from test_msp_gemv_emulation import MODES, SHAPES, Gemv2, Problem, crandn  # noqa: E402

SRC = os.path.join(HERE, "msp_gemv_cols_emu.cu")
DEPS = [SRC, os.path.join(HERE, "msp_gemv_emu.cu"),
        os.path.join(os.path.dirname(HERE), "fast_solver_lippmann_schwinger_b200", "csrc", "msp_gemv.cuh")]
OUT = os.path.join(HERE, "_build", "libmsp_gemv_cols_emu.so")


class Cols(C.Structure):
    _fields_ = [("f", C.c_long), ("x", C.c_long), ("xg", C.c_long), ("tchild", C.c_long), ("y0", C.c_long), ("out", C.c_long)]


@pytest.fixture(scope="module")
def emu():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available: the emulation library cannot be built")
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    if not os.path.exists(OUT) or os.path.getmtime(OUT) < max(os.path.getmtime(p) for p in DEPS):
        subprocess.run([nvcc, "-O1", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
                        "-o", OUT, SRC], check=True, capture_output=True)
    L = C.CDLL(OUT)
    L.emu_msp_gemv2.restype = C.c_int
    L.emu_msp_gemv2.argtypes = [C.POINTER(Gemv2), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint), C.POINTER(C.c_long)]
    L.emu_msp_gemv2_cols.restype = C.c_int
    L.emu_msp_gemv2_cols.argtypes = [C.POINTER(Gemv2), C.POINTER(Cols), C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_long)]
    L.emu_cols_choice.restype = None
    L.emu_cols_choice.argtypes = [C.c_int] * 8 + [C.c_long, C.POINTER(C.c_int)]
    assert L.emu_sizeof_gemv2() == C.sizeof(Gemv2) and L.emu_sizeof_cols() == C.sizeof(Cols)
    return L


class Batch:
    """Problem P widened to nrhs columns: every vector the sweep reads or writes gets nrhs columns at a stride a few
    elements longer than the vector (column 0 is P's own data); index arrays and the matrix are shared."""

    def __init__(self, P, nrhs, rng):
        self.P, self.nrhs = P, nrhs
        self.a = Gemv2()
        C.memmove(C.byref(self.a), C.byref(P.a), C.sizeof(Gemv2))
        self.cs = Cols()
        self.cols = {}                      # field -> (array, stride, length)
        for field in ("f", "x", "xg", "tchild", "y0"):
            base = getattr(P, field, None)
            if base is None or getattr(P.a, field) is None:
                continue
            n = len(base)
            stride = n + 3
            arr = crandn(rng, nrhs * stride)
            arr[:n] = base
            self.cols[field] = (arr, stride, n)
            setattr(self.a, field, arr.ctypes.data)
            setattr(self.cs, field, stride)
        self.ofield = "og" if P.scatter else "out"
        n = len(P.result())
        self.ostride = n + 5
        self.out = np.full(nrhs * self.ostride, 7.0 + 0j)
        setattr(self.a, self.ofield, self.out.ctypes.data)
        self.cs.out = self.ostride
        self.on = n

    def column(self, j):
        return self.out[j * self.ostride:j * self.ostride + self.on]

    def single(self, emu, j, ll):
        """the single-vector kernel on column j (UNR 4, no staging: its bits depend on LANES only)"""
        a = Gemv2()
        C.memmove(C.byref(a), C.byref(self.P.a), C.sizeof(Gemv2))
        for field, (arr, stride, _) in self.cols.items():
            setattr(a, field, arr.ctypes.data + 16 * j * stride)
        ref = np.full(self.on, 7.0 + 0j)
        setattr(a, self.ofield, ref.ctypes.data)
        assert emu.emu_msp_gemv2(C.byref(a), ll, 2, 0, None, None) > 0
        return ref


@pytest.mark.parametrize("nrhs", [1, 2, 4, 8])
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("mode", MODES)
def test_every_column_has_the_single_vector_bits(emu, nrhs, shape, mode):
    nodes, rows_p, cols_p = shape
    xmode, ymode, scatter, sign = mode
    rng = np.random.default_rng(1000 * nodes + 10 * rows_p + cols_p + xmode + 7 * nrhs)
    P = Problem(rng, nodes, rows_p, cols_p, xmode, ymode, scatter, sign)
    B = Batch(P, nrhs, rng)
    smem = C.c_long()
    for ll in range(6):
        refs = [B.single(emu, j, ll) for j in range(nrhs)]
        for ul in range(4):
            for xs in (0, 1):
                B.out[:] = 7.0 + 0j
                assert emu.emu_msp_gemv2_cols(C.byref(B.a), C.byref(B.cs), nrhs, ll, ul, xs, C.byref(smem)) > 0
                if xs:
                    assert smem.value % (16 * nrhs) == 0 and smem.value >= nrhs * cols_p * 16
                for j in range(nrhs):
                    assert np.array_equal(B.column(j), refs[j]), (ll, ul, xs, j)
                # nothing is written between the columns
                for j in range(nrhs):
                    gap = B.out[j * B.ostride + B.on:(j + 1) * B.ostride]
                    assert np.all(gap == 7.0 + 0j)


def test_columns_are_independent(emu):
    """A column full of NaN changes no bit of the others (the downward sweep, staged and not)."""
    rng = np.random.default_rng(9)
    P = Problem(rng, 9, 12, 20, 1, 1, True, -1.0)
    B = Batch(P, 4, rng)
    arr, stride, n = B.cols["xg"]
    for xs in (0, 1):
        B.out[:] = 7.0 + 0j
        emu.emu_msp_gemv2_cols(C.byref(B.a), C.byref(B.cs), 4, 3, 1, xs, None)
        clean = B.out.copy()
        keep = arr[2 * stride:3 * stride].copy()
        arr[2 * stride:2 * stride + n] = np.nan
        B.out[:] = 7.0 + 0j
        emu.emu_msp_gemv2_cols(C.byref(B.a), C.byref(B.cs), 4, 3, 1, xs, None)
        for j in (0, 1, 3):
            assert np.array_equal(B.column(j), clean[j * B.ostride:j * B.ostride + B.on])
        assert np.isnan(B.column(2)).any()
        arr[2 * stride:3 * stride] = keep


def test_cols_choice_rule(emu):
    """UNR * NRHS <= 8 (register budget of __launch_bounds__(256, 2)), LANES kept, X staged when the single plan stages it
    or X is index-chased, and only when NRHS columns of it fit the limit."""
    out = (C.c_int * 3)()
    for nrhs, unr_cap in ((1, 3), (2, 2), (4, 1), (8, 0)):
        emu.emu_cols_choice(3, 3, 0, nrhs, 40, 64, 100, 0, 48 * 1024, out)
        assert tuple(out) == (3, unr_cap, 0)
    emu.emu_cols_choice(4, 2, 0, 4, 40, 64, 100, 1, 48 * 1024, out)        # index-chased X: staged
    assert tuple(out) == (4, 1, 1)
    emu.emu_cols_choice(4, 2, 1, 8, 40, 2048, 100, 1, 113 * 1024, out)     # 8 x 2048 x 16 B > 113 KB: not staged
    assert tuple(out) == (4, 0, 0)
    emu.emu_cols_choice(4, 2, 1, 2, 40, 2048, 100, 0, 113 * 1024, out)     # 2 x 2048 x 16 B fits
    assert tuple(out) == (4, 2, 1)
