"""CPU checks of the symbolic analysis behind the device Msp factorisation (csrc/msp_symbolic.h, 2-D and 3-D grids).

tests/msp_symbolic_emu.cpp exposes the header's code as a host library: the dissection, own and ring lists, entry
routing, child / parent maps and the byte count of the memory check.  Here they are checked against independent
Python counts, and a dense multifrontal elimination that uses nothing but those lists and maps is compared with
scipy's sparse solve.  The device parity of the whole factorisation is tests/test_gpu_msp3d.py."""
import ctypes as C
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from util_sparse import stencil27  # noqa: E402

SRC = os.path.join(HERE, "msp_symbolic_emu.cpp")
HDR = os.path.join(os.path.dirname(HERE), "fast_solver_lippmann_schwinger_b200", "csrc", "msp_symbolic.h")
OUT = os.path.join(HERE, "_build", "libmsp_symbolic_emu.so")

GRIDS = [(1, 1, 1), (2, 3, 1), (3, 3, 3), (5, 6, 7), (9, 4, 3), (4, 4, 17), (12, 12, 12), (20, 20, 36)]
LEAVES = [3, 4, 8]
LS_ERR_INVALID, LS_ERR_UNSUPPORTED = -1, -2


@pytest.fixture(scope="module")
def emu():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available: the emulation library cannot be built")
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    if not os.path.exists(OUT) or os.path.getmtime(OUT) < max(os.path.getmtime(SRC), os.path.getmtime(HDR)):
        subprocess.run([nvcc, "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-o", OUT, SRC],
                       check=True, capture_output=True)
    L = C.CDLL(OUT)
    L.sym_create.restype = C.c_void_p
    L.sym_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_int]
    L.sym_destroy.argtypes = [C.c_void_p]
    L.sym_depth.argtypes = [C.c_void_p]
    L.sym_level.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.sym_box.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.sym_ints.restype = C.c_long
    L.sym_ints.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_long]
    L.sym_own_depth.argtypes = [C.c_void_p, C.c_void_p]
    L.sym_ring_index.argtypes = [C.c_void_p] + [C.c_int] * 5
    L.sym_route.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.c_int]
    L.sym_entries.restype = C.c_long
    L.sym_entries.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_long]
    L.sym_need_bytes.restype = C.c_ulonglong
    L.sym_need_bytes.argtypes = [C.c_void_p, C.c_longlong, C.c_int]
    return L


class Sym:
    """The header's analysis of one grid, read back into numpy arrays."""

    def __init__(self, L, n, m, l, leaf, lists=True):
        self.L, self.n, self.m, self.l = L, n, m, l
        err = C.create_string_buffer(512)
        self.h = L.sym_create(n, m, l, leaf, int(lists), err, len(err))
        assert self.h, err.value
        self.D = L.sym_depth(self.h)
        self.lev = []
        for d in range(self.D + 1):
            o = (C.c_int * 5)()
            L.sym_level(self.h, d, o)
            self.lev.append(dict(count=o[0], Sp=o[1], Bp=o[2], leaf=bool(o[3]), axis=o[4]))
        if lists:
            N = n * m * l
            self.own_depth = np.zeros(N, np.uint8)
            L.sym_own_depth(self.h, self.own_depth.ctypes.data_as(C.c_void_p))

    def ints(self, which, d=0):
        ln = self.L.sym_ints(self.h, which, d, None, 0)
        a = np.zeros(max(ln, 1), np.int32)
        self.L.sym_ints(self.h, which, d, a.ctypes.data_as(C.c_void_p), ln)
        return a[:ln]

    def box(self, d, t):
        o = (C.c_int * 6)()
        self.L.sym_box(self.h, d, t, o)
        return tuple(o)

    def route(self, A):
        """A: scipy CSC (0-based) -> status, message"""
        colptr = A.indptr.astype(np.int64) + 1
        rowval = A.indices.astype(np.int64) + 1
        err = C.create_string_buffer(512)
        rc = self.L.sym_route(self.h, colptr.ctypes.data_as(C.c_void_p), rowval.ctypes.data_as(C.c_void_p), err, len(err))
        return rc, err.value.decode()

    def entries(self, d):
        ln = self.L.sym_entries(self.h, d, None, None, 0)
        dest, src = np.zeros(max(ln, 1), np.int64), np.zeros(max(ln, 1), np.int32)
        self.L.sym_entries(self.h, d, dest.ctypes.data_as(C.c_void_p), src.ctypes.data_as(C.c_void_p), ln)
        return dest[:ln], src[:ln]

    def close(self):
        self.L.sym_destroy(self.h)


# ---- an independent Python statement of the dissection rule --------------------------------------------------------
def py_dissection(n, m, l, leaf):
    """per depth: (boxes, axis) with the rule of the header: split every box of a depth at its midpoint, perpendicular
    to the axis with the largest extent over the depth (ties x, y, z), until no box is wider than `leaf`."""
    levels = []
    boxes = [((0, n), (0, m), (0, l))]
    while True:
        ext = [max(b[a][1] - b[a][0] for b in boxes) for a in range(3)]
        if max(ext) <= leaf:
            levels.append((boxes, None))
            return levels
        ax = int(np.argmax(ext))                 # first maximum: ties go x, then y, then z
        levels.append((boxes, ax))
        nxt = []
        for b in boxes:
            lo, hi = b[ax]
            mid = lo + (hi - lo) // 2
            for part in ((lo, mid), (mid + 1, hi)):
                c = list(b)
                c[ax] = part
                nxt.append(tuple(c))
        boxes = nxt


def py_sizes(n, m, l, box, axis):
    ext = [box[a][1] - box[a][0] for a in range(3)]
    own = int(np.prod(ext)) if axis is None else int(np.prod([e for a, e in enumerate(ext) if a != axis]))
    dims = (n, m, l)
    shell = np.prod([min(box[a][1], dims[a] - 1) - max(box[a][0] - 1, 0) + 1 for a in range(3)])
    return own, int(shell - np.prod(ext))


def py_need_bytes(n, m, l, leaf, nnz, tight):
    """The memory check's count, restated: kept index maps + factor blocks + solve vectors of every depth, plus the
    largest per-depth transient (dense fronts of the depth and of its children, inverse, Y, pivots, child map), plus the
    matrix values and the routing of the entries, plus four N-vectors."""
    levels = py_dissection(n, m, l, leaf)
    D = len(levels) - 1
    shapes = []
    for boxes, ax in levels:
        sz = [py_sizes(n, m, l, b, ax) for b in boxes]
        shapes.append((len(boxes), max(s for s, _ in sz), max(b for _, b in sz), sz))
    keep, peak = 0, 0
    for d, (cnt, Sp, Bp, sz) in enumerate(shapes):
        Fp = Sp + Bp
        keep += 4 * cnt * Sp + 4 * cnt * max(Bp, 1) + (8 * cnt * Fp if d < D else 0)
        if tight:
            totS, totB = sum(s * s for s, _ in sz), sum(s * b for s, b in sz)
            keep += 24 * cnt
        else:
            totS, totB = cnt * Sp * Sp, cnt * Sp * Bp
        keep += 16 * (max(totS, 1) + 2 * max(totB, 1)) + 16 * (cnt * Fp + cnt * Sp + max(cnt * Bp, 1))
        tr = 16 * cnt * Fp * Fp + 16 * cnt * Sp * Sp + 16 * max(cnt * Sp * Bp, 1) + 16 * cnt + 4 * cnt * Sp + 8 * cnt
        if d < D:
            c_cnt, c_Sp, c_Bp, _ = shapes[d + 1]
            tr += 16 * c_cnt * (c_Sp + c_Bp) ** 2 + 4 * c_cnt * max(c_Bp, 1)
        peak = max(peak, tr)
    return keep + peak + 16 * max(nnz, 1) + 12 * nnz + 64 * n * m * l


def _coords(g, n, m):
    return g % n, (g // n) % m, g // (n * m)


# ---- tests ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("leaf", LEAVES)
@pytest.mark.parametrize("grid", GRIDS)
def test_owners_rings_and_routing(emu, grid, leaf):
    """Every unknown has exactly one owner; every ring lies on the box's shell in lexicographic order and ring_index
    inverts it; every entry of a full 27-point pattern routes to exactly one front position, which decodes back to
    its (row, col); the dissection follows the stated rule."""
    n, m, l = grid
    N = n * m * l
    S = Sym(emu, n, m, l, leaf)
    levels = py_dissection(n, m, l, leaf)
    assert S.D == len(levels) - 1
    owners = np.zeros(N, int)
    for d, (boxes, ax) in enumerate(levels):
        Lv = S.lev[d]
        assert Lv["count"] == len(boxes) and Lv["leaf"] == (ax is None)
        if ax is not None:
            assert Lv["axis"] == ax
        Sidx = S.ints(0, d).reshape(Lv["count"], Lv["Sp"])
        Bidx = S.ints(1, d).reshape(Lv["count"], max(Lv["Bp"], 1))
        ns, nb = S.ints(4, d), S.ints(5, d)
        for t, b in enumerate(boxes):
            assert S.box(d, t) == (b[0][0], b[0][1], b[1][0], b[1][1], b[2][0], b[2][1])
            own, ring = py_sizes(n, m, l, b, ax)
            assert (ns[t], nb[t]) == (own, ring)
            s_list = Sidx[t][Sidx[t] >= 0]
            b_list = Bidx[t][Bidx[t] >= 0]
            assert len(s_list) == own and np.all(Sidx[t][:own] >= 0) and len(b_list) == ring
            assert np.all(np.diff(s_list) > 0) and np.all(np.diff(b_list) > 0)      # lexicographic: x fastest
            owners[s_list] += 1
            for k, g in enumerate(b_list):
                i, j, p = _coords(g, n, m)
                assert max(b[0][0] - i, i - b[0][1] + 1, b[1][0] - j, j - b[1][1] + 1, b[2][0] - p, p - b[2][1] + 1) == 1
                assert emu.sym_ring_index(S.h, d, t, i, j, p) == k
    assert np.all(owners == 1)

    A = stencil27(n, m, l, seed=1, classes=False)
    rc, msg = S.route(A)
    assert rc == 0, msg
    seen = set()
    total = 0
    for d in range(S.D + 1):
        Lv = S.lev[d]
        Fp = Lv["Sp"] + Lv["Bp"]
        Sidx = S.ints(0, d).reshape(Lv["count"], Lv["Sp"])
        Bidx = S.ints(1, d).reshape(Lv["count"], max(Lv["Bp"], 1))
        dest, src = S.entries(d)
        total += len(dest)
        t, rem = dest // (Fp * Fp), dest % (Fp * Fp)
        lr, lc = rem % Fp, rem // Fp

        def unknown(t, q):
            return np.where(q < Lv["Sp"], Sidx[t, np.minimum(q, Lv["Sp"] - 1)], Bidx[t, np.maximum(q - Lv["Sp"], 0)])
        rows, cols = unknown(t, lr), unknown(t, lc)
        col_of = np.repeat(np.arange(N), np.diff(A.indptr))
        assert np.array_equal(rows, A.indices[src]) and np.array_equal(cols, col_of[src])
        assert np.all((lr < Lv["Sp"]) | (lc < Lv["Sp"]))            # never a ring-ring entry
        seen.update((d, x) for x in dest.tolist())
    assert total == A.nnz and len(seen) == A.nnz
    S.close()


def _py_ring_2d(n, m, b):
    """the 2-D ring order of the first version: row j0-1, the side columns of rows j0..j1-1, row j1 (clipped)"""
    (i0, i1), (j0, j1) = b[0], b[1]
    ia, ib = max(i0 - 1, 0), min(i1, n - 1)
    out = []
    if j0 - 1 >= 0:
        out += [i + n * (j0 - 1) for i in range(ia, ib + 1)]
    for j in range(j0, j1):
        if i0 - 1 >= 0:
            out.append(i0 - 1 + n * j)
        if i1 < n:
            out.append(i1 + n * j)
    if j1 < m:
        out += [i + n * j1 for i in range(ia, ib + 1)]
    return out


@pytest.mark.parametrize("n,m", [(1, 1), (3, 2), (9, 4), (17, 33), (40, 25), (130, 257)])
def test_planar_grids_keep_the_2d_lists(emu, n, m):
    """l = 1 gives the boxes, own lists and ring order of the 2-D analysis: the factorisation of a 2-D matrix is
    unchanged."""
    S = Sym(emu, n, m, 1, 4)
    for d, (boxes, ax) in enumerate(py_dissection(n, m, 1, 4)):
        assert ax != 2
        Lv = S.lev[d]
        Bidx = S.ints(1, d).reshape(Lv["count"], max(Lv["Bp"], 1))
        Sidx = S.ints(0, d).reshape(Lv["count"], Lv["Sp"])
        for t, b in enumerate(boxes):
            ring = _py_ring_2d(n, m, b)
            assert list(Bidx[t][:len(ring)]) == ring and np.all(Bidx[t][len(ring):] < 0)
            (i0, i1), (j0, j1) = b[0], b[1]
            if ax is None:
                own = [i + n * j for j in range(j0, j1) for i in range(i0, i1)]
            elif ax == 0:
                own = [i0 + (i1 - i0) // 2 + n * j for j in range(j0, j1)]
            else:
                own = [i + n * (j0 + (j1 - j0) // 2) for i in range(i0, i1)]
            assert list(Sidx[t][:len(own)]) == own
    S.close()


def multifrontal_solve(S, A, b):
    """Dense multifrontal elimination driven only by the shim's lists and maps: scatter the routed entries, extend-add
    the children's updates through cmap, Sinv = F_SS^-1, Y = Sinv F_SB, U = F_BB - F_BS Y; then the upward sweep
    (g = [f_S; 0] + children's t through pmap, z = Sinv g_S, t = g_B - F_BS z) and the downward one (u_S = z - Y u_B)."""
    D = S.D
    nz = A.data
    fac = [None] * (D + 1)
    U_child = None
    for d in range(D, -1, -1):
        Lv = S.lev[d]
        cnt, Sp, Bp = Lv["count"], Lv["Sp"], Lv["Bp"]
        Fp = Sp + Bp
        Sidx = S.ints(0, d).reshape(cnt, Sp)
        Fflat = np.zeros(cnt * Fp * Fp, complex)
        dest, src = S.entries(d)
        np.add.at(Fflat, dest, nz[src])
        F = Fflat.reshape(cnt, Fp, Fp).transpose(0, 2, 1).copy()         # column-major fronts
        for t in range(cnt):
            pad = np.nonzero(Sidx[t] < 0)[0]
            F[t, pad, pad] = 1.0
        if d < D:
            Lc = S.lev[d + 1]
            cmap = S.ints(3, d + 1).reshape(Lc["count"], max(Lc["Bp"], 1))
            for c in range(Lc["count"]):
                k = np.nonzero(cmap[c, :Lc["Bp"]] >= 0)[0]
                pos = cmap[c, k]
                F[c // 2][np.ix_(pos, pos)] += U_child[c][np.ix_(k, k)]
        Sinv = np.linalg.inv(F[:, :Sp, :Sp])
        Y = Sinv @ F[:, :Sp, Sp:]
        U_child = F[:, Sp:, Sp:] - F[:, Sp:, :Sp] @ Y
        fac[d] = (Sinv, F[:, Sp:, :Sp].copy(), Y)
    u = np.zeros(A.shape[0], complex)
    tvec = [None] * (D + 1)
    zvec = [None] * (D + 1)
    for d in range(D, -1, -1):
        Lv = S.lev[d]
        cnt, Sp, Bp = Lv["count"], Lv["Sp"], Lv["Bp"]
        Fp = Sp + Bp
        Sidx = S.ints(0, d).reshape(cnt, Sp)
        g = np.zeros((cnt, Fp), complex)
        g[:, :Sp] = np.where(Sidx >= 0, b[np.maximum(Sidx, 0)], 0.0)
        if d < D:
            pmap = S.ints(2, d).reshape(cnt, 2, Fp)
            for t in range(cnt):
                for side in (0, 1):
                    k = pmap[t, side]
                    ok = k >= 0
                    g[t, ok] += tvec[d + 1][2 * t + side][k[ok]]
        Sinv, FBS, _ = fac[d]
        zvec[d] = np.einsum("tij,tj->ti", Sinv, g[:, :Sp])
        tvec[d] = g[:, Sp:] - np.einsum("tij,tj->ti", FBS, zvec[d])
    for d in range(D + 1):
        Lv = S.lev[d]
        cnt, Sp, Bp = Lv["count"], Lv["Sp"], Lv["Bp"]
        Sidx = S.ints(0, d).reshape(cnt, Sp)
        Bidx = S.ints(1, d).reshape(cnt, max(Bp, 1))[:, :Bp]
        uB = np.where(Bidx >= 0, u[np.maximum(Bidx, 0)], 0.0)
        uS = zvec[d] - np.einsum("tij,tj->ti", fac[d][2], uB)
        ok = Sidx >= 0
        u[Sidx[ok]] = uS[ok]
    return u


@pytest.mark.parametrize("leaf", LEAVES)
@pytest.mark.parametrize("grid", GRIDS)
def test_multifrontal_elimination_matches_spsolve(emu, grid, leaf):
    n, m, l = grid
    N = n * m * l
    A = stencil27(n, m, l, seed=n + 10 * m + 100 * l, classes=False)
    A = (A + 8.0 * sp.identity(N, format="csc")).tocsc()
    A.sort_indices()
    S = Sym(emu, n, m, l, leaf)
    assert S.route(A)[0] == 0
    rng = np.random.default_rng(leaf)
    b = rng.standard_normal(N) + 1j * rng.standard_normal(N)
    u = multifrontal_solve(S, A, b)
    ref = spla.spsolve(A, b)
    assert np.linalg.norm(u - ref) / np.linalg.norm(ref) < 1e-12
    S.close()


@pytest.mark.parametrize("grid,leaf", [(g, lf) for g in GRIDS for lf in LEAVES]
                         + [((48, 48, 48), 4), ((64, 64, 64), 4), ((96, 96, 96), 4), ((201, 201, 1), 4), ((512, 300, 1), 4)])
def test_memory_check_counts_what_the_factorisation_allocates(emu, grid, leaf):
    n, m, l = grid
    S = Sym(emu, n, m, l, leaf, lists=False)
    nnz = 27 * n * m * l
    for tight in (0, 1):
        assert emu.sym_need_bytes(S.h, nnz, tight) == py_need_bytes(n, m, l, leaf, nnz, tight)
    assert emu.sym_need_bytes(S.h, 0, 1) == py_need_bytes(n, m, l, leaf, 0, 1)
    S.close()


def test_160_cubed_needs_more_than_one_b200(emu):
    S = Sym(emu, 160, 160, 160, 4, lists=False)
    assert emu.sym_need_bytes(S.h, 0, 1) > 180e9
    S.close()


def test_routing_refuses_duplicates_and_entries_outside_the_pattern(emu):
    n, m, l = 5, 6, 7
    N = n * m * l
    S = Sym(emu, n, m, l, 4)
    A = stencil27(n, m, l, seed=3, classes=False)
    # a duplicate (row, col): the same row twice in one column
    c = 40
    rows = A.indices[A.indptr[c]:A.indptr[c + 1]]
    indices = np.insert(A.indices, A.indptr[c] + 1, rows[0])
    indptr = A.indptr.copy()
    indptr[c + 1:] += 1
    dup = sp.csc_matrix((np.ones(len(indices), complex), indices, indptr), shape=(N, N))
    rc, msg = S.route(dup)
    assert rc == LS_ERR_INVALID and "duplicate" in msg, msg
    # two cells apart in x (inside one leaf box as well as across boxes)
    for r, col in ((0, 2), (7 + n * 2, 7 + n * 2 + 2 * n * m), (0, 4 + n * 5 + n * m * 6)):
        B = A.tolil()
        B[r, col] = 1.0
        rc, msg = S.route(B.tocsc())
        assert rc == LS_ERR_UNSUPPORTED and "27-point" in msg, msg
    # 2-D: the 9-point pattern
    S2 = Sym(emu, 8, 8, 1, 4)
    B = stencil27(8, 8, 1, seed=1).tolil()
    B[0, 2] = 1.0
    rc, msg = S2.route(B.tocsc())
    assert rc == LS_ERR_UNSUPPORTED and "9-point" in msg, msg
    S.close()
    S2.close()


def test_factor3d_argument_errors_without_gpu(built_lib):
    """ls_msp_factor3d validates its arguments before any CUDA call."""
    from fast_solver_lippmann_schwinger_b200._lib import lib
    L = lib()
    h = C.c_void_p()

    def call(n, m, l, colptr, rowval=np.ones(1, np.int64), nz=np.ones(1, complex)):
        p = (lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None)
        return L.ls_msp_factor3d(C.byref(h), n, m, l, p(colptr), p(rowval), p(nz)), L.ls_last_error()

    ok = np.ones(2 * 2 * 2 + 1, np.int64)
    rc, msg = call(2, 2, 2, None)
    assert rc == LS_ERR_INVALID and b"null pointer" in msg
    rc, msg = call(2, 2, 2, ok, None)
    assert rc == LS_ERR_INVALID and b"null pointer" in msg
    rc, msg = call(2, 2, 2, np.zeros(9, np.int64))
    assert rc == LS_ERR_INVALID and b"1-based" in msg
    for grid in ((0, 2, 2), (2, -1, 2), (2, 2, 0), (2 ** 11, 2 ** 10, 2 ** 10), (2 ** 31, 1, 1)):
        rc, msg = call(*grid, ok)
        assert rc == LS_ERR_INVALID and b"bad grid" in msg, grid
    big = np.ones(9, np.int64)
    big[-1] = 2 ** 31 + 1
    rc, msg = call(2, 2, 2, big)
    assert rc == LS_ERR_UNSUPPORTED and b"32-bit" in msg
    assert L.ls_msp_factor3d(None, 2, 2, 2, None, None, None) == LS_ERR_INVALID
