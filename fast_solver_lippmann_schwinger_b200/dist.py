"""One-process-per-GPU plumbing for the slab-decomposed 3-D operator.

torch.distributed is used only as the rendezvous (rank / world size, broadcasting the 128-byte
NCCL id, barriers, max-over-ranks of timings); the data path - both FFT transposes and the scalar
all-reduces of the Krylov dots - runs inside libls_cuda.so on its own NCCL communicator.

Sharding (SURVEY.md section 8(e)): rank r of P owns the z planes [r*l/P, (r+1)*l/P) of the
n x m x l grid, i.e. the contiguous range [r*N/P, (r+1)*N/P) of every grid vector.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _lib
from ._lib import DeviceBuffer, check, lib, ptr
from .operators import FastM3D, _Handle, _as_c128


def env_rank():
    """(rank, world_size, local_rank) from the torchrun environment."""
    return (int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")),
            int(os.environ.get("LOCAL_RANK", "0")))


def slab_range(l, rank, nranks):
    """z planes owned by `rank` (equal slabs; l must be divisible by nranks)."""
    if l % nranks:
        raise ValueError("l=%d is not divisible by the number of ranks %d" % (l, nranks))
    lloc = l // nranks
    return rank * lloc, (rank + 1) * lloc


def vector_range(n, m, l, rank, nranks):
    """[start, stop) of this rank's part of a grid vector (x fastest, z slowest)."""
    p0, p1 = slab_range(l, rank, nranks)
    return n * m * p0, n * m * p1


def scatter_vector(v, n, m, l, rank, nranks):
    a, b = vector_range(n, m, l, rank, nranks)
    return np.ascontiguousarray(v[a:b])


def exchange_bytes_per_rank(n, m, l, nranks, pad=4):
    """Bytes each rank sends over NVLink per transpose: 16 * pad*N * (P-1) / P^2 (pad = 4 literal, 2 compact)."""
    return 16 * pad * n * m * l * (nranks - 1) // (nranks * nranks)


def make_unique_id():
    buf = (C.c_char * 128)()
    check(lib().ls_nccl_unique_id(buf))
    return bytes(buf)


def broadcast_unique_id(rank, group=None):
    """Rank 0 creates the NCCL id, everyone receives it through torch.distributed (gloo or nccl)."""
    import torch.distributed as dist
    obj = [make_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(obj, src=0, group=group)
    if not (isinstance(obj[0], bytes) and len(obj[0]) == 128):
        raise _lib.LSCudaError(_lib.LS_ERR_NCCL, "NCCL id broadcast failed")
    return obj[0]


class FastM3DSharded(_Handle):
    """The FastM3D operator slab-decomposed over `nranks` GPUs (collective object: every rank
    constructs it and calls each apply).  Vectors are this rank's z slab.  ``embed=True``: any n = m, l <= 512
    with l divisible by nranks, zero-embedded on the power-of-two kernels (see FastM3D)."""

    def __init__(self, nu_slab, n, m, l, k, L, Lp, rank, nranks, unique_id, pad4=False, embed=False):
        super().__init__()
        self.n, self.m, self.l = int(n), int(m), int(l)
        self.ne, self.me, self.le = 4 * self.n, 4 * self.m, 4 * self.l
        self.omega = float(k)
        self.rank, self.nranks = int(rank), int(nranks)
        a, b = vector_range(self.n, self.m, self.l, self.rank, self.nranks)
        self.N = b - a                       # local length
        self.N_global = self.n * self.m * self.l
        nu_slab = np.ascontiguousarray(np.asarray(nu_slab, dtype=np.float64).reshape(-1))
        if nu_slab.shape[0] != self.N:
            raise ValueError("DimensionMismatch: nu slab has %d entries, expected %d" % (nu_slab.shape[0], self.N))
        idbuf = C.create_string_buffer(unique_id, 128) if self.nranks > 1 else None
        check(lib().ls_op3d_create_dist(C.byref(self._h), self.n, self.m, self.l, ptr(nu_slab), self.omega,
                                        float(L), float(Lp), self.rank, self.nranks, idbuf,
                                        (_lib.FLAG_PAD4 if pad4 else 0) | (_lib.FLAG_EMBED if embed else 0)))

    def size(self, dim=None):
        if dim is not None:
            return self.N
        return ((self.N,), (self.N,))

    def eltype(self):
        return np.dtype(np.complex128)

    def info(self):
        """(padding factor, x-slot chunks, transpose route: 'single' / 'nccl' / 'copy-engine')."""
        p, c, x = C.c_int(), C.c_int(), C.c_int()
        check(lib().ls_op3d_info(self.handle, C.byref(p), C.byref(c), C.byref(x)))
        return int(p.value), int(c.value), ("single", "nccl", "copy-engine")[x.value]

    lines = FastM3D.lines
    _apply = FastM3D._apply
    __mul__ = FastM3D.__mul__
    __matmul__ = FastM3D.__mul__
    mul_ = FastM3D.mul_


def matrix_halo(A):
    """Half bandwidth max|row - col| of a sparse matrix: the halo (in vector entries) a row slab needs from each
    z-neighbour.  For the 27-point sparsifier on an n x m x l grid this is n*m + n + 1 (SURVEY.md a11)."""
    coo = A.tocoo()
    return int(np.max(np.abs(coo.row.astype(np.int64) - coo.col.astype(np.int64)))) if coo.nnz else 1


def local_block_csc(A, a, b, halo):
    """Rows [a, b) of the global N x N matrix A with the columns re-based to the window [a - halo, b + halo):
    a (b-a) x (b-a+2*halo) scipy CSC matrix; window columns outside [0, N) are empty."""
    import scipy.sparse as sp
    N = A.shape[1]
    rows = A.tocsr()[a:b, :]
    lo, hi = max(a - halo, 0), min(b + halo, N)
    if rows[:, :lo].nnz or rows[:, hi:].nnz:
        raise ValueError("rows [%d, %d) reach beyond the halo %d" % (a, b, halo))
    mid = rows[:, lo:hi].tocsc()
    left = sp.csc_matrix((b - a, lo - (a - halo)), dtype=mid.dtype)
    right = sp.csc_matrix((b - a, (b + halo) - hi), dtype=mid.dtype)
    blk = sp.hstack([left, mid, right], format="csc")
    blk.sort_indices()
    return blk


class GPUSparseMatrixCSCSharded(_Handle):
    """Row slab of the sparsifying matrix As living next to a FastM3DSharded operator (same z-slab decomposition).
    `A` is the global scipy matrix (every rank holds it on the host, as the reference's setup does) or an already
    extracted local block (then pass halo).  mv / * take and return this rank's slab; collective over the ranks."""

    def __init__(self, A, op, halo=None, is_local_block=False):
        super().__init__()
        from .krylov import _julia_csc
        a, b = vector_range(op.n, op.m, op.l, op.rank, op.nranks)
        if is_local_block:
            if halo is None:
                raise ValueError("a local block needs its halo")
            blk = A
        else:
            halo = matrix_halo(A) if halo is None else int(halo)
            blk = local_block_csc(A, a, b, halo)
        self.halo = int(halo)
        nrows, ncols, colptr, rowval, nzval = _julia_csc(blk)
        if nrows != b - a or ncols != nrows + 2 * self.halo:
            raise ValueError("DimensionMismatch: local block is %d x %d, expected %d x %d" % (nrows, ncols, b - a, b - a + 2 * self.halo))
        self.shape = (nrows, nrows)
        self.nnz = int(colptr[-1] - 1)
        self._op = op                         # the operator (and its communicator) must outlive the matrix
        check(lib().ls_spm_create_dist(C.byref(self._h), op.handle, nrows, self.halo, ptr(colptr), ptr(rowval), ptr(nzval)))
        fmt, ncl = C.c_int(), C.c_int()
        check(lib().ls_spm_info(self.handle, None, None, None, C.byref(fmt), C.byref(ncl)))
        self.format = "stencil" if fmt.value == 1 else "csr"
        self.nclasses = int(ncl.value)

    def mv(self, x, y=None, alpha=1.0, beta=0.0):
        """y <- alpha*A*x + beta*y on this rank's slabs (device buffers or contiguous complex128 arrays)."""
        from ._lib import CDouble
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
        check(lib().ls_spm_mv(self.handle, CDouble.of(alpha), ptr(x), CDouble.of(beta), ptr(y), _lib.MEM_HOST))
        return y

    def __mul__(self, x):
        return self.mv(x)

    __matmul__ = __mul__


class ShardedSparsifyingPreconditioner:
    """``SparsifyingPreconditioner(Msp, As)`` (preconditioner.jl:27-58) next to a FastM3DSharded operator.
    ``As`` is sharded by rows on the GPUs (its halo exchange runs inside every GMRES iteration); the sparse direct
    solve with Msp is not sharded (SURVEY.md section 8(e)): rank 0 holds ``lu(Msp)`` on the host, and the ls_solve_cb
    callback gathers the slabs to it, solves, and scatters the result (CPU tensors on a gloo group)."""

    def __init__(self, Msp, As, op, group=None):
        import torch
        import torch.distributed as dist
        import scipy.sparse.linalg as spla
        from ._lib import SOLVE_CB
        self.As = GPUSparseMatrixCSCSharded(As, op)
        self.MspGPU = None
        self.rank, self.nranks = op.rank, op.nranks
        if group is None and self.nranks > 1:
            group = dist.new_group(backend="gloo") if dist.get_backend() != "gloo" else dist.group.WORLD
        self.group = group
        self.MspInv = spla.splu(Msp.tocsc()) if self.rank == 0 else None
        ranges = [vector_range(op.n, op.m, op.l, r, self.nranks) for r in range(self.nranks)]

        def _cb(user, vptr, n):
            try:
                buf = (C.c_double * (2 * n)).from_address(vptr)
                v = np.frombuffer(buf, dtype=np.complex128)
                if self.nranks == 1:
                    v[:] = self.MspInv.solve(v)
                    return 0
                mine = torch.from_numpy(v.view(np.float64))
                parts = [torch.empty(2 * (b - a), dtype=torch.float64) for a, b in ranges] if self.rank == 0 else None
                dist.gather(mine, parts, dst=0, group=self.group)
                outs = None
                if self.rank == 0:
                    full = np.concatenate([p.numpy().view(np.complex128) for p in parts])
                    sol = self.MspInv.solve(full)
                    outs = [torch.from_numpy(np.ascontiguousarray(sol[a:b]).view(np.float64)) for a, b in ranges]
                dist.scatter(mine, outs, src=0, group=self.group)
                return 0
            except Exception:      # never let an exception cross the C ABI
                return 1
        self._cb = SOLVE_CB(_cb)

    def destroy(self):
        self.As.destroy()
