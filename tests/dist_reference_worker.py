"""Worker of the sharded zero-embedded check in tests/test_gpu_kernel_reference.py, run under torchrun:

    python -m torch.distributed.run --nproc-per-node P tests/dist_reference_worker.py N L

The sharded embedded apply on an N x N x L grid (device-generated spectrum) against a single-GPU embedded handle on
rank 0 with the same spectrum: the gathered apply of a random b, FFTconvolution, and impulses at the first and the last
index of every rank's slab.  Rank 0 prints one line per check, ROW|<check>|<relative L2>|<worst / RMS>, of the
convolution part; the test holds them to its bars.  After the checks one apply of a b full of NaN, then b again: the
same bits as the first apply.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _gather_to_root(v, rank, world, dist):
    """This rank's complex slab -> the whole vector on rank 0 (None elsewhere); gloo, CPU tensors."""
    import torch
    mine = torch.from_numpy(np.ascontiguousarray(v).view(np.float64))
    parts = [torch.empty_like(mine) for _ in range(world)] if rank == 0 else None
    dist.gather(mine, parts, dst=0)
    return np.concatenate([p.numpy().view(np.complex128) for p in parts]) if rank == 0 else None


def main():
    import torch.distributed as dist
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200 import dist as lsd
    from fast_solver_lippmann_schwinger_b200._lib import ROUTE_EMBEDDED, check, lib
    from test_gpu_kernel_reference import _embed_len, _errors
    rank, world, local = lsd.env_rank()
    dist.init_process_group("gloo")
    check(lib().ls_set_device(local))
    n, l = int(sys.argv[1]), int(sys.argv[2])
    N = n * n * l
    k, L, Lp = 2 * np.pi * n / 8.3, 1.8, 4.0            # h = 1/n, 8.3 points per wavelength
    rng = np.random.default_rng([n, l, 5])              # the same nu and b on every rank
    nu = rng.standard_normal(N)
    b = rng.standard_normal(N) + 1j * rng.standard_normal(N)
    a, z = lsd.vector_range(n, n, l, rank, world)

    uid = lsd.broadcast_unique_id(rank) if world > 1 else None
    M = lsd.FastM3DSharded(nu[a:z], n, n, l, k, L, Lp, rank, world, uid, embed=True)
    assert M.lines() == {"route": ROUTE_EMBEDDED, "n_line": _embed_len(n), "m_line": _embed_len(n),
                         "l_line": _embed_len(l)}, M.lines()
    assert M.info()[:2] == (2, int(os.environ.get("LS_OP3D_CHUNKS", "1"))), M.info()
    ys = M * np.ascontiguousarray(b[a:z])
    assert np.array_equal(M * np.ascontiguousarray(b[a:z]), ys)
    y = _gather_to_root(ys, rank, world, dist)
    f = _gather_to_root(ls.FFTconvolution(M, np.ascontiguousarray(b[a:z])), rank, world, dist)
    idxs = [i for r in range(world) for i in (lsd.vector_range(n, n, l, r, world)[0],
                                              lsd.vector_range(n, n, l, r, world)[1] - 1)]
    ye = []
    for idx in idxs:
        e = np.zeros(N, complex)
        e[idx] = 1.0
        ye.append(_gather_to_root(M * np.ascontiguousarray(e[a:z]), rank, world, dist))
    M * np.full(z - a, complex(np.nan, np.nan))
    y2 = _gather_to_root(M * np.ascontiguousarray(b[a:z]), rank, world, dist)
    M.destroy()

    if rank == 0:
        assert not np.isnan(y2).any() and np.array_equal(y2, y)
        S = ls.FastM3D(None, nu, 4 * n, 4 * n, 4 * l, n, n, l, k, L=L, Lp=Lp, embed=True)
        rows = [("random b", _errors(y - b, S * b - b)), ("FFTconvolution", _errors(f, ls.FFTconvolution(S, b)))]
        for idx, yi in zip(idxs, ye):
            e = np.zeros(N, complex)
            e[idx] = 1.0
            rows.append(("impulse %d" % idx, _errors(yi - e, S * e - e, yi, (idx,))))
        S.destroy()
        for what, (l2, worst) in rows:
            print("ROW|%s|%.3e|%.3e" % (what, l2, worst), flush=True)
    dist.barrier()
    if rank == 0:
        print("DIST_REFERENCE_OK world=%d n=%d l=%d" % (world, n, l), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
