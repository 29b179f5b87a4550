"""Worker of the sharded zero-embedded 3-D tests (tests/test_gpu_apply3d_embed.py), run under torchrun:

    python -m torch.distributed.run --nproc-per-node P tests/dist_embed_worker.py N

n = l = N on P GPUs: the gathered sharded apply against the oracle and the single-GPU embedded apply, and sharded
GMRES(20) against the single-GPU embedded run.  With 8 ranks also 400^3 against the single-GPU embedded apply.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _gather_to_root(v, rank, world, dist):
    """This rank's complex slab -> the whole vector on rank 0 (None elsewhere); gloo, CPU tensors."""
    import torch
    mine = torch.from_numpy(np.ascontiguousarray(v).view(np.float64))
    parts = [torch.empty_like(mine) for _ in range(world)] if rank == 0 else None
    dist.gather(mine, parts, dst=0)
    return np.concatenate([p.numpy().view(np.complex128) for p in parts]) if rank == 0 else None


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def main():
    import torch.distributed as dist
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200 import dist as lsd
    from fast_solver_lippmann_schwinger_b200._lib import ROUTE_EMBEDDED, check, lib
    rank, world, local = lsd.env_rank()
    dist.init_process_group("gloo")
    check(lib().ls_set_device(local))
    n = int(sys.argv[1])
    l = n
    h = 1.0 / n
    k = 2 * np.pi / (8.3 * h)
    x = -0.5 + h * np.arange(n)
    Mo = None
    if rank == 0:
        from oracle import ls_oracle as O
        Mo = O.buildFastConvolution3D(x, x, x, h, k, O.nu_gaussian_3d)
    obj = [Mo.nu if rank == 0 else None]
    dist.broadcast_object_list(obj, src=0)
    nu = obj[0]
    a, b_ = lsd.vector_range(n, n, l, rank, world)

    uid = lsd.broadcast_unique_id(rank)
    M = lsd.FastM3DSharded(nu[a:b_], n, n, l, k, 1.8 * n * h, 4.0 * n * h, rank, world, uid, embed=True)
    p = 64
    while p < n:
        p *= 2
    assert M.lines() == {"route": ROUTE_EMBEDDED, "n_line": p, "m_line": p, "l_line": p}, M.lines()
    assert M.info()[0] == 2
    rng = np.random.default_rng(1234)
    b = rng.standard_normal(n ** 3) + 1j * rng.standard_normal(n ** 3)
    c = rng.standard_normal(n ** 3) + 1j * rng.standard_normal(n ** 3)
    y = _gather_to_root(M * np.ascontiguousarray(b[a:b_]), rank, world, dist)
    yc = _gather_to_root(M * np.ascontiguousarray(c[a:b_]), rank, world, dist)      # second apply, other data
    f = _gather_to_root(ls.FFTconvolution(M, np.ascontiguousarray(b[a:b_])), rank, world, dist)
    S = None
    if rank == 0:
        from oracle import ls_oracle as O
        S = ls.FastM3D(None, nu, 4 * n, 4 * n, 4 * l, n, n, l, k, L=1.8 * n * h, Lp=4.0 * n * h, embed=True)
        e_or = max(_rel(y, Mo * b), _rel(yc, Mo * c))
        assert e_or <= 1e-12, e_or
        assert _rel(f, O.FFTconvolution3D(Mo, b)) <= 1e-12
        e_single = max(_rel(y, S * b), _rel(yc, S * c), _rel(f, ls.FFTconvolution(S, b)))
        assert e_single <= 1e-13, e_single

    # sharded GMRES(20), Pl = I, against the single-GPU embedded run
    X = np.repeat(x[:, None], n * l, axis=1).reshape(-1, order="F")       # x fastest
    u_inc = np.exp(1j * k * X)
    rhs = (-(S * u_inc - u_inc)) if rank == 0 else None
    obj = [rhs]
    dist.broadcast_object_list(obj, src=0)
    rhs = obj[0]
    _, hs = ls.gmres_(np.zeros(b_ - a, complex), M, np.ascontiguousarray(rhs[a:b_]), restart=20, maxiter=40, log=True)
    hist_rel = 0.0
    if rank == 0:
        _, h1 = ls.gmres_(np.zeros(n ** 3, complex), S, rhs, restart=20, maxiter=40, log=True)
        assert hs.iters == h1.iters, (hs.iters, h1.iters)
        hist_rel = float(np.max(np.abs(np.asarray(hs["resnorm"]) - np.asarray(h1["resnorm"])) / np.asarray(h1["resnorm"])))
        assert hist_rel < 1e-8, hist_rel
        S.destroy()
    M.destroy()
    dist.barrier()

    big = ""
    if world == 8:
        nb = 400
        hb = 1.0 / nb
        kb = 2 * np.pi / (8.3 * hb)
        xb = -0.5 + hb * np.arange(nb)
        g = np.exp(-40 * xb ** 2)
        a2, b2 = lsd.vector_range(nb, nb, nb, rank, world)
        nub = (0.3 * g[:, None, None] * g[None, :, None] * g[None, None, :]).reshape(-1, order="F")
        rngb = np.random.default_rng(400)
        bb = rngb.standard_normal(nb ** 3) + 1j * rngb.standard_normal(nb ** 3)
        uidb = lsd.broadcast_unique_id(rank)
        Mb = lsd.FastM3DSharded(nub[a2:b2], nb, nb, nb, kb, 1.8, 4.0, rank, world, uidb, embed=True)
        assert Mb.lines()["n_line"] == 512 and Mb.lines()["l_line"] == 512
        yb = _gather_to_root(Mb * np.ascontiguousarray(bb[a2:b2]), rank, world, dist)
        Mb.destroy()
        dist.barrier()
        if rank == 0:
            Sb = ls.FastM3D(None, nub, 4 * nb, 4 * nb, 4 * nb, nb, nb, nb, kb, L=1.8, Lp=4.0, embed=True)
            e400 = _rel(yb, Sb * bb)
            Sb.destroy()
            assert e400 <= 1e-13, e400
            big = " e400=%.2e" % e400
    dist.barrier()
    if rank == 0:
        print("DIST_EMBED_OK world=%d n=%d apply_err_oracle=%.2e apply_err_single=%.2e gmres_iters=%d hist_rel=%.2e%s" % (
            world, n, e_or, e_single, hs.iters, hist_rel, big), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
