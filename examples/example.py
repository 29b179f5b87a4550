"""examples/example.jl of the reference, on the GPU path.

Solves the Lippmann-Schwinger equation for the shipped smooth Gaussian bump (h = 0.005, n = 201,
k = 1/h, Greengard_Vico quadrature; example.jl:30-54) with GMRES, the operator applies, the
Arnoldi kernels and the Krylov basis living on the B200.  `--n 2048` runs the power-of-two
high-frequency configuration (10 points per wavelength) instead.

    python examples/example.py [--n 201] [--reltol 1.49e-8] [--embed]

`--embed` runs the operator on the power-of-two kernels with the grid zero-embedded, which serves any n <= 4096
(`--n 1001 --embed --precond conv`: h = 1/1000).

The sparsifying preconditioner of example.jl:64-71: `--precond conv` builds As and Mapproxsp with the
convolution-sampled variants of the reference's setup code (buildSparseAConv / buildSparseAGConv,
SparsifyingMatrix2D.jl:441-532, 888-966: 61 unit-vector applies on the GPU operator + nine small SVDs);
`--precond file.npz` takes matrices computed elsewhere (e.g. by the reference's Hankel-sampled buildSparseA),
arrays As_colptr, As_rowval, As_nzval, Msp_colptr, Msp_rowval, Msp_nzval in Julia's 1-based CSC layout.
"""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fast_solver_lippmann_schwinger_b200 as ls                      # noqa: E402
from fast_solver_lippmann_schwinger_b200.problems import gv_spectrum_2d, nu_gaussian_2d   # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=201)
    ap.add_argument("--reltol", type=float, default=float(np.sqrt(np.finfo(float).eps)))
    ap.add_argument("--precond", default=None)
    ap.add_argument("--msp", default="gpu", choices=["gpu", "host"],
                    help="MspInv = lu(Msp) on the device (ls_msp_factor) or on the host (SuperLU through the solve callback)")
    ap.add_argument("--embed", action="store_true",
                    help="run the operator on the power-of-two kernels with the grid zero-embedded (LS_FLAG_EMBED): "
                         "any n <= 4096, e.g. h = 1/1000 (--n 1001), which the Bluestein general path refuses")
    ap.add_argument("--nrhs", type=int, default=1,
                    help="solve for K incident plane waves exp(ik(x cos t + y sin t)), t = 0, pi/K, ..., (K-1) pi/K, in one "
                         "lockstep GMRES: with the device Msp (--msp gpu, implies --precond conv) ls_gmres_msp_batch; with "
                         "--msp host Pl = I (ls_gmres_batch: the host Msp solve has no batched form)")
    args = ap.parse_args()
    if args.nrhs > 1:
        if args.msp == "gpu":
            args.precond = args.precond or "conv"
        else:
            args.precond = None
    n = args.n
    if n % 2 == 1:                       # example.jl: x = -a/2:h:a/2, k = 1/h
        h = 1.0 / (n - 1)
        x = -0.5 + h * np.arange(n)
        k = 1.0 / h
    else:                                # power-of-two configs: x = -a/2:h:a/2-h, 10 points per wavelength
        h = 1.0 / n
        x = -0.5 + h * np.arange(n)
        k = 2 * np.pi / (10 * h)
    X = np.repeat(x[:, None], n, axis=1).reshape(-1, order="F")
    Y = np.repeat(x[None, :], n, axis=0).reshape(-1, order="F")
    nu = nu_gaussian_2d(X, Y)
    t0 = time.time()
    fastconv = ls.FastM(gv_spectrum_2d(n, n, h, k), nu, 4 * n, 4 * n, n, n, k, quadRule="Greengard_Vico", embed=args.embed)
    info = fastconv.info()
    print("operator on the GPU in %.2f s (n = %d, padded %d, route %s, lines %d)"
          % (time.time() - t0, n, 4 * n, ("pow2", "bluestein", "embedded")[info["route"]], info["n_line"]))
    precond = None
    if args.precond == "conv":
        from fast_solver_lippmann_schwinger_b200 import sparsifier
        t0 = time.time()
        # one sampling pass (49 unit-vector applies, rows and Gram matrices kept on the device), then
        # As = buildSparseAConv(...), Mapproxsp = As + k^2 buildSparseAGConv(...) diag(nu)   (example.jl:64-67)
        As, Msp = sparsifier.sparsifying_matrices_2d(k, X, Y, fastconv, n, n, nu, strict=False)
        print("As, Mapproxsp from GPU applies in %.2f s" % (time.time() - t0))
        t0 = time.time()
        precond = (ls.SparsifyingPreconditioner(Msp, As, solverType="GPU", grid=(n, n)) if args.msp == "gpu"
                   else ls.SparsifyingPreconditioner(Msp, As))
        print("SparsifyingPreconditioner(Mapproxsp, As) with lu(Mapproxsp) on the %s in %.2f s" % (args.msp, time.time() - t0))
    elif args.precond:
        import scipy.sparse as sp
        d = np.load(args.precond)
        N = n * n
        As = sp.csc_matrix((d["As_nzval"], d["As_rowval"] - 1, d["As_colptr"] - 1), shape=(N, N))
        Msp = sp.csc_matrix((d["Msp_nzval"], d["Msp_rowval"] - 1, d["Msp_colptr"] - 1), shape=(N, N))
        precond = (ls.SparsifyingPreconditioner(Msp, As, solverType="GPU", grid=(n, n)) if args.msp == "gpu"
                   else ls.SparsifyingPreconditioner(Msp, As))
    if args.nrhs > 1:
        thetas = np.pi * np.arange(args.nrhs) / args.nrhs
        rhs = np.stack([-k ** 2 * ls.FFTconvolution(fastconv, nu * np.exp(1j * k * (X * np.cos(t) + Y * np.sin(t))))
                        for t in thetas], axis=1)
        u = np.zeros(rhs.shape, dtype=np.complex128, order="F")
        t0 = time.time()
        u, hists = ls.gmres_(u, fastconv, rhs, Pl=precond, reltol=args.reltol, log=True)
        print("gmres! for %d directions in lockstep: %.3f s" % (args.nrhs, time.time() - t0))
        for t, hq, q in zip(thetas, hists, range(args.nrhs)):
            res = np.linalg.norm(fastconv * np.ascontiguousarray(u[:, q]) - rhs[:, q]) / np.linalg.norm(rhs[:, q])
            print("direction %d theta %.4f: %d iterations, converged %s, true relative residual %.3e"
                  % (q, t, hq.iters, hq.isconverged, res))
        return
    u_inc = np.exp(1j * k * X)
    rhs = -k ** 2 * ls.FFTconvolution(fastconv, nu * u_inc)          # example.jl:77
    u = np.zeros(n * n, dtype=np.complex128)
    t0 = time.time()
    u, hist = ls.gmres_(u, fastconv, rhs, Pl=precond, reltol=args.reltol, log=True)
    print("gmres!: %d iterations, converged = %s, %.3f s" % (hist.iters, hist.isconverged, time.time() - t0))
    print(hist["resnorm"])
    res = np.linalg.norm(fastconv * u - rhs) / np.linalg.norm(rhs)
    print("true relative residual %.3e" % res)


if __name__ == "__main__":
    main()
