"""examples/example3D.jl of the reference, on the GPU path.

The shipped 3-D example: h = 1/48, k = 1/h, smooth Gaussian bump, Greengard_Vico quadrature
(example3D.jl:20-54), right-hand side -(A u_inc - u_inc) (example3D.jl:71-72), GMRES.  n = 48 takes the
general-size path (Bluestein lines); powers of two in {64, 128, 256, 512} take the pruned fast path with
the spectrum generated on the device.

    python examples/example3D.py [--n 48] [--precond [--msp {host,gpu}]]

--precond builds the sparsifying preconditioner of example3D.jl:56-67 (27-point As and
Mapproxsp = As + k^2 AG diag(nu)) from 343 unit-vector applies on the GPU operator
(fast_solver_lippmann_schwinger_b200.sparsifier) and keeps As on the GPU.  --msp host (default) factorises
Mapproxsp on the host (SuperLU here, MKL PARDISO upstream: the LU of a 3-D stencil matrix is what limits n);
--msp gpu factorises it on the device (ls_msp_factor3d), so the whole GMRES loop stays there.
"""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fast_solver_lippmann_schwinger_b200 as ls                          # noqa: E402
from fast_solver_lippmann_schwinger_b200.problems import nu_gaussian_3d_grid   # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=48)
    ap.add_argument("--ppw", type=float, default=None, help="points per wavelength (default: k = 1/h as in example3D.jl)")
    ap.add_argument("--precond", action="store_true", help="sparsifying preconditioner (example3D.jl:56-67)")
    ap.add_argument("--msp", choices=("host", "gpu"), default="host", help="where lu(Mapproxsp) is factorised and solved")
    args = ap.parse_args()
    n = args.n
    h = 1.0 / n
    k = 1.0 / h if args.ppw is None else 2 * np.pi / (args.ppw * h)
    x = -0.5 + h * np.arange(n)
    nu = nu_gaussian_3d_grid(n)
    t0 = time.time()
    fastconv = ls.FastM3D(None, nu, 4 * n, 4 * n, 4 * n, n, n, n, k, L=1.8 * n * h, Lp=4.0 * n * h)
    print("operator on the GPU in %.2f s (n = %d, padded %d^3, spectrum generated on the device)" % (time.time() - t0, n, 4 * n))
    X = np.broadcast_to(x[:, None, None], (n, n, n)).reshape(-1, order="F")
    precond = None
    if args.precond:
        from fast_solver_lippmann_schwinger_b200 import sparsifier
        Y = np.broadcast_to(x[None, :, None], (n, n, n)).reshape(-1, order="F")
        Z = np.broadcast_to(x[None, None, :], (n, n, n)).reshape(-1, order="F")
        t0 = time.time()
        As, Mapproxsp = sparsifier.sparsifying_matrices_3d(k, X, Y, Z, fastconv, n, n, n, nu)
        print("As, Mapproxsp from 343 GPU applies in %.2f s (nnz %d)" % (time.time() - t0, As.nnz))
        t0 = time.time()
        if args.msp == "gpu":
            precond = ls.SparsifyingPreconditioner(Mapproxsp, As, solverType="GPU", grid=(n, n, n))
            where = "on the GPU (%.2f GB of factors)" % (precond.MspGPU.factor_bytes / 1e9)
        else:
            precond = ls.SparsifyingPreconditioner(Mapproxsp, As, solverType="MKLPARDISO")
            where = "on the host"
        print("lu(Mapproxsp) %s in %.2f s; As on the GPU as %s (%d classes)" % (
            where, time.time() - t0, precond.As.format, precond.As.nclasses))
    u_inc = np.exp(1j * k * X)
    rhs = -(fastconv * u_inc - u_inc)
    u = np.zeros(n ** 3, dtype=np.complex128)
    t0 = time.time()
    u, hist = ls.gmres_(u, fastconv, rhs, Pl=precond, log=True)
    print("gmres!: %d iterations, converged = %s, %.3f s" % (hist.iters, hist.isconverged, time.time() - t0))
    print(hist["resnorm"])
    print("true relative residual %.3e" % (np.linalg.norm(fastconv * u - rhs) / np.linalg.norm(rhs)))


if __name__ == "__main__":
    main()
