"""Device Msp^-1 on 3-D grids (ls_msp_factor3d), measured end to end:

    python scripts/probe_msp3d.py

* examples/example3D.jl at 48^3 (k = 1/h, general-size operator) and the same problem at 64^3 (fast-path operator):
  set-up times (sparsifier sampled on the GPU, factorisation), factor bytes, depth and plan; solve time by CUDA events
  over 20 replays (the factors are larger than the 126 MB L2) with the bandwidth on factor_bytes; GMRES(20) to 1e-8 with
  Pl = I, with Msp^-1 on the device and (48^3 only, in a child process with a time limit) with the host SuperLU
  callback: iterations, wall time, true residual.
* a synthetic 96^3 27-point matrix: factorisation time, factor bytes, residual of one solve.
The card name and power limit are printed first.  HBM reference for the fraction: the 6551 GB/s copy peak measured on
the B200 (SURVEY.md)."""
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import scipy.sparse as sp  # noqa: E402

HBM_GBS = 6551.0


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:      # noqa: BLE001
        return "unknown (%s)" % e


def solve_timing(F, N, reps=20):
    import fast_solver_lippmann_schwinger_b200 as ls
    rng = np.random.default_rng(0)
    b = rng.standard_normal(N) + 1j * rng.standard_normal(N)
    db, dx = ls.DeviceBuffer.from_host(b), ls.DeviceBuffer(b.nbytes)
    for _ in range(3):
        F.solve(db, dx)
    F.sync()
    F.timer_start()
    for _ in range(reps):
        F.solve(db, dx)
    ms = F.timer_stop() / reps
    db.free(); dx.free()
    return ms


def problem(n):
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200 import sparsifier
    from fast_solver_lippmann_schwinger_b200.problems import nu_gaussian_3d_grid
    h = 1.0 / n
    k = 1.0 / h
    x = -0.5 + h * np.arange(n)
    nu = nu_gaussian_3d_grid(n)
    M = ls.FastM3D(None, nu, 4 * n, 4 * n, 4 * n, n, n, n, k, L=1.8 * n * h, Lp=4.0 * n * h)
    X = np.broadcast_to(x[:, None, None], (n, n, n)).reshape(-1, order="F")
    Y = np.broadcast_to(x[None, :, None], (n, n, n)).reshape(-1, order="F")
    Z = np.broadcast_to(x[None, None, :], (n, n, n)).reshape(-1, order="F")
    t0 = time.perf_counter()
    As, Msp = sparsifier.sparsifying_matrices_3d(k, X, Y, Z, M, n, n, n, nu)
    t_sp = time.perf_counter() - t0
    u_inc = np.exp(1j * k * X)
    rhs = -(M * u_inc - u_inc)
    return M, As, Msp, rhs, t_sp


def gmres_run(M, rhs, Pl):
    import fast_solver_lippmann_schwinger_b200 as ls
    t0 = time.perf_counter()
    u, hist = ls.gmres_(np.zeros(rhs.shape[0], complex), M, rhs, Pl=Pl, restart=20, reltol=1e-8, maxiter=2000, log=True)
    wall = time.perf_counter() - t0
    res = np.linalg.norm(M * u - rhs) / np.linalg.norm(rhs)
    return dict(iters=int(hist.iters), converged=bool(hist.isconverged), seconds=round(wall, 3), true_residual=float(res),
                msp_host_seconds=round(float(hist.msp_host_seconds), 3))


def host_route_child(path):
    """the SuperLU callback route on the saved matrices (run in a child process: it may be stopped by the time limit)"""
    import fast_solver_lippmann_schwinger_b200 as ls
    d = np.load(path, allow_pickle=True)
    n = int(d["n"])
    M, _, _, rhs, _ = problem(n)
    As = sp.csc_matrix((d["As_data"], d["As_indices"], d["As_indptr"]), shape=(n ** 3, n ** 3))
    Msp = sp.csc_matrix((d["M_data"], d["M_indices"], d["M_indptr"]), shape=(n ** 3, n ** 3))
    t0 = time.perf_counter()
    P = ls.SparsifyingPreconditioner(Msp, As)
    t_lu = time.perf_counter() - t0
    r = gmres_run(M, rhs, P)
    r["superlu_seconds"] = round(t_lu, 2)
    print("HOSTROUTE " + json.dumps(r), flush=True)


def grid_case(n, host_route):
    import fast_solver_lippmann_schwinger_b200 as ls
    out = {"n": n}
    M, As, Msp, rhs, t_sp = problem(n)
    out["sparsifier_seconds"] = round(t_sp, 2)
    out["nnz"] = int(Msp.nnz)
    t0 = time.perf_counter()
    P = ls.SparsifyingPreconditioner(Msp, As, solverType="GPU", grid=(n, n, n))
    out["factor_call_seconds"] = round(time.perf_counter() - t0, 2)
    F = P.MspGPU
    out.update(factor_seconds=round(F.factor_seconds, 2), factor_bytes=F.factor_bytes, depth=F.depth)
    plan = F.plan()
    ms = solve_timing(F, n ** 3)
    gbs = F.factor_bytes / ms / 1e6
    out.update(solve_ms=round(ms, 3), solve_GBps=round(gbs, 1), solve_fraction_of_hbm=round(gbs / HBM_GBS, 3))
    out["gmres_Pl_I"] = gmres_run(M, rhs, None)
    out["gmres_Pl_device"] = gmres_run(M, rhs, P)
    if host_route:
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "m.npz")
            A, B = As.tocsc(), Msp.tocsc()
            np.savez(path, n=n, As_data=A.data, As_indices=A.indices, As_indptr=A.indptr,
                     M_data=B.data, M_indices=B.indices, M_indptr=B.indptr)
            try:
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--host-route", path],
                                   capture_output=True, text=True, timeout=300)
                lines = [ln for ln in p.stdout.splitlines() if ln.startswith("HOSTROUTE ")]
                out["gmres_Pl_host_superlu"] = json.loads(lines[-1][10:]) if lines else "failed: " + p.stderr[-400:]
            except subprocess.TimeoutExpired:
                out["gmres_Pl_host_superlu"] = "not finished within 300 s"
    P.destroy()
    print(json.dumps(out), flush=True)
    print(plan, flush=True)


def synthetic(n):
    import fast_solver_lippmann_schwinger_b200 as ls
    from util_sparse import stencil27
    t0 = time.perf_counter()
    A = stencil27(n, n, n, seed=96)
    A = (A + (1.0 + np.abs(A).sum(axis=1).max()) * sp.identity(n ** 3, format="csc")).tocsc()    # diagonally dominant
    t_build = time.perf_counter() - t0
    t0 = time.perf_counter()
    F = ls.GPUMspFactorization(A, n, n, n)
    t_f = time.perf_counter() - t0
    rng = np.random.default_rng(1)
    b = rng.standard_normal(n ** 3) + 1j * rng.standard_normal(n ** 3)
    x = F.solve(b)
    G = ls.GPUSparseMatrixCSC(A)
    res = np.linalg.norm(G * x - b) / np.linalg.norm(b)
    ms = solve_timing(F, n ** 3)
    gbs = F.factor_bytes / ms / 1e6
    print(json.dumps(dict(synthetic=n, build_seconds=round(t_build, 1), factor_call_seconds=round(t_f, 2),
                          factor_seconds=round(F.factor_seconds, 2), factor_bytes=F.factor_bytes, depth=F.depth,
                          residual=float(res), solve_ms=round(ms, 3), solve_GBps=round(gbs, 1),
                          solve_fraction_of_hbm=round(gbs / HBM_GBS, 3))), flush=True)
    print(F.plan(), flush=True)
    G.destroy(); F.destroy()


if __name__ == "__main__":
    if "--host-route" in sys.argv:
        host_route_child(sys.argv[sys.argv.index("--host-route") + 1])
        sys.exit(0)
    print("card: " + card(), flush=True)
    grid_case(48, host_route=True)
    grid_case(64, host_route=False)
    synthetic(96)
