"""Several right-hand sides through one Msp factorisation: ls_msp_solve_batch and ls_gmres_msp_batch.

    python scripts/probe_msp_batch.py [--solve-2d 2048] [--solve-3d 48,64] [--gmres 2048] [--ks 1,2,4,8,16]

Part 1: batched Msp^-1 solve time against K (device pointers, CUDA events on the handle's stream, graphs warmed up;
median of NWIN windows of at least WINDOW_MS each, with their spread) as time per call, time per right-hand side and
the factor bytes over the time per call against the measured copy bandwidth (ls_test_device_peaks; the factors are
larger than the L2, so every call reads them from HBM).  2-D: config 3's Msp
(plasma contrast at 2048^2, sparsifier sampled from GPU applies); 3-D: examples/example3D.jl at n^3.
Part 2: config 3 GMRES(20) to reltol 1e-8 for K incident directions theta = pi q / K in lockstep (ls_gmres_msp_batch):
total time (median of NGMRES runs, with their spread), time per right-hand side, iterations per system.  The timed runs
follow a short warm-up run of the same width."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ctypes as C  # noqa: E402

import numpy as np  # noqa: E402


WINDOW_MS = 300.0   # each timed window replays the call for at least this long
NWIN = 5            # windows per row; ms_per_call is their median, ms_min / ms_max their spread
NGMRES = 3          # timed GMRES runs per K after one short warm-up run; total_s is their median


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:      # noqa: BLE001
        return "unknown (%s)" % e


def copy_gbs():
    from fast_solver_lippmann_schwinger_b200._lib import check, lib
    a, b, c = C.c_double(), C.c_double(), C.c_double()
    check(lib().ls_test_device_peaks(C.byref(a), C.byref(b), C.byref(c)))
    return c.value


def problem2d(n):
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200 import sparsifier as S
    from fast_solver_lippmann_schwinger_b200.problems import nu_plasma_2d
    h = 1.0 / n
    k = 2 * np.pi / (10 * h)
    x = -0.5 + h * np.arange(n)
    X = np.repeat(x[:, None], n, axis=1).reshape(-1, order="F")
    Y = np.repeat(x[None, :], n, axis=0).reshape(-1, order="F")
    nu = np.asarray(nu_plasma_2d(X, Y), dtype=np.float64)
    M = ls.FastM(None, nu, 4 * n, 4 * n, n, n, k, quadRule="Greengard_Vico", L=1.5 * n * h, Lp=4.0 * n * h)
    As, Msp = S.sparsifying_matrices_2d(k, X, Y, M, n, n, nu, strict=False)
    P = ls.SparsifyingPreconditioner(Msp, As, solverType="GPU", grid=(n, n))
    return dict(M=M, P=P, k=k, X=X, Y=Y)


def problem3d(n):
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200 import sparsifier as S
    from fast_solver_lippmann_schwinger_b200.problems import nu_gaussian_3d_grid
    h = 1.0 / n
    k = 1.0 / h
    x = -0.5 + h * np.arange(n)
    nu = nu_gaussian_3d_grid(n)
    M = ls.FastM3D(None, nu, 4 * n, 4 * n, 4 * n, n, n, n, k, L=1.8 * n * h, Lp=4.0 * n * h)
    X = np.broadcast_to(x[:, None, None], (n, n, n)).reshape(-1, order="F")
    Y = np.broadcast_to(x[None, :, None], (n, n, n)).reshape(-1, order="F")
    Z = np.broadcast_to(x[None, None, :], (n, n, n)).reshape(-1, order="F")
    As, Msp = S.sparsifying_matrices_3d(k, X, Y, Z, M, n, n, n, nu)
    P = ls.SparsifyingPreconditioner(Msp, As, solverType="GPU", grid=(n, n, n))
    return dict(M=M, P=P)


def solve_sweep(name, F, ks, peak):
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200._lib import MEM_DEVICE, check, lib
    N = F.N
    rng = np.random.default_rng(0)
    kmax = max(ks)
    b = rng.standard_normal(N * kmax) + 1j * rng.standard_normal(N * kmax)
    db, dx = ls.DeviceBuffer.from_host(b), ls.DeviceBuffer(b.nbytes)
    rows = []
    base = None
    for K in ks:
        call = lambda: check(lib().ls_msp_solve_batch(F.handle, C.c_void_p(db.ptr), N, C.c_void_p(dx.ptr), N, K, MEM_DEVICE))  # noqa: E731
        for _ in range(3):
            call()
        F.sync()
        F.timer_start()
        call()
        reps = max(3, int(np.ceil(WINDOW_MS / F.timer_stop())))
        wins = []
        for _ in range(NWIN):
            F.timer_start()
            for _ in range(reps):
                call()
            wins.append(F.timer_stop() / reps)
        ms = float(np.median(wins))
        base = ms if K == 1 else base
        gbs = F.factor_bytes / ms / 1e6
        row = dict(case=name, K=K, ms_per_call=round(ms, 3), ms_min=round(min(wins), 3), ms_max=round(max(wins), 3),
                   calls_per_window=reps, ms_per_rhs=round(ms / K, 3), vs_K1=round(ms / base, 2),
                   factor_GB=round(F.factor_bytes / 1e9, 3), factor_GBps=round(gbs, 1), frac_of_copy_peak=round(gbs / peak, 3))
        rows.append(row)
        print(json.dumps(row), flush=True)
    db.free(); dx.free()
    return rows


def gmres_sweep(p, ks):
    import fast_solver_lippmann_schwinger_b200 as ls
    M, P, k, X, Y = p["M"], p["P"], p["k"], p["X"], p["Y"]
    N = X.shape[0]
    ws = ls.KrylovWorkspace(N)
    rows = []
    for K in ks:
        th = np.pi * np.arange(K) / K
        B = np.stack([-(M * u - u) for u in (np.exp(1j * k * (X * np.cos(t) + Y * np.sin(t))) for t in th)], axis=1)
        if K == 1:
            b = np.ascontiguousarray(B[:, 0])
            run = lambda **kw: [ls.gmres_(np.zeros(N, complex), M, b, Pl=P, reltol=1e-8, workspace=ws, **kw)[1]]  # noqa: E731
        else:
            run = lambda **kw: ls.gmres_(np.zeros((N, K), complex, order="F"), M, B, Pl=P, reltol=1e-8,  # noqa: E731
                                         workspace=ws, **kw)[1]
        run(maxiter=3, log=True)
        runs = []
        for _ in range(NGMRES):
            t0 = time.perf_counter()
            hs = run(log=True)
            runs.append(time.perf_counter() - t0)
        dt = float(np.median(runs))
        row = dict(case="config3 gmres %d^2" % int(round(N ** 0.5)), K=K, total_s=round(dt, 3),
                   total_min_s=round(min(runs), 3), total_max_s=round(max(runs), 3), s_per_rhs=round(dt / K, 3),
                   iters=[h.iters for h in hs],
                   converged=[h.isconverged for h in hs], driver="ls_gmres_msp" if K == 1 else "ls_gmres_msp_batch")
        rows.append(row)
        print(json.dumps(row), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--solve-2d", type=int, default=2048)
    ap.add_argument("--solve-3d", default="48,64")
    ap.add_argument("--gmres", type=int, default=2048, help="grid side of the config 3 GMRES sweep (0: skip)")
    ap.add_argument("--ks", default="1,2,4,8,16")
    ap.add_argument("--gmres-ks", default="1,2,4,8")
    args = ap.parse_args()
    import fast_solver_lippmann_schwinger_b200 as ls  # noqa: F401
    ks = [int(v) for v in args.ks.split(",")]
    peak = copy_gbs()
    print("card: %s; measured copy bandwidth %.0f GB/s" % (card(), peak), flush=True)
    print("columns per chunk: %s" % os.environ.get("LS_MSP_BATCH_COLS", "4 (default; LS_MSP_BATCH_COLS unset)"), flush=True)
    p2 = None
    if args.solve_2d:
        t0 = time.perf_counter()
        p2 = problem2d(args.solve_2d)
        print("2-D %d^2 config 3 set-up %.1f s; plan:\n%s" % (args.solve_2d, time.perf_counter() - t0, p2["P"].MspGPU.plan()), flush=True)
        solve_sweep("2d %d^2" % args.solve_2d, p2["P"].MspGPU, ks, peak)
    if args.gmres and p2 is not None and args.gmres == args.solve_2d:
        gmres_sweep(p2, [int(v) for v in args.gmres_ks.split(",")])
    if p2 is not None:
        p2["P"].destroy()
        p2 = None
    for n in [int(v) for v in args.solve_3d.split(",") if v]:
        p3 = problem3d(n)
        print("3-D %d^3 plan:\n%s" % (n, p3["P"].MspGPU.plan()), flush=True)
        solve_sweep("3d %d^3" % n, p3["P"].MspGPU, ks, peak)
        p3["P"].destroy()


if __name__ == "__main__":
    main()
