"""Several right-hand sides through one operator: ls_op_apply_batch per column against K, and ls_gmres_batch against solo
ls_gmres runs.

    python scripts/probe_apply_batch.py [--out FILE] [--ks 1,2,4,8] [--rounds 5]

Part 1: ms per column of ls_op_apply_batch (device pointers, mode 0) at K = 1, 2, 4, 8 (chunks of ls_op_batch_cols
columns; K = 1 is the single apply).  Each timed window replays the call for at least WINDOW_MS and ends in ls_sync (a
device synchronise on the handle's stream); the K values alternate within each round and a row is the median over the
rounds, with min and max.  Every column has its own input and output buffer; from 2048^2 and 256^3 up (64 MB and more per
column) the inputs do not stay in the 126 MB L2 between calls, the small grids do (fits_l2 per row).
Part 2: GMRES(20), Pl = Identity, 4 random right-hand sides to reltol 1e-8 (at most 60 iterations): one ls_gmres_batch
run against the four solo ls_gmres runs, wall time (host clock around runs that end in a synchronise), after a warm-up
run of each.  The card's name and power limit head the log."""
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

WINDOW_MS = 200.0


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def op2d(ls, n, embed=False):
    h = 1.0 / n
    x = -0.5 + h * np.arange(n)
    g = np.exp(-40 * x ** 2)
    nu = np.ascontiguousarray((0.3 * g[:, None] * g[None, :]).reshape(-1, order="F"))
    k = 2 * np.pi / (10 * h)
    return ls.FastM(None, nu, 4 * n, 4 * n, n, n, k, quadRule="Greengard_Vico", L=1.5 * n * h, Lp=4.0 * n * h, embed=embed)


def op3d(ls, n, embed=False):
    h = 1.0 / n
    x = -0.5 + h * np.arange(n)
    g = np.exp(-40 * x ** 2)
    nu = np.ascontiguousarray((0.3 * g[:, None, None] * g[None, :, None] * g[None, None, :]).reshape(-1, order="F"))
    k = 2 * np.pi / (10 * h)
    return ls.FastM3D(None, nu, 4 * n, 4 * n, 4 * n, n, n, n, k, L=1.8 * n * h, Lp=4.0 * n * h, embed=embed)


def time_apply(L, M, db, dy, K, check):
    N = M.N
    call = lambda: check(L.ls_op_apply_batch(M.handle, C.c_void_p(db.ptr), N, C.c_void_p(dy.ptr), N, K, 0, 1))  # noqa: E731
    call()
    check(L.ls_sync(M.handle))
    reps, t = 0, 0.0
    t0 = time.perf_counter()
    while t * 1e3 < WINDOW_MS:
        call()
        reps += 1
        if reps % 4 == 0:
            check(L.ls_sync(M.handle))
            t = time.perf_counter() - t0
    check(L.ls_sync(M.handle))
    t = time.perf_counter() - t0
    return 1e3 * t / reps / K


def part1(ls, ks, rounds, log):
    from fast_solver_lippmann_schwinger_b200._lib import DeviceBuffer, check, lib
    L = lib()
    cases = [("2d", 256, False), ("2d", 1024, False), ("2d", 2048, False), ("2d", 4096, False), ("2d", 201, True),
             ("3d", 64, False), ("3d", 256, False), ("3d", 512, False), ("3d", 48, True)]
    rows = []
    for dim, n, embed in cases:
        M = op2d(ls, n, embed) if dim == "2d" else op3d(ls, n, embed)
        N = M.N
        Kmax = max(ks)
        rng = np.random.default_rng(n)
        db = DeviceBuffer(16 * N * Kmax)
        v = (rng.standard_normal(N) + 1j * rng.standard_normal(N)).astype(np.complex128)
        for j in range(Kmax):
            check(L.ls_memcpy_h2d(C.c_void_p(db.ptr + 16 * N * j), v.ctypes.data_as(C.c_void_p), 16 * N))
        dy = DeviceBuffer(16 * N * Kmax)
        res = {K: [] for K in ks}
        for r in range(rounds):
            order = ks if r % 2 == 0 else ks[::-1]
            for K in order:
                res[K].append(time_apply(L, M, db, dy, K, check))
        cols = ls.batch_cols(M)
        base = float(np.median(res[ks[0]]))
        for K in ks:
            med = float(np.median(res[K]))
            row = dict(dim=dim, n=n, embed=embed, N=N, batch_cols=cols, K=K, ms_per_col=med,
                       ms_min=float(min(res[K])), ms_max=float(max(res[K])), speedup_vs_k1=base / med,
                       fits_l2=bool(16 * N * K * 2 < 126e6))
            rows.append(row)
            print(json.dumps(row), file=log, flush=True)
            print(json.dumps(row), flush=True)
        del db, dy
        M.destroy() if hasattr(M, "destroy") else None
        del M
    return rows


def part2(ls, log):
    rows = []
    for dim, n in (("2d", 2048), ("3d", 256)):
        M = op2d(ls, n) if dim == "2d" else op3d(ls, n)
        N = M.N
        rng = np.random.default_rng(3)
        B = np.asfortranarray(rng.standard_normal((N, 4)) + 1j * rng.standard_normal((N, 4)))
        ws = ls.KrylovWorkspace(N)
        kw = dict(reltol=1e-8, restart=20, maxiter=60, log=True, workspace=ws)
        X = np.zeros((N, 4), complex, order="F")
        ls.gmres_(X, M, B, Pl=None, **kw)                       # warm-up
        X[...] = 0
        t0 = time.perf_counter()
        X, hs = ls.gmres_(X, M, B, Pl=None, **kw)
        tb = time.perf_counter() - t0
        x = np.zeros(N, complex)
        ls.gmres_(x, M, np.ascontiguousarray(B[:, 0]), **kw)    # warm-up
        ts, its = 0.0, []
        for q in range(4):
            x = np.zeros(N, complex)
            t0 = time.perf_counter()
            x, h = ls.gmres_(x, M, np.ascontiguousarray(B[:, q]), **kw)
            ts += time.perf_counter() - t0
            its.append(h.iters)
        row = dict(dim=dim, n=n, K=4, batch_s=tb, solo_sum_s=ts, speedup=ts / tb, iters=its,
                   batch_iters=[h.iters for h in hs], maxiter=kw["maxiter"])
        rows.append(row)
        print(json.dumps(row), file=log, flush=True)
        print(json.dumps(row), flush=True)
        del M, ws
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--ks", default="1,2,4,8")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--skip-gmres", action="store_true")
    a = ap.parse_args()
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200._lib import check, lib
    check(lib().ls_set_device(0))
    ks = [int(v) for v in a.ks.split(",")]
    log = open(a.out, "w") if a.out else sys.stdout
    print(json.dumps(dict(card=card(), window_ms=WINDOW_MS, rounds=a.rounds)), file=log, flush=True)
    part1(ls, ks, a.rounds, log)
    if not a.skip_gmres:
        part2(ls, log)


if __name__ == "__main__":
    main()
