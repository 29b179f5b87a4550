"""Timing probe of the zero-embedded 3-D route (LS_FLAG_EMBED) next to the routes it could replace.

Device-resident applies (y = M*b, mode 0) timed with CUDA events on the handle's stream: the median of ROUNDS rounds
of REPS back-to-back applies, pairs timed in alternation.  Every working set here but 48^3's is above the 126 MB L2
(b, y and the intermediates; 100^3 alone is 16 MB per vector but 2n' x m x l intermediates of 82 MB and a 268 MB
spectrum).  The spectra are generated on the device.  Create times are host clocks around a synchronised create; the
embedded route's split into lag extraction (three FP64 ZGEMM contractions) and spectrum comes from its LS_DEBUG line.

    python scripts/probe3d_embed.py [--log profiles/r3_probe3d_embed.log] [--sharded]
    (--sharded: 400^3 and 512^3 on 2 / 4 / 8 GPUs, through torchrun; skipped for world sizes above the GPU count)
"""
import argparse
import ctypes as C
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np                                                       # noqa: E402

ROUTES = ("pow2", "bluestein", "embedded")
ROUNDS, REPS = 5, 10


def nu3(n):
    h = 1.0 / n
    g = np.exp(-40 * (-0.5 + h * np.arange(n)) ** 2)
    return np.ascontiguousarray((0.3 * g[:, None, None] * g[None, :, None] * g[None, None, :]).reshape(-1, order="F"))


def make(n, embed):
    """(handle, create seconds, LS_DEBUG create line or '')"""
    import fast_solver_lippmann_schwinger_b200 as ls
    h = 1.0 / n
    k = 2 * np.pi / (8.3 * h)
    nu = nu3(n)
    with tempfile.TemporaryFile(mode="w+") as err:
        saved = os.dup(2)
        os.dup2(err.fileno(), 2)
        try:
            t0 = time.time()
            M = ls.FastM3D(None, nu, 4 * n, 4 * n, 4 * n, n, n, n, k, L=1.8, Lp=4.0, embed=embed)
            M.sync()
            dt = time.time() - t0
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        err.seek(0)
        lines = [s for s in err.read().splitlines() if "embedded create" in s]
    return M, dt, (lines[0] if lines else "")


def time_pair(Ms, ns):
    import fast_solver_lippmann_schwinger_b200 as ls
    rng = np.random.default_rng(1)
    bufs = []
    for M, n in zip(Ms, ns):
        b = rng.standard_normal(n ** 3) + 1j * rng.standard_normal(n ** 3)
        db, dy = ls.DeviceBuffer.from_host(b), ls.DeviceBuffer(b.nbytes)
        for _ in range(3):
            M.mul_(dy, db)
        M.sync()
        bufs.append((db, dy))
    ms = [[] for _ in Ms]
    for _ in range(ROUNDS):
        for i, M in enumerate(Ms):
            db, dy = bufs[i]
            M.timer_start()
            for _ in range(REPS):
                M.mul_(dy, db)
            ms[i].append(M.timer_stop() / REPS)
    return [float(np.median(t)) for t in ms]


def describe(M):
    i = M.lines()
    return "%s %dx%dx%d" % (ROUTES[i["route"]], i["n_line"], i["m_line"], i["l_line"])


def single(emit):
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200._lib import check, lib
    fma = C.c_double()
    dadd, copy = C.c_double(), C.c_double()
    check(lib().ls_test_device_peaks(C.byref(fma), C.byref(dadd), C.byref(copy)))
    emit("# FP64 FMA peak measured by ls_test_device_peaks: %.1f TFLOP/s" % fma.value)
    emit("%-18s %-24s %10s %9s %-24s %10s %9s %7s" % ("case", "A route", "A ms", "A create", "B route", "B ms",
                                                       "B create", "A/B"))
    os.environ["LS_DEBUG"] = "1"
    creates = []
    # embedded against Bluestein where the Bluestein path fits; 511 and the power-of-two sizes against the fast path
    cases = [(48, True, 48, False), (100, True, 100, False), (200, True, 200, False), (301, True, 301, False),
             (400, True, 400, False), (511, True, 512, False), (64, True, 64, False), (128, True, 128, False),
             (256, True, 256, False), (512, True, 512, False)]
    for na, ea, nb, eb in cases:
        A, ca, la = make(na, ea)
        if la:
            creates.append((na, la))
        try:
            B, cb, _ = make(nb, eb)
        except ls.LSCudaError as ex:       # the Bluestein path's full 4x spectrum no longer fits
            ta = time_pair([A], [na])[0]
            emit("%-18s %-24s %10.4f %8.2fs %-24s %10s %9s %7s" % ("n=%d vs n=%d" % (na, nb), describe(A), ta, ca,
                                                                      "bluestein: %s" % type(ex).__name__, "-", "-", "-"))
            A.destroy()
            continue
        ta, tb = time_pair([A, B], [na, nb])
        emit("%-18s %-24s %10.4f %8.2fs %-24s %10.4f %8.2fs %7.2f" % (
            "n=%d vs n=%d" % (na, nb), describe(A), ta, ca, describe(B), tb, cb, ta / tb))
        A.destroy()
        B.destroy()
    emit("# embedded create split (lag extraction: three FP64 ZGEMM contractions; rate against the FMA peak above)")
    for n, line in creates:
        m = re.search(r"lag extraction ([\d.]+) s \(([\d.e+]+) flop\), spectrum ([\d.]+) s", line)
        if m:
            tl, fl, tsp = float(m.group(1)), float(m.group(2)), float(m.group(3))
            emit("n=%-4d lag extraction %7.3f s  %.2e flop  %6.2f TFLOP/s (%4.1f %% of FMA peak)   spectrum %6.3f s" % (
                n, tl, fl, fl / tl / 1e12, 100 * fl / tl / 1e12 / fma.value, tsp))


def sharded_worker(n, embed):
    """under torchrun: create + apply time of the sharded operator, max over ranks"""
    import torch
    import torch.distributed as dist
    import fast_solver_lippmann_schwinger_b200 as ls
    from fast_solver_lippmann_schwinger_b200 import dist as lsd
    from fast_solver_lippmann_schwinger_b200._lib import check, lib
    rank, world, local = lsd.env_rank()
    check(lib().ls_set_device(local))
    dist.init_process_group("gloo")
    h = 1.0 / n
    k = 2 * np.pi / (8.3 * h)
    a, b_ = lsd.vector_range(n, n, n, rank, world)
    nu = nu3(n)[a:b_]
    uid = lsd.broadcast_unique_id(rank)
    dist.barrier()
    t0 = time.time()
    M = lsd.FastM3DSharded(nu, n, n, n, k, 1.8, 4.0, rank, world, uid, embed=embed)
    M.sync()
    dist.barrier()
    tc = time.time() - t0
    rng = np.random.default_rng(7 + rank)
    b = rng.standard_normal(b_ - a) + 1j * rng.standard_normal(b_ - a)
    db, dy = ls.DeviceBuffer.from_host(b), ls.DeviceBuffer(b.nbytes)
    for _ in range(3):
        M.mul_(dy, db)
    M.sync()
    res = []
    for _ in range(ROUNDS):
        dist.barrier()
        M.timer_start()
        for _ in range(REPS):
            M.mul_(dy, db)
        res.append(M.timer_stop() / REPS)
    t = torch.tensor([float(np.median(res))], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        print("SHARDED P=%d n=%d %s apply %.4f ms create %.2f s chunks %d exchange %s" % (
            world, n, describe(M), float(t[0]), tc, M.info()[1], M.info()[2]), flush=True)
    M.destroy()
    dist.destroy_process_group()


def sharded(emit):
    out = subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True).stdout
    ngpu = sum(1 for s in out.splitlines() if s.startswith("GPU "))
    emit("# sharded: median of %d rounds of %d device-resident applies, max over ranks; create = host clock" % (ROUNDS, REPS))
    for world in (2, 4, 8):
        if world > ngpu:
            emit("P=%d: not measured (%d GPUs visible)" % (world, ngpu))
            continue
        for n, embed in ((400, True), (512, False)):
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                   "--master-addr", "127.0.0.1", "--master-port", str(29700 + world), os.path.abspath(__file__),
                   "--worker", str(n), "1" if embed else "0"]
            p = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
            got = [s for s in p.stdout.splitlines() if s.startswith("SHARDED")]
            emit(got[0] if got else "P=%d n=%d failed: %s" % (world, n, (p.stdout + p.stderr)[-600:]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log", default=None)
    ap.add_argument("--sharded", action="store_true")
    ap.add_argument("--worker", nargs=2, type=int, default=None)
    args = ap.parse_args()
    if args.worker:
        sharded_worker(args.worker[0], bool(args.worker[1]))
        return
    out = [open(args.log, "w")] if args.log else []

    def emit(s):
        print(s, flush=True)
        for f in out:
            f.write(s + "\n")
            f.flush()

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    emit("# device: %s" % (q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"))
    emit("# median of %d alternating rounds of %d device-resident applies, CUDA events, L2 not flushed" % (ROUNDS, REPS))
    single(emit)
    if args.sharded:
        sharded(emit)


if __name__ == "__main__":
    main()
