"""Timing probe of the zero-embedded 2-D route (LS_FLAG_EMBED) next to the routes it could replace.

Device-resident applies (y = M*b, mode 0) timed with CUDA events on the handle's stream.  Each pair of operators is
timed in alternation (ROUNDS rounds of REPS back-to-back applies each) and the median round is reported; the L2 is not
flushed between applies.  Create times include the spectrum set-up (the embedded route's two ZGEMMs).  The spectra are
generated on the device (ls_op2d_create_gv): timings do not depend on their values.

    python scripts/probe2d_embed.py [--log profiles/r3_probe2d_embed.log]
"""
import argparse
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np                                                       # noqa: E402
import fast_solver_lippmann_schwinger_b200 as ls                         # noqa: E402
from fast_solver_lippmann_schwinger_b200.problems import nu_gaussian_2d  # noqa: E402

ROUTES = ("pow2", "bluestein", "embedded")
ROUNDS, REPS = 5, 20


def make(n, embed):
    h = 1.0 / n
    x = -0.5 + h * np.arange(n)
    X = np.repeat(x[:, None], n, axis=1).reshape(-1, order="F")
    Y = np.repeat(x[None, :], n, axis=0).reshape(-1, order="F")
    k = 2 * np.pi / (10 * h)
    t0 = time.time()
    M = ls.FastM(None, nu_gaussian_2d(X, Y), 4 * n, 4 * n, n, n, k, quadRule="Greengard_Vico",
                 L=1.5 * n * h, Lp=4.0 * n * h, embed=embed)
    M.sync()
    return M, time.time() - t0


def time_pair(A, B, n_a, n_b):
    rng = np.random.default_rng(1)
    bufs = []
    for M, n in ((A, n_a), (B, n_b)):
        b = rng.standard_normal(n * n) + 1j * rng.standard_normal(n * n)
        db, dy = ls.DeviceBuffer.from_host(b), ls.DeviceBuffer(b.nbytes)
        for _ in range(3):
            M.mul_(dy, db)
        M.sync()
        bufs.append((db, dy))
    ms = ([], [])
    for _ in range(ROUNDS):
        for i, M in enumerate((A, B)):
            db, dy = bufs[i]
            M.timer_start()
            for _ in range(REPS):
                M.mul_(dy, db)
            ms[i].append(M.timer_stop() / REPS)
    return float(np.median(ms[0])), float(np.median(ms[1]))


def describe(M):
    i = M.info()
    return "%s %dx%d" % (ROUTES[i["route"]], i["n_line"], i["m_line"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log", default=None)
    args = ap.parse_args()
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
    emit("%-22s %-24s %10s %10s %-24s %10s %10s %7s" % ("case", "A route", "A ms", "A create", "B route", "B ms",
                                                        "B create", "A/B"))
    # embedded at the sizes users pick (odd n from x = -0.5:h:0.5) and just above a power of two, next to the fast path
    # at the neighbouring power of two; embedded against Bluestein where both serve
    cases = [(1001, True, 1024, False), (2001, True, 2048, False), (4001, True, 4096, False),
             (1025, True, 2048, False), (201, True, 201, False), (401, True, 401, False), (801, True, 801, False)]
    for na, ea, nb, eb in cases:
        A, ca = make(na, ea)
        B, cb = make(nb, eb)
        ta, tb = time_pair(A, B, na, nb)
        emit("%-22s %-24s %10.4f %9.2fs %-24s %10.4f %9.2fs %7.2f" % (
            "n=%d vs n=%d" % (na, nb), describe(A), ta, ca, describe(B), tb, cb, ta / tb))
        A.destroy()
        B.destroy()


if __name__ == "__main__":
    main()
