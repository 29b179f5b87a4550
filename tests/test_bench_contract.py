"""bench.py's JSON line and --dump-outputs: the reference arm (the CPU path, no GPU needed) and the device arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env, *args, impl="reference", n=128, steps=2):
    env = dict(os.environ)
    env.update(extra_env)
    env.pop("DUCC0_NUM_THREADS", None)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", impl, "--n", str(n), "--steps", str(steps),
                           "--warmup", "1"] + list(args), capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)


def _json_line(p):
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    return json.loads(lines[0])


def _bench_module():
    import importlib.util
    s = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(s)
    s.loader.exec_module(m)
    return m


def _dumped(d, name="y"):
    a = np.load(os.path.join(d, name + ".npy"))
    assert a.dtype == np.float64 and a.ndim == 2 and a.shape[1] == 2
    return a[:, 0] + 1j * a[:, 1]


def _oracle_apply(n):
    """What both arms of bench.py apply: the n x n workload's operator on rng(1234)'s complex input."""
    from oracle import ls_oracle as O
    from fast_solver_lippmann_schwinger_b200.problems import gv_problem_2d
    nu, gfft, k, h = gv_problem_2d(n)
    M = O.FastM(gfft, nu, 4 * n, 4 * n, n, n, k, quadRule="Greengard_Vico")
    rng = np.random.default_rng(1234)
    return O.fastconvolution(M, rng.standard_normal(n * n) + 1j * rng.standard_normal(n * n))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    p = _run({"OMP_NUM_THREADS": "1"})                      # what torch.distributed.run exports to every rank
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ls_operator_applies_per_s_2d" and d["unit"] == "applies/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["value"] > 0
    assert abs(d["ms_per_step"] * d["value"] - 1e3) < 1e-6 * 1e3
    assert d["config"]["grid"] == [128, 128] and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["cores"] >= 1 and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "applies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_runs_on_rank_zero_only():
    p = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--gpus", "2")
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_cpu_arm_keeps_its_threads_under_torchrun():
    """OMP_NUM_THREADS=1 (exported by torch.distributed.run) must not shrink scipy's FFT pool: bench.py sets DUCC0_NUM_THREADS."""
    code = ("import os, sys; sys.argv=['bench.py']; os.environ['OMP_NUM_THREADS']='1'; os.environ.pop('DUCC0_NUM_THREADS', None); "
            "import importlib.util; s=importlib.util.spec_from_file_location('bench', %r); m=importlib.util.module_from_spec(s); "
            "s.loader.exec_module(m); print(os.environ['DUCC0_NUM_THREADS'])" % os.path.join(ROOT, "bench.py"))
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    assert int(p.stdout.strip()) == (os.cpu_count() or 1)


def test_reference_arm_runs_every_step_and_dumps_its_output(tmp_path):
    d = _json_line(_run({}, "--dump-outputs", str(tmp_path), steps=23))
    assert d["steps"] == 23 and abs(d["ms_per_step"] * d["value"] - 1e3) < 1e-6 * 1e3
    assert sorted(os.listdir(tmp_path)) == ["y.npy"]
    y = _dumped(tmp_path)
    ref = _oracle_apply(128)
    assert np.linalg.norm(y - ref) <= 1e-14 * np.linalg.norm(ref)


def test_steps_below_one_are_refused():
    p = _run({}, steps=0)
    assert p.returncode != 0 and "--steps" in p.stderr


def test_dump_of_a_long_output_is_a_fixed_sample(tmp_path):
    bench = _bench_module()
    K = bench.DUMP_MAX_POINTS
    y = np.arange(K + 1000, dtype=np.float64) * (1 - 2j)
    bench.dump_outputs(str(tmp_path / "a"), {"y": y})
    bench.dump_outputs(str(tmp_path / "b"), {"y": y})
    a, b = _dumped(tmp_path / "a"), _dumped(tmp_path / "b")
    assert a.size == K and np.array_equal(a, b)
    idx = a.real.astype(np.int64)
    assert np.all(np.diff(idx) > 0) and idx[-1] < y.size and np.array_equal(a, y[idx])
    assert os.path.getsize(tmp_path / "a" / "y.npy") <= 64 * 2 ** 20


@pytest.mark.gpu
def test_device_arm_dumps_the_output_of_its_last_step(tmp_path):
    """--dump-outputs on the timed device path: the same seeded input every run, and the output is the operator apply
    the reference arm (the CPU oracle) computes on that input."""
    n = 256
    runs = []
    for i in range(2):
        out = tmp_path / ("ours%d" % i)
        d = _json_line(_run({}, "--dump-outputs", str(out), "--no-extras", "--no-cpu-baseline", impl="ours", n=n, steps=3))
        assert d["steps"] == 3 and d["config"]["grid"] == [n, n]
        runs.append(_dumped(out))
    ref = _oracle_apply(n)
    for y in runs:
        assert y.size == n * n
        assert np.linalg.norm(y - ref) <= 1e-12 * np.linalg.norm(ref)
    assert np.linalg.norm(runs[0] - runs[1]) <= 1e-14 * np.linalg.norm(ref)
