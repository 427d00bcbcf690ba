"""bench.py's reference arm runs on the host CPU (the unmodified reference class from the build-time
copy oracle/_ref, or the oracle port where that copy was not built): its JSON line is checked here
against the contract the driver parses.  The CUDA arm's line is produced on the GPU box (`bench.py`, no flags)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "observations/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert "workload" in d["config"] and d["config"]["workload"].startswith("c3")
    cb = d["cpu_baseline"]
    # the unmodified reference (oracle/_ref, built where /root/reference exists) or else the port
    from oracle import build_ref

    assert cb["kind"] == ("reference" if build_ref.verify() else "port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_reference_arm_under_torchrun_env_only_rank0_prints():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT,
                         env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_reference_arm_is_not_pinned_to_one_thread_under_torchrun():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm opens the pools up again (VERDICT r1: the
    N > 1 reference lines were measured on one thread)."""
    env = dict(os.environ, RANK="0", WORLD_SIZE="2", LOCAL_RANK="0", OMP_NUM_THREADS="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "0", "--workload", "c2"], capture_output=True, text=True,
                         timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    ncpu = len(os.sched_getaffinity(0))
    assert d["cpu_baseline"]["cores"] == ncpu and d["n_gpus"] == 2 and d["scaling"] == "strong"
    assert d["config"]["workload"].startswith("c2")


@pytest.mark.gpu
def test_cuda_arm_times_the_requested_steps_and_dumps_reproducible_outputs(tmp_path):
    """--steps sets the number of timed LM iterations; --dump-outputs writes what the last of them
    computed (X, K, R, t and the costs of the last LM run, float64, at most 64 MB), and the same
    arguments give the same outputs."""
    def run(steps, name):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c2", "--steps", str(steps),
                              "--warmup", "1", "--extras", "none", "--no-cpu-baseline", "--dump-outputs",
                              str(tmp_path / name)], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
        files = sorted(os.listdir(tmp_path / name))
        assert files == ["E.npy", "K.npy", "R.npy", "X.npy", "t.npy"]
        arrays = {f[:-4]: np.load(tmp_path / name / f) for f in files}
        assert all(a.dtype == np.float64 for a in arrays.values())
        assert sum(os.path.getsize(tmp_path / name / f) for f in files) <= 64 << 20
        return d, arrays

    d12, a12 = run(12, "a")
    assert d12["steps"] == 12 and d12["inner_solves"] >= 12
    # 12 steps are LM runs of 10 and 2 iterations; E holds the last run's costs
    assert a12["E"].shape == (3,) and a12["X"].shape == (d12["config"]["n_points"], 3)
    assert a12["K"].shape == a12["R"].shape == (d12["config"]["n_cams"], 3, 3)
    d3, a3 = run(3, "b")
    assert d3["steps"] == 3 and a3["E"].shape == (4,)
    _, again = run(3, "c")
    for k in a3:
        np.testing.assert_allclose(again[k], a3[k], rtol=1e-12, atol=1e-12, err_msg=k)
