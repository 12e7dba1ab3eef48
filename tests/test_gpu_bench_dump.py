"""bench.py --dump-outputs: the arrays it writes are what the timed C3 pass computed (checked against the oracle on sampled
envs), and the same arguments give the same arrays from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_STEPS = 40
NAMES = ("envs", "history", "trades", "orders")


def run_bench(out_dir) -> dict:
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "3", "--envs", "64",
           "--sim-steps", str(N_STEPS), "--no-cpu", "--no-logs", "--no-secondary", "--dump-outputs", str(out_dir)]
    res = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    return json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])


@pytest.mark.gpu
def test_bench_dump_outputs_are_the_timed_pass(tmp_path, oracle):
    from bourse_b200 import workloads

    line = run_bench(tmp_path / "a")
    assert line["steps"] == 2 and line["gpu_launches"] == 4
    d = {n: np.load(tmp_path / "a" / f"c3_{n}.npy") for n in NAMES}
    assert all(a.dtype == np.float64 for a in d.values()) and sum(a.nbytes for a in d.values()) <= 64 << 20
    envs = d["envs"].astype(int)
    assert d["history"].shape == (len(envs), N_STEPS, 9)
    for i, e in enumerate(envs[:2]):
        ce = oracle.StepEnvNumpy(0, 0, 1, 1_000_000)
        ce.set_groups(workloads.c3_groups())
        ce.run_agents(N_STEPS, 101, env_id=int(e), keyed=True)
        assert np.array_equal(d["history"][i], ce._history()[:, :9]), e
        tr = d["trades"][d["trades"][:, 0] == e]
        assert len(tr) > 0 and np.array_equal(tr[:, 2:], np.array(ce.get_trades(), dtype=np.float64)), e
        orders = np.array(ce.get_orders(), dtype=np.float64)
        od = d["orders"][d["orders"][:, 0] == e]
        assert np.array_equal(od[:, 1], orders[:, 8]) and np.array_equal(od[:, 2:], orders[:, :8]), e
    run_bench(tmp_path / "b")
    for n in NAMES:
        assert np.array_equal(d[n], np.load(tmp_path / "b" / f"c3_{n}.npy")), n
