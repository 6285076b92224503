"""bench.py on a small workload: `--steps` sets the number of timed steps, and `--dump-outputs` writes what the last of
them computed, the same for the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENVS, T, B, E, STEPS = 64, 128, 4096, 2, 2
ARGS = ["--envs", str(ENVS), "--rollout-steps", str(T), "--minibatch", str(B), "--epochs", str(E), "--steps", str(STEPS),
        "--warmup", "3", "--no-kernels", "--no-cpu", "--no-variants", "--no-e2e"]


def _bench(out_dir):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *ARGS, "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    return line, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    line, out = _bench(tmp_path / "a")
    assert line["steps"] == STEPS
    assert all(a.dtype == np.float32 for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    assert out["advantage"].shape == (ENVS, T, 1) and out["current_state_value_target"].shape == (ENVS, T, 1)
    assert out["losses"].shape == (E * (ENVS * T // B), 2)
    assert out["losses"][-1].tolist() == line["final_losses"]
    params = {k[len("param."):] for k in out if k.startswith("param.")}
    assert {"actor.actor_logstd", "critic.network.last_layer.weight"} <= params
    for k in params:
        assert f"adam_exp_avg.{k}" in out and f"adam_exp_avg_sq.{k}" in out
    assert all(np.isfinite(a).all() for a in out.values())
    # seeded inputs: a second run of the same arguments computes the same outputs (up to the order of float sums)
    _, again = _bench(tmp_path / "b")
    assert sorted(again) == sorted(out)
    for k, a in out.items():
        scale = max(float(np.abs(a).max()), 1e-30)
        assert float(np.abs(again[k] - a).max()) <= 1e-5 * scale, k
