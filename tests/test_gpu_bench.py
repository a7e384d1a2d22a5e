"""GPU: bench.py's contract -- one JSON line on stdout with the keys the driver and the judge read."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import ROOT

pytestmark = pytest.mark.gpu


def _bench(*extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1000", "--warmup", "3",
                          "--steps-per-launch", "40", "--envs", "8192", "--e2e-steps", "5", *extra],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines                      # stdout carries exactly the JSON line
    return json.loads(lines[0])


def test_bench_json_line_contract(tmp_path):
    d = _bench("--cpu-seconds", "1.5", "--dump-outputs", str(tmp_path / "a"))
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert key in d, key
    assert d["unit"] == "env-steps/s" and d["n_gpus"] == 1 and d["steps"] == 1000 and d["warmup"] == 3
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and "workload" in d["config"]
    assert d["value"] > 1e8 and d["gpu_launches"] >= 1
    r = d["roofline"]
    for key in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert key in r, key
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and 0 < r["frac"] < 1.5
    # the timed region is exactly --steps steps, in launches of --steps-per-launch steps
    assert d["config"]["steps_timed"] == 1000 and r["launches_timed"] == 25 and d["gpu_launches"] == 25
    assert abs(d["ms_per_step"] * 1000 - d["config"]["timed_region_ms"]) < 1e-9 * d["config"]["timed_region_ms"]
    assert abs(d["value"] - 8192 * 1000 / (d["config"]["timed_region_ms"] * 1e-3)) < 1e-6 * d["value"]
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 8192 * 6 * 4 and e["d2h_bytes_per_step"] > 8192 * 17 * 4
    assert e["value"] < d["value"]                    # the end-to-end number is not the device-timed one
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0 and "sample" in c
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}

    # --dump-outputs: what the timed rollout returned after its last step; the same arguments give the same inputs,
    # so a second run reproduces every env's observation and state bit for bit
    a = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in ("obs", "state", "stats")}
    assert sorted(os.listdir(tmp_path / "a")) == ["obs.npy", "state.npy", "stats.npy"]
    assert a["obs"].shape == (8192, 17) and a["obs"].dtype == np.float32
    assert a["state"].shape == (8192, 20) and a["state"].dtype == np.float64
    assert a["stats"].shape == (16,) and a["stats"].dtype == np.float64 and a["stats"][0] == 8192 * 1000
    assert np.isfinite(a["obs"]).all() and np.isfinite(a["state"]).all()
    # ... the observation and state after the last timed step: the same Philox actions replayed from the same reset
    # up to that step (in one launch: how the steps are split into launches does not change the bits) give them
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    last = d["config"]["first_timed_step"] + 1000
    assert d["config"]["first_timed_step"] >= d["config"]["warmup_steps"] >= 3
    env = BatchedRendezvousEnv(8192, device="cuda:0", seed=0, auto_reset=True)
    env.reset()
    env.rollout(last, action_seed=1, step_base=0)
    assert np.array_equal(env.obs.cpu().numpy(), a["obs"]) and np.array_equal(env.get_state().cpu().numpy(), a["state"])
    env.rollout(1, action_seed=1, step_base=last)                       # one step later, the state differs
    assert not np.array_equal(env.get_state().cpu().numpy(), a["state"])
    _bench("--no-cpu-baseline", "--dump-outputs", str(tmp_path / "b"))
    b = {k: np.load(tmp_path / "b" / f"{k}.npy") for k in ("obs", "state", "stats")}
    assert np.array_equal(a["obs"], b["obs"]) and np.array_equal(a["state"], b["state"])
    np.testing.assert_allclose(a["stats"], b["stats"], rtol=1e-9)       # fp64 sums, accumulated in any order
