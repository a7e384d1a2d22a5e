"""CPU: host-side logic that needs no GPU -- factory config handling, spaces, evaluator reduction, sharding,
and the world_size-2 gloo statistics all-reduce."""
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import ROOT


def test_config_to_kwargs_matches_make_env_rules():
    """utils/environment_utils.py:22-37"""
    from reinforcement_learning_rendezvous_b200.environment_utils import config_to_kwargs
    kw = config_to_kwargs(dict(rc0=30, wt0=0.02, dt=0.5), stochastic=False)
    np.testing.assert_array_equal(kw["rc0"], [0, -30, 0])
    np.testing.assert_array_equal(kw["wt0"], [0, 0, 0.02])
    assert all(kw[k] == 0 for k in ("rc0_range", "vc0_range", "qc0_range", "wc0_range", "qt0_range", "wt0_range"))
    assert kw["dt"] == 0.5 and kw["t_max"] is None
    kw = config_to_kwargs(dict(rc0=np.array([1., 2., 3.])), stochastic=True)
    np.testing.assert_array_equal(kw["rc0"], [1, 2, 3])
    assert kw["rc0_range"] is None
    cfg = dict(dt=1)
    config_to_kwargs(cfg, stochastic=False)
    assert cfg == dict(dt=1)                          # caller's dict is not mutated


def test_box_semantics():
    """gym 0.21 Box.contains (rendezvous_env.py:367): dtype castable, shape, inclusive bounds."""
    from reinforcement_learning_rendezvous_b200.spaces import _Box
    box = _Box(-1, 1, (17,), np.float32)
    assert box.contains(np.zeros(17, dtype=np.float32)) and box.contains(np.ones(17, dtype=np.float32))
    assert not box.contains(np.full(17, 1.0000001, dtype=np.float32))
    assert not box.contains(np.zeros(17, dtype=np.float64))          # float64 is not castable to float32
    assert not box.contains(np.zeros(16, dtype=np.float32))
    assert box.sample().shape == (17,) and box.sample().dtype == np.float32


def test_terminal_error_reduction():
    """monte_carlo.py:159-189 first-index logic."""
    from reinforcement_learning_rendezvous_b200.monte_carlo import _terminal_errors
    lim = (0.5, 0.1, np.radians(5), np.radians(1))
    e = np.array([[3.0, 1.0, 0.5, 0.1], [0.4, 0.05, 0.01, 0.001], [0.2, 0.01, 0.02, 0.002]])
    out = _terminal_errors(e, lim)                      # all four met from index 1
    np.testing.assert_allclose(out, [0.3, 0.03, np.degrees(0.015), np.degrees(0.0015)])
    e2 = e.copy()
    e2[:, 3] = 1.0                                      # rot never met -> three-constraint mask (pos, vel, att)
    assert _terminal_errors(e2, lim)[0] == pytest.approx(0.3)
    e3 = np.full((4, 4), 9.0)                           # nothing met -> last sample only
    e3[-1] = [7.0, 6.0, 0.5, 0.25]
    np.testing.assert_allclose(_terminal_errors(e3, lim), [7.0, 6.0, np.degrees(0.5), np.degrees(0.25)])
    e4 = np.full((3, 4), 9.0)
    e4[1:, 0] = 0.1                                     # only position met, from index 1
    assert _terminal_errors(e4, lim)[1] == pytest.approx(9.0)


def test_terminal_error_reduction_batched_equals_per_episode():
    """evaluate_batch reduces all episodes at once (_terminal_errors_batch); same rule, episode by episode, on ragged
    random episodes that exercise every level of the first-index cascade."""
    from reinforcement_learning_rendezvous_b200.monte_carlo import _terminal_errors, _terminal_errors_batch
    lim = (0.5, 0.1, np.radians(5), np.radians(1))
    rng = np.random.default_rng(0)
    t, m = 62, 600
    err = np.abs(rng.normal(size=(t, m, 4))) * np.array([1.0, 0.2, 0.15, 0.03]) * np.linspace(2, 0.1, t)[:, None, None]
    err[:, 100:200, 3] = 1.0                            # rot never met
    err[:, 200:300, 2:] = 1.0                           # only pos / vel can be met
    err[:, 300:400, 1:] = 1.0                           # only pos
    err[:, 400:450] = 9.0                               # nothing met
    lengths = rng.integers(1, t - 1, m)
    for i in range(m):
        err[lengths[i] + 1:, i] = np.nan                # what evaluate_batch leaves after the episode's end
    one = np.array([_terminal_errors(err[:lengths[i] + 1, i], lim) for i in range(m)])
    np.testing.assert_allclose(_terminal_errors_batch(err, lengths, lim), one, rtol=1e-12, atol=0)


def test_shard_range_partitions():
    from reinforcement_learning_rendezvous_b200.distributed import shard_range
    for total, world in ((1 << 20, 8), (65536, 4), (1000, 3), (7, 8), (5, 1)):
        spans = [shard_range(total, world, r) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == total
        assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
        sizes = [hi - lo for lo, hi in spans]
        assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(10, 2, 2)


WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import torch, torch.distributed as dist
from reinforcement_learning_rendezvous_b200.distributed import all_reduce_stats, shard_range, stats_to_dict
from reinforcement_learning_rendezvous_b200 import _native as N
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
rank = dist.get_rank()
lo, hi = shard_range(1001, 2, rank)
stats = torch.zeros(N.NSTATS, dtype=torch.float64)
stats[0] = hi - lo            # steps
stats[1] = rank + 1           # episodes
stats[2] = 10.0 * (rank + 1)  # return_sum
all_reduce_stats(stats)
d = stats_to_dict(stats)
assert d["steps"] == 1001 and d["episodes"] == 3 and abs(d["mean_return"] - 10.0) < 1e-12, d
# the overlapped per-rollout reduction of the benchmark / trainer: 5 "rollouts", collective r waited for after r + 1
from reinforcement_learning_rendezvous_b200.distributed import OverlappedStatsReducer
red = OverlappedStatsReducer("cpu")
for r in range(5):
    buf = red.begin()
    buf[0] += 100 * (rank + 1) + r          # what this rank's rollout kernel would have accumulated
    buf[1] += 1
    red.end()
total = red.finish()
assert total[0] == sum(100 * 1 + r + 100 * 2 + r for r in range(5)) and total[1] == 10, total
dist.barrier()
dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_stats_all_reduce_world_size_2_gloo(tmp_path):
    import socket
    last = ""
    for attempt in range(3):                   # a free port can be taken between probing and binding: try another one
        s = socket.socket()
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
        s.close()
        script = tmp_path / f"worker{attempt}.py"
        script.write_text(WORKER.format(root=ROOT, port=port))
        procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE,
                                  stderr=subprocess.STDOUT, text=True) for r in range(2)]
        try:
            outs = [p.communicate(timeout=600)[0] for p in procs]
        except subprocess.TimeoutExpired:
            for p in procs:
                p.kill()
            last = "timeout"
            continue
        if all(p.returncode == 0 and f"rank {r} ok" in out for r, (p, out) in enumerate(zip(procs, outs))):
            return
        last = "\n".join(outs)
    raise AssertionError(last[-3000:])


def test_bench_reference_arm_runs_on_cpu():
    """bench.py --impl reference must work without a GPU (it times the CPU oracle) and print one JSON line."""
    import json
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1", "--ref-envs", "256"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["unit"] == "env-steps/s"
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["e2e"]["h2d_bytes_per_step"] == 0


def test_gae_matches_sb3_rollout_buffer_restatement():
    """ppo.gae against a numpy restatement of Stable-Baselines3 1.6.2 ``RolloutBuffer.compute_returns_and_advantage``
    (what the reference's ``PPO.learn`` runs, main.py:114): episode_starts[t + 1] = dones[t], the last row uses the
    ``dones`` argument, no time-limit bootstrapping."""
    import torch
    from reinforcement_learning_rendezvous_b200.ppo import gae
    rng = np.random.default_rng(0)
    T, n, gamma, lam = 37, 50, 0.99, 0.95
    rewards = rng.normal(size=(T, n)).astype(np.float32)
    values = rng.normal(size=(T, n)).astype(np.float32)
    dones_after = rng.random((T, n)) < 0.1                 # done flag returned by step t
    last_values = rng.normal(size=n).astype(np.float32)
    # --- SB3's buffer: episode_starts[t] marks that the observation of step t starts an episode
    episode_starts = np.zeros((T, n), dtype=np.float32)
    episode_starts[1:] = dones_after[:-1]
    dones = dones_after[-1].astype(np.float32)
    advantages = np.zeros((T, n), dtype=np.float32)
    last_gae_lam = 0
    for step in reversed(range(T)):
        if step == T - 1:
            next_non_terminal = 1.0 - dones
            next_values = last_values
        else:
            next_non_terminal = 1.0 - episode_starts[step + 1]
            next_values = values[step + 1]
        delta = rewards[step] + gamma * next_values * next_non_terminal - values[step]
        last_gae_lam = delta + gamma * lam * next_non_terminal * last_gae_lam
        advantages[step] = last_gae_lam
    returns = advantages + values
    adv, ret = gae(torch.from_numpy(rewards), torch.from_numpy(values), torch.from_numpy(dones_after),
                   torch.from_numpy(last_values), gamma, lam)
    np.testing.assert_allclose(adv.numpy(), advantages, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(ret.numpy(), returns, rtol=1e-5, atol=1e-6)


def test_ppo_defaults_are_the_references():
    """main.py:39-48: learning_rate 2e-3, batch_size 128, n_epochs 40, clip_range 0.25 (+ SB3 defaults)."""
    from reinforcement_learning_rendezvous_b200.ppo import PPOConfig
    c = PPOConfig()
    assert (c.learning_rate, c.batch_size, c.n_epochs, c.clip_range) == (2e-3, 128, 40, 0.25)
    assert (c.gamma, c.gae_lambda, c.ent_coef, c.vf_coef, c.max_grad_norm) == (0.99, 0.95, 0.0, 0.5, 0.5)


def test_info_dict_builder_cpu():
    """csrc/rdv_host.c (the VecEnv's per-env info dicts, built with the C API): fresh dicts for last step's finished
    envs, {"terminal_observation", "episode": {"r", "l", "t"}} (+ the rich keys) for this step's, errors on bad rows."""
    from reinforcement_learning_rendezvous_b200 import _native as N
    N.build_host()
    h = N.host()
    fin = np.dtype([("env", "<i4"), ("end_reason", "<i4"), ("terminal_obs", "<f4", (17,)), ("pad", "<f4"),
                    ("record", "<f8", (6,))])
    assert fin.itemsize == 128
    n, m = 1000, 37
    rng = np.random.default_rng(0)
    rows = np.zeros(m, dtype=fin)
    rows["env"] = rng.permutation(n)[:m]
    rows["end_reason"] = rng.integers(0, 4, m)
    rows["terminal_obs"] = rng.random((m, 17))
    rows["record"] = rng.random((m, 6)) * 50
    rows["record"][:, 1] = rng.integers(1, 120, m)
    rows["record"][:, 2] = rng.integers(0, 2, m)
    rows["record"][:, 3] = rng.integers(0, 2, m)
    infos = [{} for _ in range(n)]
    keep = list(infos)
    term = np.ascontiguousarray(rows["terminal_obs"])
    dirty_b = h.build_infos(infos, b"", rows, term, 12.5, True, N.END_REASONS)
    dirty = np.frombuffer(dirty_b, dtype=np.int32).tolist()            # packed int32, in the order of the rows
    assert isinstance(dirty_b, bytes) and dirty == rows["env"].tolist()
    for j in range(m):
        d = infos[int(rows["env"][j])]
        np.testing.assert_array_equal(d["terminal_observation"], rows["terminal_obs"][j])
        assert d["episode"] == {"r": round(float(rows["record"][j, 0]), 6), "l": int(rows["record"][j, 1]), "t": 12.5}
        assert d["is_success"] == bool(rows["record"][j, 2] > 0) and d["collided"] == bool(rows["record"][j, 3] > 0)
        assert d["end_reason"] == N.END_REASONS[int(rows["end_reason"][j])]
        assert d["total_delta_v"] == rows["record"][j, 4] and d["total_delta_w"] == rows["record"][j, 5]
    untouched = set(range(n)) - set(rows["env"].tolist())
    assert all(infos[i] is keep[i] for i in untouched)                 # running envs keep their own dict
    # next step: nothing finished -> last step's slots get fresh empty dicts
    dirty2 = h.build_infos(infos, dirty_b, rows[:0], term[:0], 13.0, False, N.END_REASONS)
    assert dirty2 == b"" and all(infos[i] == {} for i in dirty) and len({id(d) for d in infos}) == n
    # dicts the caller kept a reference to are never changed behind its back: they are replaced in the list ...
    assert all(keep[i] == {} for i in range(n)) and all(infos[i] is not keep[i] for i in dirty)
    # ... while a dict only the list holds is reused in place (finished -> filled, next step -> emptied)
    del keep
    ids = [id(d) for d in infos]
    dirty3_b = h.build_infos(infos, b"", rows, term, 14.0, False, N.END_REASONS)
    dirty3 = np.frombuffer(dirty3_b, dtype=np.int32).tolist()
    assert [id(d) for d in infos] == ids and set(infos[int(rows["env"][0])]) == {"terminal_observation", "episode"}
    held = infos[int(rows["env"][0])]                                  # the caller keeps one episode-end dict
    h.build_infos(infos, np.asarray(dirty3, dtype=np.int32), rows[:0], term[:0], 15.0, False, N.END_REASONS)   # any int32 buffer
    assert held["episode"]["t"] == 14.0 and infos[int(rows["env"][0])] == {} and infos[int(rows["env"][0])] is not held
    assert all(infos[i] == {} for i in dirty3) and len({id(d) for d in infos}) == n
    bad = rows[:1].copy()
    bad["env"] = n + 5
    with pytest.raises(IndexError):
        h.build_infos(infos, b"", bad, term[:1], 0.0, False, N.END_REASONS)
    with pytest.raises(ValueError):
        h.build_infos(infos, b"", np.zeros(100, dtype=np.uint8), term[:0], 0.0, False, N.END_REASONS)
    # the terminal observations are row views of the caller's array, made through the numpy C API: float32 [17] with
    # the array as base, and nothing else is accepted (wrong dtype, wrong width, too few rows, a non-contiguous view)
    import sys
    term2 = term.copy()
    base_refs = sys.getrefcount(term2)
    dirty4 = h.build_infos(infos, b"", rows, term2, 16.0, False, N.END_REASONS)
    v = infos[int(rows["env"][3])]["terminal_observation"]
    assert v.dtype == np.float32 and v.shape == (17,) and v.base is term2 and v.flags.c_contiguous and v.flags.writeable
    assert sys.getrefcount(term2) == base_refs + m                     # one reference per view ...
    del v
    h.build_infos(infos, dirty4, rows[:0], term2[:0], 17.0, False, N.END_REASONS)
    assert sys.getrefcount(term2) == base_refs                         # ... and all of them released with the dicts
    for wrong in (term.astype(np.float64), np.zeros((m, 16), np.float32), term[:m - 1], np.zeros((m, 34), np.float32)[:, ::2],
                  [[0.0] * 17] * m):
        with pytest.raises(TypeError):
            h.build_infos(infos, b"", rows, wrong, 0.0, False, N.END_REASONS)
    # `dirty` is a buffer of int32 indices (the prefetches look ahead in it): anything else fails cleanly
    with pytest.raises(TypeError):
        h.build_infos(infos, [0, 1, 2], rows[:0], term[:0], 0.0, False, N.END_REASONS)
    with pytest.raises(ValueError):
        h.build_infos(infos, b"\x00" * 7, rows[:0], term[:0], 0.0, False, N.END_REASONS)
    with pytest.raises(IndexError):
        h.build_infos(infos, np.array([2] * 30 + [n + 7], dtype=np.int32), rows[:0], term[:0], 0.0, False, N.END_REASONS)
    with pytest.raises(IndexError):
        h.build_infos(infos, np.array([5, -1], dtype=np.int32), rows[:0], term[:0], 0.0, False, N.END_REASONS)


def test_cpu_binding_helper_without_nvml():
    """distributed.bind_to_gpu_cpus: without a driver NVML has no answer -> nothing is changed and None comes back."""
    import os
    from reinforcement_learning_rendezvous_b200.distributed import bind_to_gpu_cpus, gpu_cpu_affinity
    before = os.sched_getaffinity(0)
    cores = gpu_cpu_affinity(0)
    assert isinstance(cores, set) and cores <= before
    got = bind_to_gpu_cpus(0, 0, 1)
    if not cores:
        assert got is None and os.sched_getaffinity(0) == before
    else:                                              # a box with a driver: bound to a non-empty subset, then restored
        assert got and got <= cores
        os.sched_setaffinity(0, before)


def test_bench_cpu_baseline_leg_runs_in_a_child():
    """bench.py times its cpu_baseline object in a child interpreter (`--cpu-baseline-only`): one JSON line with the
    keys the contract asks for, no CUDA needed."""
    import json, subprocess, sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--cpu-baseline-only", "--cpu-seconds", "1.0"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    c = json.loads(lines[0])
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0 and c["unit"] == "env-steps/s"
    assert "sample" in c and c["single_process_value"] > 0 and c["c_port_value"] > 0


def test_bench_dump_outputs_samples_within_the_limit(tmp_path):
    """bench.py --dump-outputs: rows that do not fit the size limit are replaced by a fixed seeded sample of envs,
    the same one on every run, with the arrays kept in float32 / float64."""
    import types
    import torch
    import bench
    n = 5000
    obs, state = torch.rand(n, 17), torch.rand(n, 20, dtype=torch.float64)
    env = types.SimpleNamespace(num_envs=n, obs=obs, get_state=lambda: state)
    stats = torch.arange(16, dtype=torch.float64)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), env, stats, limit=300_000)
        assert sum(os.path.getsize(tmp_path / d / f) for f in os.listdir(tmp_path / d)) <= 300_000
    got = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in ("obs", "state", "stats", "env_index")}
    idx = got["env_index"]
    assert got["env_index"].dtype == np.float64 and 0 < len(idx) < n and np.all(np.diff(idx) > 0)
    np.testing.assert_array_equal(idx, np.load(tmp_path / "b" / "env_index.npy"))
    rows = idx.astype(np.int64)
    np.testing.assert_array_equal(got["obs"], obs.numpy()[rows])
    np.testing.assert_array_equal(got["state"], state.numpy()[rows])
    np.testing.assert_array_equal(got["stats"], stats.numpy())
    bench.dump_outputs(str(tmp_path / "c"), env, stats)             # fits the default 64 MB: every env, no index
    assert sorted(os.listdir(tmp_path / "c")) == ["obs.npy", "state.npy", "stats.npy"]
    np.testing.assert_array_equal(np.load(tmp_path / "c" / "obs.npy"), obs.numpy())
