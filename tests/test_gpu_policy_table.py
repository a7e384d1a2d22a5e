"""GPU: policy tables -- a different actor per 128-env tile inside the fused rollout.  The oracle is exact: every
tile of a table launch must give the bits of a separate env of its envs (same seed, env_offset = tile start) rolled
with that tile's own MlpPolicy."""
import os

import numpy as np
import pytest

from helpers import GOLDEN

pytestmark = pytest.mark.gpu

T = 128                                                   # envs per policy tile
INT_STATS = ("steps", "episodes", "length_sum", "succeeded", "collided", "end_obs", "end_time", "end_bubble",
             "end_attitude", "rk_accepted", "rk_rejected", "failures")


def _policies():
    """tests/golden/policy.npz and two seeded perturbations of it, each with its own log_std."""
    from reinforcement_learning_rendezvous_b200.policy import MlpPolicy, load_state_dict
    base = load_state_dict(os.path.join(GOLDEN, "policy.npz"))
    out = [MlpPolicy(base)]
    for seed in (1, 2):
        rng = np.random.default_rng(seed)
        sd = {k: (v + rng.normal(0.0, 0.3 * float(v.std()) + 1e-3, v.shape)).astype(np.float32) for k, v in base.items()}
        sd["log_std"] = (base["log_std"] + 0.25 * seed).astype(np.float32)
        out.append(MlpPolicy(sd))
    return out


@pytest.fixture(scope="module")
def pols():
    import torch
    ps = _policies()
    # they must really act differently, or a kernel that always used entry 0 would pass
    obs = torch.rand((4096, 17), device=ps[0].device) * 2 - 1
    acts = [p.forward(obs) for p in ps]
    for i in range(3):
        for j in range(i):
            assert float((acts[i] - acts[j]).abs().max()) > 0.05, (i, j)
    return ps


def _table(ps):
    from reinforcement_learning_rendezvous_b200 import PolicyTable
    return PolicyTable(ps)


REC = dict(record_rewards=True, record_dones=True, record_obs=True, record_actions=True)


# launch shapes: "grid" -- one CTA per SM, so the small batches here give each CTA one tile and one pass; "one_cta" --
# every SM but one reserved, so a single CTA walks all tiles, two per pass (both groups active), and each group restages
# its weight set whenever the tile map hands it another entry
SHAPES = ("grid", "one_cta")


def _shape(env, shape):
    import torch
    if shape == "one_cta":
        env.sm_reserve = torch.cuda.get_device_properties(env.device).multi_processor_count - 1
    return env


def _run(env, steps, stochastic, **kw):
    return env.rollout(steps, stochastic=stochastic, action_seed=11 if stochastic else None, **REC, **kw)


def _assert_stats(big, parts):
    """stats of one launch == the sum over separate launches: integer slots exact, fp64 sums to 1e-12 (atomic order)"""
    for k, v in big.items():
        want = sum(p[k] for p in parts)
        if k in INT_STATS:
            assert v == want, k
        else:
            assert abs(v - want) <= 1e-12 * max(abs(want), 1.0), (k, v, want)


def _assert_tile_equal(env, out, lo, hi, e, o):
    import torch
    m = hi - lo
    for key in ("rewards", "dones", "actions", "obs_steps"):
        assert torch.equal(out[key][:, lo:hi], o[key]), key
    assert torch.equal(out["obs"][lo:hi], o["obs"])
    assert torch.equal(env.f64[:, lo:hi], e.f64[:, :m])
    assert torch.equal(env.i32[:, lo:hi], e.i32[:, :m])


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("stochastic", [False, True])
def test_tiles_equal_separate_launches(pols, stochastic, shape):
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    # one_cta: passes of tiles (0, 1) (2, 3) (4, 5) (6, 7): group 0 holds entries 2, 2, 1, 2 (kept once, restaged
    # twice), group 1 entries 0, 1, 0, 1 (restaged every pass); the last pass's group 1 has 37 envs
    n, tiles, K = T * 7 + 37, [2, 0, 2, 1, 1, 0, 2, 1], 24
    env = _shape(BatchedRendezvousEnv(n, seed=5, auto_reset=True), shape)
    env.reset()
    out = _run(env, K, stochastic, policy=_table(pols), policy_tiles=tiles)
    assert int(out["dones"].sum()) > 0                  # episodes end and restart inside the launch
    parts = []
    for t, entry in enumerate(tiles):
        lo, hi = T * t, min(T * (t + 1), n)
        e = BatchedRendezvousEnv(hi - lo, seed=5, env_offset=lo, auto_reset=True)
        e.reset()
        o = _run(e, K, stochastic, policy=pols[entry])
        _assert_tile_equal(env, out, lo, hi, e, o)
        parts.append(e.read_stats())
    _assert_stats(env.read_stats(), parts)


SETS = [dict(), dict(h=600e3), dict(rc0=np.array([0.0, -20.0, 0.0]))]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("stochastic", [False, True])
def test_tiles_with_parameter_table(pols, stochastic, shape):
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    sets = SETS
    per, K = 256, 24
    env = _shape(BatchedRendezvousEnv(per * 3, seed=7, auto_reset=True, param_batches=[(per, s) for s in sets]), shape)
    assert env.param_table is not None
    env.reset()
    out = _run(env, K, stochastic, policy=_table(pols), policy_tiles=[0, 0, 1, 1, 2, 2])
    parts = []
    for i, s in enumerate(sets):
        e = BatchedRendezvousEnv(per, seed=7, env_offset=per * i, auto_reset=True, **s)
        e.reset()
        o = _run(e, K, stochastic, policy=pols[i])
        _assert_tile_equal(env, out, per * i, per * (i + 1), e, o)
        parts.append(e.read_stats())
    _assert_stats(env.read_stats(), parts)


@pytest.mark.parametrize("stochastic", [False, True])
def test_one_entry_table_equals_single_policy(pols, stochastic):
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    n, K = 8192, 16
    a = BatchedRendezvousEnv(n, seed=9, auto_reset=True)
    b = BatchedRendezvousEnv(n, seed=9, auto_reset=True)
    a.reset()
    b.reset()
    oa = _run(a, K, stochastic, policy=_table([pols[1]]), policy_tiles=[0] * (n // T))
    ob = _run(b, K, stochastic, policy=pols[1])
    _assert_tile_equal(a, oa, 0, n, b, ob)
    _assert_stats(a.read_stats(), [b.read_stats()])


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("ptable", [False, True])
def test_evaluator_mode_equals_separate_launches(pols, ptable, shape):
    """Evaluator mode (mc_out): every tile's per-episode results, final state and observation equal a separate
    evaluator launch of its envs with its own model; with and without a parameter table."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    if ptable:
        per = 256
        blocks = [(per * i, per * (i + 1), SETS[i], i) for i in range(3)]
        env = BatchedRendezvousEnv(per * 3, seed=12, auto_reset=False, param_batches=[(per, s) for s in SETS])
        tiles = [0, 0, 1, 1, 2, 2]
    else:
        n, tiles = T * 7 + 37, [2, 0, 2, 1, 1, 0, 2, 1]
        blocks = [(T * t, min(T * (t + 1), n), {}, e) for t, e in enumerate(tiles)]
        env = BatchedRendezvousEnv(n, seed=12, auto_reset=False)
    _shape(env, shape)
    env.reset()
    steps = max(int(g.params.done_steps) for g in env.groups)
    mc = env.rollout(steps, policy=_table(pols), policy_tiles=tiles, monte_carlo=True)["mc"]
    for lo, hi, kw, entry in blocks:
        e = BatchedRendezvousEnv(hi - lo, seed=12, env_offset=lo, auto_reset=False, **kw)
        e.reset()
        o = e.rollout(steps, policy=pols[entry], monte_carlo=True)
        assert torch.equal(mc[lo:hi], o["mc"]), (lo, entry)
        assert torch.equal(env.obs[lo:hi], o["obs"]), (lo, entry)
        assert torch.equal(env.f64[:, lo:hi], e.f64[:, :hi - lo]) and torch.equal(env.i32[:, lo:hi], e.i32[:, :hi - lo])


def test_tile_map_upload(pols):
    """The tile map is uploaded from pinned memory without waiting for the stream and kept while it does not change:
    launches that switch maps back to back, with no synchronisation, equal the same launches with one after each."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    n = T * 7 + 37
    maps = [[2, 0, 2, 1, 1, 0, 2, 1], [2, 0, 2, 1, 1, 0, 2, 1], [0, 1, 2, 0, 1, 2, 0, 1], [1, 1, 1, 1, 0, 0, 0, 0]]
    table = _table(pols)
    envs = [_shape(BatchedRendezvousEnv(n, seed=3, auto_reset=True), "one_cta") for _ in range(2)]
    for e in envs:
        e.reset()
    torch.cuda.synchronize()
    outs = [[], []]
    kept = []
    for k, m in enumerate(maps):
        outs[0].append(envs[0].rollout(4, policy=table, policy_tiles=m, record_rewards=True)["rewards"])
        kept.append(envs[0]._tile_map[1])
        outs[1].append(envs[1].rollout(4, policy=table, policy_tiles=torch.tensor(m), record_rewards=True)["rewards"])
        torch.cuda.synchronize()
    assert kept[0] is kept[1] and kept[1] is not kept[2]
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    assert torch.equal(envs[0].f64, envs[1].f64) and torch.equal(envs[0].obs, envs[1].obs)


def test_launch_shape_invariance(pols):
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    n, tiles = T * 7 + 37, [1, 2, 0, 0, 2, 1, 1, 2]
    table = _table(pols)
    envs = [BatchedRendezvousEnv(n, seed=4, auto_reset=True) for _ in range(3)]
    for e in envs:
        e.reset()
    envs[1].sm_reserve = 7
    o0 = envs[0].rollout(16, policy=table, policy_tiles=tiles, record_rewards=True, record_dones=True)
    o1 = envs[1].rollout(16, policy=table, policy_tiles=tiles, record_rewards=True, record_dones=True)
    # four 4-step launches that carry the prefetched reset rows == one 16-step launch
    recs = [envs[2].rollout(4, policy=table, policy_tiles=tiles, record_rewards=True, record_dones=True)
            for _ in range(4)]
    for key in ("rewards", "dones"):
        assert torch.equal(o0[key], o1[key]), key
        assert torch.equal(o0[key], torch.cat([r[key] for r in recs])), key
    for e in envs[1:]:
        assert torch.equal(envs[0].f64, e.f64) and torch.equal(envs[0].i32, e.i32) and torch.equal(envs[0].obs, e.obs)


def test_evaluate_batch_with_a_policy_list(pols):
    from helpers import golden
    from reinforcement_learning_rendezvous_b200 import evaluate_batch
    ics = golden("mc.npz")["ic_raw"]
    both = evaluate_batch([pols[0], pols[2]], ics, return_raw=True)
    assert isinstance(both, list) and len(both) == 2
    for res, p in zip(both, (pols[0], pols[2])):
        one = evaluate_batch(p, ics, return_raw=True)
        assert set(res) == set(one)
        for k in one:
            assert np.array_equal(res[k], one[k], equal_nan=True), k
    assert not np.array_equal(both[0]["raw"], both[1]["raw"])


def test_evaluate_sweep_one_model_per_set(pols):
    from reinforcement_learning_rendezvous_b200 import evaluate_sweep
    sets = [dict(), dict(h=400e3), dict(dt=0.5), dict(koz_radius=10.0), dict(rc0=20.0), dict(corridor_half_angle=0.6)]
    models = [pols[i % 3] for i in range(len(sets))]
    kw = dict(episodes_per_set=256, seed=3, t_max=60)
    res = evaluate_sweep(models, sets, **kw)
    assert len(res) == len(sets)
    for i in range(len(sets)):
        assert res[i] == evaluate_sweep(models[i], sets, **kw)[i], i
    parts = evaluate_sweep(models, sets, rank=0, world_size=2, **kw) + \
        evaluate_sweep(models, sets, rank=1, world_size=2, **kw)
    assert parts == res
    with pytest.raises(ValueError):
        evaluate_sweep(models, sets, episodes_per_set=192, seed=3, t_max=60)


def _check_zeroed(run_bad, run_good, n, K, zeroed, shape):
    """Tiles in `zeroed` take zero actions (same records and state as a zero-action rollout of the same envs) and count
    one failure per env-step; every other tile equals the valid run."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    envs = [_shape(BatchedRendezvousEnv(n, seed=8, auto_reset=True), shape) for _ in range(3)]
    for e in envs:
        e.reset()
    og = run_good(envs[0])
    zeros = torch.zeros((K, n, 6), dtype=torch.float32, device=envs[2].device)
    oz = envs[2].rollout(K, actions=zeros, record_rewards=True, record_dones=True)
    ob = run_bad(envs[1])
    tiles = (n + T - 1) // T
    for t in range(tiles):
        lo, hi = T * t, min(T * (t + 1), n)
        if t not in zeroed:
            for key in ("rewards", "dones", "actions", "obs_steps"):
                assert torch.equal(ob[key][:, lo:hi], og[key][:, lo:hi]), (t, key)
            assert torch.equal(envs[1].f64[:, lo:hi], envs[0].f64[:, lo:hi]), t
        else:
            assert not bool(ob["actions"][:, lo:hi].any()), t
            for key in ("rewards", "dones"):
                assert torch.equal(ob[key][:, lo:hi], oz[key][:, lo:hi]), (t, key)
            assert torch.equal(envs[1].f64[:, lo:hi], envs[2].f64[:, lo:hi]), t
    assert envs[0].read_stats()["failures"] == 0
    assert envs[1].read_stats()["failures"] == K * sum(min(T * (t + 1), n) - T * t for t in zeroed)


@pytest.mark.parametrize("shape", SHAPES)
def test_out_of_range_tiles(pols, monkeypatch, shape):
    """An index outside the table, passed through the C ABI: that tile takes zero actions and counts one failure per
    env-step; the other tiles are unchanged.  Through Python such an index, or a wrong length, raises."""
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, batched_env
    n, K = T * 4 + 50, 12
    good, bad = [0, 1, 2, 1, 0], [0, 3, 2, -1, 0]
    table = _table(pols)
    env = BatchedRendezvousEnv(n, seed=8, auto_reset=True)
    env.reset()
    with pytest.raises(ValueError):
        env.rollout(K, policy=table, policy_tiles=bad)
    with pytest.raises(ValueError):
        env.rollout(K, policy=table, policy_tiles=good[:-1])

    def run_bad(e):
        with monkeypatch.context() as m:
            m.setattr(batched_env, "policy_tile_indices", lambda tiles, n_, c: np.asarray(tiles, dtype=np.int32))
            return e.rollout(K, policy=table, policy_tiles=bad, **REC)
    _check_zeroed(run_bad, lambda e: e.rollout(K, policy=table, policy_tiles=good, **REC), n, K, {1, 3}, shape)


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("flaw", ["hidden", "weights", "log_std"])
def test_entries_the_actor_cannot_run(pols, flaw, shape):
    """The kernel checks each table entry when a group stages it: an entry of another width, with a NULL weight, or
    without log_std in a sampling rollout is treated like an index outside the table (C callers fill the table
    themselves; PolicyTable never builds such entries)."""
    import ctypes as C
    import torch
    from reinforcement_learning_rendezvous_b200 import _native as N
    n, K, tiles = T * 4 + 50, 12, [0, 1, 2, 1, 0]
    stochastic = flaw == "log_std"
    good = _table(pols)
    flawed = _table(pols)
    size = C.sizeof(N.RdvPolicy)
    field = {"hidden": N.RdvPolicy.hidden, "weights": N.RdvPolicy.w1, "log_std": N.RdvPolicy.log_std}[flaw]
    off = size + field.offset                                       # entry 1
    flawed.table[off:off + field.size] = torch.tensor(
        list((32).to_bytes(4, "little")) if flaw == "hidden" else [0] * field.size, dtype=torch.uint8)
    run = lambda tab: (lambda e: _run(e, K, stochastic, policy=tab, policy_tiles=tiles))   # noqa: E731
    _check_zeroed(run(flawed), run(good), n, K, {1, 3}, shape)
