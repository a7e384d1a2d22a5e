"""GPU: the single-policy fused rollout (rollout_kernel<.., POLICY>) at every CTA shape it ships with, and the
Gaussian head's noise, against independent references.

* Shapes: 256 / 384 / 448 / 512 threads forced onto 3 CTAs with two passes each and a ragged last group, and the
  natural dispatch of the benchmark (sms x 443 envs: one pass of 448 threads, the fourth group 64 threads wide) and
  of twice that (two passes).  Every run is two launches with the reset rows carried, auto-reset and t_max = 12, so
  episodes restart inside and across launches.  The env is checked against the C oracle (tests/ledger.py replaying
  the recorded actions), the actor against an fp64 evaluation of the same weights on the observation the kernel
  saw, the sampled noise against tests/normals.py, and the shapes against each other bit for bit.
* Noise: with action_net = 0 and an fp16-exact bias the actor's output is exactly that bias, so the recorded draw
  is b2 + exp(log_std) z and z is checked against philox_normals_ref to the rounding of the device's float32
  logf / sqrtf / sincospif: under high words of env id, seed and step index, at every shape, across launch splits,
  shards, policy tables, and through PPO's collection, log-probabilities and GAE.
"""
import os

import numpy as np
import pytest

from helpers import GOLDEN, REL_TOL, rel_err
from ledger import FLOAT_STATS, INT_STATS, Ledger, assert_stats, short_solve_steps
from normals import philox_normals_ref

from oracle import c_oracle as CO

pytestmark = pytest.mark.gpu

T_MAX = 12
K = 9                          # steps per launch; two launches, so the time limit ends episodes inside the second
SEED, ASEED = 31, 0x0000000700000013
FORCED = (256, 384, 448, 512)
ACT_BOUND = 8e-6               # tensor-core actor vs fp64 (test_gpu_frontends.test_policy_forward_matches_torch_fp32)
OBS_TOL = 1.2e-7
EPS = 2.0 ** -23
# the draw's own error: logf within 1 ulp, correctly rounded sqrtf, sincospif within 1 ulp, the product r * cos
Z_ULPS = 4
REC = dict(record_rewards=True, record_dones=True, record_obs=True, record_actions=True)


def _tune(key, value):
    from reinforcement_learning_rendezvous_b200 import _native as N
    return N.lib().rdv_tune(key, int(value))


def _sms():
    import torch
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def launch_shape(n, sms, force_tpb=0):
    """(threads per CTA, passes) that rollout_launch picks for the single-policy fused rollout of n envs on sms SMs."""
    grid = min(n, sms)
    per_cta = -(-n // grid)
    passes = -(-per_cta // (force_tpb or 512))
    chunk = force_tpb or -(-per_cta // passes)
    return (force_tpb or next(t for t in FORCED if chunk <= t)), passes


def cta_passes(n, grid, tpb):
    """Per CTA, as rollout_kernel slices the batch: (passes, envs of the last pass, valid rows of its last group, that
    group's width)."""
    out = []
    for b in range(grid):
        lo, hi = n * b // grid, n * (b + 1) // grid
        span = hi - lo
        passes = -(-span // tpb)
        chunk = -(-span // passes)
        last = span - (passes - 1) * chunk
        g = (last - 1) // 128
        out.append((passes, last, last - 128 * g, min(128, tpb - 128 * g)))
    return out


def shapes(sms):
    """name -> (n, forced threads per CTA or 0, SMs left free)"""
    out = {f"T{t}": (3 * 2 * t - 70, t, sms - 3) for t in FORCED}
    out["bench"] = (sms * 443, 0, 0)
    out["bench_2pass"] = (2 * sms * 443, 0, 0)
    return out


# ---------------------------------------------------------------------------------------------------- policies
def _golden_sd():
    from reinforcement_learning_rendezvous_b200.policy import load_state_dict
    return load_state_dict(os.path.join(GOLDEN, "policy.npz"))


def _policy(name):
    import torch
    from reinforcement_learning_rendezvous_b200.policy import MlpPolicy
    from reinforcement_learning_rendezvous_b200.ppo import ActorCritic
    base = _golden_sd()
    if name == "golden":
        return MlpPolicy(base)
    if name == "ppo_init":                    # the first actor PPO collects with: orthogonal init, log_std 0
        with torch.random.fork_rng(devices=[]):
            torch.manual_seed(0)
            return ActorCritic().to_mlp_policy(torch.device("cuda", torch.cuda.current_device()))
    # the seeded perturbation of test_gpu_policy_table._policies (seed 1)
    rng = np.random.default_rng(1)
    sd = {k: (v + rng.normal(0.0, 0.3 * float(v.std()) + 1e-3, v.shape)).astype(np.float32) for k, v in base.items()}
    sd["log_std"] = (base["log_std"] + 0.25).astype(np.float32)
    return MlpPolicy(sd)


def _noise_policy(b2, log_std):
    """The golden hidden layers (the full tensor-core forward still runs), action_net = 0 and an fp16-exact bias:
    the actor's output is exactly b2."""
    from reinforcement_learning_rendezvous_b200.policy import MlpPolicy
    sd = _golden_sd()
    b2, log_std = np.float32(b2), np.float32(log_std)
    assert np.array_equal(b2.astype(np.float16).astype(np.float32), b2)
    sd["action_net.weight"] = np.zeros_like(sd["action_net.weight"])
    sd["action_net.bias"] = np.broadcast_to(b2, (6,)).copy()
    sd["log_std"] = np.broadcast_to(log_std, (6,)).copy()
    return MlpPolicy(sd)


UNIT = (0.0, 0.0)
SCALED = ([0.75, -0.5, 0.0, 0.25, -1.5, 2.0], [-3.0, -1.0, 0.0, 0.5, -2.0, 1.0])


def _mean64(pol, obs):
    """The actor in fp64 (torch, on the device) on float32 observations [..., 17]."""
    w = {k: v.double() for k, v in pol.w.items()}
    h = (obs.double() @ w["w0"].T + w["b0"]).tanh()
    h = (h @ w["w1"].T + w["b1"]).tanh()
    return h @ w["w2"].T + w["b2"]


def noise_bound(log_std, z, r, a, exact):
    """|a - (mean + exp(log_std) z)| allowed for a recorded draw a = fmaf(expf(log_std), z32, mean) with an exact
    mean: the draw's own error scaled by std, plus expf within 2 ulp and the rounding of the fma -- except where
    ``exact`` (mean 0 and log_std 0: fmaf(1, z32, 0) = z32)."""
    std = np.exp(np.asarray(log_std, dtype=np.float64))
    rounding = std * 2 * EPS * np.abs(z) + 0.5 * EPS * np.abs(a)
    return std * Z_ULPS * EPS * np.maximum(r, 1.0) + np.where(exact, 0.0, rounding)


def _assert_noise(acts, b2, log_std, seed, ids, steps, what):
    """Recorded unclipped draws [K, n, 6] against b2 + exp(log_std) z_ref(seed; ids, steps).  The reference with cos
    and sin swapped must fail the same bound.  Returns the worst deviation in units of the bound, and the bound."""
    b2, log_std = np.asarray(b2, dtype=np.float64), np.asarray(log_std, dtype=np.float64)
    z, r = philox_normals_ref(seed, ids, np.asarray(steps, dtype=np.int64)[:, None])
    std = np.exp(log_std)
    bound = noise_bound(log_std, z, r, acts, (b2 == 0) & (log_std == 0))
    err = np.abs(acts - (b2 + std * z))
    assert (err <= bound).all(), (what, float((err / bound).max()), np.argwhere(err > bound)[:5].tolist())
    swapped = b2 + std * z[..., [1, 0, 3, 2, 5, 4]]
    assert (np.abs(acts - swapped) > bound).mean() > 0.99, what
    return float((err / bound).max()), bound


# ---------------------------------------------------------------------------------------------------- shapes
def _run(pol, n, stochastic, tpb, reserve):
    """Two K-step launches of n envs; returns the env, the per-step records of both and the observations the actor
    saw (env.obs at a launch's start, then the previous step's record), all on the device."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, _native as N
    env = BatchedRendezvousEnv(n, seed=SEED, t_max=T_MAX)
    env.sm_reserve = reserve
    env.reset()
    outs, seen = [], []
    try:
        if tpb:
            _tune(N.TUNE_ROLLOUT_TPB, tpb)
        for j in range(2):
            obs0 = env.obs.clone()
            o = env.rollout(K, policy=pol, stochastic=stochastic, action_seed=ASEED if stochastic else None,
                            step_base=j * K, **REC)
            outs.append(o)
            seen += [obs0[None], o["obs_steps"][:-1]]
    finally:
        _tune(N.TUNE_ROLLOUT_TPB, 0)
    rec = {k: torch.cat([o[k] for o in outs]) for k in ("rewards", "dones", "obs_steps", "actions")}
    return env, rec, torch.cat(seen)


def _check_oracle(env, rec, n, stochastic, what):
    """The env against the C oracle on the actions it received; returns the worst deviations."""
    lg = Ledger(CO.make_params(t_max=T_MAX), n, SEED)
    lg.reset()
    acts, rews = rec["actions"].cpu().numpy(), rec["rewards"].cpu().numpy()
    dones, obs = rec["dones"].cpu().numpy().astype(bool), rec["obs_steps"].cpu().numpy()
    worst = dict(reward=0.0, obs=0.0)
    for k in range(2 * K):
        a = np.clip(acts[k], -1.0, 1.0) if stochastic else acts[k]
        o_rew, o_done = lg.step(np.ascontiguousarray(a, dtype=np.float32))
        np.testing.assert_array_equal(dones[k], o_done, err_msg=f"{what} step {k}")
        worst["reward"] = max(worst["reward"], rel_err(rews[k], o_rew))
        worst["obs"] = max(worst["obs"], float(np.abs(obs[k] - lg.orc.obs).max()))
    assert worst["reward"] <= REL_TOL, (what, worst)
    assert worst["obs"] <= OBS_TOL, (what, worst)
    worst["state"] = rel_err(env.get_state().cpu().numpy(), lg.state)
    assert worst["state"] <= REL_TOL, (what, worst)
    assert (lg.episode > 1).all(), what             # every env ended an episode and restarted inside a launch
    got, want = env.read_stats(), lg.stats()
    worst["short_solves"] = short_solve_steps(got, want)
    got["rk_accepted"] = want["rk_accepted"]
    assert_stats(got, want, lg.tolerance(), what)
    return worst


def _check_actor(pol, rec, seen, n, stochastic, what):
    """The recorded actions against the fp64 actor on the observation the kernel saw; returns the worst deviation
    (deterministic: |a - clip(mean64)|; sampling: of the noise, in units of its bound)."""
    import torch
    mean = _mean64(pol, seen)
    a = rec["actions"].double()
    if not stochastic:
        dev = float((a - mean.clamp(-1.0, 1.0)).abs().max())
        assert dev <= ACT_BOUND, (what, dev)
        return dict(actor=dev)
    ls = pol.log_std.double().cpu().numpy()
    std = np.exp(ls)
    z, r = philox_normals_ref(ASEED, np.arange(n), np.arange(2 * K)[:, None])
    zm = ((a - mean) / torch.as_tensor(std, device=a.device)).cpu().numpy()
    # the mean's own error (ACT_BOUND) and the draw's, both in units of std
    bound = (ACT_BOUND + noise_bound(ls, z, r, rec["actions"].cpu().numpy(), False)) / std
    err = np.abs(zm - z)
    assert (err <= bound).all(), (what, float((err / bound).max()))
    return dict(noise=float((err / bound).max()), noise_abs=float(err.max()))


def _prefix_equal(ra, rb, m, what):
    import torch
    (ea, reca), (eb, recb) = ra, rb
    for key in ("rewards", "dones", "obs_steps", "actions"):
        assert torch.equal(reca[key][:, :m], recb[key][:, :m]), (what, key)
    assert torch.equal(ea.f64[:, :m], eb.f64[:, :m]) and torch.equal(ea.i32[:, :m], eb.i32[:, :m]), what


@pytest.mark.parametrize("stochastic", [False, True], ids=["deterministic", "sampling"])
@pytest.mark.parametrize("policy", ["golden", "ppo_init", "perturbed"])
def test_shapes_against_oracle_and_fp64_actor(policy, stochastic):
    """Every shape: env against the oracle, actor against fp64, and all shapes bit-identical on their common envs;
    the forced shapes once more at a common batch size, where the statistics must agree too."""
    sms = _sms()
    pol = _policy(policy)
    runs = {}
    for name, (n, tpb, reserve) in shapes(sms).items():
        grid = sms - reserve
        t, passes = launch_shape(n, grid, tpb)
        cta = cta_passes(n, min(n, grid), t)
        if tpb:
            assert t == tpb and grid == 3 and all(c[0] == 2 and c[2] < c[3] for c in cta), (name, cta)
        else:
            assert t == 448 and passes == (1 if name == "bench" else 2), (name, t, passes)
            assert all(c[3] == 64 and c[2] == 59 for c in cta), (name, cta)       # the half group: 59 of 64 rows
        what = (policy, stochastic, name)
        env, rec, seen = _run(pol, n, stochastic, tpb, reserve)
        worst = _check_oracle(env, rec, n, stochastic, what)
        worst.update(_check_actor(pol, rec, seen, n, stochastic, what))
        print(f"\n{what}: n={n} T={t} passes={cta[-1][0]} last group {cta[-1][2]}/{cta[-1][3]} rows; worst " +
              ", ".join(f"{k} {v:.3g}" for k, v in worst.items()))
        runs[name] = (env, rec)
    m = min(e.num_envs for e, _ in runs.values())
    ref = runs["T256"]
    for name, r in runs.items():
        _prefix_equal(ref, r, m, (policy, stochastic, name))
    # the statistics depend on the batch: the other forced shapes at the batch of T256, 3 CTAs
    st_ref = ref[0].read_stats()
    for t in FORCED[1:]:
        env, rec, _ = _run(pol, m, stochastic, t, sms - 3)
        _prefix_equal(ref, (env, rec), m, (policy, stochastic, t, "common batch"))
        st = env.read_stats()
        for k in INT_STATS:
            assert st[k] == st_ref[k], (t, k, st[k], st_ref[k])
        for k in FLOAT_STATS:
            assert abs(st[k] - st_ref[k]) <= 1e-12 * max(abs(st_ref[k]), 1.0), (t, k, st[k], st_ref[k])


# ---------------------------------------------------------------------------------------------------- noise
KEYS = {                        # (env_offset, action seed, step_base)
    "plain": (0, 5, 0),
    "offset_hi": (3 * 2 ** 31 + 5, 5, 0),
    "seed_hi": (0, 0xA5A5A5A5_00000005, 0),
    "step_across_2_32": (0, 5, 2 ** 32 - 3),
}


def _noise_run(pol, n, seed, offset, step_base, steps, env_kw=None, **rollout_kw):
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    env = BatchedRendezvousEnv(n, seed=SEED, env_offset=offset, **(env_kw or {}))
    env.reset()
    out = env.rollout(steps, policy=pol, stochastic=True, action_seed=seed, step_base=step_base, **rollout_kw,
                      record_actions=True, record_rewards=True, record_dones=True)
    return env, out


@pytest.mark.parametrize("key", list(KEYS))
@pytest.mark.parametrize("head", ["unit", "scaled"])
def test_noise_exact(head, key):
    """The recorded draws are b2 + exp(log_std) z_ref(action seed; global env id, step_base + k).  A reference keyed
    by the local env id, or without the step's high word, fails where those differ.  The scaled head leaves the Box,
    so the oracle replay also shows the env got the clipped draw."""
    offset, seed, base = KEYS[key]
    b2, ls = UNIT if head == "unit" else SCALED
    n, steps = 1000, 6
    env, out = _noise_run(_noise_policy(b2, ls), n, seed, offset, base, steps, env_kw=dict(t_max=4))
    acts = out["actions"].cpu().numpy()
    ids, ks = offset + np.arange(n), base + np.arange(steps)
    worst, bound = _assert_noise(acts, b2, ls, seed, ids, ks, (head, key))
    print(f"\nnoise {head} {key}: worst {worst:.3g} of the bound")
    std = np.exp(np.float64(ls))
    if offset:
        wrong = b2 + std * philox_normals_ref(seed, np.arange(n), ks[:, None])[0]
        assert (np.abs(acts - wrong) > bound).mean() > 0.99
    if base + steps > 2 ** 32:
        hi = ks >= 2 ** 32
        wrong = b2 + std * philox_normals_ref(seed, ids, (ks & 0xFFFFFFFF)[:, None])[0]
        assert (np.abs(acts - wrong) > bound)[hi].mean() > 0.99 and hi.sum() == 3
    if head == "scaled":
        assert (np.abs(acts) > 1).mean() > 0.05
        lg = Ledger(CO.make_params(t_max=4), n, SEED, env_offset=offset)
        lg.reset()
        rews, dones = out["rewards"].cpu().numpy(), out["dones"].cpu().numpy().astype(bool)
        for k in range(steps):
            o_rew, o_done = lg.step(np.ascontiguousarray(np.clip(acts[k], -1.0, 1.0)))
            np.testing.assert_array_equal(dones[k], o_done)
            assert rel_err(rews[k], o_rew) <= REL_TOL
        assert rel_err(env.get_state().cpu().numpy(), lg.state) <= REL_TOL
        assert_stats(env.read_stats(), lg.stats(), lg.tolerance(), (head, key))


@pytest.mark.parametrize("tpb", FORCED)
def test_noise_at_every_shape(tpb):
    """Forced CTA sizes on 3 CTAs, two passes each: the same draws, keyed by the global env id across passes,
    with high words in env id, seed and step index."""
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, _native as N
    n, offset, seed, base = 3 * 2 * tpb - 70, 3 * 2 ** 31 + 5, 0xA5A5A5A5_00000005, 2 ** 32 - 2
    pol = _noise_policy(*UNIT)
    env = BatchedRendezvousEnv(n, seed=SEED, env_offset=offset, t_max=3)
    env.sm_reserve = _sms() - 3
    env.reset()
    try:
        _tune(N.TUNE_ROLLOUT_TPB, tpb)
        out = env.rollout(5, policy=pol, stochastic=True, action_seed=seed, step_base=base, record_actions=True)
    finally:
        _tune(N.TUNE_ROLLOUT_TPB, 0)
    assert all(c[0] == 2 for c in cta_passes(n, 3, tpb))
    _assert_noise(out["actions"].cpu().numpy(), *UNIT, seed, offset + np.arange(n), base + np.arange(5), tpb)


def test_noise_launch_split_and_shards():
    """One launch of 8 steps == two of 4 (step_base 0, 4); two shard_range shards == one batch; all equal the
    reference."""
    import torch
    from reinforcement_learning_rendezvous_b200.distributed import shard_range
    pol = _noise_policy(*SCALED)
    n, seed, steps = 1000, 0xA5A5A5A5_00000005, 8
    env, one = _noise_run(pol, n, seed, 0, 0, steps, env_kw=dict(t_max=5))
    _assert_noise(one["actions"].cpu().numpy(), *SCALED, seed, np.arange(n), np.arange(steps), "one launch")
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    split = BatchedRendezvousEnv(n, seed=SEED, t_max=5)
    split.reset()
    parts = [split.rollout(4, policy=pol, stochastic=True, action_seed=seed, step_base=b, record_actions=True,
                           record_rewards=True, record_dones=True) for b in (0, 4)]
    for key in ("actions", "rewards", "dones"):
        assert torch.equal(torch.cat([p[key] for p in parts]), one[key]), key
    assert torch.equal(split.f64, env.f64) and torch.equal(split.i32, env.i32) and torch.equal(split.obs, env.obs)
    for rank in range(2):
        lo, hi = shard_range(n, 2, rank)
        e, o = _noise_run(pol, hi - lo, seed, lo, 0, steps, env_kw=dict(t_max=5))
        for key in ("actions", "rewards", "dones"):
            assert torch.equal(o[key], one[key][:, lo:hi]), (rank, key)
        assert torch.equal(e.f64[:, :hi - lo], env.f64[:, lo:hi]) and torch.equal(e.obs, env.obs[lo:hi]), rank


def test_noise_policy_table():
    """A policy table whose entries carry different b2 and log_std: every tile draws b2 + std z of its own entry,
    keyed by the global env id."""
    from reinforcement_learning_rendezvous_b200 import PolicyTable
    heads = [UNIT, SCALED, ([-0.25, 0.5, 1.0, -2.0, 0.125, 0.0], [0.25, -0.5, -1.0, 0.0, 1.5, -4.0])]
    table = PolicyTable([_noise_policy(*h) for h in heads])
    n, tiles, seed, base, offset = 128 * 5 + 37, [2, 0, 1, 2, 0, 1], 0xA5A5A5A5_00000005, 2 ** 32 - 2, 3 * 2 ** 31 + 5
    env, out = _noise_run(table, n, seed, offset, base, 5, policy_tiles=tiles)
    acts = out["actions"].cpu().numpy()
    for t, entry in enumerate(tiles):
        lo, hi = 128 * t, min(128 * (t + 1), n)
        _assert_noise(acts[:, lo:hi], *heads[entry], seed, offset + np.arange(lo, hi), base + np.arange(5), (t, entry))


# ---------------------------------------------------------------------------------------------------- PPO
def _sb3_gae(rew, val, dones, last_value, gamma, lam):
    """RolloutBuffer.compute_returns_and_advantage in fp64, with SB3's episode_starts (episode_starts[t + 1] =
    dones[t]) and no time-limit bootstrapping."""
    T = rew.shape[0]
    starts = np.concatenate([np.zeros_like(dones[:1]), dones[:-1]])
    adv = np.zeros_like(rew)
    last = np.zeros_like(last_value)
    for t in reversed(range(T)):
        if t == T - 1:
            non_terminal, next_value = 1.0 - dones[-1], last_value
        else:
            non_terminal, next_value = 1.0 - starts[t + 1], val[t + 1]
        delta = rew[t] + gamma * next_value * non_terminal - val[t]
        last = delta + gamma * lam * non_terminal * last
        adv[t] = last
    return adv, adv + val


def test_ppo_fused_collection():
    """Two PPO.collect() calls with an actor whose action_net is zero: the buffer holds b2 + std z_ref(seed + 977;
    env id, iteration * n_steps + k) -- fresh noise every iteration --, the fp64 Normal log-density, the oracle's
    observations / rewards / dones on the clipped draws, and SB3's advantages and returns."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    from reinforcement_learning_rendezvous_b200.ppo import PPO, ActorCritic, PPOConfig
    b2, ls = SCALED
    n, T, seed, env_seed = 1000, 8, 3, 14
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(0)
        ac = ActorCritic()
    with torch.no_grad():
        ac.action_net.weight.zero_()
        ac.action_net.bias.copy_(torch.tensor(b2))
        ac.log_std.copy_(torch.tensor(ls))
    env = BatchedRendezvousEnv(n, seed=env_seed, t_max=6)
    cfg = PPOConfig(fused=True, n_steps=T, n_evals=8, seed=seed)
    algo = PPO(env, cfg, policy=ac)
    lg = Ledger(CO.make_params(t_max=6), n, env_seed)
    lg.reset()
    std = np.exp(np.float64(ls))
    for it in range(2):
        prev = lg.orc.obs.copy()
        adv, ret = algo.collect()
        act = algo.buf_act.cpu().numpy()
        _assert_noise(act, b2, ls, seed + 977, np.arange(n), it * T + np.arange(T), ("ppo", it))
        logp64 = (-0.5 * ((act - np.float64(b2)) / std) ** 2 - np.log(std) - 0.5 * np.log(2 * np.pi)).sum(-1)
        logp = algo.buf_logp.cpu().numpy()
        assert (np.abs(logp - logp64) <= 1e-5 * np.maximum(np.abs(logp64), 1.0)).all(), it
        obs, rew = algo.buf_obs.cpu().numpy(), algo.buf_rew.cpu().numpy()
        done = algo.buf_done.cpu().numpy()
        for k in range(T):
            assert np.abs(obs[k] - prev).max() <= OBS_TOL, (it, k)
            o_rew, o_done = lg.step(np.ascontiguousarray(np.clip(act[k], -1.0, 1.0)))
            np.testing.assert_array_equal(done[k], o_done)
            # float32 of the fp64 reward: half an ulp, plus the kernel's REL_TOL
            assert (np.abs(rew[k] - o_rew) <= (EPS + REL_TOL) * np.maximum(np.abs(o_rew), 1.0)).all(), (it, k)
            prev = lg.orc.obs.copy()
        assert done.any(), it
        with torch.no_grad():
            _, last_value = algo.policy(algo.obs)
        a64, r64 = _sb3_gae(rew.astype(np.float64), algo.buf_val.cpu().numpy().astype(np.float64),
                            done.astype(np.float64), last_value.cpu().numpy().astype(np.float64), cfg.gamma,
                            cfg.gae_lambda)
        for got, want in ((adv, a64), (ret, r64)):
            got = got.cpu().numpy()
            assert (np.abs(got - want) <= 1e-5 * np.maximum(np.abs(want), 1.0)).all(), it
