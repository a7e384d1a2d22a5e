"""The two solver forms of the rollout kernel at the benchmark's launch.  CTAs of up to 256 threads advance the chaser's
and the target's attitude solves of an env in lock-step (rk45_iso_plane_pair); the bigger ones, and the per-step kernel
(one body per lane), run the sequential solver (rk45_iso_plane).  These tests roll the benchmark's launch -- one pass of
sms x 443 envs with auto-reset in 448-thread CTAs -- on the same tensor actions as step() driven step by step, as the
256-thread variant and as the same launch with two helper warps per CTA: the attitude columns, dones, counters and every integer statistics
slot (RK steps accepted and rejected, failures) agree bit for bit, including fast spins outside the polynomials' range,
NaN quaternions and long steps."""
import numpy as np
import pytest

from helpers import rel_err

pytestmark = pytest.mark.gpu

K = 30                                    # >= 2 x the reset refill period (12): the helper-warp variant needs it
ATT = slice(6, 20)                        # qc wc qt wt: the columns the attitude solves produce
INT_STATS = ("steps", "episodes", "length_sum", "succeeded", "collided", "end_obs", "end_time", "end_bubble",
             "end_attitude", "rk_accepted", "rk_rejected", "failures")
SUM_STATS = ("return_sum", "delta_v_sum", "delta_w_sum", "reward_sum")


def _tune(key, value):
    from reinforcement_learning_rendezvous_b200 import _native as N
    return N.lib().rdv_tune(key, int(value))


def _same_bits(a, b):
    """equal values, NaN where the other is NaN"""
    import torch
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(a[~na], b[~nb])


def _close(a, b, rtol):
    return (np.isnan(a) and np.isnan(b)) or abs(a - b) <= rtol * abs(b)


def _prepare(case, n, rng):
    """ctor kwargs and a function that edits the state after reset(): the envs it marks sit in the first half of the
    batch, so the second half runs whole warps on the polynomial lock-step path"""
    kw, marked = dict(t_max=12), np.zeros(n, dtype=bool)
    idx = np.arange(n // 2)
    if case == "fast_spins":
        # outside the polynomials' range (|w| dt > ~0.35 rad): the chaser, the target or both, at up to 3 rad/s
        sets = {"wc": idx[idx % 64 == 5], "wt": idx[idx % 64 == 9], "both": idx[idx % 64 == 13]}
        scale = rng.uniform(0.4, 3.0, n)

        def edit(s):
            for k, rows in sets.items():
                cols = [(10, 13), (17, 20)] if k == "both" else [(10, 13) if k == "wc" else (17, 20)]
                for c0, c1 in cols:
                    d = rng.normal(size=(rows.size, 3))
                    s[rows, c0:c1] = d / np.linalg.norm(d, axis=1, keepdims=True) * scale[rows, None]
            return s
        for rows in sets.values():
            marked[rows] = True
    elif case == "nan":
        # a NaN quaternion in the chaser, the target or both: one failure per env-step, then the auto-reset
        sets = {"qc": idx[idx % 97 == 3], "qt": idx[idx % 97 == 50], "both": idx[idx % 389 == 11]}

        def edit(s):
            for k, rows in sets.items():
                if k in ("qc", "both"):
                    s[rows, 6] = np.nan
                if k in ("qt", "both"):
                    s[rows, 14] = np.nan
            return s
        for rows in sets.values():
            marked[rows] = True
    elif case == "long_steps":
        # dt = 4 s: several attempts and frequent rejections per solve, so far more controller norms land in the
        # 1e-3 band around the accept threshold, where the decision is taken again in fp64
        kw = dict(dt=4, t_max=48)

        def edit(s):
            return s
    else:
        def edit(s):
            return s
    return kw, edit, marked


@pytest.mark.parametrize("case", ["default", "fast_spins", "nan", "long_steps"])
def test_benchmark_variant_follows_the_sequential_solver(case):
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, _native as N
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = sms * 443                                 # 65,536 on 148 SMs: one pass of 443 envs per CTA
    rng = np.random.default_rng(7)
    kw, edit, marked = _prepare(case, n, rng)
    envs = [BatchedRendezvousEnv(n, seed=11, **kw) for _ in range(4)]
    for env in envs:
        env.reset()
    start = edit(envs[0].get_state().cpu().numpy())
    for env in envs:
        env.set_state(start)
    g = torch.Generator(device=envs[0].device)
    g.manual_seed(3)
    acts = torch.rand((K, n, 6), dtype=torch.float64, device=envs[0].device, generator=g) * 2 - 1

    plain, step, small, helper = envs
    old = _tune(N.TUNE_ROLLOUT_HELPERS, 0)
    try:
        out = plain.rollout(K, actions=acts, record_rewards=True, record_dones=True)
        _tune(N.TUNE_ROLLOUT_HELPERS, 1)
        out_help = helper.rollout(K, actions=acts, record_rewards=True, record_dones=True)
        _tune(N.TUNE_ROLLOUT_TPB, 256)
        out_small = small.rollout(K, actions=acts, record_rewards=True, record_dones=True)
    finally:
        _tune(N.TUNE_ROLLOUT_TPB, 0)
        _tune(N.TUNE_ROLLOUT_HELPERS, old)
    rews, dones = [], []
    for k in range(K):
        _, rew, done = step.step(acts[k])
        rews.append(rew.clone())
        dones.append(done.clone())
    rews, dones = torch.stack(rews), torch.stack(dones)
    torch.cuda.synchronize()

    st_h, st_s, st_m, st_w = (e.read_stats() for e in envs)
    s_h, s_s, s_m, s_w = (e.get_state() for e in envs)
    # against the 256-thread variant and the helper-warp variant: every bit
    for o, s_o, e_o in ((out_small, s_m, small), (out_help, s_w, helper)):
        assert _same_bits(s_h, s_o)
        assert _same_bits(out["rewards"], o["rewards"]) and torch.equal(out["dones"], o["dones"])
        assert torch.equal(plain.i32[:, :n], e_o.i32[:, :n])
    # against the per-step kernel: the attitude columns, dones and counters bit for bit; its lanes order a few
    # operations of the translation and the reward differently (test_gpu_rollout.test_rollout_equals_repeated_step)
    assert _same_bits(s_h[:, ATT], s_s[:, ATT])
    assert torch.equal(out["dones"], dones)
    assert torch.equal(plain.i32[:, :n], step.i32[:, :n])
    fin = ~torch.isnan(rews)
    assert torch.equal(fin, ~torch.isnan(out["rewards"]))
    assert rel_err(out["rewards"][fin].cpu().numpy(), rews[fin].cpu().numpy()) <= 1e-12
    assert rel_err(s_h.cpu().numpy(), s_s.cpu().numpy()) <= 1e-11
    for key in INT_STATS:
        assert st_h[key] == st_s[key] == st_m[key] == st_w[key], (key, st_h[key], st_s[key], st_m[key], st_w[key])
    for key in SUM_STATS:
        assert _close(st_h[key], st_m[key], 1e-12) and _close(st_h[key], st_w[key], 1e-12), key
        assert _close(st_h[key], st_s[key], 1e-9), key

    assert st_h["episodes"] > n
    if case == "nan":
        # each marked env fails its first step once, whichever body (or both) was NaN, and is reset
        assert st_h["failures"] == int(marked.sum())
        assert bool(dones[0][torch.as_tensor(marked, device=dones.device)].all())
    else:
        assert st_h["failures"] == 0
