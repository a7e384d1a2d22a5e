"""GPU: the recurrent actor step (rdv_lstm_policy_step, tcgen05) against the fp64 reference of tests/lstm_ref.py at
three weight sets, LstmPolicy's predict contract, and the recurrent Monte-Carlo evaluator (evaluate_batch) against the
single-env facade and against the C oracle driven by the fp64 reference."""
import numpy as np
import pytest
import torch

from helpers import golden
from lstm_ref import H, actor_keys, lstm_step_ref, lstm_step_split_emulation, make_state_dict

pytestmark = pytest.mark.gpu

KINDS = ("torch", "ppo", "stress")
NMAX = 65536


def _policy(kind, seed=0):
    from reinforcement_learning_rendezvous_b200 import LstmPolicy
    sd = make_state_dict(kind, seed=seed)
    return LstmPolicy(sd), actor_keys(sd)


def _observations(n, rng):
    """Observations the env produces (golden trajectories) followed by uniform draws in the Box."""
    g = golden("traj_f32.npz")
    real = np.concatenate([g["obs0"], g["obs"].reshape(-1, 17)])
    real = real[np.isfinite(real).all(axis=1)]
    return np.concatenate([real, rng.uniform(-1, 1, (n, 17))])[:n].astype(np.float32)


def _run(pol, obs, h, c, start=None):
    """Kernel step on env-major numpy inputs -> (actions, h', c') env-major numpy."""
    d = pol.device
    act, h2, c2 = pol.forward(torch.as_tensor(obs, device=d), torch.as_tensor(np.ascontiguousarray(h.T), device=d),
                              torch.as_tensor(np.ascontiguousarray(c.T), device=d),
                              None if start is None else torch.as_tensor(start, device=d))
    return act.cpu().numpy(), h2.t().cpu().numpy(), c2.t().cpu().numpy()


def _torch_fp32(sd, obs, h, c):
    """The same step in torch fp32 (nn.LSTM, TF32 off) -- printed for comparison."""
    prev = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        lstm = torch.nn.LSTM(17, H).cuda()
        w = {k: torch.as_tensor(v, device="cuda") for k, v in sd.items()}
        with torch.no_grad():
            for k in ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"):
                getattr(lstm, k).copy_(w["lstm_actor." + k])
            out, (h2, c2) = lstm(torch.as_tensor(obs, device="cuda")[None],
                                 (torch.as_tensor(h, device="cuda")[None], torch.as_tensor(c, device="cuda")[None]))
            a = torch.tanh(out[0] @ w["mlp_extractor.policy_net.0.weight"].T + w["mlp_extractor.policy_net.0.bias"])
            a = torch.tanh(a @ w["mlp_extractor.policy_net.2.weight"].T + w["mlp_extractor.policy_net.2.bias"])
            act = torch.clamp(a @ w["action_net.weight"].T + w["action_net.bias"], -1, 1)
        return act.cpu().numpy(), h2[0].cpu().numpy(), c2[0].cpu().numpy()
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev


def _errors(got, ref, c_in):
    act, h, c = got
    ra, rh, rc = ref
    return (float(np.abs(act - ra).max()), float(np.abs(h - rh).max()),
            float((np.abs(c - rc) / np.maximum(1.0, np.abs(rc))).max()))


@pytest.mark.parametrize("kind", KINDS)
def test_step_matches_fp64_reference(kind):
    """One step from identical inputs at ragged n: actions, h' and c' (relative to max(1, |c'|)) within 1e-5 of fp64;
    every env's bits independent of n and of its position in the batch."""
    rng = np.random.default_rng(10)
    pol, sd = _policy(kind)
    obs = _observations(NMAX, rng)
    h = rng.uniform(-1, 1, (NMAX, H)).astype(np.float32)
    c = (rng.standard_normal((NMAX, H)) * (4.0 if kind == "stress" else 1.0)).astype(np.float32)
    start = rng.random(NMAX) < 0.05
    ref = lstm_step_ref(sd, obs, h, c, start)
    full = _run(pol, obs, h, c, start)
    err = _errors(full, ref, c)
    t32 = _errors(_torch_fp32(sd, obs, np.where(start[:, None], 0, h), np.where(start[:, None], 0, c)), ref, c)
    print(f"{kind}: kernel |da| {err[0]:.2e} |dh| {err[1]:.2e} |dc|rel {err[2]:.2e};  "
          f"torch fp32 {t32[0]:.2e} {t32[1]:.2e} {t32[2]:.2e}")
    assert max(err) <= 1e-5, err
    for n in (1, 127, 129, 1000, NMAX - 77):             # NMAX - 77: CTAs loop over pairs, the last one ragged
        part = _run(pol, obs[:n], h[:n], c[:n], start[:n])
        for a, b in zip(part, full):
            assert np.array_equal(a, b[:n]), n
    perm = rng.permutation(1000)
    shuffled = _run(pol, obs[perm], h[perm], c[perm], start[perm])
    for a, b in zip(shuffled, full):
        assert np.array_equal(a, b[perm])


# Known limitation, not a loosened bound: at the stressed set the kernel's free run drifts to ~7e-4, where torch fp32
# (TF32 off) stays at 7.7e-5 and the numpy emulation of the kernel's split arithmetic with IEEE float32 accumulation at
# 1.0e-4.  The split itself is therefore not the cause; the tensor core's accumulation of the three products is (its
# one-step c' error is ~3x torch's, and this recurrence amplifies per-step error ~450x over 60 steps).  Removing it
# needs the K-sum moved out of the tensor core; until then this case is expected to fail.
@pytest.mark.parametrize("kind", ["torch", "ppo", pytest.param("stress", marks=pytest.mark.xfail(
    strict=True, reason="tensor-core accumulation of the split products: ~7e-4 where torch fp32 drifts 7.7e-5"))])
def test_free_run_stays_at_fp32_accuracy(kind):
    """60 recurrent steps with teacher-forced observations (episode starts mixed in): the kernel's own h, c feed its
    next step; h, c and actions stay within 1e-4 of the fp64 reference run.  The stressed set is expansive (an fp64 run
    nudged by 1e-6 after its first step ends ~1.6e-4 away), so there the bound asks for better than fp32 rounding at
    every step; torch fp32 (TF32 off) and the numpy emulation of the kernel's arithmetic are printed beside it."""
    rng = np.random.default_rng(11)
    pol, sd = _policy(kind, seed=5)
    n, d = 1000, pol.device
    h_ref = c_ref = np.zeros((n, H))
    h, c = pol.initial_state(n)
    h32 = c32 = he = ce = np.zeros((n, H), np.float32)
    worst, worst32, worst_e = np.zeros(3), np.zeros(3), np.zeros(3)
    for t in range(60):
        obs = _observations(n, rng) if t == 0 else rng.uniform(-1, 1, (n, 17)).astype(np.float32)
        start = np.ones(n, dtype=bool) if t == 0 else rng.random(n) < 0.02
        act, h, c = pol.forward(torch.as_tensor(obs, device=d), h, c, torch.as_tensor(start, device=d))
        ref = lstm_step_ref(sd, obs, h_ref, c_ref, start)
        _, h_ref, c_ref = ref
        keep = ~start[:, None]
        _, h32, c32 = _torch_fp32(sd, obs, np.where(keep, h32, 0), np.where(keep, c32, 0))
        he, ce = lstm_step_split_emulation(sd, obs, he, ce, start)
        worst = np.maximum(worst, _errors((act.cpu().numpy(), h.t().cpu().numpy(), c.t().cpu().numpy()), ref, c_ref))
        worst32 = np.maximum(worst32, _errors((ref[0], h32, c32), ref, c_ref))
        worst_e = np.maximum(worst_e, _errors((ref[0], he, ce), ref, c_ref))
    print(f"{kind}: worst over 60 steps: kernel |da| {worst[0]:.2e} |dh| {worst[1]:.2e} |dc|rel {worst[2]:.2e}; "
          f"torch fp32 |dh| {worst32[1]:.2e} |dc|rel {worst32[2]:.2e}; emulated split arithmetic |dh| "
          f"{worst_e[1]:.2e} |dc|rel {worst_e[2]:.2e}; max |c| {np.abs(c_ref).max():.2f}")
    assert worst.max() <= 1e-4, worst


def test_episode_start_and_predict_contract():
    rng = np.random.default_rng(12)
    pol, sd = _policy("torch", seed=6)
    n = 300
    obs = _observations(n, rng)
    garbage_h = rng.uniform(-1e30, 1e30, (n, H)).astype(np.float32)
    garbage_c = rng.uniform(-1e30, 1e30, (n, H)).astype(np.float32)
    for g in (garbage_h, garbage_c):                      # non-finite garbage too: the select clears it, 0 * x would not
        g[0::3, 0::5], g[1::3, 1::7], g[2::3, 2::11] = np.nan, np.inf, -np.inf
    zeros = np.zeros((n, H), np.float32)
    fresh = _run(pol, obs, zeros, zeros)
    reset = _run(pol, obs, garbage_h, garbage_c, np.ones(n, dtype=bool))
    for a, b in zip(reset, fresh):
        assert np.array_equal(a, b)                       # selected to zero exactly, whatever the old state
    mixed = rng.random(n) < 0.5
    h = rng.uniform(-1, 1, (n, H)).astype(np.float32)
    c = rng.standard_normal((n, H)).astype(np.float32)
    part = _run(pol, obs, np.where(mixed[:, None], garbage_h, h), np.where(mixed[:, None], garbage_c, c), mixed)
    free = _run(pol, obs, h, c)
    for a, b, f in zip(part, fresh, free):
        assert np.array_equal(a[mixed], b[mixed]) and np.array_equal(a[~mixed], f[~mixed])

    # predict: numpy in / out, sb3_contrib's shapes and defaults, equal to forward
    act, (hp, cp) = pol.predict(obs)
    assert act.shape == (n, 6) and act.dtype == np.float32
    assert hp.shape == cp.shape == (1, n, H) and hp.dtype == cp.dtype == np.float32
    assert np.array_equal(act, fresh[0]) and np.array_equal(hp[0], fresh[1]) and np.array_equal(cp[0], fresh[2])
    act2, (h2, c2) = pol.predict(obs, state=(hp, cp), episode_start=np.zeros(n, dtype=bool))
    nxt = _run(pol, obs, fresh[1], fresh[2])
    assert np.array_equal(act2, nxt[0]) and np.array_equal(h2[0], nxt[1]) and np.array_equal(c2[0], nxt[2])
    act3, _ = pol.predict(obs, state=(hp, cp), episode_start=np.ones(n, dtype=bool))
    assert np.array_equal(act3, act)
    one, (h1, c1) = pol.predict(obs[7], state=(hp[:, 7:8], cp[:, 7:8]), episode_start=np.zeros(1, dtype=bool))
    assert one.shape == (6,) and h1.shape == (1, 1, H) and np.array_equal(one, nxt[0][7])
    with pytest.raises(NotImplementedError):
        pol.predict(obs, deterministic=False)

    # forward on column slices of wider buffers: outputs keep the leading dimension, same bits
    d = pol.device
    wide_h = torch.zeros((H, 2 * n), device=d)
    wide_c = torch.zeros((H, 2 * n), device=d)
    wide_h[:, :n] = torch.as_tensor(h.T.copy(), device=d)
    wide_c[:, :n] = torch.as_tensor(c.T.copy(), device=d)
    obs_d = torch.as_tensor(obs, device=d)
    act_w, h_w, c_w = pol.forward(obs_d, wide_h[:, :n], wide_c[:, :n])
    assert h_w.stride(0) == 2 * n and tuple(h_w.shape) == (H, n)
    assert np.array_equal(act_w.cpu().numpy(), free[0]) and np.array_equal(h_w.t().cpu().numpy(), free[1])
    assert np.array_equal(c_w.t().cpu().numpy(), free[2])
    h_d, c_d = (torch.as_tensor(x.T.copy(), device=d) for x in (h, c))
    act_o, h_o, c_o = torch.empty((n, 6), device=d), torch.empty((H, n), device=d), torch.empty((H, n), device=d)
    with pytest.raises(ValueError, match="share memory"):
        pol.forward(obs_d, h_d, c_d, out=(act_o, h_d, c_o))                  # h' aliasing h
    with pytest.raises(ValueError):
        pol.forward(obs_d, h_d, c_d, out=(act_o, h_o.double(), c_o))          # wrong dtype
    with pytest.raises(ValueError):
        pol.forward(obs_d, h_d, c_d, out=(act_o[:-1], h_o, c_o))              # wrong shape


def test_fused_rollout_and_policy_table_reject_lstm():
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, PolicyTable
    pol, _ = _policy("torch")
    env = BatchedRendezvousEnv(256, auto_reset=False)
    env.reset()
    with pytest.raises(TypeError):
        env.rollout(1, policy=pol)
    with pytest.raises(TypeError):
        PolicyTable([pol])


def _ics(m):
    ic = np.array(golden("mc.npz")["ic_raw"][:m], dtype=np.float64)
    ic[:, 6:10] /= np.linalg.norm(ic[:, 6:10], axis=1, keepdims=True)
    ic[:, 13:17] /= np.linalg.norm(ic[:, 13:17], axis=1, keepdims=True)
    return ic


DISCRETE = ("num_collisions", "collided", "num_successes", "succeeded")
CONTINUOUS = ("total_reward", "total_delta_v", "min_dist_from_koz", "pos_error", "vel_error", "att_error", "rot_error")


def test_evaluate_batch_equals_single_env_facade():
    """evaluate_batch(lstm) against monte_carlo.evaluate(lstm, make_env(...)) (predict with state, rdv_step) on the
    first 100 published initial conditions."""
    from reinforcement_learning_rendezvous_b200 import evaluate, evaluate_batch, make_env
    pol, _ = _policy("torch", seed=7)
    m = 100
    ic = _ics(m)
    dev = evaluate_batch(pol, golden("mc.npz")["ic_raw"][:m])
    env = make_env(None, quiet=True, config=dict(dt=1, t_max=60), stochastic=False)
    host = {k: [] for k in dev}
    for s in ic:
        init = dict(rc=s[0:3].copy(), vc=s[3:6].copy(), qc=s[6:10].copy(), wc=s[10:13].copy(), qt=s[13:17].copy(),
                    wt=s[17:20].copy())
        for k, v in evaluate(pol, env, init).items():
            host[k].append(v)
    host = {k: np.asarray(v, dtype=np.float64) for k, v in host.items()}
    same = np.asarray(dev["ep_len"], dtype=float) == host["ep_len"]
    assert same.sum() >= m - 1, int((~same).sum())
    for k in DISCRETE:
        assert np.array_equal(np.asarray(dev[k])[same], host[k][same]), k
    for k in CONTINUOUS:
        a, b = np.asarray(dev[k])[same], host[k][same]
        rel = np.abs(a - b) / np.maximum(np.abs(b), 1e-2)
        assert np.median(rel) <= 1e-9 and np.quantile(rel, 0.99) <= 1e-6, (k, float(np.median(rel)), float(rel.max()))


def _oracle_closed_loop(sd, ic, config):
    """The fp64 reference policy drives the C oracle (float32-rounded actions) by monte_carlo.evaluate's rules."""
    from oracle import c_oracle as CO
    from reinforcement_learning_rendezvous_b200.environment_utils import config_to_kwargs
    from reinforcement_learning_rendezvous_b200.monte_carlo import _terminal_errors_batch
    m = ic.shape[0]
    orc = CO.COracleBatch(CO.make_params(**config_to_kwargs(config, stochastic=False)), m)
    p = orc.p
    orc.set_state(ic)
    obs = orc.observe()
    h = c = np.zeros((m, H))
    start = np.ones(m, dtype=bool)
    err, col, suc, koz = orc.errors()
    errs = [err.copy()]
    alive = np.ones(m, dtype=bool)
    length, n_col, n_suc = np.zeros(m, np.int64), col.astype(np.int64), suc.astype(np.int64)
    min_koz, total_reward, tdv = koz.copy(), np.zeros(m), np.zeros(m)
    while alive.any():
        act, h, c = lstm_step_ref(sd, obs, h, c, start)
        obs, rew, done = orc.step(act.astype(np.float32), threads=4)
        obs, done = obs.copy(), done.astype(bool)
        err, col, suc, koz = orc.errors()
        errs.append(np.where(alive[:, None], err, np.nan))
        n_col += col.astype(bool) & alive
        n_suc += suc.astype(bool) & alive
        min_koz = np.where(alive & (koz < min_koz), koz, min_koz)
        total_reward += np.where(alive, rew, 0.0)
        length += alive
        tdv = np.where(alive & done, orc.aux[:, 0], tdv)
        alive &= ~done
        start = done
    te = _terminal_errors_batch(np.array(errs), length,
                                (p.max_rd_error, p.max_vd_error, p.max_qd_error, p.max_wd_error))
    return dict(ep_len=np.round(length * p.dt, 3), num_collisions=n_col, collided=(n_col > 0).astype(np.int64),
                total_reward=total_reward, total_delta_v=tdv, num_successes=n_suc,
                succeeded=(n_suc > 0).astype(np.int64), min_dist_from_koz=min_koz, pos_error=te[:, 0],
                vel_error=te[:, 1], att_error=te[:, 2], rot_error=te[:, 3])


@pytest.mark.parametrize("kind", ("torch", "ppo"))
def test_evaluate_batch_closed_loop_against_oracle(kind):
    """All 1000 published initial conditions: the device evaluation against the C oracle driven by the fp64
    reference -- at most 5 episodes differing in any discrete column, and on rows of equal length the continuous
    columns with a median relative error below 1e-5."""
    from reinforcement_learning_rendezvous_b200 import evaluate_batch
    pol, sd = _policy(kind, seed=8)
    raw = golden("mc.npz")["ic_raw"]
    out = evaluate_batch(pol, raw, return_raw=True)
    ref = _oracle_closed_loop(sd, _ics(1000), dict(dt=1, t_max=60))
    flips = {k: int((np.asarray(out[k], dtype=float) != np.asarray(ref[k], dtype=float)).sum())
             for k in ("ep_len",) + DISCRETE}
    print(f"{kind}: episodes differing from the oracle closed loop {flips}; successes {int(out['succeeded'].sum())}, "
          f"collisions {int(out['collided'].sum())}, mean length {out['ep_len'].mean():.1f} s")
    assert max(flips.values()) <= 5, flips
    same = np.asarray(out["ep_len"], dtype=float) == ref["ep_len"]
    for k in CONTINUOUS:
        rel = np.abs(out[k][same] - ref[k][same]) / np.maximum(np.abs(ref[k][same]), 1e-3)
        assert np.median(rel) < 1e-5, (k, float(np.median(rel)))
    raw = out["raw"]
    assert raw.shape == (1000, 16)
    from reinforcement_learning_rendezvous_b200 import _native as N
    unreduced = [N.MC_LEVEL, N.MC_TAIL_COUNT, N.MC_END_REASON]                  # documented: NaN for an LstmPolicy
    assert np.isnan(raw[:, unreduced]).all()
    assert np.isfinite(np.delete(raw, unreduced, axis=1)).all()
    assert np.array_equal(raw[:, N.MC_EP_LEN], out["ep_len"]) and np.array_equal(raw[:, N.MC_POS_ERR], out["pos_error"])


def test_evaluate_batch_trajectories():
    """trajectories=True: the MLP path's fields, frozen after the first done, and consistent with the columns."""
    from reinforcement_learning_rendezvous_b200 import evaluate_batch, MlpPolicy
    from reinforcement_learning_rendezvous_b200.monte_carlo import _terminal_errors_batch
    from helpers import GOLDEN
    import os
    pol, _ = _policy("torch", seed=9)
    raw = golden("mc.npz")["ic_raw"][:200]
    out = evaluate_batch(pol, raw, trajectories=True)
    plain = evaluate_batch(pol, raw)
    mlp = evaluate_batch(MlpPolicy.load(os.path.join(GOLDEN, "policy.npz")), raw[:4], trajectories=True)
    tr = out["trajectory"]
    assert set(tr) == set(mlp["trajectory"])
    for k, v in tr.items():
        assert v.shape[1:] == mlp["trajectory"][k].shape[1:] and v.shape[0] == 200, k
    for k in plain:
        assert np.array_equal(out[k], plain[k], equal_nan=True), k
    length = tr["length"]
    assert np.array_equal(np.round(length * 1.0, 3), out["ep_len"])
    idx = np.arange(200)
    assert np.array_equal(tr["total_reward"][idx, length], out["total_reward"])
    assert np.array_equal(tr["total_delta_v"][idx, length], out["total_delta_v"])
    assert np.array_equal(tr["t"][:, -1], out["ep_len"])                     # frozen after the first done
    valid = np.arange(tr["t"].shape[1])[None, :] <= length[:, None]
    assert np.array_equal(np.where(valid, tr["dist_from_koz"], np.inf).min(axis=1), out["min_dist_from_koz"])
    assert np.array_equal((tr["collision"] & valid).sum(axis=1), out["num_collisions"])
    from reinforcement_learning_rendezvous_b200 import make_params
    p = make_params(dt=1, t_max=60)
    te = _terminal_errors_batch(tr["errors"].transpose(1, 0, 2), length,
                                (p.max_rd_error, p.max_vd_error, p.max_qd_error, p.max_wd_error))
    assert np.array_equal(te[:, 0], out["pos_error"]) and np.array_equal(te[:, 3], out["rot_error"])
