"""GPU: the statistics slots (RDV_S_*), the episode records (RDV_EP_*, RdvFinishedRow) and the VecEnv's episode
infos of every kernel path against an independent reference -- tests/ledger.py, which follows the C oracle and
accumulates what each slot should hold by the rules next to the RDV_S_* enum -- and against the launch's own
per-step records.  Integer slots must be exact; fp64 slots agree to REL_TOL of sum(max(|term|, 1)); sums the
kernel forms from its own records agree to 1e-12 (the CTAs add with atomics in no fixed order)."""
import math
import os

import numpy as np
import pytest

from helpers import GOLDEN, REL_TOL, rel_err
from ledger import INT_STATS, Ledger, assert_stats, merge_stats, short_solve_steps

from oracle import c_oracle as CO

pytestmark = pytest.mark.gpu

GENERAL = dict(inertia=np.array([[12.0, 0.8, -0.4], [0.8, 17.0, 0.5], [-0.4, 0.5, 23.0]]),
               inertia_target=np.array([[28.0, -1.5, 0.7], [-1.5, 21.0, 0.3], [0.7, 0.3, 15.0]]),
               chaser_torque=[0.01, -0.02, 0.015])


def _oracle_kw(kw):
    return {k: v for k, v in kw.items() if k != "integrator"}


def assert_own_records(stats, rewards, dones, what=""):
    """reward_sum and episodes against the launch's own per-step records."""
    r = np.asarray(rewards, dtype=np.float64).ravel()
    s = math.fsum(r.tolist())
    if math.isnan(s):
        assert math.isnan(stats["reward_sum"]), what
    else:
        assert abs(stats["reward_sum"] - s) <= 1e-12 * max(math.fsum(np.abs(r).tolist()), 1.0), (what, stats, s)
    assert stats["episodes"] == int(np.asarray(dones).astype(np.int64).sum()), what


def _tune(key, value):
    from reinforcement_learning_rendezvous_b200 import _native as N
    return N.lib().rdv_tune(key, int(value))


def _policy():
    from reinforcement_learning_rendezvous_b200 import MlpPolicy
    return MlpPolicy.load(os.path.join(GOLDEN, "policy.npz"))


def _step_case(n, steps, act_dtype, auto_reset, seed=21, offset=77, **kw):
    """rdv_step with random actions, followed by the ledger; every finished episode's record checked as it ends."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    rng = np.random.default_rng(seed)
    env = BatchedRendezvousEnv(n, seed=seed, env_offset=offset, auto_reset=auto_reset, **kw)
    env.reset()
    lg = Ledger(CO.make_params(**_oracle_kw(kw)), n, seed, env_offset=offset, auto_reset=auto_reset)
    lg.reset()
    for k in range(steps):
        a = rng.uniform(-1, 1, (n, 6)).astype(act_dtype)
        _, rew, done = env.step(torch.as_tensor(a, device=env.device))
        nrec = len(lg.records)
        o_rew, o_done = lg.step(a)
        np.testing.assert_array_equal(done.cpu().numpy().astype(bool), o_done)
        assert rel_err(rew.cpu().numpy(), o_rew) <= REL_TOL
        rec, reason = env.episode_record.cpu().numpy(), env.end_reason.cpu().numpy()
        for r in lg.records[nrec:]:
            i = r["env"]
            assert reason[i] == r["end_reason"]
            assert rec[i, 1] == r["length"] and rec[i, 2] == r["success"] and rec[i, 3] == r["collided"]
            assert rel_err(rec[i, [0, 4, 5]], [r["ret"], r["delta_v"], r["delta_w"]]) <= REL_TOL, (k, i)
    want, tol = lg.stats(), lg.tolerance()
    assert_stats(env.read_stats(), want, tol, (act_dtype, auto_reset))
    return env, lg


@pytest.mark.parametrize("act_dtype", ["float64", "float32"])
def test_step_auto_reset(act_dtype):
    """S1 / S2: rdv_step, auto-reset, short episodes; float32 actions follow NumPy-2 rules for delta_v."""
    env, lg = _step_case(1000, 20, act_dtype, True, t_max=8)
    assert lg.stats()["episodes"] > 1000 and (lg.episode > 2).any()


def test_step_past_the_end_without_auto_reset():
    """S3: an env that keeps stepping after its end counts again at every step."""
    env, lg = _step_case(700, 10, "float64", False, t_max=5)
    st = lg.stats()
    assert st["episodes"] > 700 * 5 and st["length_sum"] > 0


def test_step_general_inertia_held_torque():
    """S4: the general-inertia step kernel, a non-diagonal target inertia and a held chaser torque."""
    env, lg = _step_case(500, 14, "float64", True, t_max=6, **GENERAL)
    assert lg.stats()["rk_rejected"] >= 0 and lg.stats()["episodes"] > 500


def test_vecenv_mixed_kernel_families():
    """S5: a VecEnv whose param_batches mix isotropic and general-inertia bodies: two rdv_step launches per step
    appending to one block of finished rows (fin_append, fin_env_base) and one statistics vector."""
    from reinforcement_learning_rendezvous_b200 import RendezvousVecEnv
    n, seed, steps = 677, 5, 16
    groups = [(256, dict(t_max=6)), (n - 256, dict(t_max=6, **GENERAL))]
    vec = RendezvousVecEnv(n, seed=seed, rich_infos=True, gc_freeze=False, param_batches=groups)
    assert len(vec.env._units) == 2                     # really two launches per step
    vec.reset()
    ledgers, lo = [], 0
    for cnt, kw in groups:
        lg = Ledger(CO.make_params(**kw), cnt, seed, env_offset=lo)
        lg.reset()
        ledgers.append((lo, lg))
        lo += cnt
    rng = np.random.default_rng(2)
    finished = 0
    for k in range(steps):
        a = rng.uniform(-1, 1, (n, 6)).astype(np.float32)
        want = {}
        for base, lg in ledgers:
            nrec = len(lg.records)
            lg.step(a[base:base + lg.n])
            for r in lg.records[nrec:]:
                want[base + r["env"]] = r
        if k % 2:
            obs, rew, done, fin = vec.step_arrays(a)
            assert sorted(want) == fin["index"].tolist()
            for j, i in enumerate(fin["index"]):
                r = want[int(i)]
                assert fin["end_reason"][j] == r["end_reason"] and fin["episode_length"][j] == r["length"]
                assert fin["is_success"][j] == (r["success"] > 0) and fin["collided"][j] == bool(r["collided"])
                assert rel_err([fin["episode_return"][j], fin["total_delta_v"][j], fin["total_delta_w"][j]],
                               [r["ret"], r["delta_v"], r["delta_w"]]) <= REL_TOL
                t_obs = fin["terminal_observation"][j]
                assert (np.abs(t_obs - r["terminal_obs"]) <= np.spacing(np.abs(r["terminal_obs"]))).all(), (k, i)
        else:
            obs, rew, done, infos = vec.step(a)
            assert sorted(want) == np.flatnonzero(done).tolist()
            for i, r in want.items():
                ep = infos[i]["episode"]
                assert ep["l"] == r["length"]
                assert abs(ep["r"] - r["ret"]) <= 0.5e-6 + REL_TOL * max(1.0, abs(r["ret"])), (ep, r["ret"])
                assert infos[i]["is_success"] == (r["success"] > 0) and infos[i]["collided"] == bool(r["collided"])
                t_obs = infos[i]["terminal_observation"]
                assert (np.abs(t_obs - r["terminal_obs"]) <= np.spacing(np.abs(r["terminal_obs"]))).all(), (k, i)
        assert np.array_equal(np.asarray(rew), vec.env.reward.cpu().numpy().astype(np.float32))
        finished += len(want)
    assert finished > n
    st, tol = merge_stats([lg for _, lg in ledgers])
    assert_stats(vec.read_stats(), st, tol, "vecenv")


def _philox_ledger(n, K, seed, action_seed, offset=0, auto_reset=True, stop=False, step_base=0, **kw):
    lg = Ledger(CO.make_params(**_oracle_kw(kw)), n, seed, env_offset=offset, auto_reset=auto_reset,
                stop_at_first_done=stop)
    lg.reset()
    rews, dones = [], []
    for k in range(K):
        r, d = lg.step(CO.philox_actions(action_seed, lg.ids, step_base + k))
        rews.append(r)
        dones.append(d)
    return lg, np.array(rews), np.array(dones)


def test_rollout_launch_shapes_against_ledger():
    """R1: rollout with Philox actions at every CTA size -- the lock-step pair solver (256), the sequential solver
    with the statistics parked in tensor memory (384, 448, 512), with and without helper warps.  At 256 the
    trajectory record's rows at each done must also add up to the slots."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, _native as N
    # K - 12 and K - 24 are odd: a statistic parked under the wrong word during the solves would swap places an odd
    # number of times after the time-limit ends at steps 12 and 24, and land in the wrong slot
    n, K, seed, aseed = 1500, 31, 4, 9
    lg, o_rew, o_done = _philox_ledger(n, K, seed, aseed, t_max=12)
    want, tol = lg.stats(), lg.tolerance()
    assert want["episodes"] > n
    try:
        for tpb, helpers in ((256, 1), (384, 1), (448, 0), (448, 1), (512, 1)):
            _tune(N.TUNE_ROLLOUT_TPB, tpb)
            _tune(N.TUNE_ROLLOUT_HELPERS, helpers)
            env = BatchedRendezvousEnv(n, seed=seed, t_max=12)
            env.reset()
            out = env.rollout(K, action_seed=aseed, record_rewards=True, record_dones=True,
                              record_trajectory=tpb == 256)
            st = env.read_stats()
            what = (tpb, helpers)
            assert_stats(st, want, tol, what)
            rew, don = out["rewards"].cpu().numpy(), out["dones"].cpu().numpy()
            assert_own_records(st, rew, don, what)
            np.testing.assert_array_equal(don.astype(bool), o_done)
            if tpb == 256:
                tr = out["trajectory"].cpu().numpy()                        # [K, TR_NCOL, n]
                kk, ii = np.nonzero(don)
                rows = tr[kk, :, ii]                                         # [episodes, TR_NCOL]
                assert rows.shape[0] == st["episodes"]
                assert st["length_sum"] == rows[:, N.TR_I_STEP].sum()
                assert st["succeeded"] == (rows[:, N.TR_I_SUCCESS] > 0).sum()
                assert st["collided"] == rows[:, N.TR_I_COLLIDED].sum()
                for key, col in (("return_sum", N.EPRET), ("delta_v_sum", N.TDV), ("delta_w_sum", N.TDW)):
                    s = math.fsum(rows[:, col].tolist())
                    assert abs(st[key] - s) <= 1e-12 * max(math.fsum(np.abs(rows[:, col]).tolist()), 1.0), key
    finally:
        _tune(N.TUNE_ROLLOUT_TPB, 0)
        _tune(N.TUNE_ROLLOUT_HELPERS, 1)


def test_benchmark_shape_rk_steps():
    """R2: the benchmark's own launch (65,536 envs, automatic shape, two 20-step launches with the reset rows
    carried): every slot, including the rk_accepted that the benchmark turns into mean RK45 steps per solve."""
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    n, seed, aseed = 65536, 12, 3
    env = BatchedRendezvousEnv(n, seed=seed)
    env.reset()
    env.rollout(20, action_seed=aseed, step_base=0)
    env.rollout(20, action_seed=aseed, step_base=20)
    lg, _, _ = _philox_ledger(n, 40, seed, aseed)
    want, got = lg.stats(), env.read_stats()
    # SciPy's extra short third step (ledger.short_solve_steps; measured on this batch: 4 of 5.2 M solves)
    d_acc = short_solve_steps(got, want)
    got["rk_accepted"] = want["rk_accepted"]
    assert_stats(got, want, lg.tolerance(), "bench shape")
    print(f"\nmean RK45 steps per solve at the benchmark shape: {want['rk_accepted'] / (2 * want['steps']):.6f} "
          f"(oracle), {(want['rk_accepted'] - d_acc) / (2 * want['steps']):.6f} (kernel)")


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_rollout_tensor_actions(dtype):
    """R3: rollout with tensor actions."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    n, K, seed = 700, 25, 8
    a = np.random.default_rng(3).uniform(-1, 1, (K, n, 6)).astype(dtype)
    env = BatchedRendezvousEnv(n, seed=seed, t_max=10)
    env.reset()
    out = env.rollout(K, actions=torch.as_tensor(a, device=env.device), record_rewards=True, record_dones=True)
    lg = Ledger(CO.make_params(t_max=10), n, seed)
    lg.reset()
    for k in range(K):
        lg.step(a[k])
    st = env.read_stats()
    assert_stats(st, lg.stats(), lg.tolerance(), dtype)
    assert_own_records(st, out["rewards"].cpu().numpy(), out["dones"].cpu().numpy(), dtype)


def _policy_case(env, lg, out, K, stochastic, extra_failures=0):
    acts = out["actions"].cpu().numpy()
    for k in range(K):
        a = np.clip(acts[k], -1.0, 1.0) if stochastic else acts[k]
        lg.step(np.ascontiguousarray(a, dtype=np.float32))
    want = lg.stats()
    want["failures"] += extra_failures
    st = env.read_stats()
    assert_stats(st, want, lg.tolerance(), stochastic)
    assert_own_records(st, out["rewards"].cpu().numpy(), out["dones"].cpu().numpy(), stochastic)


@pytest.mark.parametrize("stochastic", [False, True])
def test_fused_policy(stochastic):
    """R4: the actor inside the launch; the ledger replays the recorded actions (sampling: clipped, as the env
    received them)."""
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    n, K, seed = 600, 20, 6
    env = BatchedRendezvousEnv(n, seed=seed, t_max=10)
    env.reset()
    out = env.rollout(K, policy=_policy(), stochastic=stochastic, action_seed=4 if stochastic else None,
                      record_rewards=True, record_dones=True, record_actions=True)
    lg = Ledger(CO.make_params(t_max=10), n, seed)
    lg.reset()
    _policy_case(env, lg, out, K, stochastic)


def test_policy_table_with_a_tile_it_cannot_run(monkeypatch):
    """R5: three entries, a non-monotone tile map and one index outside the table: that tile takes zero actions and
    counts one failure per env-step."""
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, PolicyTable, batched_env
    from reinforcement_learning_rendezvous_b200.policy import MlpPolicy, load_state_dict
    base = load_state_dict(os.path.join(GOLDEN, "policy.npz"))
    pols = [MlpPolicy(base)]
    for s in (1, 2):
        rng = np.random.default_rng(s)
        pols.append(MlpPolicy({k: (v + rng.normal(0.0, 0.3 * float(v.std()) + 1e-3, v.shape)).astype(np.float32)
                               for k, v in base.items()}))
    n, K, seed = 128 * 4 + 50, 14, 7
    tiles = [2, 0, 5, 1, 0]                             # tile 2 (envs 256 .. 383) names no entry
    env = BatchedRendezvousEnv(n, seed=seed, t_max=8)
    env.reset()
    with monkeypatch.context() as m:
        m.setattr(batched_env, "policy_tile_indices", lambda t, n_, c: np.asarray(t, dtype=np.int32))
        out = env.rollout(K, policy=PolicyTable(pols), policy_tiles=tiles, record_rewards=True, record_dones=True,
                          record_actions=True)
    assert not out["actions"][:, 256:384].any()
    lg = Ledger(CO.make_params(t_max=8), n, seed)
    lg.reset()
    _policy_case(env, lg, out, K, False, extra_failures=K * 128)


def test_parameter_table():
    """R6: three parameter sets in one launch (one with dt = 0.5), one ledger per set."""
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    batches = [(64, dict(h=400e3, t_max=10)), (128, dict(koz_radius=10.0, corridor_half_angle=float(np.radians(15)),
                                                        t_max=10)), (301, dict(dt=0.5, t_max=6))]
    n, K, seed, aseed = sum(c for c, _ in batches), 24, 9, 2
    env = BatchedRendezvousEnv(n, seed=seed, param_batches=batches)
    assert env.param_table is not None
    env.reset()
    out = env.rollout(K, action_seed=aseed, record_rewards=True, record_dones=True)
    ledgers, lo = [], 0
    for cnt, kw in batches:
        ledgers.append(_philox_ledger(cnt, K, seed, aseed, offset=lo, **kw)[0])
        lo += cnt
    want, tol = merge_stats(ledgers)
    st = env.read_stats()
    assert_stats(st, want, tol, "param table")
    assert_own_records(st, out["rewards"].cpu().numpy(), out["dones"].cpu().numpy())


@pytest.mark.parametrize("source", ["philox", "policy"])
def test_evaluator_mode(source):
    """R7: an env stops at its first done: steps are counted up to and including it, and equal sum(MC_EP_LEN)."""
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, _native as N
    n, K, seed = 900, 40, 10
    env = BatchedRendezvousEnv(n, seed=seed, auto_reset=False, t_max=30)
    env.reset()
    kw = dict(action_seed=5) if source == "philox" else dict(policy=_policy(), record_actions=True)
    out = env.rollout(K, monte_carlo=True, record_rewards=True, record_dones=True, **kw)
    lg = Ledger(CO.make_params(t_max=30), n, seed, auto_reset=False, stop_at_first_done=True)
    lg.reset()
    acts = out["actions"].cpu().numpy() if source == "policy" else None
    for k in range(K):
        lg.step(CO.philox_actions(5, lg.ids, k) if acts is None else np.ascontiguousarray(acts[k]))
    st = env.read_stats()
    assert_stats(st, lg.stats(), lg.tolerance(), source)
    assert_own_records(st, out["rewards"].cpu().numpy(), out["dones"].cpu().numpy(), source)
    mc = out["mc"].cpu().numpy()
    assert st["steps"] == mc[:, N.MC_EP_LEN].sum() == lg.steps_taken.sum()
    assert not lg.alive.all() and st["episodes"] == n - lg.alive.sum()


def test_general_inertia_rollout_with_torque():
    """R8: the general-inertia rollout with a held torque and auto-reset: state and rewards against the oracle,
    and every slot against the ledger."""
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    n, K, seed, aseed = 500, 24, 11, 6
    env = BatchedRendezvousEnv(n, seed=seed, t_max=8, **GENERAL)
    env.reset()
    out = env.rollout(K, action_seed=aseed, record_rewards=True, record_dones=True)
    lg, o_rew, o_done = _philox_ledger(n, K, seed, aseed, t_max=8, **GENERAL)
    np.testing.assert_array_equal(out["dones"].cpu().numpy().astype(bool), o_done)
    assert rel_err(out["rewards"].cpu().numpy(), o_rew) <= REL_TOL
    assert rel_err(env.get_state().cpu().numpy(), lg.state) <= REL_TOL
    st = env.read_stats()
    assert lg.stats()["episodes"] > n
    assert_stats(st, lg.stats(), lg.tolerance(), "general rollout")
    assert_own_records(st, out["rewards"].cpu().numpy(), out["dones"].cpu().numpy())


def test_closed_form_integrator():
    """R9: the closed-form integrator solves nothing, so both RK slots and the failures stay 0; the other slots
    agree with the launch's own records."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    n, K = 800, 20
    env = BatchedRendezvousEnv(n, seed=3, t_max=7, integrator="closed_form")
    env.reset()
    out = env.rollout(K, action_seed=1, record_rewards=True, record_dones=True)
    st = env.read_stats()
    assert_own_records(st, out["rewards"].cpu().numpy(), out["dones"].cpu().numpy())
    assert st["rk_accepted"] == st["rk_rejected"] == st["failures"] == 0 and st["episodes"] > n
    assert st["steps"] == K * n
    env.read_stats(reset=True)
    rews, dones = [], []
    for k in range(6):
        _, r, d = env.step(torch.zeros((n, 6), dtype=torch.float64, device=env.device))
        rews.append(r.cpu().numpy().copy())
        dones.append(d.cpu().numpy().copy())
    st = env.read_stats()
    assert_own_records(st, rews, dones)
    assert st["rk_accepted"] == st["rk_rejected"] == st["failures"] == 0 and st["steps"] == 6 * n


def _fast_spin_states(n, rng):
    st = np.zeros((n, 20))
    st[:, 0:3] = [0.0, -10.0, 0.0] + rng.normal(0, 0.5, (n, 3))
    st[:, 3:6] = rng.normal(0, 0.05, (n, 3))
    q = rng.normal(size=(n, 4)); q /= np.linalg.norm(q, axis=1, keepdims=True)
    qt = rng.normal(size=(n, 4)); qt /= np.linalg.norm(qt, axis=1, keepdims=True)
    st[:, 6:10], st[:, 13:17] = q, qt
    scale = np.repeat([0.02, 0.3, 1.0, 3.0, 6.0, 12.0], -(-n // 6))[:n, None]
    st[:, 10:13] = rng.uniform(-1, 1, (n, 3)) * scale
    st[:, 17:20] = rng.uniform(-1, 1, (n, 3)) * scale[::-1]
    return st


@pytest.mark.parametrize("dt", [0.25, 1.0, 4.0])
def test_fast_spins(dt):
    """R10: bodies spinning at up to 12 rad/s (the stagewise solver, pair_mixed, rejected steps) through rdv_step and
    the rollout at 256 and 448 threads per CTA."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, _native as N
    n, K = 742, 2
    rng = np.random.default_rng(int(4 * dt) + 1)
    st0 = _fast_spin_states(n, rng)
    a = rng.uniform(-1, 1, (K, n, 6))
    kw = dict(dt=dt, t_max=100 * dt)
    lg = Ledger(CO.make_params(**kw), n, 1, auto_reset=False)
    lg.set_state(st0)
    for k in range(K):
        lg.step(a[k])
    want, tol = lg.stats(), lg.tolerance()
    assert want["rk_rejected"] > 0
    try:
        for path in ("step", 256, 448):
            env = BatchedRendezvousEnv(n, seed=1, auto_reset=False, **kw)
            env.reset()
            env.set_state(st0, refresh_flags=True)
            if path == "step":
                for k in range(K):
                    env.step(torch.as_tensor(a[k], device=env.device))
            else:
                _tune(N.TUNE_ROLLOUT_TPB, path)
                env.rollout(K, actions=torch.as_tensor(a, device=env.device))
            assert rel_err(env.get_state().cpu().numpy(), lg.state) <= REL_TOL, (dt, path)
            assert_stats(env.read_stats(), want, tol, (dt, path))
    finally:
        _tune(N.TUNE_ROLLOUT_TPB, 0)


FAIL_PATHS = [("step", {}), (256, {}), (448, {}), ("step", GENERAL), ("rollout", GENERAL),
              ("step", dict(integrator="closed_form")), ("rollout", dict(integrator="closed_form"))]


@pytest.mark.parametrize("path", range(len(FAIL_PATHS)), ids=["step", "tpb256", "tpb448", "general_step",
                                                              "general_rollout", "closed_step", "closed_rollout"])
def test_non_finite_quaternion_bookkeeping(path):
    """F1: a NaN quaternion in the chaser only, the target only, and both.  The solve of that body fails; the env-step
    counts ONE failure whichever solves failed, and the accepted steps of the solve that completed still count."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, _native as N
    kind, body = FAIL_PATHS[path]
    closed = body.get("integrator") == "closed_form"
    n, K, seed = 300, 3, 13
    chaser, target, both = [3, 40, 41, 170], [7, 100, 299], [11, 250]
    a = np.random.default_rng(8).uniform(-1, 1, (K, n, 6))
    env = BatchedRendezvousEnv(n, seed=seed, t_max=30, **body)
    env.reset()
    lg = Ledger(CO.make_params(t_max=30, **_oracle_kw(body)), n, seed)
    lg.reset()
    for i in chaser + both:
        env.state_view("qc")[i, 1] = float("nan")
        lg.orc.state[i, 7] = np.nan
    for i in target + both:
        env.state_view("qt")[i, 2] = float("nan")
        lg.orc.state[i, 15] = np.nan
    rews, dones = [], []
    try:
        if kind == "step":
            for k in range(K):
                _, r, d = env.step(torch.as_tensor(a[k], device=env.device))
                rews.append(r.cpu().numpy().copy())
                dones.append(d.cpu().numpy().copy())
        else:
            if kind != "rollout":
                _tune(N.TUNE_ROLLOUT_TPB, kind)
            out = env.rollout(K, actions=torch.as_tensor(a, device=env.device), record_rewards=True,
                              record_dones=True)
            rews, dones = out["rewards"].cpu().numpy(), out["dones"].cpu().numpy()
    finally:
        _tune(N.TUNE_ROLLOUT_TPB, 0)
    for k in range(K):
        lg.step(a[k])
    st = env.read_stats()
    want = lg.stats()
    bad = chaser + target + both
    assert np.asarray(dones)[0][bad].all()                  # every such env ended at once (not in the Box)
    assert_own_records(st, rews, dones, kind)
    if closed:
        # the closed form solves nothing: no RK steps and no failures; the rest of its trajectory is not the oracle's
        want.update(rk_accepted=0.0, rk_rejected=0.0, failures=0.0)
        for k in INT_STATS:
            assert st[k] == want[k], (kind, k, st[k], want[k])
        return
    assert want["failures"] == len(bad)
    assert_stats(st, want, lg.tolerance(), (kind, path))
