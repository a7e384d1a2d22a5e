"""GPU: the trajectory record of the fused rollout (rdv_rollout_trajectory / rollout(record_trajectory=True)).  The
record must leave every other output of the launch unchanged, its rows must be the states a shorter launch ends in
(or, past an auto-reset, the states the C oracle steps through), and its evaluator columns must be what rdv_errors
returns on those states -- all bit for bit, except the oracle comparison (1e-9 of each component's scale)."""
import os

import numpy as np
import pytest

from helpers import GOLDEN, REL_TOL, STATE_FLOORS, golden

pytestmark = pytest.mark.gpu

T = 128
N_ENVS = T * 7 + 37                                       # 933: a partial last warp, tile and pass
REC = dict(record_rewards=True, record_dones=True, record_obs=True, record_actions=True)
BODIES = {"iso": {}, "closed": dict(integrator="closed_form"), "general": dict(inertia=np.diag([10.0, 16.0, 22.0]))}
SETS = [dict(), dict(h=600e3), dict(rc0=np.array([0.0, -20.0, 0.0]))]
INT_STATS = ("steps", "episodes", "length_sum", "succeeded", "collided", "end_obs", "end_time", "end_bubble",
             "end_attitude", "rk_accepted", "rk_rejected", "failures")


@pytest.fixture(scope="module")
def pols():
    from reinforcement_learning_rendezvous_b200.policy import MlpPolicy, load_state_dict
    base = load_state_dict(os.path.join(GOLDEN, "policy.npz"))
    out = [MlpPolicy(base)]
    for seed in (1, 2):
        rng = np.random.default_rng(seed)
        sd = {k: (v + rng.normal(0.0, 0.3 * float(v.std()) + 1e-3, v.shape)).astype(np.float32) for k, v in base.items()}
        sd["log_std"] = (base["log_std"] + 0.25 * seed).astype(np.float32)
        out.append(MlpPolicy(sd))
    return out


def _env(n=N_ENVS, seed=5, auto_reset=True, body="iso", param_table=False, **kw):
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    if param_table:
        per = n // 3 // 32 * 32
        kw["param_batches"] = [(per, SETS[0]), (per, SETS[1]), (n - 2 * per, SETS[2])]
    e = BatchedRendezvousEnv(n, seed=seed, auto_reset=auto_reset, **BODIES[body], **kw)
    e.reset()
    return e


def _launch(env, K, source, pols, record_trajectory, step_base=0, mc=False, **extra):
    """One rollout of `env` with the action source named by `source`; tensor actions are seeded, so repeated calls with
    the same arguments give the same inputs."""
    import torch
    kw = dict(REC, record_trajectory=record_trajectory, step_base=step_base, monte_carlo=mc, **extra)
    if source in ("f32", "f64"):
        g = torch.Generator(device=env.device).manual_seed(1234 + step_base)
        # drawn at one length and cut, so that shorter launches get a prefix of the same actions
        a = (torch.rand((max(K, 32), env.num_envs, 6), generator=g, device=env.device, dtype=torch.float64) * 2 - 1)[:K]
        kw.pop("record_actions")
        return env.rollout(K, actions=a.float() if source == "f32" else a, **kw)
    if source == "philox":
        return env.rollout(K, action_seed=21, **kw)
    if source == "policy":
        return env.rollout(K, policy=pols[0], **kw)
    if source == "sample":
        return env.rollout(K, policy=pols[1], stochastic=True, action_seed=21, **kw)
    from reinforcement_learning_rendezvous_b200 import PolicyTable
    tiles = [2, 0, 2, 1, 1, 0, 2, 1][:(env.num_envs + T - 1) // T]         # not monotone: groups restage
    return env.rollout(K, policy=PolicyTable(pols), policy_tiles=tiles, stochastic=source == "table_sample",
                       action_seed=21, **kw)


CASES = [(src, ar, False, False, "iso") for src in ("f32", "f64", "philox", "policy", "sample", "table", "table_sample")
         for ar in (True, False)]
CASES += [(src, False, True, False, "iso") for src in ("philox", "policy", "table")]                  # evaluator mode
CASES += [(src, ar, False, True, "iso") for src in ("philox", "policy", "table") for ar in (True, False)]  # param table
CASES += [(src, False, True, True, "iso") for src in ("philox", "policy", "table")]
CASES += [("philox", ar, False, False, b) for b in ("closed", "general") for ar in (True, False)]
CASES += [("f32", True, False, False, b) for b in ("closed", "general")]


@pytest.mark.parametrize("source,auto_reset,mc,ptable,body", CASES)
def test_record_changes_nothing_else(pols, source, auto_reset, mc, ptable, body):
    import torch
    from reinforcement_learning_rendezvous_b200._native import STAT_NAMES
    K = 24
    a = _env(auto_reset=auto_reset, body=body, param_table=ptable)
    b = _env(auto_reset=auto_reset, body=body, param_table=ptable)
    oa = _launch(a, K if not mc else int(a.params.done_steps), source, pols, False, mc=mc)
    ob = _launch(b, K if not mc else int(b.params.done_steps), source, pols, True, mc=mc)
    assert set(ob) == set(oa) | {"trajectory"}
    for k in oa:
        assert torch.equal(oa[k], ob[k]), k
    assert torch.equal(a.f64, b.f64) and torch.equal(a.i32, b.i32)
    # statistics: integer slots exact, fp64 sums to 1e-12 (the CTAs add them with atomics, in no fixed order)
    for name, x, y in zip(STAT_NAMES, a.stats.tolist(), b.stats.tolist()):
        assert x == y if name in INT_STATS else abs(x - y) <= 1e-12 * max(abs(y), 1.0), name
    tr = ob["trajectory"]
    assert tr.shape == (oa["rewards"].shape[0], 34, N_ENVS) and tr.dtype == torch.float64
    assert bool(torch.isfinite(tr).all())
    if auto_reset:
        assert int(oa["dones"].sum()) > 0                  # episodes end and restart inside the launch
    # the last row is the final state, except where an auto-reset replaced it
    last = tr[-1]
    keep = ~oa["dones"][-1].bool() if auto_reset else torch.ones(N_ENVS, dtype=torch.bool, device=tr.device)
    assert torch.equal(last[:23][:, keep], b.f64[:23, :N_ENVS][:, keep])
    assert torch.equal(last[23:27][:, keep], b.i32[:4, :N_ENVS][:, keep].double())


def _prefix_launches(make, K, source, pols):
    """the final f64 / i32 state of a (k + 1)-step launch from the same start, for every k"""
    out = []
    for k in range(K):
        e = make()
        _launch(e, k + 1, source, pols, False)
        out.append((e.f64[:23, :e.num_envs].clone(), e.i32[:4, :e.num_envs].double()))
    return out


@pytest.mark.parametrize("source,body", [("philox", "iso"), ("policy", "iso"), ("f64", "iso"), ("philox", "closed"),
                                         ("philox", "general"), ("f32", "general")])
def test_rows_are_prefix_states(pols, source, body):
    import torch
    K, n = 12, 300
    make = lambda: _env(n=n, seed=3, auto_reset=False, body=body)                    # noqa: E731
    tr = _launch(make(), K, source, pols, True)["trajectory"]
    for k, (f, i) in enumerate(_prefix_launches(make, K, source, pols)):
        assert torch.equal(tr[k, :23], f), k
        assert torch.equal(tr[k, 23:27], i), k


def test_auto_reset_rows(pols):
    """Rows of envs that did not finish at step k are the states of a (k + 1)-step launch; the rows of finished envs
    are their terminal states, which the C oracle stepped without a reset reaches; their step column is the episode
    length."""
    import torch
    from oracle import c_oracle as CO
    K, n, seed = 24, 512, 9
    make = lambda: _env(n=n, seed=seed, auto_reset=True)                            # noqa: E731
    out = _launch(make(), K, "philox", pols, True)
    tr, dones = out["trajectory"], out["dones"].bool()
    assert int(dones.sum()) > 0
    for k, (f, i) in enumerate(_prefix_launches(make, K, "philox", pols)):
        live = ~dones[k]
        assert torch.equal(tr[k, :23][:, live], f[:, live]), k
        assert torch.equal(tr[k, 23:27][:, live], i[:, live]), k
    trn, acts, dn = tr.cpu().numpy(), out["actions"].cpu().numpy(), dones.cpu().numpy()
    ids, episode = np.arange(n), np.ones(n, dtype=np.int32)
    orc = CO.COracleBatch(CO.make_params(), n)
    orc.reset_from_uniforms(CO.philox_uniforms(seed, ids, episode))
    length = np.zeros(n, dtype=np.int64)
    worst = 0.0
    for k in range(K):
        _, _, o_done = orc.step(np.ascontiguousarray(acts[k]), threads=4)
        assert np.array_equal(o_done.astype(bool), dn[k]), k
        length += 1
        s = trn[k, :20].T
        worst = max(worst, float(np.max(np.abs(s - orc.state) / np.maximum(np.abs(orc.state), STATE_FLOORS))))
        assert np.array_equal(trn[k, 23][dn[k]], length[dn[k]].astype(np.float64)), k
        d = np.flatnonzero(dn[k])
        if d.size:
            episode[d] += 1
            length[d] = 0
            mask = np.zeros(n, dtype=np.uint8)
            mask[d] = 1
            orc.reset_from_uniforms(CO.philox_uniforms(seed, ids, episode), mask=mask)
    assert worst <= REL_TOL, worst


@pytest.mark.parametrize("source,auto_reset,mc,body", [("philox", True, False, "iso"), ("policy", False, True, "iso"),
                                                        ("table", True, False, "iso"), ("philox", False, False, "closed"),
                                                        ("philox", True, False, "general")])
def test_error_columns_equal_rdv_errors(pols, source, auto_reset, mc, body):
    """Columns 27-33 of every row == errors() of an env holding that row's state and counters."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    n = N_ENVS
    env = _env(auto_reset=auto_reset, body=body)
    K = int(env.params.done_steps) if mc else 24
    tr = _launch(env, K, source, pols, True, mc=mc)["trajectory"]
    flat = tr.permute(1, 0, 2).reshape(34, K * n)                      # every (k, env) row as one env
    chk = BatchedRendezvousEnv(K * n, auto_reset=False, track_stats=False, **BODIES[body])
    chk.f64[:23, :K * n] = flat[:23]
    chk.i32[:4, :K * n] = flat[23:27].int()
    err, col, suc, koz = chk.errors()
    assert torch.equal(flat[27:31], err.t())
    assert torch.equal(flat[31], koz)
    assert torch.equal(flat[32], col.double())
    assert torch.equal(flat[33], suc.double())


@pytest.mark.parametrize("source", ["philox", "policy", "table"])
def test_launch_shape(pols, source):
    """Two launches of K/2 (reset rows carried, step_base advanced) concatenate to one launch of K, and the record does
    not depend on the SMs a launch leaves free."""
    import torch
    K = 16
    envs = [_env() for _ in range(3)]
    envs[1].sm_reserve = 7
    one = _launch(envs[0], K, source, pols, True)["trajectory"]
    assert torch.equal(one, _launch(envs[1], K, source, pols, True)["trajectory"])
    halves = [_launch(envs[2], K // 2, source, pols, True, step_base=h * (K // 2))["trajectory"] for h in range(2)]
    assert torch.equal(one, torch.cat(halves))
    assert torch.equal(envs[0].f64, envs[2].f64) and torch.equal(envs[0].i32, envs[2].i32)


def test_evaluate_batch_trajectories(pols):
    from reinforcement_learning_rendezvous_b200 import evaluate_batch
    from reinforcement_learning_rendezvous_b200.monte_carlo import _terminal_errors_batch
    from reinforcement_learning_rendezvous_b200.params import make_params
    ics = golden("mc.npz")["ic_raw"]
    plain = evaluate_batch(pols[0], ics, return_raw=True)
    res = evaluate_batch(pols[0], ics, return_raw=True, trajectories=True)
    tr = res.pop("trajectory")
    assert set(res) == set(plain)
    for k in plain:
        assert np.array_equal(res[k], plain[k], equal_nan=True), k
    m = len(ics)
    p = make_params(dt=1, t_max=60)
    L = int(p.done_steps)
    assert tr["rc"].shape == (m, L + 1, 3) and tr["errors"].shape == (m, L + 1, 4) and tr["t"].shape == (m, L + 1)
    length = tr["length"]
    assert np.array_equal(length, res["raw"][:, 0].astype(np.int64))
    assert np.array_equal(np.round(length * p.dt, 3), res["ep_len"])
    assert np.array_equal(tr["t"][np.arange(m), length], res["ep_len"])
    assert bool((tr["t"][:, 0] == 0).all())
    for j in range(m):
        lj = length[j]
        for key in ("rc", "vc", "qc", "wc", "qt", "wt", "errors", "dist_from_koz", "collision", "total_reward", "t"):
            assert np.array_equal(tr[key][j, lj:], np.repeat(tr[key][j, lj:lj + 1], L + 1 - lj, axis=0)), (j, key)
        assert tr["dist_from_koz"][j, :lj + 1].min() == res["min_dist_from_koz"][j], j
        assert int(tr["collision"][j, :lj + 1].sum()) == res["num_collisions"][j], j
    assert np.array_equal(tr["total_reward"][np.arange(m), length], res["total_reward"])
    assert np.array_equal(tr["total_delta_v"][np.arange(m), length], res["total_delta_v"])
    # the first sample is the normalised initial condition
    assert np.array_equal(tr["rc"][:, 0], np.asarray(ics, dtype=np.float64).reshape(-1, 20)[:, 0:3])
    limits = (p.max_rd_error, p.max_vd_error, p.max_qd_error, p.max_wd_error)
    te = _terminal_errors_batch(tr["errors"].transpose(1, 0, 2), length, limits)
    for c, key in enumerate(("pos_error", "vel_error", "att_error", "rot_error")):
        want = res[key]
        assert np.max(np.abs(te[:, c] - want) / np.maximum(np.abs(want), 1e-300)) <= 1e-12, key


def test_evaluate_batch_trajectories_with_a_policy_list(pols):
    from reinforcement_learning_rendezvous_b200 import evaluate_batch
    ics = golden("mc.npz")["ic_raw"]
    both = evaluate_batch([pols[0], pols[2]], ics, trajectories=True)
    for res, p in zip(both, (pols[0], pols[2])):
        one = evaluate_batch(p, ics, trajectories=True)
        assert set(res) == set(one) and set(res["trajectory"]) == set(one["trajectory"])
        for k in one:
            if k != "trajectory":
                assert np.array_equal(res[k], one[k], equal_nan=True), k
        for k, v in one["trajectory"].items():
            assert np.array_equal(res["trajectory"][k], v), k
    assert not np.array_equal(both[0]["trajectory"]["rc"], both[1]["trajectory"]["rc"])
