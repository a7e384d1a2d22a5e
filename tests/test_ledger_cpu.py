"""CPU: the bookkeeping reference of tests/ledger.py, checked against the unmodified reference's golden episodes and
its RK45 step counts against SciPy's own solve_ivp."""
import numpy as np
import pytest

from helpers import NO_RANGE, cfg_kwargs, golden
from ledger import END_KEYS, Ledger

from oracle import c_oracle as CO
from oracle import rdv_oracle as O


def _golden_episodes(g, idx, ctor_kwargs, reward_kwargs=None):
    """Each golden episode through the ledger in the evaluator mode (an env stops at its first done): every record
    and every slot against what the reference returned along the episode."""
    idx = np.asarray(idx)
    L = g["length"][idx].astype(int)
    lg = Ledger(CO.make_params(reward_kwargs=reward_kwargs, **ctor_kwargs), len(idx), seed=0,
                auto_reset=False, stop_at_first_done=True, threads=1)
    lg.set_state(g["ic"][idx], recompute_flags=False)
    for k in range(int(L.max())):
        lg.step(np.ascontiguousarray(g["actions"][idx, k]))
    recs = lg.records_by_env()
    assert sorted(recs) == list(range(len(idx)))
    last = L - 1
    rows = np.arange(len(idx))
    for j, c in enumerate(idx):
        (r,) = recs[j]                                   # exactly one episode, ending at the golden length
        ret = float(np.sum(g["rew"][c, :L[j]]))
        assert abs(r["ret"] - ret) <= 1e-12 * max(1.0, abs(ret)), (c, r["ret"], ret)
        assert r["length"] == L[j]
        assert r["end_reason"] == g["reason"][c, last[j]]
        assert r["delta_v"] == pytest.approx(g["tdv"][c, last[j]], rel=1e-12, abs=1e-15)
        assert r["delta_w"] == pytest.approx(g["tdw"][c, last[j]], rel=1e-12, abs=1e-15)
        assert r["success"] == g["success"][c, last[j]] and r["collided"] == g["collided"][c, last[j]]
    st = lg.stats()
    assert st["steps"] == L.sum() and st["length_sum"] == L.sum() and st["episodes"] == len(idx)
    reasons = g["reason"][idx, last]
    for j, key in enumerate(END_KEYS):
        assert st[key] == np.sum(reasons == j), key
    assert st["succeeded"] == np.sum(g["success"][idx, last] > 0)
    assert st["collided"] == np.sum(g["collided"][idx, last])
    rew_all = np.concatenate([g["rew"][c, :L[j]] for j, c in enumerate(idx)])
    assert abs(st["reward_sum"] - rew_all.sum()) <= 1e-12 * np.maximum(np.abs(rew_all), 1).sum()
    assert abs(st["delta_v_sum"] - g["tdv"][idx, last].sum()) <= 1e-12 * np.maximum(g["tdv"][idx, last], 1).sum()
    assert st["failures"] == 0 and st["rk_accepted"] >= 2 * L.sum()
    assert not lg.alive[rows].any()


def test_golden_fp64_episodes():
    g = golden("traj_f64.npz")
    for t_max in (60.0, 120.0):
        _golden_episodes(g, np.flatnonzero(g["t_max"] == t_max), dict(dt=1, t_max=t_max, **NO_RANGE))


def test_golden_fp32_episodes():
    g = golden("traj_f32.npz")
    assert g["actions"].dtype == np.float32
    _golden_episodes(g, np.arange(len(g["length"])), dict(dt=1, t_max=60, **NO_RANGE))


def test_golden_config_episodes():
    g = golden("traj_cfg.npz")
    cfgs = [str(c) for c in g["cfg"]]
    for cfg in sorted(set(cfgs)):
        kw, reward = cfg_kwargs(cfg)
        _golden_episodes(g, [i for i, c in enumerate(cfgs) if c == cfg], dict(NO_RANGE, **kw), reward)


def test_auto_reset_and_stepping_past_the_end():
    """With auto-reset an env's record restarts at every done; without it an env that keeps stepping past its end
    counts again at every step, with its step counter still growing."""
    n, seed = 40, 3
    rng = np.random.default_rng(1)
    acts = rng.uniform(-1, 1, (12, n, 6))
    for auto in (True, False):
        lg = Ledger(CO.make_params(t_max=5), n, seed=seed, auto_reset=auto, threads=1)
        lg.reset()
        for a in acts:
            lg.step(a)
        st = lg.stats()
        assert st["steps"] == 12 * n
        if auto:
            assert all(r["length"] <= 5 for r in lg.records) and st["episodes"] >= 2 * n
            assert (lg.episode >= 3).all()
        else:
            assert st["episodes"] == sum(12 - min(r["length"] for r in rs) + 1 for rs in lg.records_by_env().values())
            assert st["length_sum"] == sum(r["length"] for r in lg.records)
            assert (lg.episode == 1).all()


def _scipy_counts(y0, inertia, inv_inertia, torque, dt):
    from scipy.integrate import solve_ivp
    sol = solve_ivp(O.attitude_rhs, (0.0, dt), y0, method="RK45", rtol=1e-7, atol=1e-6,
                    args=(inertia, inv_inertia, torque))
    assert sol.success
    acc = len(sol.t) - 1
    attempts, rem = divmod(sol.nfev - 2, 6)
    assert rem == 0
    return acc, attempts - acc


@pytest.mark.parametrize("dt", [0.25, 1.0, 4.0])
def test_oracle_rk_counts_equal_scipy(dt):
    """rk_out of the C oracle (accepted steps of the chaser and of the target solve, rejected attempts of both) ==
    the step counts of scipy's solve_ivp(RK45) on the reference's attitude right-hand side."""
    pytest.importorskip("scipy")
    rng = np.random.default_rng(int(dt * 4))
    bodies = {
        "iso": dict(),
        "general_torque": dict(inertia=np.array([[10.0, 0.6, -0.3], [0.6, 16.0, 0.4], [-0.3, 0.4, 22.0]]),
                               inertia_target=np.array([[30.0, -1.0, 0.5], [-1.0, 22.0, 0.0], [0.5, 0.0, 14.0]]),
                               chaser_torque=[0.02, -0.01, 0.015]),
        "fast_iso": dict(),
        "fast_general": dict(inertia=np.diag([10.0, 16.0, 22.0]), inertia_target=np.diag([25.0, 20.0, 12.0]),
                             chaser_torque=[0.05, 0.0, -0.05]),
    }
    n = 24
    total_rej = 0
    for name, kw in bodies.items():
        p = CO.make_params(dt=dt, t_max=100 * dt, **kw)
        ic, it = np.array(p.inertia_c[:]).reshape(3, 3), np.array(p.inertia_t[:]).reshape(3, 3)
        iic, iit = np.array(p.inv_inertia_c[:]).reshape(3, 3), np.array(p.inv_inertia_t[:]).reshape(3, 3)
        tau = np.array(p.torque_c[:])
        rate = 3.0 if name.startswith("fast") else 0.05
        st = np.zeros((n, 20))
        st[:, 0:3] = [0.0, -10.0, 0.0]
        q = rng.normal(size=(n, 4)); q /= np.linalg.norm(q, axis=1, keepdims=True)
        qt = rng.normal(size=(n, 4)); qt /= np.linalg.norm(qt, axis=1, keepdims=True)
        st[:, 6:10], st[:, 13:17] = q, qt
        st[:, 10:13] = rng.uniform(-rate, rate, (n, 3))
        st[:, 17:20] = rng.uniform(-rate, rate, (n, 3))
        b = CO.COracleBatch(p, n)
        b.set_state(st)
        b.step(np.zeros((n, 6)))                        # no impulse: the solves start from the injected rates
        for i in range(n):
            ac, rc = _scipy_counts(st[i, 6:13], ic, iic, tau, dt)
            at, rt = _scipy_counts(st[i, 13:20], it, iit, np.zeros(3), dt)
            assert tuple(b.rk[i]) == (ac, at, rc + rt), (name, i, tuple(b.rk[i]), (ac, at, rc + rt))
            total_rej += rc + rt
    if dt >= 1.0:
        assert total_rej > 0                            # the rejection count was exercised
