"""GPU parity of rdv_step (through the C ABI) against
  (1) the frozen outputs of the UNMODIFIED reference (tests/golden/traj_*.npz, made by oracle/make_golden.py),
  (2) the plain-C oracle on seeded random batches, including auto-reset with the shared Philox stream.

Tolerance: BASELINE.json north_star -- 1e-9 relative on fp64 trajectories; rewards within 1e-9;
done / collided / success / end-reason exact (a mismatch is accepted only where the golden value
lies within 1e-9 of the threshold it is compared with); float32 observations within 1 ulp of 1.0.
"""
import numpy as np
import pytest

from helpers import ERROR_FLOORS, NO_RANGE, REL_TOL, cfg_kwargs, golden, rel_err

pytestmark = pytest.mark.gpu
OBS_TOL = 1.2e-7        # one float32 ulp at |x| <= 1: the fp64 value may sit on a rounding boundary


def _run_cases(g, idx, ctor_kwargs, reward_kwargs=None, integrator="rk45"):
    """Replay golden cases `idx` (same config) as one batch; returns dict of worst deviations."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    idx = np.asarray(idx)
    env = BatchedRendezvousEnv(len(idx), auto_reset=False, reward_kwargs=reward_kwargs, integrator=integrator,
                               **ctor_kwargs)
    env.reset()
    env.set_state(g["ic"][idx])
    np.testing.assert_array_equal(env.observe().cpu().numpy(), g["obs0"][idx])
    L = g["length"][idx]
    acts = g["actions"][idx]
    worst = dict(state=0.0, rew=0.0, obs=0.0, tdv=0.0, tdw=0.0, err=0.0, koz=0.0)
    flag_mismatch = 0
    for k in range(int(L.max())):
        live = k < L
        a = torch.as_tensor(acts[:, k], device=env.device)
        obs, rew, done = env.step(a)
        err, col, suc, koz = env.errors()
        worst["state"] = max(worst["state"], rel_err(env.get_state().cpu().numpy()[live], g["state"][idx, k][live]))
        worst["rew"] = max(worst["rew"], rel_err(rew.cpu().numpy()[live], g["rew"][idx, k][live]))
        worst["obs"] = max(worst["obs"], float(np.abs(obs.cpu().numpy()[live] - g["obs"][idx, k][live]).max()))
        worst["tdv"] = max(worst["tdv"], rel_err(env.total_delta_v.cpu().numpy()[live], g["tdv"][idx, k][live]))
        worst["tdw"] = max(worst["tdw"], rel_err(env.total_delta_w.cpu().numpy()[live], g["tdw"][idx, k][live]))
        worst["err"] = max(worst["err"], rel_err(err.cpu().numpy()[live], g["errors"][idx, k][live], ERROR_FLOORS))
        worst["koz"] = max(worst["koz"], rel_err(koz.cpu().numpy()[live], g["koz"][idx, k][live]))
        flag_mismatch += int((done.cpu().numpy()[live] != g["done"][idx, k][live]).sum())
        flag_mismatch += int((env.collided.cpu().numpy()[live] != g["collided"][idx, k][live]).sum())
        flag_mismatch += int((env.success.cpu().numpy()[live] != g["success"][idx, k][live]).sum())
        flag_mismatch += int((env.end_reason.cpu().numpy()[live] != g["reason"][idx, k][live]).sum())
        flag_mismatch += int((col.cpu().numpy()[live] != g["collision_now"][idx, k][live]).sum())
        steps = env.step_count.cpu().numpy()[live]
        assert (steps == k + 1).all()
    worst["flags"] = flag_mismatch
    return worst


def _assert_parity(w, tag):
    assert w["state"] <= REL_TOL, (tag, w)
    assert w["rew"] <= REL_TOL, (tag, w)
    assert w["err"] <= REL_TOL and w["koz"] <= REL_TOL, (tag, w)
    assert w["tdw"] <= REL_TOL, (tag, w)
    assert w["obs"] <= OBS_TOL, (tag, w)
    assert w["flags"] == 0, (tag, w)


def test_golden_fp64_actions():
    """96 reference episodes (12 Monte-Carlo ICs x zero/fixed/uniform/gentle fp64 actions x t_max 60/120)."""
    g = golden("traj_f64.npz")
    for t_max in (60.0, 120.0):
        idx = np.flatnonzero(g["t_max"] == t_max)
        w = _run_cases(g, idx, dict(dt=1, t_max=t_max, **NO_RANGE))
        _assert_parity(w, f"t_max={t_max}")
        assert w["tdv"] <= REL_TOL


def test_golden_fp32_policy_actions():
    """48 reference episodes driven by the shipped MLP policy's float32 actions (NumPy-2 promotion rules:
    delta_v / total_delta_v / fuel term in fp32)."""
    g = golden("traj_f32.npz")
    assert g["actions"].dtype == np.float32
    w = _run_cases(g, np.arange(len(g["length"])), dict(dt=1, t_max=60, **NO_RANGE))
    _assert_parity(w, "f32")
    assert w["tdv"] <= 1e-7          # total_delta_v accumulates in float32 in the reference


def test_golden_configs():
    """Non-default constructor parameters (sensitivity-sweep axes: h, koz, corridor, dt, rc0, wt0, reward)."""
    g = golden("traj_cfg.npz")
    cfgs = [str(c) for c in g["cfg"]]
    for cfg in sorted(set(cfgs)):
        idx = [i for i, c in enumerate(cfgs) if c == cfg]
        kw, reward = cfg_kwargs(cfg)
        w = _run_cases(g, idx, dict(NO_RANGE, **kw), reward_kwargs=reward)
        _assert_parity(w, cfg)


def test_known_answer_vector():
    """SURVEY.md section 8c: CSV row 0, fp64 action [0.5,-0.25,0.1,0.2,-0.1,0.05] applied 3 times."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    ic = golden("traj_f64.npz")["ic"][0]
    env = BatchedRendezvousEnv(1, auto_reset=False, dt=1, t_max=60, **NO_RANGE)
    env.reset()
    env.set_state(ic[None])
    a = torch.tensor([[0.5, -0.25, 0.1, 0.2, -0.1, 0.05]], dtype=torch.float64, device=env.device)
    rews = []
    for _ in range(3):
        _, rew, done = env.step(a)
        rews.append(float(rew[0]))
    np.testing.assert_allclose(rews, [2.0559846397346275, 2.058868592759961, 2.057412928302262], rtol=1e-9)
    s = env.get_state().cpu().numpy()[0]
    np.testing.assert_allclose(s[0:3], [0.2200069248780245, -9.680428164266877, -0.4026617743928622], rtol=1e-9)
    np.testing.assert_allclose(s[3:6], [0.0837701806460994, -0.0243025944639084, 0.01784886114418886], rtol=1e-9)
    np.testing.assert_allclose(s[6:10], [0.9999504147904752, 0.00836140201404473, -0.00344381757525102,
                                         -0.00417073581332044], rtol=1e-9, atol=1e-12)
    err, col, suc, koz = env.errors()
    np.testing.assert_allclose(err.cpu().numpy()[0], [7.7854802180764127, 0.098509752926333141,
                                                      0.039751831117195956, 0.0041720300952382272], rtol=1e-9)
    np.testing.assert_allclose(float(koz[0]), 4.9985334300547155, rtol=1e-9)
    assert not bool(done[0]) and int(env.collided[0]) == 0 and int(env.success[0]) == 0


@pytest.mark.parametrize("act_dtype", ["float64", "float32"])
def test_random_batch_vs_c_oracle_with_auto_reset(act_dtype):
    """4096 envs x 40 steps, random initial states and actions, auto-reset on: state, observation, reward,
    flags and the Philox-driven resets must follow the C oracle."""
    import torch
    from oracle import c_oracle as CO
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    n, steps, seed, offset = 4096, 40, 1234, 100_000
    rng = np.random.default_rng(5)
    env = BatchedRendezvousEnv(n, seed=seed, env_offset=offset, auto_reset=True, t_max=30)
    orc = CO.COracleBatch(CO.make_params(t_max=30), n)
    obs0 = env.reset().cpu().numpy()
    episode = np.ones(n, dtype=np.int32)            # reset() bumps the episode index to 1
    ids = offset + np.arange(n)
    o0 = orc.reset_from_uniforms(CO.philox_uniforms(seed, ids, episode))
    assert rel_err(env.get_state().cpu().numpy(), orc.state) <= REL_TOL
    assert np.abs(obs0 - o0).max() <= OBS_TOL
    total_done = 0
    for k in range(steps):
        scale = 1.0 if k % 2 else 0.3
        a = (scale * rng.uniform(-1, 1, (n, 6))).astype(act_dtype)
        obs, rew, done = env.step(torch.as_tensor(a, device=env.device))
        o_obs, o_rew, o_done = orc.step(a, threads=8)
        o_obs, o_rew, o_done = o_obs.copy(), o_rew.copy(), o_done.copy()
        done_np = done.cpu().numpy()
        np.testing.assert_array_equal(done_np, o_done)
        np.testing.assert_array_equal(env.end_reason.cpu().numpy(), np.where(o_done > 0, orc.reason, -1))
        assert rel_err(rew.cpu().numpy(), o_rew) <= REL_TOL
        d = np.flatnonzero(o_done)
        if d.size:
            total_done += d.size
            assert np.abs(env.terminal_obs.cpu().numpy()[d] - o_obs[d]).max() <= OBS_TOL
            rec = env.episode_record.cpu().numpy()[d]
            np.testing.assert_array_equal(rec[:, 1], np.round(orc.aux[d, 2] / 1.0))          # length = t/dt
            np.testing.assert_array_equal(rec[:, 3], orc.flags[d, 0])
            episode[d] += 1
            mask = np.zeros(n, dtype=np.uint8)
            mask[d] = 1
            o_obs = orc.reset_from_uniforms(CO.philox_uniforms(seed, ids, episode), mask=mask).copy()
        assert np.abs(obs.cpu().numpy() - o_obs).max() <= OBS_TOL
        assert rel_err(env.get_state().cpu().numpy(), orc.state) <= REL_TOL
        np.testing.assert_array_equal(env.collided.cpu().numpy(), orc.flags[:, 0])
        np.testing.assert_array_equal(env.success.cpu().numpy(), orc.flags[:, 1])
        np.testing.assert_array_equal(env.episode_index.cpu().numpy(), episode)
    assert total_done > n // 2          # the reset path really was exercised
    st = env.read_stats()
    assert st["steps"] == n * steps and st["episodes"] == total_done and st["failures"] == 0


def test_plane_solver_edge_states_vs_c_oracle():
    """The isotropic bodies are integrated in the invariant plane span{q0, M q0} (rk45_iso_plane).  States at the
    edges of that construction -- zero rates (M q0 = 0), rates at the observation bound, injected quaternions that
    are not unit vectors -- must follow the C oracle (the 4-component restatement of scipy's RK45) like any other,
    through both kernels (per-step pair kernel and fused rollout)."""
    import torch
    from oracle import c_oracle as CO
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    n = 512
    rng = np.random.default_rng(11)
    st = np.zeros((n, 20))
    st[:, 0:3] = [0.0, -10.0, 0.0] + rng.normal(0, 0.5, (n, 3))
    st[:, 3:6] = rng.normal(0, 0.05, (n, 3))
    q = rng.normal(size=(n, 4)); q /= np.linalg.norm(q, axis=1, keepdims=True)
    qt = rng.normal(size=(n, 4)); qt /= np.linalg.norm(qt, axis=1, keepdims=True)
    st[:, 6:10], st[:, 13:17] = q, qt
    st[:, 10:13] = rng.uniform(-0.17, 0.17, (n, 3))               # up to ~10 deg/s, the observation bound
    st[:, 17:20] = rng.uniform(-0.05, 0.05, (n, 3))
    st[0:64, 10:13] = 0.0                                        # chaser at rest
    st[32:128, 17:20] = 0.0                                      # target at rest (both at rest for 32..63)
    st[128:192, 6:10] *= 1.7                                     # injected non-unit quaternions
    st[160:256, 13:17] *= 0.3
    a = rng.uniform(-1, 1, (3, n, 6))
    a[:, 0:32, 3:6] = 0.0                                        # no torque impulse either: w stays exactly 0
    for fused in (False, True):
        env = BatchedRendezvousEnv(n, seed=1, auto_reset=False, t_max=100)
        env.reset()
        env.set_state(st)
        orc = CO.COracleBatch(CO.make_params(t_max=100), n)
        orc.set_state(st, recompute_flags=True)
        env.refresh_flags()
        for k in range(3):
            if fused:
                out = env.rollout(1, actions=torch.as_tensor(a[k:k + 1], device=env.device), record_rewards=True)
                rew = out["rewards"][0]
            else:
                _, rew, _ = env.step(torch.as_tensor(a[k], device=env.device))
            _, o_rew, _ = orc.step(a[k], threads=4)
            assert rel_err(env.get_state().cpu().numpy(), orc.state) <= REL_TOL, (fused, k)
            assert rel_err(rew.cpu().numpy(), o_rew.copy()) <= REL_TOL, (fused, k)
        assert env.read_stats()["failures"] == 0


@pytest.mark.parametrize("dt", [0.25, 1.0, 4.0])
def test_fast_spins_take_the_general_controller_paths(dt):
    """select_initial_step and the last attempt of a solve are shortened by bounds that hold for every body the
    reference's ranges produce (csrc/rdv_math.cuh: plane_initial_step, plane_step).  Bodies that
    spin at up to several rad/s break those bounds -- 100 h0 becomes the smallest candidate, d2 exceeds d1, steps are
    rejected, the clipped last attempt is not trivially acceptable -- and must then follow the C oracle through the
    general path, at every dt of the sensitivity grid, through both kernels."""
    import torch
    from oracle import c_oracle as CO
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    n = 768
    rng = np.random.default_rng(23)
    st = np.zeros((n, 20))
    st[:, 0:3] = [0.0, -10.0, 0.0] + rng.normal(0, 0.5, (n, 3))
    st[:, 3:6] = rng.normal(0, 0.05, (n, 3))
    q = rng.normal(size=(n, 4)); q /= np.linalg.norm(q, axis=1, keepdims=True)
    qt = rng.normal(size=(n, 4)); qt /= np.linalg.norm(qt, axis=1, keepdims=True)
    st[:, 6:10], st[:, 13:17] = q, qt
    scale = np.repeat([0.02, 0.3, 1.0, 3.0, 6.0, 12.0], n // 6)[:, None]        # rad/s, slow to absurd
    st[:, 10:13] = rng.uniform(-1, 1, (n, 3)) * scale
    st[:, 17:20] = rng.uniform(-1, 1, (n, 3)) * scale[::-1]
    a = rng.uniform(-1, 1, (2, n, 6))
    kw = dict(dt=dt, t_max=100 * dt)
    for fused in (False, True):
        env = BatchedRendezvousEnv(n, seed=1, auto_reset=False, **kw)
        env.reset()
        env.set_state(st)
        orc = CO.COracleBatch(CO.make_params(**kw), n)
        orc.set_state(st, recompute_flags=True)
        env.refresh_flags()
        for k in range(2):
            if fused:
                env.rollout(1, actions=torch.as_tensor(a[k:k + 1], device=env.device))
            else:
                env.step(torch.as_tensor(a[k], device=env.device))
            orc.step(a[k], threads=4)
            assert rel_err(env.get_state().cpu().numpy(), orc.state) <= REL_TOL, (fused, k, dt)
        stats = env.read_stats()
        assert stats["failures"] == 0 and stats["rk_rejected"] > 0, stats      # the rejection path was exercised


def test_closed_form_fast_path_within_tolerance():
    """The opt-in closed-form attitude propagation (exact for the env's isotropic, torque-free bodies) stays
    within the parity tolerance of the reference's RK45 at the default dt = 1 s."""
    g = golden("traj_f64.npz")
    idx = np.flatnonzero(g["t_max"] == 120.0)
    w = _run_cases(g, idx, dict(dt=1, t_max=120.0, **NO_RANGE), integrator="closed_form")
    assert w["state"] <= REL_TOL and w["rew"] <= 1e-6, w


def test_edge_cases():
    """n = 1, n not a multiple of the CTA size, wrong shapes / dtypes / devices."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    for n in (1, 63, 65, 1000):
        env = BatchedRendezvousEnv(n, seed=3)
        env.reset()
        a = torch.zeros((n, 6), dtype=torch.float64, device=env.device)
        obs, rew, done = env.step(a)
        assert obs.shape == (n, 17) and torch.isfinite(obs).all() and torch.isfinite(rew).all()
        ref = BatchedRendezvousEnv(1000, seed=3)
        ref.reset()
        ref.step(torch.zeros((1000, 6), dtype=torch.float64, device=env.device))
        m = min(n, 1000)
        # env i of a small batch == env i of a large batch (results independent of grid shape)
        assert torch.equal(env.get_state()[:m], ref.get_state()[:m])
    env = BatchedRendezvousEnv(8)
    env.reset()
    with pytest.raises(ValueError):
        env.step(torch.zeros((7, 6), dtype=torch.float64, device=env.device))
    with pytest.raises(TypeError):
        env.step(torch.zeros((8, 6), dtype=torch.float16, device=env.device))
    with pytest.raises(ValueError):
        env.step(torch.zeros((8, 6), dtype=torch.float64))
    with pytest.raises(TypeError):
        env.step(np.zeros((8, 6)))


def test_all_1000_published_initial_conditions_vs_c_oracle():
    """BASELINE.json north_star's protocol on ALL rows of results/data_monte_carlo_initial_conditions.csv (frozen in
    tests/golden/mc.npz): identical initial conditions and identical action sequences -- three seeded fp64 streams
    (uniform, gentle, bang-bang) -- through rdv_step and through rdv_rollout, against the C oracle over the full
    60-step episodes: trajectories within 1e-9 of each component's own scale, rewards within 1e-9, done / end
    reason / collided / success exact at every step."""
    import torch
    from oracle import c_oracle as CO
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    mc = golden("mc.npz")
    ics = mc["ic_raw"].copy()
    ics[:, 6:10] /= np.linalg.norm(ics[:, 6:10], axis=1, keepdims=True)
    ics[:, 13:17] /= np.linalg.norm(ics[:, 13:17], axis=1, keepdims=True)
    n, K = ics.shape[0], 60
    assert n == 1000
    kw = dict(dt=1, t_max=60, **NO_RANGE)
    rng = np.random.default_rng(20260101)
    streams = {"uniform": rng.uniform(-1, 1, (K, n, 6)),
               "gentle": np.clip(rng.normal(0, 0.3, (K, n, 6)), -1, 1),
               "bang": np.sign(rng.uniform(-1, 1, (K, n, 6)))}
    worst = {}
    for name, acts in streams.items():
        orc = CO.COracleBatch(CO.make_params(**kw), n)
        orc.set_state(ics)
        ref_state, ref_rew, ref_done, ref_reason, ref_flags = [], [], [], [], []
        for k in range(K):
            _, r, d = orc.step(acts[k], threads=8)
            ref_state.append(orc.state.copy()); ref_rew.append(r.copy()); ref_done.append(d.copy())
            ref_reason.append(orc.reason.copy()); ref_flags.append(orc.flags.copy())
        # per-step entry point
        env = BatchedRendezvousEnv(n, auto_reset=False, **kw)
        env.reset()
        env.set_state(ics)
        w_state = w_rew = 0.0
        for k in range(K):
            _, rew, done = env.step(torch.as_tensor(acts[k], device=env.device))
            w_state = max(w_state, rel_err(env.get_state().cpu().numpy(), ref_state[k]))
            w_rew = max(w_rew, rel_err(rew.cpu().numpy(), ref_rew[k]))
            np.testing.assert_array_equal(done.cpu().numpy(), ref_done[k])
            live = ref_done[k] > 0
            np.testing.assert_array_equal(env.end_reason.cpu().numpy()[live], ref_reason[k][live])
            np.testing.assert_array_equal(env.collided.cpu().numpy(), ref_flags[k][:, 0])
            np.testing.assert_array_equal(env.success.cpu().numpy(), ref_flags[k][:, 1])
        assert w_state <= REL_TOL and w_rew <= REL_TOL, (name, "step", w_state, w_rew)
        # fused rollout, one launch
        env2 = BatchedRendezvousEnv(n, auto_reset=False, **kw)
        env2.reset()
        env2.set_state(ics)
        out = env2.rollout(K, actions=torch.as_tensor(acts, device=env2.device), record_rewards=True, record_dones=True)
        assert rel_err(out["rewards"].cpu().numpy(), np.array(ref_rew)) <= REL_TOL, name
        np.testing.assert_array_equal(out["dones"].cpu().numpy(), np.array(ref_done))
        w2 = rel_err(env2.get_state().cpu().numpy(), ref_state[-1])
        assert w2 <= REL_TOL, (name, "rollout", w2)
        np.testing.assert_array_equal(env2.collided.cpu().numpy(), ref_flags[-1][:, 0])
        np.testing.assert_array_equal(env2.success.cpu().numpy(), ref_flags[-1][:, 1])
        worst[name] = (w_state, w_rew, w2)
    print("worst deviations (state via step, reward, state via rollout):", worst)


def test_frame_transform_vs_oracle_non_unit_quaternions():
    """rdv_frame_transform against the oracle's chaser2lvlh / lvlh2chaser (rendezvous_env.py:470-508: quat2mat
    re-normalises, utils/quaternions.py:48-68) for quaternions that are NOT unit length."""
    import ctypes as C
    import torch
    from oracle.rdv_oracle import rotation_matrix
    from reinforcement_learning_rendezvous_b200 import _native as N
    rng = np.random.default_rng(5)
    n = 4096
    q = rng.normal(size=(n, 4)) * rng.uniform(0.05, 20.0, (n, 1))          # norms from 0.05 to 20
    v = rng.normal(size=(n, 3)) * 10
    dq, dv = torch.as_tensor(q, device="cuda"), torch.as_tensor(v, device="cuda")
    out = torch.empty_like(dv)
    for transpose in (0, 1):
        N.check(N.lib().rdv_frame_transform(dq.data_ptr(), dv.data_ptr(), out.data_ptr(), n, transpose,
                                            C.c_void_p(torch.cuda.current_stream().cuda_stream)), "frame")
        got = out.cpu().numpy()
        ref = np.stack([(rotation_matrix(q[i]).T if transpose else rotation_matrix(q[i])) @ v[i] for i in range(n)])
        assert np.max(np.abs(got - ref) / np.maximum(np.abs(ref), 1.0)) <= 1e-13, transpose
