"""GPU: the collection step of RecurrentPPO (rdv_lstm_actor_critic_step: actor and critic LSTM, Gaussian draw, clip,
log-probability and value in one launch) against the fp64 reference of tests/recurrent_ref.py and against
rdv_lstm_policy_step; RecurrentPPO's collection teacher-forced and replayed through a twin env; the update's first
minibatch against the recorded log-probabilities and values; and a short training run."""
import ctypes as C

import numpy as np
import pytest
import torch

from lstm_ref import H, actor_keys, make_state_dict
from normals import philox_normals_ref
from recurrent_ref import actor_critic_step_ref
from test_gpu_lstm import _observations
from test_gpu_policy_shapes import noise_bound

pytestmark = pytest.mark.gpu

KINDS = ("torch", "ppo", "stress")
NMAX = 65536
SEED = 0x0000000500000011
STEP = 0x0000000300000007
OFFSET = 1 << 33
STATE_TOL = 1e-5                   # test_gpu_lstm.test_step_matches_fp64_reference


def _module(sd):
    from reinforcement_learning_rendezvous_b200.recurrent_ppo import RecurrentActorCritic
    m = RecurrentActorCritic().cuda()
    with torch.no_grad():
        for k, p in m.state_dict().items():
            p.copy_(torch.as_tensor(sd[k]))
    return m


def _step(m, obs, start, states, seed=SEED, step=STEP, offset=OFFSET, env_actions=True, ld=None):
    """One launch on device inputs; states: four [256, n] tensors with leading dimension ld (default n), the output
    states column slices of NaN-filled [256, ld] buffers.  Returns the outputs as device tensors."""
    from reinforcement_learning_rendezvous_b200 import _native as N
    from reinforcement_learning_rendezvous_b200.batched_env import _stream_ptr
    n, dev = obs.shape[0], obs.device
    ld = n if ld is None else ld
    out = dict(states=[torch.full((H, ld), np.nan, device=dev)[:, :n] for _ in range(4)],
               actions=torch.full((n, 6), np.nan, device=dev), env_actions=torch.full((n, 6), np.nan, device=dev),
               log_prob=torch.full((n,), np.nan, device=dev), values=torch.full((n,), np.nan, device=dev))
    w = m.kernel_weights()
    s, o = states, out["states"]
    io = N.RdvLstmStepIO(obs.data_ptr(), start.data_ptr(), s[0].data_ptr(), s[1].data_ptr(), o[0].data_ptr(),
                         o[1].data_ptr(), s[2].data_ptr(), s[3].data_ptr(), o[2].data_ptr(), o[3].data_ptr(),
                         out["actions"].data_ptr(), out["env_actions"].data_ptr() if env_actions else None,
                         out["log_prob"].data_ptr(), out["values"].data_ptr(), seed, step, offset, ld)
    N.check(N.lib().rdv_lstm_actor_critic_step(C.byref(w), C.byref(io), n, _stream_ptr(dev)), "step")
    return out


def _np(out):
    return dict(h_pi=out["states"][0].t().cpu().numpy(), c_pi=out["states"][1].t().cpu().numpy(),
                h_vf=out["states"][2].t().cpu().numpy(), c_vf=out["states"][3].t().cpu().numpy(),
                actions=out["actions"].cpu().numpy(), env_actions=out["env_actions"].cpu().numpy(),
                log_prob=out["log_prob"].cpu().numpy(), values=out["values"].cpu().numpy())


def _assert_against_ref(got, ref, sd, z, r, what):
    for k in ("h_pi", "h_vf"):
        assert np.abs(got[k] - ref[k]).max() <= STATE_TOL, (what, k, float(np.abs(got[k] - ref[k]).max()))
    for k in ("c_pi", "c_vf"):
        e = (np.abs(got[k] - ref[k]) / np.maximum(1.0, np.abs(ref[k]))).max()
        assert e <= STATE_TOL, (what, k, float(e))
    ls = np.asarray(sd["log_std"], np.float64)
    bound = STATE_TOL + noise_bound(ls, z, r, got["actions"], False)
    err = np.abs(got["actions"] - ref["actions"])
    assert (err <= bound).all(), (what, "actions", float((err / bound).max()))
    assert np.array_equal(got["env_actions"], np.clip(got["actions"], -1, 1)), what
    assert np.abs(got["log_prob"] - ref["log_prob"]).max() <= 1e-4, (what, float(np.abs(got["log_prob"] - ref["log_prob"]).max()))
    ev = np.abs(got["values"] - ref["values"]) / np.maximum(1.0, np.abs(ref["values"]))
    assert ev.max() <= 1e-5, (what, "values", float(ev.max()))
    return dict(h=max(float(np.abs(got[k] - ref[k]).max()) for k in ("h_pi", "h_vf")),
                a=float((err / bound).max()), lp=float(np.abs(got["log_prob"] - ref["log_prob"]).max()),
                v=float(ev.max()))


@pytest.mark.parametrize("kind", KINDS)
def test_actor_critic_step_matches_fp64(kind):
    """One step at n = 65536 from random states with 5 % episode starts against fp64; the actor's state bit-identical
    to rdv_lstm_policy_step; every env independent of n (1, 127, 129, 1000, and 65459, where CTAs loop over several
    tile pairs and the last pair is ragged), of its position in the batch and of the state buffers' leading
    dimension."""
    from reinforcement_learning_rendezvous_b200 import LstmPolicy
    rng = np.random.default_rng(20)
    sd = make_state_dict(kind, seed=3)
    sd["log_std"] = rng.uniform(-1.5, 0.5, 6).astype(np.float32)
    m = _module(sd)
    obs = _observations(NMAX, rng)
    st = [rng.uniform(-1, 1, (NMAX, H)).astype(np.float32),
          (rng.standard_normal((NMAX, H)) * (4.0 if kind == "stress" else 1.0)).astype(np.float32),
          rng.uniform(-1, 1, (NMAX, H)).astype(np.float32), rng.standard_normal((NMAX, H)).astype(np.float32)]
    start = rng.random(NMAX) < 0.05
    dev = torch.device("cuda")
    obs_d = torch.as_tensor(obs, device=dev)
    start_d = torch.as_tensor(start.astype(np.uint8), device=dev)
    st_d = [torch.as_tensor(np.ascontiguousarray(x.T), device=dev) for x in st]
    full = _np(_step(m, obs_d, start_d, st_d))
    z, r = philox_normals_ref(SEED, OFFSET + np.arange(NMAX), STEP)
    ref = actor_critic_step_ref(sd, obs, st[0], st[1], st[2], st[3], start, z)
    worst = _assert_against_ref(full, ref, sd, z, r, kind)
    print(f"{kind}: |dh| {worst['h']:.2e}, actions {worst['a']:.2f} of the bound, |dlogp| {worst['lp']:.2e}, "
          f"values rel {worst['v']:.2e}")
    # the actor's LSTM state: the same bits as the deterministic actor step
    pol = LstmPolicy(actor_keys(sd))
    _, h1, c1 = pol.forward(obs_d, st_d[0], st_d[1], start_d)
    assert np.array_equal(h1.t().cpu().numpy(), full["h_pi"]) and np.array_equal(c1.t().cpu().numpy(), full["c_pi"])
    # independent of n and of the position: a prefix, and a slice run with its global env offset
    for n in (1, 127, 129, 1000, NMAX - 77):
        part = _np(_step(m, obs_d[:n], start_d[:n], [x[:, :n].contiguous() for x in st_d]))
        for k, v in part.items():
            assert np.array_equal(v, full[k][:n]), (n, k)
    # column slices of wider buffers (ld > n), NaN past column n: the same bits, nothing written past column n
    n, ld = 1000, 1333
    wide = [torch.full((H, ld), np.nan, device=dev) for _ in range(4)]
    for w_, x in zip(wide, st_d):
        w_[:, :n] = x[:, :n]
    out = _step(m, obs_d[:n], start_d[:n], [w_[:, :n] for w_ in wide], ld=ld)
    for k, v in _np(out).items():
        assert np.array_equal(v, full[k][:n]), ("ld", k)
    for o in out["states"]:
        assert o.stride(0) == ld and bool(o.as_strided((H, ld), (ld, 1))[:, n:].isnan().all())
    lo, n = 3000, 1000
    part = _np(_step(m, obs_d[lo:lo + n], start_d[lo:lo + n], [x[:, lo:lo + n].contiguous() for x in st_d],
                     offset=OFFSET + lo))
    for k, v in part.items():
        assert np.array_equal(v, full[k][lo:lo + n]), k
    perm = torch.as_tensor(rng.permutation(n), device=dev)
    shuf = _np(_step(m, obs_d[:n][perm], start_d[:n][perm], [x[:, :n][:, perm].contiguous() for x in st_d]))
    p = perm.cpu().numpy()
    for k in ("h_pi", "c_pi", "h_vf", "c_vf", "values"):
        assert np.array_equal(shuf[k], full[k][:n][p]), k
    # without env_actions the rest is unchanged
    noclip = _np(_step(m, obs_d[:n], start_d[:n], [x[:, :n].contiguous() for x in st_d], env_actions=False))
    assert np.isnan(noclip["env_actions"]).all() and np.array_equal(noclip["actions"], full["actions"][:n])


def test_argument_errors():
    from reinforcement_learning_rendezvous_b200 import _native as N
    from reinforcement_learning_rendezvous_b200.batched_env import _stream_ptr
    L = N.lib()
    m = _module(make_state_dict("ppo", seed=4))
    n, dev = 200, torch.device("cuda")
    obs = torch.zeros((n, 17), device=dev)
    start = torch.zeros(n, dtype=torch.uint8, device=dev)
    st = [torch.zeros((H, n), device=dev) for _ in range(8)]
    act, lp, val = torch.zeros((n, 6), device=dev), torch.zeros(n, device=dev), torch.zeros(n, device=dev)

    def call(w=None, n_=n, ld=n, **kw):
        p = dict(obs=obs.data_ptr(), episode_start=start.data_ptr(), h_pi=st[0].data_ptr(), c_pi=st[1].data_ptr(),
                 h_pi_out=st[2].data_ptr(), c_pi_out=st[3].data_ptr(), h_vf=st[4].data_ptr(), c_vf=st[5].data_ptr(),
                 h_vf_out=st[6].data_ptr(), c_vf_out=st[7].data_ptr(), actions=act.data_ptr(), env_actions=None,
                 log_prob=lp.data_ptr(), values=val.data_ptr(), action_seed=1, step_index=0, env_offset=0, ld=ld)
        p.update(kw)
        io = N.RdvLstmStepIO(**p)
        w = w or m.kernel_weights()
        return L.rdv_lstm_actor_critic_step(C.byref(w), C.byref(io), n_, _stream_ptr(dev))

    ERR_NULL, ERR_SIZE, ERR_ALIGN, ERR_UNSUPPORTED = -1, -2, -3, -6          # RdvStatus
    assert call() == 0
    assert L.rdv_lstm_actor_critic_step(None, None, n, None) == ERR_NULL
    assert call(obs=None) == ERR_NULL and call(values=None) == ERR_NULL and call(c_vf_out=None) == ERR_NULL
    w = m.kernel_weights()
    w.log_std = None
    assert call(w=w) == ERR_NULL
    w = m.kernel_weights()
    w.critic.w2 = None
    assert call(w=w) == ERR_NULL
    assert call(n_=-1) == ERR_SIZE and call(ld=n - 1) == ERR_SIZE
    assert call(h_vf=st[4].data_ptr() + 2) == ERR_ALIGN and call(env_actions=act.data_ptr() + 1) == ERR_ALIGN
    w = m.kernel_weights()
    w.critic.hidden = 128
    assert call(w=w) == ERR_UNSUPPORTED
    assert call(n_=0, ld=0) == 0
    torch.cuda.synchronize()


def _trainer(n=4096, **cfg):
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    from reinforcement_learning_rendezvous_b200.recurrent_ppo import RecurrentPPO, RecurrentPPOConfig
    env = BatchedRendezvousEnv(n, seed=7, auto_reset=True, t_max=12)
    return RecurrentPPO(env, RecurrentPPOConfig(**cfg))


def test_collection_teacher_forced_and_replayed():
    """Two collections of 4 steps: every recorded step against fp64 from its recorded inputs, and the recorded
    env_actions through a twin env with the same seed give the same observations, rewards and dones bit for bit."""
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    T = 4
    tr = _trainer(n_steps=T, n_evals=8)
    twin = BatchedRendezvousEnv(4096, seed=7, auto_reset=True, t_max=12)
    obs = twin.reset().clone()
    sd = {k: v.detach().cpu().numpy() for k, v in tr.policy.state_dict().items()}
    n = tr.env.num_envs
    for it in range(2):
        tr.collect()
        S = tr.states.cpu().numpy()
        for t in range(T):
            start = tr.buf_start[t].cpu().numpy().astype(bool)
            assert start.all() if (it == 0 and t == 0) else True
            z, r = philox_normals_ref(tr.action_seed, np.arange(n), it * T + t)
            ref = actor_critic_step_ref(sd, tr.buf_obs[t].cpu().numpy(), *(S[k, t].T for k in range(4)), start, z)
            got = dict(h_pi=S[0, t + 1].T, c_pi=S[1, t + 1].T, h_vf=S[2, t + 1].T, c_vf=S[3, t + 1].T,
                       actions=tr.buf_act[t].cpu().numpy(), env_actions=tr.buf_env_act[t].cpu().numpy(),
                       log_prob=tr.buf_logp[t].cpu().numpy(), values=tr.buf_val[t].cpu().numpy())
            _assert_against_ref(got, ref, sd, z, r, (it, t))
            assert torch.equal(tr.buf_obs[t], obs), (it, t)
            o, rew, done = twin.step(tr.buf_env_act[t].clone())
            assert torch.equal(rew.float(), tr.buf_rew[t]) and torch.equal(done.bool(), tr.buf_done[t]), (it, t)
            obs = o.clone()
        assert torch.equal(tr.obs, obs)
        # the bootstrap value: the critic on the last observation and states
        z, r = philox_normals_ref(tr.action_seed, np.arange(n), (it + 1) * T)
        ref = actor_critic_step_ref(sd, obs.cpu().numpy(), *(S[k, T].T for k in range(4)),
                                    tr.episode_start.cpu().numpy().astype(bool), z)
        ev = np.abs(tr.last_value.cpu().numpy() - ref["values"]) / np.maximum(1.0, np.abs(ref["values"]))
        assert ev.max() <= 1e-5


def test_update_first_minibatch_reproduces_the_recorded_step():
    """The update's first minibatch of the first epoch recomputes log-probabilities and values (torch LSTMs from the
    recorded states at the sequence starts) that agree with what the kernel recorded: the ratio is 1 to 1e-4."""
    from reinforcement_learning_rendezvous_b200.recurrent_ppo import plan_minibatches
    tr = _trainer(n_steps=16, batch_size=8192, n_evals=8)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    adv, ret = tr.collect()
    tr._flat_start = tr._flat(tr.buf_start)
    starts = tr._flat_start.cpu().numpy().astype(bool)
    assert starts.any() and not starts.all()
    plan = plan_minibatches(starts, 16, 8192, int(np.random.default_rng(0).integers(starts.size)))
    pad_d, first_d = torch.as_tensor(plan.pad, device=tr.device), torch.as_tensor(plan.seq_first, device=tr.device)
    data = (tr._flat(tr.buf_obs), tr._flat(tr.buf_act), tr._flat(tr.buf_logp), tr._flat(adv), tr._flat(ret),
            tr._flat(tr.buf_val))
    with torch.no_grad():
        mask, (obs, act, old_logp, a, r, val), states, start0 = tr._minibatch(data, plan, 0, pad_d, first_d)
        assert bool(start0.any()) and int(mask.shape[0]) > 1
        _, _, _, logp, value = tr._loss(mask, obs, act, old_logp, a, r, states, start0)
    dl = float((logp - old_logp[mask]).abs().max())
    dv = float(((value - val[mask]).abs() / val[mask].abs().clamp(min=1)).max())
    print(f"first minibatch: {int(mask.sum())} samples in {mask.shape[0]} sequences, |dlogp| {dl:.2e}, dv {dv:.2e}")
    assert dl <= 1e-4 and dv <= 1e-4


def test_short_training_run_learns_and_saves(tmp_path):
    """4,096 envs, a handful of iterations with a large batch: finite losses, num_timesteps adds up, the mean step
    reward rises; save() then LstmPolicy.load() acts like the torch actor; the rejections raise.  Measured on a B200
    (1000 W): mean step reward per iteration 3.348, 3.362, 3.380, 3.440, 3.455, 3.480 (last two minus first two: +0.112);
    the threshold asks for less than half of that gain."""
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, LstmPolicy, RendezvousVecEnv
    from reinforcement_learning_rendezvous_b200.recurrent_ppo import RecurrentPPO
    iters, T = 6, 32
    tr = _trainer(n_steps=T, batch_size=16384, n_epochs=4, learning_rate=1e-3, n_evals=16)
    tr.learn(iters * T * 4096, eval_every=3)
    log = tr.cfg.log
    rewards = [row["mean_step_reward"] for row in log]
    print("mean step reward per iteration:", [f"{x:.4f}" for x in rewards],
          "eval:", [row.get("eval_mean_return") for row in log])
    assert len(log) == iters and tr.num_timesteps == iters * T * 4096
    for row in log:
        assert np.isfinite([row["pg_loss"], row["value_loss"], row["entropy"]]).all(), row
    assert np.mean(rewards[-2:]) > np.mean(rewards[:2]) + REWARD_GAIN, rewards
    assert tr.best_state is not None and np.isfinite(tr.best_eval)
    # save / load: the deterministic actor of the saved model
    path = str(tmp_path / "rnn.npz")
    tr.best_state = None
    tr.save(path)
    pol = LstmPolicy.load(path)
    rng = np.random.default_rng(5)
    n = 512
    obs = torch.as_tensor(_observations(n, rng), device="cuda")
    h, c = pol.initial_state(n)
    act, _, _ = pol.forward(obs, h, c)
    with torch.no_grad():
        zeros = torch.zeros((1, n, H), device="cuda")
        out, _ = tr.policy.lstm_actor(obs[None], (zeros, zeros))
        ref = tr.policy.action_net(tr.policy.mlp_extractor.policy_net(out[0])).clamp(-1, 1)
    assert float((act - ref).abs().max()) <= 1e-5
    # rejections
    with pytest.raises(TypeError):
        RecurrentPPO(RendezvousVecEnv(8))
    with pytest.raises(ValueError):
        RecurrentPPO(BatchedRendezvousEnv(256, auto_reset=False))
    with torch.no_grad():
        tr.policy.lstm_critic.weight_hh_l0[3, 5] = 64.0
    with pytest.raises(ValueError, match="64"):
        tr.collect()


REWARD_GAIN = 0.05
