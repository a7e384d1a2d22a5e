"""GPU: both LSTM kernels -- rdv_lstm_policy_step (LstmPolicy.forward) and rdv_lstm_actor_critic_step -- against the
fp64 step over the weights and observations the loaders accept, every output of every env within its own error bound
(tests/lstm_bound.py): LSTM and head weights from 1e-3 times torch's init to just under the limit, weights at the
limit, observations from 1e-6 to beyond the clamp and non-finite, and one poisoned env per tile that leaves every other
env's bits alone.  Each case prints its worst error / bound per output."""
import numpy as np
import pytest
import torch

from lstm_bound import ratio, step_bound
from lstm_ref import H, actor_keys, make_state_dict, scale_state_dict
from normals import philox_normals_ref
from recurrent_ref import LOG_2PI, critic_as_actor
from test_gpu_lstm import _observations
from test_gpu_policy_shapes import EPS, Z_ULPS, noise_bound
from test_gpu_recurrent_ppo import OFFSET, SEED, STEP, _module, _np, _step

pytestmark = pytest.mark.gpu

N_ENVS = 8192
LOG_STDS = (-20.0, -1.0, 2.0)           # std 2e-9, 0.37, 7.4: at 7.4 the clip of env_actions acts on most draws
U = 2.0 ** -24


def _states(n, rng):
    """[h_pi, c_pi, h_vf, c_vf] env-major: h in (-1, 1), c ~ N(0, sigma) with sigma log-uniform in [0.1, 30] per env
    (trained cells carry long memories)."""
    out = []
    for _ in range(2):
        out.append(rng.uniform(-1, 1, (n, H)).astype(np.float32))
        sigma = np.exp(rng.uniform(np.log(0.1), np.log(30.0), (n, 1)))
        out.append((rng.standard_normal((n, H)) * sigma).astype(np.float32))
    return out


def _kernels(sd, obs, states, start):
    """Both kernels on env-major numpy inputs, env-major numpy outputs: "policy" -> actions, h_pi, c_pi of
    rdv_lstm_policy_step; each log_std of LOG_STDS -> the outputs of rdv_lstm_actor_critic_step with it.  Both loaders'
    weight checks pass first."""
    from reinforcement_learning_rendezvous_b200 import LstmPolicy
    dev = torch.device("cuda")
    obs_d, start_d = torch.as_tensor(obs, device=dev), torch.as_tensor(start.astype(np.uint8), device=dev)
    st_d = [torch.as_tensor(np.ascontiguousarray(x.T), device=dev) for x in states]
    act, h, c = LstmPolicy(actor_keys(sd)).forward(obs_d, st_d[0], st_d[1], start_d)
    out = {"policy": dict(actions=act.cpu().numpy(), h_pi=h.t().cpu().numpy(), c_pi=c.t().cpu().numpy())}
    for ls in LOG_STDS:
        m = _module(dict(sd, log_std=np.full(6, ls, np.float32)))
        m.check_weights()
        out[ls] = _np(_step(m, obs_d, start_d, st_d))
    return out


def _log_prob_bound(z, r, log_std):
    """|log_prob - fp64| allowed: the draw's own error (Z_ULPS, tests/test_gpu_policy_shapes.py) times |z|, and the
    float32 roundings of the six fmas, their sum and the constant 3 ln(2 pi)."""
    return (np.abs(z) * Z_ULPS * EPS * np.maximum(r, 1.0)).sum(1) + 8 * U * ((0.5 * z * z + abs(log_std)).sum(1) + 6)


def _compare(sd, obs, states, start, got, ids):
    """Worst error / bound per output of the kernels' outputs ``got`` (of :func:`_kernels`, rows = envs ``ids`` of the
    launch) against the fp64 step of the same inputs."""
    pi = step_bound(actor_keys(sd), obs, states[0], states[1], start, device="cuda")
    vf = step_bound(critic_as_actor(sd), obs, states[2], states[3], start, device="cuda")
    g = got["policy"]
    worst = dict(h_pi=ratio(g["h_pi"], pi["h"], pi["dh"]), c_pi=ratio(g["c_pi"], pi["c"], pi["dc"]),
                 actions=ratio(g["actions"], np.clip(pi["out"], -1, 1), pi["dout"]))
    z, r = philox_normals_ref(SEED, OFFSET + ids, STEP)
    for ls in LOG_STDS:
        g = got[ls]
        assert np.array_equal(g["h_pi"], got["policy"]["h_pi"]) and np.array_equal(g["c_pi"], got["policy"]["c_pi"])
        assert np.array_equal(g["env_actions"], np.clip(g["actions"], -1, 1)), ls
        draw = pi["out"] + np.exp(ls) * z
        case = dict(h_vf=ratio(g["h_vf"], vf["h"], vf["dh"]), c_vf=ratio(g["c_vf"], vf["c"], vf["dc"]),
                    values=ratio(g["values"], vf["out"][:, 0], vf["dout"][:, 0]),
                    draw=ratio(g["actions"], draw, pi["dout"] + noise_bound(ls, z, r, g["actions"], False)),
                    log_prob=ratio(g["log_prob"], (-0.5 * z * z - ls).sum(1) - 3 * LOG_2PI, _log_prob_bound(z, r, ls)))
        worst.update({k: max(v, worst.get(k, 0.0)) for k, v in case.items()})
    return worst


def _check(sd, obs, states, start, what):
    """Both kernels on these inputs, every output within its bound; prints the worst error / bound per output."""
    got = _kernels(sd, obs, states, start)
    worst = _compare(sd, obs, states, start, got, np.arange(obs.shape[0]))
    print(f"{what}: worst error / bound " + ", ".join(f"{k} {v:.3f}" for k, v in worst.items()))
    assert max(worst.values()) <= 1.0, (what, worst)
    return got


# (LSTM scale, head scale) times torch's init; "max": the largest magnitude at 0.999 of the loaders' limit
SWEEP = [(1e-3, 1.0), (0.1, 1.0), (1.0, 1.0), (30.0, 1.0), ("max", 1.0), (1.0, 1e-3), (1.0, 30.0), (1.0, "max"),
         (1e-3, 1e-3), (1e-3, "max"), ("max", 1e-3), ("max", "max")]


@pytest.mark.parametrize("s_lstm,s_head", SWEEP, ids=[f"lstm{a}-head{b}" for a, b in SWEEP])
def test_weight_scale_sweep(s_lstm, s_head):
    """8,192 envs of golden and Box observations from random states, 5 % episode starts: both kernels within the
    bound, the actor-critic step at each log_std."""
    rng = np.random.default_rng(30)
    sd = scale_state_dict(make_state_dict("torch", seed=4), s_lstm, s_head)
    _check(sd, _observations(N_ENVS, rng), _states(N_ENVS, rng), rng.random(N_ENVS) < 0.05,
           f"LSTM x{s_lstm}, head x{s_head}")


def test_weights_at_the_limit():
    """The largest float32 the loaders accept (63.984371), with both signs, in entries of W_ih, W_hh, W0, W1 and W2 of
    both networks: finite outputs within the bound.  From 63.984375 on, fp16 rounds the staged hi half to infinity and
    the outputs would be NaN."""
    from reinforcement_learning_rendezvous_b200._native import LSTM_WEIGHT_LIMIT
    big = np.nextafter(np.float32(LSTM_WEIGHT_LIMIT), np.float32(0))
    rng = np.random.default_rng(31)
    sd = make_state_dict("torch", seed=6)
    for lstm, head, out in (("lstm_actor", "policy_net", "action_net"), ("lstm_critic", "value_net", "value_net")):
        for name in (f"{lstm}.weight_ih_l0", f"{lstm}.weight_hh_l0", f"mlp_extractor.{head}.0.weight",
                     f"mlp_extractor.{head}.2.weight", f"{out}.weight"):
            w = sd[name].copy()
            w.flat[rng.choice(w.size, 2, replace=False)] = (big, -big)
            sd[name] = w
    got = _check(sd, _observations(N_ENVS, rng), _states(N_ENVS, rng), rng.random(N_ENVS) < 0.05,
                 "weights at the limit")
    for outputs in got.values():
        for k, v in outputs.items():
            assert np.isfinite(v).all(), k


def test_observation_range():
    """Observations x1e-6 (their lo half an fp16 subnormal), x1e-3, x30 and x3000 against the fp64 step; x1e7 and
    +-inf against the fp64 step of the input clamped to +-60000, and a NaN component as -60000 (fmaxf drops the NaN),
    as include/rdv_b200.h states (lstm_bound.staged_obs)."""
    rng = np.random.default_rng(32)
    sd = make_state_dict("torch", seed=7)
    n = 2048
    base, states, start = _observations(n, rng), _states(n, rng), rng.random(n) < 0.05
    for scale in (1e-6, 1e-3, 30.0, 3000.0, 1e7):
        _check(sd, base * np.float32(scale), states, start, f"observations x{scale:g}")
    odd = base.copy()
    odd[0::4, 3], odd[1::4, 5], odd[2::4, 11] = np.inf, -np.inf, np.nan
    odd[3::4, 0], odd[3::4, 16] = np.nan, -np.inf
    _check(sd, odd, states, start, "observations +-inf and NaN")


def test_one_poisoned_env_per_tile():
    """In every 128-env tile (11, the last one ragged) one env without an episode start gets a NaN observation
    component, a non-finite h (NaN in the actor's, +inf in the critic's) or an infinite c.  Every other env's outputs,
    the critic's included, keep the bits of the clean run.  The NaN observation gives the bits of -60000 in its place.
    The non-finite h gives NaN states, NaN draws and values, actions and env_actions of -1 (the clip takes NaN to -1)
    and the clean log-probability.  The infinite c gives that unit an infinite c' of its sign and every other output
    within the bound of the fp64 step."""
    n = 11 * 128 - 51
    rng = np.random.default_rng(33)
    sd = make_state_dict("torch", seed=8)
    obs, states, start = _observations(n, rng), _states(n, rng), rng.random(n) < 0.05
    tiles = np.arange(-(-n // 128))
    victim = np.minimum(128 * tiles + (37 * tiles) % 128, n - 1)
    start[victim] = False
    v_obs, v_h, v_c = victim[tiles % 3 == 0], victim[tiles % 3 == 1], victim[tiles % 3 == 2]
    unit = 77
    clean_obs, bad_obs = obs.copy(), obs.copy()
    clean_obs[v_obs, 4], bad_obs[v_obs, 4] = -60000.0, np.nan
    bad = [x.copy() for x in states]
    bad[0][v_h, unit], bad[2][v_h, unit] = np.nan, np.inf
    bad[1][v_c, unit], bad[3][v_c, unit] = np.inf, -np.inf
    clean = _kernels(sd, clean_obs, states, start)
    got = _kernels(sd, bad_obs, bad, start)
    rest = np.setdiff1d(np.arange(n), np.concatenate([v_h, v_c]))
    for key, outputs in clean.items():
        for k, v in outputs.items():
            assert np.array_equal(got[key][k][rest], v[rest]), (key, k)
    # non-finite h: NaN everywhere but the clipped actions and the log-probability, which does not depend on the network
    assert (got["policy"]["actions"][v_h] == -1).all()
    for key in ("policy",) + LOG_STDS:
        assert all(np.isnan(got[key][k][v_h]).all() for k in ("h_pi", "c_pi")), key
    for ls in LOG_STDS:
        g = got[ls]
        assert all(np.isnan(g[k][v_h]).all() for k in ("h_vf", "c_vf", "actions", "values")), ls
        assert (g["env_actions"][v_h] == -1).all() and np.array_equal(g["log_prob"][v_h], clean[ls]["log_prob"][v_h])
    # infinite c: the fp64 step of the same inputs
    assert (got["policy"]["c_pi"][v_c, unit] == np.inf).all() and all((got[ls]["c_vf"][v_c, unit] == -np.inf).all()
                                                                       for ls in LOG_STDS)
    rows = {key: {k: v[v_c] for k, v in outputs.items()} for key, outputs in got.items()}
    worst = _compare(sd, bad_obs[v_c], [x[v_c] for x in bad], start[v_c], rows, v_c)
    print("infinite c: worst error / bound " + ", ".join(f"{k} {v:.3f}" for k, v in worst.items()))
    assert max(worst.values()) <= 1.0, worst
