"""TEST CHECKER: fp64 numpy reference of one deterministic actor step of sb3_contrib's RecurrentPPO MlpLstmPolicy
(one 256-wide LSTM layer, the default pi = [64, 64] Tanh head, action_net, clip), and builders of state dicts with
sb3_contrib's key names (critic included) at the weight scales the tests use."""
import numpy as np

H = 256
OBS, ACT = 17, 6


def sigmoid(x):
    return 0.5 * (1.0 + np.tanh(0.5 * x))


def lstm_step_ref(sd, obs, h, c, episode_start=None):
    """obs [n, 17], h, c [n, 256] (env-major), episode_start [n] bool or None -> (actions [n, 6], h', c'), all fp64.
    The state is zeroed where episode_start is set, as sb3_contrib's ``(1 - episode_start) * state``."""
    w = {k: np.asarray(v, dtype=np.float64) for k, v in sd.items()}
    obs, h, c = (np.asarray(x, dtype=np.float64) for x in (obs, h, c))
    if episode_start is not None:
        keep = ~np.asarray(episode_start, dtype=bool).reshape(-1, 1)
        h, c = np.where(keep, h, 0.0), np.where(keep, c, 0.0)
    z = (obs @ w["lstm_actor.weight_ih_l0"].T + w["lstm_actor.bias_ih_l0"]
         + h @ w["lstm_actor.weight_hh_l0"].T + w["lstm_actor.bias_hh_l0"])
    zi, zf, zg, zo = np.split(z, 4, axis=1)                   # torch's gate order
    c2 = sigmoid(zf) * c + sigmoid(zi) * np.tanh(zg)
    h2 = sigmoid(zo) * np.tanh(c2)
    a = np.tanh(h2 @ w["mlp_extractor.policy_net.0.weight"].T + w["mlp_extractor.policy_net.0.bias"])
    a = np.tanh(a @ w["mlp_extractor.policy_net.2.weight"].T + w["mlp_extractor.policy_net.2.bias"])
    act = np.clip(a @ w["action_net.weight"].T + w["action_net.bias"], -1.0, 1.0)
    return act, h2, c2


def _split16(x):
    x = np.asarray(x, dtype=np.float32)
    hi = x.astype(np.float16).astype(np.float32)
    return hi, (x - hi).astype(np.float16).astype(np.float32)


def _mm_split(a, w, scale=2.0 ** 10):
    """a [n, k] @ w[m, k].T as the kernel computes it: w times 2^10, both split into fp16 hi / lo, the three products
    a_lo w_hi + a_hi w_lo + a_hi w_hi with float32 accumulation, scaled back."""
    ah, al = _split16(a)
    wh, wl = _split16(np.asarray(w, np.float32) * np.float32(scale))
    return ((al @ wh.T + ah @ wl.T + ah @ wh.T) * np.float32(1.0 / scale)).astype(np.float32)


def gates_split_emulation(sd, obs, h, episode_start=None, mm=_mm_split):
    """The gate pre-activations z [n, 4 * 256] (float32, torch's order i, f, g, o) as rdv_lstm_policy_step computes
    them: ``mm(a, w)`` the product of a = [obs | h] (h zeroed where episode_start is set) and w = [W_ih | W_hh], then
    b_ih + b_hh added in float32.  ``mm`` defaults to the kernel's three-product split (tests pass altered ones)."""
    w = {k: np.asarray(v, dtype=np.float32) for k, v in sd.items()}
    h = np.asarray(h, np.float32)
    if episode_start is not None:
        h = np.where(~np.asarray(episode_start, dtype=bool).reshape(-1, 1), h, 0).astype(np.float32)
    a = np.concatenate([np.asarray(obs, np.float32), h], axis=1)
    wcat = np.concatenate([w["lstm_actor.weight_ih_l0"], w["lstm_actor.weight_hh_l0"]], axis=1)
    return mm(a, wcat) + (w["lstm_actor.bias_ih_l0"] + w["lstm_actor.bias_hh_l0"])


def lstm_step_split_emulation(sd, obs, h, c, episode_start=None):
    """numpy emulation of rdv_lstm_policy_step's arithmetic (fp16 hi / lo operands, three products, float32
    accumulation and activations; numpy's float32 accumulation order, not the tensor core's), state only: (h', c')."""
    c = np.asarray(c, np.float32)
    if episode_start is not None:
        c = np.where(~np.asarray(episode_start, dtype=bool).reshape(-1, 1), c, 0).astype(np.float32)
    z = gates_split_emulation(sd, obs, h, episode_start)
    zi, zf, zg, zo = np.split(z, 4, axis=1)
    sig = lambda x: np.float32(1) / (np.float32(1) + np.exp(-x))
    c2 = (sig(zf) * c + sig(zi) * np.tanh(zg)).astype(np.float32)
    return (sig(zo) * np.tanh(c2)).astype(np.float32), c2


def _uniform(rng, shape, fan_in):
    bound = 1.0 / np.sqrt(fan_in)
    return rng.uniform(-bound, bound, shape)


def _orthogonal(rng, shape, gain):
    a = rng.standard_normal((max(shape), min(shape)))
    q, r = np.linalg.qr(a)
    q = q * np.sign(np.diag(r))
    return gain * (q if shape[0] >= shape[1] else q.T)[:shape[0], :shape[1]]


def make_state_dict(kind="torch", seed=0, critic=True):
    """A full RecurrentPPO MlpLstmPolicy state dict (float32 numpy arrays).
    kind: "torch"  -- torch's default init everywhere (LSTM and Linear: U(-1/sqrt(fan_in), 1/sqrt(fan_in)));
          "ppo"    -- the LSTM at torch's init, the head as PPO's ortho_init leaves it (orthogonal, gain sqrt(2) for
                      the hidden layers and 0.01 for action_net, zero biases);
          "stress" -- the torch init with the LSTM's weights and biases times 3 and the forget-gate biases + 3
                      (saturated gates and a long memory: |c| grows over the steps); the head stays at the torch init.
    critic adds what the actor ignores: lstm_critic.*, mlp_extractor.value_net.*, value_net.* and log_std."""
    rng = np.random.default_rng(seed)
    sd = {}
    for net in ("lstm_actor", "lstm_critic") if critic else ("lstm_actor",):
        sd[f"{net}.weight_ih_l0"] = _uniform(rng, (4 * H, OBS), H)
        sd[f"{net}.weight_hh_l0"] = _uniform(rng, (4 * H, H), H)
        sd[f"{net}.bias_ih_l0"] = _uniform(rng, (4 * H,), H)
        sd[f"{net}.bias_hh_l0"] = _uniform(rng, (4 * H,), H)
    if kind == "stress":
        for k in ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"):
            sd["lstm_actor." + k] = 3.0 * sd["lstm_actor." + k]
        sd["lstm_actor.bias_ih_l0"][H:2 * H] += 3.0
    heads = [("mlp_extractor.policy_net.0", (64, H), np.sqrt(2)), ("mlp_extractor.policy_net.2", (64, 64), np.sqrt(2)),
             ("action_net", (ACT, 64), 0.01)]
    if critic:
        heads += [("mlp_extractor.value_net.0", (64, H), np.sqrt(2)), ("mlp_extractor.value_net.2", (64, 64), np.sqrt(2)),
                  ("value_net", (1, 64), 1.0)]
    for name, shape, gain in heads:
        if kind == "ppo":
            sd[name + ".weight"], sd[name + ".bias"] = _orthogonal(rng, shape, gain), np.zeros(shape[0])
        else:
            sd[name + ".weight"], sd[name + ".bias"] = _uniform(rng, shape, shape[1]), _uniform(rng, shape[0], shape[1])
    if critic:
        sd["log_std"] = np.zeros(ACT)
    return {k: np.asarray(v, dtype=np.float32) for k, v in sd.items()}


def scale_state_dict(sd, s_lstm, s_head):
    """sd with every LSTM weight and bias (actor and critic) times s_lstm and every head weight and bias times s_head
    (float32).  A factor "max" is the largest that keeps that part's largest magnitude at 0.999 of the loaders' limit
    (``_native.LSTM_WEIGHT_LIMIT``)."""
    from reinforcement_learning_rendezvous_b200._native import LSTM_WEIGHT_LIMIT
    out = dict(sd)
    parts = (("lstm_",), ("mlp_extractor.", "action_net.", "value_net."))
    for s, prefixes in zip((s_lstm, s_head), parts):
        keys = [k for k in sd if k.startswith(prefixes)]
        if s == "max":
            s = 0.999 * LSTM_WEIGHT_LIMIT / max(float(np.abs(sd[k]).max()) for k in keys)
        for k in keys:
            out[k] = (np.asarray(sd[k], dtype=np.float64) * s).astype(np.float32)
    return out


def actor_keys(sd):
    return {k: v for k, v in sd.items()
            if k.startswith(("lstm_actor.", "mlp_extractor.policy_net.", "action_net."))}
