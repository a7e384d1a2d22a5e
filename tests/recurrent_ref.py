"""TEST CHECKER: fp64 numpy reference of one collection step of sb3_contrib's RecurrentPPO MlpLstmPolicy (actor and
critic LSTM, the sampled Gaussian head with its log-probability, the value head), built on tests/lstm_ref.py, and
sb3_contrib 1.6's per-step ``_process_sequence`` loop."""
import numpy as np
import torch

from lstm_ref import ACT, H, lstm_step_ref

LOG_2PI = np.log(2.0 * np.pi)


def critic_as_actor(sd):
    """The critic's weights under the actor's key names (its value_net in place of action_net), so that
    lstm_step_ref computes the critic's LSTM step."""
    ren = {"lstm_critic.": "lstm_actor.", "mlp_extractor.value_net.": "mlp_extractor.policy_net.",
           "value_net.": "action_net."}
    out = {}
    for k, v in sd.items():
        for a, b in ren.items():
            if k.startswith(a):
                out[b + k[len(a):]] = v
    return out


def _head(sd, prefix, out, h2):
    w = {k: np.asarray(v, dtype=np.float64) for k, v in sd.items()}
    a = np.tanh(h2 @ w[prefix + ".0.weight"].T + w[prefix + ".0.bias"])
    a = np.tanh(a @ w[prefix + ".2.weight"].T + w[prefix + ".2.bias"])
    return a @ w[out + ".weight"].T + w[out + ".bias"]


def actor_critic_step_ref(sd, obs, h_pi, c_pi, h_vf, c_vf, start, z):
    """One step of RecurrentActorCriticPolicy.forward in fp64: env-major inputs ([n, 17], states [n, 256], start [n]
    bool, z [n, 6] the noise).  Returns a dict: mean (unclipped), actions = mean + exp(log_std) z, log_prob of the draw,
    values, and the four next states."""
    _, h_pi2, c_pi2 = lstm_step_ref(sd, obs, h_pi, c_pi, start)
    _, h_vf2, c_vf2 = lstm_step_ref(critic_as_actor(sd), obs, h_vf, c_vf, start)
    log_std = np.asarray(sd["log_std"], dtype=np.float64)
    mean = _head(sd, "mlp_extractor.policy_net", "action_net", h_pi2)
    values = _head(sd, "mlp_extractor.value_net", "value_net", h_vf2)[:, 0]
    z = np.asarray(z, dtype=np.float64)
    return dict(mean=mean, actions=mean + np.exp(log_std) * z,
                log_prob=(-0.5 * z * z - log_std).sum(axis=1) - 0.5 * ACT * LOG_2PI, values=values,
                h_pi=h_pi2, c_pi=c_pi2, h_vf=h_vf2, c_vf=c_vf2)


def process_sequence_loop(lstm, features, h0, c0, episode_starts):
    """sb3_contrib's ``_process_sequence`` with its per-step loop: features [n_seq * L, in] (padded sequences
    flattened), initial states [n_seq, H], episode_starts [n_seq * L].  Returns [n_seq * L, H]."""
    n_seq = h0.shape[0]
    seq = features.reshape((n_seq, -1, lstm.input_size)).swapaxes(0, 1)
    starts = episode_starts.reshape((n_seq, -1)).swapaxes(0, 1)
    states = (h0[None], c0[None])
    out = []
    for x, s in zip(seq, starts):
        keep = (1.0 - s).view(1, n_seq, 1)
        hidden, states = lstm(x.unsqueeze(dim=0), (keep * states[0], keep * states[1]))
        out.append(hidden)
    return torch.flatten(torch.cat(out).transpose(0, 1), start_dim=0, end_dim=1)


__all__ = ["H", "LOG_2PI", "actor_critic_step_ref", "critic_as_actor", "process_sequence_loop"]
