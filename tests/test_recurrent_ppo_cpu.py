"""CPU: RecurrentPPO's update semantics against sb3_contrib 1.6 restated in plain Python -- the minibatch planner
against ``RecurrentRolloutBuffer.get`` / ``_get_samples`` / ``create_sequencers`` (sequence starts, padding, mask,
initial-state indices), the single padded ``nn.LSTM`` call against ``_process_sequence``'s per-step loop -- and the
module's sb3_contrib parameter layout, initialisation and defaults."""
import numpy as np
import pytest
import torch

from lstm_ref import H, make_state_dict
from recurrent_ref import process_sequence_loop

from reinforcement_learning_rendezvous_b200 import _native as N
from reinforcement_learning_rendezvous_b200.recurrent_ppo import (RecurrentActorCritic, RecurrentPPO,
                                                                  RecurrentPPOConfig, plan_minibatches)


def sb3_get_samples(episode_starts, n_steps, batch_size, split_index):
    """sb3_contrib 1.6 ``RecurrentRolloutBuffer.get`` + ``_get_samples`` + ``create_sequencers`` + ``pad``, one
    minibatch at a time as the library does it.  ``episode_starts``: the env-major flattened flags.  Yields, per
    minibatch, (batch_inds, seq_start_indices (positions in the minibatch), padded index [n_seq, max_len] with -1
    for padding, mask [n_seq, max_len], initial-state indices (flat buffer indices of each sequence's first
    sample))."""
    total = len(episode_starts)
    indices = np.arange(total)
    indices = np.concatenate((indices[split_index:], indices[:split_index]))
    env_change = np.zeros((n_steps, total // n_steps))
    env_change[0, :] = 1.0
    env_change = env_change.swapaxes(0, 1).reshape(-1)                 # swap_and_flatten
    start_idx = 0
    while start_idx < total:
        batch_inds = indices[start_idx:start_idx + batch_size]
        seq_start = np.logical_or(np.asarray(episode_starts)[batch_inds], env_change[batch_inds]).flatten()
        seq_start[0] = True
        seq_start_indices = np.where(seq_start == True)[0]  # noqa: E712
        seq_end_indices = np.concatenate([(seq_start_indices - 1)[1:], np.array([len(batch_inds)])])
        seqs = [batch_inds[s:e + 1] for s, e in zip(seq_start_indices, seq_end_indices)]
        max_len = max(len(s) for s in seqs)
        padded = np.full((len(seqs), max_len), -1, dtype=np.int64)
        for i, s in enumerate(seqs):
            padded[i, :len(s)] = s
        yield batch_inds, seq_start_indices, padded, padded >= 0, batch_inds[seq_start_indices]
        start_idx += batch_size


def _starts(rng, n_envs, n_steps, p):
    """env-major flags as a collection leaves them: every env starts an episode at its first step of the first
    iteration (SB3's initial episode_start), then at random."""
    s = rng.random((n_envs, n_steps)) < p
    s[:, 0] |= rng.random(n_envs) < 0.5
    return s.reshape(-1)


@pytest.mark.parametrize("n_envs,n_steps,batch_size,p", [(4, 8, 8, 0.2), (5, 7, 6, 0.1), (16, 32, 100, 0.05),
                                                          (3, 16, 48, 0.0), (7, 13, 1000, 0.3), (6, 10, 1, 0.5)])
def test_planner_matches_sb3_contrib(n_envs, n_steps, batch_size, p):
    rng = np.random.default_rng(n_envs * 1000 + batch_size)
    for rep in range(4):
        starts = _starts(rng, n_envs, n_steps, p)
        split = int(rng.integers(starts.size))
        plan = plan_minibatches(starts, n_steps, batch_size, split)
        ref = list(sb3_get_samples(starts, n_steps, batch_size, split))
        assert plan.seq_lo.size == len(ref)
        covered = []
        for b, (batch_inds, seq_start, padded, mask, first) in enumerate(ref):
            lo, hi, L = plan.seq_lo[b], plan.seq_hi[b], plan.length[b]
            mine = plan.pad[plan.pad_lo[b]:plan.pad_lo[b] + (hi - lo) * L].reshape(hi - lo, L)
            assert mine.shape == padded.shape, (b, mine.shape, padded.shape)
            assert np.array_equal(mine, padded), b
            assert np.array_equal(mine >= 0, mask), b
            assert np.array_equal(plan.seq_first[lo:hi], first), b
            assert np.array_equal(mine[mine >= 0], batch_inds), b         # row-major padded order = minibatch order
            covered.append(batch_inds)
        assert np.array_equal(np.sort(np.concatenate(covered)), np.arange(starts.size))


def test_padded_lstm_equals_per_step_loop():
    """One nn.LSTM call over zero-padded sequences, the initial state zeroed at a sequence that starts an episode,
    equals sb3_contrib's per-step ``_process_sequence`` loop on the valid samples (padding only follows them)."""
    torch.manual_seed(0)
    rng = np.random.default_rng(1)
    torch.backends.cudnn.allow_tf32 = False
    lstm = torch.nn.LSTM(17, H).double()
    n_envs, n_steps = 9, 20
    starts = _starts(rng, n_envs, n_steps, 0.15)
    plan = plan_minibatches(starts, n_steps, 64, int(rng.integers(starts.size)))
    obs = torch.as_tensor(rng.uniform(-1, 1, (starts.size, 17)))
    states = torch.as_tensor(rng.standard_normal((2, starts.size, H)))
    flags = torch.as_tensor(starts.astype(np.float64))
    worst = 0.0
    for b in range(plan.seq_lo.size):
        lo, hi, L = plan.seq_lo[b], plan.seq_hi[b], plan.length[b]
        src = torch.as_tensor(plan.pad[plan.pad_lo[b]:plan.pad_lo[b] + (hi - lo) * L].reshape(hi - lo, L))
        mask = src >= 0
        x = obs[src.clamp(min=0)] * mask[..., None]
        first = torch.as_tensor(plan.seq_first[lo:hi])
        h0, c0 = states[0, first], states[1, first]
        with torch.no_grad():
            mine = RecurrentActorCritic._sequence(lstm, x, h0, c0, flags[first])
            ep = flags[src.clamp(min=0)] * mask                              # sb3 pads episode_starts with 0
            ref = process_sequence_loop(lstm, x.reshape(-1, 17), h0, c0, ep.reshape(-1)).reshape(hi - lo, L, H)
        worst = max(worst, float((mine[mask] - ref[mask]).abs().max()))
    assert worst <= 1e-6, worst


def test_module_layout_init_and_defaults():
    torch.manual_seed(3)
    m = RecurrentActorCritic()
    sd = m.state_dict()
    ref = make_state_dict("ppo", critic=True)
    assert set(sd) == set(ref), set(sd) ^ set(ref)
    for k, v in ref.items():
        assert tuple(sd[k].shape) == v.shape, k
    for name, gain in (("mlp_extractor.policy_net.2", 2.0), ("mlp_extractor.value_net.2", 2.0)):
        w = sd[name + ".weight"].double()
        assert torch.allclose(w @ w.T, gain * torch.eye(64, dtype=torch.float64), atol=1e-5), name
    for name, gain in (("mlp_extractor.policy_net.0", 2.0), ("action_net", 1e-4), ("value_net", 1.0)):
        w = sd[name + ".weight"].double()
        assert torch.allclose(w @ w.T, gain * torch.eye(w.shape[0], dtype=torch.float64), atol=1e-5 * gain), name
    for k, v in sd.items():
        if k.endswith(".bias") and not k.startswith("lstm"):
            assert not v.any(), k
    bound = 1.0 / np.sqrt(H)                                  # torch's LSTM init U(-1/sqrt(H), 1/sqrt(H))
    assert float(sd["lstm_actor.weight_hh_l0"].abs().max()) <= bound
    assert float(sd["lstm_critic.weight_ih_l0"].abs().max()) <= bound and float(sd["log_std"].abs().max()) == 0
    c = RecurrentPPOConfig()
    assert (c.learning_rate, c.n_steps, c.batch_size, c.n_epochs, c.clip_range, c.gamma, c.gae_lambda, c.ent_coef,
            c.vf_coef, c.max_grad_norm, c.normalize_advantage) == (3e-4, 128, 128, 10, 0.2, 0.99, 0.95, 0.0, 0.5, 0.5,
                                                                   True)


def test_check_weights_limit():
    """The collection step's weight check: the largest float32 below 65520 / 1024 passes, the limit itself, 64 and
    non-finite values raise, in the actor's and the critic's tensors alike."""
    assert N.LSTM_WEIGHT_LIMIT == 63.984375
    largest = float(np.nextafter(np.float32(N.LSTM_WEIGHT_LIMIT), np.float32(0)))
    m = RecurrentActorCritic()
    for p in (m.lstm_actor.weight_hh_l0, m.lstm_critic.weight_ih_l0, m.mlp_extractor.value_net[0].weight,
              m.action_net.weight):
        keep = p.detach().clone()
        with torch.no_grad():
            p[0, 1], p[-1, -1] = largest, -largest
        m.check_weights()
        for bad in (N.LSTM_WEIGHT_LIMIT, -N.LSTM_WEIGHT_LIMIT, 64.0, float("inf"), float("nan")):
            with torch.no_grad():
                p[0, 1] = bad
            with pytest.raises(ValueError, match="63.984375"):
                m.check_weights()
        with torch.no_grad():
            p.copy_(keep)
    m.check_weights()


def test_rejects_anything_but_a_batched_env():
    with pytest.raises(TypeError):
        RecurrentPPO(object())
