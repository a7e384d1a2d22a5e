"""RecurrentPPO training loop on device tensors -- what ``main_rnn.py`` does through sb3_contrib's
``RecurrentPPO("MlpLstmPolicy")`` (one 256-unit LSTM per network, the default 64-64 Tanh heads), for the case where
sb3_contrib is not installed (it is not part of this image).  Collection, the recurrent minibatches and the update
follow sb3_contrib 1.6:

* collection (``collect_rollouts``): per step ONE ``rdv_lstm_actor_critic_step`` launch -- actor and critic LSTM steps
  on the tensor cores, the Gaussian draw, its clip, its log-probability and the value -- and one ``env.step``; the
  LSTM states live in ``[T + 1][256][N]`` buffers, step t reading slice t and writing slice t + 1, so the buffer's
  per-step state record (the input states of each step, before the episode-start reset) costs no copy;
* the update (``RecurrentRolloutBuffer.get`` / ``_get_samples`` / ``create_sequencers`` and ``RecurrentPPO.train``):
  env-major flattening, a random rotation per epoch, contiguous minibatches cut into sequences at episode starts, at
  each env's first step and at the minibatch's first sample, zero-padded to the longest, both LSTMs re-run from the
  recorded states, masked losses, gradient clipping and Adam -- planned on the host from one read-back of the
  episode-start flags per iteration, gathered on the device, eager (the sequence lengths vary per minibatch);
* ``evaluate``: the callback's deterministic evaluation through ``evaluate_batch`` with an :class:`LstmPolicy` of the
  current actor.

The module has sb3_contrib's parameter names, so :meth:`RecurrentPPO.save` writes what :meth:`LstmPolicy.load` (and,
as a ``policy.pth``, sb3_contrib) reads.
"""
from __future__ import annotations

import ctypes as C
import time
from dataclasses import dataclass, field
from typing import Optional

import numpy as np
import torch
from torch import nn

from . import _native as N
from .batched_env import BatchedRendezvousEnv, _stream_ptr
from .policy import LstmPolicy
from .ppo import gae


class _Extractor(nn.Module):
    def __init__(self, hidden, net):
        super().__init__()
        self.policy_net = nn.Sequential(nn.Linear(hidden, net), nn.Tanh(), nn.Linear(net, net), nn.Tanh())
        self.value_net = nn.Sequential(nn.Linear(hidden, net), nn.Tanh(), nn.Linear(net, net), nn.Tanh())


class RecurrentActorCritic(nn.Module):
    """sb3_contrib's ``RecurrentActorCriticPolicy`` ("MlpLstmPolicy") with one 256-unit LSTM for the actor and a separate
    one for the critic (its defaults), the 64-64 Tanh heads and a state-independent ``log_std``: the same parameter
    names and shapes as its checkpoint.  Initialised as sb3_contrib does: the heads orthogonal (gain sqrt(2) for the
    hidden layers, 0.01 for ``action_net``, 1 for ``value_net``, zero biases), the LSTMs at torch's default."""

    def __init__(self, obs_dim=17, act_dim=6, hidden=256, net=64, log_std_init=0.0):
        super().__init__()
        self.lstm_actor = nn.LSTM(obs_dim, hidden)
        self.lstm_critic = nn.LSTM(obs_dim, hidden)
        self.mlp_extractor = _Extractor(hidden, net)
        self.action_net = nn.Linear(net, act_dim)
        self.value_net = nn.Linear(net, 1)
        self.log_std = nn.Parameter(torch.full((act_dim,), float(log_std_init)))
        for module, gain in ((self.mlp_extractor, np.sqrt(2)), (self.action_net, 0.01), (self.value_net, 1.0)):
            for m in module.modules():
                if isinstance(m, nn.Linear):
                    nn.init.orthogonal_(m.weight, gain=gain)
                    nn.init.zeros_(m.bias)

    def _nets(self):
        ex = self.mlp_extractor
        return ((self.lstm_actor, ex.policy_net, self.action_net), (self.lstm_critic, ex.value_net, self.value_net))

    def kernel_weights(self) -> N.RdvLstmActorCritic:
        """The ``RdvLstmActorCritic`` of this module: pointers to its own parameters (no copy; in-place optimiser steps
        are seen by the next launch)."""
        for p in self.parameters():
            if p.dtype != torch.float32 or not p.is_cuda or not p.is_contiguous():
                raise ValueError("the kernel reads float32 contiguous CUDA parameters")

        def net(lstm, mlp, out):
            return N.RdvLstmPolicy(lstm.weight_ih_l0.data_ptr(), lstm.weight_hh_l0.data_ptr(),
                                   lstm.bias_ih_l0.data_ptr(), lstm.bias_hh_l0.data_ptr(), mlp[0].weight.data_ptr(),
                                   mlp[0].bias.data_ptr(), mlp[2].weight.data_ptr(), mlp[2].bias.data_ptr(),
                                   out.weight.data_ptr(), out.bias.data_ptr(), lstm.hidden_size, 0)
        pi, vf = self._nets()
        return N.RdvLstmActorCritic(net(*pi), self.log_std.data_ptr(), net(*vf))

    def check_weights(self):
        """Raise unless every parameter the kernel reads is finite and below ``LSTM_WEIGHT_LIMIT`` in magnitude (one
        device reduction and one read-back)."""
        limit = N.LSTM_WEIGHT_LIMIT
        worst = float(torch.stack([p.detach().abs().max() for p in self.parameters()]).max())
        if not worst < limit:
            bad = [k for k, p in self.named_parameters() if not float(p.detach().abs().max()) < limit]
            raise ValueError(f"parameters {bad} have entries of magnitude >= {limit} (64 - 1/64) or non-finite ones; "
                             "the LSTM kernel stages the weights times 2^10 in fp16 halves")

    @staticmethod
    def _sequence(lstm, obs, h0, c0, start0):
        """sb3_contrib's ``_process_sequence`` on padded sequences: obs [n_seq, L, 17], initial states [n_seq, 256],
        start0 [n_seq] the episode-start flag of each sequence's first sample.  Inside a sequence only its first sample
        can start an episode, so zeroing the initial state there and one LSTM call over the padded batch is the same
        as sb3_contrib's per-step loop.  Returns the outputs [n_seq, L, 256]."""
        keep = (1.0 - start0.to(obs.dtype))[None, :, None]
        out, _ = lstm(obs.transpose(0, 1), (keep * h0[None], keep * c0[None]))
        return out.transpose(0, 1)

    def evaluate_sequences(self, obs, states, start0):
        """Padded sequences -> (mean, values) [n_seq, L, 6] and [n_seq, L]; states = (h_pi, c_pi, h_vf, c_vf) at the
        sequences' first samples, each [n_seq, 256]."""
        (lpi, mpi, out_pi), (lvf, mvf, out_vf) = self._nets()
        mean = out_pi(mpi(self._sequence(lpi, obs, states[0], states[1], start0)))
        value = out_vf(mvf(self._sequence(lvf, obs, states[2], states[3], start0))).squeeze(-1)
        return mean, value

    def distribution(self, mean):
        return torch.distributions.Normal(mean, self.log_std.exp().expand_as(mean), validate_args=False)

    def to_lstm_policy(self, device) -> LstmPolicy:
        sd = {k: v.detach().float().cpu().numpy() for k, v in self.state_dict().items()}
        return LstmPolicy(sd, device=device)


@dataclass
class MinibatchPlan:
    """The minibatches of one epoch (see :func:`plan_minibatches`).  Minibatch b holds sequences
    ``seq_lo[b] .. seq_hi[b] - 1`` and their padded samples ``pad[pad_lo[b] : pad_lo[b] + n_seq * length[b]]``
    ([n_seq, length] row-major: the flat buffer index of each sample, -1 for padding); ``seq_first`` is the flat
    buffer index of every sequence's first sample (where its initial states and episode-start flag are read)."""
    pad: np.ndarray
    seq_first: np.ndarray
    seq_lo: np.ndarray
    seq_hi: np.ndarray
    pad_lo: np.ndarray
    length: np.ndarray


def plan_minibatches(episode_starts: np.ndarray, n_steps: int, batch_size: int, split_index: int) -> MinibatchPlan:
    """sb3_contrib 1.6's ``RecurrentRolloutBuffer.get`` for one epoch, vectorised.  ``episode_starts``: flags of the
    flattened buffer, env-major (index ``env * n_steps + t``).  The indices are rotated by ``split_index`` and cut
    into contiguous minibatches of ``batch_size`` (the last one shorter when it does not divide the buffer); inside a
    minibatch a sequence starts at an episode start, at t = 0 of an env and at the minibatch's first sample
    (``create_sequencers``), and sequences are zero-padded to the minibatch's longest (``pad``)."""
    starts = np.asarray(episode_starts, dtype=bool).reshape(-1)
    total = starts.size
    idx = np.concatenate([np.arange(split_index, total), np.arange(split_index)])
    pos = np.arange(total)
    mb = pos // batch_size
    flag = starts[idx] | (idx % n_steps == 0) | (pos % batch_size == 0)
    first_pos = np.flatnonzero(flag)
    seq_id = np.cumsum(flag) - 1
    seq_len = np.diff(np.append(first_pos, total))
    seq_mb = mb[first_pos]
    n_mb = int(mb[-1]) + 1
    seq_lo = np.searchsorted(seq_mb, np.arange(n_mb))
    seq_hi = np.append(seq_lo[1:], first_pos.size)
    length = np.maximum.reduceat(seq_len, seq_lo)
    n_pad = (seq_hi - seq_lo) * length
    pad_lo = np.concatenate([[0], np.cumsum(n_pad)[:-1]])
    pad = np.full(int(n_pad.sum()), -1, dtype=np.int64)
    where = pad_lo[mb] + (seq_id - seq_lo[mb]) * length[mb] + (pos - first_pos[seq_id])
    pad[where] = idx
    return MinibatchPlan(pad, idx[first_pos], seq_lo, seq_hi, pad_lo, length)


@dataclass
class RecurrentPPOConfig:
    """sb3_contrib ``RecurrentPPO``'s defaults.  Of main_rnn.py's own settings this repository records only the
    256-unit LSTM (SURVEY.md §2), so every hyper-parameter is a field to set.  ``n_steps`` is per env; with thousands
    of envs callers normally raise ``batch_size`` with the buffer (the default 128 over 16,384 envs x 128 steps would
    be 16,384 optimiser steps per epoch)."""
    n_steps: int = 128
    batch_size: int = 128
    n_epochs: int = 10
    learning_rate: float = 3e-4
    clip_range: float = 0.2
    gamma: float = 0.99
    gae_lambda: float = 0.95
    ent_coef: float = 0.0
    vf_coef: float = 0.5
    max_grad_norm: float = 0.5
    normalize_advantage: bool = True
    n_evals: int = 50                 # custom_callbacks.py: n_evals
    seed: int = 0
    log: list = field(default_factory=list)


class RecurrentPPO:
    """``env``: an auto-resetting :class:`BatchedRendezvousEnv`.  Collection through a ``RendezvousVecEnv`` is not
    provided: with sb3_contrib installed, ``make_vec_env`` + ``sb3_contrib.RecurrentPPO`` already does that.

    Memory: besides the rollout buffers, the four LSTM state records take 4 (T + 1) 256 N 4 bytes (8.7 GB at N =
    16,384 envs and T = 128 steps)."""

    def __init__(self, env, config: Optional[RecurrentPPOConfig] = None, policy: Optional[RecurrentActorCritic] = None):
        if not isinstance(env, BatchedRendezvousEnv):
            raise TypeError("RecurrentPPO collects from a BatchedRendezvousEnv; for a VecEnv use sb3_contrib's "
                            "RecurrentPPO with make_vec_env")
        if not env.auto_reset:
            raise ValueError("training needs an auto-resetting env")
        self.env, self.cfg = env, config or RecurrentPPOConfig()
        self.device = dev = env.device
        self.lib = N.lib()
        torch.manual_seed(self.cfg.seed)
        self._rng = np.random.default_rng(self.cfg.seed)
        self.policy = (policy or RecurrentActorCritic()).to(dev)
        self.optimizer = torch.optim.Adam(self.policy.parameters(), lr=self.cfg.learning_rate, eps=1e-5)
        n, T, H = env.num_envs, self.cfg.n_steps, N.LSTM_HIDDEN
        self.buf_obs = torch.empty((T, n, N.OBS_DIM), dtype=torch.float32, device=dev)
        self.buf_act = torch.empty((T, n, N.ACT_DIM), dtype=torch.float32, device=dev)
        self.buf_env_act = torch.empty((T, n, N.ACT_DIM), dtype=torch.float32, device=dev)
        self.buf_logp = torch.empty((T, n), dtype=torch.float32, device=dev)
        self.buf_val = torch.empty((T, n), dtype=torch.float32, device=dev)
        self.buf_rew = torch.empty((T, n), dtype=torch.float32, device=dev)
        self.buf_done = torch.empty((T, n), dtype=torch.bool, device=dev)
        self.buf_start = torch.empty((T, n), dtype=torch.uint8, device=dev)
        # h_pi, c_pi, h_vf, c_vf: slice t = the input states of step t (before its episode-start reset)
        self.states = torch.zeros((4, T + 1, H, n), dtype=torch.float32, device=dev)
        self._scratch = (torch.empty((4, H, n), dtype=torch.float32, device=dev),
                         torch.empty((n, N.ACT_DIM), dtype=torch.float32, device=dev),
                         torch.empty(n, dtype=torch.float32, device=dev))
        self.last_value = torch.empty(n, dtype=torch.float32, device=dev)
        self.obs = env.reset().clone()
        self.episode_start = torch.ones(n, dtype=torch.uint8, device=dev)      # SB3 starts with every env starting
        self.action_seed = self.cfg.seed + 977
        self.num_timesteps = 0
        self._noise_step = 0
        self.best_eval = -float("inf")
        self.best_state = None
        kw = dict(env.ctor_kwargs)
        self.eval_env = BatchedRendezvousEnv(self.cfg.n_evals, device=dev, seed=env.seed + 12345, auto_reset=False, **kw)

    # -- one collection step (RecurrentActorCriticPolicy.forward) ----------------------------------------------
    def _step(self, w, obs, start, states_in, states_out, actions, env_actions, log_prob, values):
        n = self.env.num_envs
        io = N.RdvLstmStepIO(obs.data_ptr(), start.data_ptr(), *(x.data_ptr() for x in (
            states_in[0], states_in[1], states_out[0], states_out[1], states_in[2], states_in[3], states_out[2],
            states_out[3], actions)), env_actions.data_ptr() if env_actions is not None else None,
            log_prob.data_ptr(), values.data_ptr(), self.action_seed, self._noise_step, self.env.env_offset, n)
        with torch.cuda.device(self.device):
            N.check(self.lib.rdv_lstm_actor_critic_step(C.byref(w), C.byref(io), n, _stream_ptr(self.device)),
                    "rdv_lstm_actor_critic_step")

    # -- rollout collection (RecurrentPPO.collect_rollouts) -----------------------------------------------------
    @torch.no_grad()
    def collect(self):
        """T steps of every env; returns GAE's (advantages, returns) [T, N]."""
        env, T, S = self.env, self.cfg.n_steps, self.states
        self.policy.check_weights()
        w = self.policy.kernel_weights()
        S[:, 0].copy_(S[:, T])                  # the last iteration's final states (zeros before the first)
        for t in range(T):
            self.buf_obs[t].copy_(self.obs)
            self.buf_start[t].copy_(self.episode_start)
            self._step(w, self.buf_obs[t], self.buf_start[t], S[:, t], S[:, t + 1], self.buf_act[t],
                       self.buf_env_act[t], self.buf_logp[t], self.buf_val[t])
            self._noise_step += 1
            obs, rew, done = env.step(self.buf_env_act[t])
            self.buf_rew[t].copy_(rew)
            self.buf_done[t].copy_(done)
            self.obs, self.episode_start = obs, done
        self.obs, self.episode_start = self.obs.clone(), self.episode_start.clone()
        # the bootstrap value: the same launch on the last observation, its actions and next states discarded
        scratch, act, logp = self._scratch
        self._step(w, self.obs, self.episode_start, S[:, T], scratch, act, None, logp, self.last_value)
        self.num_timesteps += T * env.num_envs
        return gae(self.buf_rew, self.buf_val, self.buf_done, self.last_value, self.cfg.gamma, self.cfg.gae_lambda)

    # -- sequence-minibatch update (RecurrentPPO.train) ---------------------------------------------------------
    def _flat(self, x):
        """[T, N, ...] -> [N T, ...] env-major (index env * T + t), as sb3_contrib's swap_and_flatten."""
        return x.transpose(0, 1).reshape(-1, *x.shape[2:])

    def _minibatch(self, data, plan, b, pad_d, first_d):
        """The padded tensors of minibatch b: (mask [n_seq, L] bool, then every buffer in ``data`` gathered and
        zero-padded, then the four initial states [n_seq, 256] and the first samples' episode-start flags)."""
        lo, hi, L = int(plan.seq_lo[b]), int(plan.seq_hi[b]), int(plan.length[b])
        p0 = int(plan.pad_lo[b])
        src = pad_d[p0:p0 + (hi - lo) * L].view(hi - lo, L)
        mask = src >= 0
        src = src.clamp(min=0)
        out = [x[src] * mask.view(hi - lo, L, *([1] * (x.dim() - 1))).to(x.dtype) for x in data]
        first = first_d[lo:hi]
        env, t = first // self.cfg.n_steps, first % self.cfg.n_steps
        states = tuple(self.states[k, t, :, env] for k in range(4))
        return mask, out, states, self._flat_start[first]

    def _loss(self, mask, obs, act, old_logp, adv, ret, states, start0):
        cfg = self.cfg
        mean, value = self.policy.evaluate_sequences(obs, states, start0)
        mean, value, act, old_logp, adv, ret = (x[mask] for x in (mean, value, act, old_logp, adv, ret))
        dist = self.policy.distribution(mean)
        logp = dist.log_prob(act).sum(-1)
        if cfg.normalize_advantage:
            adv = (adv - adv.mean()) / (adv.std() + 1e-8)
        ratio = (logp - old_logp).exp()
        pg_loss = -torch.min(adv * ratio, adv * ratio.clamp(1 - cfg.clip_range, 1 + cfg.clip_range)).mean()
        v_loss = ((ret - value) ** 2).mean()
        ent_loss = -dist.entropy().sum(-1).mean()
        return pg_loss, v_loss, ent_loss, logp, value

    def update(self, adv, ret):
        cfg, T, dev = self.cfg, self.cfg.n_steps, self.device
        data = (self._flat(self.buf_obs), self._flat(self.buf_act), self._flat(self.buf_logp), self._flat(adv),
                self._flat(ret))
        self._flat_start = self._flat(self.buf_start)
        starts = self._flat_start.cpu().numpy().astype(bool)          # the one read-back of the episode starts
        total = starts.size
        stats = ()
        for _ in range(cfg.n_epochs):
            plan = plan_minibatches(starts, T, cfg.batch_size, int(self._rng.integers(total)))
            pad_d = torch.from_numpy(plan.pad).to(dev, non_blocking=True)
            first_d = torch.from_numpy(plan.seq_first).to(dev, non_blocking=True)
            for b in range(plan.seq_lo.size):
                mask, (obs, act, old_logp, a, r), states, start0 = self._minibatch(data, plan, b, pad_d, first_d)
                pg, vl, ent, _, _ = self._loss(mask, obs, act, old_logp, a, r, states, start0)
                loss = pg + cfg.ent_coef * ent + cfg.vf_coef * vl
                self.optimizer.zero_grad(set_to_none=True)
                loss.backward()
                nn.utils.clip_grad_norm_(self.policy.parameters(), cfg.max_grad_norm)
                self.optimizer.step()
                stats = (pg.detach(), vl.detach(), -ent.detach())
        # the losses of the last minibatch, read back once
        return {k: float(v) for k, v in zip(("pg_loss", "value_loss", "entropy"), stats)} if stats else {}

    # -- deterministic evaluation (CustomCallback) --------------------------------------------------------------
    @torch.no_grad()
    def evaluate(self) -> dict:
        """One deterministic episode from each of the eval env's ``n_evals`` seeded reset states, through
        ``evaluate_batch`` (``monte_carlo._evaluate_batch_lstm``) with the current actor."""
        from .environment_utils import CONFIG_KEYS
        from .monte_carlo import evaluate_batch
        env = self.eval_env
        env.reset()
        kw = dict(env.ctor_kwargs)
        config = {k: kw.pop(k) for k in CONFIG_KEYS if k in kw}
        kw.pop("quiet", None)
        reward_kwargs = kw.pop("reward_kwargs", None)
        res = evaluate_batch(self.policy.to_lstm_policy(self.device), env.get_state().cpu().numpy(), config=config,
                             reward_kwargs=reward_kwargs, device=self.device, normalize_quaternions=False, **kw)
        return {"mean_return": float(np.mean(res["total_reward"])), "mean_length": float(np.mean(res["ep_len"])),
                "success_rate": float(np.mean(res["succeeded"])), "collision_rate": float(np.mean(res["collided"]))}

    def learn(self, total_timesteps: int, eval_every: int = 1, verbose: bool = False):
        it = 0
        while self.num_timesteps < total_timesteps:
            if eval_every and it % eval_every == 0:
                ev = self.evaluate()
                if ev["mean_return"] > self.best_eval:                      # CustomCallback: keep the best model
                    self.best_eval = ev["mean_return"]
                    self.best_state = {k: v.detach().clone() for k, v in self.policy.state_dict().items()}
            else:
                ev = {}
            t0 = time.perf_counter()
            adv, ret = self.collect()
            torch.cuda.synchronize(self.device)
            t1 = time.perf_counter()
            st = self.update(adv, ret)
            torch.cuda.synchronize(self.device)
            t2 = time.perf_counter()
            row = dict(iteration=it, timesteps=self.num_timesteps, collect_s=t1 - t0, update_s=t2 - t1,
                       collect_steps_per_s=self.cfg.n_steps * self.env.num_envs / (t1 - t0),
                       mean_step_reward=float(self.buf_rew.mean()), **st, **{"eval_" + k: v for k, v in ev.items()})
            self.cfg.log.append(row)
            if verbose:
                print(row, flush=True)
            it += 1
        return self

    def save(self, path: str):
        """npz with sb3_contrib's state-dict keys ('.' -> '__'), loadable by LstmPolicy.load."""
        sd = self.best_state or self.policy.state_dict()
        np.savez(path, **{k.replace(".", "__"): v.detach().float().cpu().numpy() for k, v in sd.items()})
