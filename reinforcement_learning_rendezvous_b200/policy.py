"""Device-side MLP policy: ``model.predict(obs, deterministic=True)`` of an SB3 ``MlpPolicy``.

The reference trains ``PPO("MlpPolicy", activation_fn=Tanh)`` with the default 64-64 actor
(/root/reference/main.py:39-48) and evaluates it with
``model.predict(observation, state, episode_start, deterministic=True)``
(/root/reference/monte_carlo.py:128-133): ``clip(action_net(tanh(L2(tanh(L1(obs))))), -1, 1)``.
Here the forward pass is one fp32 kernel (rdv_policy_forward); weights come from an SB3
``.zip`` checkpoint (``policy.pth`` inside) or from an ``.npz`` with the same state-dict keys.
"""
from __future__ import annotations

import ctypes as C
import io
import zipfile

import numpy as np
import torch

from . import _native as N
from .batched_env import _stream_ptr

_KEYS = {
    "w0": "mlp_extractor.policy_net.0.weight", "b0": "mlp_extractor.policy_net.0.bias",
    "w1": "mlp_extractor.policy_net.2.weight", "b1": "mlp_extractor.policy_net.2.bias",
    "w2": "action_net.weight", "b2": "action_net.bias",
}


def load_state_dict(path: str) -> dict:
    """SB3 zip (policy.pth) or npz (keys with '.' replaced by '__') -> {key: np.ndarray fp32}."""
    if str(path).endswith(".npz"):
        d = np.load(path)
        return {k.replace("__", "."): np.asarray(d[k], dtype=np.float32) for k in d.files}
    with zipfile.ZipFile(path) as z:
        sd = torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=True)
    return {k: v.detach().cpu().numpy().astype(np.float32) for k, v in sd.items()}


class MlpPolicy:
    """Actor of an SB3 MlpPolicy (17 -> 64 -> 64 -> 6, tanh) resident on the GPU."""

    def __init__(self, state_dict: dict, device="cuda"):
        if not torch.cuda.is_available():
            raise RuntimeError("MlpPolicy needs a CUDA device; there is no CPU fallback")
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.lib = N.lib()
        self.w = {k: torch.as_tensor(np.ascontiguousarray(state_dict[name]), dtype=torch.float32,
                                     device=self.device).contiguous() for k, name in _KEYS.items()}
        hidden = self.w["w0"].shape[0]
        if tuple(self.w["w0"].shape) != (hidden, N.OBS_DIM) or tuple(self.w["w1"].shape) != (hidden, hidden) \
                or tuple(self.w["w2"].shape) != (N.ACT_DIM, hidden):
            raise ValueError("unexpected policy shapes")
        self.hidden = hidden
        ls = state_dict.get("log_std")
        self.log_std = None if ls is None else torch.as_tensor(np.ascontiguousarray(ls), dtype=torch.float32,
                                                                device=self.device).contiguous()
        self._c = N.RdvPolicy(self.w["w0"].data_ptr(), self.w["b0"].data_ptr(), self.w["w1"].data_ptr(),
                              self.w["b1"].data_ptr(), self.w["w2"].data_ptr(), self.w["b2"].data_ptr(), hidden, 0,
                              self.log_std.data_ptr() if self.log_std is not None else None)
        self._h_obs = self._h_act = None

    @classmethod
    def load(cls, path: str, device="cuda") -> "MlpPolicy":
        return cls(load_state_dict(path), device=device)

    def forward(self, obs: torch.Tensor, out: torch.Tensor = None, ffma: bool = False) -> torch.Tensor:
        """Deterministic clipped actions f32[n,6] for device observations f32[n,17] (asynchronous).  Default: the
        tcgen05 tensor-core kernel; ``ffma=True``: the plain fp32-FMA kernel (numerics reference)."""
        if obs.device != self.device or obs.dtype != torch.float32:
            raise ValueError("obs must be a float32 tensor on the policy's device")
        obs = obs.contiguous()
        n = obs.shape[0]
        out = torch.empty((n, N.ACT_DIM), dtype=torch.float32, device=self.device) if out is None else out
        with torch.cuda.device(self.device):
            fn = self.lib.rdv_policy_forward_ffma if ffma else self.lib.rdv_policy_forward
            N.check(fn(C.byref(self._c), obs.data_ptr(), out.data_ptr(), n, _stream_ptr(self.device)),
                    "rdv_policy_forward")
        return out

    def predict(self, observation, state=None, episode_start=None, deterministic=True):
        """SB3 ``BaseAlgorithm.predict`` signature (numpy in, numpy out)."""
        if not deterministic:
            raise NotImplementedError("stochastic sampling is done by the trainer, not by predict()")
        obs = np.asarray(observation, dtype=np.float32)
        single = obs.ndim == 1
        obs2 = obs.reshape(-1, N.OBS_DIM)
        n = obs2.shape[0]
        if self._h_obs is None or self._h_obs.shape[0] != n:
            self._h_obs = torch.zeros((n, N.OBS_DIM), dtype=torch.float32).pin_memory()
            self._h_act = torch.zeros((n, N.ACT_DIM), dtype=torch.float32).pin_memory()
            self._d_obs = torch.zeros((n, N.OBS_DIM), dtype=torch.float32, device=self.device)
            self._d_act = torch.zeros((n, N.ACT_DIM), dtype=torch.float32, device=self.device)
        self._h_obs.numpy()[...] = obs2
        self._d_obs.copy_(self._h_obs, non_blocking=True)
        self.forward(self._d_obs, out=self._d_act)
        self._h_act.copy_(self._d_act, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        act = self._h_act.numpy().copy()
        return (act[0] if single else act), state


_LSTM_KEYS = {
    "weight_ih": "lstm_actor.weight_ih_l0", "weight_hh": "lstm_actor.weight_hh_l0",
    "bias_ih": "lstm_actor.bias_ih_l0", "bias_hh": "lstm_actor.bias_hh_l0",
    "w0": "mlp_extractor.policy_net.0.weight", "b0": "mlp_extractor.policy_net.0.bias",
    "w1": "mlp_extractor.policy_net.2.weight", "b1": "mlp_extractor.policy_net.2.bias",
    "w2": "action_net.weight", "b2": "action_net.bias",
}


def _overlap(a: torch.Tensor, b: torch.Tensor) -> bool:
    """Whether the address ranges spanned by the 2-D tensors a and b intersect."""
    def span(x):
        last = sum((d - 1) * st for d, st in zip(x.shape, x.stride()))
        return x.data_ptr(), x.data_ptr() + (last + 1) * x.element_size()
    if a.numel() == 0 or b.numel() == 0:
        return False
    (a0, a1), (b0, b1) = span(a), span(b)
    return a0 < b1 and b0 < a1


class LstmPolicy:
    """Actor of an sb3_contrib RecurrentPPO ``MlpLstmPolicy`` (main_rnn.py) resident on the GPU: one LSTM layer of
    256 units on the observation, then the default 64-64 Tanh head and ``action_net``.  One step for n envs is one
    tensor-core kernel (``rdv_lstm_policy_step``).  Only the actor is loaded: the critic's LSTM and value head and
    ``log_std`` are ignored.  The state is kept hidden-major, ``h`` and ``c`` as float32 ``[256, n]`` device tensors
    (unit j of env i at ``[j, i]``)."""

    def __init__(self, state_dict: dict, device="cuda"):
        extra = [k for k in state_dict if k.startswith("lstm_actor.") and k not in _LSTM_KEYS.values()]
        if extra:
            raise ValueError(f"only a single-layer LSTM actor is supported, got {sorted(extra)}")
        missing = [name for name in _LSTM_KEYS.values() if name not in state_dict]
        if missing:
            raise ValueError(f"not a RecurrentPPO MlpLstmPolicy state dict: missing {missing}")
        hid, obs, act = N.LSTM_HIDDEN, N.OBS_DIM, N.ACT_DIM
        shapes = dict(weight_ih=(4 * hid, obs), weight_hh=(4 * hid, hid), bias_ih=(4 * hid,), bias_hh=(4 * hid,),
                      w0=(64, hid), b0=(64,), w1=(64, 64), b1=(64,), w2=(act, 64), b2=(act,))
        for k, name in _LSTM_KEYS.items():
            if tuple(np.shape(state_dict[name])) != shapes[k]:
                raise ValueError(f"{name} has shape {tuple(np.shape(state_dict[name]))}, expected {shapes[k]} "
                                 f"(LSTM of {hid} units, 64-64 head)")
            if not np.all(np.abs(state_dict[name]) < N.LSTM_WEIGHT_LIMIT):
                raise ValueError(f"{name} has entries of magnitude >= {N.LSTM_WEIGHT_LIMIT} (64 - 1/64) or non-finite "
                                 "ones; the kernel stages the weights times 2^10 in fp16 halves")
        if not torch.cuda.is_available():
            raise RuntimeError("LstmPolicy needs a CUDA device; there is no CPU fallback")
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.lib = N.lib()
        self.hidden = hid
        self.w = {k: torch.as_tensor(np.ascontiguousarray(state_dict[name]), dtype=torch.float32,
                                     device=self.device).contiguous() for k, name in _LSTM_KEYS.items()}
        self._c = N.RdvLstmPolicy(*(self.w[k].data_ptr() for k in _LSTM_KEYS), hid, 0)

    @classmethod
    def load(cls, path: str, device="cuda") -> "LstmPolicy":
        """A RecurrentPPO ``.zip`` (its ``policy.pth``) or an ``.npz`` with the same keys ('.' written as '__')."""
        return cls(load_state_dict(path), device=device)

    def initial_state(self, n: int):
        """Zero ``(h, c)``, each float32 ``[256, n]`` on the policy's device."""
        return (torch.zeros((self.hidden, n), dtype=torch.float32, device=self.device),
                torch.zeros((self.hidden, n), dtype=torch.float32, device=self.device))

    def forward(self, obs: torch.Tensor, h: torch.Tensor, c: torch.Tensor, episode_start: torch.Tensor = None,
                out=None):
        """One deterministic step for the n envs of device observations f32 ``[n, 17]``: returns ``(actions f32
        [n, 6], h', c')`` with ``h', c'`` f32 ``[256, n]`` (asynchronous).  ``h, c``: f32 ``[256, >= n]`` with unit
        stride along envs (a column slice of a wider buffer works; the returned h', c' then are column slices of
        buffers with the same leading dimension).  ``episode_start`` (bool / uint8 ``[n]``, optional) zeroes the state
        of the envs where it is set first.  ``out``: optional ``(actions f32 [n, 6], h', c')`` buffers to write into,
        h' and c' shaped and strided like ``h``; they must not share memory with ``h``, ``c`` or each other (the
        kernel reads h' back for the head)."""
        if obs.device != self.device or obs.dtype != torch.float32 or obs.dim() != 2 or obs.shape[1] != N.OBS_DIM:
            raise ValueError("obs must be a float32 [n, 17] tensor on the policy's device")
        obs = obs.contiguous()
        n = obs.shape[0]
        ld = h.stride(0)

        def check_state(name, x):
            if x.device != self.device or x.dtype != torch.float32 or x.dim() != 2 or x.shape[0] != self.hidden \
                    or x.shape[1] < n or (n > 1 and x.stride(1) != 1) or x.stride(0) != ld:
                raise ValueError(f"{name} must be a float32 [{self.hidden}, >= n] tensor on the policy's device with "
                                 f"unit stride along envs and h's leading dimension {ld}")

        check_state("h", h)
        check_state("c", c)
        start = None
        if episode_start is not None:
            start = torch.as_tensor(episode_start, device=self.device).reshape(-1)
            if start.numel() != n:
                raise ValueError(f"episode_start must have {n} entries")
            start = start.to(torch.uint8).contiguous()
        if out is None:
            act = torch.empty((n, N.ACT_DIM), dtype=torch.float32, device=self.device)
            h_out, c_out = (torch.zeros((self.hidden, max(ld, n)), dtype=torch.float32, device=self.device)[:, :n]
                            for _ in range(2))
        else:
            act, h_out, c_out = out
            if act.device != self.device or act.dtype != torch.float32 or tuple(act.shape) != (n, N.ACT_DIM) \
                    or not act.is_contiguous():
                raise ValueError(f"out actions must be a contiguous float32 [{n}, 6] tensor on the policy's device")
            check_state("out h'", h_out)
            check_state("out c'", c_out)
            bufs = (("h", h), ("c", c), ("h'", h_out), ("c'", c_out), ("actions", act))
            for i, (na, a) in enumerate(bufs):
                for nb, b in bufs[i + 1:]:
                    if not (na in ("h", "c") and nb in ("h", "c")) and _overlap(a, b):
                        raise ValueError(f"the buffers {na} and {nb} share memory")
        if n == 0:
            return act, h_out, c_out
        with torch.cuda.device(self.device):
            N.check(self.lib.rdv_lstm_policy_step(C.byref(self._c), obs.data_ptr(),
                                                  start.data_ptr() if start is not None else None, h.data_ptr(),
                                                  c.data_ptr(), h_out.data_ptr(), c_out.data_ptr(), act.data_ptr(),
                                                  n, ld, _stream_ptr(self.device)),
                    "rdv_lstm_policy_step")
        self._keepalive = (obs, start)
        return act, h_out, c_out

    def predict(self, observation, state=None, episode_start=None, deterministic=True):
        """sb3_contrib ``RecurrentActorCriticPolicy.predict`` (numpy in, numpy out): returns ``(actions, (h, c))``
        with ``h, c`` float32 ``(1, n, 256)``.  ``state=None`` starts from zeros, ``episode_start=None`` means no env
        starts an episode; a single 1-D observation gives a ``(6,)`` action."""
        if not deterministic:
            raise NotImplementedError("stochastic sampling is done by the trainer, not by predict()")
        obs = np.asarray(observation, dtype=np.float32)
        single = obs.ndim == 1
        obs2 = obs.reshape(-1, N.OBS_DIM)
        n = obs2.shape[0]
        if state is None:
            h, c = self.initial_state(n)
        else:
            h, c = (torch.as_tensor(np.asarray(s, dtype=np.float32).reshape(n, self.hidden).T.copy(),
                                    device=self.device) for s in state)
        start = None if episode_start is None else np.asarray(episode_start, dtype=bool).reshape(n)
        act, h, c = self.forward(torch.as_tensor(obs2, device=self.device), h, c,
                                 None if start is None else torch.as_tensor(start.astype(np.uint8)))
        act = act.cpu().numpy()
        states = tuple(x.t().cpu().numpy().reshape(1, n, self.hidden) for x in (h, c))
        return (act[0] if single else act), states


class PolicyTable:
    """Several :class:`MlpPolicy` actors for ONE fused rollout (``BatchedRendezvousEnv.rollout(policy=table,
    policy_tiles=...)``): entry ``e`` acts for every tile of 128 consecutive envs whose index in ``policy_tiles`` is
    ``e`` (``RdvRolloutIO.policy_table``).  Holds the entries' ``RdvPolicy`` structs as a device ``uint8`` tensor and
    keeps the policies (which own the weights the structs point to) alive.  Every entry must live on one device and
    have the 64-wide actor the fused kernel is built for."""

    def __init__(self, policies):
        policies = list(policies)
        if not policies:
            raise ValueError("a policy table needs at least one policy")
        if not all(isinstance(p, MlpPolicy) for p in policies):
            raise TypeError("policy table entries must be MlpPolicy objects")
        if any(p.device != policies[0].device for p in policies):
            raise ValueError("policy table entries live on different devices")
        if any(p.hidden != 64 for p in policies):
            raise ValueError("the fused actor needs hidden width 64 for every entry")
        self.policies = policies
        self.device = policies[0].device
        self.table = torch.frombuffer(bytearray(self.pack([p._c for p in policies])), dtype=torch.uint8).to(self.device)

    @staticmethod
    def pack(structs) -> bytes:
        """``RdvPolicy`` structs -> the bytes of a C array ``RdvPolicy[len(structs)]``."""
        return b"".join(bytes(s) for s in structs)

    def __len__(self):
        return len(self.policies)

    @property
    def stochastic_ready(self) -> bool:
        """Every entry has the Gaussian head's ``log_std`` (needed for sampling rollouts)."""
        return all(p.log_std is not None for p in self.policies)
