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
