"""BatchedRendezvousEnv -- N independent RendezvousEnv instances resident in B200 HBM.

State lives in two torch tensors laid out structure-of-arrays ([row][env], see
include/rdv_b200.h): ``f64`` = rc vc qc wc qt wt + total_delta_v/w + episode return,
``i32`` = step counter, success counter, sticky collided flag, episode index.
Every method launches hand-written sm_100a kernels through the C ABI on the
current torch CUDA stream and returns device tensors without synchronising;
nothing here computes environment math on the host.

Reference semantics (/root/reference/rendezvous_env.py): ``step`` = :160-221,
``reset`` = :223-270, auto-reset + ``terminal_observation`` = what SB3's
DummyVecEnv.step_wait adds around them (main.py:33-34).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import _native as N
from .params import copy_params, make_params

STATE_SLICES = {"rc": (N.RCX, 3), "vc": (N.VCX, 3), "qc": (N.QCW, 4), "wc": (N.WCX, 3), "qt": (N.QTW, 4),
                "wt": (N.WTX, 3)}


def _stream_ptr(device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def policy_tile_indices(policy_tiles, num_envs: int, count: int) -> np.ndarray:
    """Host-side check of a policy-table tile map: one int per tile of 128 envs (``ceil(num_envs / 128)``), each in
    ``[0, count)``.  Returns it as int32 (``RdvRolloutIO.policy_tile``)."""
    if policy_tiles is None:
        raise ValueError("a PolicyTable needs policy_tiles (one entry index per tile of 128 envs)")
    if isinstance(policy_tiles, torch.Tensor):
        policy_tiles = policy_tiles.detach().cpu().numpy()
    tiles = np.asarray(policy_tiles)
    if tiles.dtype.kind not in "iu":
        raise ValueError("policy_tiles must hold integers")
    tiles = tiles.reshape(-1).astype(np.int64)
    want = (int(num_envs) + N.POLICY_TILE - 1) // N.POLICY_TILE
    if tiles.size != want:
        raise ValueError(f"policy_tiles has {tiles.size} entries, expected {want} (one per {N.POLICY_TILE} envs)")
    if tiles.size and (tiles.min() < 0 or tiles.max() >= count):
        raise ValueError(f"policy_tiles holds an index outside [0, {count})")
    return tiles.astype(np.int32)


class ParamGroup:
    """A contiguous env range [lo, hi) sharing one RdvParams block."""

    def __init__(self, params: N.RdvParams, lo: int, hi: int):
        self.params, self.lo, self.hi = params, int(lo), int(hi)

    @property
    def n(self):
        return self.hi - self.lo


class BatchedRendezvousEnv:
    """``num_envs`` environments on one GPU.

    :param num_envs: number of environments on this device
    :param device: CUDA device (no CPU path exists)
    :param seed: Philox key for reset(); results depend only on (seed, global env id, episode index)
    :param env_offset: global index of env 0 of this shard (multi-GPU sharding keeps results invariant)
    :param auto_reset: finished envs are reset inside ``step`` (VecEnv semantics); the returned obs is then
        the post-reset observation and ``terminal_obs`` holds the last observation of the episode
    :param param_batches: optional list of ``(count, ctor_kwargs)``: per-env parameter batches (the
        sensitivity-sweep axes of sensitivity_analysis.py:97-134) as contiguous groups of envs
    :param ctor_kwargs: the reference ``RendezvousEnv`` constructor arguments (+ ``integrator``, ``inertia``,
        ``inertia_target``, ``chaser_torque``)
    """

    def __init__(self, num_envs: int, device="cuda", seed: int = 0, env_offset: int = 0, auto_reset: bool = True,
                 param_batches: Optional[Sequence] = None, track_stats: bool = True, ld: Optional[int] = None,
                 **ctor_kwargs):
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedRendezvousEnv needs a CUDA device (B200); there is no CPU fallback")
        self.lib = N.lib()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("BatchedRendezvousEnv only runs on CUDA devices")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.num_envs = n = int(num_envs)
        if n <= 0:
            raise ValueError("num_envs must be positive")
        self._seed, self.env_offset, self.auto_reset = int(seed), int(env_offset), bool(auto_reset)
        self.ctor_kwargs = dict(ctor_kwargs)
        self.reset_rows = None          # prefetched reset rows carried from rollout to rollout (allocated on first use)
        self._tile_map = None           # (bytes, device int32 tensor): the last policy-table tile map uploaded
        self.sm_reserve = 0             # SMs a rollout launch leaves free (distributed.py: overlapped stats all-reduce)

        if param_batches:
            groups, lo = [], 0
            for count, kw in param_batches:
                merged = dict(ctor_kwargs)
                merged.update(kw)
                if lo % 32:
                    raise ValueError("every param batch but the last must hold a multiple of 32 envs "
                                     "(keeps each group's rows 256-byte aligned)")
                groups.append(ParamGroup(make_params(**merged), lo, lo + int(count)))
                lo += int(count)
            if lo != n:
                raise ValueError(f"param_batches cover {lo} envs, expected {n}")
        else:
            groups = [ParamGroup(make_params(**ctor_kwargs), 0, n)]
        self.groups = groups
        self.params = groups[0].params
        # Per-env parameter batches travel as a device table of RdvParams + one entry index per block of 32 envs, so
        # that every method is ONE launch over the whole batch (RdvState.param_table).  The table form exists for the
        # reference's bodies with the RK45 integrator; anything else falls back to one launch per group.
        self.param_table = self.param_block = None
        self._units = groups
        if len(groups) > 1 and all(g.params.iso_c and g.params.iso_t and g.params.integrator == N.INTEGRATOR_RK45
                                   for g in groups):
            raw = b"".join(bytes(g.params) for g in groups)
            self.param_table = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(self.device)
            blocks = np.zeros((n + 31) // 32, dtype=np.int32)
            for gi, g in enumerate(groups):
                blocks[g.lo // 32:(g.hi + 31) // 32] = gi
            self.param_block = torch.as_tensor(blocks, device=self.device)
            self._units = [ParamGroup(groups[0].params, 0, n)]

        # leading dimension padded to 32 envs so every SoA row starts 256-byte aligned
        self.ld = ld = (n + 31) // 32 * 32 if ld is None else int(ld)
        if ld < n:
            raise ValueError("ld must be >= num_envs")
        dev = self.device
        self.f64 = torch.zeros((N.NF64, ld), dtype=torch.float64, device=dev)
        self.i32 = torch.zeros((N.NI32, ld), dtype=torch.int32, device=dev)
        self.obs = torch.zeros((n, N.OBS_DIM), dtype=torch.float32, device=dev)
        self.reward = torch.zeros(n, dtype=torch.float64, device=dev)
        self.done = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.terminal_obs = torch.zeros((n, N.OBS_DIM), dtype=torch.float32, device=dev)
        self.end_reason = torch.full((n,), -1, dtype=torch.int8, device=dev)
        self.episode_record = torch.zeros((n, N.EP_NCOL), dtype=torch.float64, device=dev)
        self.stats = torch.zeros(N.NSTATS, dtype=torch.float64, device=dev) if track_stats else None
        self.host_block = None          # see enable_host_block()
        self.reward_f32 = self.fin_count = self.fin_rows = None
        self._keepalive = None

    # ------------------------------------------------------------------ plumbing
    @property
    def seed(self) -> int:
        return self._seed

    @seed.setter
    def seed(self, value: int):
        self._seed = int(value)
        self.invalidate_reset_rows()

    def invalidate_reset_rows(self):
        """The prefetched reset rows are a function of (seed, parameters, env id, episode): forget them when the
        first two change (the episode tag row covers the rest)."""
        if self.reset_rows is not None:
            self.reset_rows[N.RESET_ROWS - 1].zero_()

    def _reset_rows_ptr(self, g: "ParamGroup"):
        if not self.auto_reset:
            return None
        if self.reset_rows is None:
            self.reset_rows = torch.zeros((N.RESET_ROWS, self.ld), dtype=torch.float64, device=self.device)
        return self.reset_rows.data_ptr() + 8 * g.lo

    def _state_of(self, g: ParamGroup) -> N.RdvState:
        if self.param_table is not None:
            return N.RdvState(self.f64.data_ptr(), self.i32.data_ptr(), self.ld, self.param_table.data_ptr(),
                              self.param_block.data_ptr())
        return N.RdvState(self.f64.data_ptr() + 8 * g.lo, self.i32.data_ptr() + 4 * g.lo, self.ld, None, None)

    def enable_host_block(self):
        """Re-home everything one ``step`` returns to a host-side VecEnv into ONE contiguous device block, so that a
        single device-to-host copy fetches it: ``[count | reward f32[N] | done u8[N] | obs f32[N,17] | finished rows]``
        (every section 256-byte aligned).  ``obs`` / ``done`` become views of the block; ``step`` then also writes
        float32 rewards and appends one 128-byte :class:`RdvFinishedRow` per finished env (index, end reason, terminal
        observation, episode record) through one atomic counter.  Returns the section offsets in bytes."""
        if self.host_block is not None:
            return self.block_layout
        n = self.num_envs

        def up(x):
            return (x + 255) // 256 * 256
        off_rew = 256
        off_done = up(off_rew + 4 * n)
        off_obs = up(off_done + n)
        off_rows = up(off_obs + 4 * N.OBS_DIM * n)
        total = off_rows + C.sizeof(N.RdvFinishedRow) * n
        blk = torch.zeros(total, dtype=torch.uint8, device=self.device)
        self.host_block = blk
        self.block_layout = dict(count=0, reward=off_rew, done=off_done, obs=off_obs, rows=off_rows, total=total,
                                 row_bytes=C.sizeof(N.RdvFinishedRow))
        self.fin_count = blk[0:4].view(torch.int32)
        self.reward_f32 = blk[off_rew:off_rew + 4 * n].view(torch.float32)
        new_done = blk[off_done:off_done + n]
        new_obs = blk[off_obs:off_obs + 4 * N.OBS_DIM * n].view(torch.float32).view(n, N.OBS_DIM)
        new_done.copy_(self.done)
        new_obs.copy_(self.obs)
        self.done, self.obs = new_done, new_obs
        self.fin_rows = blk[off_rows:]
        return self.block_layout

    def _check_actions(self, actions: torch.Tensor) -> torch.Tensor:
        if not isinstance(actions, torch.Tensor):
            raise TypeError("actions must be a torch tensor on the env's device (use RendezvousVecEnv for numpy)")
        if actions.device != self.device:
            raise ValueError(f"actions live on {actions.device}, env on {self.device}")
        if actions.dtype not in (torch.float32, torch.float64):
            raise TypeError("actions must be float32 or float64")
        if tuple(actions.shape) != (self.num_envs, N.ACT_DIM):
            raise ValueError(f"actions must have shape ({self.num_envs}, {N.ACT_DIM})")
        return actions if actions.is_contiguous() else actions.contiguous()

    # ------------------------------------------------------------------ hot path
    def step(self, actions: torch.Tensor):
        """One step of every env.  Returns (obs f32[N,17], reward f64[N], done u8[N]) -- views of the
        env's output buffers, valid until the next ``step``.  Asynchronous on the current stream."""
        actions = self._check_actions(actions)
        mode = 1 if self.auto_reset else 0
        act_f64 = 1 if actions.dtype == torch.float64 else 0
        esz = 8 if act_f64 else 4
        stream = _stream_ptr(self.device)
        blk = self.host_block is not None
        with torch.cuda.device(self.device):
            for gi, g in enumerate(self._units):
                io = N.RdvStepIO(
                    actions.data_ptr() + g.lo * N.ACT_DIM * esz, act_f64, mode,
                    self.obs.data_ptr() + g.lo * N.OBS_DIM * 4, self.reward.data_ptr() + g.lo * 8,
                    self.done.data_ptr() + g.lo,
                    self.terminal_obs.data_ptr() + g.lo * N.OBS_DIM * 4, self.end_reason.data_ptr() + g.lo,
                    self.episode_record.data_ptr() + g.lo * N.EP_NCOL * 8,
                    self.stats.data_ptr() if self.stats is not None else None,
                    self.reward_f32.data_ptr() + g.lo * 4 if blk else None,
                    self.fin_count.data_ptr() if blk else None, self.fin_rows.data_ptr() if blk else None,
                    self.num_envs if blk else 0, 1 if gi else 0, g.lo, 0)
                st = self._state_of(g)
                N.check(self.lib.rdv_step(C.byref(g.params), C.byref(st), C.byref(io), g.n, self.seed,
                                          self.env_offset + g.lo, stream), "rdv_step")
        self._keepalive = actions
        return self.obs, self.reward, self.done

    def rollout(self, steps: int, actions: Optional[torch.Tensor] = None, action_seed: Optional[int] = None,
                step_base: int = 0, record_rewards: bool = False, record_dones: bool = False,
                record_obs: bool = False, record_actions: bool = False, policy=None,
                stochastic: bool = False, carry_reset_rows: bool = True, monte_carlo: bool = False,
                policy_tiles=None, record_trajectory: bool = False) -> dict:
        """``steps`` consecutive env steps in ONE kernel launch (state stays in registers, finished envs restart
        in place when ``auto_reset``).  Actions come from ``actions`` ([steps, N, 6] float32/float64 on the device) or,
        when it is None, from the device Philox stream ``(action_seed; global env id, step_base + k)`` as U(-1,1) fp64
        draws -- the "random actions" workload -- or from ``policy`` (an :class:`MlpPolicy`): the deterministic actor
        output ``clip(pi(obs), -1, 1)`` evaluated inside the launch on the tensor cores from the observation the
        previous step returned (closed loop, float32 actions); with ``stochastic`` the action is drawn from the
        policy's Gaussian head N(pi(obs), exp(log_std)^2) with Philox noise keyed by ``action_seed`` (SB3's
        collect_rollouts: the env gets the clipped draw, ``actions`` records the unclipped one).  Returns a dict with ``obs`` (final observation, f32 [N,17]) and the
        requested per-step records (``rewards`` f64 [steps,N], ``dones`` u8 [steps,N], ``obs_steps`` f32 [steps,N,17],
        ``actions`` f64 [steps,N,6] for Philox actions).  ``carry_reset_rows``: keep every env's prefetched next reset
        state in a device scratch between launches (short launches then run at the rate of long ones).
        ``monte_carlo`` (needs ``auto_reset=False``): evaluator mode -- an env stops at its first done and the launch
        returns ``mc`` f64 [N, MC_NCOL], the per-episode columns of monte_carlo.py:190-203 accumulated on the device.
        ``policy`` may also be a :class:`~.policy.PolicyTable`: then ``policy_tiles`` (ints or an int tensor, one per
        tile of 128 envs) names the entry that acts for envs ``128 t .. 128 t + 127``, all in the same launch; every
        tile gives the bits a separate env of its envs (same seed, ``env_offset`` = tile start) rolled with that entry
        would give.  Asynchronous on the current stream (the tile map is checked on the host: a device tensor given as
        ``policy_tiles`` is read back for that, which waits for the stream; a host sequence does not).
        ``record_trajectory``: the launch also records the fp64 trajectory (``rdv_rollout_trajectory``) and returns it
        as ``trajectory`` f64 [steps, TR_NCOL, N] on the device -- 272 B per env-step.  Row k is every env after step k
        and before an auto-reset (a finished env's terminal state): columns 0 .. NF64 - 1 the ``f64`` state rows,
        ``TR_I_STEP`` .. ``TR_I_EPISODE`` the ``i32`` rows, ``TR_POS_ERR`` .. ``TR_SUCCESS`` what :meth:`errors`
        returns for that state.  Every other output is the same as without the record."""
        steps = int(steps)
        n, dev = self.num_envs, self.device
        if steps < 0:
            raise ValueError("steps must be >= 0")
        table = None                    # policy tables: the tile map on the device
        if actions is not None:
            if actions.device != dev or actions.dtype not in (torch.float32, torch.float64):
                raise ValueError("actions must be a float32/float64 tensor on the env's device")
            if tuple(actions.shape) != (steps, n, N.ACT_DIM):
                raise ValueError(f"actions must have shape ({steps}, {n}, {N.ACT_DIM})")
            actions = actions.contiguous()
            source = N.ACTIONS_F64 if actions.dtype == torch.float64 else N.ACTIONS_F32
            esz = 8 if actions.dtype == torch.float64 else 4
        elif policy is not None:
            from .policy import PolicyTable
            if policy.device != dev:
                raise ValueError("policy and env live on different devices")
            if isinstance(policy, PolicyTable):
                tiles = policy_tile_indices(policy_tiles, n, len(policy))
                if stochastic and (not policy.stochastic_ready or action_seed is None):
                    raise ValueError("stochastic policy-table rollouts need log_std in every entry and an action_seed")
                if len(self._units) > 1:
                    raise NotImplementedError("policy tables with param_batches of general-inertia or closed-form "
                                              "groups (one launch per group)")
                table = self._policy_tile_map(tiles)
            elif stochastic and (policy.log_std is None or action_seed is None):
                raise ValueError("stochastic policy rollouts need policy.log_std and an action_seed")
            source, esz = (N.ACTIONS_POLICY_SAMPLE if stochastic else N.ACTIONS_POLICY), 0
        else:
            if action_seed is None:
                raise ValueError("give an actions tensor, an action_seed (device-generated actions) or a policy")
            source, esz = N.ACTIONS_PHILOX, 0
        if policy_tiles is not None and table is None:
            raise ValueError("policy_tiles needs a PolicyTable policy")
        out = {"obs": self.obs}
        rew = torch.empty((steps, n), dtype=torch.float64, device=dev) if record_rewards else None
        don = torch.empty((steps, n), dtype=torch.uint8, device=dev) if record_dones else None
        obs_steps = torch.empty((steps, n, N.OBS_DIM), dtype=torch.float32, device=dev) if record_obs else None
        act_out = torch.empty((steps, n, N.ACT_DIM), dtype=torch.float32 if policy is not None else torch.float64,
                              device=dev) if (record_actions and actions is None) else None
        mc_out = None
        if monte_carlo:
            if self.auto_reset:
                raise ValueError("monte_carlo mode needs an env with auto_reset=False")
            mc_out = torch.empty((n, N.MC_NCOL), dtype=torch.float64, device=dev)
        traj = torch.empty((steps, N.TR_NCOL, n), dtype=torch.float64, device=dev) if record_trajectory else None
        if len(self._units) > 1 and (rew is not None or don is not None or obs_steps is not None or act_out is not None
                                     or actions is not None or traj is not None):
            raise NotImplementedError("per-step records / tensor actions with param_batches of general-inertia or "
                                      "closed-form groups (one launch per group): use step()")
        stream = _stream_ptr(dev)
        with torch.cuda.device(dev):
            for g in self._units:
                io = N.RdvRolloutIO(
                    steps, source, int(self.auto_reset), 0,
                    actions.data_ptr() if actions is not None else None,
                    int(action_seed or 0) & 0xFFFFFFFFFFFFFFFF, int(step_base),
                    act_out.data_ptr() if act_out is not None else None,
                    self.obs.data_ptr() + g.lo * N.OBS_DIM * 4,
                    rew.data_ptr() if rew is not None else None, don.data_ptr() if don is not None else None,
                    obs_steps.data_ptr() if obs_steps is not None else None,
                    self.stats.data_ptr() if self.stats is not None else None,
                    policy._c if policy is not None and table is None else N.RdvPolicy(),
                    self._reset_rows_ptr(g) if carry_reset_rows else None, int(self.sm_reserve), 0,
                    mc_out.data_ptr() + g.lo * N.MC_NCOL * 8 if mc_out is not None else None,
                    policy.table.data_ptr() if table is not None else None,
                    table.data_ptr() if table is not None else None, len(policy) if table is not None else 0, 0)
                st = self._state_of(g)
                if traj is None:
                    N.check(self.lib.rdv_rollout(C.byref(g.params), C.byref(st), C.byref(io), g.n, self.seed,
                                                 self.env_offset + g.lo, stream), "rdv_rollout")
                else:
                    N.check(self.lib.rdv_rollout_trajectory(C.byref(g.params), C.byref(st), C.byref(io),
                                                            traj.data_ptr(), g.n, self.seed, self.env_offset + g.lo,
                                                            stream), "rdv_rollout_trajectory")
        self._keepalive = (actions, policy, table)
        if rew is not None:
            out["rewards"] = rew
        if don is not None:
            out["dones"] = don
        if obs_steps is not None:
            out["obs_steps"] = obs_steps
        if act_out is not None:
            out["actions"] = act_out
        if mc_out is not None:
            out["mc"] = mc_out
        if traj is not None:
            out["trajectory"] = traj
        return out

    def _policy_tile_map(self, tiles: np.ndarray) -> torch.Tensor:
        """The checked tile map on the device.  The last one is kept, so repeated rollouts with the same map upload
        nothing; a new one goes through pinned memory with a non-blocking copy, so the call does not wait for the
        stream."""
        key = tiles.tobytes()
        if self._tile_map is None or self._tile_map[0] != key:
            dev_map = torch.empty(tiles.shape, dtype=torch.int32, device=self.device)
            dev_map.copy_(torch.from_numpy(tiles).pin_memory(), non_blocking=True)
            self._tile_map = (key, dev_map)
        return self._tile_map[1]

    def reset(self, mask: Optional[torch.Tensor] = None, uniforms: Optional[torch.Tensor] = None,
              bump_episode: bool = True) -> torch.Tensor:
        """reset() for all envs, or those where ``mask`` (uint8/bool [N]) is set.  ``uniforms`` ([N,24] fp64 in
        [0,1)) replaces the Philox draws (test hook that pins the reference's draw order)."""
        m_ptr = u_ptr = None
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            if mask.numel() != self.num_envs:
                raise ValueError("mask must have num_envs elements")
        if uniforms is not None:
            uniforms = uniforms.to(device=self.device, dtype=torch.float64).contiguous()
            if tuple(uniforms.shape) != (self.num_envs, N.N_UNIFORMS):
                raise ValueError(f"uniforms must have shape ({self.num_envs}, {N.N_UNIFORMS})")
        stream = _stream_ptr(self.device)
        with torch.cuda.device(self.device):
            for g in self._units:
                if mask is not None:
                    m_ptr = mask.data_ptr() + g.lo
                if uniforms is not None:
                    u_ptr = uniforms.data_ptr() + g.lo * N.N_UNIFORMS * 8
                st = self._state_of(g)
                N.check(self.lib.rdv_reset(C.byref(g.params), C.byref(st), m_ptr, u_ptr,
                                           self.obs.data_ptr() + g.lo * N.OBS_DIM * 4, g.n, self.seed,
                                           self.env_offset + g.lo, int(bump_episode), stream), "rdv_reset")
        self._keepalive = (mask, uniforms)
        return self.obs

    def observe(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """get_observation() of the current state (rendezvous_env.py:294-311)."""
        out = torch.empty((self.num_envs, N.OBS_DIM), dtype=torch.float32, device=self.device) if out is None else out
        stream = _stream_ptr(self.device)
        with torch.cuda.device(self.device):
            for g in self._units:
                st = self._state_of(g)
                N.check(self.lib.rdv_observe(C.byref(g.params), C.byref(st), out.data_ptr() + g.lo * N.OBS_DIM * 4,
                                             g.n, stream), "rdv_observe")
        return out

    def errors(self):
        """(errors f64[N,4], collision u8[N], success u8[N], dist_from_koz f64[N]) of the current state:
        get_errors / check_collision / check_success / dist_from_koz (rendezvous_env.py:388-468, :510-537)."""
        n, dev = self.num_envs, self.device
        err = torch.empty((n, 4), dtype=torch.float64, device=dev)
        col = torch.empty(n, dtype=torch.uint8, device=dev)
        suc = torch.empty(n, dtype=torch.uint8, device=dev)
        koz = torch.empty(n, dtype=torch.float64, device=dev)
        stream = _stream_ptr(dev)
        with torch.cuda.device(dev):
            for g in self._units:
                st = self._state_of(g)
                N.check(self.lib.rdv_errors(C.byref(g.params), C.byref(st), err.data_ptr() + g.lo * 32,
                                            col.data_ptr() + g.lo, suc.data_ptr() + g.lo, koz.data_ptr() + g.lo * 8,
                                            g.n, stream), "rdv_errors")
        return err, col, suc, koz

    def refresh_flags(self):
        """Recompute collided/success from the current state the way reset() does (:260-261)."""
        stream = _stream_ptr(self.device)
        with torch.cuda.device(self.device):
            for g in self._units:
                st = self._state_of(g)
                N.check(self.lib.rdv_refresh_flags(C.byref(g.params), C.byref(st), g.n, stream), "rdv_refresh_flags")

    # ------------------------------------------------------------------ state access
    def state_view(self, name: str) -> torch.Tensor:
        """Writable [N, k] view of one state vector ('rc','vc','qc','wc','qt','wt') into the SoA rows."""
        row, k = STATE_SLICES[name]
        return self.f64[row:row + k, :self.num_envs].t()

    def get_state(self) -> torch.Tensor:
        """[N,20] fp64 copy: rc vc qc wc qt wt."""
        return self.f64[:N.TDV, :self.num_envs].t().contiguous()

    def set_state(self, state20, reset_counters: bool = True, refresh_flags: bool = False):
        """Inject states (what monte_carlo.evaluate does after reset(), monte_carlo.py:106-112).  The sticky
        collided/success flags are zeroed with the counters (a reset() at the nominal state leaves them 0) and are
        NOT recomputed from the injected state unless ``refresh_flags`` -- exactly like the reference evaluator."""
        s = torch.as_tensor(np.asarray(state20, dtype=np.float64) if not isinstance(state20, torch.Tensor) else state20)
        s = s.to(device=self.device, dtype=torch.float64).reshape(self.num_envs, 20)
        self.f64[:N.TDV, :self.num_envs] = s.t()
        if reset_counters:
            self.f64[N.TDV:, :] = 0
            self.i32[N.I_STEP:N.I_COLLIDED + 1, :] = 0
        if refresh_flags:
            self.refresh_flags()

    @property
    def step_count(self):
        return self.i32[N.I_STEP, :self.num_envs]

    @property
    def collided(self):
        return self.i32[N.I_COLLIDED, :self.num_envs]

    @property
    def success(self):
        return self.i32[N.I_SUCCESS, :self.num_envs]

    @property
    def episode_index(self):
        return self.i32[N.I_EPISODE, :self.num_envs]

    @property
    def total_delta_v(self):
        return self.f64[N.TDV, :self.num_envs]

    @property
    def total_delta_w(self):
        return self.f64[N.TDW, :self.num_envs]

    @property
    def episode_return(self):
        return self.f64[N.EPRET, :self.num_envs]

    # ------------------------------------------------------------------ statistics / checkpoint
    def read_stats(self, reset: bool = False) -> dict:
        """Rollout statistics accumulated on the device by the step kernel (warp-shuffle + one atomic per CTA)."""
        if self.stats is None:
            raise RuntimeError("env was created with track_stats=False")
        v = self.stats.cpu().numpy()
        if reset:
            self.stats.zero_()
        return dict(zip(N.STAT_NAMES, v.tolist()))

    def state_dict(self) -> dict:
        return {"f64": self.f64.clone(), "i32": self.i32.clone(), "obs": self.obs.clone(),
                "seed": self.seed, "env_offset": self.env_offset,
                "stats": None if self.stats is None else self.stats.clone()}

    def load_state_dict(self, sd: dict):
        self.f64.copy_(sd["f64"])
        self.i32.copy_(sd["i32"])
        self.obs.copy_(sd["obs"])
        self.seed, self.env_offset = int(sd["seed"]), int(sd["env_offset"])      # the setter forgets the reset rows
        if self.stats is not None and sd.get("stats") is not None:
            self.stats.copy_(sd["stats"])

    def clone(self) -> "BatchedRendezvousEnv":
        other = BatchedRendezvousEnv.__new__(BatchedRendezvousEnv)
        other.__dict__.update(self.__dict__)
        other.groups = [ParamGroup(copy_params(g.params), g.lo, g.hi) for g in self.groups]
        other.params = other.groups[0].params
        other._units = other.groups if self.param_table is None else [ParamGroup(other.params, 0, self.num_envs)]
        for name in ("f64", "i32", "obs", "reward", "done", "terminal_obs", "end_reason", "episode_record"):
            setattr(other, name, getattr(self, name).clone())
        if self.host_block is not None:
            other.host_block = None
            other.enable_host_block()
        other.stats = None if self.stats is None else self.stats.clone()
        other.reset_rows = None if self.reset_rows is None else self.reset_rows.clone()
        other._keepalive = None
        return other
