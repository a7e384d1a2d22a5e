"""Monte-Carlo evaluator (/root/reference/monte_carlo.py:94-207).

``evaluate(model, env, initial_state)`` keeps the reference's single-episode signature and works with
the single-env facade.  ``evaluate_batch`` runs every initial condition as one env of a GPU batch in ONE
launch: the actor, the env step, the get_errors / check_collision / check_success / dist_from_koz queries
and the per-episode reduction (counts, running minimum, first-index terminal-error averaging of
monte_carlo.py:159-189) all happen inside the policy-fused rollout kernel, and one [M, 16] array comes back.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native as N
from .batched_env import BatchedRendezvousEnv
from .environment_utils import config_to_kwargs
from .policy import PolicyTable

MC_COLS = ("ep_len", "num_collisions", "collided", "total_reward", "total_delta_v", "num_successes", "succeeded",
           "min_dist_from_koz", "pos_error", "vel_error", "att_error", "rot_error")


def _terminal_errors(errors, limits):
    """monte_carlo.py:159-189: errors [T,4] of one episode -> averaged terminal errors from the first index
    at which the most constraints are met."""
    pos, vel, att, rot = errors[:, 0], errors[:, 1], errors[:, 2], errors[:, 3]
    pm, vm, am, rm = pos < limits[0], vel < limits[1], att < limits[2], rot < limits[3]
    all_mask = pm & vm & am & rm
    if all_mask.any():
        index = int(np.argmax(all_mask))
    else:
        three = (pm & vm & am) | (pm & vm & rm)
        if three.any():
            index = int(np.argmax(three))
        elif (pm & vm).any():
            index = int(np.argmax(pm & vm))
        elif pm.any():
            index = int(np.argmax(pm))
        else:
            index = -1
    return (pos[index:].mean(), vel[index:].mean(), np.degrees(att[index:].mean()), np.degrees(rot[index:].mean()))


def _terminal_errors_batch(errors, lengths, limits):
    """``_terminal_errors`` for M episodes at once.  errors [T, M, 4] (rows >= lengths[i] + 1 of episode i are
    ignored), lengths [M] = steps taken; returns [M, 4] (pos, vel, att deg, rot deg).  Same rule as
    monte_carlo.py:159-189: the first index at which all four constraints hold, else the first with three
    (pos, vel and att or rot), else pos and vel, else pos, else the last sample; then the mean of the tail."""
    errors = np.asarray(errors, dtype=np.float64)
    t_max, m = errors.shape[0], errors.shape[1]
    valid = np.arange(t_max)[:, None] <= np.asarray(lengths)[None, :]                     # [T, M]
    lim = np.asarray(limits, dtype=np.float64)
    ok = (errors < lim[None, None, :]) & valid[:, :, None]                                  # NaN rows compare False
    pm, vm, am, rm = ok[..., 0], ok[..., 1], ok[..., 2], ok[..., 3]
    levels = (pm & vm & am & rm, (pm & vm & am) | (pm & vm & rm), pm & vm, pm)
    last = np.asarray(lengths, dtype=np.int64)
    index = last.copy()                                                                     # the "-1" case: last sample
    decided = np.zeros(m, dtype=bool)
    for mask in levels:
        hit = mask.any(axis=0) & ~decided
        index = np.where(hit, mask.argmax(axis=0), index)
        decided |= hit
    tail = valid & (np.arange(t_max)[:, None] >= index[None, :])                            # [T, M]
    count = tail.sum(axis=0)
    mean = np.where(tail[:, :, None], np.nan_to_num(errors), 0.0).sum(axis=0) / count[:, None]
    mean[:, 2:] = np.degrees(mean[:, 2:])
    return mean


def evaluate(model, env, initial_state):
    """One deterministic episode from ``initial_state`` (dict rc vc qc wc qt wt) -- monte_carlo.py:94-207."""
    num_collisions = num_successes = 0
    total_reward = 0
    env.reset()
    for k in ("rc", "vc", "qc", "wc", "qt", "wt"):
        setattr(env, k, initial_state[k])
    obs = env.get_observation()
    lstm_states, ep_start, done = None, np.ones((1,), dtype=bool), False
    errors, times = [env.get_errors()], [env.t]
    collision = env.check_collision()
    num_collisions += int(collision)
    if not env.collided:
        num_successes += int(env.check_success())
    min_dist = env.dist_from_koz()
    while not done:
        action, lstm_states = model.predict(observation=obs, state=lstm_states, episode_start=ep_start,
                                            deterministic=True)
        obs, reward, done, _ = env.step(action)
        ep_start[0] = done
        errors.append(env.get_errors())
        times.append(env.t)
        collision = env.check_collision()
        num_collisions += int(collision)
        if not env.collided:
            num_successes += int(env.check_success())
        min_dist = min(min_dist, env.dist_from_koz())
        total_reward += reward
    te = _terminal_errors(np.array(errors), (env.max_rd_error, env.max_vd_error, env.max_qd_error, env.max_wd_error))
    return dict(ep_len=times[-1], num_collisions=num_collisions, collided=int(num_collisions > 0),
                total_reward=total_reward, total_delta_v=env.total_delta_v, num_successes=num_successes,
                succeeded=int(num_successes > 0), min_dist_from_koz=min_dist, pos_error=te[0], vel_error=te[1],
                att_error=te[2], rot_error=te[3])


def evaluate_batch(policy, initial_states, config=None, reward_kwargs=None, device="cuda", normalize_quaternions=True,
                   return_raw=False, trajectories=False, **extra) -> dict:
    """All rows of ``initial_states`` ([M,20]: rc vc qc wc qt wt) as one GPU batch: ONE kernel launch and ONE
    device-to-host copy.  The launch is the policy-fused rollout in evaluator mode (``RdvRolloutIO.mc_out``): the actor
    runs on the tensor cores inside the kernel, and per-episode collision / success counts, the running minimum of
    ``dist_from_koz``, the return and the first-index terminal-error averages of monte_carlo.py:159-189 are
    accumulated in registers until the env's first done.  Returns a dict of length-M arrays with the columns of the
    reference's results workbook.  ``config`` defaults to the evaluator's ``dict(dt=1, t_max=60)`` with
    ``stochastic=False`` (monte_carlo.py:26-27).

    ``policy`` may be a list or tuple of :class:`~.policy.MlpPolicy` (e.g. the checkpoints of a training run, or the models
    of a sweep): every model then runs all M initial conditions in its own block of envs, padded to a multiple of 128
    (one tile of the policy table; the padding rows are discarded), still in ONE launch with ONE read-back, and a list
    with one result dict per model is returned.  Each dict equals what ``evaluate_batch(model, ...)`` returns.

    ``trajectories``: the same launch also records every env's fp64 trajectory (``rdv_rollout_trajectory``), and each
    result dict gains ``trajectory``: the reference evaluator's per-step ``errors`` and ``times`` lists (and the state
    behind them) for every episode at once, over L + 1 samples (L = ``done_steps``; sample 0 is the state at launch,
    whose errors come from one :meth:`~.BatchedRendezvousEnv.errors` call before it).  See :func:`trajectory_fields`."""
    ics = np.array(initial_states, dtype=np.float64, copy=True).reshape(-1, 20)
    if normalize_quaternions:                                   # monte_carlo.py:66-67
        ics[:, 6:10] /= np.linalg.norm(ics[:, 6:10], axis=1, keepdims=True)
        ics[:, 13:17] /= np.linalg.norm(ics[:, 13:17], axis=1, keepdims=True)
    m = ics.shape[0]
    models = list(policy) if isinstance(policy, (list, tuple)) else None
    block = m
    if models is not None:
        policy = PolicyTable(models)
        block = (m + N.POLICY_TILE - 1) // N.POLICY_TILE * N.POLICY_TILE
        # the reset state of the evaluator's config does not depend on the env id (zero ranges), so the last row
        # repeated is a valid padding state
        ics = np.tile(np.concatenate([ics, np.repeat(ics[-1:], block - m, axis=0)]), (len(models), 1))
    kw = config_to_kwargs(dict(dt=1, t_max=60) if config is None else config, stochastic=False)
    env = BatchedRendezvousEnv(ics.shape[0], device=device, auto_reset=False, track_stats=False,
                               reward_kwargs=reward_kwargs, **kw, **extra)
    p = env.params
    env.reset()
    env.set_state(ics, reset_counters=False)        # flags stay as reset() left them (monte_carlo.py:106-112)
    tiles = None if models is None else np.repeat(np.arange(len(models)), block // N.POLICY_TILE)
    row0 = _record_row_of_state(env) if trajectories else None
    out = env.rollout(int(p.done_steps), policy=policy, monte_carlo=True, policy_tiles=tiles,
                      record_trajectory=trajectories)
    mc = out["mc"].cpu().numpy()                    # the one read-back: [M, MC_NCOL] (models x block with a list)
    rec = torch.cat([row0[None], out["trajectory"]]).cpu().numpy() if trajectories else None
    results = []
    for b in range(1 if models is None else len(models)):
        raw = mc[b * block:b * block + m]
        res = mc_columns(raw, p.dt)
        if return_raw:
            res["raw"] = raw
        if trajectories:
            res["trajectory"] = trajectory_fields(rec[:, :, b * block:b * block + m], p.dt)
        results.append(res)
    return results[0] if models is None else results


def _record_row_of_state(env) -> torch.Tensor:
    """The current state of every env as one row of the trajectory record, [TR_NCOL, N] on the device."""
    n = env.num_envs
    err, col, suc, koz = env.errors()
    return torch.cat([env.f64[:N.NF64, :n], env.i32[:N.NI32, :n].double(), err.t(), koz[None], col[None].double(),
                      suc[None].double()])


def trajectory_fields(record: np.ndarray, dt: float) -> dict:
    """[L + 1, TR_NCOL, M] trajectory record (sample 0 = the state at launch, then one row per step of an evaluator
    launch) -> per-episode series, every array [M, L + 1, ...]: ``t`` (s, round(step * dt, 3) as RendezvousEnv.t),
    ``rc vc wc wt`` [.., 3] and ``qc qt`` [.., 4] (the state), ``errors`` [.., 4] (get_errors: m, m/s, rad, rad/s),
    ``dist_from_koz``, ``collision`` (check_collision), ``total_delta_v``, ``total_reward`` (the return so far);
    ``length`` [M] is the episode length in steps.  Samples after ``length`` repeat the last one (a finished env stops
    stepping)."""
    rec = np.asarray(record, dtype=np.float64).transpose(2, 0, 1)          # [M, L + 1, TR_NCOL]
    out = dict(t=np.round(rec[:, :, N.TR_I_STEP] * dt, 3))
    for name, (row, k) in (("rc", (N.RCX, 3)), ("vc", (N.VCX, 3)), ("wc", (N.WCX, 3)), ("wt", (N.WTX, 3)),
                           ("qc", (N.QCW, 4)), ("qt", (N.QTW, 4))):
        out[name] = rec[:, :, row:row + k].copy()
    out["errors"] = rec[:, :, N.TR_POS_ERR:N.TR_ROT_ERR + 1].copy()
    out["dist_from_koz"] = rec[:, :, N.TR_KOZ].copy()
    out["collision"] = rec[:, :, N.TR_COLLISION] != 0
    out["total_delta_v"] = rec[:, :, N.TDV].copy()
    out["total_reward"] = rec[:, :, N.EPRET].copy()
    out["length"] = (rec[:, -1, N.TR_I_STEP] - rec[:, 0, N.TR_I_STEP]).astype(np.int64)
    return out


def mc_columns(mc: np.ndarray, dt: float) -> dict:
    """[M, MC_NCOL] device results -> the workbook columns (monte_carlo.py:190-203): seconds and degrees."""
    return dict(
        ep_len=np.round(mc[:, N.MC_EP_LEN] * dt, 3), num_collisions=mc[:, N.MC_NUM_COLLISIONS].astype(np.int64),
        collided=mc[:, N.MC_COLLIDED].astype(np.int64), total_reward=mc[:, N.MC_TOTAL_REWARD].copy(),
        total_delta_v=mc[:, N.MC_TOTAL_DELTA_V].copy(), num_successes=mc[:, N.MC_NUM_SUCCESSES].astype(np.int64),
        succeeded=mc[:, N.MC_SUCCEEDED].astype(np.int64), min_dist_from_koz=mc[:, N.MC_MIN_KOZ].copy(),
        pos_error=mc[:, N.MC_POS_ERR].copy(), vel_error=mc[:, N.MC_VEL_ERR].copy(),
        att_error=np.degrees(mc[:, N.MC_ATT_ERR]), rot_error=np.degrees(mc[:, N.MC_ROT_ERR]))


def sensitivity_grid(include_invalid: bool = False) -> list:
    """The parameter grid of /root/reference/sensitivity_analysis.py:97-134 as a list of ``make_env`` config dicts:
    rc0 {10..50} x wt0 rad{0, 1.25, 2.5} x koz_radius {2, 5, 10} x corridor_half_angle rad{15, 25, 30, 35, 45} x
    h {400, 600, 800, 1000, 2000} km x dt {0.25, 0.5, 1, 2, 4}.  koz_radius = 2 violates the constructor's assertion
    ``|rd| < koz_radius`` (rendezvous_env.py:155 -- the reference raises there), so those 1,875 of the 5,625
    combinations are left out unless ``include_invalid``."""
    import itertools
    rad = np.radians
    axes = dict(rc0=[10, 20, 30, 40, 50], wt0=[float(rad(v)) for v in (0, 1.25, 2.5)], koz_radius=[2, 5, 10],
                corridor_half_angle=[float(rad(v)) for v in (15, 25, 30, 35, 45)],
                h=[400e3, 600e3, 800e3, 1000e3, 2000e3], dt=[0.25, 0.5, 1, 2, 4])
    grid = [dict(zip(axes, combo)) for combo in itertools.product(*axes.values())]
    return grid if include_invalid else [g for g in grid if g["koz_radius"] > 2]


def evaluate_sweep(policy, param_sets, episodes_per_set=1024, reward_kwargs=None, device="cuda", seed=0,
                   rank=0, world_size=1, **common) -> list:
    """Sensitivity sweep as ONE batch (BASELINE.json configs[4]; the axes of sensitivity_analysis.py:97-134 --
    ``rc0, wt0, koz_radius, corridor_half_angle, h, dt``): every entry of ``param_sets`` (a dict of ``make_env``
    config keys) becomes a contiguous block of ``episodes_per_set`` stochastic envs with its own constants; the
    blocks run under the deterministic policy fused into the rollout in evaluator mode (one launch per block, the
    first episode of every env is scored on the device).  With ``world_size`` > 1 the parameter sets are sharded over
    ranks by :func:`~.distributed.shard_range` (every rank returns its own sets; reset streams are keyed by the
    global env id, so a set's result does not depend on the sharding).  Returns one dict per set: mean return /
    length, success and collision rates (the metrics of custom_callbacks.py:285-298).

    ``policy`` may be a list or tuple of :class:`~.policy.MlpPolicy`, as long as ``param_sets``: set i is then scored with
    model i (sensitivity_analysis.py trains one model per set), all sets still in one launch through a policy table.
    The list is global, sharded with the sets; ``episodes_per_set`` must then be a multiple of 128 (one table tile)."""
    from .distributed import shard_range
    models = list(policy) if isinstance(policy, (list, tuple)) else None
    if models is not None:
        if len(models) != len(param_sets):
            raise ValueError(f"{len(models)} policies for {len(param_sets)} parameter sets")
        if episodes_per_set % N.POLICY_TILE:
            raise ValueError(f"episodes_per_set must be a multiple of {N.POLICY_TILE} with one policy per set")
    if episodes_per_set % 32:
        raise ValueError("episodes_per_set must be a multiple of 32")
    lo_set, hi_set = shard_range(len(param_sets), world_size, rank)
    mine = list(param_sets[lo_set:hi_set])
    if not mine:
        return []
    tiles = None
    if models is not None:
        policy = PolicyTable(models[lo_set:hi_set])
        tiles = np.repeat(np.arange(len(mine)), episodes_per_set // N.POLICY_TILE)
    batches = []
    for ps in mine:
        kw = config_to_kwargs(dict(common, **ps), stochastic=True)
        batches.append((episodes_per_set, {k: v for k, v in kw.items() if v is not None}))
    n = episodes_per_set * len(batches)
    env = BatchedRendezvousEnv(n, device=device, seed=seed, env_offset=lo_set * episodes_per_set, auto_reset=False,
                               track_stats=False, reward_kwargs=reward_kwargs, param_batches=batches)
    env.reset()
    steps = max(int(g.params.done_steps) for g in env.groups)
    mc = env.rollout(steps, policy=policy, monte_carlo=True, policy_tiles=tiles)["mc"]
    res = torch.stack([mc[:, N.MC_TOTAL_REWARD], mc[:, N.MC_EP_LEN], (env.success > 0).double(),
                       (env.collided > 0).double()], dim=1).cpu().numpy()        # flags are frozen at the first done
    out = []
    for ps, g in zip(mine, env.groups):
        r = res[g.lo:g.hi]
        out.append(dict(params=dict(ps), episodes=g.n, mean_return=float(r[:, 0].mean()),
                        mean_length_s=float(r[:, 1].mean() * g.params.dt), success_rate=float(r[:, 2].mean()),
                        collision_rate=float(r[:, 3].mean())))
    return out
