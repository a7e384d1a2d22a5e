"""The bookkeeping a batch of envs should report, from the C oracle.

``Ledger`` steps ``oracle.c_oracle.COracleBatch`` and accumulates, in numpy, what the 16 statistics slots (RDV_S_*)
and the per-episode record (RDV_EP_*, RdvFinishedRow) should hold by the rules stated next to the RDV_S_* enum in
include/rdv_b200.h:

* steps, reward_sum: every env-step taken and its reward (evaluator mode: up to and including the first done);
* episodes, end_*: every env-step that returned done, by end reason -- again at every step of an env that keeps
  stepping past its end without auto-reset;
* return_sum, length_sum, delta_v_sum, delta_w_sum, succeeded, collided: at each such step, the episode return,
  the step counter, total_delta_v / total_delta_w, success counter > 0 and the sticky collided flag;
* rk_accepted: accepted steps of every solve that completed; rk_rejected: rejected attempts of every solve;
* failures: one per env-step in which any solve failed.

The episode return is a sequential fp64 sum per env (how RDV_EPRET accumulates it); the slots are summed with
math.fsum, and ``tolerance()`` gives each fp64 slot's scale, sum(max(|term|, 1)).
"""
import math

import numpy as np

from helpers import REL_TOL
from oracle import c_oracle as CO

STAT_NAMES = ("steps", "episodes", "return_sum", "length_sum", "succeeded", "collided", "delta_v_sum",
              "delta_w_sum", "end_obs", "end_time", "end_bubble", "end_attitude", "reward_sum",
              "rk_accepted", "rk_rejected", "failures")
FLOAT_STATS = ("return_sum", "delta_v_sum", "delta_w_sum", "reward_sum")
INT_STATS = tuple(k for k in STAT_NAMES if k not in FLOAT_STATS)
END_KEYS = ("end_obs", "end_time", "end_bubble", "end_attitude")


class Ledger:
    """n envs with global ids ``env_offset + arange(n)``, reset from the Philox stream (seed; env id, episode).

    :param auto_reset: envs whose step returned done restart from (seed; env id, episode + 1) before the next step
    :param stop_at_first_done: evaluator mode -- an env takes no further step after its first done
    :param threads: host threads of the oracle's step
    """

    def __init__(self, params, n, seed, env_offset=0, auto_reset=True, stop_at_first_done=False, threads=8):
        self.p, self.n, self.seed = params, int(n), int(seed)
        self.ids = int(env_offset) + np.arange(self.n)
        self.auto_reset, self.stop = bool(auto_reset), bool(stop_at_first_done)
        self.threads = threads
        self.orc = CO.COracleBatch(params, self.n)
        self.episode = np.zeros(self.n, dtype=np.int32)
        self.length = np.zeros(self.n, dtype=np.int64)
        self.ret = np.zeros(self.n)
        self.alive = np.ones(self.n, dtype=bool)
        self.steps_taken = np.zeros(self.n, dtype=np.int64)
        self.terms = {k: [] for k in STAT_NAMES}
        self.records = []          # one dict per finished episode, in step order
        self.last_rk = None

    # ---- state -------------------------------------------------------------------------------------------------
    def reset(self, episode=1):
        """reset() of every env with episode index ``episode`` (BatchedRendezvousEnv.reset() bumps 0 -> 1)."""
        self.episode[:] = episode
        self.orc.reset_from_uniforms(CO.philox_uniforms(self.seed, self.ids, self.episode))
        self.length[:] = 0
        self.ret[:] = 0.0
        self.alive[:] = True

    def set_state(self, state20, recompute_flags=True):
        """Inject states with zeroed counters (BatchedRendezvousEnv.set_state + refresh_flags)."""
        self.orc.set_state(state20, recompute_flags=recompute_flags)
        self.length[:] = 0
        self.ret[:] = 0.0
        self.alive[:] = True

    @property
    def state(self):
        return self.orc.state

    # ---- one env-step of every env ------------------------------------------------------------------------------
    def step(self, actions):
        """Returns (rewards, dones) of the envs that took this step (0 / 0 for an evaluator env that has stopped)."""
        o = self.orc
        live = self.alive.copy()
        frozen = (o.state.copy(), o.aux.copy(), o.flags.copy()) if not live.all() else None
        o.step(actions, threads=self.threads)
        rew, done, reason, rk = o.rew.copy(), o.done.astype(bool), o.reason.copy(), o.rk.copy()
        if frozen is not None:     # an env that has stopped keeps its state
            o.state[~live], o.aux[~live], o.flags[~live] = frozen[0][~live], frozen[1][~live], frozen[2][~live]
        rew[~live] = 0.0
        done &= live
        self.last_rk = rk
        self.ret[live] += rew[live]
        self.length[live] += 1
        self.steps_taken[live] += 1
        t = self.terms
        t["steps"].append(np.ones(int(live.sum())))
        t["reward_sum"].append(rew[live])
        rk_l = rk[live]
        t["rk_accepted"].append((np.maximum(rk_l[:, 0], 0) + np.maximum(rk_l[:, 1], 0)).astype(float))
        t["rk_rejected"].append(rk_l[:, 2].astype(float))
        t["failures"].append(((rk_l[:, 0] < 0) | (rk_l[:, 1] < 0)).astype(float))
        d = np.flatnonzero(done)
        if d.size:
            tdv, tdw = o.aux[d, 0].copy(), o.aux[d, 1].copy()        # before a reset overwrites them
            collided, success = o.flags[d, 0].copy(), o.flags[d, 1].copy()
            t["episodes"].append(np.ones(d.size))
            for j, key in enumerate(END_KEYS):
                t[key].append((reason[d] == j).astype(float))
            t["return_sum"].append(self.ret[d].copy())
            t["length_sum"].append(self.length[d].astype(float))
            t["delta_v_sum"].append(tdv)
            t["delta_w_sum"].append(tdw)
            t["succeeded"].append((success > 0).astype(float))
            t["collided"].append(collided.astype(float))
            term_obs = o.obs[d].copy()
            for j, i in enumerate(d):
                self.records.append(dict(env=int(i), end_reason=int(reason[i]), ret=float(self.ret[i]),
                                         length=int(self.length[i]), success=int(success[j]),
                                         collided=int(collided[j]), delta_v=float(tdv[j]), delta_w=float(tdw[j]),
                                         terminal_obs=term_obs[j]))
            if self.stop:
                self.alive[d] = False
            elif self.auto_reset:
                self.episode[d] += 1
                mask = np.zeros(self.n, dtype=np.uint8)
                mask[d] = 1
                o.reset_from_uniforms(CO.philox_uniforms(self.seed, self.ids, self.episode), mask=mask)
                self.ret[d] = 0.0
                self.length[d] = 0
        return rew, done

    # ---- results ---------------------------------------------------------------------------------------------------
    def _all(self, key):
        return np.concatenate(self.terms[key]) if self.terms[key] else np.zeros(0)

    def stats(self):
        """The 16 slots (STAT_NAMES order), each an fsum of its terms."""
        return {k: math.fsum(self._all(k).tolist()) for k in STAT_NAMES}

    def tolerance(self):
        """Per fp64 slot: sum(max(|term|, 1)), the scale REL_TOL applies to."""
        return {k: math.fsum(np.maximum(np.abs(self._all(k)), 1.0).tolist()) for k in FLOAT_STATS}

    def records_by_env(self):
        """Finished episodes grouped by env, each env's in step order."""
        out = {}
        for r in self.records:
            out.setdefault(r["env"], []).append(r)
        return out


def merge_stats(ledgers):
    """The slots of several ledgers that share one statistics vector (parameter sets, kernel-family groups)."""
    out, tol = {}, {}
    for k in STAT_NAMES:
        out[k] = math.fsum(np.concatenate([lg._all(k) for lg in ledgers]).tolist())
    for k in FLOAT_STATS:
        tol[k] = math.fsum(lg.tolerance()[k] for lg in ledgers)
    return out, tol


def short_solve_steps(got, want):
    """rk_accepted the oracle counts beyond the kernel's, checked and returned.  The kernel forms select_initial_step's
    h0 in float32 (plane_initial_step); SciPy's h0 of a slow body is close to dt / 11 and h grows by the capped factor
    10, so after two steps SciPy can stop up to one float32 ulp of h0 short of dt and take a third step of ~1e-7 s
    that the kernel does not take (e.g. SciPy's 0.0909090857, 0.909090857, 5.7e-8 against the kernel's two).  The
    state after the step agrees to REL_TOL either way; the count may then differ by one step per such solve, a few
    per million."""
    d = want["rk_accepted"] - got["rk_accepted"]
    assert 0 <= d <= 1e-6 * want["rk_accepted"], (got["rk_accepted"], want["rk_accepted"])
    return d


def assert_stats(got, want, tol, what=""):
    """A launch's slots against a ledger's: integer slots exact, fp64 slots within REL_TOL of their scale."""
    for k in INT_STATS:
        assert got[k] == want[k], (what, k, got[k], want[k])
    for k in FLOAT_STATS:
        if math.isnan(want[k]):
            assert math.isnan(got[k]), (what, k, got[k])
        else:
            assert abs(got[k] - want[k]) <= REL_TOL * tol[k], (what, k, got[k], want[k])
