"""Cost of the trajectory record of the fused rollout (development tool).

(a) Rollouts of N envs (auto-reset, carried reset rows) in K-step launches, with and without ``record_trajectory``, for
    Philox and closed-loop policy actions: microseconds per step, CUDA events around ``launches`` back-to-back launches.
    The two variants run on two envs from the same reset state; their final states are checked to be identical.
(b) ``evaluate_batch`` on the 1,000 initial conditions of tests/golden/mc.npz: without and with ``trajectories``, and the
    host loop of tests/mc_hostloop.py (rdv_policy_forward + rdv_step + rdv_errors per step), host clock around each
    call (each ends in a device-to-host copy).
Variants are alternated and every measurement is repeated to show the spread.

    python tools/trajectory_timing.py [--envs 65536] [--reps 5] [--json out.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, MlpPolicy, evaluate_batch  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name()


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def rollouts(n, K, launches, source, pol, reps):
    envs = {v: BatchedRendezvousEnv(n, seed=2, auto_reset=True, track_stats=False) for v in ("plain", "record")}
    for e in envs.values():
        e.reset()
    kw = dict(policy=pol) if source == "policy" else dict(action_seed=7)
    base = {"plain": 0, "record": 0}

    def run(v):
        def go():
            for _ in range(launches):
                envs[v].rollout(K, step_base=base[v], record_trajectory=v == "record", **kw)
                base[v] += K
        return go
    for v in envs:
        run(v)()                                                # warm-up (module load, allocator)
    torch.cuda.synchronize()
    res = {"plain": [], "record": []}
    for r in range(reps):
        for v in (("plain", "record") if r % 2 == 0 else ("record", "plain")):
            res[v].append(1e3 * timed(run(v)) / (launches * K))
    same = bool(torch.equal(envs["plain"].f64, envs["record"].f64) and torch.equal(envs["plain"].i32, envs["record"].i32))
    return dict(envs=n, source=source, steps_per_launch=K, launches=launches, identical=same,
                plain_us_per_step=res["plain"], record_us_per_step=res["record"])


def evaluator(pol, reps):
    from helpers import golden
    from mc_hostloop import evaluate_batch_hostloop
    ics = golden("mc.npz")["ic_raw"]
    run = {"plain": lambda: evaluate_batch(pol, ics), "trajectories": lambda: evaluate_batch(pol, ics, trajectories=True),
           "hostloop": lambda: evaluate_batch_hostloop(pol, ics)}
    outs = {k: f() for k, f in run.items()}                     # warm-up
    same = all(np.array_equal(outs["plain"][k], outs["trajectories"][k]) for k in outs["plain"])
    res = {k: [] for k in run}
    for r in range(reps):
        order = list(run) if r % 2 == 0 else list(run)[::-1]
        for k in order:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run[k]()
            torch.cuda.synchronize()
            res[k].append(1e3 * (time.perf_counter() - t0))
    return dict(episodes=len(ics), identical_columns=same, ms=res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", default=None, help="also write the results to this file")
    args = ap.parse_args()
    pol = MlpPolicy.load(os.path.join(ROOT, "tests", "golden", "policy.npz"))
    info = dict(card=card())
    print("card (name, power limit, max SM clock):", info["card"], flush=True)
    rows = []
    for source in ("philox", "policy"):
        for K, launches in ((16, 40), (250, 4)):
            r = rollouts(args.envs, K, launches, source, pol, args.reps)
            rows.append(r)
            pm, rm = np.median(r["plain_us_per_step"]), np.median(r["record_us_per_step"])
            print(f"(a) {r['envs']} envs, {source} actions, {launches} launches of {K} steps; final state identical: "
                  f"{r['identical']}")
            print("    without record us/step:", " ".join(f"{x:.2f}" for x in r["plain_us_per_step"]))
            print("    with record    us/step:", " ".join(f"{x:.2f}" for x in r["record_us_per_step"]))
            print(f"    median cost of the record {rm - pm:+.2f} us/step ({100 * (rm / pm - 1):+.1f} %), "
                  f"{args.envs * 272 / (rm * 1e-6) / 1e9:.0f} GB/s of record stores", flush=True)
    ev = evaluator(pol, args.reps)
    print(f"(b) evaluate_batch, {ev['episodes']} golden initial conditions; columns identical with and without "
          f"trajectories: {ev['identical_columns']}")
    for k, v in ev["ms"].items():
        print(f"    {k:13s} ms:", " ".join(f"{x:.2f}" for x in v), f"(median {np.median(v):.2f})", flush=True)
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(info, rollouts=rows, evaluator=ev), f, indent=1)


if __name__ == "__main__":
    main()
