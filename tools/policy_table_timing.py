"""Policy tables against the launches they replace (development tool).

(a) M models x E episodes in evaluator mode (nominal config, t_max = 60, dt = 1): ONE policy-table launch against the
    M single-policy launches of E envs each that scoring M models takes without a table.  Both start from the same
    reset states, restored outside the timed window; the outputs are checked to be identical first.
(b) Closed-loop rollout of N envs in K-step launches: a one-entry policy table against the existing fused variant
    (the per-env-step cost of the table path).
Variants are alternated and every measurement is repeated to show the spread.  CUDA events time the launches.

    python tools/policy_table_timing.py [--models 64] [--episodes 1024] [--envs 65536] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, MlpPolicy, PolicyTable  # noqa: E402
from reinforcement_learning_rendezvous_b200.policy import load_state_dict  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name()


def models(m):
    base = load_state_dict(os.path.join(ROOT, "tests", "golden", "policy.npz"))
    out = [MlpPolicy(base)]
    for seed in range(1, m):
        rng = np.random.default_rng(seed)
        out.append(MlpPolicy({k: (v + rng.normal(0.0, 0.1 * float(v.std()) + 1e-4, v.shape)).astype(np.float32)
                              for k, v in base.items()}))
    return out


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def evaluator(m, episodes, reps):
    pols = models(m)
    table = PolicyTable(pols)
    tiles = np.repeat(np.arange(m), episodes // 128)
    kw = dict(auto_reset=False, track_stats=False, dt=1, t_max=60)
    big = BatchedRendezvousEnv(m * episodes, seed=1, **kw)
    big.reset()
    singles = [BatchedRendezvousEnv(episodes, seed=1, env_offset=k * episodes, **kw) for k in range(m)]
    for e in singles:
        e.reset()
    steps = int(big.params.done_steps)
    snap = [(e.f64.clone(), e.i32.clone()) for e in [big] + singles]

    def restore():
        for e, (f, i) in zip([big] + singles, snap):
            e.f64.copy_(f)
            e.i32.copy_(i)
        torch.cuda.synchronize()

    outs = {}

    def run_table():
        outs["table"] = big.rollout(steps, policy=table, policy_tiles=tiles, monte_carlo=True)["mc"]

    def run_singles():
        outs["singles"] = [e.rollout(steps, policy=p, monte_carlo=True)["mc"] for e, p in zip(singles, pols)]

    restore(); run_table(); restore(); run_singles(); torch.cuda.synchronize()        # warm-up of both shapes
    same = bool(torch.equal(outs["table"], torch.cat(outs["singles"])))
    t_tab, t_one = [], []
    for r in range(reps):
        for which in ((0, 1) if r % 2 == 0 else (1, 0)):
            restore()
            (t_tab if which == 0 else t_one).append(timed(run_table if which == 0 else run_singles))
    return dict(models=m, episodes=episodes, steps=steps, identical=same, table_ms=t_tab, singles_ms=t_one)


def closed_loop(n, K, launches, reps):
    pol = models(1)[0]
    table = PolicyTable([pol])
    tiles = [0] * ((n + 127) // 128)
    a = BatchedRendezvousEnv(n, seed=2, auto_reset=True, track_stats=False)
    b = BatchedRendezvousEnv(n, seed=2, auto_reset=True, track_stats=False)
    a.reset()
    b.reset()
    run = {"table": lambda: [a.rollout(K, policy=table, policy_tiles=tiles) for _ in range(launches)],
           "single": lambda: [b.rollout(K, policy=pol) for _ in range(launches)]}
    for f in run.values():
        f()                                                     # warm-up
    torch.cuda.synchronize()
    res = {"table": [], "single": []}
    for r in range(reps):
        for name in (("table", "single") if r % 2 == 0 else ("single", "table")):
            res[name].append(1e3 * timed(run[name]) / (launches * K))
    same = bool(torch.equal(a.f64, b.f64) and torch.equal(a.obs, b.obs))
    return dict(envs=n, steps_per_launch=K, launches=launches, identical=same,
                table_us_per_step=res["table"], single_us_per_step=res["single"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--models", type=int, default=64)
    ap.add_argument("--episodes", type=int, default=1024)
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--launches", type=int, default=40)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", default=None, help="also write the results to this file")
    args = ap.parse_args()
    if args.episodes % 128:
        raise SystemExit("--episodes must be a multiple of 128")
    info = dict(card=card())
    print("card (name, power limit, max SM clock):", info["card"], flush=True)
    ev = evaluator(args.models, args.episodes, args.reps)
    print(f"(a) {ev['models']} models x {ev['episodes']} episodes, evaluator mode, {ev['steps']} steps; outputs "
          f"identical: {ev['identical']}")
    print("    one table launch   ms:", " ".join(f"{x:.2f}" for x in ev["table_ms"]))
    print(f"    {ev['models']} single launches ms:", " ".join(f"{x:.2f}" for x in ev["singles_ms"]))
    print(f"    median speed-up {np.median(ev['singles_ms']) / np.median(ev['table_ms']):.2f}x", flush=True)
    cl = closed_loop(args.envs, args.steps, args.launches, args.reps)
    print(f"(b) {cl['envs']} envs, {cl['launches']} launches of {cl['steps_per_launch']} steps; final state identical: "
          f"{cl['identical']}")
    print("    one-entry table us/step:", " ".join(f"{x:.2f}" for x in cl["table_us_per_step"]))
    print("    fused single    us/step:", " ".join(f"{x:.2f}" for x in cl["single_us_per_step"]), flush=True)
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(info, evaluator=ev, closed_loop=cl), f, indent=1)


if __name__ == "__main__":
    main()
