#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched RendezvousEnv step/reset hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # this repo's CUDA path
    python bench.py --impl reference [--steps K] [--warmup W]    # the reference algorithm on the host cores

Workload (BASELINE.json configs[1]): 65,536 envs per GPU, default constructor parameters, uniform random
actions, auto-reset on, fp64 state.  A "step" is one env step of every env of the batch.  Prints ONE JSON line
(rank 0).  Keys:

  value / ms_per_step   device-resident loop: exactly K timed steps as fused rollouts (rdv_rollout, --steps-per-launch
                        steps per launch), fp64 U(-1,1) actions drawn on the device (Philox), CUDA events, max over
                        ranks
  step_api              the same workload through the one-launch-per-step entry point (rdv_step) with fp64 actions
                        from a pre-generated 64-step device ring (201 MB, larger than L2)
  e2e                   same metric through RendezvousVecEnv.step(numpy actions): pinned H2D of the actions and
                        D2H of obs / reward / done / terminal obs / episode records inside the timed region
  roofline              dominant kernel (rollout_kernel, the only kernel of the timed region) timed per launch with
                        CUDA events inside the timed region; fp64-pipe bound: algorithmic flop per env-step
                        (SURVEY.md 8d) x envs x steps / duration vs the DFMA peak measured in this run; the HBM view
                        is in roofline["hbm"]
  cpu_baseline          the reference algorithm (numpy restatement incl. scipy's RK45, bit-exact vs the reference)
                        under a SubprocVecEnv-protocol harness on all host cores, bounded sample
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ENVS_PER_GPU = 65536
WARMUP_MIN = 1000
LEAD_IN_LAUNCHES = 10
RING = 64
METRIC = "env-steps/sec"
UNIT = "env-steps/s"
# SURVEY.md 8(d): F_step = 1202 + 1930 * k fp64 flop with k = mean accepted RK45 steps per solve_ivp call;
# B_step = 511 B (fp64 actions) / 487 B (fp32 actions) of state + action + output traffic per env-step.
F_STEP_BASE, F_STEP_PER_RK = 1202.0, 1930.0
B_STEP_F64, B_STEP_F32 = 511.0, 487.0
F_STEP_CLOSED_FORM = 560.0


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons during the timed region (pynvml; nvidia-smi as a fallback)."""

    def __init__(self, index=0, period=0.01):
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nvml = None
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        return self

    def _run(self):
        names = {}
        if self._nvml is not None:
            n = self._nvml
            for key in ("nvmlClocksEventReasonHwSlowdown", "nvmlClocksEventReasonHwThermalSlowdown",
                        "nvmlClocksEventReasonSwThermalSlowdown", "nvmlClocksEventReasonSwPowerCap",
                        "nvmlClocksThrottleReasonHwSlowdown", "nvmlClocksThrottleReasonHwThermalSlowdown",
                        "nvmlClocksThrottleReasonSwThermalSlowdown", "nvmlClocksThrottleReasonSwPowerCap"):
                if hasattr(n, key):
                    label = key.replace("nvmlClocksEventReason", "").replace("nvmlClocksThrottleReason", "")
                    names[getattr(n, key)] = {"HwSlowdown": "hw_slowdown", "HwThermalSlowdown": "hw_thermal_slowdown",
                                              "SwThermalSlowdown": "sw_thermal_slowdown",
                                              "SwPowerCap": "sw_power_cap"}[label]
        while not self._stop.is_set():
            try:
                if self._nvml is not None:
                    n = self._nvml
                    self.samples.append(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM))
                    get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                        getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
                    mask = get(self._h)
                    for bit, label in names.items():
                        if mask & bit:
                            self.reasons.add(label)
                else:
                    import subprocess
                    out = subprocess.run(
                        ["nvidia-smi", f"--id={self.index}", "--format=csv,noheader,nounits",
                         "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
                         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                         "clocks_event_reasons.sw_power_cap"], capture_output=True, text=True, timeout=5).stdout
                    f = [x.strip() for x in out.strip().split(",")]
                    self.samples.append(int(f[0]))
                    self.max_mhz = int(f[1])
                    for label, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                        f[2:6]):
                        if v.lower().startswith("active"):
                            self.reasons.add(label)
            except Exception:
                pass
            self._stop.wait(self.period)

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=5)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# --------------------------------------------------------------------------------------------------------------
# reference arm: the reference algorithm on the host cores
# --------------------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle.subproc_vec_env import time_subproc_baseline
    cores = args.ref_procs or os.cpu_count() or 1
    res = time_subproc_baseline(steps=args.steps, warmup=max(args.warmup, 1), n_procs=cores, seed=0,
                                max_seconds=args.ref_max_seconds, min_seconds=args.ref_min_seconds)
    sample = (f"{res['steps']} VecEnv steps of {cores} envs (one env per process, Pipe protocol, auto-reset in the "
              f"worker), random fp64 actions, default RendezvousEnv parameters; {res['seconds']:.1f} s")
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": res["steps"], "warmup": max(args.warmup, 1), "ms_per_step": 1e3 * res["seconds"] / max(res["steps"], 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "RendezvousEnv step/reset, random actions, reference algorithm on host cores "
                               "(bounded sample of the 65,536-env workload: one env per core)",
                   "envs": cores, "harness": "SubprocVecEnv protocol (oracle/subproc_vec_env.py)",
                   "env": "oracle/rdv_oracle.py OracleEnv: numpy restatement of the reference env incl. scipy's adaptive "
                          "RK45, bit-exact vs the reference (the Python reference tree cannot travel)"},
        "cpu_baseline": {"value": res["value"], "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# --------------------------------------------------------------------------------------------------------------
# this repo's arm
# --------------------------------------------------------------------------------------------------------------
def cpu_baseline_leg(args):
    """The oracle timed on the host cores (SubprocVecEnv protocol, single process, plain-C port): bench.py's
    `cpu_baseline` object.  Runs in a child interpreter of the CUDA arm (`--cpu-baseline-only`)."""
    from oracle.subproc_vec_env import time_c_port, time_single_process, time_subproc_baseline
    cores = os.cpu_count() or 1
    res = time_subproc_baseline(steps=100000, warmup=2, n_procs=cores, seed=0, max_seconds=args.cpu_seconds)
    single = time_single_process(seconds=min(3.0, args.cpu_seconds))
    cport = time_c_port(n_envs=4096, steps=10, threads=cores)
    return {
        "value": res["value"], "unit": UNIT, "cores": cores, "kind": "port",
        "sample": f"{res['steps']} VecEnv steps x {cores} envs (one per process, SubprocVecEnv protocol), "
                  f"random fp64 actions, numpy restatement of the reference env (bit-exact), "
                  f"{res['seconds']:.1f} s",
        "single_process_value": single["value"],
        "single_process_sample": f"one env in-process (DummyVecEnv style, main.py:33-34), {single['steps']} steps",
        "c_port_value": cport["value"],
        "c_port_sample": f"plain-C oracle, {cport['envs']} envs x {cport['steps']} steps on {cores} threads",
    }


def dump_outputs(out_dir, env, stats, limit=64 << 20):
    """Write what the timed rollout hands its caller after its last step, so that two builds can be compared output
    for output (the inputs are a function of the arguments alone): obs.npy (float32 [envs, 17], the observation the
    last step returned), state.npy (float64 [envs, 20], the env state it left) and stats.npy (float64 [16], the
    statistics of the timed steps summed over ranks, _native.STAT_NAMES order).  When the rows do not fit in `limit`
    bytes, a fixed seeded sample of envs is written instead, their indices in env_index.npy (float64)."""
    import numpy as np
    from reinforcement_learning_rendezvous_b200 import _native as N
    arrays = {"obs": env.obs.cpu().numpy(), "state": env.get_state().cpu().numpy()}
    n = env.num_envs
    per_env = sum(a.itemsize * a.shape[1] for a in arrays.values())
    budget = limit - 8 * N.NSTATS - 4096                   # 4 KB for the .npy headers
    if n * per_env > budget:
        rows = np.sort(np.random.default_rng(0).choice(n, budget // (per_env + 8), replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["env_index"] = rows.astype(np.float64)
    arrays["stats"] = stats.cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_cuda(args):
    import numpy as np
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    # CPU baseline first (rank 0, N = 1 only), in a child interpreter: the 16 worker processes, the numpy oracle's
    # object churn and the C oracle's threads leave this process untouched.  (Run in-process, whatever the leg left
    # behind -- most likely a fragmented small-object heap -- made the end-to-end leg's host side 18 % slower:
    # 1.14 against 0.96 ms per step, measured with and without --no-cpu-baseline.)
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        child = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-baseline-only",
                                "--cpu-seconds", str(args.cpu_seconds)], capture_output=True, text=True)
        try:
            if child.returncode != 0:
                raise RuntimeError(child.stderr[-2000:])
            cpu_baseline = json.loads(child.stdout.strip().splitlines()[-1])
        except Exception as exc:                      # no child interpreter to be had: time the leg in this process
            print("cpu baseline leg: child failed, running in-process:", exc, file=sys.stderr)
            cpu_baseline = cpu_baseline_leg(args)

    import torch
    import torch.distributed as dist
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, RendezvousVecEnv, _native as N
    from reinforcement_learning_rendezvous_b200.distributed import OverlappedStatsReducer, all_reduce_stats

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device for its own arm (there is no CPU fallback); "
                         "use --impl reference for the host baseline")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = args.envs
    K, W = args.steps, args.warmup

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t[0])
        return ms

    # ---------------- device-resident leg: fused rollouts, KL steps per launch, Philox actions ----------------
    # The timed region is exactly K steps: one K-step rollout (launches of at most KL steps).  The statistics
    # all-reduce (NCCL, N > 1) is issued asynchronously on the rollout's statistics row at its end and waited for
    # after the region, and one SM is left free for it (RdvRolloutIO.sm_reserve).
    KL = max(1, min(args.steps_per_launch, K))
    launches = [KL] * (K // KL) + ([K % KL] if K % KL else [])
    env = BatchedRendezvousEnv(n, device=dev, seed=args.seed, env_offset=rank * n, auto_reset=True,
                               integrator=args.integrator)
    env.sm_reserve = 1 if world > 1 else 0
    env.reset()
    done_steps = 0
    # at least WARMUP_MIN warm-up steps: every episode of the batch starts at the reset above, and until their ends
    # have spread out, the resets come in bursts (profiles/bench_short_region.md)
    W_eff = max(W, WARMUP_MIN)
    env.rollout(W_eff, action_seed=args.seed + 1, step_base=0)
    done_steps = W_eff
    red = OverlappedStatsReducer(dev, capacity=4096)
    # one untimed pass of the timed launches: warms the K-step launch shapes and every torch op and the collective
    # the timed region issues
    env.stats = red.begin()
    for kl in launches:
        env.rollout(kl, action_seed=args.seed + 1, step_base=done_steps)
        done_steps += kl
    red.end()
    red.reset()
    n_l = len(launches)
    sampler = ClockSampler(local_rank).start() if rank == 0 else None
    # region start and end are the first and last of the per-launch events: one event record between two launches,
    # as between any two timed launches (every record costs the stream a few microseconds)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(n_l + 1)]
    barrier()
    # untimed lead-in launches queued ahead of the region: the first timed launch then starts as a launch inside a
    # long stream of them does, not after the host's launch latency (one lead-in launch is not enough: see
    # profiles/bench_short_region.md)
    env.stats = None
    for _ in range(LEAD_IN_LAUNCHES):
        env.rollout(KL, action_seed=args.seed + 1, step_base=done_steps)
        done_steps += KL
    ev[0].record()
    first_timed_step = done_steps
    env.stats = red.begin()
    for j, kl in enumerate(launches):
        env.rollout(kl, action_seed=args.seed + 1, step_base=done_steps)
        done_steps += kl
        ev[j + 1].record()
    red.end()
    total_stats = red.finish()
    barrier()
    ms = max_over_ranks(ev[0].elapsed_time(ev[-1]))
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env, total_stats)
    stats = dict(zip(N.STAT_NAMES, total_stats.cpu().tolist()))
    total_steps = stats["steps"]
    assert total_steps == world * n * K, (total_steps, world, n, K)
    value = world * n * K / (ms * 1e-3)
    rk_mean = stats["rk_accepted"] / (2.0 * max(total_steps, 1.0))
    # dominant kernel: rollout_kernel, per-launch durations of the full-size launches inside the timed region
    full = [ev[q].elapsed_time(ev[q + 1]) for q in range(n_l) if launches[q] == KL]
    t_launch = sum(full) / len(full)
    t_step = t_launch / KL
    env.stats = torch.zeros(N.NSTATS, dtype=torch.float64, device=dev)

    # fp64 peak: DFMA probe, best of 6
    blocks, threads, iters = 148 * 8, 256, 4096
    sink = torch.empty(blocks * threads, dtype=torch.float64, device=dev)
    best = 1e30
    for _ in range(6):
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        N.check(N.lib().rdv_fp64_peak_probe(sink.data_ptr(), blocks, threads, iters,
                                            torch.cuda.current_stream().cuda_stream), "fp64 probe")
        p1.record()
        torch.cuda.synchronize()
        best = min(best, p0.elapsed_time(p1))
    fp64_peak = 2.0 * iters * 16 * blocks * threads / (best * 1e-3) / 1e12

    closed = args.integrator == "closed_form"
    f_step = F_STEP_CLOSED_FORM if closed else F_STEP_BASE + F_STEP_PER_RK * rk_mean
    peaks, peak_src = _peaks()
    # state load + store, the reset-row scratch load + store and the final observation, once per launch
    b_step = (386.0 + 2 * 8.0 * N.RESET_ROWS + 68.0) / KL
    ach_tf = f_step * n / (t_step * 1e-3) / 1e12
    ach_gbs = b_step * n / (t_step * 1e-3) / 1e9
    traffic, f_exec, ncu_pipe, ncu_issue, ncu_src, ncu_steady = None, None, None, None, None, None
    try:                                # per-launch facts of the committed ncu capture of this kernel
        with open(os.path.join(ROOT, "profiles", "rollout_traffic.json")) as f:
            tr = json.load(f)
        if tr.get("envs") == n:
            traffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]
            f_exec = tr.get("fp64_flop_per_env_step_executed")
            ncu_pipe = tr.get("fp64_pipe_pct")
            ncu_issue = tr.get("issue_active_pct")
            ncu_src = tr.get("source")
        with open(os.path.join(ROOT, "profiles", "rollout_traffic_250steps.json")) as f:
            ts = json.load(f)
        if ts.get("envs") == n:         # the same kernel in one 250-step launch (steady state)
            ncu_steady = {"steps_per_launch": ts["steps_per_launch"], "fp64_pipe_pct": ts["fp64_pipe_pct"],
                          "issue_slots_pct": ts["issue_active_pct"], "xu_pipe_pct": ts["xu_pipe_pct"],
                          "warp_instructions_per_warp_step": ts["warp_instructions_per_warp_step"],
                          "fp64_instructions_per_warp_step": ts["fp64_instructions_per_warp_step"],
                          "source": ts["source"]}
    except Exception:
        pass
    roofline = {
        "kernel": "rollout_kernel", "bound": "fp64",
        "achieved": ach_tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": ach_tf / fp64_peak, "traffic": traffic,
        "algorithmic_bytes_per_launch": b_step * n * KL,
        "peak_source": "rdv_fp64_peak_probe (DFMA microbenchmark, this run; MEASURED_PEAKS.json has no fp64 entry; "
                       "nominal 37 TFLOP/s)",
        "flop_per_env_step": f_step, "rk45_steps_per_solve": rk_mean, "steps_per_launch": KL,
        # `achieved` counts the reference's formulation (SURVEY.md 8d: 4-component quaternion RK45, 6.65 kflop per
        # env-step).  The kernel integrates the same equation in the invariant plane of the motion (2 components,
        # same step sizes and results) and executes fewer operations; that figure comes from the ncu source page.
        "note": "achieved counts the flops of the reference's formulation (SURVEY.md 8d), as the contract defines "
                "it; the kernel reaches the same results with fewer executed operations (see `executed`), so frac "
                "measures delivered reference arithmetic per second against the fp64 peak and can exceed 1; "
                "ncu_fp64_pipe_pct is what the profiler reports for the fp64 pipe of this kernel",
        "executed": (None if closed or f_exec is None else
                     {"flop_per_env_step": f_exec, "achieved": f_exec * n / (t_step * 1e-3) / 1e12, "unit": "TFLOP/s",
                      "frac": f_exec * n / (t_step * 1e-3) / 1e12 / fp64_peak, "source": ncu_src}),
        "ncu_fp64_pipe_pct": ncu_pipe,
        # the busiest unit of the SM in the same capture: the warp schedulers' issue slots (smsp__issue_active)
        "ncu_issue_slots_pct": ncu_issue,
        "ncu_steady_state": ncu_steady,
        "launch_ms": t_launch, "launch_ms_min": min(full), "launch_ms_max": max(full), "launches_timed": len(full),
        "hbm": {"achieved": ach_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach_gbs / peaks["hbm_gbs"],
                "bytes_per_env_step": b_step, "peak_source": peak_src},
    }

    # ---------------- the same launches with L2 flushed in between (a 256 MB write before each) ----------------
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    F = 8
    fe = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(F)]
    for j in range(F):
        flush.fill_(j & 0xFF)
        fe[j][0].record()
        env.rollout(KL, action_seed=args.seed + 1, step_base=done_steps)
        done_steps += KL
        fe[j][1].record()
    torch.cuda.synchronize()
    ms_flushed = sum(a.elapsed_time(b) for a, b in fe) / F / KL
    del flush

    # ---------------- the same kernel without auto-reset: the first 16 steps after a batch reset ----------------
    env_nr = BatchedRendezvousEnv(n, device=dev, seed=args.seed, env_offset=rank * n, auto_reset=False,
                                  track_stats=False, integrator=args.integrator)
    KN, RN = 16, 16
    ne = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(RN)]
    for j in range(RN + 2):
        env_nr.reset()
        if j >= 2:
            ne[j - 2][0].record()
        env_nr.rollout(KN, action_seed=args.seed + 1, step_base=j * KN)
        if j >= 2:
            ne[j - 2][1].record()
    torch.cuda.synchronize()
    ms_no_reset = sum(a.elapsed_time(b) for a, b in ne) / RN / KN
    del env_nr

    # ---------------- per-step API (rdv_step, one launch per step, fp64 actions from a device ring) ----------------
    gen = torch.Generator(device=dev)
    gen.manual_seed(1 + rank)
    ring = torch.rand((RING, n, 6), dtype=torch.float64, device=dev, generator=gen) * 2 - 1
    KS = min(max(K, 200), 500)
    for k in range(10):
        env.step(ring[k % RING])
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    s0.record()
    for k in range(KS):
        env.step(ring[k % RING])
    s1.record()
    barrier()
    step_ms = max_over_ranks(s0.elapsed_time(s1))
    step_api = {"value": world * n * KS / (step_ms * 1e-3), "unit": UNIT, "steps": KS, "ms_per_step": step_ms / KS,
                "gpu_launches": KS, "kernel": "step_kernel",
                "roofline_frac_fp64": f_step * n / (step_ms / KS * 1e-3) / 1e12 / fp64_peak,
                "actions": f"fp64 U(-1,1), pre-generated {RING}-step device ring ({RING * n * 48 / 1e6:.0f} MB > L2)"}

    # ---------------- closed-loop rollouts with the shipped policy fused into the launch (tensor-core MLP) --------
    # policy_rollout: this workload's batch (65,536 envs per GPU); policy_rollout_1m: BASELINE.json configs[3],
    # 131,072 envs per GPU = 1,048,576 envs on 8 GPUs, with the per-rollout statistics all-reduce in the region.
    policy_rollout = policy_rollout_1m = None
    pol_path = os.path.join(ROOT, "tests", "golden", "policy.npz")
    if os.path.exists(pol_path) and not closed:
        from reinforcement_learning_rendezvous_b200 import MlpPolicy
        pol = MlpPolicy.load(pol_path, device=dev)
        what = ("SB3 MlpPolicy actor 17-64-64-6 tanh (models/mlp_model_best weights), deterministic, "
                "split-fp16 (3 MMAs per product, fp32-level accuracy) tcgen05.mma with TMEM-resident activations inside rollout_kernel")

        def policy_leg(penv, kl):
            penv.sm_reserve = 1 if world > 1 else 0
            for _ in range(2):
                penv.rollout(kl, policy=pol)
            q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            q0.record()
            penv.rollout(kl, policy=pol)
            q1.record()
            torch.cuda.synchronize()
            reps = max(3, math.ceil(args.min_region_ms / max(max_over_ranks(q0.elapsed_time(q1)), 1e-3)))
            if world > 1:
                rt = torch.tensor([reps], dtype=torch.int64, device=dev)
                dist.all_reduce(rt, op=dist.ReduceOp.MAX)
                reps = int(rt[0])
            pred = OverlappedStatsReducer(dev)
            barrier()
            q0.record()
            for r in range(reps):
                penv.stats = pred.begin()
                penv.rollout(kl, policy=pol)
                pred.end()
            pred.finish()
            q1.record()
            barrier()
            pms = max_over_ranks(q0.elapsed_time(q1))
            m = penv.num_envs
            return {"value": world * m * reps * kl / (pms * 1e-3), "unit": UNIT, "ms_per_step": pms / (reps * kl),
                    "steps": reps * kl, "steps_per_launch": kl, "repeats": reps, "envs_per_gpu": m,
                    "total_envs": world * m, "policy": what}

        policy_rollout = policy_leg(env, min(KL, max(K, 16)))
        big = BatchedRendezvousEnv(2 * n, device=dev, seed=args.seed, env_offset=rank * 2 * n, auto_reset=True)
        big.reset()
        policy_rollout_1m = policy_leg(big, 64)
        policy_rollout_1m["config"] = ("BASELINE.json configs[3]: 131,072 envs per GPU (1,048,576 on 8 GPUs), fused "
                                       "MLP policy inference, 64 steps per launch, one NCCL statistics all-reduce per "
                                       "launch (overlapped with the next launch)")
        del big

    # ---------------- end-to-end leg: numpy actions in, numpy results out, through the VecEnv ----------------
    del env
    venv = RendezvousVecEnv(n, device=dev, seed=args.seed, env_offset=rank * n, integrator=args.integrator)
    venv.reset()
    rng = np.random.default_rng(100 + rank)
    host_ring = rng.uniform(-1, 1, (RING, n, 6)).astype(np.float32)
    KE = max(args.e2e_steps, 1)              # a floor of its own: ~2 s of steps whatever --steps is
    for k in range(max(10, min(W, 50))):
        venv.step(host_ring[k % RING])
    checksum = 0.0
    d2h_before = venv.d2h_bytes_total
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for k in range(KE):
        obs, rew, done, infos = venv.step(host_ring[k % RING])
        checksum += float(rew[0])
    e1.record()
    barrier()
    wall = (time.perf_counter() - t0) * 1e3
    e2e_ms = max_over_ranks(max(e0.elapsed_time(e1), wall))
    d2h_e2e = (venv.d2h_bytes_total - d2h_before) // KE       # obs + reward + done of every env, rows of finished ones
    e2e = {"value": world * n * KE / (e2e_ms * 1e-3), "unit": UNIT, "steps": KE,
           "ms_per_step": e2e_ms / KE, "h2d_bytes_per_step": venv.h2d_bytes_per_step,
           "d2h_bytes_per_step": d2h_e2e,
           "extra_fetches": venv.extra_fetches,
           "api": "RendezvousVecEnv.step(np.float32[N,6]) -> (obs, rewards, dones, infos) numpy: one pinned H2D copy, "
                  "one launch, one D2H copy of [count | rewards | dones | obs | finished rows], one synchronise"}

    # the same loop through the array-returning variant (no per-env Python objects)
    barrier()
    t0 = time.perf_counter()
    for k in range(KE):
        obs, rew, done, fin = venv.step_arrays(host_ring[k % RING])
        checksum += float(rew[0]) + fin["episode_return"].sum()
    barrier()
    arr_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    e2e["arrays_api"] = {"value": world * n * KE / (arr_ms * 1e-3), "unit": UNIT, "ms_per_step": arr_ms / KE,
                         "api": "RendezvousVecEnv.step_arrays: same transfers, finished episodes as arrays"}

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return 0
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"batched RendezvousEnv, {n:,} envs per GPU, random actions, fp64 step/reset "
                               "(BASELINE.json configs[1])",
                   "envs_per_gpu": n, "total_envs": world * n, "auto_reset": True, "integrator": args.integrator,
                   "actions": "fp64 U(-1,1) drawn on the device every step from the Philox4x32-10 stream "
                              "(action seed; global env id, step index)",
                   "steps_per_launch": KL, "steps_timed": K, "timed_region_ms": ms,
                   "warmup_steps": W_eff, "first_timed_step": first_timed_step,
                   "timing": "the timed region is one `steps`-step rollout, queued behind %d untimed launches"
                             % LEAD_IN_LAUNCHES,
                   "stats_all_reduce": ("one 16-double NCCL all-reduce per rollout, issued asynchronously in place on the "
                                        "rollout's own statistics row at the end of the region and waited for after it; "
                                        "the rollout leaves 1 SM free for it" if world > 1 else "no-op at N = 1"),
                   "l2": "state lives in registers for the steps of a launch and is re-read from memory once per "
                         "launch; ms_per_step_l2_flushed repeats the launches with a 256 MB L2 flush before each; "
                         "ms_per_step_no_auto_reset = 16-step launches right after a batch reset, auto_reset off "
                         "(includes 1/16 of a launch latency per step)",
                   "ms_per_step_l2_flushed": ms_flushed,
                   "ms_per_step_no_auto_reset": ms_no_reset,
                   "parallelism": f"{world} x independent env shards, no data-path collective; one "
                                  "16-double statistics all-reduce per rollout"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": n_l,
        "roofline": roofline, "cpu_baseline": cpu_baseline, "step_api": step_api,
        "policy_rollout": policy_rollout, "policy_rollout_1m": policy_rollout_1m,
        "episode_stats": {"episodes": stats["episodes"], "mean_length": stats["length_sum"] / max(stats["episodes"], 1),
                          "success_rate": stats["succeeded"] / max(stats["episodes"], 1),
                          "rk_rejected": stats["rk_rejected"], "failures": stats["failures"]},
    }
    print(json.dumps(line), flush=True)
    return 0


def _json_only_stdout():
    """Route everything libraries print on fd 1 (e.g. the NCCL version banner) to stderr and return a file
    object on the original stdout, so that stdout carries exactly one JSON line."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", choices=("cuda", "reference"), default="cuda")
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="envs per GPU")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--integrator", choices=("rk45", "closed_form"), default="rk45")
    ap.add_argument("--e2e-steps", type=int, default=1000)
    ap.add_argument("--min-region-ms", type=float, default=80.0,
                    help="minimum length of a timed region of the policy_rollout legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what they computed as DIR/<name>.npy (see dump_outputs)")
    ap.add_argument("--ref-min-seconds", type=float, default=8.0, help="time floor of the reference arm")
    ap.add_argument("--steps-per-launch", type=int, default=250, help="env steps fused into one rollout launch")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-baseline-only", action="store_true", help="(internal) print the cpu_baseline object and exit")
    ap.add_argument("--ref-procs", type=int, default=0)
    ap.add_argument("--ref-envs", type=int, default=0, help="(ignored; kept for compatibility)")
    ap.add_argument("--ref-max-seconds", type=float, default=150.0)
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "cuda":
        args.warmup = 3
    out = _json_only_stdout()
    sys.stdout = out
    try:
        if args.cpu_baseline_only:
            print(json.dumps(cpu_baseline_leg(args)))
            return 0
        if args.impl == "reference":
            return run_reference(args)
        return run_cuda(args)
    finally:
        out.flush()


if __name__ == "__main__":
    sys.exit(main())
