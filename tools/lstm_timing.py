"""Timing of the recurrent actor step (rdv_lstm_policy_step) against the same step in torch fp32 with TF32 disabled
(nn.LSTM single step + the 64-64 head), alternated launch by launch with CUDA events, and of evaluate_batch with an
LstmPolicy on the 1000 published initial conditions end to end.  Prints the card and its power limit first.

    python tools/lstm_timing.py [--reps 50]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from lstm_ref import H, actor_keys, make_state_dict                        # noqa: E402

# per env-step: executed = 3 fp16 products over the padded K (gates K = 288, N = 1024; head 256->64, 64->64, 64->16)
EXEC_FLOP = 3 * 2 * (4 * H * 288 + 64 * H + 64 * 64 + 16 * 64)
ALGO_FLOP = 2 * (4 * H * (17 + H) + 64 * H + 64 * 64 + 6 * 64)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def event_time(fn, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) * 1e3 / reps                             # us per call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    from reinforcement_learning_rendezvous_b200 import LstmPolicy, evaluate_batch
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    print("card (name, power limit, max SM clock):", card())
    sd = make_state_dict("torch", seed=0)
    pol = LstmPolicy(sd)
    lstm = torch.nn.LSTM(17, H).cuda()
    w = {k: torch.as_tensor(v, device="cuda") for k, v in actor_keys(sd).items()}
    with torch.no_grad():
        for k in ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"):
            getattr(lstm, k).copy_(w["lstm_actor." + k])
    rng = np.random.default_rng(0)
    print(f"FLOP per env-step: algorithmic {ALGO_FLOP / 1e6:.3f} M, executed on the tensor cores {EXEC_FLOP / 1e6:.3f} M")
    print(f"{'n':>8} {'kernel us':>10} {'torch fp32 us':>14} {'speed-up':>9} {'kernel TFLOP/s exec':>20} "
          f"{'fp32 TFLOP/s algo':>18}")
    for n in (1000, 65536, 131072):
        obs = torch.as_tensor(rng.uniform(-1, 1, (n, 17)).astype(np.float32), device="cuda")
        h = torch.as_tensor(rng.uniform(-1, 1, (H, n)).astype(np.float32), device="cuda")
        c = torch.as_tensor(rng.standard_normal((H, n)).astype(np.float32), device="cuda")
        out = (torch.empty((n, 6), device="cuda"), torch.empty((H, n), device="cuda"), torch.empty((H, n), device="cuda"))
        ht, ct = h.t().contiguous()[None], c.t().contiguous()[None]

        def kernel():
            pol.forward(obs, h, c, None, out=out)

        def reference():
            with torch.no_grad():
                o, _ = lstm(obs[None], (ht, ct))
                a = torch.tanh(o[0] @ w["mlp_extractor.policy_net.0.weight"].T + w["mlp_extractor.policy_net.0.bias"])
                a = torch.tanh(a @ w["mlp_extractor.policy_net.2.weight"].T + w["mlp_extractor.policy_net.2.bias"])
                torch.clamp(a @ w["action_net.weight"].T + w["action_net.bias"], -1, 1)

        for f in (kernel, reference):                                       # warm-up of both shapes
            event_time(f, 5)
        tk, tr = [], []
        for _ in range(5):                                                  # alternate the two, 5 rounds
            tk.append(event_time(kernel, args.reps))
            tr.append(event_time(reference, args.reps))
        k_us, r_us = float(np.median(tk)), float(np.median(tr))
        print(f"{n:>8} {k_us:>10.1f} {r_us:>14.1f} {r_us / k_us:>8.2f}x {EXEC_FLOP * n / k_us / 1e6:>20.1f} "
              f"{ALGO_FLOP * n / r_us / 1e6:>18.1f}   (kernel rounds {np.round(tk, 1).tolist()}, torch "
              f"{np.round(tr, 1).tolist()})")
    ics = np.load(os.path.join(ROOT, "tests", "golden", "mc.npz"))["ic_raw"]
    evaluate_batch(pol, ics)                                                # warm-up
    times = []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = evaluate_batch(pol, ics)
        times.append(time.perf_counter() - t0)
    print(f"evaluate_batch(LstmPolicy, 1000 ICs, dt 1 s, t_max 60 s): {np.median(times) * 1e3:.1f} ms end to end "
          f"(runs {np.round(np.array(times) * 1e3, 1).tolist()}), mean episode {res['ep_len'].mean():.1f} s")


if __name__ == "__main__":
    main()
