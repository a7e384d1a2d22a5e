"""Timing of RecurrentPPO's collection step and training loop.  Prints the card and its power limit first.

(a) rdv_lstm_actor_critic_step (actor + critic LSTM steps, Gaussian draw, log-probability, value in ONE launch)
    against the same step in torch fp32 with TF32 off (two nn.LSTM single steps, the heads and the sampling) and
    against two rdv_lstm_policy_step launches (what two networks cost as separate launches of the actor kernel),
    alternated round by round with CUDA events, at 1,000, 16,384 and 65,536 envs;
(b) RecurrentPPO.collect env-steps/s at 16,384 envs and n_steps 128 (host clock around a device synchronise);
(c) RecurrentPPO.update seconds per iteration at that size (batch size and epochs printed).

    python tools/recurrent_ppo_timing.py [--reps 50] [--rounds 3] [--batch 65536] [--epochs 10]
"""
import argparse
import ctypes as C
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from lstm_ref import H, actor_keys, make_state_dict                        # noqa: E402
from lstm_timing import card, event_time                                    # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--epochs", type=int, default=10)
    ap.add_argument("--sizes", type=str, default="1000,16384,65536")
    ap.add_argument("--collect-envs", type=int, default=16384)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, LstmPolicy, _native as N
    from reinforcement_learning_rendezvous_b200.batched_env import _stream_ptr
    from reinforcement_learning_rendezvous_b200.recurrent_ppo import RecurrentActorCritic, RecurrentPPO, RecurrentPPOConfig
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    print("card (name, power limit, max SM clock):", card())
    dev = torch.device("cuda")
    sd = make_state_dict("ppo", seed=0)
    m = RecurrentActorCritic().to(dev)
    with torch.no_grad():
        for k, p in m.state_dict().items():
            p.copy_(torch.as_tensor(sd[k]))
    w = m.kernel_weights()
    actor = LstmPolicy(actor_keys(sd))
    print("(a) one collection step, us per call (median of rounds; each round alternates the three)")
    for n in (int(x) for x in args.sizes.split(",")):
        rng = np.random.default_rng(0)
        obs = torch.as_tensor(rng.uniform(-1, 1, (n, 17)).astype(np.float32), device=dev)
        start = torch.as_tensor((rng.random(n) < 0.05).astype(np.uint8), device=dev)
        st = [torch.as_tensor(rng.uniform(-1, 1, (H, n)).astype(np.float32), device=dev) for _ in range(8)]
        act, env_act = torch.empty((n, 6), device=dev), torch.empty((n, 6), device=dev)
        lp, val = torch.empty(n, device=dev), torch.empty(n, device=dev)
        io = N.RdvLstmStepIO(obs.data_ptr(), start.data_ptr(), *(x.data_ptr() for x in st), act.data_ptr(),
                             env_act.data_ptr(), lp.data_ptr(), val.data_ptr(), 977, 0, 0, n)
        lib, stream = N.lib(), _stream_ptr(dev)

        def fused():
            N.check(lib.rdv_lstm_actor_critic_step(C.byref(w), C.byref(io), n, stream), "step")

        acts2 = torch.empty((n, 6), device=dev)

        def two_launches():
            actor.forward(obs, st[0], st[1], start, out=(act, st[2], st[3]))
            actor.forward(obs, st[4], st[5], start, out=(acts2, st[6], st[7]))

        keep = (1.0 - start.float())[None, :, None]
        h_pi, c_pi, h_vf, c_vf = (x.t().contiguous()[None] for x in st[:4])
        log_std = m.log_std.detach()

        @torch.no_grad()
        def torch_fp32():
            o_pi, _ = m.lstm_actor(obs[None], (keep * h_pi, keep * c_pi))
            o_vf, _ = m.lstm_critic(obs[None], (keep * h_vf, keep * c_vf))
            mean = m.action_net(m.mlp_extractor.policy_net(o_pi[0]))
            v = m.value_net(m.mlp_extractor.value_net(o_vf[0]))[:, 0]
            z = torch.randn_like(mean)
            a = mean + log_std.exp() * z
            logp = (-0.5 * z * z - log_std).sum(-1) - 3 * np.log(2 * np.pi)
            return a.clamp(-1, 1), logp, v

        for fn in (fused, two_launches, torch_fp32):
            event_time(fn, 5)
        rounds = {"fused": [], "two_launches": [], "torch_fp32": []}
        for _ in range(args.rounds):
            for name, fn in (("fused", fused), ("two_launches", two_launches), ("torch_fp32", torch_fp32)):
                rounds[name].append(event_time(fn, args.reps))
        med = {k: float(np.median(v)) for k, v in rounds.items()}
        print(f"  n {n:6d}: rdv_lstm_actor_critic_step {med['fused']:8.1f}  two rdv_lstm_policy_step {med['two_launches']:8.1f}"
              f"  torch fp32 {med['torch_fp32']:8.1f}   rounds {({k: [round(x, 1) for x in v] for k, v in rounds.items()})}")
        del st, obs
        torch.cuda.empty_cache()

    n, T = args.collect_envs, 128
    env = BatchedRendezvousEnv(n, seed=3, auto_reset=True)
    tr = RecurrentPPO(env, RecurrentPPOConfig(n_steps=T, batch_size=args.batch, n_epochs=args.epochs, n_evals=16))
    print(f"(b) RecurrentPPO.collect at {n} envs x {T} steps; (c) update with batch {args.batch}, {args.epochs} epochs")
    adv, ret = tr.collect()                                                 # warm-up (and a buffer for the update)
    torch.cuda.synchronize()
    for r in range(args.rounds):
        t0 = time.perf_counter()
        adv, ret = tr.collect()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        tr.update(adv, ret)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        print(f"  round {r}: collect {t1 - t0:.3f} s = {T * n / (t1 - t0) / 1e6:.2f} M env-steps/s; update {t2 - t1:.2f} s")


if __name__ == "__main__":
    main()
