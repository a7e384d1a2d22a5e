"""TEST CHECKER: the fp64 reference of one LSTM step (rdv_lstm_policy_step, each network of
rdv_lstm_actor_critic_step) together with a per-env, per-output bound on how far the kernel's arithmetic may land from
it, so that one test covers weights from 1e-4 to the loaders' limit and observations from 1e-6 to the clamp.

The kernel (csrc/rdv_lstm.cuh) forms every product of a layer z = W a + b as three tensor-core products of fp16 halves,
a_lo w_hi + a_hi w_lo + a_hi w_hi, the weights staged times 2^10, accumulated in float32 in K-steps of 16 (three MMAs
per K-step into one accumulator); it adds the bias in float32 after the sum and uses expf / tanhf.  Each
pre-activation is bounded by (:func:`layer_bound`)

    |z^ - z| <= TAU sum_k |a_k| |w_k|          the split: the dropped a_lo w_lo, the roundings of the halves
              + 3 ACC sum_s max(|S_s-1|, |S_s|)  the accumulation: S_s the fp64 partial sum after K-step s
              + sum_k min(|a_k|, 2^-25) |w_k|   a lo half below the fp16 normal range: absolute error 2^-25
              + 2^-35 sum_k |a_k|               the same for a staged weight (2^-25 / 2^10)
              + 2^-23 |b| + 2^-24 |z|           the float32 bias (b_ih + b_hh for the gates) and the rounding of z
              + sum_k |w_k| da_k                the error bound da of the layer's own input (head layers)

and the bound is carried to first order through the cell and the head in fp64, each derivative taken at the point of
[z - dz, z + dz] where it is largest (sigma' and tanh' peak at 0), so the bound of a saturated gate stays a bound.
expf, tanhf and the sigmoid's 1 / (1 + e) add FN = 2^-21 (4 ulps) of their value each, a sigmoid that underflows
float32 an absolute 2^-126.

TAU = 2^-20 (9.5e-7).  lstm_step_split_emulation (the split with IEEE float32 accumulation in numpy's order), 2000
rows of random states, LSTM weights from 1e-2 to 1000 times torch's init: the largest |z^ - z| / sum_k |a_k| |w_k| is
2.8e-7 to 3.2e-7 at every scale (at 1e-3 the fp16 subnormal floor makes it 1.0e-6; the floor term covers that).
Dropping one of the three products makes it 2.4e-4 to 2.8e-4, and leaving the weights unscaled 1.1e-3 at weight scale
1e-3 and 1.1e-4 at 1e-2: these break the whole bound 50 to 280 fold (tests/test_lstm_bound_cpu.py).

ACC = 2^-22, two float32 ulps per MMA.  The accumulation term is what a sum whose large terms come first needs: each
later MMA then rounds on the grid of a large partial sum, which sum_k |a_k| |w_k| cannot see.  On a B200 (1000 W) with
TAU alone the kernels' outputs reached 2.7 times the bound with single weights at the limit and 1.5 times with
observations x30 (they fill the first K-step); with one ulp per MMA at most 0.84, with two 0.79 at the limit and 0.44
in every other case of tests/test_gpu_lstm_ranges.py (it prints the worst ratio of each case).
"""
import numpy as np
import torch

from lstm_ref import H

TAU = 2.0 ** -20
ACC = 2.0 ** -22                 # two float32 ulps: what one MMA's accumulation may lose of the partial sum
U = 2.0 ** -24                   # float32 unit roundoff
FN = 2.0 ** -21                  # expf, tanhf, the sigmoid: within 4 ulps of their value
A_FLOOR = 2.0 ** -25             # half the fp16 subnormal spacing: the split's absolute error of a small operand
W_FLOOR = 2.0 ** -35             # the same for a weight staged times 2^10
TINY = 2.0 ** -126               # float32 underflow of a product or a sum
OBS_CLAMP = 60000.0              # the kernels clamp every observation component to +-60000 before the split


def staged_obs(obs):
    """Observations [n, 17] as the kernels stage them: clamped to +-60000, a NaN component as -60000 (fmaxf(-60000,
    NaN) is -60000).  fp64 tensor."""
    obs = torch.as_tensor(obs).double()
    return torch.where(torch.isnan(obs), -OBS_CLAMP, obs.clamp(-OBS_CLAMP, OBS_CLAMP))


def layer_bound(a, w, b_abs, z, da=None, ksteps=None):
    """Bound [n, m] on the kernel's error of z = a w^T + b for the inputs a [n, k] it reads, w [m, k], |b| [m] and the
    fp64 value z [n, m]; da [n, k]: the error bound of a, or None where a is exact.  ``ksteps``: the column edges of
    the kernel's K-steps in a (default: every 16 columns).  fp64 tensors."""
    aa, ww = a.abs(), w.abs()
    out = (TAU * aa + aa.clamp(max=A_FLOOR)) @ ww.T + W_FLOOR * aa.sum(1, keepdim=True) + 2 * U * b_abs + U * z.abs()
    if da is not None:
        out = out + da @ ww.T
    edges = list(range(0, a.shape[1], 16)) + [a.shape[1]] if ksteps is None else ksteps
    partial, seen = torch.zeros_like(z), torch.zeros_like(z)
    for lo, hi in zip(edges[:-1], edges[1:]):
        after = partial + a[:, lo:hi] @ w[:, lo:hi].T
        seen += torch.maximum(partial.abs(), after.abs())
        partial = after
    return out + 3 * ACC * seen + TINY


def _nearest_zero(z, dz):
    """The point of [z - dz, z + dz] nearest to 0."""
    return torch.where(z.abs() <= dz, torch.zeros_like(z), z - torch.sign(z) * dz)


def _dsigmoid(z, dz):
    x = _nearest_zero(z, dz)
    return torch.sigmoid(x) * torch.sigmoid(-x)


def _dtanh(z, dz):
    return torch.cosh(_nearest_zero(z, dz)).pow(-2)


def _head(a, da, layers):
    """Tanh layers then a linear output: (out, dout) of the head [(w0, b0), (w1, b1), (w2, b2)] on a, da."""
    for i, (w, b) in enumerate(layers):
        z = a @ w.T + b
        dz = layer_bound(a, w, b.abs(), z, da)
        if i == len(layers) - 1:
            return z, dz
        a = torch.tanh(z)
        da = _dtanh(z, dz) * dz + FN * a.abs() + TINY


def step_bound(sd, obs, h, c, episode_start=None, device="cpu"):
    """One step of the network in ``sd`` (lstm_ref's actor key names; recurrent_ref.critic_as_actor gives the critic
    under them) on env-major float32 inputs obs [n, 17], h, c [n, 256], episode_start [n] bool or None: the state is
    zeroed where it is set and the observations are staged as the kernel stages them (:func:`staged_obs`).
    Returns fp64 numpy arrays: ``z`` [n, 1024] the gate pre-activations, ``h``, ``c`` [n, 256] the next state, ``out``
    the head's output before any clip (action_net: the mean, value_net: the value), each with its bound ``dz``, ``dh``,
    ``dc``, ``dout``.  An infinite c' has tanh(c') = +-1 exactly in the kernel and here, so it adds nothing to h'."""
    dev = torch.device(device)
    w = {k: torch.as_tensor(np.asarray(v, dtype=np.float64), device=dev) for k, v in sd.items()}
    obs = staged_obs(obs).to(dev)
    h, c = (torch.as_tensor(np.asarray(x, dtype=np.float64), device=dev) for x in (h, c))
    if episode_start is not None:
        keep = ~torch.as_tensor(np.asarray(episode_start, dtype=bool).reshape(-1, 1), device=dev)
        h, c = torch.where(keep, h, 0.0), torch.where(keep, c, 0.0)
    a = torch.cat([obs, h], dim=1)
    wg = torch.cat([w["lstm_actor.weight_ih_l0"], w["lstm_actor.weight_hh_l0"]], dim=1)
    z = a @ wg.T + (w["lstm_actor.bias_ih_l0"] + w["lstm_actor.bias_hh_l0"])
    # the kernel's A is [obs(17) | 0 x 15 | h]: K-step 0 holds obs 0..15, K-step 1 obs 16, then 16 units of h each
    dz = layer_bound(a, wg, w["lstm_actor.bias_ih_l0"].abs() + w["lstm_actor.bias_hh_l0"].abs(), z,
                     ksteps=[0, 16] + list(range(17, a.shape[1] + 1, 16)))
    (zi, zf, zg, zo), (di, df, dg, do) = z.split(H, dim=1), dz.split(H, dim=1)
    si, sf, so, tg = torch.sigmoid(zi), torch.sigmoid(zf), torch.sigmoid(zo), torch.tanh(zg)
    c2 = sf * c + si * tg
    # a sigmoid below 2^-126 may come out as 0 (expf overflows past 88.7): an absolute error TINY times its factor
    dc2 = (_dsigmoid(zf, df) * c.abs() * df + _dsigmoid(zi, di) * tg.abs() * di + si * _dtanh(zg, dg) * dg
           + (2 * FN + 2 * U) * (sf * c.abs() + si * tg.abs()) + TINY * (c.abs() + 2))
    tc = torch.tanh(c2)
    h2 = so * tc
    dtc = torch.where(torch.isinf(c2), 0.0, _dtanh(c2, dc2) * dc2)
    dh2 = _dsigmoid(zo, do) * tc.abs() * do + so * dtc + (2 * FN + U) * h2.abs() + 2 * TINY
    layers = [(w[f"mlp_extractor.policy_net.{i}.weight"], w[f"mlp_extractor.policy_net.{i}.bias"]) for i in (0, 2)]
    out, dout = _head(h2, dh2, layers + [(w["action_net.weight"], w["action_net.bias"])])
    res = dict(z=z, dz=dz, h=h2, dh=dh2, c=c2, dc=dc2, out=out, dout=dout)
    return {k: v.cpu().numpy() for k, v in res.items()}


def ratio(got, ref, bound):
    """Largest |got - ref| / bound (a NaN anywhere, or an error where the bound is 0, counts as infinite; equal values,
    infinities included, as 0)."""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        r = np.where(got == ref, 0.0, np.abs(got - ref) / bound)
    r = np.where(np.isnan(r), np.inf, r)
    return float(r.max()) if r.size else 0.0
