"""GPU: the polynomial form of the attempted plane step (csrc/rdv_math.cuh, rk45_iso_plane) -- the device polynomials
against the stagewise attempt, bodies on both sides of the polynomials' range against the C oracle, and launch shapes."""
import ctypes as C

import numpy as np
import pytest

from helpers import REL_TOL, rel_err
from test_plane_poly_cpu import _header, _horner

pytestmark = pytest.mark.gpu


def _probe(x, op):
    import torch
    from reinforcement_learning_rendezvous_b200 import _native as N
    xd = torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device="cuda")
    yd = torch.empty_like(xd)
    N.check(N.lib().rdv_math_probe(xd.data_ptr(), yd.data_ptr(), xd.numel(), op,
                                   C.c_void_p(torch.cuda.current_stream().cuda_stream)), "rdv_math_probe")
    return yd.cpu().numpy()


def test_polynomial_attempt_matches_the_stagewise_attempt():
    """P, Q (the new point) agree with the six-stage attempt to a few ulp; R, I (the error estimate) to the stagewise
    form's own rounding, which is absolute (~1e-16 h from the cancellation in the E-weighted sum of slopes)."""
    x_max, c = _header()
    x = np.linspace(0.0, x_max, 2001)[1:]
    s = np.sqrt(x)
    P, Q, R, I = (_probe(x, op) for op in (6, 7, 8, 9))
    Ps, Qs, Rs, Is = (_probe(x, op) for op in (10, 11, 12, 13))
    ulps = lambda a, b: np.abs(a - b) / np.spacing(np.abs(b))
    # the device evaluates the header's polynomials (with FMA) as the host does
    assert ulps(P, 1.0 + x * _horner(c["P1"], x)).max() <= 2.0
    assert ulps(Q, 1.0 + x * _horner(c["Q1"], x)).max() <= 2.0
    assert np.abs(R - _horner(c["R"], x)).max() <= 1e-15 * np.abs(R).max()
    assert np.abs(I - _horner(c["I"], x)).max() <= 1e-15 * np.abs(I).max()
    assert ulps(P, Ps).max() <= 4.0 and ulps(Q, Qs).max() <= 8.0
    assert (np.abs(R - Rs) * x ** 3).max() <= 1e-15 * s.max()           # Re E = x^3 R
    assert (np.abs(I - Is) * s * x ** 2 <= 1e-15 * s).all()                # Im E = s x^2 I
    big = x > 0.25 * x_max                                                  # where the stagewise estimate is sharp
    assert np.abs(R - Rs)[big].max() <= 1e-6 * np.abs(R).max() and np.abs(I - Is)[big].max() <= 1e-6 * np.abs(I).max()


def _bodies(n, rng, x_max, dt):
    """States whose chaser / target solve sees om2 dt^2 = 0.25 |w|^2 dt^2 / |q|^2 spread around X_MAX (0.5 to 2 times),
    with quaternions that are not unit vectors and bodies at rest."""
    st = np.zeros((n, 20))
    st[:, 0:3] = [0.0, -10.0, 0.0] + rng.normal(0, 0.5, (n, 3))
    st[:, 3:6] = rng.normal(0, 0.05, (n, 3))
    for qs, ws in ((slice(6, 10), slice(10, 13)), (slice(13, 17), slice(17, 20))):
        q = rng.normal(size=(n, 4))
        q *= rng.uniform(0.5, 2.0, (n, 1)) / np.linalg.norm(q, axis=1, keepdims=True)
        u = rng.normal(size=(n, 3))
        u /= np.linalg.norm(u, axis=1, keepdims=True)
        x = x_max * np.exp(rng.uniform(np.log(0.5), np.log(2.0), n))
        x[::7] = x_max * (1.0 - 4e-6)                                   # just inside / outside the gate's margin
        x[1::7] = x_max * (1.0 + 1e-7)
        x[2::7] = 0.0                                                    # w = 0
        w = u * (2.0 * np.sqrt(x) / dt * np.linalg.norm(q, axis=1))[:, None]
        st[:, qs], st[:, ws] = q, w
    return st


@pytest.mark.parametrize("dt", [1.0, 4.0])
def test_bodies_around_the_polynomial_range_follow_the_oracle(dt):
    """Solves just inside and just outside X_MAX (polynomial and stagewise attempts, mixed within one env), with
    non-unit quaternions and bodies at rest, follow the C oracle through both kernels."""
    import torch
    from oracle import c_oracle as CO
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv
    x_max, _ = _header()
    n = 700
    rng = np.random.default_rng(41)
    st = _bodies(n, rng, x_max, dt)
    a = rng.uniform(-1, 1, (2, n, 6))
    a[:, :, 3:6] = 0.0                                                   # keep the rates where _bodies put them
    kw = dict(dt=dt, t_max=100 * dt)
    for fused in (False, True):
        env = BatchedRendezvousEnv(n, seed=1, auto_reset=False, **kw)
        env.reset()
        env.set_state(st)
        orc = CO.COracleBatch(CO.make_params(**kw), n)
        orc.set_state(st, recompute_flags=True)
        env.refresh_flags()
        for k in range(2):
            if fused:
                env.rollout(1, actions=torch.as_tensor(a[k:k + 1], device=env.device))
            else:
                env.step(torch.as_tensor(a[k], device=env.device))
            orc.step(a[k], threads=4)
            assert rel_err(env.get_state().cpu().numpy(), orc.state) <= REL_TOL, (fused, k, dt)
        assert env.read_stats()["failures"] == 0


def test_mixed_batch_is_bit_identical_across_launch_shapes():
    """A batch with bodies on both sides of X_MAX gives the same bits from the step API, the lock-step solver (<= 256
    envs per CTA, which sends a pair with an out-of-range body through the sequential form) and the larger CTAs."""
    import torch
    from reinforcement_learning_rendezvous_b200 import BatchedRendezvousEnv, _native as N
    x_max, _ = _header()
    n = 3000
    rng = np.random.default_rng(43)
    st = _bodies(n, rng, x_max, 1.0)
    a = torch.as_tensor(rng.uniform(-1, 1, (3, n, 6)) * [1, 1, 1, 0, 0, 0])
    got = []
    try:
        for tpb in (None, 256, 384, 448, 512):
            env = BatchedRendezvousEnv(n, seed=2, auto_reset=False, t_max=1000)
            env.reset()
            env.set_state(st)
            env.refresh_flags()
            if tpb is None:
                for k in range(3):
                    env.step(a[k].to(env.device))
            else:
                N.lib().rdv_tune(N.TUNE_ROLLOUT_TPB, tpb)
                env.rollout(3, actions=a.to(env.device))
            got.append((env.get_state().clone(), env.read_stats()))
    finally:
        N.lib().rdv_tune(N.TUNE_ROLLOUT_TPB, 0)
    for s, stats in got[1:]:
        assert torch.equal(got[0][0], s)
        assert all(stats[k] == got[0][1][k] for k in ("rk_accepted", "rk_rejected", "failures"))
