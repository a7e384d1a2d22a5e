"""CPU: the bounds behind the three controller shortcuts of csrc/rdv_math.cuh (plane_initial_step, plane_step),
checked against SciPy's own ``select_initial_step`` / ``rk_step`` on the reference's right-hand side -- no GPU
involved.  What the kernel skips when a bound holds must be what SciPy would have computed anyway:

* ``select_initial_step`` returns min(100 h0, h1, dt); with the kernel's conditions satisfied it equals
  min((0.01 / d1)^(1/5), dt) with d1 from the quaternion components alone (d2 <= d1, and 100 h0 is not the minimum);
* an attempted step whose upper bound  2 sum(e_i^2) / (7 atol^2)  is below 0.99 has SciPy's error norm below 1.

The conditions are restated here in float64 exactly as the kernel forms them in float32 (its 5 % / 1e-4 / 0.975 margins
are what covers the difference)."""
import numpy as np
import pytest
from scipy.integrate._ivp.common import norm, select_initial_step
from scipy.integrate._ivp.rk import RK45, rk_step

from oracle.rdv_oracle import RK_ATOL, RK_RTOL, attitude_rhs

INERTIA = np.diag([100.0 / 6.0] * 3)
INV_INERTIA = np.linalg.inv(INERTIA)


def _fun(t, y):
    return attitude_rhs(t, y, INERTIA, INV_INERTIA, np.zeros(3))


def _bodies(rng, n, rate):
    q = rng.normal(size=(n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    q *= rng.uniform(0.3, 1.7, (n, 1)) ** rng.integers(0, 2, (n, 1))          # half of them injected non-unit
    w = rng.uniform(-1, 1, (n, 3)) * rate
    return np.hstack([q, w])


def _plane(y0):
    q0, w = y0[:4], y0[4:]
    f0 = _fun(0.0, y0)
    p = f0[:4]                                                                 # 0.5 Omega(w) q0 / |q0|
    om2 = 0.25 * np.dot(w, w) / np.dot(q0, q0)
    return q0, p, om2, f0


def _kernel_initial_step_shortcut(y0, dt):
    """The common-case branch of plane_initial_step: its value, or None when the kernel takes the general path."""
    q0, p, om2, _ = _plane(y0)
    inv_sc = 1.0 / (RK_ATOL + RK_RTOL * np.abs(q0))
    d0q = np.sum((q0 * inv_sc) ** 2) / 7.0
    d1s = np.sum((p * inv_sc) ** 2) / 7.0
    room = 0.975 - 0.5 * dt * om2
    if not (d0q >= 1e-10 and d1s >= 1e-10 and room > 0.0 and om2 * om2 * d0q <= d1s * room * room):
        return None
    h1 = (min(d1s, 1e30) * 1e4) ** -0.1
    lim = min(h1, dt)
    if not d0q >= lim * lim * d1s * 1.0001:
        return None
    return min(h1, dt)


@pytest.mark.parametrize("dt", [0.25, 1.0, 4.0])
def test_initial_step_shortcut_equals_scipy(dt):
    rng = np.random.default_rng(5)
    taken = {}
    for rate in (0.0, 0.003, 0.05, 0.17, 1.0, 3.0, 12.0):
        hits = 0
        for y0 in _bodies(rng, 150, rate):
            mine = _kernel_initial_step_shortcut(y0, dt)
            if mine is None:
                continue
            hits += 1
            ref = select_initial_step(_fun, 0.0, y0, dt, np.inf, _fun(0.0, y0), 1.0, 4, RK_RTOL, RK_ATOL)
            assert abs(mine - ref) <= 1e-12 * ref, (rate, mine, ref)
        taken[rate] = hits
    # every body in the reference's ranges (rates up to the 10 deg/s observation bound) takes the shortcut ...
    assert taken[0.003] == 150 and taken[0.05] == 150 and taken[0.17] == 150, taken
    # ... a body at rest (f0 = 0) never does, and neither does one that spins fast enough to break a bound
    assert taken[0.0] == 0 and taken[12.0] < 150, taken


def test_last_attempt_bound_implies_scipy_accepts():
    rng = np.random.default_rng(6)
    accepted_by_bound = total = 0
    for rate in (0.003, 0.05, 0.17, 1.0, 3.0):
        for y0 in _bodies(rng, 60, rate):
            q0, p, om2, f0 = _plane(y0)
            for h in (1e-3, 0.03, 0.1, 0.3, 0.9, 2.0):
                y_new, f_new = rk_step(_fun, 0.0, y0, f0, h, RK45.A, RK45.B, RK45.C, K := np.empty((7, 7)))
                e = np.dot(K.T, RK45.E) * h
                assert np.all(np.abs(e[4:]) < 1e-15)           # the rates carry no error (w' = w x I w / I: rounding noise)
                # the kernel's bound, from the plane coordinates of the error estimate (q0 is orthogonal to p)
                ea = np.dot(e[:4], q0) / np.dot(q0, q0)
                eb = np.dot(e[:4], p) / np.dot(p, p) if np.dot(p, p) > 0 else 0.0
                ub = (ea * ea * np.dot(q0, q0) + eb * eb * np.dot(p, p)) * (2.0 / 7.0 * 1.0e12)
                scale = RK_ATOL + np.maximum(np.abs(y0), np.abs(y_new)) * RK_RTOL
                err2 = norm(e / scale) ** 2
                total += 1
                if ub < 0.99:
                    accepted_by_bound += 1
                    assert err2 < 1.0, (rate, h, ub, err2)
                    assert err2 <= ub + 1e-16          # an upper bound (SciPy's 7-component rounding noise lies off the plane)
    # the bound decides a good share of these attempts (the clipped last step of a solve is a short one)
    assert accepted_by_bound > 0.3 * total, (accepted_by_bound, total)
