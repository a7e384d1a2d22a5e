"""CPU: the polynomial form of one attempted plane step (csrc/rdv_plane_poly.h) against its generator and mpmath."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

mp = pytest.importorskip("mpmath")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "reinforcement_learning_rendezvous_b200", "csrc", "rdv_plane_poly.h")


def _header():
    defs = dict(re.findall(r"^#define RDV_PP_(\w+) (.*)$", open(HEADER).read(), flags=re.M))
    coef = {k: [float.fromhex(v.strip()) for v in defs[k].split(",")] for k in ("P1", "Q1", "R", "I")}
    return float.fromhex(defs["X_MAX"]), coef


def _horner(c, x):
    r = np.full_like(x, c[-1])
    for v in reversed(c[:-1]):
        r = r * x + v
    return r


def test_generator_reproduces_the_header():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gen_plane_poly.py"), "--check"],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr


def test_header_polynomials_match_mpmath():
    """Evaluated in fp64 (Horner, no FMA), 1 + x P1 and 1 + x Q1 are within 2 ulp of Re S and Im S / s, and R, I within
    1e-13 of their largest magnitude, on a dense grid of [0, X_MAX] -- S and E from the Dormand-Prince tableau itself."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import gen_plane_poly as G
    finally:
        sys.path.pop(0)
    x_max, c = _header()
    assert x_max == float(G.X_MAX)
    x = np.linspace(0.0, x_max, 1501)[1:]
    truth = np.array([[float(v) for v in (1 + xi * p, 1 + xi * q, r, i)]
                      for xi, (p, q, r, i) in ((xi, G.parts(mp.mpf(xi))) for xi in x)])
    P = 1.0 + x * _horner(c["P1"], x)
    Q = 1.0 + x * _horner(c["Q1"], x)
    for got, want in ((P, truth[:, 0]), (Q, truth[:, 1])):
        assert (np.abs(got - want) / np.spacing(np.abs(want))).max() <= 2.0
    for got, want in ((_horner(c["R"], x), truth[:, 2]), (_horner(c["I"], x), truth[:, 3])):
        assert np.abs(got - want).max() <= 1e-13 * np.abs(want).max()
