"""CPU: the error bound of tests/lstm_bound.py against the numpy emulation of the LSTM kernels' arithmetic
(tests/lstm_ref.py) at every weight scale the loaders accept -- it holds for the kernel's arithmetic and fails for two
subtly wrong versions of it, so the GPU tests that use it can tell a right kernel from a wrong one."""
import numpy as np
import pytest

from lstm_bound import ratio, step_bound
from lstm_ref import (H, _mm_split, _split16, actor_keys, gates_split_emulation, lstm_step_ref,
                      lstm_step_split_emulation, make_state_dict, scale_state_dict)

SCALES = (1e-3, 1e-2, 0.1, 1.0, 30.0, "max")          # times torch's init; "max": largest |w| just under the limit


def _inputs(n=2000, seed=0):
    """Observations in the Box, h in (-1, 1), c ~ N(0, sigma) with sigma log-uniform in [0.1, 30] per env (trained
    cells carry long memories), 5 % episode starts."""
    rng = np.random.default_rng(seed)
    obs = rng.uniform(-1, 1, (n, 17)).astype(np.float32)
    h = rng.uniform(-1, 1, (n, H)).astype(np.float32)
    c = (rng.standard_normal((n, H)) * np.exp(rng.uniform(np.log(0.1), np.log(30.0), (n, 1)))).astype(np.float32)
    return obs, h, c, rng.random(n) < 0.05


def _actor(scale):
    return actor_keys(scale_state_dict(make_state_dict("torch", seed=0), scale, 1.0))


def _mm_without(product):
    """The kernel's product with one of its three fp16 products left out."""
    def mm(a, w, scale=2.0 ** 10):
        ah, al = _split16(a)
        wh, wl = _split16(np.asarray(w, np.float32) * np.float32(scale))
        terms = {"lo_hi": al @ wh.T, "hi_lo": ah @ wl.T, "hi_hi": ah @ wh.T}
        return (sum(v for k, v in terms.items() if k != product) * np.float32(1.0 / scale)).astype(np.float32)
    return mm


def _mm_unstaged(a, w):
    """The kernel's product with the weights split as they are, not times 2^10."""
    return _mm_split(a, w, scale=1.0)


@pytest.mark.parametrize("scale", SCALES)
def test_bound_holds_for_split_emulation(scale):
    """The emulated kernel step is within the bound on the gates, c' and h'; the bound's own fp64 reference is
    lstm_step_ref's."""
    sd = _actor(scale)
    obs, h, c, start = _inputs()
    b = step_bound(sd, obs, h, c, start)
    act, h_ref, c_ref = lstm_step_ref(sd, obs, h, c, start)
    for mine, ref in ((np.clip(b["out"], -1, 1), act), (b["h"], h_ref), (b["c"], c_ref)):
        assert np.abs(mine - ref).max() <= 1e-12 * max(1.0, float(np.abs(ref).max()))
    with np.errstate(over="ignore"):                      # float32 expf overflow of a saturated gate, as on the device
        h_e, c_e = lstm_step_split_emulation(sd, obs, h, c, start)
    worst = dict(z=ratio(gates_split_emulation(sd, obs, h, start), b["z"], b["dz"]), c=ratio(c_e, b["c"], b["dc"]),
                 h=ratio(h_e, b["h"], b["dh"]))
    print(f"scale {scale}: emulation / bound {worst}")
    assert max(worst.values()) <= 1.0, worst


@pytest.mark.parametrize("product", ["lo_hi", "hi_lo"])
def test_bound_catches_a_dropped_product(product):
    """Leaving out a_lo w_hi or a_hi w_lo breaks the gates' bound at every scale.  Checked on the pre-activations:
    after a fully saturated gate an error need not show in c', h' or the actions."""
    obs, h, c, start = _inputs()
    for scale in SCALES:
        sd = _actor(scale)
        b = step_bound(sd, obs, h, c, start)
        r = ratio(gates_split_emulation(sd, obs, h, start, mm=_mm_without(product)), b["z"], b["dz"])
        print(f"without {product}, scale {scale}: {r:.1f} x the bound")
        assert r > 10.0, (scale, r)


def test_bound_catches_unstaged_weights():
    """Without the 2^10 staging the lo half of a small weight is an fp16 subnormal: the gates break the bound at
    weight scales up to 1e-2 (85 times at 1e-2; 7 times at 0.1; from torch's init on, the staging changes nothing)."""
    obs, h, c, start = _inputs()
    for scale in (1e-3, 1e-2):
        sd = _actor(scale)
        b = step_bound(sd, obs, h, c, start)
        r = ratio(gates_split_emulation(sd, obs, h, start, mm=_mm_unstaged), b["z"], b["dz"])
        print(f"unstaged, scale {scale}: {r:.1f} x the bound")
        assert r > 10.0, (scale, r)

