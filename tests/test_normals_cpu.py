"""CPU: tests/normals.py, the reference of the fused rollout's random streams, against the C oracle -- the raw
Philox block on random counters and keys, and the counter layout the Gaussian head's noise shares with the U(-1,1)
action stream, through the action stream the oracle implements.  All bit for bit."""
import numpy as np
import pytest

from normals import philox4x32_10, philox_actions_ref, philox_block, philox_normals_ref

from oracle import c_oracle as CO


def test_philox_block_against_oracle():
    rng = np.random.default_rng(0)
    ctr = rng.integers(0, 2 ** 32, (300, 4), dtype=np.uint64)
    ctr[:10] = 0
    ctr[10:20] = 2 ** 32 - 1
    keys = rng.integers(0, 2 ** 64, 300, dtype=np.uint64)
    keys[:5] = 0
    keys[5:10] &= np.uint64(0xFFFFFFFF)                          # high word 0
    keys[10:15] |= np.uint64(0xFFFFFFFF00000000)
    got = np.stack(philox4x32_10(ctr[:, 0], ctr[:, 1], ctr[:, 2], ctr[:, 3], keys), axis=-1)
    for i in range(len(keys)):
        k = int(keys[i])
        want = CO.philox_raw([int(x) for x in ctr[i]], k & 0xFFFFFFFF, k >> 32)
        np.testing.assert_array_equal(got[i], want, err_msg=str(i))
    # the Random123 known answer (counter 0, key 0) through the vectorised form
    np.testing.assert_array_equal(got[0], [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8])


SEEDS = (0, 9, 0x123456789ABCDEF0, 2 ** 64 - 1)
STEPS = (0, 17, 2 ** 32 - 1, 2 ** 32, 5 * 2 ** 32 + 7)


@pytest.mark.parametrize("seed", SEEDS)
def test_counter_layout_against_oracle_action_stream(seed):
    """The U(-1,1) actions from the shared layout (tag 0x40000000) equal the oracle's at step indices around and
    past 2^32, and for env ids with a nonzero high word; dropping the step's high word would not."""
    ids = np.concatenate([np.arange(40), [2 ** 31 - 1, 2 ** 31, 3 * 2 ** 31 + 5, 2 ** 40 + 3, 2 ** 62 + 11]])
    for step in STEPS:
        want = CO.philox_actions(seed, ids, step)
        np.testing.assert_array_equal(philox_actions_ref(seed, ids, step), want, err_msg=str(step))
        if step >= 2 ** 32:
            wrong = philox_actions_ref(seed, ids, step & 0xFFFFFFFF)
            assert (wrong != want).all(), step
    # broadcast [steps, envs] == one call per step
    steps = np.array(STEPS, dtype=np.int64)[:, None]
    both = philox_actions_ref(seed, ids, steps)
    for j, step in enumerate(STEPS):
        np.testing.assert_array_equal(both[j], CO.philox_actions(seed, ids, step))


def test_normals_layout_and_transform():
    """The noise uses the same counters under tag 0x20000000 (three blocks), the float32 uniforms of the device and
    the Box-Muller pair (r cos, r sin) of each block."""
    seed, ids, step = 0x0000000500000003, np.array([0, 1, 3 * 2 ** 31 + 5]), 2 ** 32 + 9
    z, r = philox_normals_ref(seed, ids, step)
    assert z.shape == r.shape == (3, 6) and z.dtype == np.float64
    for b in range(3):
        w = philox_block(seed, ids, step, 0x20000000, b)
        hi = (step >> 32) << 4
        for e in range(3):
            c = [ids[e] & 0xFFFFFFFF, ids[e] >> 32, step & 0xFFFFFFFF, 0x20000000 | b | hi]
            np.testing.assert_array_equal([x[e] for x in w], CO.philox_raw(c, seed & 0xFFFFFFFF, seed >> 32))
        u1 = (np.float32(w[0] >> 8) + np.float32(0.5)) * np.float32(2.0 ** -24)
        u2 = (np.float32(w[1] >> 8) + np.float32(0.5)) * np.float32(2.0 ** -24)
        rr = np.sqrt(-2.0 * np.log(np.float64(u1)))
        np.testing.assert_array_equal(r[:, 2 * b], rr)
        np.testing.assert_array_equal(r[:, 2 * b + 1], rr)
        np.testing.assert_array_equal(z[:, 2 * b], rr * np.cos(2 * np.pi * np.float64(u2)))
        np.testing.assert_array_equal(z[:, 2 * b + 1], rr * np.sin(2 * np.pi * np.float64(u2)))


def test_uniforms_are_formed_in_float32():
    """(w >> 8) + 0.5 rounds to even in float32 above 2^23: the largest word gives u = 1 exactly (r = 0), the
    smallest u = 2^-25."""
    from normals import _uniform_f32
    w = np.array([0, 255, 2 ** 31, 2 ** 32 - 256, 2 ** 32 - 1], dtype=np.uint32)
    u = _uniform_f32(w)
    assert u.dtype == np.float32
    np.testing.assert_array_equal(u, np.float32([2.0 ** -25, 2.0 ** -25, 0.5, 1.0, 1.0]))


def test_normal_moments():
    """The reference is a N(0,1) stream: 600,000 draws, mean, variance and the pair's correlation."""
    z, _ = philox_normals_ref(11, np.arange(10000), np.arange(10)[:, None])
    z = z.reshape(-1, 6)
    assert np.abs(z.mean(axis=0)).max() < 0.01
    assert np.abs(z.var(axis=0) - 1.0).max() < 0.02
    assert abs(np.corrcoef(z[:, 0], z[:, 1])[0, 1]) < 0.01
