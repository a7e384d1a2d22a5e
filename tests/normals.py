"""CPU reference of the fused rollout's device random streams, vectorised over arrays of counters.

Both streams key Philox4x32-10 with the 64-bit action seed and use one counter layout (rdv_policy.cuh,
rdv_step.cuh): (env id lo, env id hi, step index lo, tag | block | (step index hi & 0xFFFFFF) << 4).

* ``philox_normals_ref``: the Gaussian head's noise (tag 0x20000000, blocks 0..2, one Box-Muller pair per block).
  The uniforms are formed exactly as the device forms them in float32, u = ((w >> 8) + 0.5) 2^-24; the rest is fp64,
  so the device's float32 logf / sqrtf / sincospif are compared against the exact transform of the same uniforms.
* ``philox_actions_ref``: the U(-1,1) fp64 actions (tag 0x40000000, blocks 0..1), a = (w + 0.5) 2^-31 - 1.
"""
import numpy as np

_M = np.uint64(0xFFFFFFFF)
NORMAL_TAG, ACTION_TAG = 0x20000000, 0x40000000


def _u64(x):
    """Integers below 2^64 -> uint64 array (signed ones in two's complement, as the device's uint64 casts)."""
    a = np.asarray(x)
    return a.astype(np.uint64) if a.dtype.kind == "u" else a.astype(np.int64).astype(np.uint64)


def philox4x32_10(c0, c1, c2, c3, seed):
    """Philox4x32-10 (Salmon et al., SC'11) over broadcast arrays of 32-bit counter words; ``seed`` is the 64-bit
    key (lo word k0, hi word k1).  Returns the four output words as uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint64) & _M for x in np.broadcast_arrays(c0, c1, c2, c3)]
    key = _u64(seed)
    k0, k1 = key & _M, key >> np.uint64(32)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _M, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _M]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & _M, (k1 + np.uint64(0xBB67AE85)) & _M
    return [x.astype(np.uint32) for x in c]


def philox_block(seed, env_ids, step_index, tag, blk):
    """The block ``tag | blk`` of (seed; env id, step index) for broadcast arrays of env ids and step indices."""
    ids, step = np.broadcast_arrays(_u64(env_ids), _u64(step_index))
    hi = (step >> np.uint64(32)) & np.uint64(0x00FFFFFF)
    return philox4x32_10(ids & _M, ids >> np.uint64(32), step & _M, np.uint64(tag | blk) | (hi << np.uint64(4)), seed)


def _uniform_f32(w):
    """((w >> 8) + 0.5) 2^-24 in float32 arithmetic, as the device forms it: in (0, 1]."""
    return ((w >> np.uint32(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)


def philox_normals_ref(seed, env_ids, step_index):
    """The six N(0,1) draws of (seed; env id, step index) over broadcast ``env_ids`` / ``step_index``.
    Returns (z, r), both float64 [..., 6]: z[2b] = r cos(2 pi u2), z[2b+1] = r sin(2 pi u2) of block b, and r =
    sqrt(-2 ln u1) of the component's pair (the scale of the device's rounding errors)."""
    zs, rs = [], []
    for blk in range(3):
        w = philox_block(seed, env_ids, step_index, NORMAL_TAG, blk)
        u1, u2 = _uniform_f32(w[0]).astype(np.float64), _uniform_f32(w[1]).astype(np.float64)
        r = np.sqrt(-2.0 * np.log(u1))
        zs += [r * np.cos(2.0 * np.pi * u2), r * np.sin(2.0 * np.pi * u2)]
        rs += [r, r]
    return np.stack(zs, axis=-1), np.stack(rs, axis=-1)


def philox_actions_ref(seed, env_ids, step_index):
    """The U(-1,1) fp64 actions of (seed; env id, step index), [..., 6]: words 0..3 of block 0 and 0..1 of block 1
    (exact in fp64)."""
    w0 = philox_block(seed, env_ids, step_index, ACTION_TAG, 0)
    w1 = philox_block(seed, env_ids, step_index, ACTION_TAG, 1)
    w = np.stack(w0 + w1[:2], axis=-1).astype(np.float64)
    return w * 4.656612873077392578125e-10 + (-1.0 + 2.3283064365386962890625e-10)
