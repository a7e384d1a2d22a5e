"""CPU: the trajectory record of the fused rollout -- rdv_rollout_trajectory's declaration and column enum against the
binding, the argument checks it makes before it touches the device (each returns its own code here, where a device call
would give RDV_ERR_CUDA), and the numpy assembly of evaluate_batch(trajectories=True).  No kernels are launched."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from reinforcement_learning_rendezvous_b200 import _native as N
from reinforcement_learning_rendezvous_b200.monte_carlo import trajectory_fields
from reinforcement_learning_rendezvous_b200.params import make_params

RDV_ERR_NULL, RDV_ERR_SIZE, RDV_ERR_ALIGN, RDV_ERR_UNSUPPORTED = -1, -2, -3, -6
HEADER = os.path.join(N.INCLUDE_DIR, "rdv_b200.h")


@pytest.fixture(scope="module")
def lib():
    N.build()
    return N.lib()


def test_declared_exported_and_mirrored(lib):
    text = open(HEADER).read()
    assert re.search(r"int rdv_rollout_trajectory\(const RdvParams \*p, const RdvState \*s, const RdvRolloutIO \*io, "
                     r"double \*traj, int64_t n,\s+uint64_t seed, int64_t env_offset, void \*cuda_stream\);", text)
    assert "rdv_rollout_trajectory" in N.PROTOTYPES and hasattr(lib, "rdv_rollout_trajectory")
    body = re.search(r"enum \{ (RDV_TR_I_STEP = RDV_NF64,[^}]*)\};", text).group(1)
    names = [x.strip().split("=")[0].strip() for x in body.split(",") if x.strip()]
    assert names[-1] == "RDV_TR_NCOL"
    for k, name in enumerate(names):
        assert getattr(N, name[len("RDV_"):]) == N.NF64 + k, name
    assert N.TR_NCOL == 34 and N.TR_NCOL * 8 == 272
    # the ABI the existing binaries were built against is unchanged
    assert lib.rdv_abi_version() == N.ABI_VERSION == 16
    assert C.sizeof(N.RdvRolloutIO) == N.RdvRolloutIO.reserved3.offset + 4


def _call(lib, params=None, traj=0x700000, n=256, table=True, **fields):
    """rdv_rollout_trajectory with fake (never dereferenced) aligned device pointers, by default with a policy table."""
    p = make_params() if params is None else params
    st = N.RdvState(0x100000, 0x200000, n, None, None)
    io = N.RdvRolloutIO()
    io.steps, io.action_source, io.obs = 4, N.ACTIONS_POLICY, 0x300000
    if table:
        io.policy_table, io.policy_tile, io.policy_count = 0x400000, 0x500000, 3
    for k, v in fields.items():
        setattr(io, k, v)
    return lib.rdv_rollout_trajectory(C.byref(p), C.byref(st), C.byref(io), traj, n, 1, 0, None)


def test_rejects_bad_arguments_before_the_device(lib):
    assert _call(lib, traj=None) == RDV_ERR_NULL
    assert _call(lib, traj=0x700004) == RDV_ERR_ALIGN
    assert _call(lib, traj=0x700001) == RDV_ERR_ALIGN
    # rdv_rollout's own checks still apply: a bad policy table returns its codes
    assert _call(lib, action_source=N.ACTIONS_PHILOX) == RDV_ERR_SIZE
    assert _call(lib, policy_tile=None) == RDV_ERR_NULL
    assert _call(lib, policy_count=0) == RDV_ERR_SIZE
    assert _call(lib, policy_table=0x400004) == RDV_ERR_ALIGN
    assert _call(lib, make_params(inertia=np.diag([10.0, 16.0, 22.0]))) == RDV_ERR_UNSUPPORTED
    assert _call(lib, make_params(integrator="closed_form")) == RDV_ERR_UNSUPPORTED
    # ... and so do the others
    assert _call(lib, obs=None) == RDV_ERR_NULL
    assert _call(lib, steps=-1) == RDV_ERR_SIZE
    assert _call(lib, auto_reset=2) == RDV_ERR_SIZE
    assert _call(lib, table=False) == RDV_ERR_NULL                  # no table and NULL policy weights
    assert _call(lib, table=False, action_source=N.ACTIONS_F32) == RDV_ERR_NULL   # no actions tensor
    assert _call(lib, table=False, action_source=N.ACTIONS_PHILOX, rewards=0x800004) == RDV_ERR_ALIGN
    # an empty launch is accepted without a device, but the record is still required
    assert _call(lib, n=0) == 0
    assert _call(lib, steps=0) == 0
    assert _call(lib, traj=None, steps=0) == RDV_ERR_NULL


def _synthetic_record(m=3, steps=6):
    """[steps + 1, TR_NCOL, m]: env j runs lengths[j] steps from step counter 0, then repeats its last row."""
    lengths = np.array([steps, 2, 4])[:m]
    rec = np.zeros((steps + 1, N.TR_NCOL, m))
    for j in range(m):
        for k in range(steps + 1):
            kk = min(k, lengths[j])
            r = np.random.default_rng(100 * j + kk).normal(size=N.TR_NCOL)
            r[N.TR_I_STEP] = kk
            r[N.TR_COLLISION] = float(kk % 2)
            rec[k, :, j] = r
    return rec, lengths


def test_trajectory_fields_from_a_synthetic_record():
    dt = 0.5
    rec, lengths = _synthetic_record()
    steps, m = rec.shape[0] - 1, rec.shape[2]
    tr = trajectory_fields(rec, dt)
    assert set(tr) == {"t", "rc", "vc", "wc", "wt", "qc", "qt", "errors", "dist_from_koz", "collision",
                       "total_delta_v", "total_reward", "length"}
    for k, width in (("rc", 3), ("vc", 3), ("wc", 3), ("wt", 3), ("qc", 4), ("qt", 4), ("errors", 4)):
        assert tr[k].shape == (m, steps + 1, width), k
    for k in ("t", "dist_from_koz", "collision", "total_delta_v", "total_reward"):
        assert tr[k].shape == (m, steps + 1), k
    assert tr["length"].dtype == np.int64 and tr["length"].tolist() == lengths.tolist()
    assert tr["collision"].dtype == bool
    for j in range(m):
        for k in range(steps + 1):
            row = rec[k, :, j]
            assert tr["t"][j, k] == round(min(k, lengths[j]) * dt, 3)
            assert np.array_equal(tr["rc"][j, k], row[N.RCX:N.RCX + 3])
            assert np.array_equal(tr["vc"][j, k], row[N.VCX:N.VCX + 3])
            assert np.array_equal(tr["qc"][j, k], row[N.QCW:N.QCW + 4])
            assert np.array_equal(tr["wc"][j, k], row[N.WCX:N.WCX + 3])
            assert np.array_equal(tr["qt"][j, k], row[N.QTW:N.QTW + 4])
            assert np.array_equal(tr["wt"][j, k], row[N.WTX:N.WTX + 3])
            # errors in the units of get_errors (rad, not the workbook's degrees)
            assert np.array_equal(tr["errors"][j, k], row[N.TR_POS_ERR:N.TR_ROT_ERR + 1])
            assert tr["dist_from_koz"][j, k] == row[N.TR_KOZ]
            assert tr["collision"][j, k] == bool(row[N.TR_COLLISION])
            assert tr["total_delta_v"][j, k] == row[N.TDV]
            assert tr["total_reward"][j, k] == row[N.EPRET]
        # sample 0 is the state at launch, and the tail after the episode's length repeats its last sample
        assert tr["t"][j, 0] == 0.0
        last = lengths[j]
        for key in ("rc", "qc", "errors", "dist_from_koz", "total_reward", "t"):
            assert np.array_equal(tr[key][j, last:], np.repeat(tr[key][j, last:last + 1], steps + 1 - last, axis=0))
