"""CPU: the policy-table fields of RdvRolloutIO -- layout of the ctypes mirror, the argument checks rdv_rollout makes
before it touches the device (so each returns its own code here, where a device call would give RDV_ERR_CUDA), the
packed RdvPolicy array of PolicyTable, and the host-side validation of the tile map and of the evaluators' policy
lists.  No kernels are launched here."""
import ctypes as C

import numpy as np
import pytest
import torch

from reinforcement_learning_rendezvous_b200 import _native as N
from reinforcement_learning_rendezvous_b200.batched_env import policy_tile_indices
from reinforcement_learning_rendezvous_b200.params import make_params


@pytest.fixture(scope="module")
def lib():
    N.build()
    return N.lib()


def test_rollout_io_mirror(lib):
    assert lib.rdv_abi_version() == N.ABI_VERSION == 16
    assert lib.rdv_sizeof(3) == C.sizeof(N.RdvRolloutIO)
    # the new fields are appended: everything before them keeps its offset
    assert N.RdvRolloutIO.policy_table.offset == N.RdvRolloutIO.mc_out.offset + 8
    assert N.RdvRolloutIO.policy_tile.offset == N.RdvRolloutIO.policy_table.offset + 8
    assert N.RdvRolloutIO.policy_count.offset == N.RdvRolloutIO.policy_tile.offset + 8
    assert C.sizeof(N.RdvRolloutIO) == N.RdvRolloutIO.reserved3.offset + 4
    assert N.POLICY_TILE == 128


def _call(lib, params=None, n=256, **fields):
    """rdv_rollout with fake (never dereferenced) aligned device pointers and a policy table."""
    p = make_params() if params is None else params
    st = N.RdvState(0x100000, 0x200000, n, None, None)
    io = N.RdvRolloutIO()
    io.steps, io.action_source, io.obs = 4, N.ACTIONS_POLICY, 0x300000
    io.policy_table, io.policy_tile, io.policy_count = 0x400000, 0x500000, 3
    for k, v in fields.items():
        setattr(io, k, v)
    return lib.rdv_rollout(C.byref(p), C.byref(st), C.byref(io), n, 1, 0, None)


def test_rollout_rejects_bad_policy_tables_before_the_device(lib):
    RDV_ERR_NULL, RDV_ERR_SIZE, RDV_ERR_ALIGN, RDV_ERR_UNSUPPORTED = -1, -2, -3, -6
    # a table needs an action source that evaluates the actor
    for src in (N.ACTIONS_F32, N.ACTIONS_F64, N.ACTIONS_PHILOX):
        assert _call(lib, action_source=src, actions=0x600000) == RDV_ERR_SIZE, src
    assert _call(lib, policy_tile=None) == RDV_ERR_NULL
    assert _call(lib, policy_count=0) == RDV_ERR_SIZE
    assert _call(lib, policy_count=-1) == RDV_ERR_SIZE
    assert _call(lib, policy_table=0x400004) == RDV_ERR_ALIGN
    assert _call(lib, policy_tile=0x500002) == RDV_ERR_ALIGN
    assert _call(lib, make_params(inertia=np.diag([10.0, 16.0, 22.0]))) == RDV_ERR_UNSUPPORTED
    assert _call(lib, make_params(integrator="closed_form")) == RDV_ERR_UNSUPPORTED
    assert _call(lib, action_source=N.ACTIONS_POLICY_SAMPLE, policy_count=0) == RDV_ERR_SIZE
    # with a table the call's own policy weights may be NULL: an empty launch is accepted without a device
    assert _call(lib, n=0) == 0
    assert _call(lib, steps=0) == 0
    assert _call(lib, action_source=N.ACTIONS_POLICY_SAMPLE, steps=0) == 0
    # without a table the NULL weights are still an error
    assert _call(lib, policy_table=None, policy_tile=None, policy_count=0) == RDV_ERR_NULL


def test_policy_table_packs_a_c_array():
    from reinforcement_learning_rendezvous_b200.policy import PolicyTable
    structs = [N.RdvPolicy(*(0x1000 * (8 * e + j + 1) for j in range(6)), 64, 0, 0x9000 + 0x100 * e if e else None)
               for e in range(3)]
    raw = PolicyTable.pack(structs)
    size = C.sizeof(N.RdvPolicy)
    assert size == 64 and len(raw) == 3 * size
    assert raw == bytes((N.RdvPolicy * 3)(*structs))
    for e, s in enumerate(structs):
        back = N.RdvPolicy.from_buffer_copy(raw, e * size)
        assert (back.w0, back.b0, back.w1, back.b1, back.w2, back.b2) == (s.w0, s.b0, s.w1, s.b1, s.w2, s.b2)
        assert back.hidden == 64 and back.log_std == s.log_std


def test_policy_table_rejects_bad_entries():
    from reinforcement_learning_rendezvous_b200.policy import PolicyTable
    with pytest.raises(ValueError):
        PolicyTable([])
    with pytest.raises(TypeError):
        PolicyTable([object()])


def test_policy_tile_indices():
    t = policy_tile_indices([2, 0, 2, 1, 1, 0, 2, 1], 128 * 7 + 37, 3)
    assert t.dtype == np.int32 and t.tolist() == [2, 0, 2, 1, 1, 0, 2, 1]
    assert policy_tile_indices(torch.tensor([0, 1], dtype=torch.int64), 256, 2).tolist() == [0, 1]
    assert policy_tile_indices(np.zeros(1, dtype=np.uint8), 1, 1).tolist() == [0]
    with pytest.raises(ValueError):
        policy_tile_indices(None, 256, 2)
    with pytest.raises(ValueError):
        policy_tile_indices([0, 1], 257, 2)                  # 3 tiles
    with pytest.raises(ValueError):
        policy_tile_indices([0, 1, 0], 256, 2)               # 2 tiles
    with pytest.raises(ValueError):
        policy_tile_indices([0, 2], 256, 2)                  # index == count
    with pytest.raises(ValueError):
        policy_tile_indices([-1, 0], 256, 2)
    with pytest.raises(ValueError):
        policy_tile_indices([0.0, 1.0], 256, 2)              # not integers


def test_evaluator_policy_lists_are_checked_before_the_device():
    from reinforcement_learning_rendezvous_b200.monte_carlo import evaluate_sweep
    sets = [dict(), dict(h=400e3), dict(dt=0.5)]
    with pytest.raises(ValueError):
        evaluate_sweep([None, None], sets, episodes_per_set=256)              # one policy per set
    with pytest.raises(ValueError):
        evaluate_sweep([None, None, None], sets, episodes_per_set=192)        # not a multiple of 128
