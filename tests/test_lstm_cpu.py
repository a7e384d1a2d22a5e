"""CPU: the fp64 reference of the recurrent actor against torch.nn.LSTM, the RecurrentPPO checkpoint loader, and the
C ABI of rdv_lstm_policy_step (struct layout, argument errors) -- no kernel is launched."""
import ctypes as C
import io
import zipfile

import numpy as np
import pytest
import torch

from lstm_ref import H, lstm_step_ref, make_state_dict

from reinforcement_learning_rendezvous_b200 import _native as N
from reinforcement_learning_rendezvous_b200.policy import LstmPolicy, load_state_dict


def test_reference_equals_torch_lstm_fp64():
    """60 steps driven like sb3_contrib's _process_sequence: one step per call, the state times (1 - episode_start)."""
    sd = make_state_dict("stress", seed=1)
    n, rng = 40, np.random.default_rng(2)
    lstm = torch.nn.LSTM(17, H).double()
    with torch.no_grad():
        for k in ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"):
            getattr(lstm, k).copy_(torch.as_tensor(sd["lstm_actor." + k], dtype=torch.float64))
    w = {k: torch.as_tensor(v, dtype=torch.float64) for k, v in sd.items()}
    h_t = c_t = torch.zeros((1, n, H), dtype=torch.float64)
    h = c = np.zeros((n, H))
    worst = 0.0
    for t in range(60):
        obs = rng.uniform(-1, 1, (n, 17))
        start = np.ones(n, dtype=bool) if t == 0 else rng.random(n) < 0.1
        es = torch.as_tensor(start, dtype=torch.float64)[None, :, None]
        with torch.no_grad():
            out, (h_t, c_t) = lstm(torch.as_tensor(obs)[None], ((1.0 - es) * h_t, (1.0 - es) * c_t))
            a = torch.tanh(out[0] @ w["mlp_extractor.policy_net.0.weight"].T + w["mlp_extractor.policy_net.0.bias"])
            a = torch.tanh(a @ w["mlp_extractor.policy_net.2.weight"].T + w["mlp_extractor.policy_net.2.bias"])
            act_t = torch.clamp(a @ w["action_net.weight"].T + w["action_net.bias"], -1, 1)
        act, h, c = lstm_step_ref(sd, obs, h, c, start)
        for mine, theirs in ((act, act_t), (h, h_t[0]), (c, c_t[0])):
            worst = max(worst, float(np.abs(mine - theirs.numpy()).max()))
    assert float(np.abs(c).max()) > 3.0                  # the stressed cell has a long memory
    assert worst <= 1e-13, worst


def _zip_of(sd, path):
    buf = io.BytesIO()
    torch.save({k: torch.as_tensor(v) for k, v in sd.items()}, buf)
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("policy.pth", buf.getvalue())
        z.writestr("data", "{}")
    return str(path)


def _construct(sd):
    """LstmPolicy(sd): a valid actor passes the shape checks and then needs a GPU (no CPU fallback)."""
    if torch.cuda.is_available():
        return LstmPolicy(sd)
    with pytest.raises(RuntimeError, match="CUDA"):
        LstmPolicy(sd)


def test_loader_reads_recurrent_ppo_zip(tmp_path):
    full = make_state_dict("torch", seed=3, critic=True)
    sd = load_state_dict(_zip_of(full, tmp_path / "rnn_model.zip"))
    assert set(sd) == set(full) and "log_std" in sd and "lstm_critic.weight_hh_l0" in sd
    for k in full:
        assert np.array_equal(sd[k], full[k]), k
    pol = _construct(sd)                                  # critic keys and log_std are ignored
    if pol is not None:
        assert np.array_equal(pol.w["weight_hh"].cpu().numpy(), full["lstm_actor.weight_hh_l0"])


def test_loader_rejects_other_shapes():
    sd = make_state_dict("torch", seed=4)
    two = dict(sd)
    two["lstm_actor.weight_ih_l1"] = np.zeros((4 * H, H), np.float32)
    two["lstm_actor.weight_hh_l1"] = np.zeros((4 * H, H), np.float32)
    with pytest.raises(ValueError, match="single-layer"):
        LstmPolicy(two)
    small = dict(sd)
    small["lstm_actor.weight_hh_l0"] = np.zeros((4 * 64, 64), np.float32)
    with pytest.raises(ValueError):
        LstmPolicy(small)
    wide_head = dict(sd)
    wide_head["mlp_extractor.policy_net.0.weight"] = np.zeros((128, H), np.float32)
    with pytest.raises(ValueError):
        LstmPolicy(wide_head)
    missing = {k: v for k, v in sd.items() if k != "lstm_actor.bias_hh_l0"}
    with pytest.raises(ValueError, match="missing"):
        LstmPolicy(missing)


@pytest.fixture(scope="module")
def lib():
    N.build()
    return N.lib()


def test_struct_mirror_and_argument_errors(lib):
    assert lib.rdv_sizeof(6) == C.sizeof(N.RdvLstmPolicy) == 10 * 8 + 8
    f = lib.rdv_lstm_policy_step
    buf = (C.c_double * 8192)()
    b = C.addressof(buf)
    pi = N.RdvLstmPolicy(*([b] * 10), 256, 0)
    ok = (b, None, b, b, b + 16384, b + 16384, b + 32768)                      # obs, start, h_in, c_in, h_out, ...
    assert f(None, *ok, 4, 4, None) == -1
    assert f(C.byref(pi), None, *ok[1:], 4, 4, None) == -1
    assert f(C.byref(pi), *ok[:2], None, *ok[3:], 4, 4, None) == -1
    assert f(C.byref(N.RdvLstmPolicy(*([b] * 9), None, 256, 0)), *ok, 4, 4, None) == -1
    assert f(C.byref(pi), *ok, 4, 3, None) == -2                               # ld < n
    assert f(C.byref(pi), *ok, -1, 4, None) == -2
    assert f(C.byref(pi), b + 2, *ok[1:], 4, 4, None) == -3                    # misaligned observations
    assert f(C.byref(pi), *ok[:6], b + 1, 4, 4, None) == -3                    # misaligned actions
    assert f(C.byref(N.RdvLstmPolicy(b + 2, *([b] * 9), 256, 0)), *ok, 4, 4, None) == -3
    assert f(C.byref(N.RdvLstmPolicy(*([b] * 10), 64, 0)), *ok, 4, 4, None) == -6
    assert f(C.byref(pi), *ok, 0, 0, None) == 0                                # n = 0: no-op
    if not torch.cuda.is_available():
        assert f(C.byref(pi), *ok, 4, 4, None) == -5                           # no GPU: RDV_ERR_CUDA
