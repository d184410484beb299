"""CPU checks of the deterministic-reduction entry points and of the training-state pieces that need no device: the workspace sizes,
argument validation before any CUDA call, and the Adam state round trip into the existing flat arenas."""
import ctypes

import pytest

torch = pytest.importorskip("torch")

MARL_EINVAL = -1
FAKE = 256                      # a non-null device address that is never dereferenced: the calls below are rejected first


def _L():
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    return _lib.lib()


def test_message_bwd_workspace_bytes():
    L = _L()
    assert L.marl_dhgn_message_bwd_workspace_bytes(8, 176, 128) == 148 * 8 * 19 * 128 * 4      # grouped path: 8 CTAs per SM
    assert L.marl_dhgn_message_bwd_workspace_bytes(16, 256, 128) == 148 * 8 * 19 * 128 * 4
    assert L.marl_dhgn_message_bwd_workspace_bytes(20, 176, 64) == 148 * 4 * 19 * 64 * 4        # per-row path: 4 CTAs per SM
    assert L.marl_dhgn_message_bwd_workspace_bytes(64, 176, 128) == 148 * 4 * 19 * 128 * 4
    assert L.marl_dhgn_message_bwd_workspace_bytes(8, 300, 128) == 148 * 4 * 19 * 128 * 4       # O > 256: per-row path
    for n, o, e in ((0, 176, 128), (8, 0, 128), (8, 176, 96), (129, 176, 128)):
        assert L.marl_dhgn_message_bwd_workspace_bytes(n, o, e) == -1, (n, o, e)


def test_ppo_head_workspace_bytes():
    L = _L()
    assert L.marl_ppo_head_workspace_bytes(1) == 3 * 4
    assert L.marl_ppo_head_workspace_bytes(4 * 100) == 100 * 3 * 4
    assert L.marl_ppo_head_workspace_bytes(1 << 40) == 148 * 8 * 3 * 4
    assert L.marl_ppo_head_workspace_bytes(0) == -1 and L.marl_ppo_head_workspace_bytes(-5) == -1


def _msg_args(S=64, N=8, O=176, E=128, null=None):
    args = [S, N, O, E] + [FAKE] * 8 + [0] + [FAKE] * 6 + [FAKE] + [FAKE] * 6 + [FAKE]
    if null is not None:
        args[null] = None
    return args


def test_message_bwd_det_rejects_bad_arguments():
    L = _L()
    cases = [(_msg_args(E=96), b"E=96"), (_msg_args(S=0), b"S=0"), (_msg_args(null=4), b"null pointer"),
             (_msg_args(null=19), b"null pointer"), (_msg_args(null=25), b"null pointer"), (_msg_args(null=26), b"null workspace")]
    for args, what in cases:
        assert L.marl_dhgn_message_bwd_det(*args, None) == MARL_EINVAL, args
        assert what in L.marl_last_error_string(), L.marl_last_error_string()


def _head_args(R=64, E=128, A=9, null=None, workspace=FAKE):
    args = [R, E, A] + [FAKE] * 12 + [ctypes.c_float(0.2), ctypes.c_float(0.01)] + [FAKE] * 6 + [workspace]
    if null is not None:
        args[null] = None
    return args


def test_ppo_head_det_rejects_bad_arguments():
    L = _L()
    cases = [(_head_args(R=0), b"R=0"), (_head_args(A=5), b"A=5"), (_head_args(E=48), b"E=48"), (_head_args(null=3), b"null pointer"),
             (_head_args(null=22), b"null pointer"), (_head_args(workspace=None), b"null workspace")]
    for args, what in cases:
        assert L.marl_ppo_head_det(*args, None) == MARL_EINVAL, args
        assert what in L.marl_last_error_string(), L.marl_last_error_string()


def test_flat_adam_state_round_trip_in_place():
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import _FlatAdam
    params = [torch.nn.Parameter(torch.randn(3, 4)), torch.nn.Parameter(torch.randn(5))]
    opt = _FlatAdam(params, lr=1e-3)
    opt.exp_avg.copy_(torch.randn(17))
    opt.exp_avg_sq.copy_(torch.rand(17))
    opt.step_count, opt.param_groups[0]["lr"] = 7, 4.5e-4
    sd = opt.state_dict()
    assert sd["step_count"] == 7 and sd["lr"] == 4.5e-4 and sd["exp_avg"].device.type == "cpu"

    params2 = [torch.nn.Parameter(torch.randn(3, 4)), torch.nn.Parameter(torch.randn(5))]
    opt2 = _FlatAdam(params2, lr=1e-3)
    ptrs = [p.data_ptr() for p in params2] + [opt2.exp_avg.data_ptr(), opt2.exp_avg_sq.data_ptr()]
    opt2.load_state_dict(sd)
    assert torch.equal(opt2.exp_avg, opt.exp_avg) and torch.equal(opt2.exp_avg_sq, opt.exp_avg_sq)
    assert opt2.step_count == 7 and opt2.param_groups[0]["lr"] == 4.5e-4
    assert [p.data_ptr() for p in params2] + [opt2.exp_avg.data_ptr(), opt2.exp_avg_sq.data_ptr()] == ptrs

    small = _FlatAdam([torch.nn.Parameter(torch.randn(4))], lr=1e-3)
    before = small.exp_avg.clone()
    with pytest.raises(_lib.MarlError, match="exp_avg"):
        small.load_state_dict(sd)
    assert torch.equal(small.exp_avg, before) and small.step_count == 0
