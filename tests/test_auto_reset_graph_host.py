"""CPU checks of auto-reset segments replayed from CUDA graphs (MAPPO.explore_batched(carry=..., auto_reset=AutoReset(..., tape="device"))):
every misuse is refused before any CUDA call, the AutoReset's tape kind is validated, the device-seeded entry points are declared and
bound, and seeds reach a device word as the u64 bit pattern a by-value call passes."""
import ctypes
from types import SimpleNamespace

import pytest

torch = pytest.importorskip("torch")

B, N, L, E, D, T_EP = 4, 8, 2, 128, 3, 150


def _fake_mappo():
    """The attributes explore_batched reads before its first CUDA call."""
    return SimpleNamespace(embedding_dim=E, depth=D, num_layers=L, device=torch.device("cpu"), action_dim=9, rnn_hidden_dim=E,
                           cfg=SimpleNamespace(env=SimpleNamespace(max_steps=T_EP)))


def _carry(t0=0, **kw):
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    z = torch.zeros
    return RolloutCarry(t0, z(L, B * N, E), z(L, B * N, E), z(D, B, N, E), z(D, B, N, E), **kw)


def _auto(tape="device"):
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import AutoReset
    return AutoReset(reset_seed=lambda e: 1000 + e, sample_seed=lambda e: e, tape=tape)


def _explore(T=64, carry="default", auto="default", **kw):
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    engine, arena = SimpleNamespace(B=B, N=N), SimpleNamespace(T=T_EP)      # no tensors: a CUDA call would fail here
    carry = _carry() if carry == "default" else carry
    auto = _auto() if auto == "default" else auto
    return MAPPO.explore_batched(_fake_mappo(), engine, arena, T, carry=carry, auto_reset=auto, **kw)


def _refused(match, **kw):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    with pytest.raises(_lib.MarlError, match=match):
        _explore(**kw)


@pytest.mark.parametrize("T", [64, 50, 7])
def test_the_torch_tape_is_a_type_error_before_the_segment_checks(T):
    with pytest.raises(TypeError, match="tape='device'"):
        _explore(T=T, auto=_auto("torch"))
    with pytest.raises(TypeError, match="tape='device'"):
        _explore(T=T, auto=_auto("torch"), carry=None, seed=3)


@pytest.mark.parametrize("auto", [dict(reset_seed=0), 3])
def test_explore_batched_auto_reset_must_be_an_auto_reset(auto):
    with pytest.raises(TypeError):
        _explore(auto=auto)


def test_explore_batched_auto_reset_refuses_a_seed():
    _refused("seed=7 with auto_reset", seed=7)


def test_explore_batched_auto_reset_needs_a_carry():
    _refused("needs a carry", carry=None)


@pytest.mark.parametrize("kw", [dict(host_state={}), dict(host_out={}), dict(host_state={}, host_out={})], ids=["state", "out", "both"])
def test_explore_batched_auto_reset_refuses_host_buffers(kw):
    _refused("host_state / host_out do not combine with auto_reset", **kw)


@pytest.mark.parametrize("S", [0, -1, 151])
def test_explore_batched_auto_reset_segment_length_must_fit_the_episode(S):
    _refused(r"the length must lie in \[1, 150\]", T=S)


@pytest.mark.parametrize("t0", [-1, 150])
def test_explore_batched_auto_reset_segment_must_start_inside_the_episode(t0):
    _refused(r"the start must lie in \[0, 150\)", carry=_carry(t0=t0))


def test_explore_batched_auto_reset_checks_the_carry():
    z = torch.zeros
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    _refused("must be a RolloutCarry", carry=dict(t0=0))
    _refused("rollout carry: emb_a is", carry=RolloutCarry(0, z(L, B * N, E), z(L, B * N, E), z(D + 1, B, N, E), z(D, B, N, E)))


def test_auto_reset_tape_kind():
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import AutoReset
    a = AutoReset(lambda e: e, lambda e: e)
    assert a.tape == "torch" and a.tape_len == 16
    assert AutoReset(lambda e: e, lambda e: e, 8, "device").tape == "device"
    with pytest.raises(ValueError, match="tape='cuda'"):
        AutoReset(lambda e: e, lambda e: e, tape="cuda")


def test_rollout_batched_accepts_the_device_tape_in_its_checks():
    """The host checks of rollout_batched do not depend on the tape kind: a device-tape AutoReset fails where a torch-tape one does."""
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    engine, arena = SimpleNamespace(B=B, N=N), SimpleNamespace(T=T_EP)
    with pytest.raises(_lib.MarlError, match=r"the length must lie in \[1, 150\]"):
        MAPPO.rollout_batched(_fake_mappo(), engine, arena, 151, carry=_carry(), auto_reset=_auto())


@pytest.mark.parametrize("v,bits", [(0, 0), (5, 5), (2 ** 63 - 1, 2 ** 63 - 1), (2 ** 63, -2 ** 63), (2 ** 64 - 1, -1), (-1, -1),
                                    (2 ** 64 + 3, 3)])
def test_u64_bits_is_the_c_uint64_value(v, bits):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    assert _lib.u64_bits(v) == bits
    assert ctypes.c_int64(bits).value == bits
    assert ctypes.c_uint64(bits).value == ctypes.c_uint64(int(v) & (2 ** 64 - 1)).value


def test_device_seeded_entry_points_refuse_a_null_seed_without_a_gpu():
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.config import env_params_dict
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    lib = _lib.lib()
    p = ctypes.byref(_lib.EnvParams.from_dict(env_params_dict(default_config())))
    d = ctypes.c_double
    assert lib.marl_map_generate_dseed(p, 4, 10, d(1.0), d(1.0), d(1.0), None, 256, 256, None) == -1
    assert b"d_seed is NULL" in lib.marl_last_error_string()
    assert lib.marl_env_reset_place_dseed(p, 4, 4, 256, None, None, d(4.0), 2, 10, 256, 256, 256, 256, None, None) == -1
    assert b"d_seed is NULL" in lib.marl_last_error_string()
    assert lib.marl_target_tape_generate(p, 4, 0, 256, 256, None) == -1
    assert lib.marl_target_tape_generate(p, 4, 16, None, 256, None) == -1
    from distributed_multi_agent_reinforcement_learning_b200 import fused_policy
    s = fused_policy.PolicyStep()
    s.B, s.N, s.O, s.E, s.depth, s.action_dim = 4, 8, 16, 128, 1, 9
    w, io = fused_policy.DhgnWeights(), fused_policy.PolicyNetIO()
    r = ctypes.byref
    assert lib.marl_policy_rollout_step_dseed(r(s), r(w), r(io), r(w), r(io), None, None) == -1
    assert b"d_seed is NULL" in lib.marl_last_error_string()
