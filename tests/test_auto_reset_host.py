"""CPU checks of auto-reset rollout segments (MAPPO.rollout_batched(carry=..., auto_reset=AutoReset(...))): every misuse is refused
before any CUDA call, any segment length up to the episode's passes the host checks from any step, and without auto_reset the
divisor rule and its messages stay as they are."""
from types import SimpleNamespace

import pytest

torch = pytest.importorskip("torch")

B, N, L, E, D, T_EP = 4, 8, 2, 128, 3, 150


def _fake_mappo(E=E):
    """The attributes rollout_batched reads before its first CUDA call."""
    return SimpleNamespace(embedding_dim=E, depth=D, num_layers=L, device=torch.device("cpu"), action_dim=9, rnn_hidden_dim=E,
                           cfg=SimpleNamespace(env=SimpleNamespace(max_steps=T_EP)))


def _carry(t0=0, **kw):
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    z = torch.zeros
    return RolloutCarry(t0, z(L, B * N, E), z(L, B * N, E), z(D, B, N, E), z(D, B, N, E), **kw)


def _auto():
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import AutoReset
    return AutoReset(reset_seed=lambda e: 1000 + e, sample_seed=lambda e: e)


def _refused(match, T=64, carry="default", auto="default", mappo=None, **kw):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    engine, arena = SimpleNamespace(B=B, N=N), SimpleNamespace(T=T_EP)
    carry = _carry() if carry == "default" else carry
    auto = _auto() if auto == "default" else auto
    with pytest.raises(_lib.MarlError, match=match):
        MAPPO.rollout_batched(mappo or _fake_mappo(), engine, arena, T, carry=carry, auto_reset=auto, **kw)


def test_auto_reset_needs_a_carry():
    _refused("needs a carry", carry=None)


@pytest.mark.parametrize("S", [0, -1, 151, 300])
def test_auto_reset_segment_length_must_fit_the_episode(S):
    _refused(r"the length must lie in \[1, 150\]", T=S)


@pytest.mark.parametrize("t0", [-1, 150, 151])
def test_auto_reset_segment_must_start_inside_the_episode(t0):
    _refused(r"the start must lie in \[0, 150\)", carry=_carry(t0=t0))


def test_auto_reset_refuses_actor_only():
    _refused("actor_only .* takes no auto_reset", actor_only=True)


def test_auto_reset_refuses_the_unfused_path():
    _refused("auto_reset needs the fused policy step", use_fused=False)
    _refused("auto_reset needs the fused policy step", mappo=_fake_mappo(E=64))        # a shape the fused step does not cover


def test_auto_reset_refuses_an_explicit_seed():
    _refused("seed=7 with auto_reset", seed=7)


@pytest.mark.parametrize("auto", [dict(reset_seed=0), 3, "x"])
def test_auto_reset_must_be_an_auto_reset(auto):
    _refused("auto_reset must be an AutoReset", auto=auto)


def test_auto_reset_carry_must_be_a_rollout_carry_of_the_right_shape():
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    _refused("must be a RolloutCarry", carry=dict(t0=0))
    z = torch.zeros
    _refused("rollout carry: ha is", carry=RolloutCarry(0, z(L, B * N + 1, E), z(L, B * N, E), z(D, B, N, E), z(D, B, N, E)))


@pytest.mark.parametrize("t0", [0, 120, 149])
@pytest.mark.parametrize("S", [1, 7, 40, 64, 149, 150])
def test_any_segment_passes_the_host_checks_with_auto_reset(S, t0):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import check_auto_reset, check_segment
    check_auto_reset(_auto(), _carry(t0=t0), S, T_EP, B, N, L, E, D, "cpu")
    if T_EP % S != 0:                   # without auto_reset: the existing divisor rule and message
        with pytest.raises(_lib.MarlError, match="positive divisor of the episode length 150"):
            check_segment(_carry(t0=t0), S, T_EP, B, N, L, E, D, "cpu")
    elif t0 + S > T_EP:
        with pytest.raises(_lib.MarlError, match="does not lie inside the episode"):
            check_segment(_carry(t0=t0), S, T_EP, B, N, L, E, D, "cpu")
    else:
        check_segment(_carry(t0=t0), S, T_EP, B, N, L, E, D, "cpu")


@pytest.mark.parametrize("t0,S,match", [(0, 7, "positive divisor"), (0, 40, "positive divisor"), (0, 64, "positive divisor"),
                                        (120, 50, "does not lie inside the episode")])
def test_without_auto_reset_crossing_segments_are_still_refused(t0, S, match):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    engine, arena = SimpleNamespace(B=B, N=N), SimpleNamespace(T=T_EP)
    with pytest.raises(_lib.MarlError, match=match):
        MAPPO.rollout_batched(_fake_mappo(), engine, arena, S, carry=_carry(t0=t0))


def test_rollout_carry_positional_construction_and_episode_default():
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    c = _carry(t0=5)
    assert c.t0 == 5 and c.episode == 0
    assert _carry(t0=5, episode=3).episode == 3
    z = RolloutCarry.zeros(_fake_mappo(), B, N, 0)
    assert z.t0 == 0 and z.episode == 0 and tuple(z.ha.shape) == (L, B * N, E)
    assert RolloutCarry.zeros(_fake_mappo(), B, N, t0=2, episode=4).episode == 4
    c.copy_(_carry(t0=9, episode=2))
    assert c.t0 == 9 and c.episode == 2


def test_explore_batched_takes_no_auto_reset():
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    with pytest.raises(TypeError):
        MAPPO.explore_batched(_fake_mappo(), SimpleNamespace(B=B, N=N), SimpleNamespace(T=T_EP), 64, carry=_carry(), auto_reset=_auto())
