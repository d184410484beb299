"""CPU checks of rollout segments (MAPPO.rollout_batched / explore_batched with a RolloutCarry): a bad segment length, a carry of the
wrong shape, step or device, and the evaluator's actor-only rollout with a carry are all refused before any CUDA call."""
from types import SimpleNamespace

import pytest

torch = pytest.importorskip("torch")

B, N, L, E, D, T_EP = 4, 8, 2, 128, 3, 150


def _fake_mappo():
    """The attributes rollout_batched / explore_batched read before their first CUDA call."""
    return SimpleNamespace(embedding_dim=E, depth=D, num_layers=L, device=torch.device("cpu"),
                           cfg=SimpleNamespace(env=SimpleNamespace(max_steps=T_EP)))


def _carry(t0=0, b=B, n=N, l=L, e=E, d=D, dtype=torch.float32):
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    z = lambda *s: torch.zeros(*s, dtype=dtype)      # noqa: E731
    return RolloutCarry(t0, z(l, b * n, e), z(l, b * n, e), z(d, b, n, e), z(d, b, n, e))


def _refused(match, T=50, carry=None, actor_only=False, explore=False):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    engine, arena = SimpleNamespace(B=B, N=N), SimpleNamespace(T=T_EP)
    carry = _carry() if carry is None else carry
    with pytest.raises(_lib.MarlError, match=match):
        if explore:
            MAPPO.explore_batched(_fake_mappo(), engine, arena, T, carry=carry)
        else:
            MAPPO.rollout_batched(_fake_mappo(), engine, arena, T, carry=carry, actor_only=actor_only)


@pytest.mark.parametrize("explore", [False, True], ids=["rollout", "graph"])
@pytest.mark.parametrize("S", [0, -50, 7, 40, 151, 300])
def test_segment_length_must_divide_the_episode(S, explore):
    _refused("positive divisor of the episode length 150", T=S, explore=explore)


@pytest.mark.parametrize("explore", [False, True], ids=["rollout", "graph"])
@pytest.mark.parametrize("t0,S", [(-50, 50), (150, 50), (120, 50), (1, 150)])
def test_segment_must_lie_inside_the_episode(t0, S, explore):
    _refused("does not lie inside the episode", T=S, carry=_carry(t0=t0), explore=explore)


@pytest.mark.parametrize("explore", [False, True], ids=["rollout", "graph"])
@pytest.mark.parametrize("what,kw", [("ha", dict(b=B + 1)), ("ha", dict(n=N - 1)), ("ha", dict(l=1)), ("ha", dict(e=64)),
                                     ("emb_a", dict(d=D - 1)), ("ha", dict(dtype=torch.float64))])
def test_carry_shape_must_match(what, kw, explore):
    _refused(f"rollout carry: {what} is", carry=_carry(**kw), explore=explore)


def test_carry_on_another_device_is_refused():
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import check_segment
    with pytest.raises(_lib.MarlError, match="on cpu, this rollout needs .* on cuda"):
        check_segment(_carry(), 50, T_EP, B, N, L, E, D, "cuda")


def test_carry_must_be_a_rollout_carry():
    _refused("must be a RolloutCarry", carry=dict(t0=0))


def test_actor_only_rollout_takes_no_carry():
    _refused("actor_only", actor_only=True)


def test_valid_segment_passes_the_host_checks():
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import check_segment
    for t0, S in ((0, 50), (100, 50), (0, 150), (149, 1), (75, 75)):
        check_segment(_carry(t0=t0), S, T_EP, B, N, L, E, D, "cpu")
