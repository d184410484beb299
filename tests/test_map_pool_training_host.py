"""CPU checks of training on an installed map pool: the map modes of `reset_device` and `AutoReset` are validated, a reset that keeps
the maps is refused before any CUDA call on an engine whose maps were never set, the `train_loop.py --map-pool` argument errors, and
`marl_map_draw` refuses bad arguments with MARL_EINVAL and a message."""
import ctypes
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B, N, L, E, D, T_EP = 4, 8, 2, 128, 1, 150


def _fake_engine(maps_set):
    """The attributes reset_device reads before its first CUDA call."""
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    return SimpleNamespace(maps_set=maps_set, MAP_MODES=BatchedPursuitEnv.MAP_MODES)


@pytest.mark.parametrize("maps", ["pool", "", None, "Draw"])
def test_reset_device_refuses_an_unknown_map_mode(maps):
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    for maps_set in (False, True):
        with pytest.raises(ValueError, match="'generate', 'keep' or 'draw'"):
            BatchedPursuitEnv.reset_device(_fake_engine(maps_set), seed=1, maps=maps)


@pytest.mark.parametrize("maps", ["keep", "draw"])
def test_reset_device_keeping_maps_that_were_never_set_raises_before_any_cuda_call(maps):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    with pytest.raises(_lib.MarlError, match="never set"):
        BatchedPursuitEnv.reset_device(_fake_engine(False), seed=1, maps=maps)
    with pytest.raises(_lib.MarlError, match="never set"):          # whatever the seed and tape
        BatchedPursuitEnv.reset_device(_fake_engine(False), seed=torch.zeros(1, dtype=torch.int64), tape="device", maps=maps)


def test_engine_maps_are_unset_until_set():
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    assert BatchedPursuitEnv.maps_set is False and BatchedPursuitEnv.MAP_MODES == ("generate", "keep", "draw")


def test_auto_reset_map_mode():
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import AutoReset
    assert AutoReset(lambda e: e, lambda e: e).maps == "generate"
    for maps in ("generate", "keep", "draw"):
        assert AutoReset(lambda e: e, lambda e: e, 8, "device", maps=maps).maps == maps
    with pytest.raises(ValueError, match="maps='pool'"):
        AutoReset(lambda e: e, lambda e: e, maps="pool")


def _carry():
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    z = torch.zeros
    return RolloutCarry(0, z(L, B * N, E), z(L, B * N, E), z(D, B, N, E), z(D, B, N, E))


def _fake_mappo():
    return SimpleNamespace(embedding_dim=E, depth=D, num_layers=L, device=torch.device("cpu"), action_dim=9, rnn_hidden_dim=E,
                           cfg=SimpleNamespace(env=SimpleNamespace(max_steps=T_EP)))


def test_check_auto_reset_validates_the_map_mode():
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import AutoReset, check_auto_reset
    auto = AutoReset(lambda e: e, lambda e: e, maps="draw")
    check_auto_reset(auto, _carry(), 64, T_EP, B, N, L, E, D, "cpu")
    with pytest.raises(_lib.MarlError, match="never set"):
        check_auto_reset(auto, _carry(), 64, T_EP, B, N, L, E, D, "cpu", maps_set=False)
    check_auto_reset(AutoReset(lambda e: e, lambda e: e), _carry(), 64, T_EP, B, N, L, E, D, "cpu", maps_set=False)
    auto.maps = "pool"                                      # changed after construction
    with pytest.raises(_lib.MarlError, match="auto_reset.maps='pool'"):
        check_auto_reset(auto, _carry(), 64, T_EP, B, N, L, E, D, "cpu")


@pytest.mark.parametrize("tape", ["torch", "device"])
@pytest.mark.parametrize("maps", ["keep", "draw"])
def test_auto_reset_keeping_unset_maps_is_refused_before_any_cuda_call(maps, tape):
    """rollout_batched and explore_batched refuse a stream whose resets would keep maps the engine never had, before the first
    segment runs (the reset itself would raise only at the boundary, after the segment's first piece)."""
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO, AutoReset
    engine, arena = SimpleNamespace(B=B, N=N), SimpleNamespace(T=T_EP)     # no tensors: a CUDA call would fail here
    auto = AutoReset(lambda e: e, lambda e: e, tape=tape, maps=maps)
    with pytest.raises(_lib.MarlError, match="never set"):
        MAPPO.rollout_batched(_fake_mappo(), engine, arena, 64, carry=_carry(), auto_reset=auto)
    if tape == "device":
        with pytest.raises(_lib.MarlError, match="never set"):
            MAPPO.explore_batched(_fake_mappo(), engine, arena, 64, carry=_carry(), auto_reset=auto)


def test_map_draw_refuses_bad_arguments_without_a_gpu():
    from distributed_multi_agent_reinforcement_learning_b200 import _lib, default_config
    from distributed_multi_agent_reinforcement_learning_b200.config import env_params_dict
    lib = _lib.lib()
    p = ctypes.byref(_lib.EnvParams.from_dict(env_params_dict(default_config())))
    u64 = ctypes.c_uint64
    for Bx, M, out in ((0, 4, 256), (-1, 4, 256), (4, 0, 256), (4, -3, 256), (4, 4, None)):
        assert lib.marl_map_draw(p, Bx, M, u64(1), out, None) == -1, (Bx, M, out)                # MARL_EINVAL
        assert b"marl_map_draw: bad arguments" in lib.marl_last_error_string()
        assert lib.marl_map_draw_dseed(p, Bx, M, 256, out, None) == -1, (Bx, M, out)
        assert b"marl_map_draw: bad arguments" in lib.marl_last_error_string()
    assert lib.marl_map_draw_dseed(p, 4, 4, None, 256, None) == -1
    assert b"d_seed is NULL" in lib.marl_last_error_string()
    assert lib.marl_map_draw(None, 4, 4, u64(1), 256, None) == -1


# ------------------------------------------------------------------------------------------------ tools/train_loop.py
def _pool_dir(tmp_path, M=5, W=60, H=55, O=4):
    """A structurally valid pool on disk (its tables are not checked before the GPU runs)."""
    from distributed_multi_agent_reinforcement_learning_b200.map_pool import MapPool
    z = np.zeros
    MapPool(z((M, W, H), np.uint8), z((M, W, H), np.uint8), z((M, W, H, O), np.uint8), z((0, 2), np.int64), z(M, np.int64),
            z((0, 2), np.int64), z(M, np.int64)).save(str(tmp_path))
    return str(tmp_path)


def _arg_error(*args):
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.join(ROOT, "tools", "train_loop.py")] + list(args)
    r = subprocess.run(cmd, cwd=ROOT, timeout=300, capture_output=True, text=True)
    assert r.returncode == 2, (r.returncode, r.stdout, r.stderr)           # argparse's error exit, before any CUDA call
    return r.stderr


def test_train_loop_map_pool_argument_errors(tmp_path):
    pool = _pool_dir(tmp_path / "pool")
    assert "does not combine with --host-reset" in _arg_error("--map-pool", pool, "--host-reset")
    assert "does not combine with --maps" in _arg_error("--map-pool", pool, "--maps", "32")
    assert "does not combine with --maps" in _arg_error("--map-pool", pool, "--maps", "3")
    assert "--held-out needs --map-pool" in _arg_error("--held-out", "2")
    assert "leaves no training map" in _arg_error("--map-pool", pool, "--held-out", "5")
    assert "--held-out must be >= 0" in _arg_error("--map-pool", pool, "--held-out", "-1")
    assert "--eval-every and --eval-envs >= 1" in _arg_error("--map-pool", pool, "--held-out", "2", "--eval-every", "0")
    assert "--eval-every and --eval-envs >= 1" in _arg_error("--map-pool", pool, "--held-out", "2", "--eval-envs", "0")
    assert "missing" in _arg_error("--map-pool", str(tmp_path / "nowhere"))
