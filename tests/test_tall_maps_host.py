"""CPU-side checks of the evader's map limits: maps the column-bitmap search cannot hold are refused with MARL_EUNSUPPORTED and a
message naming the limits, before any CUDA call (so this runs without a GPU)."""
import ctypes

import pytest

LIMITS = b"H <= 63 needs W <= 254, H <= 127 needs W <= 162"


def _params(W, H):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib, default_config, env_params_dict
    d = env_params_dict(default_config(env__num_defender=4, map__map_size=[W, H]))
    return _lib.EnvParams.from_dict(d)


@pytest.mark.parametrize("W,H", [(128, 128), (64, 200), (163, 64), (163, 100), (255, 63)])
def test_evader_refuses_maps_beyond_the_search_limits(W, H):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    L = _lib.lib()
    p = _params(W, H)
    buf = ctypes.create_string_buffer(4096)      # never dereferenced: the size check comes first
    a = ctypes.addressof(buf)
    rc = L.marl_evader_step(ctypes.byref(p), 4, 4, a, a, a, a, a, 16, a, a, a, None, a, 1, a, a, None, None)
    assert rc == -3                              # MARL_EUNSUPPORTED
    msg = L.marl_last_error_string()
    assert b"%dx%d" % (W, H) in msg and LIMITS in msg, msg
    rc = L.marl_evader_replan(ctypes.byref(p), 4, 4, a, a, a, a, a, 16, a, a, None, a, None)
    assert rc == -3
    assert LIMITS in L.marl_last_error_string()
