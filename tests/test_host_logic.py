"""CPU-side checks: the C-ABI library loads and exports every declared symbol; the config loader accepts the
reference's YAML schema; the host reset reproduces the reference's initial state from the same global seeds."""
import ctypes
import os
import random
import re

import numpy as np
import pytest

from conftest import ROOT, env_fixture_names, golden

PKG = "distributed_multi_agent_reinforcement_learning_b200"


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "marl_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(marl_[a-z_0-9]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    handle = ctypes.CDLL(_lib.LIB_PATH)
    declared = _header_symbols()
    assert len(declared) >= 10
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in include/marl_b200.h but not exported"
    assert sorted(_lib.exported_symbols()) == declared, "python prototypes out of sync with the header"
    handle.marl_version.restype = ctypes.c_int
    assert handle.marl_version() == 1


def test_params_struct_matches_header_and_oracle(oracle):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    assert [f[0] for f in _lib.EnvParams._fields_] == [f[0] for f in oracle.EnvParams._fields_]
    assert ctypes.sizeof(_lib.EnvParams) == ctypes.sizeof(oracle.EnvParams) == 10 * 4 + 11 * 8


def test_bad_arguments_fail_loudly_without_a_gpu():
    """Validation happens before any CUDA call, so error behaviour is testable on a CPU-only box."""
    from distributed_multi_agent_reinforcement_learning_b200 import _lib, default_config, env_params_dict
    L = _lib.lib()
    d = env_params_dict(default_config())
    d["N"] = 1          # the reference indexes adjacency column 1: N=1 cannot work there either
    p = _lib.EnvParams.from_dict(d)
    rc = L.marl_env_step(ctypes.byref(p), 4, 4, *([None] * 12))
    assert rc == -1 and b"N=1" in L.marl_last_error_string()
    with pytest.raises(_lib.MarlError):
        _lib.check(rc, "marl_env_step")
    p = _lib.EnvParams.from_dict(env_params_dict(default_config()))
    assert L.marl_env_step(ctypes.byref(p), 4, 4, *([None] * 12)) == -1       # null pointers
    assert L.marl_gae(0, 1, 1, None, None, None, 0, 0.99, 0.94, 1, None, None, None, None) == -1


CONFIG_YAML = """
defaults:
  - _self_
hydra:
  run:
    dir: .
main:
env:
  env_class:
    _target_: environment.pursuit_evasion_game.pursuit_env.Pursuit_Env
  state_dim: 4
  action_dim: 9
  max_steps: 150
  num_attacker: 1
  num_defender: 15
  num_target: 1
  step_size: 0.1
  difficulty: 10
sensor: {num_beams: 36, radius: 8}
map: {center: [30, 25], map_size: [60, 55], num_obstacle_block: 5, resolution: 1, variance: 10, num_max_obstacle: 176}
attacker: {collision_radius: 0.5, comm_range: 16, sen_range: 8, step_size: 0.1, tau: 0.2, vmax: 4, extend_dis: 1}
defender: {collision_radius: 0.5, comm_range: 16, sen_range: 8, step_size: 0.1, tau: 0.2, vmax: 2}
algo: {depth: 1, gamma: 0.99, lamda: 0.95, epochs: 1}
"""


def test_config_loader_accepts_the_hydra_schema(tmp_path):
    from distributed_multi_agent_reinforcement_learning_b200 import env_params_dict, load_conf_dir, load_config
    f = tmp_path / "config.yaml"
    f.write_text(CONFIG_YAML)
    cfg = load_config(str(f))
    assert cfg.env.num_defender == 15 and cfg.map.map_size == [60, 55] and cfg["algo"]["depth"] == 1
    assert cfg.env.env_class._target_.endswith("Pursuit_Env")
    d = env_params_dict(cfg)
    assert (d["W"], d["H"], d["N"], d["O"], d["e_extend_dis"]) == (60, 55, 15, 176, 1)
    # flat per-group dumps: tuple tags, `max_num_obstacle`, x_dim/y_dim, K_epochs (conf/*.yaml schema)
    conf = tmp_path / "conf"
    conf.mkdir()
    (conf / "env.yaml").write_text("max_steps: 250\nnum_attacker: 1\nnum_defender: 10\nnum_target: 1\nstep_size: 0.1\n")
    (conf / "sensor.yaml").write_text("num_beams: 36\nradius: 8\n")
    (conf / "mao.yaml").write_text("center: !!python/tuple\n- 30\n- 30\nmap_size: !!python/tuple\n- 60\n- 60\n"
                                   "max_num_obstacle: 110\nnum_obstacle_block: 5\nresolution: 1\nvariance: 10\n")
    (conf / "attacker.yaml").write_text("collision_radius: 0.5\ncomm_range: 16\nextend_dis: 3\nsen_range: 8\n"
                                        "step_size: 0.1\ntau: 0.2\nvmax: 4\n")
    (conf / "defender.yaml").write_text("collision_radius: 0.5\ncomm_range: 16\nsen_range: 8\nstep_size: 0.1\ntau: 0.2\nvmax: 2\n")
    (conf / "algo.yaml").write_text("K_epochs: 1\naction_dim: 9\nstate_dim: 4\ndepth: 3\n")
    c2 = load_conf_dir(str(conf))
    d2 = env_params_dict(c2)
    assert (d2["W"], d2["H"], d2["N"], d2["O"], d2["max_steps"], d2["e_extend_dis"]) == (60, 60, 10, 110, 250, 3)
    assert c2.algo.epochs == 1 and c2.env.action_dim == 9


def _cfg_for(fx):
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    g = lambda k: fx["param_" + k].item()
    W, H = g("W"), g("H")
    return default_config(env__num_defender=g("N"), env__max_steps=g("max_steps"), map__map_size=[W, H],
                          map__center=[30, 25] if H == 55 else [30, 30], map__num_max_obstacle=g("O"),
                          attacker__extend_dis=g("e_extend_dis"))


@pytest.mark.parametrize("name", [n for n in env_fixture_names() if "edge" not in n])
def test_reset_reproduces_reference_initial_state(name):
    """Same global seeds -> the reference's map, target, pursuers and evader, bit for bit."""
    from distributed_multi_agent_reinforcement_learning_b200 import maps
    fx = golden(name)
    seed = int(fx["seed"])
    random.seed(seed)
    np.random.seed(seed)
    r = maps.reset_one(_cfg_for(fx), maps.RefRng())
    assert np.array_equal(r["grid"], fx["grid"])
    assert np.array_equal(r["inflated"], fx["inflated"])
    assert tuple(r["target"]) == tuple(fx["target"][0])
    assert np.array_equal(r["p_state"].view(np.int64), fx["p_state"][0].view(np.int64))
    assert np.array_equal(r["e_state"].view(np.int64), fx["e_before"][0].view(np.int64))


def test_tables_match_reference():
    from distributed_multi_agent_reinforcement_learning_b200 import maps
    fx = golden("env_n8_s2")
    assert np.array_equal(maps.action_table(2), fx["action_table"])
    assert np.array_equal(maps.beam_directions(36), fx["beam_dir"])


def test_pack_unpack_roundtrip():
    from distributed_multi_agent_reinforcement_learning_b200 import maps
    rng = np.random.default_rng(0)
    g = (rng.random((3, 60, 55)) < 0.2).astype(np.uint8)
    w = maps.pack_grid(g)
    assert w.shape == (3, 60, 2) and w.dtype == np.int32
    assert np.array_equal(maps.unpack_words(w, 55), g)
    assert ((w.view(np.uint32)[..., 1] >> (55 - 32)) == 0).all()    # padding bits stay clear


def test_dilate_matches_oracle(oracle):
    from distributed_multi_agent_reinforcement_learning_b200 import maps
    fx = golden("env_n8_s2")
    p = oracle.EnvParams.from_fixture(fx)
    for e in (0, 1, 2, 3):
        assert np.array_equal(maps.dilate(fx["grid"], e), oracle.dilate(p, fx["grid"], e))
