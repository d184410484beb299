"""CPU checks of the history-replay interface: the fused step's `flags` field and bits agree between include/marl_b200.h and the
ctypes binding, bad flags are rejected before any CUDA call, and the stored-history size the rollout decides on."""
import ctypes
import os
import re

from conftest import ROOT


def _header():
    src = open(os.path.join(ROOT, "include", "marl_b200.h")).read()
    return re.sub(r"/\*.*?\*/", "", src, flags=re.S)


def _struct_fields(src, name):
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), src, flags=re.S).group(1)
    fields = []
    for decl in body.split(";"):
        fields += re.findall(r"(\w+)\s*(?=,|$)", decl.strip())
    return fields


def test_policy_step_flags_match_header():
    from distributed_multi_agent_reinforcement_learning_b200 import fused_policy
    src = _header()
    assert _struct_fields(src, "marl_policy_step") == [f[0] for f in fused_policy.PolicyStep._fields_]
    assert fused_policy.PolicyStep._fields_[-1] == ("flags", ctypes.c_int32)
    assert ctypes.sizeof(fused_policy.PolicyStep) == 160                  # the field replaced `reserved`: same size and offsets
    assert fused_policy.PolicyStep.flags.offset == 156
    bits = dict(re.findall(r"#define MARL_POLICY_(\w+) (\d+)", src))
    assert {k: int(v) for k, v in bits.items()} == {"STATE_F32": fused_policy.STATE_F32, "EMBED_ONLY": fused_policy.EMBED_ONLY}


def _step_args(flags, variant):
    from distributed_multi_agent_reinforcement_learning_b200 import fused_policy
    s = fused_policy.PolicyStep()
    s.B, s.N, s.O, s.E, s.depth, s.action_dim, s.variant, s.flags = 4, 8, 16, 128, 1, 9, variant, flags
    for f in ("d_p_state", "d_e_state", "d_oxy", "d_map_id", "d_o_count", "d_p_adj_bits", "d_e_adj", "d_o_adj_bits"):
        setattr(s, f, 256)                      # never dereferenced: the arguments are rejected first
    w, io = fused_policy.DhgnWeights(), fused_policy.PolicyNetIO()
    return s, w, io


def test_bad_flags_fail_without_a_gpu():
    from distributed_multi_agent_reinforcement_learning_b200 import _lib, fused_policy
    L = _lib.lib()
    for flags, variant, what in ((4, 0, b"unknown flags"), (1 << 30, 3, b"unknown flags"),
                                 (fused_policy.STATE_F32, 2, b"variant 2"), (fused_policy.EMBED_ONLY, 2, b"variant 2")):
        s, w, io = _step_args(flags, variant)
        rc = L.marl_policy_rollout_step(ctypes.byref(s), ctypes.byref(w), ctypes.byref(io), ctypes.byref(w), ctypes.byref(io), None)
        assert rc == -1, (flags, variant)
        assert what in L.marl_last_error_string(), L.marl_last_error_string()


def test_history_bytes():
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import history_bytes
    assert history_bytes(150, 4096, 8, 128, 1) == 2 * 151 * 4096 * 8 * 128 * 4              # bench shape: 5.1 GB
    assert round(history_bytes(250, 32768, 64, 128, 3) / 1e9) == 543                        # configs[4]: 543 GB
