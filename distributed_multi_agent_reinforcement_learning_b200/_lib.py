"""ctypes binding of libmarl_b200.so (C-ABI declared in include/marl_b200.h).

There is NO CPU fallback: if the CUDA library is missing or a call fails, this module raises.  The library is
built in-tree by `__graft_entry__.build()` (or `make -C distributed_multi_agent_reinforcement_learning_b200/csrc`).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmarl_b200.so")

MARL_OK = 0
EV_HEAP_OVERFLOW, EV_PATH_OVERFLOW, EV_TAPE_EXHAUSTED, EV_MISSED_REPLAN = 1, 2, 4, 8


class MarlError(RuntimeError):
    pass


class EnvParams(C.Structure):
    """marl_env_params (include/marl_b200.h)."""
    _INT = ("W", "H", "N", "O", "max_steps", "difficulty", "sensor_beams", "sensor_radius", "e_extend_dis",
            "e_sen_range")
    _DBL = ("d_step", "d_tau", "d_vmax", "d_collision_radius", "d_comm_range", "d_sen_range", "e_step", "e_tau",
            "e_vmax", "e_collision_radius", "resolution")
    _fields_ = [(n, C.c_int32) for n in _INT] + [(n, C.c_double) for n in _DBL]

    @classmethod
    def from_dict(cls, d):
        p = cls()
        for n in cls._INT:
            setattr(p, n, int(d[n]))
        for n in cls._DBL:
            setattr(p, n, float(d[n]))
        return p

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}

    @property
    def HW(self):
        return (self.H + 31) // 32

    @property
    def OW(self):
        return (self.O + 31) // 32

    @property
    def NW(self):
        return (self.N + 31) // 32


class RolloutRecords(C.Structure):
    """marl_rollout_records: device pointers of the time-major rollout arena (NULL = not recorded)."""
    FIELDS = ("p_state_f32", "e_state_f32", "p_adj_bits", "e_adj", "o_adj_bits", "a_n", "r", "raw_reward", "active",
              "p_adj_f32", "e_adj_f32", "o_adj_f32")
    _fields_ = [(n, C.c_void_p) for n in FIELDS]


_VP, _I32, _I64, _U64, _F32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_float
_PP = C.POINTER(EnvParams)

_PROTOTYPES = {
    "marl_version": (C.c_int, []),
    "marl_last_error_string": (C.c_char_p, []),
    "marl_env_step": (C.c_int, [_PP, _I32, _I32] + [_VP] * 12),
    "marl_env_observe": (C.c_int, [_PP, _I32, _I32] + [_VP] * 12),
    "marl_raser_map_build": (C.c_int, [_PP, _I32] + [_VP] * 7),
    "marl_evader_step": (C.c_int, [_PP, _I32, _I32, _VP, _VP, _VP, _VP, _VP, _I32, _VP, _VP, _VP, _VP, _VP, _I32, _VP,
                                   _VP, _VP, _VP]),
    "marl_evader_replan": (C.c_int, [_PP, _I32, _I32, _VP, _VP, _VP, _VP, _VP, _I32, _VP, _VP, _VP, _VP, _VP]),
    "marl_rollout_closed": (C.c_int, [_PP, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _VP, _VP, _VP, _VP, _VP, _I32, _VP, _VP, _I32,
                                      _VP, _VP, _VP, _U64, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP,
                                      C.POINTER(RolloutRecords), _VP]),
    "marl_dhgn_message_fwd": (C.c_int, [_I32] * 4 + [_VP] * 8 + [_I32] + [_VP] * 8),
    "marl_dhgn_message_bwd": (C.c_int, [_I32] * 4 + [_VP] * 8 + [_I32] + [_VP] * 14),
    "marl_dhgn_message_bwd_workspace_bytes": (_I64, [_I32, _I32, _I32]),
    "marl_dhgn_message_bwd_det": (C.c_int, [_I32] * 4 + [_VP] * 8 + [_I32] + [_VP] * 15),
    "marl_fcra_agg": (C.c_int, [_I32, _I32, _I32, _VP, _I64, _I64, _VP, _I32, _VP, _VP]),
    "marl_gru_cell_fwd": (C.c_int, [_I64, _I32] + [_VP] * 9),
    "marl_gru_cell_bwd": (C.c_int, [_I64, _I32] + [_VP] * 10),
    "marl_ppo_head": (C.c_int, [_I64, _I32, _I32] + [_VP] * 12 + [_F32, _F32] + [_VP] * 7),
    "marl_ppo_head_workspace_bytes": (_I64, [_I64]),
    "marl_ppo_head_det": (C.c_int, [_I64, _I32, _I32] + [_VP] * 12 + [_F32, _F32] + [_VP] * 8),
    "marl_act_head": (C.c_int, [_I64, _I32, _I32] + [_VP] * 6 + [_U64, _I32, _I32] + [_VP] * 5),
    "marl_gemm_tf32x3": (C.c_int, [_I32, _I32, _I32, _I32, _VP, _I64, _VP, _I64, _VP, _I64, _VP, _VP, _I64, _VP, _I64, _I32, _VP]),
    "marl_policy_pack_bytes": (_I64, [_I32, _I32]),
    "marl_policy_pack": (C.c_int, [_VP, _I32, _I32, _I32, _VP, _VP]),
    "marl_policy_rollout_step": (C.c_int, [_VP] * 6),
    "marl_policy_pack_bytes": (_I64, [_I32, _I32]),
    "marl_policy_pack": (C.c_int, [_VP, _I32, _I32, _I32, _VP, _VP]),
    "marl_policy_rollout_step": (C.c_int, [_VP] * 6),
    "marl_entity_agg_fwd": (C.c_int, [_I64, _I32, _I32, _I32, _I32, _VP, _I32, _VP, _I64, _I64, _I64, _VP, _VP]),
    "marl_entity_agg_bwd": (C.c_int, [_I64, _I32, _I32, _VP, _I32, _VP, _VP, _VP]),
    "marl_gru_pack_bytes": (_I64, []),
    "marl_gru_pack": (C.c_int, [_VP, _VP, _VP]),
    "marl_gru_seq_fwd": (C.c_int, [_I32, _I64, _I32, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "marl_gru_seq_bwd": (C.c_int, [_I32, _I64, _I32, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "marl_relu_bwd": (C.c_int, [_I64, _VP, _VP, _VP, _VP]),
    "marl_skinny_wgrad_workspace_bytes": (_I64, [_I64, _I32, _I32]),
    "marl_skinny_wgrad": (C.c_int, [_I64, _I32, _I32, _VP, _I64, _VP, _I64, _VP, _I64, _VP, _VP, _VP]),
    "marl_wgrad_workspace_bytes": (_I64, [_I64, _I32, _I32]),
    "marl_wgrad_tf32x3": (C.c_int, [_I64, _I32, _I32, _VP, _I64, _VP, _I64, _VP, _I64, _VP, _I32, _VP, _VP]),
    "marl_rowgemm_pack_bytes": (_I64, [_I32, _I32]),
    "marl_rowgemm_pack": (C.c_int, [_VP, _I64, _I64, _I32, _I32, _VP, _VP]),
    "marl_rowgemm_tf32x3": (C.c_int, [_I64, _I32, _I32, _I32, _VP, _I64, _VP, _I64, _VP, _VP, _VP, _I64, _VP, _I64, _I32, _VP]),
    "marl_map_generate": (C.c_int, [_PP, _I32, _I32, C.c_double, C.c_double, C.c_double, _U64, _VP, _VP, _VP]),
    "marl_env_reset_place": (C.c_int, [_PP, _I32, _I32, _VP, _VP, _U64, C.c_double, _I32, _I32, _VP, _VP, _VP, _VP, _VP, _VP]),
    "marl_clip_workspace_bytes": (_I64, [_I64]),
    "marl_clip_grad_norm": (C.c_int, [_I64, _VP, _F32, _VP, _VP, _VP]),
    "marl_adam_step": (C.c_int, [_I64, _VP, _VP, _VP, _VP, _F32, _F32, _F32, _F32, _I64, _VP]),
    "marl_welford_update": (C.c_int, [_I32, _I32, _VP, _VP, _VP, _VP, _VP, _VP, _I32, _VP]),
    "marl_welford_update_f64": (C.c_int, [_I32, _I32, _VP, _VP, _VP, _VP, _VP, _VP, _I32, _VP]),
    "marl_gae_workspace_bytes": (_I64, [_I32, _I32, _I32]),
    "marl_gae": (C.c_int, [_I32, _I32, _I32, _VP, _VP, _VP, _I32, _F32, _F32, _I32, _VP, _VP, _VP, _VP]),
    "marl_gather_rows": (C.c_int, [_VP, _VP, _VP, _I32, _I64, _I64, _VP]),
    "marl_env3d_step": (C.c_int, [_VP, _I32] + [_VP] * 10),
    "marl_env3d_evader_step": (C.c_int, [_VP, _I32] + [_VP] * 4),
    "marl_env3d_adjacency": (C.c_int, [_VP, _I32] + [_VP] * 8),
    "marl_env3d_rollout": (C.c_int, [_VP, _I32, _I32, _I32, _I32] + [_VP] * 8 + [_U64, _VP, _VP]),
    "marl_envn2n_step": (C.c_int, [_VP, _I32] + [_VP] * 10),
    "marl_envn2n_evader_step": (C.c_int, [_VP, _I32] + [_VP] * 4),
    "marl_envn2n_observe": (C.c_int, [_VP, _I32] + [_VP] * 8),
    "marl_envn2n_rollout": (C.c_int, [_VP, _I32, _I32, _I32, _I32] + [_VP] * 8 + [_U64, _VP, _VP]),
    "marl_rollout_steps": (C.c_int, [_PP, _I32, _I32, _I32, _I32, _I32, _VP, _VP, _VP, _U64, _VP, _VP, _VP, _VP, _VP,
                                     _VP, _VP, _VP, _VP, _VP, C.POINTER(RolloutRecords), _VP]),
}

_lib = None


def exported_symbols():
    """Every entry point include/marl_b200.h declares."""
    return sorted(_PROTOTYPES)


def lib():
    """Loads the CUDA library (once).  Raises MarlError if it has not been built: there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MarlError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(the product path has no CPU fallback)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOTYPES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


CALLS = 0   # successful C-ABI calls so far (each launches >= 1 of our kernels); bench.py reports the delta


def check(rc, what=""):
    global CALLS
    CALLS += 1
    if rc != MARL_OK:
        msg = lib().marl_last_error_string().decode("utf-8", "replace")
        raise MarlError(f"{what or 'marl call'} failed (code {rc}): {msg}")


def ptr(t):
    """Device (or host) address of a torch tensor / None -> NULL.  Tensors must be contiguous, and device tensors must live on
    the CURRENT device: the kernels are launched on the current device's stream (one process per GPU; a rank that forgot
    `torch.cuda.set_device` would otherwise launch on cuda:0 with another device's pointers)."""
    if t is None:
        return None
    if not t.is_contiguous():
        raise MarlError("non-contiguous tensor passed to the C-ABI")
    if t.is_cuda:
        import torch
        if t.device.index != torch.cuda.current_device():
            raise MarlError(f"tensor on {t.device} passed to a launch on cuda:{torch.cuda.current_device()}: call "
                            "torch.cuda.set_device(...) (or wrap the call in torch.cuda.device(...)) first")
    return t.data_ptr()


def stream_ptr(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return s.cuda_stream


def ptr_or_int(v):
    return v
