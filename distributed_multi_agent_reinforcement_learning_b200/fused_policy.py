"""Binding of the fused rollout-step kernel (csrc/policy_fused.cu): one launch runs the DHGN encoder, both GRU layers and
the heads of the actor AND the critic for all B envs of a step (DHGN/mappo_parallel.py:758-801, network half).

`FusedRolloutStep` owns the packed (hi/lo TF32, pre-swizzled) weight images and the ctypes structs; it is rebuilt (re-packed)
whenever the weights change, i.e. once per rollout.  Built with `snapshot=True` it also keeps its own copy of every weight the
kernel reads unpacked (message layers, biases, head rows), so it keeps computing the rollout-time networks after the optimizer
has stepped the live parameters - what a replay of the episode's history embeddings needs."""
import ctypes as C
import os

import torch

from . import _lib


class DhgnWeights(C.Structure):
    _fields_ = [("msg_w", C.c_void_p * 3), ("msg_b", C.c_void_p * 3), ("agg_v_w", C.c_void_p), ("agg_v_b", C.c_void_p),
                ("sem_w", C.c_void_p), ("sem_b", C.c_void_p), ("agg_f_w", C.c_void_p * 3), ("agg_f_b", C.c_void_p * 3),
                ("fcra_w", C.c_void_p * 3), ("fcra_b", C.c_void_p * 3), ("gru_w_ih", C.c_void_p * 2),
                ("gru_w_hh", C.c_void_p * 2), ("gru_b_ih", C.c_void_p * 2), ("gru_b_hh", C.c_void_p * 2),
                ("head_w", C.c_void_p), ("head_b", C.c_void_p)]


class PolicyNetIO(C.Structure):
    _fields_ = [("d_packed", C.c_void_p), ("d_hist", C.c_void_p * 3), ("d_emb_out", C.c_void_p), ("d_hidden", C.c_void_p),
                ("d_hidden_out", C.c_void_p)]


class PolicyStep(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("B", "N", "O", "E", "depth", "action_dim", "t", "deterministic", "force_action",
                                         "variant")] + \
               [("seed", C.c_uint64)] + \
               [(n, C.c_void_p) for n in ("d_p_state", "d_e_state", "d_oxy", "d_map_id", "d_o_count", "d_p_adj_bits",
                                          "d_e_adj", "d_o_adj_bits", "d_action", "d_logp", "d_value", "d_debug")] + \
               [("row_offset", C.c_int64), ("tile_rows", C.c_int32), ("flags", C.c_int32)]


# marl_policy_step.flags (include/marl_b200.h)
STATE_F32 = 1       # d_p_state / d_e_state are float [B,N,4] / [B,4] (the rollout arena's records) instead of double
EMBED_ONLY = 2      # encoder + FCRA chain only: write the embeddings; hidden states, actions, log-probs and values untouched


# Kernel variant used when the caller does not ask for one (marl_policy_step.variant): 3 = the actor and the critic chain of a row
# tile interleaved in ONE CTA (policy_pair_kernel) whenever both networks are stepped, 1 = one (tile, network) item per CTA.
DEFAULT_VARIANT = int(os.environ.get("MARL_POLICY_VARIANT", "3"))


def supported(mappo):
    return (mappo.embedding_dim == 128 and mappo.num_layers == 2 and 1 <= mappo.depth <= 3 and mappo.action_dim == 9
            and mappo.rnn_hidden_dim == 128)


def _c(t):
    t = t.detach()
    assert t.dtype == torch.float32 and t.is_cuda
    return t if t.is_contiguous() else t.contiguous()


class FusedRolloutStep:
    def __init__(self, mappo, critic_w_eff, snapshot=False):
        """critic_w_eff: effective [E] critic head row (weight_orig / sigma), constant while the weights are fixed.
        snapshot: copy the weights instead of pointing at the live parameters (see the module docstring)."""
        if not supported(mappo):
            raise _lib.MarlError("fused rollout step needs embedding_dim = rnn_hidden_dim = 128, 2 GRU layers, depth 1..3")
        self.lib = _lib.lib()
        self.depth, self.E, self.A = int(mappo.depth), 128, int(mappo.action_dim)
        dev = mappo.device
        self._keep = []
        self._next_hidden = {}
        enc = mappo.actor.shared_net
        self.w = {}
        self.packed = {}
        keep = self._keep

        def P(t):
            keep.append(_c(t).clone() if snapshot else _c(t))
            return keep[-1].data_ptr()

        for name, net in (("actor", mappo.actor), ("critic", mappo.critic)):
            w = DhgnWeights()
            for r in range(3):
                w.msg_w[r], w.msg_b[r] = P(enc.MSG_layers[r].weight), P(enc.MSG_layers[r].bias)
            av, sem = enc.AGG_layers["AGG_vertex_0"], enc.semantic_layer
            w.agg_v_w, w.agg_v_b, w.sem_w, w.sem_b = P(av.weight), P(av.bias), P(sem.weight), P(sem.bias)
            for k in range(self.depth):
                af, ff = enc.AGG_layers[f"AGG_fcra_{k}"], enc.FCRA_layers[k]
                w.agg_f_w[k], w.agg_f_b[k], w.fcra_w[k], w.fcra_b[k] = P(af.weight), P(af.bias), P(ff.weight), P(ff.bias)
            for l in range(2):
                g = net.GRU
                w.gru_w_ih[l], w.gru_w_hh[l] = P(getattr(g, f"weight_ih_l{l}")), P(getattr(g, f"weight_hh_l{l}"))
                w.gru_b_ih[l], w.gru_b_hh[l] = P(getattr(g, f"bias_ih_l{l}")), P(getattr(g, f"bias_hh_l{l}"))
            if name == "actor":
                w.head_w, w.head_b = P(net.Mean.weight), P(net.Mean.bias)
            else:
                w.head_w, w.head_b = P(critic_w_eff.reshape(-1)), P(net.Mean.bias)
            is_actor = 1 if name == "actor" else 0
            nbytes = int(self.lib.marl_policy_pack_bytes(self.depth, is_actor))
            buf = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
            off = (-buf.data_ptr()) % 1024
            packed = buf[off:off + nbytes]
            _lib.check(self.lib.marl_policy_pack(C.byref(w), self.depth, is_actor, self.A, packed.data_ptr(), _lib.stream_ptr()),
                       "marl_policy_pack")
            self.w[name], self.packed[name] = w, packed
            keep.append(buf)

    def step(self, engine, oxy_i32, o_count, t, seed, deterministic, hist_a, hist_c, emb_a, emb_c, ha, hc, action, logp, value,
             nets=("actor", "critic"), force_action=False, debug=None, variant=0, row_offset=0, tile_rows=0, flags=0):
        """hist_*: list (k = 0 newest) of [B,N,E] tensors or None (zeros); emb_*: [B,N,E] outputs; ha/hc: [2,B*N,E] in/out;
        action i32 [B,N], logp / value f32 [B,N] outputs.
        flags: STATE_F32 (engine.p_state / e_state are the fp32 records [B,N,4] / [B,4]) | EMBED_ONLY (ha / hc / action / logp /
        value may be None and are not touched).
        variant: 0 = DEFAULT_VARIANT, 1 = one (tile, network) item per CTA (hidden state updated in place), 2 = two such CTAs per
        SM, 3 = both networks' chains of a tile interleaved in one CTA.  Variant 2 reads the previous hidden state from one
        buffer and writes the new one to another; afterwards the two tensors trade their storage, so for the caller `ha` / `hc`
        are still updated "in place" (views taken before the call keep the old state)."""
        if int(variant) == 0 and DEFAULT_VARIANT == 3 and "actor" in nets and "critic" in nets:
            variant = 3          # (16-agent envs run the pair kernel with 8 worker warps: their message path needs a whole env per warp)
        if int(variant) == 3 and not ("actor" in nets and "critic" in nets):
            variant = 1          # a single network (the critic-only bootstrap step): nothing to interleave
        s = PolicyStep()
        s.B, s.N, s.O, s.E, s.depth, s.action_dim = engine.B, engine.N, engine.O, self.E, self.depth, self.A
        s.t, s.deterministic, s.seed = int(t), 1 if deterministic else 0, int(seed) & 0xFFFFFFFFFFFFFFFF
        s.force_action = 1 if force_action else 0
        s.variant = int(variant)
        s.row_offset = int(row_offset)
        s.tile_rows = int(tile_rows)
        s.flags = int(flags)
        P = _lib.ptr
        s.d_debug = P(debug) if debug is not None else None
        s.d_p_state, s.d_e_state, s.d_oxy, s.d_map_id, s.d_o_count = (P(engine.p_state), P(engine.e_state), P(oxy_i32),
                                                                        P(engine.map_id), P(o_count))
        s.d_p_adj_bits, s.d_e_adj, s.d_o_adj_bits = P(engine.p_adj_bits), P(engine.e_adj), P(engine.o_adj_bits)
        s.d_action, s.d_logp, s.d_value = P(action), P(logp), P(value)
        ios, swaps = {}, []
        for name, hist, emb, hid in (("actor", hist_a, emb_a, ha), ("critic", hist_c, emb_c, hc)):
            if name not in nets:
                continue
            io = PolicyNetIO()
            io.d_packed = self.packed[name].data_ptr()
            for k in range(self.depth):
                io.d_hist[k] = P(hist[k]) if hist[k] is not None else None
            assert hid is None or hid.is_contiguous()
            io.d_emb_out, io.d_hidden, io.d_hidden_out = P(emb), P(hid), None
            if int(variant) == 2:                            # the two-CTA-per-SM kernel re-reads the previous state: separate output buffer
                # the partner buffer belongs to THIS hidden-state tensor (env-group pipelines step their own states concurrently)
                nxt = getattr(hid, "_marl_next", None)
                if nxt is None or nxt.shape != hid.shape or nxt.device != hid.device:
                    nxt = torch.empty_like(hid)
                    hid._marl_next = nxt
                io.d_hidden_out = P(nxt)
                swaps.append((hid, nxt))
            ios[name] = io
        a_w, a_io = (C.byref(self.w["actor"]), C.byref(ios["actor"])) if "actor" in ios else (None, None)
        c_w, c_io = (C.byref(self.w["critic"]), C.byref(ios["critic"])) if "critic" in ios else (None, None)
        _lib.check(self.lib.marl_policy_rollout_step(C.byref(s), a_w, a_io, c_w, c_io, _lib.stream_ptr()),
                   "marl_policy_rollout_step")
        for hid, nxt in swaps:                               # the caller's tensor now holds the new state, its partner the old buffer
            hid.data, nxt.data = nxt.data, hid.data
