"""MAPPO with the DHGN heterogeneous-graph encoder — B200 mirror of the reference `DHGN/mappo_parallel.py`.

Same class names, constructor signatures, sub-module names (`shared_net`, `GRU`, `Mean`) and state_dict keys as the
reference (`DHGN`, `SharedActor`, `SharedCritic`, `MAPPO`: DHGN/mappo_parallel.py:116-831), so checkpoints written by
`torch.save(actor)` / `state_dict()` interchange (main.py:149-169, evaluator.py:329-330), and — because layers are
created in the reference's order with the same torch initialisers — `torch.manual_seed(s); MAPPO(cfg, ...)` yields the
reference's initial weights.

The compute path is not the reference's: adjacency stays bit-packed, the three relations are message-passed and
aggregated by one fused kernel, history averaging / GRU cells / heads+PPO loss / clip / Adam are our kernels
(csrc/policy_kernels.cu via policy_ops.py); only the dense E-wide layers are library GEMMs.  The whole rollout for B
envs runs on the GPU (`MAPPO.rollout_batched`); `explore_env(env, n)` keeps the reference's single-env signature.

Reference quirks kept on purpose (SURVEY 7.4-5; parity is defined per phase):
  * one encoder instance shared by actor and critic (:582-616); only `critic.Mean` is spectrally normalised (:485);
  * rollout history: actor and critic datasets alias ONE list (:750-752), so both see [C(t-1), A(t-1), C(t-2), ...];
  * critic "all ones" adjacency spans the O_b real boundary cells in rollout but all O padded slots in training;
  * gradients accumulate over minibatches and clip_grad_norm_ acts on the running accumulation (:708-711);
  * minibatches are sequential, unshuffled index ranges (:665).
"""
import os
import time
from types import SimpleNamespace

import numpy as np
import torch
import torch.nn as nn
from torch.nn.utils import spectral_norm

from . import _lib, fused_policy, policy_ops as ops
from .normalization import Normalization
from .replay_buffer import BigBuffer, ReplayBuffer
from .train_stats import TrainStats


TWO_STREAM_TRAIN = True     # actor and critic branches of a training minibatch on two CUDA streams
import os as _os
CONCURRENT_MINIBATCHES = int(_os.environ.get("MARL_CONCURRENT_MB", "3"))  # minibatches of an epoch in flight at once (their clip-accumulate order is replayed afterwards)
# A rollout stores the full [T+D,B,N,E] history of both networks when it takes at most this share of the device memory free at the
# call (free to the driver plus what the caching allocator holds unused); otherwise it keeps a ring of D+1 slabs per network and
# training regenerates each minibatch's history (HistoryReplay).  The share leaves the rest for the arena and the training epoch.
STORE_HISTORY_SHARE = 0.5
REPLAY_EMBED_ONLY = True    # the replay runs the embeddings-only fused step (MARL_POLICY_EMBED_ONLY), not the full step


def history_bytes(T, B, N, E, D):
    """Bytes of the stored history of both networks, [T+D,B,N,E] fp32 each."""
    return 2 * (T + D) * B * N * E * 4


def _history_inputs(hist_a, hist_c, t, D, quirks, net, slot, sl=slice(None), t0=0):
    """The D history inputs of step t for `net` (k = 0 newest; None = zeros, before the episode's first step), read from the
    [*, B, N, E] buffers at index slot(i) for history step i (t + D is what step t writes).  reference_quirks: the ONE list actor and
    critic alias (:750-752), C(t-1), A(t-1), C(t-2), ...; otherwise each network's own embeddings.  t is local to a segment that
    starts at the episode's step t0; indices 0..D-1 hold the embeddings carried in from the previous segment."""
    out = []
    for k in range(D):
        if quirks:
            back, src = k // 2 + 1, (hist_c if k % 2 == 0 else hist_a)
        else:
            back, src = k + 1, (hist_a if net == "actor" else hist_c)
        out.append(src[slot(t - back + D)][sl] if t0 + t - back >= 0 else None)
    return out


def _bootstrap_history(hist_a, hist_c, T, D, quirks, slot, sl=slice(None), t0=0):
    """The critic's D history inputs of the bootstrap value after a segment's last step T-1 (None = zeros).  reference_quirks: only the
    critic's dataset is updated once more (:806-825), so the aliased list is C(T-1), then the list of step T-1 without its oldest entry;
    otherwise the critic's own history of step T."""
    if quirks:
        return [hist_c[slot(T - 1 + D)][sl]] + _history_inputs(hist_a, hist_c, T - 1, D, True, "actor", slot, sl, t0)[:D - 1]
    return _history_inputs(hist_a, hist_c, T, D, False, "critic", slot, sl, t0)


class RolloutCarry:
    """The recurrent state one rollout segment hands to the next segment of the same episode.

    t0: the episode's env step at which the next segment starts.  ha / hc: the actor's and the critic's GRU hidden states
    [L, B*N, E] after step t0-1.  emb_a / emb_c: the last D embeddings of each network [D, B, N, E], index j = step t0-D+j (zeros
    for steps before the episode's first).  A carry with t0 = 0 is the start of an episode: zero hidden states and zero history."""

    def __init__(self, t0, ha, hc, emb_a, emb_c, episode=0):
        self.t0, self.ha, self.hc, self.emb_a, self.emb_c = int(t0), ha, hc, emb_a, emb_c
        self.episode = int(episode)     # index of the episode that step t0 belongs to (counted by an auto-reset rollout stream)

    @classmethod
    def zeros(cls, mappo, B, N, t0=0, episode=0):
        """An episode start (t0 = 0) for B envs of N agents, on the networks' device."""
        f32 = dict(dtype=torch.float32, device=mappo.device)
        L, E, D = mappo.num_layers, mappo.embedding_dim, mappo.depth
        return cls(t0, torch.zeros(L, B * N, E, **f32), torch.zeros(L, B * N, E, **f32), torch.zeros(D, B, N, E, **f32),
                   torch.zeros(D, B, N, E, **f32), episode=episode)

    def shapes(self):
        return dict(ha=tuple(self.ha.shape), hc=tuple(self.hc.shape), emb_a=tuple(self.emb_a.shape), emb_c=tuple(self.emb_c.shape))

    def copy_(self, other):
        """Copies `other`'s step, episode and tensors into this carry's tensors (same shapes)."""
        self.t0, self.episode = int(other.t0), int(other.episode)
        for k in ("ha", "hc", "emb_a", "emb_c"):
            if getattr(self, k).data_ptr() != getattr(other, k).data_ptr():
                getattr(self, k).copy_(getattr(other, k))
        return self


def check_segment(carry, S, T_ep, B, N, L, E, D, device, actor_only=False):
    """Host-side checks of a rollout segment of S steps continuing `carry` in an episode of T_ep steps; raises MarlError before any
    CUDA call.  S must divide T_ep (a segment never crosses an episode boundary) and the segment must end inside the episode."""
    if actor_only:
        raise _lib.MarlError("rollout_batched: actor_only (the evaluator's episode) runs whole episodes and takes no carry")
    if not isinstance(carry, RolloutCarry):
        raise _lib.MarlError(f"rollout_batched: carry must be a RolloutCarry, not {type(carry).__name__}")
    if S <= 0 or T_ep % S != 0:
        raise _lib.MarlError(f"rollout segment of {S} steps: the length must be a positive divisor of the episode length {T_ep}")
    if carry.t0 < 0 or carry.t0 + S > T_ep:
        raise _lib.MarlError(f"rollout segment [{carry.t0}, {carry.t0 + S}) does not lie inside the episode of {T_ep} steps")
    _check_carry_tensors(carry, B, N, L, E, D, device)


def _check_carry_tensors(carry, B, N, L, E, D, device):
    want = dict(ha=(L, B * N, E), hc=(L, B * N, E), emb_a=(D, B, N, E), emb_c=(D, B, N, E))
    have = carry.shapes()
    dev = torch.device(device)
    for k in want:
        x = getattr(carry, k)
        if (have[k] != want[k] or x.dtype != torch.float32 or x.device.type != dev.type
                or (dev.index is not None and x.device.index != dev.index)):
            raise _lib.MarlError(f"rollout carry: {k} is {have[k]} {x.dtype} on {x.device}, this rollout needs {want[k]} float32 on "
                                 f"{device}")


class AutoReset:
    """Lets a rollout segment run across an episode boundary (`rollout_batched(carry=..., auto_reset=AutoReset(...))`).

    All envs of a batch step in lock-step and an episode ends only at cfg.env.max_steps, so the boundary falls at the same step of the
    segment for every env.  There the rollout bootstraps the finished episode e, resets every env on the device with
    `engine.reset_device(seed=reset_seed(e + 1), tape_len=tape_len)`, zeroes both networks' hidden states and history, and continues
    with episode e + 1.  The actions of episode e are sampled with seed `sample_seed(e)` (keyed by row and the episode's step, as in a
    whole-episode rollout), so a stream of segments collects the episodes that `reset_device(reset_seed(e))` followed by
    `rollout_batched(max_steps, seed=sample_seed(e))` collects, bit for bit.  reset_seed / sample_seed: host callables, episode
    index -> int.  tape: the target tape's draw, as in `reset_device` - "torch" (a torch.Generator) or "device"
    (marl_target_tape_generate), which `explore_batched` needs to replay the reset from a CUDA graph.  maps: the reset's map mode, as in
    `reset_device` - "generate" (new maps every episode), "keep" (the engine's maps and map assignment) or "draw" (every env draws one
    of the engine's M maps, e.g. an installed pool, per episode)."""

    def __init__(self, reset_seed, sample_seed, tape_len=16, tape="torch", maps="generate"):
        if tape not in ("torch", "device"):
            raise ValueError(f"AutoReset: tape={tape!r}, 'torch' or 'device'")
        if maps not in ("generate", "keep", "draw"):
            raise ValueError(f"AutoReset: maps={maps!r}, 'generate', 'keep' or 'draw'")
        self.reset_seed, self.sample_seed, self.tape_len, self.tape = reset_seed, sample_seed, int(tape_len), tape
        self.maps = maps


def check_auto_reset(auto_reset, carry, S, T_ep, B, N, L, E, D, device, actor_only=False, use_fused=True, seed=0, maps_set=True):
    """Host-side checks of an auto-reset rollout segment (any 1 <= S <= T_ep from any step 0 <= carry.t0 < T_ep); raises MarlError
    before any CUDA call.  maps_set: whether the engine's maps were ever set (a reset that keeps them needs them)."""
    if not isinstance(auto_reset, AutoReset):
        raise _lib.MarlError(f"rollout_batched: auto_reset must be an AutoReset, not {type(auto_reset).__name__}")
    if auto_reset.maps not in ("generate", "keep", "draw"):
        raise _lib.MarlError(f"rollout_batched: auto_reset.maps={auto_reset.maps!r}, 'generate', 'keep' or 'draw'")
    if auto_reset.maps != "generate" and not maps_set:
        raise _lib.MarlError(f"rollout_batched: AutoReset(maps={auto_reset.maps!r}) keeps the engine's maps, but they were never set "
                             "(MapPool.install, set_maps or a reset_device(maps='generate') first)")
    if carry is None:
        raise _lib.MarlError("rollout_batched: auto_reset continues a stream of segments and needs a carry (RolloutCarry.zeros at the "
                             "start)")
    if actor_only:
        raise _lib.MarlError("rollout_batched: actor_only (the evaluator's episode) runs whole episodes and takes no auto_reset")
    if not use_fused:
        raise _lib.MarlError("rollout_batched: auto_reset needs the fused policy step (embedding_dim = rnn_hidden_dim = 128, "
                             "2 GRU layers, depth 1..3, 9 actions)")
    if seed != 0:
        raise _lib.MarlError(f"rollout_batched: seed={seed} with auto_reset: the sampling seeds come from auto_reset.sample_seed")
    if not isinstance(carry, RolloutCarry):
        raise _lib.MarlError(f"rollout_batched: carry must be a RolloutCarry, not {type(carry).__name__}")
    if S <= 0 or S > T_ep:
        raise _lib.MarlError(f"auto-reset rollout segment of {S} steps: the length must lie in [1, {T_ep}], the episode length")
    if carry.t0 < 0 or carry.t0 >= T_ep:
        raise _lib.MarlError(f"auto-reset rollout segment from step {carry.t0}: the start must lie in [0, {T_ep})")
    _check_carry_tensors(carry, B, N, L, E, D, device)


def orthogonal_init(layer, gain=1.0):
    for name, param in layer.named_parameters():
        if "bias" in name:
            nn.init.constant_(param, 0)
        elif "weight" in name:
            nn.init.orthogonal_(param, gain=gain)
    return layer


def preproc_layer(input_size, output_size, is_sn=False):
    layer = orthogonal_init(nn.Linear(input_size, output_size))
    return spectral_norm(layer) if is_sn else layer


# ---- dataset shims: same constructors as the reference's (they only carry tensors to the encoder) -----------------
class AttributeDataset:
    def __init__(self, attribute, adjacent, is_critic=False):
        self.attribute, self.adjacent, self.is_critic = attribute, adjacent, is_critic

    def __len__(self):
        return len(self.attribute)


class EmbeddingDataset:
    def __init__(self, attribute, adjacent, is_critic=False, depth=1):
        self.attribute, self.adjacent, self.is_critic, self.depth = attribute, adjacent, is_critic, depth

    def __len__(self):
        return len(self.attribute)

    def update(self, embedding, adjacent):
        del self.attribute[0]
        self.attribute.append(embedding)
        self.adjacent = adjacent


class EmbeddingDataset2(EmbeddingDataset):
    def __len__(self):
        return self.depth


def _dataset_of(loader):
    return getattr(loader, "dataset", loader)


class DHGN(nn.Module):
    """Encoder parameters (reference names).  `encode` is the fused forward used by both networks."""

    def __init__(self, input_dim, embedding_dim, is_sn, algo_config, device):
        super().__init__()
        if algo_config.vertex_level_aggregator != "mean" or algo_config.fcra_aggregator != "mean":
            # the reference's 'pool' / 'att' branches cannot run (Parameter(required_grad=...), masked_fill(mask, value=...))
            raise NotImplementedError("only the 'mean' aggregators are functional in the reference")
        self.ReLU = nn.ReLU()
        self.MSG_layers = nn.ModuleList()
        self.AGG_layers = nn.ModuleDict()
        self.FCRA_layers = nn.ModuleList()
        self.alpha = nn.ModuleDict()
        self.algo_config, self.device = algo_config, device
        self.input_dim, self.embedding_dim, self.depth = input_dim, embedding_dim, int(algo_config.depth)
        mk = (lambda a, b: preproc_layer(a, b)) if is_sn else (lambda a, b: nn.Linear(a, b))
        self.semantic_layer = mk(3 * embedding_dim + input_dim, embedding_dim)
        for r in range(algo_config.num_relation):
            self.MSG_layers.append(mk(2 * input_dim if r == 0 else input_dim, embedding_dim))
        for _ in range(self.depth):
            self.FCRA_layers.append(mk(2 * embedding_dim, embedding_dim))
        self.AGG_layers["AGG_vertex_0"] = mk(embedding_dim, embedding_dim)
        for k in range(self.depth):
            self.AGG_layers[f"AGG_fcra_{k}"] = mk(embedding_dim, embedding_dim)

    def encode(self, graph, all_ones, hist):
        """graph: ops.GraphBatch of S samples; hist: list over k of (tensor, sample_stride, agent_stride) or contiguous
        [S,N,E] tensors, k=0 the most recent.  Returns the FCRA output [S,N,E] (what the reference calls `embedding`)."""
        S, N, E = graph.S, graph.N, self.embedding_dim
        m = self.MSG_layers
        agg = ops.message_agg(graph, all_ones, m[0].weight, m[0].bias, m[1].weight, m[1].bias, m[2].weight, m[2].bias)
        av, sem = self.AGG_layers["AGG_vertex_0"], self.semantic_layer
        emb3 = ops.linear(agg.view(S * N * 3, E), av.weight, av.bias, relu=True).view(S * N, 3 * E)
        # semantic layer on [p | emb0 | emb1 | emb2] without materialising the concatenation: the 4-wide state part is
        # a rank-4 update handed to the GEMM as its additive input
        p_term = ops.skinny_linear(graph.p.view(S * N, 4), sem.weight[:, :4], sem.bias)
        h = ops.linear(emb3, sem.weight[:, 4:], None, add=p_term)
        for k in range(self.depth):
            hk = hist[k]
            if isinstance(hk, tuple):
                nb = ops.fcra_agg(hk[0], graph.p_adj_bits, all_ones, S, N, E, hk[1], hk[2])
            else:
                nb = ops.fcra_agg(hk, graph.p_adj_bits, all_ones, S, N, E)
            af, ff = self.AGG_layers[f"AGG_fcra_{k}"], self.FCRA_layers[k]
            mk = ops.linear(nb.view(S * N, E), af.weight, af.bias, relu=True)
            h = ops.linear(mk, ff.weight, ff.bias, relu=True, x2=h)      # FCRA_k([m_k | h]) without the concatenation
        return h.view(S, N, E)

    # reference signature: forward(attributes: DataLoader, historical_embeddings: DataLoader)
    def forward(self, attributes, historical_embeddings):
        graph, all_ones, lead = _graph_from_datasets(_dataset_of(attributes))
        hd = _dataset_of(historical_embeddings)
        hist = _history_from_dataset(hd, graph, lead)
        out = self.encode(graph, all_ones, hist)
        return out.view(*lead, graph.N, self.embedding_dim).unsqueeze(0)   # DataLoader(batch_size=1) adds a leading 1


def _graph_from_datasets(ds):
    """AttributeDataset(attribute=[p,e,o], adjacent=[p_adj,e_adj,o_adj]) -> GraphBatch (dense fp32 0/1 -> packed bits)."""
    p, e, o = ds.attribute
    p_adj, e_adj, o_adj = ds.adjacent
    lead = tuple(p.shape[:-2])
    N, O = p.shape[-2], o.shape[-2]
    S = int(np.prod(lead)) if lead else 1
    dev = p.device
    pf = p.reshape(S, N, 4).float().contiguous()
    ef = e.reshape(S, 4).float().contiguous()
    oxy = o.reshape(S, O, 4)[..., :2].float().contiguous()
    graph = ops.GraphBatch(pf, ef, oxy, torch.arange(S, dtype=torch.int32, device=dev),
                           torch.full((S,), O, dtype=torch.int32, device=dev),
                           ops.pack_bits(p_adj.reshape(S, N, N)), (e_adj.reshape(S, N) != 0).to(torch.uint8).contiguous(),
                           ops.pack_bits(o_adj.reshape(S, N, O)))
    return graph, bool(ds.is_critic), lead


def _history_from_dataset(hd, graph, lead):
    D = hd.depth
    S, N = graph.S, graph.N
    if isinstance(hd.attribute, (list, tuple)):          # rollout: list of [N,E], newest last (EmbeddingDataset)
        return [hd.attribute[D - 1 - k].reshape(S, N, -1).float().contiguous() for k in range(D)]
    T = lead[-1]                                           # training: [mb, T+D, N, E] (EmbeddingDataset2)
    return [hd.attribute[:, D - 1 - k: D - 1 - k + T].reshape(S, N, -1).float().contiguous() for k in range(D)]


class _SharedNet(nn.Module):
    def _gru_weights(self):
        g = self.GRU
        return [(getattr(g, f"weight_ih_l{l}"), getattr(g, f"weight_hh_l{l}"), getattr(g, f"bias_ih_l{l}"),
                 getattr(g, f"bias_hh_l{l}")) for l in range(self.num_layers)]

    def features(self, emb_TRE, hidden_state):
        """emb [T,R,E], hidden [L,R,E] -> (GRU outputs [T,R,E], new hidden [L,R,E])."""
        return ops.gru_forward(emb_TRE, hidden_state, self._gru_weights(), self.num_layers)

    def get_weights(self):
        return {k: v.cpu() for k, v in self.state_dict().items()}

    def set_weights(self, weights):
        self.load_state_dict(weights)

    def get_gradients(self):
        return [None if p.grad is None else p.grad.data.cpu().numpy() for p in self.parameters()]

    def set_gradients(self, gradients, device):
        for g, p in zip(gradients, self.parameters()):
            if g is not None:
                g = torch.as_tensor(g).to(device)
                if p.grad is not None and p.grad.shape == g.shape:
                    p.grad.copy_(g)            # keeps the flat-arena view alive
                else:
                    p.grad = g


class SharedActor(_SharedNet):
    def __init__(self, shared_net, rnn_input_dim, action_dim, num_layers, rnn_hidden_dim, is_sn=False):
        super().__init__()
        self.shared_net = shared_net
        self.num_layers, self.rnn_input_dim, self.rnn_hidden_dim = num_layers, rnn_input_dim, rnn_hidden_dim
        self.GRU = nn.GRU(rnn_input_dim, rnn_hidden_dim, num_layers)
        self.Mean = preproc_layer(rnn_hidden_dim, action_dim) if is_sn else nn.Linear(rnn_hidden_dim, action_dim)

    def forward(self, attributes, historical_embeddings, hidden_state, mode):
        embedding = self.shared_net(attributes, historical_embeddings)          # [1, (mb, T,) N, E]
        if mode == 0:
            feat, hidden_state = self.features(embedding, hidden_state)
            feature = feat.squeeze(0)
        else:
            emb = embedding.squeeze(0)
            mb, T, N, E = emb.shape
            feat, hidden_state = self.features(emb.permute(1, 0, 2, 3).reshape(T, mb * N, E), hidden_state)
            feature = feat.reshape(T, mb, N, E).permute(1, 0, 2, 3)
        prob = torch.softmax(torch.nn.functional.linear(feature, self.Mean.weight, self.Mean.bias), dim=-1)
        return prob, hidden_state, embedding

    def choose_action(self, attributes, historical_embeddings, hidden_state, deterministic=True, seed=0, t=0):
        embedding = self.shared_net(attributes, historical_embeddings)
        feat, hidden_state = self.features(embedding, hidden_state)
        a, _, logp, _ = ops.act_head(feat[0], None, self.Mean.weight, self.Mean.bias, None, None, seed, t, deterministic)
        if deterministic:
            return a.long(), hidden_state, embedding
        return a.long(), logp, hidden_state, embedding

    def get_logprob_and_entropy(self, attributes, historical_embeddings, hidden_state, action):
        prob, _, _ = self.forward(attributes, historical_embeddings, hidden_state, mode=1)
        dist = torch.distributions.Categorical(prob)
        return dist.log_prob(action), dist.entropy()


class SharedCritic(_SharedNet):
    def __init__(self, shared_net, rnn_input_dim, value_dim, num_layers, rnn_hidden_dim, is_sn=False):
        super().__init__()
        self.shared_net = shared_net
        self.num_layers, self.rnn_input_dim, self.rnn_hidden_dim = num_layers, rnn_input_dim, rnn_hidden_dim
        self.is_sn = is_sn
        self.GRU = nn.GRU(rnn_input_dim, rnn_hidden_dim, num_layers)
        self.Mean = preproc_layer(rnn_hidden_dim, value_dim, is_sn=is_sn)

    def head_weight(self, update_buffers=True):
        """Effective [1,E] weight.  With spectral norm the power iteration runs on every forward, rollout included
        (the reference never calls .eval()), and updates weight_u / weight_v in place."""
        if not self.is_sn:
            return self.Mean.weight, None
        W, u = self.Mean.weight_orig, self.Mean.weight_u
        sigma, u2, v = ops.spectral_sigma(W, u)
        if update_buffers:
            with torch.no_grad():
                self.Mean.weight_u.copy_(u2)
                self.Mean.weight_v.copy_(v)
        return W / sigma, u

    def forward(self, attributes, historical_embeddings, hidden_state, mode):
        embedding = self.shared_net(attributes, historical_embeddings)
        w_eff, _ = self.head_weight()
        if mode == 0:
            feat, hidden_state = self.features(embedding, hidden_state)
            val = torch.nn.functional.linear(feat.squeeze(0), w_eff, self.Mean.bias)
            return val, hidden_state, embedding
        emb = embedding.squeeze(0)
        mb, T, N, E = emb.shape
        feat, _ = self.features(emb.permute(1, 0, 2, 3).reshape(T, mb * N, E), hidden_state)
        feature = feat.reshape(T, mb, N, E).permute(1, 0, 2, 3)
        return torch.nn.functional.linear(feature, w_eff, self.Mean.bias)


class _FlatAdam:
    """torch.optim.Adam(lr, eps=1e-5) over one flat parameter/gradient arena, stepped by our fused kernel.
    Exposes the slice of the optimizer API the reference touches: zero_grad(), step(), param_groups[i]['lr']."""

    def __init__(self, params, lr, eps=1e-5, betas=(0.9, 0.999)):
        self.params = params
        self.param_groups = [dict(lr=lr, eps=eps, betas=betas, params=params)]
        n = sum(p.numel() for p in params)
        dev = params[0].device
        self.flat_param = torch.empty(n, dtype=torch.float32, device=dev)
        self.flat_grad = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros_like(self.flat_param)
        self.exp_avg_sq = torch.zeros_like(self.flat_param)
        self.step_count = 0
        off = 0
        self._views = []
        for p in params:
            k = p.numel()
            self.flat_param[off:off + k].copy_(p.data.reshape(-1))
            p.data = self.flat_param[off:off + k].view_as(p.data)
            p.grad = self.flat_grad[off:off + k].view_as(p.data)
            self._views.append((off, k))
            off += k

    def _sync_grads(self):
        for p, (off, k) in zip(self.params, self._views):
            view = self.flat_grad[off:off + k]
            if p.grad is None:
                view.zero_()
                p.grad = view.view_as(p.data)
            elif p.grad.data_ptr() != view.data_ptr():
                view.copy_(p.grad.reshape(-1))
                p.grad = view.view_as(p.data)

    def zero_grad(self, set_to_none=False):
        self.flat_grad.zero_()
        self._sync_grads()

    def state_dict(self):
        """Adam state as CPU tensors and plain values: both moments, the step count and the current learning rate."""
        return dict(exp_avg=self.exp_avg.cpu(), exp_avg_sq=self.exp_avg_sq.cpu(), step_count=int(self.step_count),
                    lr=float(self.param_groups[0]["lr"]))

    def load_state_dict(self, sd):
        """Copies a `state_dict()` into the existing arenas in place: the parameters stay views into `flat_param`."""
        for k in ("exp_avg", "exp_avg_sq"):
            if tuple(sd[k].shape) != tuple(self.exp_avg.shape) or sd[k].dtype != self.exp_avg.dtype:
                raise _lib.MarlError(f"Adam state: {k} is {tuple(sd[k].shape)} {sd[k].dtype}, the optimizer's arena is "
                                     f"{tuple(self.exp_avg.shape)} {self.exp_avg.dtype}")
        self.exp_avg.copy_(sd["exp_avg"])
        self.exp_avg_sq.copy_(sd["exp_avg_sq"])
        self.step_count = int(sd["step_count"])
        for g in self.param_groups:
            g["lr"] = float(sd["lr"])

    def step(self):
        self._sync_grads()
        self.step_count += 1
        g = self.param_groups[0]
        ops.adam_step_(self.flat_param, self.flat_grad, self.exp_avg, self.exp_avg_sq, g["lr"], self.step_count,
                       betas=g["betas"], eps=g["eps"])


class TrainBatch:
    """Training data in the engine's canonical form: time-major, bit-packed adjacency.  Built from a reference-layout
    dict (`from_reference`, [B,T,...] dense fp32 as in DHGN/replay_buffer.py:28-40) or directly from a rollout."""

    KEYS = ("p", "e", "p_adj_bits", "e_adj", "o_adj_bits", "hist_a", "hist_c", "v", "a", "logp", "r", "active")
    replay = None       # HistoryReplay of a batch whose history was not stored (hist_a = hist_c = None); minibatches regenerate it
    map_id = None       # i32 [B] (replay only; a batch that crossed an episode boundary: the ids of the episode that ended)
    # A rollout segment (rollout_batched(carry=...)) starts at the episode's step t0 from the GRU hidden states h0_a / h0_c
    # [L, B*N, E]; a replay-mode segment also keeps its D history-prefix slabs prefix_a / prefix_c [D, B, N, E] (a store-mode one has
    # them as slabs 0..D-1 of hist_a / hist_c).  `carry` is the RolloutCarry the next segment continues from.  A whole-episode batch
    # has t0 = 0 and None for all of them: zero hidden states and zero history.
    t0 = 0
    h0_a = h0_c = prefix_a = prefix_c = carry = None
    # A segment that crossed an episode boundary (rollout_batched(auto_reset=...)) has boundary = k: steps [0, k) end one episode and
    # [k, T) start the next, which trains from zero hidden states and zero history, on its own maps oxy2 / o_count_train2 (replay2:
    # its HistoryReplay; map_id2: its map ids, which a reset that draws the maps changes).  v_boot [B,N] is the bootstrap value after
    # step k-1.  `pieces()` views it as those two ordinary batches; a minibatch of it holds the minibatches of both pieces in `parts`.
    # ended_collision / ended_evader_status [B]: the flags of the episode that ended during the segment (the reset cleared the engine's).
    boundary = v_boot = oxy2 = o_count_train2 = replay2 = map_id2 = parts = None
    ended_collision = ended_evader_status = None
    zero_prefix = False     # a store-mode piece whose history slabs 0..D-1 belong to the previous episode: they read as zeros

    def __init__(self, **kw):
        self.__dict__.update(kw)
        self.T, self.B, self.N = self.p.shape[:3]

    @classmethod
    def from_reference(cls, d, depth):
        tm = lambda x: x.transpose(0, 1).contiguous()
        B = d["p_state"].shape[0]
        O = d["o_state"].shape[2]
        dev = d["p_state"].device
        return cls(p=tm(d["p_state"]).float(), e=tm(d["e_state"])[:, :, 0].contiguous().float(),
                   oxy=d["o_state"][:, 0, :, :2].contiguous().float(),
                   o_count_train=torch.full((B,), O, dtype=torch.int32, device=dev),
                   p_adj_bits=ops.pack_bits(tm(d["p_adj"])), e_adj=(tm(d["e_adj"])[..., 0] != 0).to(torch.uint8).contiguous(),
                   o_adj_bits=ops.pack_bits(tm(d["o_adj"])), hist_a=tm(d["actor_historical_embedding"]).float(),
                   hist_c=tm(d["critic_historical_embedding"]).float(), v=tm(d["v_n"]).float(), a=tm(d["a_n"]).float(),
                   logp=tm(d["a_logprob_n"]).float(), r=tm(d["r"]).float(), active=tm(d["active"]).float(), depth=depth)

    def _select(self, tm, em):
        """The minibatch of the envs that `tm` selects from a time-major slab ([X, B, ...] -> [X, mb, ...]) and `em` from an env-major
        tensor ([B, ...] -> [mb, ...]).  A replay-mode batch regenerates the minibatch's history from its slabs (on the current stream)."""
        if self.boundary is not None:
            parts = [pc._select(tm, em) for pc in self.pieces()]
            cat = lambda k: torch.cat([getattr(x, k) for x in parts])     # noqa: E731
            return TrainBatch(p=cat("p"), a=cat("a"), logp=cat("logp"), r=cat("r"), active=cat("active"), v=tm(self.v), depth=self.depth,
                              boundary=self.boundary, parts=parts)

        def opt(x):
            if x is None or not self.zero_prefix:
                return None if x is None else tm(x)
            h = tm(x[self.depth:])                      # the minibatch's own copy, with D zero slabs in front
            return torch.cat([h.new_zeros((self.depth,) + tuple(h.shape[1:])), h])
        mb = TrainBatch(p=tm(self.p), e=tm(self.e), oxy=em(self.oxy), o_count_train=em(self.o_count_train), p_adj_bits=tm(self.p_adj_bits),
                        e_adj=tm(self.e_adj), o_adj_bits=tm(self.o_adj_bits), hist_a=opt(self.hist_a), hist_c=opt(self.hist_c),
                        v=tm(self.v), a=tm(self.a), logp=tm(self.logp), r=tm(self.r), active=tm(self.active), depth=self.depth)
        if self.h0_a is not None:                   # hidden states [L, B*N, E], selected as the time-major [L, B, N, E]
            L, E = self.h0_a.shape[0], self.h0_a.shape[-1]
            mb.t0 = self.t0
            mb.h0_a, mb.h0_c = (tm(h.view(L, self.B, self.N, E)).view(L, -1, E) for h in (self.h0_a, self.h0_c))
            mb.prefix_a, mb.prefix_c = opt(self.prefix_a), opt(self.prefix_c)
        if self.replay is not None:
            mb.replay, mb.map_id = self.replay, em(self.map_id)
            self.replay.regenerate(mb)
        return mb

    def pieces(self):
        """A batch that crossed an episode boundary at step k as two ordinary batches sharing its slabs: steps [0, k) (the segment's
        start state, the ended episode's maps, bootstrapped with v_boot) and steps [k, T) (an episode start on the new maps)."""
        k, D = self.boundary, self.depth
        first = lambda x, n=k: None if x is None else x[:n]     # noqa: E731
        last = lambda x: None if x is None else x[k:]           # noqa: E731
        keys = ("p", "e", "p_adj_bits", "e_adj", "o_adj_bits", "a", "logp", "r", "active")
        common = lambda f: {n: f(getattr(self, n)) for n in keys}     # noqa: E731
        one = TrainBatch(**common(first), oxy=self.oxy, o_count_train=self.o_count_train, hist_a=first(self.hist_a, k + D),
                         hist_c=first(self.hist_c, k + D), v=torch.cat([self.v[:k], self.v_boot.unsqueeze(0)]), depth=D, t0=self.t0,
                         h0_a=self.h0_a, h0_c=self.h0_c, prefix_a=self.prefix_a, prefix_c=self.prefix_c, replay=self.replay,
                         map_id=self.map_id)
        two = TrainBatch(**common(last), oxy=self.oxy2, o_count_train=self.o_count_train2, hist_a=last(self.hist_a),
                         hist_c=last(self.hist_c), v=self.v[k:], depth=D, replay=self.replay2, map_id=self.map_id2,
                         zero_prefix=self.hist_a is not None)
        return one, two

    def minibatch(self, lo, hi):
        """Envs [lo, hi): contiguous copies of the slabs (the reference's sequential `batch[key][index]`)."""
        return self._select(lambda x: x[:, lo:hi].contiguous(), lambda x: x[lo:hi].contiguous())

    def minibatch_indexed(self, index):
        """Envs `index` (int64 device tensor, any order): the reference's `batch[key][index]` (:665-679) for an arbitrary index list,
        every slab gathered by `marl_gather_rows` (one launch per tensor: row = one env at one step, source row t*B + index[b])."""
        T, B = self.T, self.B
        index = index.to(torch.int64).contiguous()
        mb = index.numel()
        rows = {}

        def g(x, lead_t=True):
            x = x.contiguous()
            Tx = x.shape[0] if lead_t else 1
            if Tx not in rows:          # source row of (t, b) in the [Tx*B, row] view of a time-major slab
                rows[Tx] = ((torch.arange(Tx, device=x.device, dtype=torch.int64) * B).unsqueeze(1) + index.unsqueeze(0)).reshape(-1).contiguous()
            idx = rows[Tx]
            tail = tuple(x.shape[2:]) if lead_t else tuple(x.shape[1:])
            out = torch.empty(((Tx, mb) if lead_t else (mb,)) + tail, dtype=x.dtype, device=x.device)
            row_bytes = (x.numel() // (Tx * B)) * x.element_size()
            _lib.check(_lib.lib().marl_gather_rows(x.data_ptr(), out.data_ptr(), idx.data_ptr(), idx.numel(), row_bytes, Tx * B,
                                                   _lib.stream_ptr()), "marl_gather_rows")
            return out

        return self._select(g, lambda x: g(x, False)), g

    def graph(self):
        T, B, N = self.T, self.B, self.N
        o_index = torch.arange(B, dtype=torch.int32, device=self.p.device).repeat(T)
        return ops.GraphBatch(self.p.view(T * B, N, 4), self.e.view(T * B, 4), self.oxy, o_index, self.o_count_train,
                              self.p_adj_bits.view(T * B, N, -1), self.e_adj.view(T * B, N),
                              self.o_adj_bits.view(T * B, N, -1))

    def history(self, which):
        """EmbeddingDataset2 (:95-113): k-th history = slabs [D-1-k, D-1-k+T) of the [T+D,B,N,E] arena — addressed in
        place through strides, no copy."""
        h = self.hist_a if which == "actor" else self.hist_c
        D, T, B, N = self.depth, self.T, self.B, self.N
        E = h.shape[-1]
        return [(h[D - 1 - k:], N * E, E) for k in range(D)]


class HistoryReplay:
    """What regenerating a rollout's history embeddings needs, carried by a replay-mode TrainBatch: the rollout-time weights (a
    snapshot FusedRolloutStep, so the batch stays valid after `update()` steps the optimizer), the per-map boundary cells (i32) with the
    rollout's REAL cell counts, and the aliasing rule.  The per-env inputs - fp32 states, packed adjacency, actions, map ids - are the
    minibatch's own slabs.  The fused step's per-row output does not depend on how the batch is split into launches, and the arena
    records are (float) of the fp64 states the rollout's step converted, so the regenerated history is the stored one bit for bit."""

    def __init__(self, fused, oxy_i32, o_count, quirks, t0=0):
        self.fused, self.oxy_i32, self.o_count, self.quirks, self.t0 = fused, oxy_i32, o_count, bool(quirks), int(t0)

    def regenerate(self, mb, embed_only=None):
        """Fills mb.hist_a / mb.hist_c [T+D, mb, N, E] with T fused steps on the current stream (forced actions, history read from the
        tensors being filled; a segment's slabs 0..D-1 are its history prefix).  embed_only (default REPLAY_EMBED_ONLY) False runs the
        full step from the batch's start hidden states and returns the replayed (log-prob, value) [T, mb, N] - the same numbers the
        rollout stored."""
        embed_only = REPLAY_EMBED_ONLY if embed_only is None else embed_only
        T, B, N, D, E, t0 = mb.T, mb.B, mb.N, mb.depth, self.fused.E, self.t0
        f32 = dict(dtype=torch.float32, device=mb.p.device)
        mb.hist_a, mb.hist_c = torch.zeros(T + D, B, N, E, **f32), torch.zeros(T + D, B, N, E, **f32)
        if mb.prefix_a is not None:
            mb.hist_a[:D].copy_(mb.prefix_a)
            mb.hist_c[:D].copy_(mb.prefix_c)
        flags = fused_policy.STATE_F32 | (fused_policy.EMBED_ONLY if embed_only else 0)
        ha = hc = act = logp = v = None
        if not embed_only:
            if mb.h0_a is None:
                ha, hc = torch.zeros(2, B * N, E, **f32), torch.zeros(2, B * N, E, **f32)
            else:
                ha, hc = mb.h0_a.clone(), mb.h0_c.clone()
            act = mb.a.to(torch.int32)
            logp, v = torch.empty(T, B, N, **f32), torch.empty(T, B, N, **f32)
        view = SimpleNamespace(B=B, N=N, O=self.oxy_i32.shape[1], map_id=mb.map_id)
        ident = lambda i: i      # noqa: E731
        for t in range(T):
            view.p_state, view.e_state = mb.p[t], mb.e[t]
            view.p_adj_bits, view.e_adj, view.o_adj_bits = mb.p_adj_bits[t], mb.e_adj[t], mb.o_adj_bits[t]
            h_a = _history_inputs(mb.hist_a, mb.hist_c, t, D, self.quirks, "actor", ident, t0=t0)
            h_c = _history_inputs(mb.hist_a, mb.hist_c, t, D, self.quirks, "critic", ident, t0=t0)
            self.fused.step(view, self.oxy_i32, self.o_count, t0 + t, 0, True, h_a, h_c, mb.hist_a[t + D], mb.hist_c[t + D], ha, hc,
                            None if act is None else act[t], None if logp is None else logp[t], None if v is None else v[t],
                            force_action=True, flags=flags)
        return None if embed_only else (logp, v)


class RolloutGraph:
    """`MAPPO.rollout_batched` for all envs of an engine (networks in the loop) captured as ONE CUDA graph: the fused schedule of
    G env-group pipelines, per env step and group observe -> fused policy step (encoder + GRU + heads of both networks, one launch)
    || A* replan when due -> fused evader-move / step / reward-norm / store kernel; no host involvement on replay.  The engine state
    the episode starts from is whatever the engine holds at replay time.  With `carry` (a RolloutCarry whose tensors stay put: the
    graph reads them on every replay) the graph is one segment of T steps starting at the episode's step carry.t0.
    policy_dbg: an instrumented capture for measurements, not for production replays - an int64 tensor [T, G, >= CTAs per launch,
    16] that every policy launch of the G pipelines writes its per-CTA record to (see MAPPO.rollout_batched)."""

    def __init__(self, mappo, engine, arena, T, seed, policy_dbg=None, history=None, carry=None):
        snap = engine.snapshot()
        kw = {} if policy_dbg is None else dict(policy_dbg=policy_dbg, pipelines=policy_dbg.shape[1])
        # decided once: the warm-up's allocations would otherwise change the free memory the captured rollout sees
        kw["history"] = history or mappo.history_mode(T, engine.B, engine.N)
        kw["carry"] = self.carry = carry
        mappo.rollout_batched(engine, arena, T, seed=seed, history=kw["history"], carry=carry)   # eager warm-up (kernel attributes, stream pool)
        torch.cuda.synchronize()
        engine.restore(snap)
        self.graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        c0 = _lib.CALLS
        with torch.cuda.stream(side):
            with torch.cuda.graph(self.graph, stream=side):
                self.batch = mappo.rollout_batched(engine, arena, T, seed=seed, **kw)
        self.our_launches = _lib.CALLS - c0                           # C-ABI calls (>= 1 of our kernels each) per replay
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        engine.restore(snap)

    def replay(self):
        self.graph.replay()


class AutoResetStream:
    """The CUDA graphs of one auto-reset segment stream of `explore_batched`: one graph per segment start t0 (a stream of S-step
    segments visits T_ep / gcd(S, T_ep) of them), all sharing the stream's memory.

    * Inputs: one RolloutCarry (the segment's start state, copied in before each replay) and one int64 [3] seed word (sample_seed(e),
      reset_seed(e + 1), sample_seed(e + 1), filled from the host before each replay).  The policy launches and the reset read the seeds
      through the device-seeded entry points, so a graph is not tied to the episode it was captured in.
    * Outputs: the batch's S-sized slabs (history or ring, values, log-probs, actions) and the next carry, owned by the stream, not by a
      graph.  Everything else a graph allocates comes from one memory pool shared by the stream's graphs, which is safe because a
      stream's replays never overlap.  So a batch is valid until the next call of the same stream, whatever that call's start is.
    * Capture: an eager warm-up of the segment (kernel attributes, stream pool), then the engine is put back from device clones of
      every tensor it keeps across episodes (BatchedPursuitEnv._STATE and reset_fail; the warm-up may have reset the maps) and the
      critic's spectral-norm vectors, then the capture."""

    def __init__(self, mappo, engine, arena, S, tape_len, history):
        B, N, E, D, L = engine.B, engine.N, mappo.embedding_dim, mappo.depth, mappo.num_layers
        f32 = dict(dtype=torch.float32, device=mappo.device)
        self.engine, self.arena = engine, arena      # the stream is keyed by their ids: keeping them alive keeps the ids unique
        self.S, self.history = S, history or mappo.history_mode(S, B, N)
        rows = D + 1 if self.history == "replay" else S + D
        self.carry = RolloutCarry.zeros(mappo, B, N)
        self.seeds = torch.zeros(3, dtype=torch.int64, device=mappo.device)
        self.out = SimpleNamespace(hist_a=torch.zeros(rows, B, N, E, **f32), hist_c=torch.zeros(rows, B, N, E, **f32),
                                   v=torch.zeros(S + 1, B, N, **f32), logp=torch.zeros(S, B, N, **f32),
                                   act=torch.zeros(S, B, N, dtype=torch.int32, device=mappo.device),
                                   carry=RolloutCarry.zeros(mappo, B, N))
        self.pool = torch.cuda.graph_pool_handle()
        self.graphs = {}                # t0 -> (CUDAGraph, TrainBatch, next (t0, episode increment))
        self.tape_ptr = engine.target_tape.data_ptr()

    def capture(self, mappo, engine, arena, t0, auto_reset):
        carry = RolloutCarry(t0, self.carry.ha, self.carry.hc, self.carry.emb_a, self.carry.emb_c)
        kw = dict(history=self.history, carry=carry, auto_reset=auto_reset, out=self.out, device_seeds=self.seeds)
        engine._reset_buffers()
        names = engine._STATE + ("reset_fail",)
        saved = {n: getattr(engine, n).clone() for n in names}
        cm = mappo.critic.Mean
        sn = (cm.weight_u.clone(), cm.weight_v.clone()) if mappo.sn else None
        mappo.rollout_batched(engine, arena, self.S, **kw)        # eager warm-up
        torch.cuda.synchronize()
        for n in names:
            getattr(engine, n).copy_(saved[n])
        if sn is not None:
            cm.weight_u.copy_(sn[0])
            cm.weight_v.copy_(sn[1])
        del saved
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side, pool=self.pool):
                batch = mappo.rollout_batched(engine, arena, self.S, **kw)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        nxt = (batch.carry.t0, 0 if batch.ended_collision is None else 1)
        self.graphs[t0] = (graph, batch, nxt)
        return self.graphs[t0]


class MAPPO:
    def __init__(self, cfg, batch_size, mini_batch_size, agent_type, reference_quirks=None):
        """reference_quirks (default True, or `cfg.algo.reference_quirks`): keep the two reference behaviours that make its rollout
        forward differ from its training forward at identical weights (SURVEY 7.4-5) - the history list that actor and critic
        alias during the rollout, and the critic's all-ones obstacle adjacency spanning the padded slots in training.  False is the
        self-consistent variant: per-network histories in the rollout, the map's real boundary cells in training (PPO ratios are then
        1 on the first epoch); never the parity default."""
        a = cfg.algo
        self.reference_quirks = bool(getattr(a, "reference_quirks", True)) if reference_quirks is None else bool(reference_quirks)
        self.batch_size, self.mini_batch_size = batch_size, mini_batch_size
        self.max_train_steps, self.lr, self.gamma, self.lamda = a.max_train_steps, a.lr, a.gamma, a.lamda
        self.epsilon, self.K_epochs, self.entropy_coef = a.epsilon, a.epochs, a.entropy_coef
        self.use_grad_clip, self.use_lr_decay = a.use_grad_clip, a.use_lr_decay
        self.use_adv_norm, self.use_value_clip = a.use_adv_norm, a.use_value_clip
        self.action_dim, self.input_dim = cfg.env.action_dim, cfg.env.state_dim
        self.num_layers, self.embedding_dim = a.num_layers, a.embedding_dim
        self.rnn_input_dim, self.rnn_hidden_dim = a.embedding_dim, a.rnn_hidden_dim
        self.sn = a.use_spectral_norm
        key = "learner_device" if "Learner" in agent_type else ("worker_device" if "Worker" in agent_type else "evaluator_device")
        self.device = torch.device(getattr(a, key))
        if self.device.type != "cuda":
            raise _lib.MarlError(f"algo.{key}={self.device}: this engine runs on CUDA only (no CPU fallback)")
        if a.use_reward_norm:
            self.reward_norm = Normalization(shape=cfg.env.num_defender, device=self.device)
        encoder = DHGN(self.input_dim, self.embedding_dim, self.sn, a, self.device)
        self.depth = a.depth
        self.actor = SharedActor(encoder, self.rnn_input_dim, self.action_dim, self.num_layers, self.rnn_hidden_dim, self.sn)
        self.critic = SharedCritic(encoder, self.rnn_input_dim, 1, self.num_layers, self.rnn_hidden_dim, self.sn)
        self.actor, self.critic = self.actor.to(self.device), self.critic.to(self.device)
        self.ac_parameters = (list(self.actor.shared_net.parameters()) + list(self.actor.GRU.parameters()) +
                              list(self.critic.GRU.parameters()) + list(self.critic.Mean.parameters()) +
                              list(self.actor.Mean.parameters()))
        self.ac_optimizer = _FlatAdam(self.ac_parameters, lr=self.lr, eps=1e-5)
        self.minibuffer, self.total_step, self.cfg = None, 0, cfg
        self.last_train_stats = None     # TrainStats of the last train(stats=True)

    # ------------------------------------------------------------------------------------------------ training
    def _forward_losses(self, mb, adv, v_target, side=None):
        T, B, N, E = mb.T, mb.B, mb.N, self.embedding_dim
        if mb.parts is None:
            feat_a, feat_c = self._features(mb, side)
        else:                           # a segment that crossed an episode boundary: the GRU and the history restart with each piece
            feats = [self._features(part, side) for part in mb.parts]
            feat_a, feat_c = (torch.cat([f[i] for f in feats]) for i in (0, 1))
        cm = self.critic.Mean
        R = T * B * N
        flat = lambda x: x.reshape(R)
        la, lc, logp, ent, val, u2, v2 = ops.ppo_head(
            feat_a.reshape(R, E), feat_c.reshape(R, E), self.actor.Mean.weight, self.actor.Mean.bias,
            cm.weight_orig if self.sn else cm.weight, cm.bias, cm.weight_u if self.sn else torch.ones(1, device=self.device),
            flat(mb.a), flat(mb.logp), flat(adv), flat(mb.v[:-1]) if self.use_value_clip else None, flat(v_target), flat(mb.active), self.epsilon,
            self.entropy_coef)
        if self.sn:
            with torch.no_grad():
                cm.weight_u.copy_(u2)
                cm.weight_v.copy_(v2)
        return la, lc, logp.view(T, B, N), ent.view(T, B, N), val.view(T, B, N)

    def _features(self, mb, side=None):
        """The GRU outputs [T, B*N, E] of the actor and the critic over a minibatch's steps, from its start state."""
        T, B, N, E = mb.T, mb.B, mb.N, self.embedding_dim
        graph = mb.graph()
        enc = self.actor.shared_net
        if mb.h0_a is None:             # a whole episode starts from zero hidden states
            h0_a = h0_c = torch.zeros(self.num_layers, B * N, E, dtype=torch.float32, device=self.device)
        else:                           # a segment from the hidden states the rollout carried into it
            h0_a, h0_c = mb.h0_a, mb.h0_c
        # The two networks are independent until the loss: the critic branch runs on a side stream, concurrently with the actor
        # branch (forward here, and backward too: autograd replays each node on the stream of its forward).  The GRU sequence
        # kernels of a minibatch only fill 50-100 of the 148 SMs, so the pair overlaps almost perfectly.
        main = torch.cuda.current_stream()
        if TWO_STREAM_TRAIN and not torch.cuda.is_current_stream_capturing():
            if side is None:
                if getattr(self, "_critic_stream", None) is None:
                    self._critic_stream = torch.cuda.Stream(device=self.device)
                side = self._critic_stream
            side.wait_stream(main)
            with torch.cuda.stream(side):
                emb_c = enc.encode(graph, True, mb.history("critic"))
                feat_c, _ = self.critic.features(emb_c.view(T, B * N, E), h0_c)
            emb_a = enc.encode(graph, False, mb.history("actor"))
            feat_a, _ = self.actor.features(emb_a.view(T, B * N, E), h0_a)
            main.wait_stream(side)
            feat_c.record_stream(main)
        else:
            emb_a = enc.encode(graph, False, mb.history("actor"))
            feat_a, _ = self.actor.features(emb_a.view(T, B * N, E), h0_a)
            emb_c = enc.encode(graph, True, mb.history("critic"))
            feat_c, _ = self.critic.features(emb_c.view(T, B * N, E), h0_c)
        return feat_a, feat_c

    def gae(self, tb):
        """GAE + advantage normalisation on a time-major TrainBatch (kernel 3b; marl_gae_boundary for a batch that crossed an
        episode boundary)."""
        L = _lib.lib()
        import ctypes
        T, B, N = tb.T, tb.B, tb.N
        adv, vt = torch.empty_like(tb.r), torch.empty_like(tb.r)
        ws = torch.zeros(int(L.marl_gae_workspace_bytes(B, T, N)), dtype=torch.uint8, device=tb.r.device)
        if tb.boundary is not None:     # a segment that crossed an episode boundary: the recursion restarts there
            _lib.check(L.marl_gae_boundary(B, T, N, int(tb.boundary), _lib.ptr(tb.r), _lib.ptr(tb.v), _lib.ptr(tb.v_boot),
                                           _lib.ptr(tb.active), ctypes.c_float(self.gamma), ctypes.c_float(self.gamma * self.lamda),
                                           1 if self.use_adv_norm else 0, _lib.ptr(adv), _lib.ptr(vt), _lib.ptr(ws), _lib.stream_ptr()),
                       "marl_gae_boundary")
            return adv, vt
        _lib.check(L.marl_gae(B, T, N, _lib.ptr(tb.r), _lib.ptr(tb.v), _lib.ptr(tb.active), 1, ctypes.c_float(self.gamma),
                              ctypes.c_float(self.gamma * self.lamda), 1 if self.use_adv_norm else 0, _lib.ptr(adv),
                              _lib.ptr(vt), _lib.ptr(ws), _lib.stream_ptr()), "marl_gae")
        return adv, vt

    def train(self, replay_buffer, total_steps, return_numpy=True, trace=None, allreduce=None, mean=False, shuffle=None,
              shuffle_seed=None, permutation=None, stats=False):
        """MAPPO.train (:638-723): GAE, then for each sequential minibatch forward / PPO losses / backward with gradients
        accumulating and the global-norm clip applied to the running accumulation; no optimizer step here.

        allreduce: None (default, the reference's protocol: the accumulated gradients are summed across replicas once per update,
        in `update()` - main.py:121-129) or "minibatch" (north star: ONE all-reduce per PPO minibatch - every minibatch's gradient
        is summed over the replicas (`mean=True`: averaged) before it enters the running, clipped accumulation, so the clip acts on
        the global gradient and all replicas leave `train` with identical gradients; `update()` then only steps).
        shuffle (default `cfg.algo.shuffle_minibatches`, false = the reference's SequentialSampler :665): minibatches are drawn from a
        device permutation of the envs (seeded by `shuffle_seed`, or given as `permutation`) and gathered by `marl_gather_rows`.
        stats=True: PPO diagnostics of the update (entropy, KL, clip fractions, explained variance, gradient norms) are reduced on the
        device - one `marl_ppo_stats` row per minibatch, on that minibatch's stream, then one `marl_ppo_stats_combine` - and left in
        `self.last_train_stats` (a TrainStats; this replica's rows: `allreduce_()` makes them global).  Training is unchanged, and the
        return value too."""
        if allreduce not in (None, "update", "minibatch"):
            raise ValueError(f"allreduce={allreduce!r}: None / 'update' (one all-reduce per update) or 'minibatch'")
        per_mb = allreduce == "minibatch"
        t_issue = time.perf_counter()
        if shuffle is None:
            shuffle = bool(getattr(self.cfg.algo, "shuffle_minibatches", False)) or permutation is not None
        data = replay_buffer.get_training_data(self.device) if hasattr(replay_buffer, "get_training_data") else replay_buffer
        tb = data if isinstance(data, TrainBatch) else TrainBatch.from_reference(data, self.depth)
        adv, v_target = self.gae(tb)
        if trace is not None:
            trace["adv"], trace["v_target"] = adv, v_target
        self.ac_optimizer.zero_grad()
        B = tb.B
        bs = self.batch_size or B
        mbs = self.mini_batch_size or bs
        # The weights are fixed for the whole epoch, so the minibatches are independent except for the ORDER in which their
        # gradients enter the running, clipped accumulation (:708-711).  Their forward/backward passes therefore run concurrently
        # (CONCURRENT_MINIBATCHES in flight, each with its own actor / critic stream pair, gradients into per-minibatch arenas),
        # and the accumulate-then-clip sequence is replayed afterwards in minibatch order — same result, ~4x the kernels in flight
        # for the launch-latency-bound GRU sequence kernels.
        starts = list(range(0, bs, mbs))
        n_mb = len(starts)
        perm = None
        if shuffle:
            if permutation is not None:
                perm = torch.as_tensor(permutation, dtype=torch.int64, device=self.device)
                if perm.numel() != bs or not torch.equal(torch.sort(perm).values, torch.arange(bs, device=self.device)):
                    raise ValueError("permutation must be a permutation of range(batch_size)")
            else:
                gen = torch.Generator(device=self.device)
                gen.manual_seed(int(total_steps) if shuffle_seed is None else int(shuffle_seed))
                perm = torch.randperm(bs, device=self.device, generator=gen)
            if trace is not None:
                trace["permutation"] = perm.clone()
        flat = self.ac_optimizer.flat_grad
        views = self.ac_optimizer._views
        gbuf = torch.zeros(n_mb, flat.numel(), dtype=torch.float32, device=self.device)
        losses = torch.zeros(n_mb, 2, dtype=torch.float32, device=self.device)
        if stats:       # row m belongs to minibatch m alone, so the result does not depend on which minibatch finishes first
            mb_sums = torch.empty(n_mb, ops.PPO_STATS_SUMS, dtype=torch.float64, device=self.device)
            norms = torch.empty(n_mb, dtype=torch.float32, device=self.device) if self.use_grad_clip else None
        main = torch.cuda.current_stream()
        P = max(1, min(CONCURRENT_MINIBATCHES, n_mb))
        if getattr(self, "_mb_streams", None) is None or len(self._mb_streams) < P:
            self._mb_streams = [(torch.cuda.Stream(device=self.device), torch.cuda.Stream(device=self.device)) for _ in range(P)]
        with torch.enable_grad(), ops.pack_scope():       # weights are fixed for the whole epoch: pack them once (per stream)
            for m, lo in enumerate(starts):
                hi = min(lo + mbs, bs)
                st, side = self._mb_streams[m % P]
                st.wait_stream(main)
                with torch.cuda.stream(st):
                    if perm is None:
                        mb = tb.minibatch(lo, hi)
                        adv_mb, vt_mb = adv[:, lo:hi].contiguous(), v_target[:, lo:hi].contiguous()
                    else:
                        mb, gather = tb.minibatch_indexed(perm[lo:hi])
                        adv_mb, vt_mb = gather(adv), gather(v_target)
                    la, lc, logp, ent, val = self._forward_losses(mb, adv_mb, vt_mb, side=side)
                    grads = torch.autograd.grad(la + lc, self.ac_parameters, allow_unused=True)
                    for g, (off, k) in zip(grads, views):
                        if g is not None:
                            gbuf[m, off:off + k].copy_(g.reshape(-1))
                    losses[m, 0], losses[m, 1] = la.detach(), lc.detach()
                    if stats:
                        ops.ppo_stats(logp, mb.logp, ent, val, mb.v[:-1] if self.use_value_clip else None, vt_mb, mb.active,
                                      self.epsilon, out=mb_sums[m])
                    if trace is not None:
                        trace.setdefault("mb", []).append(dict(logp=logp.detach(), ent=ent.detach(), val=val.detach()))
                    del grads, la, lc, logp, ent, val, mb
            for st, _ in self._mb_streams[:P]:
                main.wait_stream(st)
            if trace is not None:
                trace["mb_grads"] = gbuf.clone()            # this replica's per-minibatch gradients, before any reduction
            for m in range(n_mb):                           # gradients accumulate; clip_grad_norm_ acts on the running sum
                if per_mb:                                  # one all-reduce per PPO minibatch: the clip then sees the global gradient
                    from . import parallel
                    parallel.allreduce_sum_(gbuf[m], mean=mean)
                flat.add_(gbuf[m])
                if self.use_grad_clip:
                    norm = ops.clip_grad_norm_(flat, 5.0, out=norms[m:m + 1] if stats else None)
                    if trace is not None:
                        trace.setdefault("grad_norms", []).append(norm.clone())
            if stats:
                stats_sums = ops.ppo_stats_combine(mb_sums, norms, 5.0)
        self.ac_optimizer._sync_grads()
        self._grads_reduced = per_mb
        self.last_train_issue_s = time.perf_counter() - t_issue     # host time to ISSUE the epoch (the device may still be running)
        lh = losses.cpu()
        if stats:
            self.last_train_stats = TrainStats.from_sums(stats_sums, self.epsilon, 5.0 if self.use_grad_clip else None)
        if trace is not None:
            for m, rec in enumerate(trace["mb"]):
                rec["actor_loss"], rec["critic_loss"] = float(lh[m, 0]), float(lh[m, 1])
        obj_a, obj_c, n_updates = float(lh[:, 0].sum()), float(lh[:, 1].sum()), n_mb
        if self.use_lr_decay:
            self.lr_decay(total_steps)
        if return_numpy:
            return obj_c / n_updates, obj_a / n_updates, self.actor.get_gradients(), self.critic.get_gradients()
        return obj_c / n_updates, obj_a / n_updates, None, None

    # ------------------------------------------------------------------------------------------------ data parallel
    def sync_weights(self, src=0):
        """All replicas start from rank `src`'s weights (main.py:73-75) — one broadcast of the flat parameter arena."""
        from . import parallel
        parallel.broadcast_(self.ac_optimizer.flat_param, src)
        if self.sn:
            parallel.broadcast_(self.critic.Mean.weight_u, src)
            parallel.broadcast_(self.critic.Mean.weight_v, src)

    def update(self, total_steps, mean=False):
        """Learner.set_gradients_and_update across replicas (main.py:121-129, runner.py:72-78): ONE all-reduce (SUM) of
        the flat gradient arena over NCCL, then the same fused Adam step on every replica."""
        from . import parallel
        if not getattr(self, "_grads_reduced", False):    # train(allreduce="minibatch") already reduced every minibatch's gradient
            parallel.allreduce_sum_(self.ac_optimizer.flat_grad, mean=mean)
        self._grads_reduced = False
        self.ac_optimizer.step()
        if self.use_lr_decay:
            self.lr_decay(total_steps)

    def lr_decay(self, total_steps):
        lr_now = self.lr * (1 - total_steps / self.max_train_steps)
        for p in self.ac_optimizer.param_groups:
            p["lr"] = lr_now
        self.total_step = total_steps

    def save_model(self, cwd):
        torch.save(self.actor.state_dict(), cwd + "actor.pth")
        torch.save(self.critic.state_dict(), cwd + "critic.pth")

    # ------------------------------------------------------------------------------------------------ rollout
    def history_mode(self, T, B, N):
        """'store' when the full history of both networks fits STORE_HISTORY_SHARE of the free device memory, else 'replay'."""
        free = torch.cuda.mem_get_info(self.device)[0] + torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)
        return "store" if history_bytes(T, B, N, self.embedding_dim, self.depth) <= STORE_HISTORY_SHARE * free else "replay"

    @torch.no_grad()
    def rollout_batched(self, engine, arena, T=None, seed=0, deterministic=False, use_fused=None, timers=None, pipelines=None,
                        actor_only=False, history=None, carry=None, policy_dbg=None, auto_reset=None, out=None, device_seeds=None):
        """MAPPO.run_episode (:742-827) for all B envs of a BatchedPursuitEnv at once, entirely on the GPU.
        Per step: observe kernel -> fused encoder (actor, then critic with all-ones adjacency) -> GRU cell -> heads ->
        closed-loop env kernel (evader move + pursuer step + reward-norm + store).  Fills `arena` plus the history /
        value / log-prob slabs and returns a TrainBatch ready for `train`.

        With the fused policy step (use_fused; default: whenever the networks' shape has one) the envs are cut into G contiguous
        env-group pipelines, each stepping through the episode on its own stream: observe -> ONE policy launch for both networks ->
        env step, with the A* replan due every `difficulty` steps on the group's side stream beside the policy launch (it needs the
        env state, not the action) and joined before the env step.  One group's small kernels and the long tail of its replanning
        (the slowest of its searches gates its env step) then overlap with the other groups' policy kernels instead of idling the
        GPU.  Results are the same for any G (the envs are independent and the sampling RNG is keyed by the global row).  G is 1 for
        actor_only, else `pipelines`, else 1 with `timers`, else MARL_PIPELINES or `default_pipelines(B, N)`.  Without the fused
        step (network shapes it does not cover) the unfused kernels run one after another on the current stream.

        timers: dict name -> list of (start, end) CUDA events around every launch of the T steps (env_observe_kernel,
        policy_step_kernel, evader_kernel(replan), rollout_kernel(closed)); the replan then runs on the group's own stream, after the
        policy launch.  The bootstrap step is not timed.  policy_dbg: int64 [T, G, >= CTAs per launch, 16]; every policy launch of
        the T steps writes its per-CTA record there (slots 13 / 14 = %globaltimer at CTA start / end in ns, 15 = SM id;
        csrc/policy_fused.cu) - usable under CUDA-graph capture, which is how bench.py times the kernel inside the schedule.

        actor_only=True is the EVALUATOR's episode (evaluator.py:118-156): no critic, and the actor's history is its OWN
        embeddings A(t-1), A(t-2), ... (its dataset is not aliased with a critic's there); values / bootstrap stay zero.

        history: 'store' keeps the full [T+D,B,N,E] history of both networks in the batch; 'replay' keeps only a ring of D+1 slabs
        per network during the episode (step t reads at most D steps back) and returns a batch with hist_a = hist_c = None that
        regenerates each minibatch's history in training (HistoryReplay).  None chooses with `history_mode` (store when it fits
        comfortably).  Replay needs the fused step; actor_only rollouts always store.

        carry: None (a whole episode from the engine's state at step 0) or a RolloutCarry: one segment of T = S steps of an episode of
        cfg.env.max_steps steps (S divides it), starting at the episode's step carry.t0 from the carried hidden states and history.
        The history rule, the sampling RNG key and the A* replan schedule use the episode's step; the engine must be at carry.t0.
        The batch records its start state (t0, h0_a / h0_c, the history prefix) and its `carry` is where the next segment starts.

        auto_reset: None, or an AutoReset with a carry: the segment may be any 1 <= S <= cfg.env.max_steps steps from any step carry.t0 of
        episode carry.episode, and when the episode ends inside it (at the segment's step k) the rollout bootstraps that episode, resets
        the envs on the device and continues with the next episode (see AutoReset; the fused step only, seeds from the AutoReset).  A
        batch that crosses the boundary has `boundary` = k, `v_boot` [B,N] (the finished episode's bootstrap value) and the two episodes'
        map data, and trains as two pieces with their own start states (`TrainBatch.pieces`).  A segment that ends exactly at the
        episode's end resets at its end.  Whenever the envs were reset, `ended_collision` / `ended_evader_status` [B] keep the finished
        episode's flags that the reset clears, and the next carry starts episode carry.episode + 1.

        out / device_seeds (internal, for `explore_batched`'s auto-reset graphs): `out` is a SimpleNamespace of preallocated slabs
        (hist_a, hist_c, v, logp, act) and a RolloutCarry `carry` that the batch and its next carry are written into instead of fresh
        tensors; `device_seeds` an int64 [3] device tensor (sample_seed(e), reset_seed(e + 1), sample_seed(e + 1) as u64 bit patterns)
        that the policy launches and the reset read when they run, in place of the AutoReset's host seeds."""
        B, N, E, D, L = engine.B, engine.N, self.embedding_dim, self.depth, self.num_layers
        dev = self.device
        if auto_reset is not None:
            T = arena.T if T is None else int(T)
            fused_ok = use_fused is not False and fused_policy.supported(self)
            check_auto_reset(auto_reset, carry, T, int(self.cfg.env.max_steps), B, N, L, E, D, dev, actor_only, fused_ok, seed,
                             getattr(engine, "maps_set", False))
            if not torch.cuda.is_current_stream_capturing() and not bool((engine.time_step == carry.t0).all()):
                raise _lib.MarlError(f"rollout segment from step {carry.t0}: the engine's envs are at steps "
                                     f"{sorted(set(engine.time_step.tolist()))[:4]}")
            seed = auto_reset.sample_seed(carry.episode)
        elif carry is not None:
            T = arena.T if T is None else int(T)
            check_segment(carry, T, int(self.cfg.env.max_steps), B, N, L, E, D, dev, actor_only)
            if not torch.cuda.is_current_stream_capturing() and not bool((engine.time_step == carry.t0).all()):
                raise _lib.MarlError(f"rollout segment from step {carry.t0}: the engine's envs are at steps "
                                     f"{sorted(set(engine.time_step.tolist()))[:4]}")
        T = T or arena.T
        t0 = 0 if carry is None else carry.t0
        f32 = dict(dtype=torch.float32, device=dev)
        if use_fused is None:
            use_fused = fused_policy.supported(self)
        if history not in (None, "store", "replay"):
            raise ValueError(f"history={history!r}: None, 'store' or 'replay'")
        if actor_only:
            history = "store"
        elif history is None:
            history = self.history_mode(T, B, N)
        replay = history == "replay"
        if replay and not use_fused:
            raise _lib.MarlError(f"rollout_batched: the history of this rollout ({history_bytes(T, B, N, E, D) / 1e9:.1f} GB) is not "
                                 "stored, and regenerating it needs the fused policy step (embedding_dim = rnn_hidden_dim = 128, "
                                 "2 GRU layers, depth 1..3, 9 actions)")
        slot = (lambda i: i % (D + 1)) if replay else (lambda i: i)     # history step i -> index into hist_a / hist_c
        if out is None:
            hist_a, hist_c = (torch.zeros(D + 1 if replay else T + D, B, N, E, **f32) for _ in range(2))
            v = torch.zeros(T + 1, B, N, **f32)
            logp = torch.zeros(T, B, N, **f32)
            act = torch.zeros(T, B, N, dtype=torch.int32, device=dev)
        else:
            hist_a, hist_c, v, logp, act = (getattr(out, k).zero_() for k in ("hist_a", "hist_c", "v", "logp", "act"))
        if carry is None:
            ha, hc = torch.zeros(L, B * N, E, **f32), torch.zeros(L, B * N, E, **f32)
        else:                                   # history steps 0..D-1 (slot(i) = i in both modes) are the carried embeddings
            ha, hc = carry.ha.clone(), carry.hc.clone()
            hist_a[:D].copy_(carry.emb_a)
            hist_c[:D].copy_(carry.emb_c)
        oxy = engine.boundary_xy.to(torch.float32).contiguous()                 # [M,O,2]
        o_count = torch.clamp(engine.boundary_count, max=engine.O).contiguous()  # rollout: the O_b real cells

        if use_fused:
            # ONE launch per env step and group for both networks (csrc/policy_fused.cu); embeddings / values / log-probs / actions
            # land directly in their rollout slabs.  The critic's effective head row is constant while the weights are (one power
            # iteration on a [1,E] matrix is already converged), so it is computed once.  A replay-mode batch keeps the step (its own
            # copy of the weights) to regenerate the history in training.
            w, _ = self.critic.head_weight()
            fused = fused_policy.FusedRolloutStep(self, w.reshape(E).contiguous(), snapshot=replay)
            oxy_i = engine.boundary_xy.clone() if replay else engine.boundary_xy.contiguous()
            rep_ = HistoryReplay(fused, oxy_i, o_count, self.reference_quirks, t0) if replay else None
            G = (1 if actor_only else int(pipelines) if pipelines is not None else 1 if timers is not None
                 else int(os.environ.get("MARL_PIPELINES") or self.default_pipelines(B, N)))
            nxt, ended = self._rollout_fused(engine, arena, T, seed, deterministic, G, fused, oxy_i, o_count, hist_a, hist_c, ha, hc, act,
                                             logp, v, slot, carry, actor_only, timers, policy_dbg, auto_reset, oxy, replay,
                                             None if out is None else out.carry, device_seeds)
            return self._train_batch(engine, arena, T, oxy, hist_a, hist_c, v, logp, rep_, carry, nxt, ended)

        enc = self.actor.shared_net
        quirks = self.reference_quirks and not actor_only
        zeros_hist = torch.zeros(B, N, E, **f32)
        zeros_for_none = lambda hs: [zeros_hist if h is None else h for h in hs]     # noqa: E731
        observed = lambda: ops.GraphBatch(engine.p_state.to(torch.float32), engine.e_state.to(torch.float32), oxy,   # noqa: E731
                                          engine.map_id, o_count, engine.p_adj_bits, engine.e_adj, engine.o_adj_bits)
        for t in range(T):
            engine.observe()
            graph = observed()
            emb_a = enc.encode(graph, False, zeros_for_none(_history_inputs(hist_a, hist_c, t, D, quirks, "actor", slot, t0=t0)))
            feat_a, ha = self.actor.features(emb_a.view(1, B * N, E), ha)
            if actor_only:
                a_i, _, lp, _ = ops.act_head(feat_a[0], None, self.actor.Mean.weight, self.actor.Mean.bias, None, None, seed, t0 + t,
                                             deterministic)
                hist_a[t + D] = emb_a
            else:
                emb_c = enc.encode(graph, True, zeros_for_none(_history_inputs(hist_a, hist_c, t, D, quirks, "critic", slot, t0=t0)))
                feat_c, hc = self.critic.features(emb_c.view(1, B * N, E), hc)
                w, _ = self.critic.head_weight()
                a_i, _, lp, val = ops.act_head(feat_a[0], feat_c[0], self.actor.Mean.weight, self.actor.Mean.bias,
                                               w.reshape(E).contiguous(), self.critic.Mean.bias, seed, t0 + t, deterministic)
                hist_a[t + D], hist_c[t + D] = emb_a, emb_c
                v[t] = val.view(B, N)
            logp[t], act[t] = lp.view(B, N), a_i.view(B, N)
            engine.rollout_closed(arena, 1, t0=t, action_tape=act[t:t + 1], env_t0=t0 + t)
        if actor_only:
            return self._train_batch(engine, arena, T, oxy, hist_a, hist_c, v, logp)
        # bootstrap value of the final state (:806-825)
        engine.observe()
        graph = observed()
        nxt = None if carry is None else self._next_carry(carry, T, hist_a, hist_c, slot, ha, hc)
        emb_c = enc.encode(graph, True, zeros_for_none(_bootstrap_history(hist_a, hist_c, T, D, quirks, slot, t0=t0)))
        feat_c, _ = self.critic.features(emb_c.view(1, B * N, E), hc)
        w, _ = self.critic.head_weight()
        v[T] = torch.nn.functional.linear(feat_c[0], w, self.critic.Mean.bias).view(B, N)
        return self._train_batch(engine, arena, T, oxy, hist_a, hist_c, v, logp, None, carry, nxt)

    @staticmethod
    def default_pipelines(B, N):
        """Env-group pipelines of a batched rollout: one per 8192 (env, agent) rows, at most 8."""
        return max(1, min(8, (B * N) // 8192))

    def _rollout_fused(self, engine, arena, T, seed, deterministic, G, fused, oxy_i, o_count, hist_a, hist_c, h0_a, h0_c, act, logp, v,
                       slot, carry, actor_only, timers, policy_dbg, auto_reset=None, oxy=None, replay=False, out_carry=None, device_seeds=None):
        """The fused schedule of `rollout_batched`: G independent env-group pipelines, one stream (+ one A* side stream) each.  Each
        group starts from its rows of the hidden states h0_a / h0_c [L, B*N, E] (one group steps them in place).  Returns the
        RolloutCarry of the segment's end (None without a carry) and, when auto_reset reset the envs during the segment, a namespace of
        what the batch needs about the episode that ended (else None).  out_carry: the RolloutCarry the next carry is written into (else
        fresh tensors); device_seeds: see `rollout_batched`."""
        B, N, E, D, L = engine.B, engine.N, self.embedding_dim, self.depth, self.num_layers
        f32 = dict(dtype=torch.float32, device=self.device)
        quirks = self.reference_quirks and not actor_only
        nets = ("actor",) if actor_only else ("actor", "critic")
        t0 = 0 if carry is None else carry.t0
        T_ep = int(self.cfg.env.max_steps)
        # auto_reset: the episode ends after the segment's step k-1 when k = T_ep - t0 <= T; k < T crosses the boundary
        k = T_ep - t0 if auto_reset is not None and t0 + T >= T_ep else None
        # The bootstrap value v[T] is a critic-only step at the episode's end.  A segment that ends inside the episode computes it with
        # the step of both networks instead (the actor's outputs are discarded): that is the kernel the next segment's first step runs
        # on the same state, and the critic-only kernel rounds the GRU cell and the value sum differently, so v[T] is then bit for bit
        # the value the next segment starts with.
        pair_bootstrap = carry is not None and t0 + T < T_ep
        if len(getattr(engine, "_pipe_streams", [])) < 2 * G:
            engine._pipe_streams = [torch.cuda.Stream(device=self.device) for _ in range(2 * G)]
        rec_ptrs = arena.record_pointers()
        diff = int(engine.params.difficulty)
        # A lone launch takes the kernel's wave model (tile_rows 0: see policy_fused.cu); concurrent launches take full tiles and leave
        # SMs over for the neighbouring groups' kernels.
        tile = 0
        if G > 1:
            tile = int(os.environ.get("MARL_PIPE_TILE_ROWS") or ((128 // N) * N if N <= 128 else 0))     # (the knob: tools/)

        def timed(name, stream, fn):
            if timers is None:
                return fn()
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record(stream)
            fn()
            b_.record(stream)
            timers.setdefault(name, []).append((a_, b_))

        main = torch.cuda.current_stream()
        if out_carry is not None:
            next_ha, next_hc = out_carry.ha, out_carry.hc
        elif carry is not None:         # every group writes its rows of the next carry's hidden states
            next_ha, next_hc = torch.empty_like(carry.ha), torch.empty_like(carry.hc)
        dseed = (lambda i: None) if device_seeds is None else (lambda i: device_seeds[i:i + 1])     # noqa: E731

        def into(nc):
            return nc if out_carry is None else out_carry.copy_(nc)

        def pipelines(t_lo, t_hi, off, seed, oxy_i, o_count, v_end, pair, h0_a, h0_c, last, d_seed=None):
            """Segment steps [t_lo, t_hi) of one episode, at its steps t + off, then the bootstrap value after step t_hi - 1 into v_end;
            forked from and joined back into the current stream.  h0_a / h0_c: the hidden states at t_lo (None: zeros).  last: the
            piece that ends the segment (it writes the next carry's hidden states)."""
            fork = torch.cuda.Event()
            fork.record(main)
            for g in range(G):
                lo, hi = g * B // G, (g + 1) * B // G
                sl, rows = slice(lo, hi), slice(lo * N, hi * N)
                st, side = engine._pipe_streams[2 * g], engine._pipe_streams[2 * g + 1]
                st.wait_event(fork)
                with torch.cuda.stream(st):
                    # what FusedRolloutStep.step reads from an engine, for envs [lo, hi) (views: the kernels update them in place)
                    view = SimpleNamespace(B=hi - lo, N=N, O=engine.O, p_state=engine.p_state[sl], e_state=engine.e_state[sl],
                                           map_id=engine.map_id[sl], p_adj_bits=engine.p_adj_bits[sl], e_adj=engine.e_adj[sl],
                                           o_adj_bits=engine.o_adj_bits[sl])
                    if h0_a is None:
                        ha, hc = torch.zeros(L, (hi - lo) * N, E, **f32), torch.zeros(L, (hi - lo) * N, E, **f32)
                    else:
                        ha, hc = h0_a[:, rows].contiguous(), h0_c[:, rows].contiguous()

                    def hist_of(t, net):
                        return _history_inputs(hist_a, hist_c, t, D, quirks, net, slot, sl, t0=off)

                    for t in range(t_lo, t_hi):
                        replan, join = (off + t) % diff == 0, None
                        if replan and timers is None:
                            ev = torch.cuda.Event()
                            ev.record(st)
                            side.wait_event(ev)
                            engine.evader_replan(lo, hi, side)
                            join = torch.cuda.Event()
                            join.record(side)
                        timed("env_observe_kernel", st, lambda: engine.observe(lo=lo, hi=hi))
                        timed("policy_step_kernel", st, lambda: fused.step(
                            view, oxy_i, o_count, off + t, seed, deterministic, hist_of(t, "actor"), hist_of(t, "critic"),
                            hist_a[slot(t + D)][sl], hist_c[slot(t + D)][sl], ha, hc, act[t][sl], logp[t][sl], v[t][sl], nets=nets,
                            row_offset=lo * N, tile_rows=tile, debug=None if policy_dbg is None else policy_dbg[t, g], d_seed=d_seed))
                        if join is not None:
                            st.wait_event(join)
                        elif replan:
                            timed("evader_kernel(replan)", st, lambda: engine.evader_replan(lo, hi, st))
                        timed("rollout_kernel(closed)", st, lambda: engine._closed_chunk(arena, rec_ptrs, lo, hi, t, 1, act[t:t + 1], 0,
                                                                                          seed, st))
                    if not actor_only:
                        engine.observe(lo=lo, hi=hi)
                        h_fin = _bootstrap_history(hist_a, hist_c, t_hi, D, quirks, slot, sl, off)
                        scratch = torch.empty(hi - lo, N, E, **f32)
                        if carry is not None and last:  # before the bootstrap step, which updates the hidden states in place
                            next_ha[:, rows].copy_(ha)
                            next_hc[:, rows].copy_(hc)
                        if pair:
                            fused.step(view, oxy_i, o_count, off + t_hi, seed, deterministic, hist_of(t_hi, "actor"), h_fin,
                                       torch.empty_like(scratch), scratch, ha, hc, torch.empty_like(act[0][sl]),
                                       torch.empty_like(logp[0][sl]), v_end[sl], row_offset=lo * N, tile_rows=tile, d_seed=d_seed)
                        else:
                            fused.step(view, oxy_i, o_count, off + t_hi, seed, deterministic, h_fin, h_fin, scratch, scratch, ha, hc,
                                       None, None, v_end[sl], nets=("critic",), row_offset=lo * N, tile_rows=tile, d_seed=d_seed)
                    done = torch.cuda.Event()
                    done.record(st)
                main.wait_event(done)

        if k is None:
            pipelines(0, T, t0, seed, oxy_i, o_count, v[T], pair_bootstrap, h0_a, h0_c, True, dseed(0))
            if carry is not None:
                return into(self._next_carry(carry, T, hist_a, hist_c, slot, next_ha, next_hc)), None
            return None, None
        # auto-reset: episode e ends after step k-1.  Its pipelines end with the whole-episode rollout's critic-only bootstrap step.
        e = carry.episode
        v_boot = v[T] if k == T else torch.empty(B, N, **f32)
        pipelines(0, k, t0, seed, oxy_i, o_count, v_boot, False, h0_a, h0_c, k == T, dseed(0))
        # All groups are joined: the maps and their sensor tables are shared by envs of different groups, and the reset regenerates
        # them in place.  Keep what the reset clears or the batch's first piece still needs.
        oxy_env, o_count_train = self._train_map_data(engine, oxy)
        ended = SimpleNamespace(k=k, collision=engine.collision.clone(), evader_status=engine.evader_status.clone(), oxy=oxy_env,
                                o_count_train=o_count_train, map_id=engine.map_id.clone() if replay else None)
        reset_seed = auto_reset.reset_seed(e + 1) if device_seeds is None else dseed(1)
        engine.reset_device(seed=reset_seed, tape_len=auto_reset.tape_len, tape=auto_reset.tape, maps=auto_reset.maps)
        if k == T:
            return into(RolloutCarry.zeros(self, B, N, episode=e + 1)), ended
        ended.v_boot = v_boot
        oxy_i = engine.boundary_xy.clone() if replay else engine.boundary_xy.contiguous()
        o_count = torch.clamp(engine.boundary_count, max=engine.O).contiguous()
        ended.oxy_i, ended.o_count = oxy_i, o_count
        pipelines(k, T, -k, auto_reset.sample_seed(e + 1), oxy_i, o_count, v[T], True, None, None, True, dseed(2))
        return into(self._next_carry(carry, T, hist_a, hist_c, slot, next_ha, next_hc, start=k)), ended

    def explore_batched(self, engine, arena, T=None, seed=0, host_state=None, host_out=None, reset_reward_norm=False, history=None,
                        carry=None, auto_reset=None):
        """The batched counterpart of `explore_env` (:731-740) - the call a user makes once per training iteration: one whole
        episode of ALL envs of `engine` with both networks in the loop, replayed from a CUDA graph that is captured on the first
        call (per engine / arena / T / seed; the weight images are re-packed inside the graph, so it follows the optimizer).

        host_state: optional dict of HOST tensors (pinned for asynchronous copies) - `p_state` f64 [B,N,4], `e_state` f64 [B,4],
        `target` i32 [B,2] - copied to the device before the episode (`BatchedPursuitEnv.load_host_state`, which also clears the
        episode bookkeeping; `reset_reward_norm` additionally restarts the running reward statistics).
        host_out: optional dict of HOST tensors filled after the episode - `episode_reward` i64 [B] (sum of the raw rewards over
        pursuers and steps, the evaluator's return), `collision` u8 [B]; the call then synchronises the stream.
        history: as in `rollout_batched`, chosen when the graph is captured.
        Returns the TrainBatch of the episode (device resident, ready for `train`).  It lives in the graph's memory: it is valid until
        the next call with the same engine / arena / T / seed, which overwrites it - for a replay-mode batch this includes the weight
        snapshot its history is regenerated with (the graph re-packs it in place).

        carry: as in `rollout_batched` - one segment of T steps from carry.t0, usually the previous segment's `batch.carry` (or
        `RolloutCarry.zeros` at an episode's start).  One graph is captured per segment start; the carry is copied into that graph's
        own input buffers before the replay, so consecutive segments chain.  The engine must be at step carry.t0 (checked: one
        synchronisation), and host_state (an episode start) is only accepted with t0 = 0.

        auto_reset: an AutoReset with tape="device" (TypeError otherwise) and a carry: one auto-reset segment of T = S steps, with the
        semantics and the TrainBatch fields of `rollout_batched(carry=carry, auto_reset=auto_reset)` (boundary, v_boot, ended_*, the
        pieces, and `carry` with its episode index), replayed from a CUDA graph.  The stream of such calls with the same engine / arena
        / S / tape_len / history keeps one graph per segment start, its input buffers (carry, seeds), the batch's S-sized slabs and the
        next carry, and one memory pool for the graphs (`AutoResetStream`): the returned batch is valid until the next call of the same
        stream, whatever its start.  The seeds of the segment's episodes are written to a device word before the replay, so the graphs
        serve every episode.  The engine's target tape must have auto_reset.tape_len entries.  seed must be 0 (the seeds come from
        auto_reset), and host_state / host_out are not accepted: the stream resets itself, and the batch holds the per-episode data."""
        if auto_reset is not None:
            return MAPPO._explore_auto_reset(self, engine, arena, T, seed, host_state, host_out, history, carry, auto_reset)
        T = (T or arena.T) if carry is None else (arena.T if T is None else int(T))
        if carry is not None:
            check_segment(carry, T, int(self.cfg.env.max_steps), engine.B, engine.N, self.num_layers, self.embedding_dim,
                          self.depth, self.device)
            if host_state is not None and carry.t0 != 0:
                raise _lib.MarlError(f"explore_batched: host_state starts an episode, the carry continues one at step {carry.t0}")
        key = (id(engine), id(arena), int(T), int(seed)) + (() if carry is None else (carry.t0,))
        graphs = self.__dict__.setdefault("_episode_graphs", {})
        if host_state is not None:
            engine.load_host_state(reset_reward_norm=reset_reward_norm, **host_state)
        if carry is not None:
            at = engine.time_step.tolist()
            if any(s != carry.t0 for s in at):
                raise _lib.MarlError(f"explore_batched: segment from step {carry.t0}, the engine's envs are at steps {sorted(set(at))[:4]}")
        if key not in graphs:
            graphs[key] = RolloutGraph(self, engine, arena, T, seed, history=history,
                                       carry=None if carry is None else RolloutCarry.zeros(self, engine.B, engine.N, carry.t0))
        g = graphs[key]
        if carry is not None:
            g.carry.copy_(carry)
        g.replay()
        if host_out is not None:
            if "episode_reward" in host_out:
                host_out["episode_reward"].copy_(arena.raw_reward[:T].sum(dim=(0, 2), dtype=torch.int64), non_blocking=True)
            if "collision" in host_out:
                host_out["collision"].copy_(engine.collision, non_blocking=True)
            status = engine.evader_status.max()
            torch.cuda.current_stream().synchronize()
            if int(status):                                  # the evader's search overflowed or its target tape ran out: not an episode
                raise _lib.MarlError(f"explore_batched: evader status {int(status)} (A* OPEN / path overflow or target tape exhausted)")
        return g.batch

    def _explore_auto_reset(self, engine, arena, T, seed, host_state, host_out, history, carry, auto_reset):
        """explore_batched(auto_reset=...): every refusal before any CUDA call, then one replay of the stream's graph for carry.t0."""
        if not isinstance(auto_reset, AutoReset) or auto_reset.tape != "device":
            raise TypeError("explore_batched: auto_reset must be an AutoReset(..., tape='device'): the graph replays the reset, and the "
                            "torch tape's generator is not graph-safe")
        if seed != 0:
            raise _lib.MarlError(f"explore_batched: seed={seed} with auto_reset: the sampling seeds come from auto_reset.sample_seed")
        if carry is None:
            raise _lib.MarlError("explore_batched: auto_reset continues a stream of segments and needs a carry (RolloutCarry.zeros at the "
                                 "start)")
        if host_state is not None or host_out is not None:
            raise _lib.MarlError("explore_batched: host_state / host_out do not combine with auto_reset (the stream resets the envs "
                                 "itself; per-episode returns are in the batch)")
        S = arena.T if T is None else int(T)
        check_auto_reset(auto_reset, carry, S, int(self.cfg.env.max_steps), engine.B, engine.N, self.num_layers, self.embedding_dim,
                         self.depth, self.device, use_fused=fused_policy.supported(self), maps_set=getattr(engine, "maps_set", False))
        if engine._tape_len != auto_reset.tape_len or tuple(engine.target_tape.shape) != (engine.B, auto_reset.tape_len, 2):
            raise _lib.MarlError(f"explore_batched: the engine's target tape has {engine._tape_len} entries, auto_reset.tape_len is "
                                 f"{auto_reset.tape_len} (reset the envs with reset_device(..., tape_len={auto_reset.tape_len}))")
        at = engine.time_step.tolist()
        if any(x != carry.t0 for x in at):
            raise _lib.MarlError(f"explore_batched: segment from step {carry.t0}, the engine's envs are at steps {sorted(set(at))[:4]}")
        key = (id(engine), id(arena), S, auto_reset.tape_len, history, auto_reset.maps)
        streams = self.__dict__.setdefault("_auto_reset_streams", {})
        st = streams.get(key)
        if st is None:
            st = streams[key] = AutoResetStream(self, engine, arena, S, auto_reset.tape_len, history)
        if st.tape_ptr != engine.target_tape.data_ptr():    # the tape was reallocated: the graphs read the old one
            st.graphs.clear()
            st.tape_ptr = engine.target_tape.data_ptr()
        e = carry.episode
        st.seeds.copy_(torch.tensor([_lib.u64_bits(x) for x in (auto_reset.sample_seed(e), auto_reset.reset_seed(e + 1),
                                                                 auto_reset.sample_seed(e + 1))], dtype=torch.int64))
        st.carry.copy_(carry)
        graph, batch, (t_next, de) = st.graphs.get(carry.t0) or st.capture(self, engine, arena, carry.t0, auto_reset)
        graph.replay()
        batch.carry.t0, batch.carry.episode = t_next, e + de
        return batch

    def _next_carry(self, carry, T, hist_a, hist_c, slot, ha, hc, start=None):
        """The carry after a segment of T steps: its hidden states and the embeddings of its history steps T..T+D-1.  start: the
        segment's step at which a new episode began (auto-reset); history steps before it are zeros in the carry."""
        D = self.depth
        if start is None:
            last = lambda h: torch.stack([h[slot(T + j)] for j in range(D)])     # noqa: E731
            return RolloutCarry(carry.t0 + T, ha, hc, last(hist_a), last(hist_c), episode=carry.episode)
        last = lambda h: torch.stack([h[slot(T + j)] if T + j - D >= start else torch.zeros_like(h[0]) for j in range(D)])  # noqa: E731
        return RolloutCarry(T - start, ha, hc, last(hist_a), last(hist_c), episode=carry.episode + 1)

    def _train_map_data(self, engine, oxy):
        """Per-env obstacle cells [B,O,2] and the cell counts the training forward's critic uses, from the maps `oxy` [M,O,2] (f32)."""
        oxy_env = oxy[engine.map_id.long()].contiguous()
        if self.reference_quirks:      # the critic's all-ones adjacency spans all O padded slots in training (:65,677): 76 phantom cells at (0,0)
            o_count_train = torch.full((engine.B,), engine.O, dtype=torch.int32, device=self.device)
        else:                          # ... or the map's real boundary cells, as in the rollout
            o_count_train = torch.clamp(engine.boundary_count, max=engine.O)[engine.map_id.long()].to(torch.int32).contiguous()
        return oxy_env, o_count_train

    def _train_batch(self, engine, arena, T, oxy, hist_a, hist_c, v, logp, replay=None, carry=None, next_carry=None, ended=None):
        D = self.depth
        seg = {}
        if carry is not None:
            seg = dict(t0=carry.t0, h0_a=carry.ha, h0_c=carry.hc, carry=next_carry)
            if replay is not None:
                seg.update(prefix_a=carry.emb_a, prefix_c=carry.emb_c)
        if replay is not None:         # the ring holds the last D+1 steps only: the history is regenerated per minibatch
            hist_a = hist_c = None
        if ended is None:
            oxy_env, o_count_train = self._train_map_data(engine, oxy)
        else:                          # the envs were reset during the segment: the maps of the episode that ended
            oxy_env, o_count_train = ended.oxy, ended.o_count_train
            seg.update(ended_collision=ended.collision, ended_evader_status=ended.evader_status)
            if ended.k < T:            # the segment's second piece: the next episode's start, on the new maps
                oxy2, o_count_train2 = self._train_map_data(engine, engine.boundary_xy.to(torch.float32).contiguous())
                seg.update(boundary=ended.k, v_boot=ended.v_boot, oxy2=oxy2, o_count_train2=o_count_train2)
                if replay is not None:
                    seg.update(replay2=HistoryReplay(replay.fused, ended.oxy_i, ended.o_count, replay.quirks),
                               map_id2=engine.map_id.to(torch.int32).clone())
        map_id = None
        if replay is not None:         # the map ids of the steps the batch (its first piece) ran: taken before any reset
            map_id = engine.map_id.to(torch.int32).clone() if ended is None else ended.map_id
        return TrainBatch(p=arena.p_state_f32[:T], e=arena.e_state_f32[:T, :, 0].contiguous(), oxy=oxy_env,
                          o_count_train=o_count_train,
                          p_adj_bits=arena.p_adj_bits[:T], e_adj=arena.e_adj[:T], o_adj_bits=arena.o_adj_bits[:T],
                          hist_a=hist_a, hist_c=hist_c, v=v, a=arena.a_n[:T], logp=logp, r=arena.r[:T],
                          active=arena.active[:T], depth=D, replay=replay, map_id=map_id, **seg)

    def explore_env(self, env, num_episode):
        """Reference signature (:731-740) for the single-env facade `Pursuit_Env`: returns
        (mean episode reward, ReplayBuffer in the reference layout, steps)."""
        from .pursuit_env import RolloutArena
        self.minibuffer = ReplayBuffer(cfg=self.cfg, device=self.device)
        self.minibuffer.reset_buffer()
        total_r, steps = 0.0, 0
        for k in range(num_episode):
            env.reset()
            eng = env.engine
            self.reward_norm.to_engine(eng)
            arena = RolloutArena(eng.params, 1, env.max_steps, eng.device)
            env.begin_batched_episode()
            tb = self.rollout_batched(eng, arena, env.max_steps, seed=int(torch.randint(0, 2 ** 31, (1,)).item()))
            self.reward_norm.from_engine(eng)
            env.end_batched_episode()
            total_r += float(arena.raw_reward.sum().item())
            steps += env.max_steps
            self.minibuffer.store_episode(k, arena, tb)
        return total_r / num_episode, self.minibuffer, steps

    def run_episode(self, env, num_episode=0):
        r, _, steps = self.explore_env(env, 1)
        return r, steps
