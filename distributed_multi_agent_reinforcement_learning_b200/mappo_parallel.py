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

import numpy as np
import torch
import torch.nn as nn
from torch.nn.utils import spectral_norm

from . import _lib, fused_policy, policy_ops as ops
from .normalization import Normalization
from .replay_buffer import BigBuffer, ReplayBuffer


PIPELINE_STAGGER = 0        # env steps by which consecutive env-group pipelines of a rollout are offset (see _rollout_pipelined)
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


def _history_inputs(hist_a, hist_c, t, D, quirks, net, slot, sl=slice(None)):
    """The D history inputs of step t for `net` (k = 0 newest; None = zeros, before the episode's first step), read from the
    [*, B, N, E] buffers at index slot(i) for history step i (t + D is what step t writes).  reference_quirks: the ONE list actor and
    critic alias (:750-752), C(t-1), A(t-1), C(t-2), ...; otherwise each network's own embeddings."""
    out = []
    for k in range(D):
        if quirks:
            back, src = k // 2 + 1, (hist_c if k % 2 == 0 else hist_a)
        else:
            back, src = k + 1, (hist_a if net == "actor" else hist_c)
        out.append(src[slot(t - back + D)][sl] if t - back >= 0 else None)
    return out


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
    map_id = None       # i32 [B] (replay only)

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

    def minibatch(self, lo, hi):
        """Envs [lo, hi): contiguous copies of the time-major slabs (the reference's sequential `batch[key][index]`).  A replay-mode
        batch regenerates the minibatch's history from its slabs (on the current stream)."""
        s = lambda x: None if x is None else x[:, lo:hi].contiguous()     # noqa: E731
        mb = TrainBatch(p=s(self.p), e=s(self.e), oxy=self.oxy[lo:hi].contiguous(),
                        o_count_train=self.o_count_train[lo:hi].contiguous(), p_adj_bits=s(self.p_adj_bits),
                        e_adj=s(self.e_adj), o_adj_bits=s(self.o_adj_bits), hist_a=s(self.hist_a), hist_c=s(self.hist_c),
                        v=s(self.v), a=s(self.a), logp=s(self.logp), r=s(self.r), active=s(self.active), depth=self.depth)
        if self.replay is not None:
            mb.replay, mb.map_id = self.replay, self.map_id[lo:hi].contiguous()
            self.replay.regenerate(mb)
        return mb

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

        gh = lambda x: None if x is None else g(x)      # noqa: E731
        out = TrainBatch(p=g(self.p), e=g(self.e), oxy=g(self.oxy, False), o_count_train=g(self.o_count_train, False),
                         p_adj_bits=g(self.p_adj_bits), e_adj=g(self.e_adj), o_adj_bits=g(self.o_adj_bits), hist_a=gh(self.hist_a),
                         hist_c=gh(self.hist_c), v=g(self.v), a=g(self.a), logp=g(self.logp), r=g(self.r), active=g(self.active),
                         depth=self.depth)
        if self.replay is not None:
            out.replay, out.map_id = self.replay, g(self.map_id, False)
            self.replay.regenerate(out)
        return out, g

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

    def __init__(self, fused, oxy_i32, o_count, quirks):
        self.fused, self.oxy_i32, self.o_count, self.quirks = fused, oxy_i32, o_count, bool(quirks)

    def regenerate(self, mb, embed_only=None):
        """Fills mb.hist_a / mb.hist_c [T+D, mb, N, E] with T fused steps on the current stream (forced actions, history read from the
        tensors being filled).  embed_only (default REPLAY_EMBED_ONLY) False runs the full step from zero hidden states and returns the
        replayed (log-prob, value) [T, mb, N] - the same numbers the rollout stored."""
        from types import SimpleNamespace
        embed_only = REPLAY_EMBED_ONLY if embed_only is None else embed_only
        T, B, N, D, E = mb.T, mb.B, mb.N, mb.depth, self.fused.E
        f32 = dict(dtype=torch.float32, device=mb.p.device)
        mb.hist_a, mb.hist_c = torch.zeros(T + D, B, N, E, **f32), torch.zeros(T + D, B, N, E, **f32)
        flags = fused_policy.STATE_F32 | (fused_policy.EMBED_ONLY if embed_only else 0)
        ha = hc = act = logp = v = None
        if not embed_only:
            ha, hc = torch.zeros(2, B * N, E, **f32), torch.zeros(2, B * N, E, **f32)
            act = mb.a.to(torch.int32)
            logp, v = torch.empty(T, B, N, **f32), torch.empty(T, B, N, **f32)
        view = SimpleNamespace(B=B, N=N, O=self.oxy_i32.shape[1], map_id=mb.map_id)
        ident = lambda i: i      # noqa: E731
        for t in range(T):
            view.p_state, view.e_state = mb.p[t], mb.e[t]
            view.p_adj_bits, view.e_adj, view.o_adj_bits = mb.p_adj_bits[t], mb.e_adj[t], mb.o_adj_bits[t]
            h_a = _history_inputs(mb.hist_a, mb.hist_c, t, D, self.quirks, "actor", ident)
            h_c = _history_inputs(mb.hist_a, mb.hist_c, t, D, self.quirks, "critic", ident)
            self.fused.step(view, self.oxy_i32, self.o_count, t, 0, True, h_a, h_c, mb.hist_a[t + D], mb.hist_c[t + D], ha, hc,
                            None if act is None else act[t], None if logp is None else logp[t], None if v is None else v[t],
                            force_action=True, flags=flags)
        return None if embed_only else (logp, v)


class RolloutGraph:
    # (policy_dbg: see MAPPO._rollout_pipelined - an instrumented capture for measurements, not for production replays)
    """`MAPPO.rollout_batched` for all envs of an engine (networks in the loop) captured as ONE CUDA graph: per env step
    observe -> fused policy step (encoder + GRU + heads of both networks, one launch per env group) -> A* replan when due ->
    fused evader-move / step / reward-norm / store kernel; no host involvement on replay.  The engine state the episode starts
    from is whatever the engine holds at replay time."""

    def __init__(self, mappo, engine, arena, T, seed, policy_dbg=None, history=None):
        snap = engine.snapshot()
        kw = {} if policy_dbg is None else dict(timers={"_policy_dbg": policy_dbg}, pipelines=policy_dbg.shape[1])
        # decided once: the warm-up's allocations would otherwise change the free memory the captured rollout sees
        kw["history"] = history or mappo.history_mode(T, engine.B, engine.N)
        mappo.rollout_batched(engine, arena, T, seed=seed, history=kw["history"])   # eager warm-up (kernel attributes, stream pool)
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

    # ------------------------------------------------------------------------------------------------ training
    def _forward_losses(self, mb, adv, v_target, side=None):
        T, B, N, E = mb.T, mb.B, mb.N, self.embedding_dim
        graph = mb.graph()
        enc = self.actor.shared_net
        h0 = torch.zeros(self.num_layers, B * N, E, dtype=torch.float32, device=self.device)
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
                feat_c, _ = self.critic.features(emb_c.view(T, B * N, E), h0)
            emb_a = enc.encode(graph, False, mb.history("actor"))
            feat_a, _ = self.actor.features(emb_a.view(T, B * N, E), h0)
            main.wait_stream(side)
            feat_c.record_stream(main)
        else:
            emb_a = enc.encode(graph, False, mb.history("actor"))
            feat_a, _ = self.actor.features(emb_a.view(T, B * N, E), h0)
            emb_c = enc.encode(graph, True, mb.history("critic"))
            feat_c, _ = self.critic.features(emb_c.view(T, B * N, E), h0)
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

    def gae(self, tb):
        """GAE + advantage normalisation on a time-major TrainBatch (kernel 3b)."""
        L = _lib.lib()
        import ctypes
        T, B, N = tb.T, tb.B, tb.N
        adv, vt = torch.empty_like(tb.r), torch.empty_like(tb.r)
        ws = torch.zeros(int(L.marl_gae_workspace_bytes(B, T, N)), dtype=torch.uint8, device=tb.r.device)
        _lib.check(L.marl_gae(B, T, N, _lib.ptr(tb.r), _lib.ptr(tb.v), _lib.ptr(tb.active), 1, ctypes.c_float(self.gamma),
                              ctypes.c_float(self.gamma * self.lamda), 1 if self.use_adv_norm else 0, _lib.ptr(adv),
                              _lib.ptr(vt), _lib.ptr(ws), _lib.stream_ptr()), "marl_gae")
        return adv, vt

    def train(self, replay_buffer, total_steps, return_numpy=True, trace=None, allreduce=None, mean=False, shuffle=None,
              shuffle_seed=None, permutation=None):
        """MAPPO.train (:638-723): GAE, then for each sequential minibatch forward / PPO losses / backward with gradients
        accumulating and the global-norm clip applied to the running accumulation; no optimizer step here.

        allreduce: None (default, the reference's protocol: the accumulated gradients are summed across replicas once per update,
        in `update()` - main.py:121-129) or "minibatch" (north star: ONE all-reduce per PPO minibatch - every minibatch's gradient
        is summed over the replicas (`mean=True`: averaged) before it enters the running, clipped accumulation, so the clip acts on
        the global gradient and all replicas leave `train` with identical gradients; `update()` then only steps).
        shuffle (default `cfg.algo.shuffle_minibatches`, false = the reference's SequentialSampler :665): minibatches are drawn from a
        device permutation of the envs (seeded by `shuffle_seed`, or given as `permutation`) and gathered by `marl_gather_rows`."""
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
                    ops.clip_grad_norm_(flat, 5.0)
        self.ac_optimizer._sync_grads()
        self._grads_reduced = per_mb
        self.last_train_issue_s = time.perf_counter() - t_issue     # host time to ISSUE the epoch (the device may still be running)
        lh = losses.cpu()
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
    def rollout_batched(self, engine, arena, T=None, seed=0, deterministic=False, groups=1, use_fused=None, timers=None,
                        pipelines=None, actor_only=False, history=None):
        """MAPPO.run_episode (:742-827) for all B envs of a BatchedPursuitEnv at once, entirely on the GPU.
        Per step: observe kernel -> fused encoder (actor, then critic with all-ones adjacency) -> GRU cell -> heads ->
        closed-loop env kernel (evader move + pursuer step + reward-norm + store).  Fills `arena` plus the history /
        value / log-prob slabs and returns a TrainBatch ready for `train`.

        actor_only=True is the EVALUATOR's episode (evaluator.py:118-156): no critic, and the actor's history is its OWN
        embeddings A(t-1), A(t-2), ... (its dataset is not aliased with a critic's there); values / bootstrap stay zero.

        history: 'store' keeps the full [T+D,B,N,E] history of both networks in the batch; 'replay' keeps only a ring of D+1 slabs
        per network during the episode (step t reads at most D steps back) and returns a batch with hist_a = hist_c = None that
        regenerates each minibatch's history in training (HistoryReplay).  None chooses with `history_mode` (store when it fits
        comfortably).  Replay needs the fused step; actor_only rollouts always store."""
        T = T or arena.T
        B, N, E, D, L = engine.B, engine.N, self.embedding_dim, self.depth, self.num_layers
        dev = self.device
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
        hist_a, hist_c = (torch.zeros(D + 1 if replay else T + D, B, N, E, **f32) for _ in range(2))
        v = torch.zeros(T + 1, B, N, **f32)
        logp = torch.zeros(T, B, N, **f32)
        act = torch.zeros(T, B, N, dtype=torch.int32, device=dev)
        ha, hc = torch.zeros(L, B * N, E, **f32), torch.zeros(L, B * N, E, **f32)
        oxy = engine.boundary_xy.to(torch.float32).contiguous()                 # [M,O,2]
        o_count = torch.clamp(engine.boundary_count, max=engine.O).contiguous()  # rollout: the O_b real cells
        enc = self.actor.shared_net
        zeros_hist = torch.zeros(B, N, E, **f32)
        w_eff = None

        quirks = self.reference_quirks

        def history(t, net="actor"):
            # reference: one aliased list for both nets (:750-752): newest first = C(t-1), A(t-1), C(t-2), A(t-2), ...
            # actor_only (the evaluator) / reference_quirks=False: each network's own embeddings, newest first
            out = []
            for k in range(D):
                own = actor_only or not quirks
                back = (k + 1) if own else (k // 2 + 1)
                src = (hist_a if (net == "actor" or actor_only) else hist_c) if own else (hist_c if k % 2 == 0 else hist_a)
                out.append(src[slot(t - back + D)] if t - back >= 0 else zeros_hist)
            return out

        def critic_step(t, graph):
            nonlocal hc, w_eff
            emb_c = enc.encode(graph, True, history(t, "critic"))
            feat_c, hc = self.critic.features(emb_c.view(1, B * N, E), hc)
            w, _ = self.critic.head_weight()
            w_eff = w.reshape(E).contiguous()
            return emb_c, feat_c[0]

        if use_fused:
            # ONE launch per env step for both networks (csrc/policy_fused.cu); embeddings / values / log-probs / actions
            # land directly in their rollout slabs.  The critic's effective head row is constant while the weights are
            # (one power iteration on a [1,E] matrix is already converged), so it is computed once.  A replay-mode batch keeps the
            # step (its own copy of the weights) to regenerate the history in training.
            w, _ = self.critic.head_weight()
            fused = fused_policy.FusedRolloutStep(self, w.reshape(E).contiguous(), snapshot=replay)
            oxy_i = engine.boundary_xy.clone() if replay else engine.boundary_xy.contiguous()
            rep_ = HistoryReplay(fused, oxy_i, o_count, quirks) if replay else None
            none_if_zero = lambda lst: [None if h is zeros_hist else h for h in lst]   # noqa: E731
            def timed(name, fn):
                if timers is None:
                    return fn()
                a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_.record()
                fn()
                b_.record()
                timers.setdefault(name, []).append((a_, b_))

            # Env-group pipelines: the envs are independent, so the batch is cut into G contiguous groups, each stepping through
            # the episode on its own stream (observe -> policy step || A* replan -> env step).  One group's small kernels and the
            # long tail of its replanning (the slowest of its searches gates its env step) then overlap with the other groups'
            # policy kernels instead of idling the GPU.  Same results for any G (the sampling RNG is keyed by the global row).
            auto = pipelines is None
            if auto:
                pipelines = self.default_pipelines(B, N) if (timers is None and groups == 1) else 1
                if os.environ.get("MARL_PIPELINES") and timers is None and groups == 1:      # tuning knob for tools/
                    pipelines = int(os.environ["MARL_PIPELINES"])
            if pipelines > 1 and (timers is None or not auto) and groups == 1 and not actor_only:
                # (an explicit pipelines=G together with timers: CUDA events around every launch of the pipelined schedule itself)
                self._rollout_pipelined(engine, arena, T, seed, deterministic, int(pipelines), fused, oxy_i, o_count, hist_a, hist_c,
                                        act, logp, v, zeros_hist, timers=timers, slot=slot)
                return self._train_batch(engine, arena, T, oxy, hist_a, hist_c, v, logp, rep_)
            # Single pipeline.  The A* replanning due every `difficulty` steps only needs the env state, not the action: it runs
            # on a side stream concurrently with the policy kernel and is joined before the env kernel consumes the paths.
            overlap = timers is None and groups == 1
            main = torch.cuda.current_stream()
            if overlap:
                if getattr(engine, "_replan_stream", None) is None:
                    engine._replan_stream = torch.cuda.Stream(device=dev)
                side = engine._replan_stream
            diff = int(engine.params.difficulty)
            for t in range(T):
                join = None
                if overlap and t % diff == 0:
                    fork = torch.cuda.Event()
                    fork.record(main)
                    side.wait_event(fork)
                    engine.evader_replan(0, B, side)
                    join = torch.cuda.Event()
                    join.record(side)
                timed("env_observe_kernel", engine.observe)
                h_t, h_tc = none_if_zero(history(t)), none_if_zero(history(t, "critic"))
                timed("policy_step_kernel", lambda: fused.step(engine, oxy_i, o_count, t, seed, deterministic, h_t, h_tc,
                                                               hist_a[slot(t + D)], hist_c[slot(t + D)], ha, hc, act[t], logp[t], v[t],
                                                               nets=("actor",) if actor_only else ("actor", "critic")))
                if join is not None:
                    main.wait_event(join)
                engine.rollout_closed(arena, 1, t0=t, action_tape=act[t:t + 1], env_t0=t, groups=groups, timers=timers,
                                      skip_replan=join is not None)
            if actor_only:
                return self._train_batch(engine, arena, T, oxy, hist_a, hist_c, v, logp)
            engine.observe()
            h_fin = none_if_zero(([hist_c[slot(T - 1 + D)]] + history(T - 1)[:D - 1]) if quirks else history(T, "critic"))
            scratch = torch.empty(B, N, E, **f32)
            fused.step(engine, oxy_i, o_count, T, seed, deterministic, h_fin, h_fin, scratch, scratch, ha, hc, None, None, v[T],
                       nets=("critic",))
            return self._train_batch(engine, arena, T, oxy, hist_a, hist_c, v, logp, rep_)

        for t in range(T):
            engine.observe()
            graph = ops.GraphBatch(engine.p_state.to(torch.float32), engine.e_state.to(torch.float32), oxy, engine.map_id,
                                   o_count, engine.p_adj_bits, engine.e_adj, engine.o_adj_bits)
            emb_a = enc.encode(graph, False, history(t))
            feat_a, ha = self.actor.features(emb_a.view(1, B * N, E), ha)
            if actor_only:
                a_i, _, lp, _ = ops.act_head(feat_a[0], None, self.actor.Mean.weight, self.actor.Mean.bias, None, None, seed, t,
                                             deterministic)
                hist_a[t + D] = emb_a
            else:
                emb_c, feat_c = critic_step(t, graph)
                a_i, _, lp, val = ops.act_head(feat_a[0], feat_c, self.actor.Mean.weight, self.actor.Mean.bias, w_eff,
                                               self.critic.Mean.bias, seed, t, deterministic)
                hist_a[t + D], hist_c[t + D] = emb_a, emb_c
                v[t] = val.view(B, N)
            logp[t], act[t] = lp.view(B, N), a_i.view(B, N)
            engine.rollout_closed(arena, 1, t0=t, action_tape=act[t:t + 1], env_t0=t, groups=groups)
        if actor_only:
            return self._train_batch(engine, arena, T, oxy, hist_a, hist_c, v, logp)
        # bootstrap value of the final state (:806-825): only the critic's dataset is updated once more
        engine.observe()
        graph = ops.GraphBatch(engine.p_state.to(torch.float32), engine.e_state.to(torch.float32), oxy, engine.map_id,
                               o_count, engine.p_adj_bits, engine.e_adj, engine.o_adj_bits)
        hist_final = ([hist_c[T - 1 + D]] + history(T - 1)[:D - 1]) if quirks else history(T, "critic")
        emb_c = enc.encode(graph, True, hist_final)
        feat_c, hc = self.critic.features(emb_c.view(1, B * N, E), hc)
        w, _ = self.critic.head_weight()
        v[T] = torch.nn.functional.linear(feat_c[0], w, self.critic.Mean.bias).view(B, N)
        return self._train_batch(engine, arena, T, oxy, hist_a, hist_c, v, logp)

    @staticmethod
    def default_pipelines(B, N):
        """Env-group pipelines of a batched rollout: one per 8192 (env, agent) rows, at most 8."""
        return max(1, min(8, (B * N) // 8192))

    def _rollout_pipelined(self, engine, arena, T, seed, deterministic, G, fused, oxy_i, o_count, hist_a, hist_c, act, logp, v,
                           zeros_hist, timers=None, slot=lambda i: i):
        """G independent env-group pipelines, one stream (+ one A* side stream) each; see rollout_batched.
        timers: dict name -> list of (start, end) CUDA events recorded on the launching stream around every launch.  If it holds a
        "_policy_dbg" int64 tensor [T, G, >= CTAs per launch, 16], every policy launch instead writes its per-CTA record there (slots
        13 / 14 = %globaltimer at CTA start / end in ns, 15 = SM id; csrc/policy_fused.cu) - usable under CUDA-graph capture, which
        is how bench.py times the kernel inside the schedule it reports."""
        dbg = timers.pop("_policy_dbg", None) if timers is not None else None
        if timers is not None and not timers and dbg is not None:
            timers = None                                   # only the in-kernel records were asked for: no events (graph capture)
        B, N, E, D, L = engine.B, engine.N, self.embedding_dim, self.depth, self.num_layers
        dev = self.device
        main = torch.cuda.current_stream()
        if len(getattr(engine, "_pipe_streams", [])) < 2 * G:
            # MARL_PIPE_PRIORITY (measurement knob): "astar" / "policy" gives the A* side streams / the policy streams the high priority
            prio = os.environ.get("MARL_PIPE_PRIORITY", "")
            engine._pipe_streams = [torch.cuda.Stream(device=dev, priority=(-1 if (prio == "astar" and i % 2 == 1) or (prio == "policy" and i % 2 == 0) else 0))
                                    for i in range(2 * G)]
        rec_ptrs = arena.record_pointers()
        diff = int(engine.params.difficulty)
        full_tile = (128 // N) * N if N <= 128 else 0      # concurrent launches: full tiles, SMs left over for the neighbours
        if os.environ.get("MARL_PIPE_TILE_ROWS"):            # tuning knob for tools/
            full_tile = int(os.environ["MARL_PIPE_TILE_ROWS"])
        fork = torch.cuda.Event(enable_timing=timers is not None)
        fork.record(main)
        if timers is not None:
            timers["_t0"] = fork

        def timed(name, stream, fn):
            if timers is None:
                return fn()
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record(stream)
            fn()
            b_.record(stream)
            timers.setdefault(name, []).append((a_, b_))

        class _View:                                     # what FusedRolloutStep.step reads from an engine, for envs [lo, hi)
            pass

        # Stagger: every group replans at the same env steps (t % difficulty == 0), and a replan stalls its group for the length of
        # its slowest A* search; groups that run in lockstep would all be stalled at once.  Group g therefore starts when group g-1
        # has launched its policy step number `stagger`: the stalls then fall on different wall-clock times and the other groups'
        # policy kernels fill the SMs meanwhile.
        stagger = int(os.environ.get("MARL_STAGGER", PIPELINE_STAGGER))
        stagger_ev = None
        for g in range(G):
            lo, hi = g * B // G, (g + 1) * B // G
            st, side = engine._pipe_streams[2 * g], engine._pipe_streams[2 * g + 1]
            st.wait_event(fork)
            if stagger_ev is not None:
                st.wait_event(stagger_ev)
                stagger_ev = None
            with torch.cuda.stream(st):
                view = _View()
                view.B, view.N, view.O = hi - lo, N, engine.O
                ha = torch.zeros(L, (hi - lo) * N, E, dtype=torch.float32, device=dev)
                hc = torch.zeros(L, (hi - lo) * N, E, dtype=torch.float32, device=dev)
                sl = slice(lo, hi)

                def hist_of(t, net="actor"):
                    return _history_inputs(hist_a, hist_c, t, D, self.reference_quirks, net, slot, sl)

                def refresh():
                    view.p_state, view.e_state, view.map_id = engine.p_state[sl], engine.e_state[sl], engine.map_id[sl]
                    view.p_adj_bits, view.e_adj, view.o_adj_bits = engine.p_adj_bits[sl], engine.e_adj[sl], engine.o_adj_bits[sl]

                refresh()
                for t in range(T):
                    join = None
                    if t % diff == 0:
                        ev = torch.cuda.Event()
                        ev.record(st)
                        side.wait_event(ev)
                        timed("evader_kernel", side, lambda: engine.evader_replan(lo, hi, side))
                        join = torch.cuda.Event()
                        join.record(side)
                    timed("env_observe_kernel", st, lambda: engine.observe(lo=lo, hi=hi))
                    h_t, h_tc = hist_of(t), hist_of(t, "critic")
                    timed("policy_step_kernel", st, lambda: fused.step(
                        view, oxy_i, o_count, t, seed, deterministic, h_t, h_tc, hist_a[slot(t + D)][sl], hist_c[slot(t + D)][sl], ha, hc,
                        act[t][sl], logp[t][sl], v[t][sl], row_offset=lo * N, tile_rows=full_tile,
                        debug=dbg[t, g] if dbg is not None else None))
                    if stagger > 0 and t == min(stagger, T - 1) - 1 and g + 1 < G:
                        stagger_ev = torch.cuda.Event()
                        stagger_ev.record(st)
                    if join is not None:
                        st.wait_event(join)
                    timed("rollout_kernel", st, lambda: engine._closed_chunk(arena, rec_ptrs, lo, hi, t, 1, act[t:t + 1], 0, seed, st))
                engine.observe(lo=lo, hi=hi)
                h_fin = ([hist_c[slot(T - 1 + D)][sl]] + hist_of(T - 1)[:D - 1]) if self.reference_quirks else hist_of(T, "critic")
                scratch = torch.empty(hi - lo, N, E, dtype=torch.float32, device=dev)
                fused.step(view, oxy_i, o_count, T, seed, deterministic, h_fin, h_fin, scratch, scratch, ha, hc, None, None, v[T][sl],
                           nets=("critic",), row_offset=lo * N, tile_rows=full_tile)
                done = torch.cuda.Event()
                done.record(st)
            main.wait_event(done)

    def explore_batched(self, engine, arena, T=None, seed=0, host_state=None, host_out=None, reset_reward_norm=False, history=None):
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
        snapshot its history is regenerated with (the graph re-packs it in place)."""
        T = T or arena.T
        key = (id(engine), id(arena), int(T), int(seed))
        graphs = self.__dict__.setdefault("_episode_graphs", {})
        if key not in graphs:
            graphs[key] = RolloutGraph(self, engine, arena, T, seed, history=history)
        g = graphs[key]
        if host_state is not None:
            engine.load_host_state(reset_reward_norm=reset_reward_norm, **host_state)
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

    def _train_batch(self, engine, arena, T, oxy, hist_a, hist_c, v, logp, replay=None):
        B, D, dev = engine.B, self.depth, self.device
        if replay is not None:         # the ring holds the last D+1 steps only: the history is regenerated per minibatch
            hist_a = hist_c = None
        oxy_env = oxy[engine.map_id.long()].contiguous()
        if self.reference_quirks:      # the critic's all-ones adjacency spans all O padded slots in training (:65,677): 76 phantom cells at (0,0)
            o_count_train = torch.full((B,), engine.O, dtype=torch.int32, device=dev)
        else:                          # ... or the map's real boundary cells, as in the rollout
            o_count_train = torch.clamp(engine.boundary_count, max=engine.O)[engine.map_id.long()].to(torch.int32).contiguous()
        return TrainBatch(p=arena.p_state_f32[:T], e=arena.e_state_f32[:T, :, 0].contiguous(), oxy=oxy_env,
                          o_count_train=o_count_train,
                          p_adj_bits=arena.p_adj_bits[:T], e_adj=arena.e_adj[:T], o_adj_bits=arena.o_adj_bits[:T],
                          hist_a=hist_a, hist_c=hist_c, v=v, a=arena.a_n[:T], logp=logp, r=arena.r[:T],
                          active=arena.active[:T], depth=D, replay=replay,
                          map_id=None if replay is None else engine.map_id.to(torch.int32).clone())

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
