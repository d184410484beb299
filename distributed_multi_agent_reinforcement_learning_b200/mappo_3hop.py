"""Second network family — B200 mirror of `obstacle_differ_3hop/mappo_parallel.py` (SURVEY §8 a22): `GnnExtractor`,
`SharedActor`, `SharedCritic`, `MAPPO.train`, with the reference's class / sub-module names (`shared_net.one_hop`,
`shared_net.bottleneck`, `GRU`, `Mean`) so that state_dicts interchange, and the reference's layer construction order so that
equal torch seeds give equal initial weights.

Compute path: the 128-wide dense layers go through the tcgen05 3xTF32 GEMM (policy_ops.linear), the adjacency-normalised
entity means through csrc/gnn_kernels.cu (forward and backward), GRU / heads / PPO loss / clip / Adam through the same kernels as
the DHGN family.  The env of this family is not part of the reference tree, so there is no rollout engine here: the classes
consume the reference's buffer layout (`module/replay_buffer.py:21-30`).

Deviation: the reference `MAPPO.__init__` unconditionally loads `./model/actor.pth` / `critic.pth` (:320-324); here that is
optional (`pretrain_dir`)."""
import ctypes

import numpy as np
import torch
import torch.nn as nn
from torch.nn.utils import spectral_norm

from . import _lib, policy_ops as ops
from .mappo_parallel import _FlatAdam, orthogonal_init
from .train_stats import TrainStats


def preproc_layer(input_size, output_size, is_sn=False):
    layer = nn.Linear(input_size, output_size)
    orthogonal_init(layer)
    return spectral_norm(layer) if is_sn else layer


class _EntityAgg(torch.autograd.Function):
    """out[s,i,:] = sum_j w_ij x[s,i,j,:], w = L1-normalised adjacency (or 1/J when all_ones)."""

    @staticmethod
    def forward(ctx, x, adj, all_ones):
        S, N, J, E = x.shape
        x, adj = x.contiguous(), adj.contiguous()
        out = torch.empty(S, N, E, dtype=torch.float32, device=x.device)
        _lib.check(_lib.lib().marl_entity_agg_fwd(S * N, N, J, J, E, _lib.ptr(adj), 1 if all_ones else 0, _lib.ptr(x), N * J * E,
                                                  J * E, E, _lib.ptr(out), _lib.stream_ptr()), "marl_entity_agg_fwd")
        ctx.save_for_backward(adj)
        ctx.all_ones, ctx.shape = all_ones, (S, N, J, E)
        return out

    @staticmethod
    def backward(ctx, dout):
        (adj,) = ctx.saved_tensors
        S, N, J, E = ctx.shape
        dx = torch.empty(S, N, J, E, dtype=torch.float32, device=dout.device)
        _lib.check(_lib.lib().marl_entity_agg_bwd(S * N, J, E, _lib.ptr(adj), 1 if ctx.all_ones else 0, _lib.ptr(dout.contiguous()),
                                                  _lib.ptr(dx), _lib.stream_ptr()), "marl_entity_agg_bwd")
        return dx, None, None


def comm_agg(last_comm, adj, all_ones):
    """adj_normalised[..., :N] @ last_comm_embedding (no gradient: the embeddings are buffer data).  last_comm [S,N,C]."""
    S, N, C = last_comm.shape
    J = adj.shape[-1]
    out = torch.empty(S, N, C, dtype=torch.float32, device=last_comm.device)
    _lib.check(_lib.lib().marl_entity_agg_fwd(S * N, N, J, N, C, _lib.ptr(adj.contiguous()), 1 if all_ones else 0,
                                              _lib.ptr(last_comm.contiguous()), N * C, 0, C, _lib.ptr(out), _lib.stream_ptr()),
               "marl_entity_agg_fwd")
    return out


class GnnExtractor(nn.Module):
    def __init__(self, input_size, middle_size, output_size, n_hops: int = 1, is_sn: bool = False):
        super().__init__()
        self.n_hop = n_hops
        self.one_hop = nn.Sequential(
            preproc_layer(input_size, middle_size) if is_sn else nn.Linear(input_size, middle_size), nn.ReLU(),
            preproc_layer(middle_size, output_size) if is_sn else nn.Linear(middle_size, output_size), nn.ReLU())
        self.bottleneck = nn.Sequential(
            preproc_layer(output_size + 2 * output_size, output_size) if is_sn else nn.Linear(3 * output_size, output_size), nn.ReLU())

    def forward(self, obs, last_comm_embedding=None, adj=None, all_ones=False):
        """obs [*, N, J, F]; adj [*, N, J]; last_comm_embedding [*, N, 2*out] -> [*, N, out]."""
        lead = tuple(obs.shape[:-3])
        N, J, F = obs.shape[-3:]
        S = int(np.prod(lead)) if lead else 1
        l1, l2, lb = self.one_hop[0], self.one_hop[2], self.bottleneck[0]
        h1 = ops.linear(obs.reshape(S * N * J, F).float().contiguous(), l1.weight, l1.bias, relu=True)
        h0 = ops.linear(h1, l2.weight, l2.bias, relu=True)
        E = h0.shape[-1]
        adj2 = adj.reshape(S, N, J).float().contiguous()
        h0_agg = _EntityAgg.apply(h0.view(S, N, J, E), adj2, all_ones)
        c_agg = comm_agg(last_comm_embedding.reshape(S, N, -1).float(), adj2, all_ones)
        feat = ops.linear(h0_agg.view(S * N, E), lb.weight, lb.bias, relu=True, x2=c_agg.view(S * N, -1))
        return feat.view(*lead, N, E)


class _Shared(nn.Module):
    def _gru_weights(self):
        g = self.GRU
        return [(getattr(g, f"weight_ih_l{l}"), getattr(g, f"weight_hh_l{l}"), getattr(g, f"bias_ih_l{l}"), getattr(g, f"bias_hh_l{l}"))
                for l in range(self.num_layers)]

    def _features(self, comm_embedding, hidden_state, mode):
        if mode == 0:
            feat, hidden_state = ops.gru_forward(comm_embedding.unsqueeze(0).contiguous(), hidden_state, self._gru_weights(), self.num_layers)
            return feat.squeeze(0), hidden_state
        batch, steps, num_agent = comm_embedding.shape[:3]
        x = comm_embedding.permute(1, 0, 2, 3).reshape(steps, batch * num_agent, self.rnn_input_size)
        feat, hidden_state = ops.gru_forward(x, hidden_state, self._gru_weights(), self.num_layers)
        return feat.reshape(steps, batch, num_agent, self.hidden_size).permute(1, 0, 2, 3), hidden_state

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
                    p.grad.copy_(g)
                else:
                    p.grad = g


class SharedActor(_Shared):
    def __init__(self, shared_net, rnn_input_dim, output_size, num_layers, hidden_size, is_sn=False):
        super().__init__()
        self.shared_net = shared_net
        self.num_layers, self.rnn_input_size, self.hidden_size = num_layers, rnn_input_dim, hidden_size
        self.GRU = nn.GRU(self.rnn_input_size, hidden_size, num_layers)
        self.Mean = preproc_layer(hidden_size, output_size) if is_sn else nn.Linear(hidden_size, output_size)

    def forward(self, state, adj, hidden_state, last_comm_embedding, mode):
        comm_embedding = self.shared_net(state, last_comm_embedding, adj)
        assert 2 * comm_embedding.shape[-1] == last_comm_embedding.shape[-1]
        feature, hidden_state = self._features(comm_embedding, hidden_state, mode)
        prob = torch.softmax(torch.nn.functional.linear(feature, self.Mean.weight, self.Mean.bias), dim=-1)
        return prob, hidden_state, comm_embedding

    def choose_action(self, state, adj, hidden_state, last_comm_embedding, deterministic=True):
        prob, hidden_state, comm_embedding = self.forward(state, adj, hidden_state, last_comm_embedding, mode=0)
        if deterministic:
            return prob.argmax(dim=-1), hidden_state, comm_embedding
        dist = torch.distributions.Categorical(probs=prob)
        a_n = dist.sample()
        return a_n, dist.log_prob(a_n), hidden_state, comm_embedding

    def get_logprob_and_entropy(self, state, adj, hidden_state, last_comm_embedding, action):
        prob, _, __ = self.forward(state, adj, hidden_state, last_comm_embedding, mode=1)
        dist = torch.distributions.Categorical(prob)
        return dist.log_prob(action), dist.entropy()


class SharedCritic(_Shared):
    def __init__(self, shared_net, rnn_input_dim, output_size, num_layers, hidden_size, is_sn=False):
        super().__init__()
        self.shared_net = shared_net
        self.num_layers, self.rnn_input_size, self.hidden_size, self.is_sn = num_layers, rnn_input_dim, hidden_size, is_sn
        self.GRU = nn.GRU(rnn_input_dim, hidden_size, num_layers)
        self.Mean = preproc_layer(hidden_size, output_size, is_sn=is_sn)

    def head_weight(self):
        if not self.is_sn:
            return self.Mean.weight
        sigma, u2, v = ops.spectral_sigma(self.Mean.weight_orig, self.Mean.weight_u)
        with torch.no_grad():
            self.Mean.weight_u.copy_(u2)
            self.Mean.weight_v.copy_(v)
        return self.Mean.weight_orig / sigma

    def forward(self, state, adj, hidden_state, last_comm_embedding, mode):
        comm_embedding = self.shared_net(state, last_comm_embedding, adj, all_ones=True)     # ones_like(adj) (:171)
        assert 2 * comm_embedding.shape[-1] == last_comm_embedding.shape[-1]
        feature, hidden_state = self._features(comm_embedding, hidden_state, mode)
        val = torch.nn.functional.linear(feature, self.head_weight(), self.Mean.bias)
        return (val, hidden_state, comm_embedding) if mode == 0 else val


class MAPPO:
    """obstacle_differ_3hop/mappo_parallel.py:237-425 (constructor arguments and `train` contract)."""

    def __init__(self, args, batch_size, mini_batch_size, agent_type, pretrain_dir=None):
        self.batch_size, self.mini_batch_size = batch_size, mini_batch_size
        self.max_train_steps, self.lr, self.gamma, self.lamda = args.max_train_steps, args.lr, args.gamma, args.lamda
        self.epsilon, self.K_epochs, self.entropy_coef = args.epsilon, args.K_epochs, args.entropy_coef
        self.use_grad_clip, self.use_lr_decay = args.use_grad_clip, args.use_lr_decay
        self.use_adv_norm, self.use_value_clip = args.use_adv_norm, args.use_value_clip
        self.actor_input_dim = self.critic_input_dim = args.state_dim + 1
        self.num_layers, self.gnn_output_dim = args.num_layers, args.gnn_output_dim
        self.rnn_input_dim, self.rnn_hidden_dim, self.n_hops = args.gnn_output_dim, args.rnn_hidden_dim, args.n_hops
        key = "learner_device" if "Learner" in agent_type else ("worker_device" if "Worker" in agent_type else "evaluator_device")
        self.device = torch.device(getattr(args, key))
        if self.device.type != "cuda":
            raise _lib.MarlError(f"{key}={self.device}: this engine runs on CUDA only (no CPU fallback)")
        sn = args.use_spectral_norm
        actor_gnn = GnnExtractor(self.actor_input_dim, args.gnn_middle_dim, args.gnn_output_dim, args.n_hops, sn)
        critic_gnn = GnnExtractor(self.critic_input_dim, args.gnn_middle_dim, args.gnn_output_dim, args.n_hops, sn)
        self.actor = SharedActor(actor_gnn, self.rnn_input_dim, args.action_dim, args.num_layers, args.rnn_hidden_dim, sn)
        self.critic = SharedCritic(critic_gnn, self.rnn_input_dim, 1, args.num_layers, args.rnn_hidden_dim, sn)
        if pretrain_dir is not None:
            self.actor.load_state_dict(torch.load(pretrain_dir + "/actor.pth", map_location="cpu").state_dict())
            self.critic.load_state_dict(torch.load(pretrain_dir + "/critic.pth", map_location="cpu").state_dict())
        self.sn, self.args, self.minibuffer = sn, args, None
        self.last_train_stats = None     # TrainStats of the last train(stats=True)
        self.finalize()

    def finalize(self):
        """Moves the networks to the device and builds the flat parameter / gradient arenas (call again after replacing
        parameters wholesale, e.g. load_state_dict on CPU modules)."""
        self.actor, self.critic = self.actor.to(self.device), self.critic.to(self.device)
        self.ac_parameters = (list(self.critic.shared_net.parameters()) + list(self.actor.shared_net.parameters()) +
                              list(self.actor.GRU.parameters()) + list(self.critic.GRU.parameters()) +
                              list(self.critic.Mean.parameters()) + list(self.actor.Mean.parameters()))
        self.ac_optimizer = _FlatAdam(self.ac_parameters, lr=self.lr, eps=1e-5)

    def gae(self, batch, T):
        L = _lib.lib()
        r, v, act = (batch[k][:, :n].contiguous().float() for k, n in (("r", T), ("v_n", T + 1), ("active", T)))
        B, _, N = r.shape
        adv, vt = torch.empty_like(r), torch.empty_like(r)
        ws = torch.zeros(int(L.marl_gae_workspace_bytes(B, T, N)), dtype=torch.uint8, device=r.device)
        _lib.check(L.marl_gae(B, T, N, _lib.ptr(r), _lib.ptr(v), _lib.ptr(act), 0, ctypes.c_float(self.gamma),
                              ctypes.c_float(self.gamma * self.lamda), 1 if self.use_adv_norm else 0, _lib.ptr(adv), _lib.ptr(vt),
                              _lib.ptr(ws), _lib.stream_ptr()), "marl_gae")
        return adv, vt

    def train(self, replay_buffer, total_steps, stats=False):
        """stats=True: PPO diagnostics of the update, one `marl_ppo_stats` row per team-size minibatch, left in
        `self.last_train_stats` (a TrainStats, see mappo_parallel.MAPPO.train); training and the return value are unchanged."""
        per_team = []
        for num in self.args.pursuer_num:
            batch, T = replay_buffer.get_training_data(num, self.device)
            batch = {k: v.to(self.device) for k, v in batch.items()}
            per_team.append((num, batch, T) + self.gae(batch, T))
        object_critics = object_actors = 0.0
        update_time = 0
        self.ac_optimizer.zero_grad()
        E, L = self.rnn_hidden_dim, self.num_layers
        cm = self.critic.Mean
        if stats:
            n_mb = len(per_team) * len(range(0, self.batch_size, self.mini_batch_size))
            mb_sums = torch.empty(n_mb, ops.PPO_STATS_SUMS, dtype=torch.float64, device=self.device)
            norms = torch.empty(n_mb, dtype=torch.float32, device=self.device) if self.use_grad_clip else None
        with torch.enable_grad(), ops.pack_scope():
            for num, batch, T, adv, v_target in per_team:
                for lo in range(0, self.batch_size, self.mini_batch_size):
                    idx = slice(lo, min(lo + self.mini_batch_size, self.batch_size))
                    mb = idx.stop - idx.start
                    h0 = torch.zeros(L, mb * num, E, dtype=torch.float32, device=self.device)
                    st, ad = batch["state"][idx, :T], batch["adj"][idx, :T]
                    emb_a = self.actor.shared_net(st, batch["actor_comm_embedding"][idx, :T], ad)
                    feat_a, _ = self.actor._features(emb_a, h0, mode=1)                          # [mb,T,N,E]
                    emb_c = self.critic.shared_net(st, batch["critic_comm_embedding"][idx, :T], ad, all_ones=True)
                    feat_c, _ = self.critic._features(emb_c, h0, mode=1)
                    flat = lambda x: x.reshape(-1).contiguous()     # noqa: E731
                    la, lc, logp, ent, val, u2, v2 = ops.ppo_head(
                        feat_a.reshape(-1, E), feat_c.reshape(-1, E), self.actor.Mean.weight, self.actor.Mean.bias,
                        cm.weight_orig if self.sn else cm.weight, cm.bias, cm.weight_u if self.sn else torch.ones(1, device=self.device),
                        flat(batch["a_n"][idx, :T]), flat(batch["a_logprob_n"][idx, :T]), flat(adv[idx]),
                        flat(batch["v_n"][idx, :T]) if self.use_value_clip else None,
                        flat(v_target[idx]), flat(batch["active"][idx, :T]), self.epsilon, self.entropy_coef)
                    if self.sn:
                        with torch.no_grad():
                            cm.weight_u.copy_(u2)
                            cm.weight_v.copy_(v2)
                    if stats:
                        ops.ppo_stats(logp, batch["a_logprob_n"][idx, :T], ent, val,
                                      batch["v_n"][idx, :T] if self.use_value_clip else None, v_target[idx],
                                      batch["active"][idx, :T], self.epsilon, out=mb_sums[update_time])
                    (la + lc).backward()
                    if self.use_grad_clip:
                        ops.clip_grad_norm_(self.ac_optimizer.flat_grad, 10.0,                    # (:405)
                                            out=norms[update_time:update_time + 1] if stats else None)
                    object_critics += float(lc.detach())
                    object_actors += float(la.detach())
                    update_time += 1
        if stats:
            self.last_train_stats = TrainStats.from_sums(ops.ppo_stats_combine(mb_sums, norms, 10.0), self.epsilon,
                                                         10.0 if self.use_grad_clip else None)
        if self.use_lr_decay:
            self.lr_decay(total_steps)
        return object_critics / update_time, object_actors / update_time, self.actor.get_gradients(), self.critic.get_gradients()

    def lr_decay(self, total_steps):
        lr_now = self.lr * (1 - total_steps / self.max_train_steps)
        for p in self.ac_optimizer.param_groups:
            p["lr"] = lr_now

    def save_model(self, cwd):
        torch.save(self.actor.state_dict(), cwd + "actor.pth")
        torch.save(self.critic.state_dict(), cwd + "critic.pth")
