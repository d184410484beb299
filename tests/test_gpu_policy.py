"""GPU parity tests of kernel family 5 (DHGN encoder pieces, GRU, heads + PPO loss, clip, Adam) and of the MAPPO
mirror built on them.

Two oracles:
  * tests/golden/algo_*.npz — produced by executing the unmodified reference (explore_env + train + Adam step);
  * oracle/policy_ref.py — the torch fp32 restatement pinned to those fixtures, used here on random inputs at the
    production width (E=128) and odd shapes.
Tolerances (north_star): 1e-5 relative for GAE / statistics / forward activations, 1e-4 for losses and gradients."""
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR, AlgoFixture

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

FIXTURES = sorted(glob.glob(os.path.join(GOLDEN_DIR, "algo_*.npz")))
IDS = [os.path.basename(p)[:-4] for p in FIXTURES]


def _cfg(depth, n_def, T, emb):
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    return default_config(env__num_defender=n_def, env__max_steps=T, algo__depth=depth, algo__embedding_dim=emb,
                          algo__rnn_hidden_dim=emb, algo__learner_device="cuda", algo__worker_device="cuda")


def _load(path):
    fx = AlgoFixture(path)
    depth, n_def, T, episodes, mb, seed, emb = (int(v) for v in fx["meta"])
    return fx, depth, n_def, T, episodes, mb, seed, emb


def _load_weights(mappo, fx, prefix="w."):
    for net, mod in (("actor", mappo.actor), ("critic", mappo.critic)):
        sd = {k[len(prefix) + len(net) + 1:]: torch.from_numpy(fx[k]) for k in fx.files if k.startswith(prefix + net + ".")}
        mod.load_state_dict(sd)


class _Big:
    def __init__(self, d):
        self.buffer = d

    def get_training_data(self, device):
        return {k: v.to(device) for k, v in self.buffer.items()}


@pytest.mark.parametrize("path", FIXTURES, ids=IDS)
def test_initial_weights_equal_reference(path):
    """Same torch seed -> the reference's initial weights, key for key (checkpoint layout + init order)."""
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    fx, depth, n_def, T, episodes, mb, seed, emb = _load(path)
    torch.manual_seed(seed)
    m = MAPPO(_cfg(depth, n_def, T, emb), None, None, "Worker")
    for net, mod in (("actor", m.actor), ("critic", m.critic)):
        sd = mod.state_dict()
        want = [k[len("w." + net + "."):] for k in fx.files if k.startswith("w." + net + ".")]
        assert list(sd.keys()) == want
        for k in want:
            gold = fx[f"w_init.{net}.{k}"] if f"w_init.{net}.{k}" in fx.files else fx[f"w.{net}.{k}"]
            assert np.array_equal(sd[k].cpu().numpy(), gold), (net, k)


def _reference_adam_step(fx, m):
    """Weights after the reference's optimizer step (runner.py:72-78: stock torch.optim.Adam(lr, eps=1e-5), DHGN/mappo_parallel.py:631-632)
    on the fixture's weights and gradients - for the wide fixtures, which do not store them."""
    names = [(net, name) for net, mod in (("actor", m.actor), ("critic", m.critic)) for name, _ in mod.named_parameters()]
    seen, params = {}, []
    for net, name in names:
        key = name if name.startswith("shared_net.") else f"{net}.{name}"      # one encoder instance under both networks
        if key in seen:
            continue
        p = torch.nn.Parameter(torch.from_numpy(np.array(fx[f"w.{net}.{name}"])).clone())
        p.grad = torch.from_numpy(np.array(fx[f"grad.{net}.{name}"])).clone()
        seen[key] = p
        params.append(p)
    torch.optim.Adam(params, lr=float(fx["lr_used"]), eps=1e-5).step()
    out = {}
    for net, name in names:
        key = name if name.startswith("shared_net.") else f"{net}.{name}"
        out[f"{net}.{name}"] = seen[key].detach().numpy()
    return out


@pytest.mark.parametrize("concurrent", [1, 3], ids=["sequential_minibatches", "three_minibatches_in_flight"])
@pytest.mark.parametrize("path", FIXTURES, ids=IDS)
def test_train_matches_reference(path, concurrent, monkeypatch):
    """MAPPO.train on the reference's own buffer and weights: advantages, per-minibatch forward outputs, both losses,
    every accumulated (and clipped) gradient, then one optimizer step.  At E = 128 (the production width) every dense layer
    must have gone through the tcgen05 kernels - rowgemm, wgrad, gru_seq - and none through a library GEMM; the minibatches run
    one at a time and three in flight (the schedule the bench's `train` number uses)."""
    from distributed_multi_agent_reinforcement_learning_b200 import mappo_parallel as mp, policy_ops as ops
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    fx, depth, n_def, T, episodes, mb, seed, emb = _load(path)
    monkeypatch.setattr(mp, "CONCURRENT_MINIBATCHES", concurrent)
    monkeypatch.setattr(ops, "ROWGEMM_MIN_ROWS", 1)      # performance thresholds only: the fixtures are small
    monkeypatch.setattr(ops, "WGRAD_MIN_ROWS", 1)
    m = MAPPO(_cfg(depth, n_def, T, emb), episodes, mb, "Learner")
    _load_weights(m, fx)
    buf = {k[4:]: torch.from_numpy(fx[k]) for k in fx.files if k.startswith("buf.")}
    trace = {}
    ops.CALLS.clear()
    objC, objA, ag, cg = m.train(_Big(buf), int(fx["total_steps"]), trace=trace)
    calls = dict(ops.CALLS)
    if emb == 128:
        n_mb = int(fx["n_mb"])
        assert calls.get("rowgemm", 0) >= 10 * n_mb and calls.get("wgrad", 0) >= 10 * n_mb, calls
        assert calls.get("gru_seq_fwd", 0) == 4 * n_mb and calls.get("gru_seq_bwd", 0) == 4 * n_mb, calls
        assert calls.get("linear_library", 0) == 0 and calls.get("wgrad_library", 0) == 0 and calls.get("gemm_tile", 0) == 0, calls
    tm = lambda x: torch.from_numpy(x).transpose(0, 1).cuda()
    torch.testing.assert_close(trace["adv"], tm(fx["adv"]), rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(trace["v_target"], tm(fx["v_target"]), rtol=1e-6, atol=1e-7)
    assert len(trace["mb"]) == int(fx["n_mb"])
    for i, t in enumerate(trace["mb"]):
        torch.testing.assert_close(t["logp"], tm(fx[f"mb{i}.logp"]), rtol=1e-5, atol=2e-6)
        torch.testing.assert_close(t["ent"], tm(fx[f"mb{i}.ent"]), rtol=1e-5, atol=2e-6)
        torch.testing.assert_close(t["val"], tm(fx[f"mb{i}.val"]), rtol=1e-5, atol=2e-6)
        lc, la = fx[f"mb{i}.losses"]
        assert abs(t["critic_loss"] - lc) <= 1e-4 * max(1.0, abs(lc)) and abs(t["actor_loss"] - la) <= 1e-4 * max(1.0, abs(la))
    assert abs(objC - float(fx["objC"])) < 1e-5 and abs(objA - float(fx["objA"])) < 1e-5
    for net, mod, grads in (("actor", m.actor, ag), ("critic", m.critic, cg)):
        for (name, _), g in zip(mod.named_parameters(), grads):
            gold = fx[f"grad.{net}.{name}"]
            np.testing.assert_allclose(g, gold, rtol=1e-4, atol=2e-6, err_msg=f"{net}.{name}")
    # optimizer step (runner.py:72-78): lr after lr_decay, eps 1e-5
    assert abs(m.ac_optimizer.param_groups[0]["lr"] - float(fx["lr_used"])) < 1e-12
    m.ac_optimizer.step()
    after = None if "w_after.actor.Mean.weight" in fx else _reference_adam_step(fx, m)
    for net, mod in (("actor", m.actor), ("critic", m.critic)):
        for k, v in mod.state_dict().items():
            if k.endswith(("weight_u", "weight_v")):
                continue
            # (Adam normalises the update to ~lr per element: near-zero gradients make its sign - not its size - sensitive to 1e-8
            # gradient differences, so the comparison of our step on OUR gradients allows 2 % of one lr)
            if after is None:
                np.testing.assert_allclose(v.cpu().numpy(), fx[f"w_after.{net}.{k}"], rtol=1e-5, atol=1e-6, err_msg=f"{net}.{k}")
            else:
                np.testing.assert_allclose(v.cpu().numpy(), after[f"{net}.{k}"], rtol=1e-5, atol=1e-5, err_msg=f"{net}.{k}")


@pytest.mark.parametrize("path", FIXTURES, ids=IDS)
def test_rollout_forward_reproduces_reference_buffer(path):
    """Replays the reference's own rollout observations through the rollout-mode forward (aliased history list, critic
    adjacency over the O_b real boundary cells): embeddings, values and log-probs stored by the reference come back."""
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    fx, depth, n_def, T, episodes, mb, seed, emb = _load(path)
    m = MAPPO(_cfg(depth, n_def, T, emb), None, None, "Worker")
    _load_weights(m, fx)
    buf = {k[4:]: torch.from_numpy(fx[k]).cuda() for k in fx.files if k.startswith("buf.")}
    N, E, D, L = n_def, emb, depth, 2
    enc = m.actor.shared_net
    with torch.no_grad():
        for b in range(episodes):
            ob = int(fx["o_counts"][b])
            ha = torch.zeros(L, N, E, device="cuda")
            hc = torch.zeros(L, N, E, device="cuda")
            hist_a, hist_c = buf["actor_historical_embedding"][b], buf["critic_historical_embedding"][b]   # [T+D,N,E]
            for t in range(T):
                graph = ops.GraphBatch(buf["p_state"][b, t].reshape(1, N, 4).contiguous(), buf["e_state"][b, t].reshape(1, 4).contiguous(),
                                       buf["o_state"][b, t, :, :2].reshape(1, -1, 2).contiguous(),
                                       torch.zeros(1, dtype=torch.int32, device="cuda"),
                                       torch.full((1,), ob, dtype=torch.int32, device="cuda"),
                                       ops.pack_bits(buf["p_adj"][b, t].reshape(1, N, N)),
                                       (buf["e_adj"][b, t].reshape(1, N) != 0).to(torch.uint8), ops.pack_bits(buf["o_adj"][b, t].reshape(1, N, -1)))
                hist = []
                for k in range(D):
                    back = k // 2 + 1
                    src = hist_c if k % 2 == 0 else hist_a
                    hist.append((src[t - back + D] if t - back >= 0 else torch.zeros(N, E, device="cuda")).reshape(1, N, E).contiguous())
                emb_a = enc.encode(graph, False, hist)
                fa, ha = m.actor.features(emb_a.view(1, N, E), ha)
                emb_c = enc.encode(graph, True, hist)
                fc, hc = m.critic.features(emb_c.view(1, N, E), hc)
                w_eff, _ = m.critic.head_weight()
                val = torch.nn.functional.linear(fc[0], w_eff, m.critic.Mean.bias)[:, 0]
                logp_all = torch.log_softmax(torch.nn.functional.linear(fa[0], m.actor.Mean.weight, m.actor.Mean.bias), -1)
                lp = logp_all.gather(-1, buf["a_n"][b, t].long().unsqueeze(-1))[:, 0]
                # 1e-5 relative; the absolute floor is 1e-5 of the activations' scale (embeddings of the 128-wide networks reach
                # ~0.5: an element that cancels to 0.03 still carries the rounding of its O(1) summands)
                tol = dict(rtol=1e-5, atol=2e-6 if emb == 32 else 5e-6)
                torch.testing.assert_close(emb_a[0], hist_a[t + D], **tol)
                torch.testing.assert_close(emb_c[0], hist_c[t + D], **tol)
                torch.testing.assert_close(val, buf["v_n"][b, t], **tol)
                torch.testing.assert_close(lp, buf["a_logprob_n"][b, t], **tol)


# ---------------------------------------------------------------------------------------------------------------
# kernels against the pinned torch restatement on random inputs


def _rand_graph(S, N, O, Bo, seed):
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    g = torch.Generator(device="cuda").manual_seed(seed)
    p = torch.rand(S, N, 4, device="cuda", generator=g) * 50
    e = torch.rand(S, 4, device="cuda", generator=g) * 50
    oxy = torch.randint(0, 55, (Bo, O, 2), device="cuda", generator=g).float()
    o_index = torch.randint(0, Bo, (S,), device="cuda", generator=g, dtype=torch.int32)
    o_count = torch.randint(1, O + 1, (Bo,), device="cuda", generator=g, dtype=torch.int32)
    p_adj = (torch.rand(S, N, N, device="cuda", generator=g) < 0.5).float()
    e_adj = (torch.rand(S, N, 1, device="cuda", generator=g) < 0.5).float()
    o_adj = (torch.rand(S, N, O, device="cuda", generator=g) < 0.1).float()
    p_adj[0] = 0                                         # an agent with no neighbour at all: normalised row is zero
    o_adj[1] = 0
    graph = ops.GraphBatch(p, e, oxy, o_index, o_count, ops.pack_bits(p_adj), (e_adj[..., 0] != 0).to(torch.uint8).contiguous(),
                           ops.pack_bits(o_adj))
    return graph, p_adj, e_adj, o_adj


def _ref_message_agg(graph, p_adj, e_adj, o_adj, all_ones, W):
    import torch.nn.functional as F
    p, e = graph.p, graph.e.unsqueeze(1)
    o4 = torch.cat([graph.oxy, torch.zeros_like(graph.oxy)], -1)[graph.o_index.long()]          # [S,O,4]
    if all_ones:
        p_adj, e_adj = torch.ones_like(p_adj), torch.ones_like(e_adj)
        cnt = graph.o_count[graph.o_index.long()]
        o_adj = (torch.arange(graph.O, device="cuda")[None, None, :] < cnt[:, None, None]).float().expand_as(o_adj)
    rel_pp = p.unsqueeze(-2) - p.unsqueeze(-3)
    rel_pe = p.unsqueeze(-2) - e.unsqueeze(-3)
    rel_po = p.unsqueeze(-2) - o4.unsqueeze(-3)
    a0 = torch.cat([rel_pp, rel_pe.expand(*rel_pp.shape[:-1], 4)], -1)
    outs = []
    for (attr, adj, (w, b)) in ((a0, p_adj, W[0]), (rel_pe, e_adj, W[1]), (rel_po, o_adj, W[2])):
        msg = torch.relu(F.linear(attr, w, b))
        outs.append(torch.matmul(F.normalize(adj.unsqueeze(-2), p=1, dim=-1), msg).squeeze(-2))
    return torch.stack(outs, dim=2)


@pytest.mark.parametrize("E,N,O,all_ones", [(128, 8, 176, False), (128, 8, 176, True), (32, 5, 40, False), (64, 33, 70, True)])
def test_message_agg_forward_backward(E, N, O, all_ones):
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    S, Bo = 23, 4
    graph, p_adj, e_adj, o_adj = _rand_graph(S, N, O, Bo, seed=E + N)
    g = torch.Generator(device="cuda").manual_seed(1)
    W = [(torch.randn(E, k, device="cuda", generator=g) * 0.3, torch.randn(E, device="cuda", generator=g) * 0.1) for k in (8, 4, 4)]
    leaves = [t.clone().requires_grad_(True) for pair in W for t in pair]
    out = ops.message_agg(graph, all_ones, *leaves)
    refl = [t.clone().requires_grad_(True) for pair in W for t in pair]
    ref = _ref_message_agg(graph, p_adj, e_adj, o_adj, all_ones, [(refl[0], refl[1]), (refl[2], refl[3]), (refl[4], refl[5])])
    torch.testing.assert_close(out, ref, rtol=1e-5, atol=1e-5)
    dout = torch.randn(out.shape, device="cuda", generator=g)
    out.backward(dout)
    ref.backward(dout)
    for a, b in zip(leaves, refl):
        torch.testing.assert_close(a.grad, b.grad, rtol=1e-4, atol=1e-4 * float(b.grad.abs().max()))


def test_fcra_agg_and_strided_history():
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    import torch.nn.functional as F
    T, B, N, E, D = 6, 5, 7, 128, 3
    g = torch.Generator(device="cuda").manual_seed(2)
    arena = torch.randn(T + D, B, N, E, device="cuda", generator=g)
    adj = (torch.rand(T * B, N, N, device="cuda", generator=g) < 0.4).float()
    bits = ops.pack_bits(adj)
    for k in range(D):
        hist = arena[D - 1 - k: D - 1 - k + T].reshape(T * B, N, E)
        ref = torch.matmul(F.normalize(adj, p=1, dim=-1), hist)
        got = ops.fcra_agg(arena[D - 1 - k:], bits, False, T * B, N, E, N * E, E)
        torch.testing.assert_close(got, ref, rtol=1e-5, atol=1e-5)
        got1 = ops.fcra_agg(arena[D - 1 - k:], bits, True, T * B, N, E, N * E, E)
        torch.testing.assert_close(got1, hist.mean(1, keepdim=True).expand(-1, N, -1), rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("E,T,R", [(128, 9, 37), (32, 4, 5), (128, 1, 64), (128, 23, 333)])
def test_gru_layer_forward_backward(E, T, R):
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    from oracle import policy_ref
    g = torch.Generator(device="cuda").manual_seed(3)
    mk = lambda *s: (torch.randn(*s, device="cuda", generator=g) * 0.2)
    w = {"G.weight_ih_l0": mk(3 * E, E), "G.weight_hh_l0": mk(3 * E, E), "G.bias_ih_l0": mk(3 * E), "G.bias_hh_l0": mk(3 * E)}
    x, h0 = mk(T, R, E), mk(R, E)
    a = [t.clone().requires_grad_(True) for t in (x, h0, w["G.weight_ih_l0"], w["G.weight_hh_l0"], w["G.bias_ih_l0"], w["G.bias_hh_l0"])]
    out = ops._GRULayer.apply(*a)
    b = [t.clone().requires_grad_(True) for t in (x, h0, w["G.weight_ih_l0"], w["G.weight_hh_l0"], w["G.bias_ih_l0"], w["G.bias_hh_l0"])]
    wr = {"G.weight_ih_l0": b[2], "G.weight_hh_l0": b[3], "G.bias_ih_l0": b[4], "G.bias_hh_l0": b[5]}
    ref, _ = policy_ref.gru_layer(wr, "G", 0, b[0], b[1])
    # atol: 23 recurrent steps of fp32 GEMMs in a different summation order (3xTF32 tensor-core vs library sgemm)
    torch.testing.assert_close(out, ref, rtol=1e-5, atol=5e-6)
    # and against torch.nn.GRU itself (the module the reference uses)
    gru = torch.nn.GRU(E, E, 1).cuda()
    torch.backends.cudnn.allow_tf32 = False               # cuDNN's RNN path would otherwise round the GEMMs to TF32
    with torch.no_grad():
        gru.weight_ih_l0.copy_(w["G.weight_ih_l0"]); gru.weight_hh_l0.copy_(w["G.weight_hh_l0"])
        gru.bias_ih_l0.copy_(w["G.bias_ih_l0"]); gru.bias_hh_l0.copy_(w["G.bias_hh_l0"])
        lib_out, _ = gru(x, h0.unsqueeze(0))
    torch.testing.assert_close(out.detach(), lib_out, rtol=1e-4, atol=2e-5)
    dout = mk(T, R, E)
    out.backward(dout)
    ref.backward(dout)
    for u, v in zip(a, b):
        torch.testing.assert_close(u.grad, v.grad, rtol=1e-4, atol=1e-5 * max(1.0, float(v.grad.abs().max())))


@pytest.mark.parametrize("E,value_clip", [(128, True), (32, True), (128, False)])
def test_ppo_head_forward_backward(E, value_clip):
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    from oracle import policy_ref
    R, A = 301, 9
    g = torch.Generator(device="cuda").manual_seed(4)
    rn = lambda *s: torch.randn(*s, device="cuda", generator=g)
    feat_a, feat_c = rn(R, E), rn(R, E)
    Wa, ba, Wc, bc = rn(A, E) * 0.4, rn(A) * 0.1, rn(1, E) * 0.3, rn(1) * 0.1
    Wa[0] *= 6.0                      # some rows become near-deterministic: exercises the probability clamp
    u = torch.nn.functional.normalize(rn(1), dim=0)
    action = torch.randint(0, A, (R,), device="cuda", generator=g).float()
    old_logp = torch.log_softmax(rn(R, A), -1)[:, 0] * 0.05 + torch.log(torch.tensor(1.0 / A))
    adv, v_old, v_t = rn(R), rn(R) * 0.2, rn(R) * 0.2
    active = (torch.rand(R, device="cuda", generator=g) < 0.9).float()
    la = [t.clone().requires_grad_(True) for t in (feat_a, feat_c, Wa, ba, Wc, bc)]
    out = ops.ppo_head(*la, u, action, old_logp, adv, v_old if value_clip else None, v_t, active, 0.05, 0.05)
    (out[0] + out[1]).backward()
    # restatement: Categorical(probs=softmax) exactly as torch.distributions does it
    lb = [t.clone().requires_grad_(True) for t in (feat_a, feat_c, Wa, ba, Wc, bc)]
    prob = torch.softmax(torch.nn.functional.linear(lb[0], lb[2], lb[3]), -1)
    dist = torch.distributions.Categorical(probs=prob)
    logp, ent = dist.log_prob(action), dist.entropy()
    w = {"critic.Mean.weight_orig": lb[4], "critic.Mean.weight_u": u}
    Weff, _, _ = policy_ref.critic_head_weight(w)
    val = torch.nn.functional.linear(lb[1], Weff, lb[5])[:, 0]
    la_ref, lc_ref = policy_ref.ppo_losses(logp[None], ent[None], val[None], {"active": active[None], "a_logprob_n": old_logp[None],
                                                                            "v_n": torch.cat([v_old[None], v_old[None, -1:]], 1)},
                                           adv[None], v_t[None], use_value_clip=value_clip)
    torch.testing.assert_close(out[2], logp, rtol=1e-5, atol=2e-6)
    torch.testing.assert_close(out[3], ent, rtol=1e-5, atol=2e-6)
    torch.testing.assert_close(out[4], val, rtol=1e-5, atol=2e-6)
    assert abs(float(out[0]) - float(la_ref)) < 1e-5 and abs(float(out[1]) - float(lc_ref)) < 1e-5
    (la_ref + lc_ref).backward()
    for a_, b_ in zip(la, lb):
        torch.testing.assert_close(a_.grad, b_.grad, rtol=1e-4, atol=1e-6 + 1e-4 * float(b_.grad.abs().max()))


def test_act_head_sampling_and_argmax():
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    R, E, A = 4096, 128, 9
    g = torch.Generator(device="cuda").manual_seed(5)
    feat = torch.randn(R, E, device="cuda", generator=g)
    Wa, ba = torch.randn(A, E, device="cuda", generator=g) * 0.2, torch.randn(A, device="cuda", generator=g) * 0.1
    wc, bc = torch.randn(E, device="cuda", generator=g) * 0.1, torch.randn(1, device="cuda", generator=g)
    prob = torch.softmax(torch.nn.functional.linear(feat, Wa, ba), -1)
    a, af, lp, val = ops.act_head(feat, feat, Wa, ba, wc, bc, seed=9, t=3, deterministic=True)
    assert torch.equal(a.long(), prob.argmax(-1)) and torch.equal(af, a.float())
    torch.testing.assert_close(val, feat @ wc + bc, rtol=1e-5, atol=1e-5)
    a2, _, lp2, _ = ops.act_head(feat, None, Wa, ba, None, None, seed=9, t=3, deterministic=False)
    torch.testing.assert_close(lp2, torch.log(prob.gather(-1, a2.long()[:, None])[:, 0]), rtol=1e-5, atol=2e-6)
    a3, _, _, _ = ops.act_head(feat, None, Wa, ba, None, None, seed=9, t=3, deterministic=False)
    assert torch.equal(a2, a3)                                            # counter RNG: same key, same draw
    a4, _, _, _ = ops.act_head(feat, None, Wa, ba, None, None, seed=9, t=4, deterministic=False)
    assert not torch.equal(a2, a4)
    # sampled frequencies follow the probabilities (chi-square-ish bound on the pooled histogram)
    many = torch.stack([ops.act_head(feat, None, Wa, ba, None, None, seed=s, t=0, deterministic=False)[0] for s in range(64)])
    freq = torch.stack([(many == k).float().mean() for k in range(A)])
    torch.testing.assert_close(freq, prob.mean(0), rtol=0.05, atol=0.005)


def test_clip_and_adam_match_torch():
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    n = 614538                                            # parameter count of the depth-3 model (SURVEY 8a)
    g = torch.Generator(device="cuda").manual_seed(6)
    p = torch.randn(n, device="cuda", generator=g)
    grad = torch.randn(n, device="cuda", generator=g) * 0.1
    ref_p = torch.nn.Parameter(p.clone())
    ref_p.grad = grad.clone()
    opt = torch.optim.Adam([ref_p], lr=5e-4, eps=1e-5)
    m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    mine, gmine = p.clone(), grad.clone()
    for step in range(1, 4):
        tn = torch.nn.utils.clip_grad_norm_([ref_p], 5.0)
        got = ops.clip_grad_norm_(gmine, 5.0)
        assert abs(float(got) - float(tn)) <= 1e-5 * float(tn)
        torch.testing.assert_close(gmine, ref_p.grad, rtol=1e-6, atol=1e-8)
        opt.step()
        ops.adam_step_(mine, gmine, m, v, 5e-4, step)
        torch.testing.assert_close(mine, ref_p.data, rtol=1e-6, atol=1e-7)
        ref_p.grad.mul_(0.5).add_(0.01)
        gmine.mul_(0.5).add_(0.01)
    small = torch.full((10,), 1e-3, device="cuda")
    before = small.clone()
    ops.clip_grad_norm_(small, 5.0)                       # below the threshold: untouched
    assert torch.equal(small, before)


def test_batched_rollout_then_train_end_to_end():
    """run_episode for a batch of envs on the GPU (observe -> encoder -> GRU -> heads -> env kernels), checked for
    self-consistency against a teacher-forced replay of what it stored, then fed to train()."""
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena
    import bench
    B, N, M, T, E, D = 12, 4, 3, 14, 32, 3
    cfg = _cfg(D, N, T, E)
    torch.manual_seed(0)
    m = MAPPO(cfg, B, 5, "Learner")
    wl = bench.host_workload(cfg, B, M, seed=3)
    env = BatchedPursuitEnv(cfg, B, num_maps=M)
    env.set_maps(wl["grids"], wl["inflated"])
    env.set_state(wl["p_state"], wl["e_state"], wl["target"], wl["map_id"], time_step=0)
    env.set_target_tape(wl["tape"])
    env.start_episode()
    arena = RolloutArena(env.params, B, T, env.device)
    tb = m.rollout_batched(env, arena, T, seed=11)
    torch.cuda.synchronize()
    assert int(env.evader_status.max()) == 0 and (env.time_step == T).all()
    assert tb.p.shape == (T, B, N, 4) and tb.hist_a.shape == (T + D, B, N, E) and tb.v.shape == (T + 1, B, N)
    assert torch.equal(tb.a, arena.a_n) and (tb.a >= 0).all() and (tb.a <= 8).all()
    assert (tb.hist_a[:D] == 0).all() and tb.hist_a[D:].abs().sum() > 0 and torch.isfinite(tb.v).all()
    # teacher-forced replay of step t from the stored observations (rollout-mode history, O_b critic slots)
    oxy = env.boundary_xy.float()
    o_count = torch.clamp(env.boundary_count, max=env.O)
    enc = m.actor.shared_net
    with torch.no_grad():
        ha = torch.zeros(2, B * N, E, device="cuda")
        hc = torch.zeros(2, B * N, E, device="cuda")
        for t in range(T):
            graph = ops.GraphBatch(tb.p[t].contiguous(), tb.e[t].contiguous(), oxy, env.map_id, o_count,
                                   tb.p_adj_bits[t].contiguous(), tb.e_adj[t].contiguous(), tb.o_adj_bits[t].contiguous())
            hist = []
            for k in range(D):
                back, src = k // 2 + 1, (tb.hist_c if k % 2 == 0 else tb.hist_a)
                hist.append(src[t - back + D] if t - back >= 0 else torch.zeros(B, N, E, device="cuda"))
            ea = enc.encode(graph, False, hist)
            fa, ha = m.actor.features(ea.view(1, B * N, E), ha)
            ec = enc.encode(graph, True, hist)
            fc, hc = m.critic.features(ec.view(1, B * N, E), hc)
            w_eff, _ = m.critic.head_weight()
            torch.testing.assert_close(ea, tb.hist_a[t + D], rtol=1e-6, atol=1e-6)
            torch.testing.assert_close(ec, tb.hist_c[t + D], rtol=1e-6, atol=1e-6)
            val = torch.nn.functional.linear(fc[0], w_eff, m.critic.Mean.bias).view(B, N)
            torch.testing.assert_close(val, tb.v[t], rtol=1e-5, atol=1e-6)
            lp = torch.log_softmax(torch.nn.functional.linear(fa[0], m.actor.Mean.weight, m.actor.Mean.bias), -1)
            torch.testing.assert_close(lp.gather(-1, tb.a[t].long().view(-1, 1)).view(B, N), tb.logp[t], rtol=1e-5, atol=2e-6)
    # training on the rollout: first-epoch ratios are NOT 1 in this algorithm (rollout != training forward, SURVEY 7.4-5)
    before = [p.detach().clone() for p in m.ac_parameters]
    objC, objA, ag, cg = m.train(tb, total_steps=B * T)
    assert np.isfinite(objC) and np.isfinite(objA)
    assert all(g is not None and np.isfinite(g).all() for g in ag + cg)
    assert float(m.ac_optimizer.flat_grad.norm()) <= 5.0 + 1e-4
    m.ac_optimizer.step()
    assert any(not torch.equal(a, b) for a, b in zip(before, m.ac_parameters))


def test_explore_env_reference_signature():
    """MAPPO.explore_env(env, n) with the single-env facade returns (float, ReplayBuffer, steps) in the reference's
    buffer layout, and the result trains."""
    import random
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import Pursuit_Env
    from distributed_multi_agent_reinforcement_learning_b200.replay_buffer import BigBuffer
    N, T, E, D = 4, 9, 32, 1
    cfg = _cfg(D, N, T, E)
    random.seed(4); np.random.seed(4); torch.manual_seed(4)
    env = Pursuit_Env(cfg)
    worker = MAPPO(cfg, None, None, "Worker")
    big = BigBuffer()
    for _ in range(2):
        r, buf, steps = worker.explore_env(env, 1)
        assert steps == T and isinstance(r, float)
        big.concat_buffer(buf)
    O = cfg.map.num_max_obstacle
    shapes = {k: tuple(v.shape) for k, v in big.buffer.items()}
    assert shapes == dict(p_state=(2, T, N, 4), e_state=(2, T, 1, 4), o_state=(2, T, O, 4), p_adj=(2, T, N, N),
                          e_adj=(2, T, N, 1), o_adj=(2, T, N, O), actor_historical_embedding=(2, T + D, N, E),
                          critic_historical_embedding=(2, T + D, N, E), v_n=(2, T + 1, N), a_n=(2, T, N),
                          a_logprob_n=(2, T, N), r=(2, T, N), active=(2, T, N))
    assert (big.buffer["p_adj"][..., 1] == 1).all() and (big.buffer["active"] == 1).all()
    assert worker.reward_norm.running_ms.n == 2 * T            # the estimate persists across episodes
    learner = MAPPO(cfg, 2, 1, "Learner")
    learner.actor.set_weights(worker.actor.get_weights())
    learner.critic.set_weights(worker.critic.get_weights())
    objC, objA, ag, cg = learner.train(big, 2 * T)
    assert np.isfinite(objC) and np.isfinite(objA) and len(ag) == len(list(learner.actor.parameters()))


def test_checkpoint_file_set_round_trip(tmp_path):
    """The reference driver's eight-file checkpoint set (main.py:149-169) + recorder.npy, written and read back."""
    from distributed_multi_agent_reinforcement_learning_b200 import checkpoint
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    cfg = _cfg(1, 4, 5, 32)
    torch.manual_seed(1)
    a = MAPPO(cfg, None, None, "Worker")
    checkpoint.save_checkpoint(a, str(tmp_path), recorder=[(10, 1.0, 0.5, 0.9, 0.1, -0.1)])
    checkpoint.save_checkpoint(a, str(tmp_path), final=True)
    names = sorted(os.listdir(tmp_path))
    for n in checkpoint.FILES:
        assert f"{n}.pth" in names and f"{n}_final.pth" in names and f"{n}.state_dict.pth" in names
    assert np.load(os.path.join(tmp_path, "recorder.npy")).shape == (1, 6)
    torch.manual_seed(2)
    b = MAPPO(cfg, None, None, "Worker")
    assert not torch.equal(a.actor.GRU.weight_hh_l0, b.actor.GRU.weight_hh_l0)
    assert sorted(checkpoint.load_checkpoint(b, str(tmp_path))) == sorted(checkpoint.FILES)
    for (k, u), (_, v) in zip(a.actor.state_dict().items(), b.actor.state_dict().items()):
        assert torch.equal(u, v), k
    for (k, u), (_, v) in zip(a.critic.state_dict().items(), b.critic.state_dict().items()):
        assert torch.equal(u, v), k
    # pickled whole module, as evaluator.py:329-330 consumes it
    sd = torch.load(os.path.join(tmp_path, "actor.pth"), weights_only=False).state_dict()
    assert list(sd.keys()) == list(a.actor.state_dict().keys())


def _train_grads(m, buf, total_steps, **kw):
    trace = {}
    m.train(_Big(buf), total_steps, return_numpy=False, trace=trace, **kw)
    return m.ac_optimizer.flat_grad.clone(), trace


def test_shuffled_minibatches_through_the_gather_kernel():
    """algo.shuffle_minibatches / train(permutation=...) (north star part 4; the reference is sequential, :665, so the default is
    off): with the identity permutation the gathered epoch equals the sequential epoch bit for bit, and with a random permutation
    it equals the sequential epoch on the correspondingly permuted buffer."""
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    path = os.path.join(GOLDEN_DIR, "algo_d1_n8_e128.npz")
    fx, depth, n_def, T, episodes, mb, seed, emb = _load(path)
    m = MAPPO(_cfg(depth, n_def, T, emb), episodes, mb, "Learner")
    _load_weights(m, fx)
    u0, v0 = m.critic.Mean.weight_u.clone(), m.critic.Mean.weight_v.clone()

    def reset_sn():          # the power-iteration buffers advance on every critic forward: same start for every run
        m.critic.Mean.weight_u.copy_(u0)
        m.critic.Mean.weight_v.copy_(v0)
    buf = {k[4:]: torch.from_numpy(fx[k]) for k in fx.files if k.startswith("buf.")}
    steps = int(fx["total_steps"])
    # the gathered minibatch IS the sliced minibatch, tensor for tensor, bit for bit
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import TrainBatch
    tb = TrainBatch.from_reference({k: v.cuda() for k, v in buf.items()}, depth)
    sliced = tb.minibatch(1, 4)
    gathered, _ = tb.minibatch_indexed(torch.arange(1, 4, device="cuda"))
    for key in TrainBatch.KEYS + ("oxy", "o_count_train"):
        assert torch.equal(getattr(sliced, key), getattr(gathered, key)), key
    g_seq, tr_seq = _train_grads(m, buf, steps)
    reset_sn()
    g_id, tr = _train_grads(m, buf, steps, permutation=list(range(episodes)))
    assert torch.equal(tr["permutation"].cpu(), torch.arange(episodes))
    for a_, b_ in zip(tr_seq["mb"], tr["mb"]):            # identity permutation: the forward passes are bit-identical ...
        assert torch.equal(a_["logp"], b_["logp"]) and torch.equal(a_["ent"], b_["ent"]) and torch.equal(a_["val"], b_["val"])
    # ... and so are the gradients: both epochs feed the same minibatches to kernels that reduce in a fixed order
    assert torch.equal(g_id, g_seq)
    perm = [3, 0, 4, 2, 1]
    reset_sn()
    g_perm, _ = _train_grads(m, buf, steps, permutation=perm)
    reset_sn()
    g_ref, _ = _train_grads(m, {k: v[perm] for k, v in buf.items()}, steps)
    # (the advantage statistics are summed in a different env order in the two runs: equal up to fp64 rounding of the mean / std)
    torch.testing.assert_close(g_perm, g_ref, rtol=1e-5, atol=1e-7)
    assert not torch.allclose(g_perm, g_seq, rtol=1e-3, atol=1e-6)
    # the config switch draws a seeded device permutation
    reset_sn()
    _, tr2 = _train_grads(m, buf, steps, shuffle=True, shuffle_seed=11)
    assert sorted(tr2["permutation"].cpu().tolist()) == list(range(episodes))


@pytest.mark.parametrize("depth", [1, 3])
def test_reference_quirks_off_makes_rollout_and_training_forward_agree(depth):
    """SURVEY 7.4-5: in the reference the rollout forward differs from the training forward at identical weights (the history list that
    actor and critic alias during the rollout; the critic's all-ones obstacle adjacency over the 76 padded slots in training), so PPO
    ratios are != 1 on the first epoch.  `MAPPO(..., reference_quirks=False)` is the self-consistent variant (never the parity
    default): the training forward then reproduces the rollout's log-probs and values, and with the quirks on it does not."""
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena
    B, N, T = 16, 8, 12
    cfg = default_config(env__num_defender=N, env__max_steps=T, algo__depth=depth, algo__learner_device="cuda", algo__worker_device="cuda")
    out = {}
    for quirks in (False, True):
        torch.manual_seed(7)
        m = MAPPO(cfg, B, B // 2, "Learner", reference_quirks=quirks)
        with torch.no_grad():
            for p in m.ac_parameters:
                if p.dim() == 1:
                    p.add_(0.05 * torch.randn_like(p))
        env = BatchedPursuitEnv(cfg, B, num_maps=4)
        env.reset(seed=13)
        arena = RolloutArena(env.params, B, T, env.device)
        tb = m.rollout_batched(env, arena, T, seed=3)
        if not quirks:                                        # the env-group pipelines give the same episode
            snap_logp, snap_v = tb.logp.clone(), tb.v.clone()
            env.reset(seed=13)
            tb = m.rollout_batched(env, arena, T, seed=3, pipelines=2)
            assert torch.equal(tb.logp, snap_logp) and torch.equal(tb.v, snap_v)
        trace = {}
        m.train(tb, B * T, return_numpy=False, trace=trace)
        logp = torch.cat([t["logp"] for t in trace["mb"]], dim=1)
        val = torch.cat([t["val"] for t in trace["mb"]], dim=1)
        out[quirks] = (float((logp - tb.logp).abs().max()), float((val - tb.v[:-1]).abs().max()))
        if not quirks:
            torch.testing.assert_close(logp, tb.logp, rtol=1e-5, atol=2e-5)
            torch.testing.assert_close(val, tb.v[:-1], rtol=1e-5, atol=2e-5)
    assert out[True][0] > 1e-3 and out[True][1] > 1e-3, out      # the reference's behaviour: the two forwards disagree
