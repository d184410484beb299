"""GPU parity of the fused rollout-step kernel (csrc/policy_fused.cu: encoder + GRU + heads of actor and critic in one
launch, tcgen05 3xTF32) against
  (a) the reference's OWN rollout buffer at the production width E=128 (tests/golden/rollout128_*.npz, recorded by executing
      the unmodified reference, oracle/gen_golden_rollout128.py), teacher-forced on the reference's actions, and
  (b) the unfused kernel path (policy_ops) on live env observations at ragged / multi-tile shapes.
Tolerance: 1e-5 relative + 2e-5 absolute on embeddings, values and log-probs (north_star: 1e-5 forward activations)."""
import glob
import os
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import GOLDEN_DIR

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

FIXTURES = sorted(glob.glob(os.path.join(GOLDEN_DIR, "rollout128_*.npz")))


def _cfg(depth, n_def, T):
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    return default_config(env__num_defender=n_def, env__max_steps=T, algo__depth=depth, algo__embedding_dim=128,
                          algo__rnn_hidden_dim=128, algo__learner_device="cuda", algo__worker_device="cuda")


def _words(packed_bytes, n_bits):
    """np.packbits(..., bitorder='little') bytes [..., nb] -> int32 words [..., ceil(n_bits/32)]."""
    nw = (n_bits + 31) // 32
    pad = nw * 4 - packed_bytes.shape[-1]
    b = np.pad(packed_bytes, [(0, 0)] * (packed_bytes.ndim - 1) + [(0, pad)])
    return np.ascontiguousarray(b).view(np.uint32).astype(np.int64).astype(np.uint32).view(np.int32).reshape(*packed_bytes.shape[:-1], nw)


@pytest.mark.parametrize("variant", [1, 3], ids=["one_cta_per_sm", "actor_critic_pair_cta"])
@pytest.mark.parametrize("path", FIXTURES, ids=[os.path.basename(p)[:-4] for p in FIXTURES])
def test_fused_step_reproduces_reference_rollout_buffer(path, variant):
    from distributed_multi_agent_reinforcement_learning_b200.fused_policy import FusedRolloutStep
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    fx = np.load(path)
    depth, N, T, episodes, seed, E = (int(v) for v in fx["meta"])
    torch.manual_seed(seed)
    m = MAPPO(_cfg(depth, N, T), None, None, "Worker")       # same seed -> the reference's initial weights
    for net, mod in (("actor", m.actor), ("critic", m.critic)):
        for k, v in mod.state_dict().items():
            assert abs(float(v.double().abs().sum()) - float(fx[f"wsum.{net}.{k}"])) <= 1e-9 * max(1.0, float(fx[f"wsum.{net}.{k}"])), (net, k)
    w_eff, _ = m.critic.head_weight()
    fused = FusedRolloutStep(m, w_eff)
    B, O, dev = episodes, fx["o_xy"].shape[1], "cuda"
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    eng = SimpleNamespace(B=B, N=N, O=O, map_id=torch.arange(B, dtype=torch.int32, device=dev))
    oxy, o_count = cu(fx["o_xy"].astype(np.int32)), cu(fx["o_counts"].astype(np.int32))
    hist_a, hist_c = cu(fx["hist_a"]), cu(fx["hist_c"])                 # [B,T+D,N,E]
    ha, hc = torch.zeros(2, B * N, E, device=dev), torch.zeros(2, B * N, E, device=dev)
    emb_a, emb_c = torch.empty(B, N, E, device=dev), torch.empty(B, N, E, device=dev)
    logp, value = torch.empty(B, N, device=dev), torch.empty(B, N, device=dev)
    p_adj, o_adj = _words(fx["p_adj"], N), _words(fx["o_adj"], O)
    for t in range(T):
        eng.p_state = cu(fx["p_state"][:, t].astype(np.float64))
        eng.e_state = cu(fx["e_state"][:, t, 0].astype(np.float64))
        eng.p_adj_bits, eng.e_adj, eng.o_adj_bits = cu(p_adj[:, t]), cu(fx["e_adj"][:, t]), cu(o_adj[:, t])
        hist = []
        for k in range(depth):                               # one aliased list for both networks (:750-752)
            back, src = k // 2 + 1, (hist_c if k % 2 == 0 else hist_a)
            hist.append(src[:, t - back + depth].contiguous() if t - back >= 0 else None)
        action = cu(fx["a_n"][:, t].astype(np.int32))
        fused.step(eng, oxy, o_count, t, 0, False, hist, hist, emb_a, emb_c, ha, hc, action, logp, value, force_action=True, variant=variant)
        torch.cuda.synchronize()
        tol = dict(rtol=1e-5, atol=2e-5)
        torch.testing.assert_close(emb_a, hist_a[:, t + depth], **tol)
        torch.testing.assert_close(emb_c, hist_c[:, t + depth], **tol)
        torch.testing.assert_close(value, cu(fx["v_n"][:, t]), **tol)
        torch.testing.assert_close(logp, cu(fx["a_logprob_n"][:, t]), **tol)


@pytest.mark.parametrize("variant", [1, 3], ids=["one_cta_per_sm", "actor_critic_pair_cta"])
@pytest.mark.parametrize("B,N,D,steps", [(300, 8, 1, 4), (70, 5, 3, 5), (9, 16, 2, 3), (7, 20, 1, 2), (45, 4, 1, 3)])
def test_fused_step_matches_unfused_kernels(B, N, D, steps, variant):
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    from distributed_multi_agent_reinforcement_learning_b200.fused_policy import FusedRolloutStep
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena
    import bench
    E, M, T = 128, 4, steps
    cfg = _cfg(D, N, T)
    torch.manual_seed(5)
    m = MAPPO(cfg, B, max(1, B // 4), "Learner")
    with torch.no_grad():                                    # biases are zero-initialised: make them matter
        for p in m.ac_parameters:
            if p.dim() == 1:
                p.add_(0.05 * torch.randn_like(p))
    wl = bench.host_workload(cfg, B, M, seed=9)
    env = BatchedPursuitEnv(cfg, B, num_maps=M)
    env.set_maps(wl["grids"], wl["inflated"])
    env.set_state(wl["p_state"], wl["e_state"], wl["target"], wl["map_id"], time_step=0)
    env.set_target_tape(wl["tape"])
    env.start_episode()
    arena = RolloutArena(env.params, B, T, env.device)
    dev = env.device
    w_eff, _ = m.critic.head_weight()
    fused = FusedRolloutStep(m, w_eff)
    oxy_i = env.boundary_xy.contiguous()
    oxy_f = oxy_i.float().contiguous()
    o_count = torch.clamp(env.boundary_count, max=env.O).contiguous()
    enc = m.actor.shared_net
    ha = 0.1 * torch.randn(2, B * N, E, device=dev)
    hc = 0.1 * torch.randn(2, B * N, E, device=dev)
    prev = [0.3 * torch.randn(B, N, E, device=dev) for _ in range(D)]
    hist_in = [prev[k] if k != 1 else None for k in range(D)]            # one zero (None) slot when D >= 2
    tol = dict(rtol=1e-5, atol=2e-5)
    with torch.no_grad():
        for t in range(steps):
            env.observe()
            graph = ops.GraphBatch(env.p_state.float(), env.e_state.float(), oxy_f, env.map_id, o_count, env.p_adj_bits,
                                   env.e_adj, env.o_adj_bits)
            hist_ref = [h if h is not None else torch.zeros(B, N, E, device=dev) for h in hist_in]
            ea = enc.encode(graph, False, hist_ref)
            fa, ha_ref = m.actor.features(ea.view(1, B * N, E), ha)
            ec = enc.encode(graph, True, hist_ref)
            fc, hc_ref = m.critic.features(ec.view(1, B * N, E), hc)
            a_ref, _, lp_ref, v_ref = ops.act_head(fa[0], fc[0], m.actor.Mean.weight, m.actor.Mean.bias, w_eff.reshape(E).contiguous(),
                                                   m.critic.Mean.bias, 77, t, False)
            ha_f, hc_f = ha.clone(), hc.clone()
            emb_a, emb_c = torch.empty(B, N, E, device=dev), torch.empty(B, N, E, device=dev)
            act, logp, value = (torch.zeros(B, N, dtype=torch.int32, device=dev), torch.empty(B, N, device=dev),
                                torch.empty(B, N, device=dev))
            fused.step(env, oxy_i, o_count, t, 77, False, hist_in, hist_in, emb_a, emb_c, ha_f, hc_f, act, logp, value, variant=variant)
            torch.cuda.synchronize()
            torch.testing.assert_close(emb_a, ea, **tol)
            torch.testing.assert_close(emb_c, ec, **tol)
            torch.testing.assert_close(ha_f, ha_ref, **tol)
            torch.testing.assert_close(hc_f, hc_ref, **tol)
            torch.testing.assert_close(value.view(-1), v_ref, **tol)
            same = (act.view(-1) == a_ref)
            assert same.float().mean() > 0.995, float(same.float().mean())   # inverse-CDF ties at 1e-6 may flip a sample
            torch.testing.assert_close(logp.view(-1)[same], lp_ref[same], **tol)
            # teacher forcing on the unfused path's actions
            ha_g, hc_g = ha.clone(), hc.clone()
            forced = a_ref.view(B, N).clone()
            fused.step(env, oxy_i, o_count, t, 77, False, hist_in, hist_in, emb_a, emb_c, ha_g, hc_g, forced, logp, value,
                       force_action=True, variant=variant)
            torch.testing.assert_close(logp.view(-1), lp_ref, **tol)
            # critic-only launch (bootstrap value)
            hc_h, val2 = hc.clone(), torch.empty(B, N, device=dev)
            fused.step(env, oxy_i, o_count, t, 77, False, hist_in, hist_in, emb_a, emb_c, ha_g, hc_h, None, None, val2,
                       nets=("critic",), variant=1)
            if variant == 3:      # the single-network launch runs the one-chain kernel: same products, but the value's 128-term dot is summed in another order
                torch.testing.assert_close(val2, value, rtol=1e-6, atol=2e-7)
            else:
                torch.testing.assert_close(val2, value, rtol=0, atol=0)
            ha, hc = ha_ref, hc_ref
            hist_in = [ec.view(B, N, E)] + hist_in[:-1] if D > 1 else [ec.view(B, N, E)]
            env.rollout_closed(arena, 1, t0=t, action_tape=a_ref.view(1, B, N).contiguous(), env_t0=t)


def test_rollout_batched_fused_equals_unfused_rollout():
    """MAPPO.rollout_batched with the fused step vs the unfused kernel path from the same initial state and seed."""
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena
    import bench
    B, N, M, T, D = 20, 4, 3, 12, 2
    cfg = _cfg(D, N, T)
    torch.manual_seed(2)
    m = MAPPO(cfg, B, 5, "Learner")
    wl = bench.host_workload(cfg, B, M, seed=4)
    env = BatchedPursuitEnv(cfg, B, num_maps=M)
    env.set_maps(wl["grids"], wl["inflated"])
    env.set_state(wl["p_state"], wl["e_state"], wl["target"], wl["map_id"], time_step=0)
    env.set_target_tape(wl["tape"])
    env.start_episode()
    snap = env.snapshot()
    out = []
    for fused in (True, False):
        env.restore(snap)
        arena = RolloutArena(env.params, B, T, env.device)
        tb = m.rollout_batched(env, arena, T, seed=3, use_fused=fused)
        torch.cuda.synchronize()
        out.append((tb, arena.raw_reward.clone(), env.p_state.clone()))
    (f, rf, pf), (u, ru, pu) = out
    assert torch.equal(f.a, u.a) and torch.equal(rf, ru) and torch.equal(pf, pu)
    tol = dict(rtol=1e-4, atol=5e-5)
    torch.testing.assert_close(f.hist_a, u.hist_a, **tol)
    torch.testing.assert_close(f.hist_c, u.hist_c, **tol)
    torch.testing.assert_close(f.v, u.v, **tol)
    torch.testing.assert_close(f.logp, u.logp, **tol)
    objC, objA, _, _ = m.train(f, total_steps=B * T)
    assert np.isfinite(objC) and np.isfinite(objA)


@pytest.mark.parametrize("N,D", [(8, 1), (5, 2)])
def test_rollout_pipelines_give_identical_episodes(N, D):
    """Env-group pipelines (independent sub-batches on their own streams) must not change anything: actions, rewards, states,
    embeddings, values, log-probs and Welford state are bit-identical for 1, 3 and 4 pipelines (the sampling RNG is keyed by the
    global row; rows do not interact across envs)."""
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena
    import bench
    B, M, T = 50, 5, 23
    cfg = _cfg(D, N, T)
    torch.manual_seed(2)
    m = MAPPO(cfg, B, 5, "Learner")
    wl = bench.host_workload(cfg, B, M, seed=6)
    env = BatchedPursuitEnv(cfg, B, num_maps=M)
    env.set_maps(wl["grids"], wl["inflated"])
    env.set_state(wl["p_state"], wl["e_state"], wl["target"], wl["map_id"], time_step=0)
    env.set_target_tape(wl["tape"])
    env.start_episode()
    snap = env.snapshot()
    out = []
    for pipes in (1, 3, 4):
        env.restore(snap)
        arena = RolloutArena(env.params, B, T, env.device)
        tb = m.rollout_batched(env, arena, T, seed=9, pipelines=pipes)
        torch.cuda.synchronize()
        assert int(env.evader_status.max().item()) == 0
        out.append([tb.a.clone(), tb.logp.clone(), tb.v.clone(), tb.hist_a.clone(), tb.hist_c.clone(), arena.raw_reward.clone(),
                    arena.r.clone(), env.p_state.clone(), env.e_state.clone(), env.wf_mean.clone(), env.path_len.clone()])
    for other in out[1:]:
        for a, b in zip(out[0], other):
            assert torch.equal(a, b)


def test_fused_step_full_size_env_permutation_equivariance():
    """BASELINE config 2 size (4096 envs x 8 pursuers): envs are independent, so permuting the envs of the batch must permute every
    output of the fused step bit for bit (embeddings, hidden states, values, arg-max actions, log-probs) - whatever tile, CTA or
    warp an env lands in.  Also checks that the outputs are finite and that the critic does not depend on the adjacency."""
    from distributed_multi_agent_reinforcement_learning_b200.fused_policy import FusedRolloutStep
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    B, N, D, E = 4096, 8, 1, 128
    cfg = _cfg(D, N, 150)
    torch.manual_seed(11)
    m = MAPPO(cfg, B, B // 10, "Learner")
    with torch.no_grad():
        for p in m.ac_parameters:
            if p.dim() == 1:
                p.add_(0.05 * torch.randn_like(p))
    env = BatchedPursuitEnv(cfg, B, num_maps=64)
    env.reset_device(seed=21)
    dev = env.device
    w_eff, _ = m.critic.head_weight()
    fused = FusedRolloutStep(m, w_eff)
    oxy_i = env.boundary_xy.contiguous()
    o_count = torch.clamp(env.boundary_count, max=env.O).contiguous()
    g = torch.Generator(device=dev).manual_seed(4)
    ha0 = 0.1 * torch.randn(2, B, N, E, device=dev, generator=g)
    hc0 = 0.1 * torch.randn(2, B, N, E, device=dev, generator=g)
    hist0 = 0.3 * torch.randn(B, N, E, device=dev, generator=g)
    perm = torch.randperm(B, device=dev, generator=g)

    def run(order):
        e = BatchedPursuitEnv(cfg, B, num_maps=64)
        for name in ("grid_bits", "inflated_bits", "boundary_bits", "boundary_count", "boundary_xy", "raser_bits"):
            getattr(e, name).copy_(getattr(env, name))
        e.p_state.copy_(env.p_state[order]); e.e_state.copy_(env.e_state[order]); e.map_id.copy_(env.map_id[order])
        e.observe()
        ha, hc = ha0[:, order].reshape(2, B * N, E).contiguous(), hc0[:, order].reshape(2, B * N, E).contiguous()
        hist = [hist0[order].contiguous()]
        emb_a, emb_c = torch.empty(B, N, E, device=dev), torch.empty(B, N, E, device=dev)
        act, logp, val = torch.zeros(B, N, dtype=torch.int32, device=dev), torch.empty(B, N, device=dev), torch.empty(B, N, device=dev)
        fused.step(e, oxy_i, o_count, 3, 1, True, hist, hist, emb_a, emb_c, ha, hc, act, logp, val)
        torch.cuda.synchronize()
        return emb_a, emb_c, ha.view(2, B, N, E), hc.view(2, B, N, E), act, logp, val

    ident = torch.arange(B, device=dev)
    a, b = run(ident), run(perm)
    for x, y, batch_dim in zip(a, b, (0, 0, 1, 1, 0, 0, 0)):
        assert torch.isfinite(x.float()).all()
        assert torch.equal(x.index_select(batch_dim, perm), y)
    assert len(torch.unique(a[4])) > 1                      # the arg-max policy is not degenerate on this batch
