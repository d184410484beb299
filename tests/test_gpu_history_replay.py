"""History replay (mappo_parallel.HistoryReplay): a rollout that keeps only a ring of D+1 history slabs, and training that regenerates
each minibatch's [T+D, mb, N, E] history with the fused step (MARL_POLICY_STATE_F32 | MARL_POLICY_EMBED_ONLY) from the arena's
records, must give exactly what storing the history gives: the same episode, the same history bit for bit, the same minibatch
forward and gradients."""
from types import SimpleNamespace

import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

E = 128


def _cfg(depth, n_def, T, **over):
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    return default_config(env__num_defender=n_def, env__max_steps=T, algo__depth=depth, algo__learner_device="cuda",
                          algo__worker_device="cuda", **over)


def _setup(B, N, D, T, mbs=None, M=4, seed=3, quirks=True, **over):
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    cfg = _cfg(D, N, T, **over)
    torch.manual_seed(seed)
    m = MAPPO(cfg, B, mbs or max(1, B // 4), "Learner", reference_quirks=quirks)
    with torch.no_grad():                                    # biases are zero-initialised: make them matter
        for p in m.ac_parameters:
            if p.dim() == 1:
                p.add_(0.05 * torch.randn_like(p))
    env = BatchedPursuitEnv(cfg, B, num_maps=M)
    env.reset_device(seed=seed + 10, tape_len=32)            # (bounded placement draws: 64 pursuers need not all find a spot)
    return m, env, env.snapshot()


def _rollout(m, env, snap, T, history, seed=5, **kw):
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    env.restore(snap)
    arena = RolloutArena(env.params, env.B, T, env.device)
    tb = m.rollout_batched(env, arena, T, seed=seed, history=history, **kw)
    torch.cuda.synchronize()
    assert int(env.evader_status.max()) == 0
    return tb, arena


# ------------------------------------------------------------------------------------------------ 1, 2: the fused step's new modes
@pytest.mark.parametrize("variant", [1, 3])
@pytest.mark.parametrize("D", [1, 3])
@pytest.mark.parametrize("B,N", [(37, 4), (45, 8), (11, 16), (29, 5), (5, 64)])
def test_state_f32_and_embed_only_steps_equal_fp64_step(B, N, D, variant):
    """STATE_F32 on (float) copies of the state - what the arena records - equals the fp64 step bit for bit (embeddings, new hidden
    states, sampled action, log-prob, value); EMBED_ONLY writes the same embeddings and nothing else."""
    from distributed_multi_agent_reinforcement_learning_b200.fused_policy import EMBED_ONLY, STATE_F32, FusedRolloutStep
    m, env, _ = _setup(B, N, D, 4)
    dev = env.device
    env.observe()
    w_eff, _ = m.critic.head_weight(update_buffers=False)
    fused = FusedRolloutStep(m, w_eff.reshape(E).contiguous())
    oxy_i = env.boundary_xy.contiguous()
    o_count = torch.clamp(env.boundary_count, max=env.O).contiguous()
    g = torch.Generator(device=dev).manual_seed(7)
    hist = [0.3 * torch.randn(B, N, E, device=dev, generator=g) for _ in range(D)]
    if D == 3:
        hist[1] = None                                       # a zero (not yet written) slot
    ha0, hc0 = (0.1 * torch.randn(2, B * N, E, device=dev, generator=g) for _ in range(2))
    f32_view = SimpleNamespace(B=B, N=N, O=env.O, map_id=env.map_id, p_state=env.p_state.float().contiguous(),
                               e_state=env.e_state.float().contiguous(), p_adj_bits=env.p_adj_bits, e_adj=env.e_adj,
                               o_adj_bits=env.o_adj_bits)

    def run(engine, flags, full=True):
        emb_a, emb_c = torch.full((B, N, E), float("nan"), device=dev), torch.full((B, N, E), float("nan"), device=dev)
        ha, hc = ha0.clone(), hc0.clone()
        act = torch.full((B, N), -1, dtype=torch.int32, device=dev)
        logp, val = torch.full((B, N), float("nan"), device=dev), torch.full((B, N), float("nan"), device=dev)
        if full:
            fused.step(engine, oxy_i, o_count, 2, 11, False, hist, hist, emb_a, emb_c, ha, hc, act, logp, val, variant=variant, flags=flags)
        else:
            fused.step(engine, oxy_i, o_count, 2, 11, False, hist, hist, emb_a, emb_c, None, None, None, None, None, variant=variant,
                       flags=flags)
        torch.cuda.synchronize()
        return emb_a, emb_c, ha, hc, act, logp, val

    ref = run(env, 0)
    assert all(torch.isfinite(x.float()).all() for x in ref)
    for x, y in zip(ref, run(f32_view, STATE_F32)):
        assert torch.equal(x, y)
    for engine, flags in ((f32_view, STATE_F32 | EMBED_ONLY), (env, EMBED_ONLY)):
        emb_a, emb_c = run(engine, flags, full=False)[:2]
        assert torch.equal(emb_a, ref[0]) and torch.equal(emb_c, ref[1])


# ------------------------------------------------------------------------------------------------ 3: a replay-mode episode
EPISODES = [pytest.param(64, 8, 40, D, q, pipes, id=f"B64-N8-T40-d{D}-{'quirks' if q else 'own'}-{pipes}pipe")
            for D in (1, 3) for q in (True, False) for pipes in (1, 4)] + \
           [pytest.param(12, 16, 20, 3, True, 1, id="B12-N16-T20-d3"), pytest.param(3, 64, 12, 3, True, 1, id="B3-N64-T12-d3")]


@pytest.mark.parametrize("B,N,T,D,quirks,pipes", EPISODES)
def test_replayed_history_equals_stored_history(B, N, T, D, quirks, pipes):
    m, env, snap = _setup(B, N, D, T, quirks=quirks)
    tb_s, ar_s = _rollout(m, env, snap, T, "store", pipelines=pipes)
    hist_a, hist_c, logp, v, a, rew = tb_s.hist_a.clone(), tb_s.hist_c.clone(), tb_s.logp.clone(), tb_s.v.clone(), tb_s.a.clone(), ar_s.raw_reward.clone()
    tb_r, ar_r = _rollout(m, env, snap, T, "replay", pipelines=pipes)
    assert tb_r.hist_a is None and tb_r.hist_c is None and tb_r.replay is not None
    # the ring does not change the episode (the bootstrap value reads the ring too)
    assert torch.equal(tb_r.a, a) and torch.equal(tb_r.logp, logp) and torch.equal(tb_r.v, v) and torch.equal(ar_r.raw_reward, rew)
    mb = tb_r.minibatch(0, B)
    torch.cuda.synchronize()
    assert torch.equal(mb.hist_a, hist_a) and torch.equal(mb.hist_c, hist_c)
    # the full step (EMBED_ONLY off) from zero hidden states reproduces the stored log-probs and values
    lp2, v2 = tb_r.replay.regenerate(mb, embed_only=False)
    torch.cuda.synchronize()
    assert torch.equal(mb.hist_a, hist_a) and torch.equal(mb.hist_c, hist_c)
    assert torch.equal(lp2, logp) and torch.equal(v2, v[:T])
    # a sub-batch, contiguous and gathered
    lo, hi = B // 3, B // 3 + max(1, B // 2)
    mb = tb_r.minibatch(lo, hi)
    assert torch.equal(mb.hist_a, hist_a[:, lo:hi]) and torch.equal(mb.hist_c, hist_c[:, lo:hi])
    idx = torch.randperm(B, device=env.device, generator=torch.Generator(device=env.device).manual_seed(1))[:hi - lo]
    mb, _ = tb_r.minibatch_indexed(idx)
    torch.cuda.synchronize()
    assert torch.equal(mb.hist_a, hist_a[:, idx]) and torch.equal(mb.hist_c, hist_c[:, idx])


def test_explore_batched_graph_replay_history():
    """The CUDA-graph episode (explore_batched) in replay mode: same episode as a stored rollout, same regenerated history."""
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    B, N, T, D = 48, 8, 30, 3
    m, env, snap = _setup(B, N, D, T)
    tb_s, _ = _rollout(m, env, snap, T, "store", seed=9)
    env.restore(snap)
    arena = RolloutArena(env.params, B, T, env.device)
    tb_g = m.explore_batched(env, arena, T, seed=9, history="replay")
    torch.cuda.synchronize()
    assert tb_g.hist_a is None and tb_g.replay is not None
    assert torch.equal(tb_g.a, tb_s.a) and torch.equal(tb_g.logp, tb_s.logp) and torch.equal(tb_g.v, tb_s.v)
    mb = tb_g.minibatch(0, B)
    torch.cuda.synchronize()
    assert torch.equal(mb.hist_a, tb_s.hist_a) and torch.equal(mb.hist_c, tb_s.hist_c)


# ------------------------------------------------------------------------------------------------ 4: training on a replay batch
@pytest.mark.parametrize("in_flight", [1, 3])
@pytest.mark.parametrize("shuffle", [False, True], ids=["sequential", "shuffled"])
def test_train_on_replay_batch_equals_store_batch(shuffle, in_flight, monkeypatch):
    """Same epoch on the stored and the replay-mode batch of one episode, twice with an optimizer step in between (the second round
    only matches if the replay uses the rollout-time weights): per-minibatch log-probs, entropies, values, losses and gradients
    bit-identical.  Every reduction of the epoch, the message layers' weight gradients and the loss sums included, is summed in a
    fixed order (DESIGN §2)."""
    from distributed_multi_agent_reinforcement_learning_b200 import mappo_parallel
    monkeypatch.setattr(mappo_parallel, "CONCURRENT_MINIBATCHES", in_flight)
    B, N, T, D = 48, 8, 24, 3
    m, env, snap = _setup(B, N, D, T, mbs=16)
    tb_s, _ = _rollout(m, env, snap, T, "store")
    tb_r, _ = _rollout(m, env, snap, T, "replay")
    u = m.critic.Mean
    for rnd in range(2):
        traces = []
        sn0 = (u.weight_u.clone(), u.weight_v.clone()) if m.sn else None
        for tb in (tb_s, tb_r):
            if sn0 is not None:                              # the spectral-norm power iteration advances on every forward
                u.weight_u.copy_(sn0[0])
                u.weight_v.copy_(sn0[1])
            tr = {}
            m.train(tb, B * T * (rnd + 1), return_numpy=False, trace=tr, shuffle=shuffle, shuffle_seed=4)
            torch.cuda.synchronize()
            traces.append(tr)
        ts, tr_ = traces
        assert len(ts["mb"]) == len(tr_["mb"]) == 3
        for a, b in zip(ts["mb"], tr_["mb"]):
            for k in ("logp", "ent", "val"):
                assert torch.equal(a[k], b[k]), (rnd, k)
            assert a["actor_loss"] == b["actor_loss"] and a["critic_loss"] == b["critic_loss"], rnd
        gs, gr = ts["mb_grads"], tr_["mb_grads"]
        assert torch.equal(gs, gr), [i for i, (off, k) in enumerate(m.ac_optimizer._views)
                                     if not torch.equal(gs[:, off:off + k], gr[:, off:off + k])]
        m.update(B * T * (rnd + 1))


# ------------------------------------------------------------------------------------------------ 5: memory
def test_replay_mode_peak_memory():
    """Peak allocation of rollout + epoch: replay mode saves at least the stored history minus the ring and the replay scratch of
    the minibatches in flight (all from shapes)."""
    from distributed_multi_agent_reinforcement_learning_b200 import mappo_parallel
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import history_bytes
    B, N, T, D, mbs = 256, 8, 60, 1, 32
    m, env, snap = _setup(B, N, D, T, mbs=mbs)
    peaks = {}
    for mode in ("replay", "store", "replay"):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        tb, arena = _rollout(m, env, snap, T, mode)
        m.train(tb, B * T, return_numpy=False)
        torch.cuda.synchronize()
        peaks[mode] = torch.cuda.max_memory_allocated() - base
        del tb, arena
    in_flight = min(mappo_parallel.CONCURRENT_MINIBATCHES, B // mbs)
    ring = 2 * (D + 1) * B * N * E * 4
    scratch = in_flight * history_bytes(T, mbs, N, E, D)
    saved = peaks["store"] - peaks["replay"]
    assert saved >= history_bytes(T, B, N, E, D) - ring - scratch, (peaks, history_bytes(T, B, N, E, D), ring, scratch)


# ------------------------------------------------------------------------------------------------ 6: automatic selection
def test_automatic_history_selection(monkeypatch):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib, mappo_parallel
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    torch.manual_seed(0)
    m = MAPPO(_cfg(1, 8, 150), 4096, 410, "Learner")
    assert m.history_mode(150, 4096, 8) == "store"                  # the bench shape: 5.1 GB
    monkeypatch.setattr(mappo_parallel, "STORE_HISTORY_SHARE", 0.0)
    assert m.history_mode(150, 4096, 8) == "replay"
    m, env, snap = _setup(8, 4, 1, 6)
    tb, _ = _rollout(m, env, snap, 6, None)
    assert tb.hist_a is None and tb.replay is not None
    # networks the fused step cannot run: the history must be stored, and it does not fit
    m, env, snap = _setup(8, 4, 1, 6, algo__embedding_dim=64, algo__rnn_hidden_dim=64)
    with pytest.raises(_lib.MarlError, match="GB"):
        _rollout(m, env, snap, 6, None)
    monkeypatch.setattr(mappo_parallel, "STORE_HISTORY_SHARE", 0.5)
    tb, _ = _rollout(m, env, snap, 6, None)
    assert tb.hist_a is not None and tb.replay is None
