"""Training and evaluation on an installed map pool: the per-env map draw (marl_map_draw), resets that keep the maps
(reset_device(maps="keep" | "draw")), auto-reset streams that draw each episode's maps from the pool (eager and from CUDA graphs), the
map ids of a crossing batch's two pieces, the Evaluator on held-out maps, and tools/train_loop.py --map-pool."""
import ctypes
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T_EP, B, M = 150, 600, 97
RECORDS = ("p_state_f32", "e_state_f32", "p_adj_bits", "e_adj", "o_adj_bits", "a_n", "r", "raw_reward", "active")
TABLES = ("grid_bits", "inflated_bits", "boundary_bits", "boundary_count", "boundary_xy", "raser_bits")
RESET_SEED = lambda e: 70 + e                 # noqa: E731
SAMPLE_SEED = lambda e: 9 + 5 * e             # noqa: E731
TAG = 0x6472617700000000                      # the map draw's stream tag (csrc/reset_kernels.cu)


def _cfg(N=8, D=1, T=T_EP):
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    return default_config(env__num_defender=N, env__max_steps=T, algo__depth=D, algo__learner_device="cuda", algo__worker_device="cuda",
                          algo__evaluator_device="cuda")


@functools.lru_cache(maxsize=None)
def _pool(n_maps=M, seed=11):
    """A pool of maps generated on the device, read back through MapPool.from_engine."""
    from distributed_multi_agent_reinforcement_learning_b200.map_pool import MapPool
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    env = BatchedPursuitEnv(_cfg(), n_maps, num_maps=n_maps)
    env.reset_device(seed=seed)
    return MapPool.from_engine(env)


def _pool_engine(Bx=B, N=8, D=1, T=T_EP):
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    env = BatchedPursuitEnv(_cfg(N, D, T), Bx, num_maps=M)
    _pool().install(env, verify=True)
    return env


# ------------------------------------------------------------------------------------------------ marl_map_draw
def _splitmix64(z):
    z = (z + np.uint64(0x9E3779B97F4A7C15)).astype(np.uint64)
    z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)).astype(np.uint64)
    z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)).astype(np.uint64)
    return z ^ (z >> np.uint64(31))


def _draw_ref(seed, Bx, Mx):
    """numpy restatement: env b's Stream64 keyed by splitmix64(seed ^ TAG) ^ splitmix64(b), first draw, randint(0, M-1)."""
    with np.errstate(over="ignore"):
        key = _splitmix64(np.array([(seed & (2 ** 64 - 1)) ^ TAG], np.uint64)) ^ _splitmix64(np.arange(Bx, dtype=np.uint64))
        x = _splitmix64(key ^ _splitmix64(np.zeros(1, np.uint64)))
    u = (x >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)
    return (u * float(Mx)).astype(np.int32)


def _draw(env, seed, Bx=None, Mx=None, device_seed=False):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    Bx, Mx = Bx or env.B, Mx or env.M
    out = torch.full((Bx,), -1, dtype=torch.int32, device=env.device)
    if device_seed:
        word = torch.tensor([_lib.u64_bits(seed)], dtype=torch.int64, device=env.device)
        rc = env.lib.marl_map_draw_dseed(env._pp(), Bx, Mx, _lib.ptr(word), _lib.ptr(out), _lib.stream_ptr())
    else:
        rc = env.lib.marl_map_draw(env._pp(), Bx, Mx, ctypes.c_uint64(seed & (2 ** 64 - 1)), _lib.ptr(out), _lib.stream_ptr())
    _lib.check(rc, "marl_map_draw")
    torch.cuda.synchronize()
    return out.cpu().numpy()


def test_map_draw_is_the_stream64_draw():
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    env = BatchedPursuitEnv(_cfg(), 8, num_maps=8)
    for seed, Bx, Mx in ((1, 1000, 97), (2 ** 64 - 5, 777, 2000), (123456789, 4096, 1), (5, 300, 2 ** 31 - 1)):
        got = _draw(env, seed, Bx, Mx)
        assert np.array_equal(got, _draw_ref(seed, Bx, Mx)), seed
        assert got.min() >= 0 and got.max() < Mx
        assert np.array_equal(_draw(env, seed, Bx, Mx), got)                                  # deterministic
        assert np.array_equal(_draw(env, seed, Bx, Mx, device_seed=True), got)                # the dseed twin
        assert np.array_equal(_draw(env, seed, 64, Mx), got[:64])                             # env b's id does not depend on B
    assert (_draw(env, 1, 1000, 97) != _draw(env, 2, 1000, 97)).mean() > 0.9                  # and changes with the seed


def test_map_draw_is_uniform():
    from scipy import stats
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    env = BatchedPursuitEnv(_cfg(), 8, num_maps=8)
    for seed, Mx in ((3, 97), (4, 2000), (5, 7)):
        counts = np.bincount(_draw(env, seed, 200_000, Mx), minlength=Mx)
        assert counts.shape == (Mx,)
        assert stats.chisquare(counts).pvalue > 1e-4, (seed, Mx)


def test_captured_draw_reset_follows_its_seed_word():
    env = _pool_engine(256)
    word = torch.zeros(1, dtype=torch.int64, device=env.device)
    env.reset_device(seed=word, tape_len=16, tape="device", maps="draw")       # warm-up, allocates the reset's buffers
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            env.reset_device(seed=word, tape_len=16, tape="device", maps="draw")
    torch.cuda.current_stream().wait_stream(side)
    names = ("map_id", "p_state", "e_state", "target", "target_tape")
    for seed in (21, 22):
        word.fill_(seed)
        graph.replay()
        torch.cuda.synchronize()
        got = {n: getattr(env, n).clone() for n in names}
        env.reset_device(seed=seed, tape_len=16, tape="device", maps="draw")
        torch.cuda.synchronize()
        for n in names:
            assert torch.equal(got[n], getattr(env, n)), (seed, n)
        assert np.array_equal(got["map_id"].cpu().numpy(), _draw_ref(seed, env.B, M))


# ------------------------------------------------------------------------------------------------ keep / draw resets
def _check_placements(cfg, env):
    """The placement rules test_gpu_reset.py checks, for every env on the map it was placed on."""
    from distributed_multi_agent_reinforcement_learning_b200 import maps
    W, H, N = env.params.W, env.params.H, env.N
    infl = maps.unpack_words(env.inflated_bits.cpu().numpy(), H)
    ps, es, tg, mid = (t.cpu().numpy() for t in (env.p_state, env.e_state, env.target, env.map_id))
    comm, sen = float(cfg.defender.comm_range), float(cfg.defender.sen_range)
    for b in range(env.B):
        I = infl[mid[b]]
        assert not I[tg[b, 0], tg[b, 1]]
        work = I.copy()
        cells = []
        for i in range(N):
            x, y = ps[b, i, :2]
            assert 0 <= x <= W - 1 and 0 <= y <= H - 1 and ps[b, i, 2] == 0 and ps[b, i, 3] == 0
            cx, cy = round(float(x)), round(float(y))
            assert not work[cx, cy], (b, i)
            if i:
                d = np.hypot(ps[b, :i, 0] - x, ps[b, :i, 1] - y)
                assert (d >= 4).all() and 0 < (d < comm).sum() <= 2, (b, i)
            work[max(0, cx - 2):cx + 3, max(0, cy - 2):cy + 3] = 1
            cells.append((cx, cy))
        ex, ey = es[b, :2]
        assert not work[round(float(ex)), round(float(ey))]
        assert min(np.hypot(c[0] - ex, c[1] - ey) for c in cells) < sen


@pytest.mark.parametrize("tape", ["torch", "device"])
def test_keep_and_draw_resets_keep_the_tables(tape):
    env = _pool_engine()
    tables = {n: getattr(env, n).clone() for n in TABLES}
    env.map_id.copy_(torch.arange(B, dtype=torch.int32, device=env.device).flip(0) % M)
    ids = env.map_id.clone()
    env.reset_device(seed=5, tape=tape, maps="keep")
    torch.cuda.synchronize()
    assert torch.equal(env.map_id, ids) and int(env.reset_fail.sum()) == 0
    _check_placements(env.cfg, env)
    kept = {n: getattr(env, n).clone() for n in ("p_state", "e_state", "target", "target_tape")}
    env.reset_device(seed=6, tape=tape, maps="draw")
    torch.cuda.synchronize()
    assert np.array_equal(env.map_id.cpu().numpy(), _draw_ref(6, B, M)) and int(env.reset_fail.sum()) == 0
    _check_placements(env.cfg, env)
    for n in TABLES:
        assert torch.equal(getattr(env, n), tables[n]), n
    env.map_id.copy_(ids)                                          # placements depend on (seed, map): the same with the same map ids
    env.reset_device(seed=5, tape=tape, maps="keep")
    for n, x in kept.items():
        assert torch.equal(getattr(env, n), x), n
    assert env.time_step.abs().sum() == 0 and env.tape_pos.abs().sum() == 0


def test_draw_reset_places_every_env_at_the_bench_config():
    """4096 envs x 8 pursuers on a 2000-map pool."""
    from distributed_multi_agent_reinforcement_learning_b200.map_pool import MapPool
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    gen = BatchedPursuitEnv(_cfg(), 2000, num_maps=2000)
    gen.reset_device(seed=1)
    env = BatchedPursuitEnv(_cfg(), 4096, num_maps=2000)
    MapPool.from_engine(gen).install(env, verify=False)
    for seed in range(3):
        env.reset_device(seed=seed, tape="device", maps="draw")
        torch.cuda.synchronize()
        assert int(env.reset_fail.sum()) == 0, seed
        assert int(env.map_id.min()) >= 0 and int(env.map_id.max()) < 2000


@pytest.mark.parametrize("maps", ["keep", "draw"])
def test_keeping_maps_that_were_never_set_raises_before_any_launch(maps):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    env = BatchedPursuitEnv(_cfg(), 16, num_maps=4)
    calls, launches = _lib.CALLS, env.launches
    before = {n: getattr(env, n).clone() for n in ("map_id", "p_state", "target_tape") + TABLES}
    for seed in (3, torch.zeros(1, dtype=torch.int64, device=env.device)):
        with pytest.raises(_lib.MarlError, match="never set"):
            env.reset_device(seed=seed, tape="device", maps=maps)
    assert _lib.CALLS == calls and env.launches == launches and getattr(env, "_reset_scratch", None) is None
    for n, x in before.items():
        assert torch.equal(getattr(env, n), x), n
    env.reset_device(seed=3)                                     # a "generate" reset sets them
    env.reset_device(seed=4, maps=maps)
    env2 = BatchedPursuitEnv(_cfg(), 16, num_maps=4)
    env2.load_state_dict(env.state_dict())                      # ... and so does loading a state
    env2.reset_device(seed=4, maps=maps)
    torch.cuda.synchronize()
    assert torch.equal(env2.p_state, env.p_state) and torch.equal(env2.map_id, env.map_id)


# ------------------------------------------------------------------------------------------------ auto-reset streams on the pool
def _setup(D=1, quirks=True, seed=3):
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    env = _pool_engine(D=D)
    torch.manual_seed(seed)
    m = MAPPO(env.cfg, B, B // 3, "Learner", reference_quirks=quirks)
    with torch.no_grad():
        for p in m.ac_parameters:
            if p.dim() == 1:
                p.add_(0.05 * torch.randn_like(p))
    env.wf0 = {k: getattr(env, k).clone() for k in ("wf_n", "wf_mean", "wf_S", "wf_std")}
    return m, env


def _auto():
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import AutoReset
    return AutoReset(RESET_SEED, SAMPLE_SEED, tape_len=32, tape="device", maps="draw")


def _first_episode(env):
    env.restore(env.wf0)
    env.reset_device(seed=RESET_SEED(0), tape_len=32, tape="device", maps="draw")


def _state(env):
    out = {k: x.clone() for k, x in env.snapshot().items()}
    out["path"] = out["path"] * (torch.arange(out["path"].shape[1], device=env.device)[None, :, None] < out["path_len"][:, None, None].long())
    for n in ("map_id", "target_tape") + TABLES:
        out[n] = getattr(env, n).clone()
    return out


def _episodes(m, env, history):
    """Two whole episodes, episode e from reset_device(RESET_SEED(e), maps="draw") sampled with SAMPLE_SEED(e), and the engine at the
    start of episode 2."""
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    arena = RolloutArena(env.params, env.B, T_EP, env.device)
    eps = []
    _first_episode(env)
    for e in range(3):
        if e:
            env.reset_device(seed=RESET_SEED(e), tape_len=32, tape="device", maps="draw")
        if e == 2:
            return eps, _state(env)
        ids = env.map_id.clone()
        tb = m.rollout_batched(env, arena, T_EP, seed=SAMPLE_SEED(e), history=history)
        mb = tb.minibatch(0, env.B)
        torch.cuda.synchronize()
        eps.append(dict(a=tb.a.clone(), logp=tb.logp.clone(), v=tb.v.clone(), hist_a=mb.hist_a.clone(), hist_c=mb.hist_c.clone(),
                        rec={k: getattr(arena, k).clone() for k in RECORDS}, collision=env.collision.clone(),
                        evader_status=env.evader_status.clone(), map_id=ids))


def _stream(m, env, S, history, graph=False):
    """Segments of S steps with the pool auto-reset from episode 0's start until two episodes are collected."""
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    arena = RolloutArena(env.params, env.B, S, env.device)
    _first_episode(env)
    carry, segs, auto = RolloutCarry.zeros(m, env.B, env.N), [], _auto()
    for _ in range(-(-2 * T_EP // S)):
        start = (carry.episode, carry.t0)
        if graph:
            tb = m.explore_batched(env, arena, S, history=history, carry=carry, auto_reset=auto)
        else:
            tb = m.rollout_batched(env, arena, S, history=history, carry=carry, auto_reset=auto)
        torch.cuda.synchronize()
        assert int(env.evader_status.max()) == 0 and int(env.reset_fail.sum()) == 0
        c = tb.carry
        segs.append(dict(a=tb.a.clone(), logp=tb.logp.clone(), v=tb.v.clone(), rec={k: getattr(arena, k).clone() for k in RECORDS},
                         start=start, boundary=tb.boundary, v_boot=None if tb.v_boot is None else tb.v_boot.clone(),
                         ended=None if tb.ended_collision is None else (tb.ended_collision.clone(), tb.ended_evader_status.clone()),
                         carry=(c.episode, c.t0) + tuple(getattr(c, k).clone() for k in ("ha", "hc", "emb_a", "emb_c")),
                         map_id=None if tb.map_id is None else tb.map_id.clone(),
                         map_id2=None if tb.map_id2 is None else tb.map_id2.clone()))
        carry = RolloutCarry(c.t0, *(x.clone() for x in (c.ha, c.hc, c.emb_a, c.emb_c)), episode=c.episode)
    return segs, _state(env)


@functools.lru_cache(maxsize=None)
def _runs(history):
    m, env = _setup()
    out = {None: _episodes(m, env, history)}
    for S in (64, 150):
        out[S] = _stream(m, env, S, history)
    out["graph"] = _stream(m, env, 64, history, graph=True)
    return out


@pytest.mark.parametrize("history", ["store", "replay"])
@pytest.mark.parametrize("S", [64, 150])
def test_pool_stream_equals_the_episodes(S, history):
    runs = _runs(history)
    eps, final = runs[None]
    segs, final_s = runs[S]
    assert not torch.equal(eps[0]["map_id"], eps[1]["map_id"])                                  # the draw changed the maps
    assert np.array_equal(eps[0]["map_id"].cpu().numpy(), _draw_ref(RESET_SEED(0), B, M))
    ep_cat = lambda k: torch.cat([e[k] for e in eps])                                       # noqa: E731
    ep_v = torch.cat([e["v"][:-1] for e in eps])
    n = 2 * T_EP
    cut = lambda x: x[:n]                                                                   # noqa: E731
    assert torch.equal(cut(torch.cat([s["a"] for s in segs])), ep_cat("a"))
    assert torch.equal(cut(torch.cat([s["logp"] for s in segs])), ep_cat("logp"))
    assert torch.equal(cut(torch.cat([s["v"][:-1] for s in segs])), ep_v)
    for k in RECORDS:
        assert torch.equal(cut(torch.cat([s["rec"][k] for s in segs])), torch.cat([e["rec"][k] for e in eps])), k
    crossings = 0
    for i, s in enumerate(segs):
        e, t0 = divmod(i * S, T_EP)
        assert s["start"] == (e, t0), i
        if history == "replay":                                  # the batch's (first piece's) map ids are the episode's
            assert torch.equal(s["map_id"], eps[e]["map_id"]), i
        if t0 + S >= T_EP:
            k = T_EP - t0
            boot = s["v"][-1] if k == S else s["v_boot"]
            assert torch.equal(boot, eps[e]["v"][T_EP]), i
            assert torch.equal(s["ended"][0], eps[e]["collision"]) and torch.equal(s["ended"][1], eps[e]["evader_status"]), i
            crossings += k < S
            if k < S and history == "replay" and e + 1 < len(eps):
                assert torch.equal(s["map_id2"], eps[e + 1]["map_id"]), i
        else:
            assert s["boundary"] is None and s["ended"] is None, i
        e2, t2 = divmod((i + 1) * S, T_EP)
        assert s["carry"][:2] == (e2, t2), i
        if t2 == 0:
            assert all(float(x.abs().max()) == 0 for x in s["carry"][2:]), i
        elif e2 < len(eps):
            D = eps[e2]["hist_a"].shape[0] - T_EP
            assert torch.equal(s["carry"][4], eps[e2]["hist_a"][t2:t2 + D]) and torch.equal(s["carry"][5], eps[e2]["hist_c"][t2:t2 + D]), i
    assert crossings == {64: 2, 150: 0}[S]
    if S == T_EP:                                                # the stream stops at episode 2's start, maps drawn
        for k in final:
            assert torch.equal(final_s[k], final[k]), k


@pytest.mark.parametrize("history", ["store", "replay"])
def test_pool_graph_stream_equals_the_eager_stream(history):
    runs = _runs(history)
    (eager, fin_e), (graph, fin_g) = runs[64], runs["graph"]
    assert len(eager) == len(graph)
    for i, (a, b) in enumerate(zip(eager, graph)):
        for k in ("a", "logp", "v", "v_boot", "map_id", "map_id2"):
            assert (a[k] is None and b[k] is None) or torch.equal(a[k], b[k]), (i, k)
        for k in RECORDS:
            assert torch.equal(a["rec"][k], b["rec"][k]), (i, k)
        assert a["start"] == b["start"] and a["boundary"] == b["boundary"], i
        assert (a["ended"] is None) == (b["ended"] is None) and (a["ended"] is None or all(map(torch.equal, a["ended"], b["ended"]))), i
        assert a["carry"][:2] == b["carry"][:2] and all(map(torch.equal, a["carry"][2:], b["carry"][2:])), i
    for k in fin_e:
        assert torch.equal(fin_e[k], fin_g[k]), k


# ------------------------------------------------------------------------------------------------ the pieces' map ids
def _crossing_batch(m, env, history):
    """The third segment of an S = 64 pool stream: steps 128..149 of episode 0 and 0..41 of episode 1 (on newly drawn maps)."""
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    arena = RolloutArena(env.params, env.B, 64, env.device)
    _first_episode(env)
    carry, auto = RolloutCarry.zeros(m, env.B, env.N), _auto()
    for _ in range(3):
        tb = m.rollout_batched(env, arena, 64, history=history, carry=carry, auto_reset=auto)
        carry = tb.carry
    torch.cuda.synchronize()
    assert tb.boundary == 22
    return tb


def _forward(m, tb, sn0):
    u = m.critic.Mean
    u.weight_u.copy_(sn0[0])
    u.weight_v.copy_(sn0[1])
    tr = {}
    m.train(tb, B * 64, return_numpy=False, trace=tr)
    torch.cuda.synchronize()
    return torch.cat([t["logp"] for t in tr["mb"]], dim=1), torch.cat([t["val"] for t in tr["mb"]], dim=1)


@pytest.mark.parametrize("D", [1, 3])
def test_replay_crossing_batch_trains_each_piece_on_its_own_maps(D):
    """reference_quirks=False, replay mode: the training forward reproduces the rollout's log-probs and values on both pieces, and
    does not on the first piece when it is given the new episode's map ids."""
    m, env = _setup(D=D, quirks=False)
    tb = _crossing_batch(m, env, "replay")
    k = tb.boundary
    assert tb.hist_a is None and tb.map_id2 is not None
    assert float((tb.map_id != tb.map_id2).float().mean()) > 0.9
    u = m.critic.Mean
    sn0 = (u.weight_u.clone(), u.weight_v.clone())
    logp, val = _forward(m, tb, sn0)
    torch.testing.assert_close(logp, tb.logp, rtol=1e-5, atol=2e-5)
    torch.testing.assert_close(val, tb.v[:-1], rtol=1e-5, atol=2e-5)
    tb.map_id = tb.map_id2                                       # negative control: piece 1 on the new maps
    logp0, val0 = _forward(m, tb, sn0)
    assert float((logp0[:k] - tb.logp[:k]).abs().max()) > 1e-3 and float((val0[:k] - tb.v[:k]).abs().max()) > 1e-3
    torch.testing.assert_close(logp0[k:], tb.logp[k:], rtol=1e-5, atol=2e-5)


# ------------------------------------------------------------------------------------------------ Evaluator on held-out maps
def test_evaluator_plays_the_held_out_maps():
    from distributed_multi_agent_reinforcement_learning_b200.evaluator import Evaluator
    from distributed_multi_agent_reinforcement_learning_b200.map_pool import MapPool
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena
    T, n_env = 40, 24
    cfg = _cfg(T=T)
    pool, held = _pool(), np.arange(80, 87)
    torch.manual_seed(5)
    agent = MAPPO(cfg, None, None, "Evaluator")
    evs = [Evaluator(cfg, n_env, agent, seed=3, pool=pool, pool_indices=held) for _ in range(2)]
    rs = [ev.get_rewards_and_step() for ev in evs]
    assert torch.equal(rs[0], rs[1])
    eng = evs[0]._engine
    assert eng.M == len(held) and np.array_equal(eng.map_id.cpu().numpy(), np.arange(n_env) % len(held))
    got = MapPool.from_engine(eng)
    for f in ("obstacle_map_list", "boundary_map_list", "hash_map_list"):
        assert np.array_equal(getattr(got, f), getattr(pool, f)[held]), f
    assert np.array_equal(got.boundary_obstacle_num_list, pool.boundary_obstacle_num_list[held])
    rs2 = evs[0].get_rewards_and_step()                          # the next evaluation: same maps, new placements
    assert np.array_equal(eng.map_id.cpu().numpy(), np.arange(n_env) % len(held)) and not torch.equal(rs2, rs[0])
    # the returns are an actor_only arg-max rollout from the same engine state
    env = BatchedPursuitEnv(cfg, n_env, num_maps=len(held))
    pool.install(env, held)
    arena = RolloutArena(env.params, n_env, T, env.device)
    for seed, r in ((4, rs[0]), (5, rs2)):
        env.reset_device(seed=seed, tape_len=64, maps="keep")
        agent.rollout_batched(env, arena, T, seed=seed, deterministic=True, actor_only=True)
        ret = arena.raw_reward[:T].sum(dim=(0, 2)).float().cpu()
        assert torch.equal(ret, r[:, 0]), seed


# ------------------------------------------------------------------------------------------------ tools/train_loop.py
def _subpool(pool, n):
    """The pool of the first n maps of `pool`."""
    from distributed_multi_agent_reinforcement_learning_b200.map_pool import MapPool
    no, nb = int(pool.obstacle_num_list[:n].sum()), int(pool.boundary_obstacle_num_list[:n].sum())
    return MapPool(pool.obstacle_map_list[:n], pool.boundary_map_list[:n], pool.hash_map_list[:n], pool.obstacle_list[:no],
                   pool.obstacle_num_list[:n], pool.boundary_obstacle_list[:nb], pool.boundary_obstacle_num_list[:n])


def _train_loop(*args):
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.join(ROOT, "tools", "train_loop.py"), "--envs", "32",
                                                                         "--steps", "150"] + list(args)
    out = subprocess.run(cmd, check=True, cwd=ROOT, timeout=900, capture_output=True, text=True).stdout
    lines = out.splitlines()
    train = {int(ln.split("exact ")[1].split()[0]): ln.split("exact ")[1] for ln in lines if ln.startswith("iter")}
    evals = {int(ln.split("hex ")[1].split()[0]): ln.split("hex ")[1] for ln in lines if ln.startswith("eval")}
    return train, evals


@pytest.fixture(scope="module")
def pools(tmp_path_factory):
    d = tmp_path_factory.mktemp("pools")
    full = _pool(12, seed=4)
    full.save(str(d / "full"))
    _subpool(full, 9).save(str(d / "first9"))
    return str(d / "full"), str(d / "first9")


@pytest.mark.parametrize("mode", [[], ["--auto-reset"], ["--auto-reset", "--graph"]], ids=["plain", "auto", "graph"])
def test_train_loop_on_a_pool_is_reproducible(pools, mode):
    seg = ["--segment", "50" if not mode else "64"]
    a, _ = _train_loop("--map-pool", pools[1], "--iters", "4", *seg, *mode)
    b, _ = _train_loop("--map-pool", pools[1], "--iters", "4", *seg, *mode)
    assert sorted(a) == list(range(4)) and a == b


def test_train_loop_on_a_pool_resumes_inside_a_stream_and_ignores_the_held_out_maps(pools, tmp_path):
    args = ("--segment", "64", "--auto-reset", "--iters", "5")
    straight, _ = _train_loop("--map-pool", pools[1], *args)
    held, evals = _train_loop("--map-pool", pools[0], "--held-out", "3", "--eval-every", "2", "--eval-envs", "6", *args)
    assert held == straight                                      # the evaluation changes nothing in the training
    assert sorted(evals) == [1, 3]
    first, ev1 = _train_loop("--map-pool", pools[0], "--held-out", "3", "--eval-every", "2", "--eval-envs", "6", "--segment", "64",
                             "--auto-reset", "--iters", "3", "--save-dir", str(tmp_path))       # stops after the first crossing
    resumed, ev2 = _train_loop("--map-pool", pools[0], "--held-out", "3", "--eval-every", "2", "--eval-envs", "6", *args, "--resume",
                               str(tmp_path))
    assert first == {i: straight[i] for i in range(3)} and resumed == {i: straight[i] for i in range(3, 5)}
    assert ev1 == {1: evals[1]} and ev2 == {3: evals[3]}
