"""Maps 64 to 127 cells tall on the GPU: the A* evader's two-word column search (csrc/evader.cu, CW = 2) against the CPU oracle,
and the env, observe, sensor-table and reset kernels with three or four bitmap words per column.  The lattice of the search is
[0, W] x [0, H], so H = 64 is already a two-word map and H = 127 the tallest (128 x 128 would need a 129th row); rows 63 / 64 are
the word boundary every case below crosses."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

WIDEST = 162          # widest map whose two-word search fits one block's shared memory (marl_b200.h)


def _cfg(W, H, **over):
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    kw = dict(env__num_defender=4, map__map_size=[W, H], map__center=[W // 2, H // 2], map__num_max_obstacle=256)
    kw.update(over)
    return default_config(**kw)


def _bits(a):
    return np.ascontiguousarray(a).view(np.int64)


def _evader_vs_oracle(oracle, cfg, grids, p_state, e_state, target):
    """One attacker_step per env (env b on map b, replan due), compared with the oracle's: path, path length, the evader's move."""
    from distributed_multi_agent_reinforcement_learning_b200 import maps
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    B = len(grids)
    env = BatchedPursuitEnv(cfg, B, num_maps=B)
    env.set_maps(grids)
    env.set_state(p_state, e_state, target, np.arange(B), time_step=0)
    env.start_episode()
    env.set_target_tape(np.zeros((B, 0, 2), np.int32))
    env.evader_step()
    torch.cuda.synchronize()
    assert not (env.evader_status.cpu().numpy() & 3).any(), "search heap / path overflow"
    p = oracle.EnvParams.from_dict(env.params.as_dict())
    infl = maps.dilate(grids, 2)
    lens = []
    for b in range(B):
        ev = oracle.EvaderState(e_state[b], target[b])
        assert oracle.evader_step(p, ev, p_state[b], 0, grids[b], infl[b], np.zeros((0, 2), np.int32)) in (0, -2)
        L = ev.path_len.value
        assert int(env.path_len[b]) == L, (b, int(env.path_len[b]), L)
        assert np.array_equal(env.path[b, :L].cpu().numpy(), ev.path[:L]), b
        np.testing.assert_allclose(env.e_state[b].cpu().numpy(), ev.e_state, rtol=1e-9, atol=1e-9)
        lens.append(L)
    return lens, [env.path[b, :lens[b]].cpu().numpy() for b in range(B)]


@pytest.mark.parametrize("size", [(64, 64), (96, 96), (128, 127), (129, 127), (WIDEST, 64), (WIDEST, 101)])
def test_tall_cup_trap_search_vs_oracle(oracle, size):
    """The cup trap of test_gpu_env.py on two-word maps: the evader starts inside a cup that opens away from its target, so the
    weighted A* floods the cup (long OPEN stripes, dead-end pops, more columns than lanes) before it finds the way round.
    (162 x 101 is also a map whose W * H is 2 mod 4: the sensor-table kernel's shared-memory carve must stay aligned there.)"""
    W, H = size
    grid = np.zeros((W, H), np.uint8)
    x0 = W // 2
    grid[x0, 4:H - 4] = 1
    grid[x0 - W // 4:x0 + 1, 4] = 1
    grid[x0 - W // 4:x0 + 1, H - 5] = 1
    p_state = np.zeros((1, 4, 4))
    p_state[0, :, 0] = [1, 2, 3, 4]                            # pursuers parked in a corner
    p_state[0, :, 1] = 1.0
    e_state = np.array([[x0 - 5.2, H // 2 + 0.1, 0, 0]], np.float64)
    target = np.array([[W - 4, H // 2]], np.int32)
    (L,), _ = _evader_vs_oracle(oracle, _cfg(W, H), grid[None], p_state, e_state, target)
    assert L > W // 4                                          # out of the cup and round the wall


@pytest.mark.parametrize("extend_dis", [1, 3])
def test_word_boundary_searches_vs_oracle(oracle, extend_dis):
    """Cases that put the search's bit operations on rows 63 / 64 of a 128 x 127 map: the only way through a wall, an obstacle
    dilated across the boundary, pursuers inflated across it, and the evader's view window straddling it."""
    W, H = 128, 127
    N = 4
    grids = np.zeros((4, W, H), np.uint8)
    p_state = np.zeros((4, N, 4))
    p_state[:, :, 0] = [[2, 3, 4, 5]] * 4                      # parked far away unless a case places them
    p_state[:, :, 1] = 1.0
    e_state = np.zeros((4, 4))
    target = np.zeros((4, 2), np.int32)
    # 0: a wall whose only gap is rows 62..65 (63 / 64 after the inflation by 1; closed at extend_dis 3, so the search retries)
    grids[0, 60, :62] = grids[0, 60, 66:] = 1
    e_state[0, :2], target[0] = (20.2, 30.1), (110, 100)
    # 1: a block on rows 63 / 64 right across the straight line
    grids[1, 40:44, 63:65] = 1
    e_state[1, :2], target[1] = (30.2, 63.9), (60, 63)
    # 2: pursuers on and around the boundary, inside the evader's view: their inflation crosses the word boundary
    p_state[2, :, :2] = [(38.0, 63.0), (38.0, 64.0), (40.0, 62.0), (41.0, 66.0)]
    e_state[2, :2], target[2] = (34.3, 63.6), (50, 63)
    # 3: view window [cy - 8, cy + 8) = rows 52..67 straddling the boundary; pursuers inside and just outside it
    p_state[3, :, :2] = [(44.0, 66.0), (44.0, 68.0), (36.0, 58.0), (48.0, 64.0)]
    e_state[3, :2], target[3] = (40.2, 60.1), (60, 72)
    lens, paths = _evader_vs_oracle(oracle, _cfg(W, H, attacker__extend_dis=extend_dis), grids, p_state, e_state, target)
    assert min(lens) > 2
    for b, path in enumerate(paths):                           # every search crosses the word boundary (start row included:
        ys = np.append(path[:, 1], round(e_state[b, 1]))       # the move may already have consumed the start cell)
        assert ys.min() <= 63 and ys.max() >= 64, b


def test_tall_hard_searches_vs_oracle(oracle):
    """Searches that run past the reachability-check budget on a 128 x 127 map: (a) the goal sealed inside a ring that straddles
    the word boundary - the reference's A* exhausts the component and returns [start]; (b) a serpentine maze whose path is longer
    than the pop budget."""
    W, H = 128, 127
    ring = np.zeros((W, H), np.uint8)
    ring[84:97, 58] = ring[84:97, 72] = 1
    ring[84, 58:73] = ring[96, 58:73] = 1                      # closed ring around (90, 65)
    maze = np.zeros((W, H), np.uint8)
    maze[43, 0:H - 6] = 1                                      # walls with alternating gaps
    maze[86, 6:H] = 1
    p_state = np.zeros((2, 4, 4))
    p_state[:, :, 0] = [[2, 3, 4, 5]] * 2
    p_state[:, :, 1] = 120.0
    e_state = np.array([[5.2, 5.1, 0, 0], [2.3, 2.2, 0, 0]], np.float64)
    target = np.array([[90, 65], [124, 3]], np.int32)
    lens, _ = _evader_vs_oracle(oracle, _cfg(W, H), np.stack([ring, maze]), p_state, e_state, target)
    assert lens[0] == 1                                        # sealed goal -> [start]
    assert lens[1] > 192                                       # longer than the pop budget before the reachability check


@pytest.mark.parametrize("size", [(128, 127), (80, 90)])
def test_tall_closed_loop_rollout_vs_oracle(oracle, size):
    """The whole closed loop (A* replanning, fused evader move, env / observe kernels, sensor tables) on maps with four and three
    bitmap words per column, against the oracle's closed loop: every discrete record and the fp64 pursuer state exact."""
    from distributed_multi_agent_reinforcement_learning_b200 import maps
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena
    from test_gpu_env import _rand_actions_numpy
    import bench
    W, H = size
    B, N, M, K = 64, 8, 8, 45
    cfg = _cfg(W, H, env__num_defender=N, env__max_steps=K, map__num_max_obstacle=176)
    wl = bench.host_workload(cfg, B, M, seed=21)
    env = BatchedPursuitEnv(cfg, B, num_maps=M)
    env.set_maps(wl["grids"], wl["inflated"])
    env.set_state(wl["p_state"], wl["e_state"], wl["target"], wl["map_id"], time_step=0)
    env.set_target_tape(wl["tape"])
    env.start_episode()
    actions = _rand_actions_numpy(99, B, N, 0, K)
    p = oracle.EnvParams.from_dict(env.params.as_dict())
    O = env.O
    st = dict(p_state=wl["p_state"].copy(), e_state=wl["e_state"].copy(), target=wl["target"].copy(),
              path=np.zeros((B, env.PATH_CAP, 2), np.int16), path_len=np.zeros(B, np.int32),
              grid=np.ascontiguousarray(wl["grids"]), inflated=np.ascontiguousarray(wl["inflated"]),
              raser=np.ascontiguousarray(maps.unpack_words(env.raser_bits.cpu().numpy(), O).reshape(M, W * H, O)),
              ob_count=np.minimum(env.boundary_count.cpu().numpy(), O).astype(np.int32), map_id=wl["map_id"].copy(),
              action_table=env.action_table.cpu().numpy().copy(), tape=np.ascontiguousarray(wl["tape"]),
              tape_pos=np.zeros(B, np.int32), p_adj=np.zeros((B, N, N), np.uint8), o_adj=np.zeros((B, N, O), np.uint8),
              e_adj=np.zeros((B, N), np.uint8), reward=np.zeros((B, N), np.int32), can_apply=np.zeros((B, N), np.uint8),
              collision=np.zeros(B, np.uint8), time_step=np.zeros(B, np.int32), done=np.zeros(B, np.uint8),
              wf_n=np.zeros(B, np.int64), wf_mean=np.zeros((B, N)), wf_S=np.zeros((B, N)), wf_std=np.zeros((B, N)),
              r_norm=np.zeros((B, N), np.float32), status=np.zeros(B, np.int32))
    rec = dict(reward=[], e_adj=[], o_adj=[], p_adj=[])
    for k in range(K):
        st["action"] = np.ascontiguousarray(actions[k])
        oracle.rollout_iteration_closed(p, st)
        for key in rec:
            rec[key].append(st[key].copy())
    assert not st["status"].any()
    assert np.stack(rec["o_adj"]).any() and np.stack(rec["e_adj"]).any()   # obstacles and the evader are actually seen
    arena = RolloutArena(env.params, B, K, env.device)
    env.rollout_closed(arena, K, 0, action_tape=torch.from_numpy(actions).cuda())
    torch.cuda.synchronize()
    assert int(env.evader_status.max().item()) == 0
    assert np.array_equal(env.path_len.cpu().numpy(), st["path_len"])
    assert np.array_equal(env.target.cpu().numpy(), st["target"])
    assert np.array_equal(env.tape_pos.cpu().numpy(), st["tape_pos"])
    np.testing.assert_allclose(env.e_state.cpu().numpy(), st["e_state"], rtol=1e-9, atol=1e-9)
    assert np.array_equal(arena.raw_reward.cpu().numpy(), np.stack(rec["reward"]))
    assert np.array_equal(arena.e_adj.cpu().numpy(), np.stack(rec["e_adj"]))
    assert np.array_equal(maps.unpack_words(arena.o_adj_bits.cpu().numpy(), O), np.stack(rec["o_adj"]))
    assert np.array_equal(maps.unpack_words(arena.p_adj_bits.cpu().numpy(), N), np.stack(rec["p_adj"]))
    assert np.array_equal(_bits(env.p_state.cpu().numpy()), _bits(st["p_state"]))
    assert (env.time_step == K).all()


def test_tall_device_reset_places_64_pursuers():
    """configs[4]'s 64 pursuers on 128 x 127 maps: the device reset seats every pursuer of every env under the reference's rule
    (>= 4 from every earlier pursuer, within comm range of one or two of them), which a 60 x 60 map has no room for."""
    from distributed_multi_agent_reinforcement_learning_b200 import maps
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    B, N, M, W, H = 1024, 64, 64, 128, 127
    cfg = _cfg(W, H, env__num_defender=N, map__num_max_obstacle=110)
    env = BatchedPursuitEnv(cfg, B, num_maps=M)
    env.reset_device(seed=5)
    torch.cuda.synchronize()
    assert int((env.reset_fail != 0).sum()) == 0
    grid = maps.unpack_words(env.grid_bits.cpu().numpy(), H)
    infl = maps.unpack_words(env.inflated_bits.cpu().numpy(), H)
    assert np.array_equal(infl, maps.dilate(grid, 2))
    ps, es, tg, mid = (t.cpu().numpy() for t in (env.p_state, env.e_state, env.target, env.map_id))
    comm, sen = float(cfg.defender.comm_range), float(cfg.defender.sen_range)
    for b in range(B):
        I = infl[mid[b]]
        assert not I[tg[b, 0], tg[b, 1]]
        work = I.copy()
        x, y = ps[b, :, 0], ps[b, :, 1]
        assert ((x >= 0) & (x <= W - 1) & (y >= 0) & (y <= H - 1)).all()
        d = np.hypot(x[:, None] - x[None, :], y[:, None] - y[None, :])
        cells = []
        for i in range(N):
            cx, cy = round(float(x[i])), round(float(y[i]))
            assert not work[cx, cy], (b, i)
            if i:
                assert (d[i, :i] >= 4).all() and 0 < (d[i, :i] < comm).sum() <= 2, (b, i)
            work[max(0, cx - 2):cx + 3, max(0, cy - 2):cy + 3] = 1
            cells.append((cx, cy))
        ex, ey = es[b, :2]
        assert not work[round(float(ex)), round(float(ey))]
        assert min(np.hypot(c[0] - ex, c[1] - ey) for c in cells) < sen
    assert (ps[:, :, 1] > 64).any() and (ps[:, :, 1] < 63).any()      # the pursuers use both halves of the map


def test_tall_map_end_to_end():
    """128 x 127 with the networks in the loop: the fused closed-loop rollout (1 and 4 env-group pipelines bit-identical), the
    CUDA-graph episode of explore_batched, and one train epoch + update."""
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena
    B, N, M, T, D = 64, 8, 8, 32, 1
    cfg = _cfg(128, 127, env__num_defender=N, env__max_steps=T, map__num_max_obstacle=176, algo__depth=D,
               algo__learner_device="cuda", algo__worker_device="cuda")
    torch.manual_seed(2)
    m = MAPPO(cfg, B, 16, "Learner")
    env = BatchedPursuitEnv(cfg, B, num_maps=M)
    env.reset_device(seed=7, tape_len=32)
    assert int((env.reset_fail != 0).sum()) == 0
    snap = env.snapshot()
    out = []
    for pipes in (1, 4):
        env.restore(snap)
        arena = RolloutArena(env.params, B, T, env.device)
        tb = m.rollout_batched(env, arena, T, seed=9, pipelines=pipes, history="store")
        torch.cuda.synchronize()
        assert int(env.evader_status.max().item()) == 0
        out.append([tb.a.clone(), tb.logp.clone(), tb.v.clone(), tb.hist_a.clone(), tb.hist_c.clone(), arena.raw_reward.clone(),
                    arena.r.clone(), env.p_state.clone(), env.e_state.clone(), env.path_len.clone(), env.target.clone()])
    for a, b in zip(*out):
        assert torch.equal(a, b)
    assert (out[0][9] > 1).any()                               # the evader planned real paths
    env.restore(snap)
    arena = RolloutArena(env.params, B, T, env.device)
    tb_g = m.explore_batched(env, arena, T, seed=9, history="store")
    torch.cuda.synchronize()
    assert int(env.evader_status.max().item()) == 0
    assert torch.equal(tb_g.a, out[0][0]) and torch.equal(tb_g.v, out[0][2])
    obj_c, obj_a, _, _ = m.train(tb, B * T * N, return_numpy=False)
    m.update(B * T * N)
    torch.cuda.synchronize()
    assert np.isfinite(obj_c) and np.isfinite(obj_a)
