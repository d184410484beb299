"""Rollout segments: an episode of T_ep steps collected as T_ep / S segments of S steps, with the GRU hidden states and the last D history
embeddings carried from one segment to the next (mappo_parallel.RolloutCarry), must be the episode collected in one piece, and training
on a segment must start from the state the rollout carried into it."""
import functools
import os
import subprocess
import sys

import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T_EP, B, SEED = 150, 24, 5
RECORDS = ("p_state_f32", "e_state_f32", "p_adj_bits", "e_adj", "o_adj_bits", "a_n", "r", "raw_reward", "active")


def _setup(N, D, quirks, mbs=None, seed=3, history_mode=None):
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    cfg = default_config(env__num_defender=N, env__max_steps=T_EP, algo__depth=D, algo__learner_device="cuda",
                         algo__worker_device="cuda")
    torch.manual_seed(seed)
    m = MAPPO(cfg, B, mbs or B // 3, "Learner", reference_quirks=quirks)
    with torch.no_grad():                                    # biases are zero-initialised: make them matter
        for p in m.ac_parameters:
            if p.dim() == 1:
                p.add_(0.05 * torch.randn_like(p))
    env = BatchedPursuitEnv(cfg, B, num_maps=4)
    env.reset_device(seed=seed + 10, tape_len=32)
    return m, env, env.snapshot()


def _episode(m, env, snap, S, history, pipes):
    """The episode from `snap` as T_EP / S segments (S = T_EP: one segment from a zero carry; S = None: carry=None).  Per segment: the
    batch's step outputs, its history (a whole minibatch regenerates it in replay mode), its start and next carry, the arena records."""
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    env.restore(snap)
    arena = RolloutArena(env.params, env.B, S or T_EP, env.device)
    carry = None if S is None else RolloutCarry.zeros(m, env.B, env.N)
    segs = []
    for _ in range(T_EP // (S or T_EP)):
        tb = m.rollout_batched(env, arena, S, seed=SEED, history=history, pipelines=pipes, carry=carry)
        mb = tb.minibatch(0, env.B)
        torch.cuda.synchronize()
        assert int(env.evader_status.max()) == 0
        segs.append(dict(a=tb.a.clone(), logp=tb.logp.clone(), v=tb.v.clone(), hist_a=mb.hist_a.clone(), hist_c=mb.hist_c.clone(),
                         rec={k: getattr(arena, k).clone() for k in RECORDS}, t0=tb.t0, carry=tb.carry))
        carry = tb.carry
    return segs, {k: x.clone() for k, x in env.snapshot().items()}


CASES = [pytest.param(N, D, q, pipes, h, id=f"N{N}-d{D}-{'quirks' if q else 'own'}-{pipes}pipe-{h}")
         for N in (8, 5) for D in (1, 3) for q in (True, False) for pipes in (1, 4) for h in ("store", "replay")
         if N == 8 or (pipes == 4 and h == "replay") or (pipes == 1 and h == "store")]


@functools.lru_cache(maxsize=None)
def _runs(N, D, quirks, pipes, history):
    m, env, snap = _setup(N, D, quirks)
    return {S: _episode(m, env, snap, S, history, pipes) for S in (None, T_EP, 50)}


@pytest.mark.parametrize("N,D,quirks,pipes,history", CASES)
def test_segments_equal_the_episode(N, D, quirks, pipes, history):
    runs = _runs(N, D, quirks, pipes, history)
    (ep,), final = runs[None]
    for S in (T_EP, 50):
        segs, final_s = runs[S]
        cat = lambda k: torch.cat([s[k] for s in segs])       # noqa: E731
        assert torch.equal(cat("a"), ep["a"]) and torch.equal(cat("logp"), ep["logp"]), S
        assert torch.equal(torch.cat([s["v"][:-1] for s in segs]), ep["v"][:-1]), S
        assert torch.equal(segs[-1]["v"][-1], ep["v"][-1]), S              # the episode's bootstrap value
        for k in RECORDS:
            assert torch.equal(torch.cat([s["rec"][k] for s in segs]), ep["rec"][k]), (S, k)
        for i, s in enumerate(segs):                          # history [S+D]: the carried prefix, then the segment's embeddings
            assert s["t0"] == i * S
            for k in ("hist_a", "hist_c"):
                assert torch.equal(s[k], ep[k][i * S:(i + 1) * S + D]), (S, i, k)
        for k in final:
            assert torch.equal(final_s[k], final[k]), (S, k)
        assert segs[-1]["carry"].t0 == T_EP


@pytest.mark.parametrize("N,D,quirks,pipes,history", CASES)
def test_bootstrap_value_equals_next_segment_value(N, D, quirks, pipes, history):
    if quirks and D >= 2:
        pytest.skip("under reference_quirks the bootstrap's history is [C(T-1), A(T-1) ... ] with the critic's newest embedding "
                    "first (h_fin in rollout_batched), the next step's aliased list is C(T-1), A(T-1), C(T-2): they differ for D >= 2")
    segs, _ = _runs(N, D, quirks, pipes, history)[50]
    for k in range(len(segs) - 1):
        assert torch.equal(segs[k]["v"][-1], segs[k + 1]["v"][0]), k


def _trace(m, tb, shuffle=False):
    tr = {}
    m.train(tb, B * 50, return_numpy=False, trace=tr, shuffle=shuffle, shuffle_seed=4)
    torch.cuda.synchronize()
    return tr


def _second_segment(m, env, snap, history, pipes=1):
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    env.restore(snap)
    arena = RolloutArena(env.params, env.B, 50, env.device)
    tb = m.rollout_batched(env, arena, 50, seed=SEED, history=history, pipelines=pipes, carry=RolloutCarry.zeros(m, env.B, env.N))
    tb = m.rollout_batched(env, arena, 50, seed=SEED, history=history, pipelines=pipes, carry=tb.carry)
    torch.cuda.synchronize()
    return tb, arena


@pytest.mark.parametrize("history", ["store", "replay"])
@pytest.mark.parametrize("D", [1, 3])
def test_training_forward_starts_from_the_carried_state(D, history):
    """reference_quirks=False: the training forward of segment 1 (steps 50..99) reproduces the log-probs and values the rollout stored
    (the tolerance of the whole-episode check in test_gpu_policy), and does not when it starts from zero hidden states and history."""
    import copy
    m, env, snap = _setup(8, D, False)
    tb, _ = _second_segment(m, env, snap, history)
    assert tb.t0 == 50 and tb.h0_a is not None and float(tb.h0_a.abs().max()) > 0
    u = m.critic.Mean
    sn0 = (u.weight_u.clone(), u.weight_v.clone())
    tr = _trace(m, tb)
    logp = torch.cat([t["logp"] for t in tr["mb"]], dim=1)
    val = torch.cat([t["val"] for t in tr["mb"]], dim=1)
    torch.testing.assert_close(logp, tb.logp, rtol=1e-5, atol=2e-5)
    torch.testing.assert_close(val, tb.v[:-1], rtol=1e-5, atol=2e-5)
    zero = copy.copy(tb)                                     # same segment, started like an episode: zero hidden states, zero prefix
    zero.h0_a = zero.h0_c = None
    if history == "store":
        zero.hist_a, zero.hist_c = tb.hist_a.clone(), tb.hist_c.clone()
        zero.hist_a[:D] = 0
        zero.hist_c[:D] = 0
    else:
        zero.prefix_a, zero.prefix_c = torch.zeros_like(tb.prefix_a), torch.zeros_like(tb.prefix_c)
    u.weight_u.copy_(sn0[0])
    u.weight_v.copy_(sn0[1])
    tr = _trace(m, zero)
    logp0 = torch.cat([t["logp"] for t in tr["mb"]], dim=1)
    val0 = torch.cat([t["val"] for t in tr["mb"]], dim=1)
    assert float((logp0 - tb.logp).abs().max()) > 1e-3 and float((val0 - tb.v[:-1]).abs().max()) > 1e-3


@pytest.mark.parametrize("shuffle", [False, True], ids=["sequential", "shuffled"])
@pytest.mark.parametrize("D", [1, 3])
def test_store_and_replay_segment_batches_train_identically(D, shuffle):
    m, env, snap = _setup(8, D, True)
    tbs = [_second_segment(m, env, snap, h)[0] for h in ("store", "replay")]
    assert tbs[1].hist_a is None and tbs[1].prefix_a is not None
    u = m.critic.Mean
    sn0 = (u.weight_u.clone(), u.weight_v.clone())
    traces, flats = [], []
    for tb in tbs:
        u.weight_u.copy_(sn0[0])
        u.weight_v.copy_(sn0[1])
        traces.append(_trace(m, tb, shuffle))
        flats.append(m.ac_optimizer.flat_grad.clone())
    ts, tr = traces
    assert torch.equal(ts["mb_grads"], tr["mb_grads"]) and torch.equal(flats[0], flats[1])
    for a, b in zip(ts["mb"], tr["mb"]):
        assert a["actor_loss"] == b["actor_loss"] and a["critic_loss"] == b["critic_loss"]
        for k in ("logp", "ent", "val"):
            assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize("history", ["store", "replay"])
def test_graph_segments_equal_eager_segments(history):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    m, env, snap = _setup(8, 3, True)
    eager, final = _episode(m, env, snap, 50, history, None)
    arena = RolloutArena(env.params, env.B, 50, env.device)
    for _ in range(2):                                       # the second episode replays the three captured graphs
        env.restore(snap)
        carry = RolloutCarry.zeros(m, env.B, env.N)
        for i in range(3):
            tb = m.explore_batched(env, arena, 50, seed=SEED, history=history, carry=carry)
            mb = tb.minibatch(0, env.B)
            torch.cuda.synchronize()
            e = eager[i]
            assert tb.t0 == 50 * i
            assert torch.equal(tb.a, e["a"]) and torch.equal(tb.logp, e["logp"]) and torch.equal(tb.v, e["v"]), i
            assert torch.equal(mb.hist_a, e["hist_a"]) and torch.equal(mb.hist_c, e["hist_c"]), i
            for k in RECORDS:
                assert torch.equal(getattr(arena, k), e["rec"][k]), (i, k)
            carry = tb.carry
        for k, x in env.snapshot().items():
            assert torch.equal(x, final[k]), k
    with pytest.raises(_lib.MarlError, match="engine's envs are at steps"):
        m.explore_batched(env, arena, 50, seed=SEED, history=history, carry=RolloutCarry.zeros(m, env.B, env.N, t0=50))


def test_training_state_carry_round_trip(tmp_path):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.checkpoint import load_training_state, save_training_state
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    m, env, snap = _setup(8, 3, False)
    tb, _ = _second_segment(m, env, snap, "store")
    plain, mid = str(tmp_path / "plain.pt"), str(tmp_path / "mid.pt")
    save_training_state(plain, m, env)                       # no carry: at an episode boundary
    save_training_state(mid, m, env, carry=tb.carry)
    got = RolloutCarry(7, *(torch.full_like(getattr(tb.carry, k), 3.0) for k in ("ha", "hc", "emb_a", "emb_c")))
    load_training_state(plain, m, env, carry=got)
    assert got.t0 == 0 and all(float(getattr(got, k).abs().max()) == 0 for k in ("ha", "hc", "emb_a", "emb_c"))
    load_training_state(plain, m, env)
    load_training_state(mid, m, env, carry=got)
    assert got.t0 == 100
    for k in ("ha", "hc", "emb_a", "emb_c"):
        assert torch.equal(getattr(got, k), getattr(tb.carry, k)), k
    with pytest.raises(_lib.MarlError, match="stopped inside an episode"):
        load_training_state(mid, m, env)
    small = RolloutCarry.zeros(m, B - 1, 8)
    with pytest.raises(_lib.MarlError, match="carry ha is"):
        load_training_state(mid, m, env, carry=small)
    assert small.t0 == 0


def _train_loop(*args):
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.join(ROOT, "tools", "train_loop.py"), "--envs", "32",
                                                                         "--maps", "8", "--steps", "150", "--segment", "50"] + list(args)
    out = subprocess.run(cmd, check=True, cwd=ROOT, timeout=900, capture_output=True, text=True).stdout
    return {int(line.split("exact ")[1].split()[0]): line.split("exact ")[1] for line in out.splitlines() if "exact " in line}


def test_resume_mid_episode_in_a_new_process_equals_uninterrupted_run(tmp_path):
    straight = _train_loop("--iters", "6")
    assert sorted(straight) == list(range(6))
    assert [straight[i].split()[2] == "-" for i in range(6)] == [True, True, False, True, True, False]
    first = _train_loop("--iters", "2", "--save-dir", str(tmp_path))            # stops after segment 1 of episode 0
    resumed = _train_loop("--iters", "6", "--resume", str(tmp_path))
    assert first == {i: straight[i] for i in range(2)}
    assert resumed == {i: straight[i] for i in range(2, 6)}
