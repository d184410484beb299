"""Auto-reset segment streams replayed from CUDA graphs (explore_batched(carry=..., auto_reset=AutoReset(..., tape="device"))): the
device-drawn target tape, the device-seeded entry points, and a graph stream that equals the eager stream and the whole episodes bit for
bit, shares its slabs across segment starts, trains like the eager batch and drives tools/train_loop.py --graph."""
import contextlib
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T_EP, B, TAPE = 150, 24, 32
RECORDS = ("p_state_f32", "e_state_f32", "p_adj_bits", "e_adj", "o_adj_bits", "a_n", "r", "raw_reward", "active")
RESET_SEED = lambda e: 40 + e                 # noqa: E731
SAMPLE_SEED = lambda e: 5 + 3 * e             # noqa: E731


def _cfg(N=8, D=1):
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    return default_config(env__num_defender=N, env__max_steps=T_EP, algo__depth=D, algo__learner_device="cuda", algo__worker_device="cuda")


def _engine(n_envs=B, n_maps=4, N=8):
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    return BatchedPursuitEnv(_cfg(N), n_envs, num_maps=n_maps)


def _setup(N, D, quirks, seed=3):
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    torch.manual_seed(seed)
    m = MAPPO(_cfg(N, D), B, B // 3, "Learner", reference_quirks=quirks)
    with torch.no_grad():                                    # biases are zero-initialised: make them matter
        for p in m.ac_parameters:
            if p.dim() == 1:
                p.add_(0.05 * torch.randn_like(p))
    env = _engine(N=N)
    env.wf0 = {k: getattr(env, k).clone() for k in ("wf_n", "wf_mean", "wf_S", "wf_std")}
    return m, env


def _state(env):
    torch.cuda.synchronize()
    out = {n: getattr(env, n).clone() for n in env._STATE}
    out["reset_fail"] = env.reset_fail.clone()
    return out


def _assert_same(a, b, what=""):
    assert a.keys() == b.keys()
    for k in a:
        assert torch.equal(a[k], b[k]), (what, k)


# ------------------------------------------------------------------------------------------------ device target tape
def _tape(env, seed, L=TAPE):
    env.reset_device(seed=seed, tape_len=L, tape="device")
    torch.cuda.synchronize()
    return env.target_tape.clone()


def test_device_tape_is_deterministic_per_seed_and_differs_across_seeds():
    env = _engine()
    a, b, c = _tape(env, 7), _tape(env, 7), _tape(env, 8)
    assert tuple(a.shape) == (B, TAPE, 2) and a.dtype == torch.int32
    assert torch.equal(a, b) and not torch.equal(a, c)
    assert float((a != c).float().mean()) > 0.9


def test_device_tape_range_and_uniformity():
    from scipy import stats
    env = _engine(n_envs=64, n_maps=8)
    W, H = env.params.W, env.params.H
    t = _tape(env, 2 ** 63 + 11, L=1024).cpu().numpy().reshape(-1, 2)          # 65 536 draws per coordinate
    assert t[:, 0].min() >= 0 and t[:, 0].max() < W and t[:, 1].min() >= 0 and t[:, 1].max() < H
    for col, n in ((0, W), (1, H)):
        counts = np.bincount(t[:, col], minlength=n)
        assert counts.min() > 0
        assert stats.chisquare(counts).pvalue > 1e-4, col
    cells = np.bincount(t[:, 0] * H + t[:, 1], minlength=W * H)                  # the pairs: independent coordinates
    assert stats.chisquare(cells).pvalue > 1e-4


def test_device_tape_row_does_not_depend_on_the_batch():
    small, large = _engine(24, 4), _engine(48, 4)
    assert torch.equal(_tape(small, 99), _tape(large, 99)[:24])


def test_device_and_torch_tapes_differ_only_in_the_tape():
    env = _engine()
    env.reset_device(seed=31, tape_len=TAPE, tape="torch")
    torch_state = _state(env)
    env.reset_device(seed=31, tape_len=TAPE, tape="device")
    dev_state = _state(env)
    assert not torch.equal(torch_state.pop("target_tape"), dev_state.pop("target_tape"))
    _assert_same(torch_state, dev_state)


@pytest.mark.parametrize("tape", ["torch", "device"])
def test_target_tape_storage_survives_reset_device(tape):
    env = _engine()
    env.reset_device(seed=1, tape_len=TAPE, tape=tape)
    ptr = env.target_tape.data_ptr()
    before = env.target_tape.clone()
    env.reset_device(seed=2, tape_len=TAPE, tape=tape)
    assert env.target_tape.data_ptr() == ptr and not torch.equal(env.target_tape, before)
    env.reset_device(seed=2, tape_len=TAPE + 1, tape=tape)                     # another length: new storage
    assert tuple(env.target_tape.shape) == (B, TAPE + 1, 2)


# ------------------------------------------------------------------------------------------------ device-seeded entry points
@pytest.mark.parametrize("seed", [0, 12345, 2 ** 63 + 5, 2 ** 64 - 1])
def test_device_seeded_reset_equals_the_by_value_reset(seed):
    """marl_map_generate_dseed / marl_env_reset_place_dseed / the tape from a device word equal the by-value calls with the same seed."""
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    env = _engine()
    env.reset_device(seed=seed, tape_len=TAPE, tape="device")
    by_value = _state(env)
    env.reset_device(seed=seed + 1, tape_len=TAPE, tape="device")
    word = torch.tensor([_lib.u64_bits(seed)], dtype=torch.int64, device=env.device)
    env.reset_device(seed=word, tape_len=TAPE, tape="device")
    _assert_same(by_value, _state(env))
    with pytest.raises(_lib.MarlError, match="needs tape='device'"):
        env.reset_device(seed=word, tape_len=TAPE)


def _policy_fixture():
    from distributed_multi_agent_reinforcement_learning_b200.fused_policy import FusedRolloutStep
    m, env = _setup(8, 2, True)
    env.reset_device(seed=5, tape_len=TAPE, tape="device")
    env.observe()
    w_eff, _ = m.critic.head_weight(update_buffers=False)
    fused = FusedRolloutStep(m, w_eff.reshape(-1).contiguous())
    g = torch.Generator(device="cuda").manual_seed(1)
    E = 128
    hist = [0.3 * torch.randn(B, 8, E, device="cuda", generator=g) for _ in range(2)]
    h0 = [0.1 * torch.randn(2, B * 8, E, device="cuda", generator=g) for _ in range(2)]
    o_count = torch.clamp(env.boundary_count, max=env.O).contiguous()
    oxy = env.boundary_xy.contiguous()
    outs = dict(emb_a=torch.empty(B, 8, E, device="cuda"), emb_c=torch.empty(B, 8, E, device="cuda"),
                act=torch.empty(B, 8, dtype=torch.int32, device="cuda"), logp=torch.empty(B, 8, device="cuda"),
                val=torch.empty(B, 8, device="cuda"), ha=torch.empty_like(h0[0]), hc=torch.empty_like(h0[1]))

    def step(seed=0, d_seed=None):
        outs["ha"].copy_(h0[0])
        outs["hc"].copy_(h0[1])
        fused.step(env, oxy, o_count, 17, seed, False, hist, hist, outs["emb_a"], outs["emb_c"], outs["ha"], outs["hc"], outs["act"],
                   outs["logp"], outs["val"], d_seed=d_seed)

    def result():
        torch.cuda.synchronize()
        return {k: v.clone() for k, v in outs.items()}
    return step, result


def test_device_seeded_policy_step_equals_the_by_value_step():
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    step, result = _policy_fixture()
    for seed in (3, 2 ** 63 + 9):
        step(seed)
        ref = result()
        step(seed + 1, d_seed=torch.tensor([_lib.u64_bits(seed)], dtype=torch.int64, device="cuda"))     # s->seed is ignored
        _assert_same(ref, result(), seed)


def test_captured_policy_step_follows_the_seed_word():
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    step, result = _policy_fixture()
    word = torch.tensor([_lib.u64_bits(11)], dtype=torch.int64, device="cuda")
    step(0, d_seed=word)                                     # warm-up (kernel attributes)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            step(0, d_seed=word)
    torch.cuda.current_stream().wait_stream(side)
    refs = {}
    for seed in (11, 12):
        step(seed)
        refs[seed] = result()
    assert not torch.equal(refs[11]["act"], refs[12]["act"])
    for seed in (12, 11):
        word.fill_(_lib.u64_bits(seed))
        graph.replay()
        _assert_same(refs[seed], result(), seed)


# ------------------------------------------------------------------------------------------------ graph streams
@contextlib.contextmanager
def _pipelines(n):
    old = os.environ.get("MARL_PIPELINES")
    os.environ["MARL_PIPELINES"] = str(n)
    try:
        yield
    finally:
        if old is None:
            os.environ.pop("MARL_PIPELINES")
        else:
            os.environ["MARL_PIPELINES"] = old


def _auto():
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import AutoReset
    return AutoReset(RESET_SEED, SAMPLE_SEED, tape_len=TAPE, tape="device")


def _first_episode(env):
    env.restore(env.wf0)
    env.reset_device(seed=RESET_SEED(0), tape_len=TAPE, tape="device")


def _stream(m, env, S, history, pipes, graph, steps=2 * T_EP):
    """Segments of S steps with auto_reset (eager, or replayed from the stream's graphs) from episode 0's start."""
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    arena = RolloutArena(env.params, env.B, S, env.device)
    _first_episode(env)
    carry, segs, auto = RolloutCarry.zeros(m, env.B, env.N), [], _auto()
    batches = []
    with _pipelines(pipes):
        for _ in range(-(-steps // S)):
            start = (carry.episode, carry.t0)
            if graph:
                tb = m.explore_batched(env, arena, S, history=history, carry=carry, auto_reset=auto)
            else:
                tb = m.rollout_batched(env, arena, S, history=history, pipelines=pipes, carry=carry, auto_reset=auto)
            torch.cuda.synchronize()
            assert int(env.evader_status.max()) == 0
            c = tb.carry
            segs.append(dict(a=tb.a.clone(), logp=tb.logp.clone(), v=tb.v.clone(), rec={k: getattr(arena, k).clone() for k in RECORDS},
                             start=start, boundary=tb.boundary, v_boot=None if tb.v_boot is None else tb.v_boot.clone(),
                             ended=None if tb.ended_collision is None else (tb.ended_collision.clone(), tb.ended_evader_status.clone()),
                             carry=(c.episode, c.t0) + tuple(getattr(c, k).clone() for k in ("ha", "hc", "emb_a", "emb_c"))))
            batches.append(tb)
            carry = tb.carry
    return segs, _state(env), batches


def _episodes(m, env, history, pipes, n=2):
    """Whole episodes: reset_device(RESET_SEED(e), tape="device") + rollout_batched(seed=SAMPLE_SEED(e))."""
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    arena = RolloutArena(env.params, env.B, T_EP, env.device)
    eps = []
    _first_episode(env)
    for e in range(n):
        if e:
            env.reset_device(seed=RESET_SEED(e), tape_len=TAPE, tape="device")
        tb = m.rollout_batched(env, arena, T_EP, seed=SAMPLE_SEED(e), history=history, pipelines=pipes)
        torch.cuda.synchronize()
        eps.append(dict(a=tb.a.clone(), logp=tb.logp.clone(), v=tb.v.clone(), rec={k: getattr(arena, k).clone() for k in RECORDS}))
    return eps


CASES = [pytest.param(D, pipes, h, id=f"d{D}-{pipes}pipe-{h}") for D in (1, 3) for pipes, h in ((1, "store"), (4, "replay"))]


@functools.lru_cache(maxsize=None)
def _runs(D, pipes, history):
    m, env = _setup(8, D, True)
    out = {None: _episodes(m, env, history, pipes)}
    for S in (50, 64, 76, 150):
        eager = _stream(m, env, S, history, pipes, graph=False)[:2]
        graph = _stream(m, env, S, history, pipes, graph=True)[:2]
        out[S] = (eager, graph)
    return out


@pytest.mark.parametrize("D,pipes,history", CASES)
@pytest.mark.parametrize("S", [50, 64, 76, 150])
def test_graph_stream_equals_the_eager_stream_and_the_episodes(S, D, pipes, history):
    runs = _runs(D, pipes, history)
    (eager, final_e), (graph, final_g) = runs[S]
    assert len(eager) == len(graph) == -(-2 * T_EP // S)
    for i, (x, y) in enumerate(zip(eager, graph)):
        for k in ("a", "logp", "v"):
            assert torch.equal(x[k], y[k]), (i, k)
        for k in RECORDS:
            assert torch.equal(x["rec"][k], y["rec"][k]), (i, k)
        assert x["start"] == y["start"] == divmod(i * S, T_EP), i
        assert x["boundary"] == y["boundary"], i
        assert (x["v_boot"] is None) == (y["v_boot"] is None) and (x["v_boot"] is None or torch.equal(x["v_boot"], y["v_boot"])), i
        assert (x["ended"] is None) == (y["ended"] is None), i
        if x["ended"] is not None:
            assert torch.equal(x["ended"][0], y["ended"][0]) and torch.equal(x["ended"][1], y["ended"][1]), i
        assert x["carry"][:2] == y["carry"][:2] == divmod((i + 1) * S, T_EP), i
        for a, b in zip(x["carry"][2:], y["carry"][2:]):
            assert torch.equal(a, b), i
    _assert_same(final_e, final_g, "engine where the stream stops")
    eps = runs[None]                                         # both streams collect the whole episodes
    n = 2 * T_EP
    ep = lambda k: torch.cat([e[k] for e in eps])            # noqa: E731
    assert torch.equal(torch.cat([s["a"] for s in graph])[:n], ep("a"))
    assert torch.equal(torch.cat([s["logp"] for s in graph])[:n], ep("logp"))
    assert torch.equal(torch.cat([s["v"][:-1] for s in graph])[:n], torch.cat([e["v"][:-1] for e in eps]))
    for k in RECORDS:
        assert torch.equal(torch.cat([s["rec"][k] for s in graph])[:n], torch.cat([e["rec"][k] for e in eps])), k
    for i, s in enumerate(graph):
        e, t0 = divmod(i * S, T_EP)
        if t0 + S >= T_EP and e < len(eps):                  # the episode ends in this segment: the whole episode's bootstrap value
            boot = s["v"][-1] if t0 + S == T_EP else s["v_boot"]
            assert torch.equal(boot, eps[e]["v"][T_EP]), i


def test_graph_stream_batches_of_different_starts_share_their_slabs():
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    m, env = _setup(8, 1, True)
    arena = RolloutArena(env.params, env.B, 64, env.device)
    _first_episode(env)
    carry, tbs = RolloutCarry.zeros(m, env.B, env.N), []
    for _ in range(3):
        tbs.append(m.explore_batched(env, arena, 64, history="store", carry=carry, auto_reset=_auto()))
        carry = tbs[-1].carry
    assert [tb.t0 for tb in tbs] == [0, 64, 128]
    for k in ("hist_a", "hist_c", "v", "logp"):
        assert len({getattr(tb, k).data_ptr() for tb in tbs}) == 1, k
    assert len({tb.carry.ha.data_ptr() for tb in tbs}) == 1
    assert (tbs[-1].carry.episode, tbs[-1].carry.t0, tbs[-1].boundary) == (1, 42, 22)


# ------------------------------------------------------------------------------------------------ training on a crossing graph batch
def _crossing(m, env, history, graph):
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    arena = RolloutArena(env.params, env.B, 64, env.device)
    _first_episode(env)
    carry, auto = RolloutCarry.zeros(m, env.B, env.N), _auto()
    for _ in range(3):
        if graph:
            tb = m.explore_batched(env, arena, 64, history=history, carry=carry, auto_reset=auto)
        else:
            tb = m.rollout_batched(env, arena, 64, history=history, carry=carry, auto_reset=auto)
        carry = tb.carry
    torch.cuda.synchronize()
    assert tb.boundary == 22
    return tb


@pytest.mark.parametrize("history", ["store", "replay"])
def test_training_on_a_crossing_graph_batch_equals_the_eager_batch(history):
    m, env = _setup(8, 3, True)
    u = m.critic.Mean
    sn0 = (u.weight_u.clone(), u.weight_v.clone())
    traces = []
    for graph in (False, True):
        u.weight_u.copy_(sn0[0])
        u.weight_v.copy_(sn0[1])
        tb = _crossing(m, env, history, graph)
        u.weight_u.copy_(sn0[0])
        u.weight_v.copy_(sn0[1])
        tr = {}
        m.train(tb, B * 64, return_numpy=False, trace=tr)
        torch.cuda.synchronize()
        traces.append((tr, m.ac_optimizer.flat_grad.clone()))
    (te, ge), (tg, gg) = traces
    assert torch.equal(te["adv"], tg["adv"]) and torch.equal(te["v_target"], tg["v_target"])
    assert torch.equal(te["mb_grads"], tg["mb_grads"]) and torch.equal(ge, gg)
    for a, b in zip(te["mb"], tg["mb"]):
        assert a["actor_loss"] == b["actor_loss"] and a["critic_loss"] == b["critic_loss"]
        for k in ("logp", "ent", "val"):
            assert torch.equal(a[k], b[k]), k


# ------------------------------------------------------------------------------------------------ tools/train_loop.py --graph
def _train_loop(*args):
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.join(ROOT, "tools", "train_loop.py"), "--envs", "32",
                                                                         "--maps", "8", "--steps", "150", "--segment", "64",
                                                                         "--auto-reset"] + list(args)
    out = subprocess.run(cmd, check=True, cwd=ROOT, timeout=900, capture_output=True, text=True).stdout
    return {int(line.split("exact ")[1].split()[0]): line.split("exact ")[1] for line in out.splitlines() if "exact " in line}


def test_train_loop_graph_equals_device_tape_and_resumes(tmp_path):
    eager = _train_loop("--device-tape", "--iters", "5")
    assert sorted(eager) == list(range(5))
    assert _train_loop("--graph", "--iters", "5") == eager
    first = _train_loop("--graph", "--iters", "3", "--save-dir", str(tmp_path))
    resumed = _train_loop("--graph", "--iters", "5", "--resume", str(tmp_path))
    assert first == {i: eager[i] for i in range(3)}
    assert resumed == {i: eager[i] for i in range(3, 5)}
