"""Auto-reset rollout segments: a stream of segments of any length S <= T_ep that run across episode boundaries
(rollout_batched(carry=..., auto_reset=AutoReset(...))) must collect the episodes that whole-episode rollouts collect from the same reset
and sampling seeds, bit for bit; its batches must train as the two episodes' pieces; and marl_gae_boundary must be marl_gae on each
piece."""
import copy
import ctypes
import functools
import math
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T_EP, B = 150, 24
RECORDS = ("p_state_f32", "e_state_f32", "p_adj_bits", "e_adj", "o_adj_bits", "a_n", "r", "raw_reward", "active")
RESET_SEED = lambda e: 40 + e                 # noqa: E731
SAMPLE_SEED = lambda e: 5 + 3 * e             # noqa: E731
EPISODES = 3


def _setup(N, D, quirks, mbs=None, seed=3):
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
    env.wf0 = {k: getattr(env, k).clone() for k in ("wf_n", "wf_mean", "wf_S", "wf_std")}
    return m, env


def _first_episode(env):
    """Episode 0's start, with the running reward statistics of a fresh engine (a device reset keeps them)."""
    env.restore(env.wf0)
    env.reset_device(seed=RESET_SEED(0), tape_len=32)


def _auto():
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import AutoReset
    return AutoReset(RESET_SEED, SAMPLE_SEED, tape_len=32)


def _episodes(m, env, history, pipes):
    """EPISODES whole-episode rollouts, episode e from reset_device(RESET_SEED(e)) sampled with SAMPLE_SEED(e), and the engine state at
    the start of episode 2, where an auto-reset stream of two episodes leaves it."""
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    arena = RolloutArena(env.params, env.B, T_EP, env.device)
    eps = []
    _first_episode(env)
    for e in range(EPISODES):
        if e:
            env.reset_device(seed=RESET_SEED(e), tape_len=32)
        if e == 2:
            final = {k: x.clone() for k, x in env.snapshot().items()}
        tb = m.rollout_batched(env, arena, T_EP, seed=SAMPLE_SEED(e), history=history, pipelines=pipes)
        mb = tb.minibatch(0, env.B)
        torch.cuda.synchronize()
        eps.append(dict(a=tb.a.clone(), logp=tb.logp.clone(), v=tb.v.clone(), hist_a=mb.hist_a.clone(), hist_c=mb.hist_c.clone(),
                        rec={k: getattr(arena, k).clone() for k in RECORDS}, collision=env.collision.clone(),
                        evader_status=env.evader_status.clone()))
    return eps, final


def _stream(m, env, S, history, pipes, steps):
    """Segments of S steps with auto_reset from episode 0's start until `steps` env steps are collected."""
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    arena = RolloutArena(env.params, env.B, S, env.device)
    _first_episode(env)
    carry, segs, auto = RolloutCarry.zeros(m, env.B, env.N), [], _auto()
    for _ in range(-(-steps // S)):
        start = (carry.episode, carry.t0)
        tb = m.rollout_batched(env, arena, S, history=history, pipelines=pipes, carry=carry, auto_reset=auto)
        torch.cuda.synchronize()
        assert int(env.evader_status.max()) == 0
        segs.append(dict(a=tb.a.clone(), logp=tb.logp.clone(), v=tb.v.clone(), rec={k: getattr(arena, k).clone() for k in RECORDS},
                         start=start, boundary=tb.boundary, v_boot=None if tb.v_boot is None else tb.v_boot.clone(),
                         ended=None if tb.ended_collision is None else (tb.ended_collision.clone(), tb.ended_evader_status.clone()),
                         carry=tb.carry))
        carry = tb.carry
    return segs, {k: x.clone() for k, x in env.snapshot().items()}


CASES = [pytest.param(N, D, q, pipes, h, id=f"N{N}-d{D}-{'quirks' if q else 'own'}-{pipes}pipe-{h}")
         for N in (8, 5) for D in (1, 3) for q in (True, False) for pipes, h in ((1, "store"), (4, "replay"))]


@functools.lru_cache(maxsize=None)
def _runs(N, D, quirks, pipes, history):
    m, env = _setup(N, D, quirks)
    out = {None: _episodes(m, env, history, pipes)}
    for S in (64, 76, 150):
        out[S] = _stream(m, env, S, history, pipes, 2 * T_EP)
    out["part"] = {r: _episode_2_start(m, env, out[None][1], r, history, pipes) for r in (20, 4)}
    return out


def _episode_2_start(m, env, start, r, history, pipes):
    """The engine after the first r steps of episode 2, collected without auto_reset from its start state `start` as segments whose
    length divides the episode (a segmented episode is the whole episode, test_gpu_rollout_segments)."""
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    env.restore(start)
    env.reset_device(seed=RESET_SEED(2), tape_len=32)         # the maps, which a snapshot does not hold
    S = math.gcd(r, T_EP)
    arena = RolloutArena(env.params, env.B, S, env.device)
    carry = RolloutCarry.zeros(m, env.B, env.N)
    for _ in range(r // S):
        carry = m.rollout_batched(env, arena, S, seed=SAMPLE_SEED(2), history=history, pipelines=pipes, carry=carry).carry
    torch.cuda.synchronize()
    return {k: x.clone() for k, x in env.snapshot().items()}


def _live(snap):
    """A snapshot without the A* path entries beyond path_len, which hold no state (a reset sets path_len to 0)."""
    out = dict(snap)
    out["path"] = snap["path"] * (torch.arange(snap["path"].shape[1], device=snap["path"].device)[None, :, None]
                                  < snap["path_len"][:, None, None].long())
    return out


@pytest.mark.parametrize("N,D,quirks,pipes,history", CASES)
@pytest.mark.parametrize("S", [64, 76, 150])
def test_stream_equals_the_episodes(S, N, D, quirks, pipes, history):
    runs = _runs(N, D, quirks, pipes, history)
    eps, final = runs[None]
    segs, final_s = runs[S]
    ep_cat = lambda k: torch.cat([e[k] for e in eps])                                       # noqa: E731
    ep_v = torch.cat([e["v"][:-1] for e in eps])
    n = len(segs) * S
    assert torch.equal(torch.cat([s["a"] for s in segs]), ep_cat("a")[:n])
    assert torch.equal(torch.cat([s["logp"] for s in segs]), ep_cat("logp")[:n])
    assert torch.equal(torch.cat([s["v"][:-1] for s in segs]), ep_v[:n])
    for k in RECORDS:
        assert torch.equal(torch.cat([s["rec"][k] for s in segs]), torch.cat([e["rec"][k] for e in eps])[:n]), k
    crossings = 0
    for i, s in enumerate(segs):
        e, t0 = divmod(i * S, T_EP)
        assert s["start"] == (e, t0), i
        # the bootstrap of a segment that ends inside an episode is the next step's value (see test_gpu_rollout_segments for why
        # not under reference_quirks with D >= 2)
        next_value = not (quirks and D >= 2)
        if t0 + S < T_EP:                                    # inside an episode: no reset
            assert s["boundary"] is None and s["ended"] is None
            assert not next_value or torch.equal(s["v"][-1], ep_v[(i + 1) * S]), i
        else:                                                # the episode ends at step k of the segment
            k = T_EP - t0
            ref = eps[e]
            assert s["boundary"] == (None if k == S else k), i
            boot = s["v"][-1] if k == S else s["v_boot"]
            assert torch.equal(boot, ref["v"][T_EP]), i      # the whole episode's critic-only bootstrap value
            assert torch.equal(s["ended"][0], ref["collision"]) and torch.equal(s["ended"][1], ref["evader_status"]), i
            assert int(s["ended"][1].max()) == 0
            crossings += k < S
            if k < S and next_value:
                assert torch.equal(s["v"][-1], ep_v[(i + 1) * S]), i
        c = s["carry"]                                       # the next segment's start and its history (zeros before the episode)
        e2, t2 = divmod((i + 1) * S, T_EP)
        assert (c.episode, c.t0) == (e2, t2), i
        if t2 == 0:
            assert all(float(getattr(c, x).abs().max()) == 0 for x in ("ha", "hc", "emb_a", "emb_c")), i
        else:
            assert torch.equal(c.emb_a, eps[e2]["hist_a"][t2:t2 + D]) and torch.equal(c.emb_c, eps[e2]["hist_c"][t2:t2 + D]), i
    assert crossings == {64: 2, 76: 2, 150: 0}[S]
    # the engine where the stream stops: at episode 2's start (S = 150), or after its first 320 - 300 = 20 (S = 64) / 4 (S = 76) steps
    ref = final if S == T_EP else runs["part"][n - 2 * T_EP]
    got, ref = _live(final_s), _live(ref)
    for k in ref:
        assert torch.equal(got[k], ref[k]), k


def test_stream_carry_after_a_late_crossing_has_zero_history():
    """S = 76: the boundary falls 2 steps before a segment's end (segment 1 covers steps 76..151), fewer than D = 3: the carried slab of
    the step before the new episode is zero, the next two are the new episode's embeddings."""
    segs, _ = _runs(8, 3, False, 1, "store")[76]
    c = segs[1]["carry"]
    assert (c.episode, c.t0) == (1, 2)
    assert float(c.emb_a[0].abs().max()) == 0 and float(c.emb_c[0].abs().max()) == 0
    assert float(c.emb_a[1:].abs().max()) > 0 and float(c.emb_c[1:].abs().max()) > 0


# ------------------------------------------------------------------------------------------------ marl_gae_boundary
def _gae(B_, T, N, r, v, active, norm, k=None, v_boot=None):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    L = _lib.lib()
    adv, vt = torch.empty_like(r), torch.empty_like(r)
    ws = torch.zeros(int(L.marl_gae_workspace_bytes(B_, T, N)), dtype=torch.uint8, device=r.device)
    g, gl = ctypes.c_float(0.99), ctypes.c_float(0.99 * 0.95)
    if k is None:
        rc = L.marl_gae(B_, T, N, _lib.ptr(r), _lib.ptr(v), _lib.ptr(active), 1, g, gl, int(norm), _lib.ptr(adv), _lib.ptr(vt),
                        _lib.ptr(ws), _lib.stream_ptr())
    else:
        rc = L.marl_gae_boundary(B_, T, N, k, _lib.ptr(r), _lib.ptr(v), _lib.ptr(v_boot), _lib.ptr(active), g, gl, int(norm),
                                 _lib.ptr(adv), _lib.ptr(vt), _lib.ptr(ws), _lib.stream_ptr())
    _lib.check(rc, "gae")
    torch.cuda.synchronize()
    return adv, vt


def _gae_f64(r, v, v_boot, active, k):
    T = r.shape[0]
    adv = np.zeros_like(r, dtype=np.float64)
    g, gl = np.float64(np.float32(0.99)), np.float64(np.float32(0.99 * 0.95))
    for lo, hi, v_end in ((k, T, v[T]), (0, k, v_boot)):
        gae, v_next = 0.0, v_end.astype(np.float64)
        for t in range(hi - 1, lo - 1, -1):
            delta = (r[t] + g * v_next - v[t]) * active[t]
            gae = delta + gl * gae
            adv[t] = gae
            v_next = v[t].astype(np.float64)
    return adv, adv + v[:T]


@pytest.mark.parametrize("B_,T,N,k", [(3, 7, 4, 3), (24, 64, 8, 50), (257, 33, 15, 1), (16, 76, 5, 75)])
def test_gae_boundary_is_gae_on_each_piece(B_, T, N, k):
    gen = torch.Generator(device="cuda").manual_seed(T * 100 + k)
    rnd = lambda *s: torch.randn(*s, generator=gen, device="cuda")       # noqa: E731
    r, v, v_boot = rnd(T, B_, N), rnd(T + 1, B_, N), rnd(B_, N)
    active = (torch.rand(T, B_, N, generator=gen, device="cuda") < 0.9).float()
    adv, vt = _gae(B_, T, N, r, v, active, False, k, v_boot)
    a2, vt2 = _gae(B_, T - k, N, r[k:].contiguous(), v[k:].contiguous(), active[k:].contiguous(), False)
    a1, vt1 = _gae(B_, k, N, r[:k].contiguous(), torch.cat([v[:k], v_boot[None]]).contiguous(), active[:k].contiguous(), False)
    assert torch.equal(adv, torch.cat([a1, a2])) and torch.equal(vt, torch.cat([vt1, vt2]))
    # piece 1 ends an episode of T_ep = 150 steps: its advantages are that whole episode's at the same steps
    t_ep = 150
    r_ep, v_ep, act_ep = rnd(t_ep, B_, N), rnd(t_ep + 1, B_, N), torch.ones(t_ep, B_, N, device="cuda")
    r_ep[t_ep - k:], v_ep[t_ep - k:t_ep], act_ep[t_ep - k:], v_ep[t_ep] = r[:k], v[:k], active[:k], v_boot
    a_ep, vt_ep = _gae(B_, t_ep, N, r_ep, v_ep, act_ep, False)
    assert torch.equal(adv[:k], a_ep[t_ep - k:]) and torch.equal(vt[:k], vt_ep[t_ep - k:])
    # a float64 restatement of the whole computation: the two recursions and the normalisation over all T*B*N samples (the float32
    # recursions of the kernel round at every step, hence 1e-5) ...
    adv_n, vt_n = _gae(B_, T, N, r, v, active, True, k, v_boot)
    act64 = active.double().cpu().numpy()
    ref_adv, ref_vt = _gae_f64(*(x.double().cpu().numpy() for x in (r, v, v_boot, active)), k)
    norm = lambda a: (a - a.mean()) / (a.reshape(-1).std(ddof=1) + 1e-5) * act64       # noqa: E731
    np.testing.assert_allclose(adv.cpu().numpy(), ref_adv, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(vt_n.cpu().numpy(), ref_vt, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(adv_n.cpu().numpy(), norm(ref_adv), rtol=1e-5, atol=1e-5)
    # ... and the normalisation step alone, in float64 from the kernel's own un-normalised advantages, to 1e-6
    np.testing.assert_allclose(adv_n.cpu().numpy(), norm(adv.double().cpu().numpy()), rtol=1e-6, atol=1e-6)


def test_gae_boundary_refuses_bad_arguments():
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    L = _lib.lib()
    x = torch.zeros(8, 2, 3, device="cuda")
    v = torch.zeros(9, 2, 3, device="cuda")
    vb = torch.zeros(2, 3, device="cuda")
    ws = torch.zeros(int(L.marl_gae_workspace_bytes(2, 8, 3)), dtype=torch.uint8, device="cuda")
    p = _lib.ptr
    for Bx, T, N, k, vb_ptr in ((2, 8, 3, 0, p(vb)), (2, 8, 3, 8, p(vb)), (2, 8, 3, -1, p(vb)), (2, 1, 3, 1, p(vb)), (0, 8, 3, 4, p(vb)),
                                (2, 8, 0, 4, p(vb)), (2, 8, 3, 4, None)):
        rc = L.marl_gae_boundary(Bx, T, N, k, p(x), p(v), vb_ptr, p(x), ctypes.c_float(0.99), ctypes.c_float(0.9), 1, p(x), p(x),
                                 p(ws), _lib.stream_ptr())
        assert rc == -1, (Bx, T, N, k)                       # MARL_EINVAL


# ------------------------------------------------------------------------------------------------ training on a crossing batch
def _crossing_batch(m, env, history, S=64):
    """The second segment of an S = 64 stream: steps 64..127 of episode 0 - no boundary; the third: 128..149 of episode 0 and 0..41 of
    episode 1, crossing at k = 22."""
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutCarry
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    arena = RolloutArena(env.params, env.B, S, env.device)
    _first_episode(env)
    carry, auto = RolloutCarry.zeros(m, env.B, env.N), _auto()
    for _ in range(3):
        tb = m.rollout_batched(env, arena, S, history=history, carry=carry, auto_reset=auto)
        carry = tb.carry
    torch.cuda.synchronize()
    assert tb.boundary == T_EP - 2 * S
    return tb


def _trace(m, tb, shuffle=False):
    tr = {}
    m.train(tb, B * 64, return_numpy=False, trace=tr, shuffle=shuffle, shuffle_seed=4)
    torch.cuda.synchronize()
    return tr


@pytest.mark.parametrize("history", ["store", "replay"])
@pytest.mark.parametrize("D", [1, 3])
def test_training_forward_of_a_crossing_segment_reproduces_the_rollout(D, history):
    """reference_quirks=False: the training forward of a crossing segment reproduces the log-probs and values the rollout stored, and
    does not when the segment runs as one GRU / history pass (no reset at the boundary)."""
    m, env = _setup(8, D, False)
    tb = _crossing_batch(m, env, history)
    u = m.critic.Mean
    sn0 = (u.weight_u.clone(), u.weight_v.clone())
    tr = _trace(m, tb)
    logp = torch.cat([t["logp"] for t in tr["mb"]], dim=1)
    val = torch.cat([t["val"] for t in tr["mb"]], dim=1)
    torch.testing.assert_close(logp, tb.logp, rtol=1e-5, atol=2e-5)
    torch.testing.assert_close(val, tb.v[:-1], rtol=1e-5, atol=2e-5)
    if history == "replay":
        return
    whole = copy.copy(tb)                                    # the same segment without the split
    whole.boundary = None
    u.weight_u.copy_(sn0[0])
    u.weight_v.copy_(sn0[1])
    tr = _trace(m, whole)
    logp0 = torch.cat([t["logp"] for t in tr["mb"]], dim=1)
    val0 = torch.cat([t["val"] for t in tr["mb"]], dim=1)
    k = tb.boundary
    assert float((logp0[k:] - tb.logp[k:]).abs().max()) > 1e-3 and float((val0[k:] - tb.v[k:-1]).abs().max()) > 1e-3


@pytest.mark.parametrize("shuffle", [False, True], ids=["sequential", "shuffled"])
@pytest.mark.parametrize("D", [1, 3])
def test_store_and_replay_crossing_batches_train_identically(D, shuffle):
    m, env = _setup(8, D, True)
    tbs = [_crossing_batch(m, env, h) for h in ("store", "replay")]
    assert tbs[1].hist_a is None and tbs[1].replay2 is not None
    u = m.critic.Mean
    sn0 = (u.weight_u.clone(), u.weight_v.clone())
    traces, flats = [], []
    for tb in tbs:
        u.weight_u.copy_(sn0[0])
        u.weight_v.copy_(sn0[1])
        traces.append(_trace(m, tb, shuffle))
        flats.append(m.ac_optimizer.flat_grad.clone())
    ts, tr = traces
    assert torch.equal(ts["adv"], tr["adv"]) and torch.equal(ts["v_target"], tr["v_target"])
    assert torch.equal(ts["mb_grads"], tr["mb_grads"]) and torch.equal(flats[0], flats[1])
    for a, b in zip(ts["mb"], tr["mb"]):
        assert a["actor_loss"] == b["actor_loss"] and a["critic_loss"] == b["critic_loss"]
        for k in ("logp", "ent", "val"):
            assert torch.equal(a[k], b[k]), k


# ------------------------------------------------------------------------------------------------ tools/train_loop.py
def _train_loop(*args):
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.join(ROOT, "tools", "train_loop.py"), "--envs", "32",
                                                                         "--maps", "8", "--steps", "150"] + list(args)
    out = subprocess.run(cmd, check=True, cwd=ROOT, timeout=900, capture_output=True, text=True).stdout
    return {int(line.split("exact ")[1].split()[0]): line.split("exact ")[1] for line in out.splitlines() if "exact " in line}


def test_train_loop_auto_reset_is_reproducible_and_resumable(tmp_path):
    straight = _train_loop("--segment", "64", "--auto-reset", "--iters", "5")
    assert sorted(straight) == list(range(5))
    assert [straight[i].split()[2] == "-" for i in range(5)] == [True, True, False, True, False]   # episodes end in segments 2 and 4
    assert _train_loop("--segment", "64", "--auto-reset", "--iters", "5") == straight
    first = _train_loop("--segment", "64", "--auto-reset", "--iters", "3", "--save-dir", str(tmp_path))   # after the first crossing
    resumed = _train_loop("--segment", "64", "--auto-reset", "--iters", "5", "--resume", str(tmp_path))
    assert first == {i: straight[i] for i in range(3)}
    assert resumed == {i: straight[i] for i in range(3, 5)}


def test_train_loop_auto_reset_equals_divisor_segments():
    assert _train_loop("--segment", "50", "--auto-reset", "--iters", "6") == _train_loop("--segment", "50", "--iters", "6")
