"""GPU checks of the PPO diagnostics (csrc/train_stats.cu, MAPPO.train(stats=True), tools/train_loop.py --stats / --target-kl):
the kernel and the combine against float64 numpy restatements (bit-stable, graph-capturable), the statistics of train() against a
restatement from its trace in every batch mode, training bit-identical with the statistics on and off, independence of the number of
minibatches in flight, the reference's own per-minibatch values, two ranks, and the driver."""
import math
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN_DIR, AlgoFixture

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("entropy", "approx_kl", "approx_kl_k1", "clip_frac", "ratio_min", "ratio_max", "value_clip_frac", "explained_variance",
        "rollout_explained_variance", "adv_mean", "adv_std", "return_mean", "grad_norm_max", "grad_norm_last", "clipped_minibatches",
        "rows")


def np_sums(logp, old, ent, val, v_old, vt, active, eps):
    """The 16 minibatch slots in float64 (include/marl_b200.h), and per slot the sum of its terms' absolute values."""
    f = lambda x: np.asarray(x, np.float64).reshape(-1)           # noqa: E731
    a = f(active)
    on = a != 0
    a, lr = a[on], (f(logp) - f(old))[on]
    r = np.exp(lr)
    e, vt_ = f(ent)[on], f(vt)[on]
    res = vt_ - f(val)[on]
    terms = {0: a, 1: a * e, 2: -a * lr, 3: a * ((r - 1) - lr), 4: a * (np.abs(r - 1) > eps), 8: a * vt_, 9: a * vt_ * vt_,
             10: a * res, 11: a * res * res}
    if v_old is not None:
        vo = f(v_old)[on]
        x = vt_ - vo
        terms.update({7: a * (np.abs(f(val)[on] - vo) > eps), 12: a * x, 13: a * x * x})
    s, mag = np.zeros(16), np.zeros(16)
    for j, t in terms.items():
        s[j], mag[j] = t.sum(), np.abs(t).sum()
    s[5] = lr.max() if lr.size else -np.inf
    s[6] = lr.min() if lr.size else np.inf
    s[14] = 0.0 if v_old is None else 1.0
    s[15] = f(logp).size
    return s, mag


def _check_sums(got, want, mag):
    got = got.cpu().numpy()
    for j in range(16):
        if j in (5, 6, 14, 15):
            assert got[j] == want[j], (j, got[j], want[j])
        else:
            assert abs(got[j] - want[j]) <= 1e-12 * mag[j], (j, got[j], want[j], mag[j])


def _inputs(R, p_active, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    rn = lambda s=1.0: s * torch.randn(R, device="cuda", generator=g)       # noqa: E731
    old = rn() - 2.0
    logp = old + rn(0.1)
    active = (torch.rand(R, device="cuda", generator=g) < p_active).float()
    return logp, old, rn().abs(), rn(), rn(), rn(), active


# ------------------------------------------------------------------------------------------------ 1: kernel and combine
@pytest.mark.parametrize("with_v_old", [False, True], ids=["no_value_clip", "value_clip"])
@pytest.mark.parametrize("R,p_active", [(1, 1.0), (1000, 0.7), (1000, 0.0), ((1 << 20) + 7, 0.8)])
def test_kernel_matches_float64_restatement(R, p_active, with_v_old):
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    logp, old, ent, val, v_old, vt, active = _inputs(R, p_active, R)
    vo = v_old if with_v_old else None
    eps = 0.05
    got = ops.ppo_stats(logp, old, ent, val, vo, vt, active, eps)
    want, mag = np_sums(*(None if t is None else t.cpu().numpy() for t in (logp, old, ent, val, vo, vt, active)), eps=np.float32(eps))
    _check_sums(got, want, mag)
    if p_active == 0.0:
        assert got[5].item() == -math.inf and got[6].item() == math.inf and got[0].item() == 0.0
    again = ops.ppo_stats(logp, old, ent, val, vo, vt, active, eps)
    assert torch.equal(got, again)
    # the same call captured in a CUDA graph (workspace and output allocated by the graph's pool) gives the same bits
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.ppo_stats(logp, old, ent, val, vo, vt, active, eps)       # warm-up on the side stream
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = ops.ppo_stats(logp, old, ent, val, vo, vt, active, eps)
    captured.fill_(0)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, got)


@pytest.mark.parametrize("with_norms", [False, True])
def test_combine_adds_rows_in_index_order(with_norms):
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    n = 7
    g = torch.Generator(device="cuda").manual_seed(2)
    rows = torch.randn(n, 16, device="cuda", dtype=torch.float64, generator=g) * 1e3
    rows[3, 5], rows[2, 6] = -math.inf, math.inf                   # a minibatch without active rows
    norms = (torch.rand(n, device="cuda", generator=g) * 10).float() if with_norms else None
    out = ops.ppo_stats_combine(rows, norms, 5.0).cpu().numpy()
    h = rows.cpu().numpy()
    want = h[0].copy()
    for m in range(1, n):
        for j in range(16):
            want[j] = max(want[j], h[m, j]) if j == 5 else (min(want[j], h[m, j]) if j == 6 else want[j] + h[m, j])
    assert np.array_equal(out[:16], want)
    assert out[16] == n
    if with_norms:
        nh = norms.cpu().numpy().astype(np.float64)
        assert (out[17], out[18], out[19], out[20]) == (n, nh.max(), nh[-1], float((nh > 5.0).sum()))
    else:
        assert (out[17:21] == 0).all()
    assert (out[21:] == 0).all()


# ------------------------------------------------------------------------------------------------ 2-4: through MAPPO.train
def _restated(trace, tb, perm, mbs, eps, max_norm, value_clip):
    """The TrainStats of one epoch from its trace and the batch: every minibatch's rows restated in float64, added in index order."""
    from distributed_multi_agent_reinforcement_learning_b200.train_stats import TrainStats
    B = tb.B
    total = np.zeros(24)
    total[5], total[6] = -np.inf, np.inf
    for m, lo in enumerate(range(0, B, mbs)):
        idx = torch.arange(lo, min(lo + mbs, B), device="cuda") if perm is None else perm[lo:lo + mbs]
        sel = lambda x: x[:, idx].cpu().numpy()                   # noqa: E731
        rec = trace["mb"][m]
        s, _ = np_sums(rec["logp"].cpu().numpy(), sel(tb.logp), rec["ent"].cpu().numpy(), rec["val"].cpu().numpy(),
                       sel(tb.v[:-1]) if value_clip else None, sel(trace["v_target"]), sel(tb.active), np.float32(eps))
        for j in range(16):
            total[j] = max(total[j], s[j]) if j == 5 else (min(total[j], s[j]) if j == 6 else total[j] + s[j])
    n_mb = len(trace["mb"])
    total[16] = n_mb
    if max_norm is not None:
        norms = np.array([float(x) for x in trace["grad_norms"]])
        total[17:21] = n_mb, norms.max(), norms[-1], (norms > max_norm).sum()
    return TrainStats.from_sums(total, eps, max_norm)


def _assert_stats_close(got, want, rtol=1e-9):
    for k in KEYS:
        a, b = getattr(got, k), getattr(want, k)
        if b is None or a is None:
            assert a is None and b is None, k
        elif isinstance(b, float) and math.isnan(b):
            assert math.isnan(a), k
        else:
            assert a == pytest.approx(b, rel=rtol, abs=1e-12), (k, a, b)


def _mappo(B, N, D, T_ep, mbs, seed=3, **over):
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    cfg = default_config(env__num_defender=N, env__max_steps=T_ep, algo__depth=D, algo__learner_device="cuda", algo__worker_device="cuda",
                         **over)
    torch.manual_seed(seed)
    m = MAPPO(cfg, B, mbs, "Learner")
    with torch.no_grad():                                    # biases are zero-initialised: make them matter
        for p in m.ac_parameters:
            if p.dim() == 1:
                p.add_(0.05 * torch.randn_like(p))
    env = BatchedPursuitEnv(cfg, B, num_maps=4)
    env.reset_device(seed=seed + 10, tape_len=32)
    return m, env


def _batch(mode, m, env):
    """A small real rollout batch: a whole episode (store or replay history), or an auto-reset segment that crosses the boundary."""
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import AutoReset, RolloutCarry
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    T_ep = int(m.cfg.env.max_steps)
    if mode in ("store", "replay"):
        arena = RolloutArena(env.params, env.B, T_ep, env.device)
        return m.rollout_batched(env, arena, T_ep, seed=5, history=mode), arena
    S = 16
    arena = RolloutArena(env.params, env.B, S, env.device)
    auto = AutoReset(lambda e: 20 + e, lambda e: 5 + e, tape_len=32)
    env.reset_device(seed=20, tape_len=32)
    carry = RolloutCarry.zeros(m, env.B, env.N)
    tb = m.rollout_batched(env, arena, S, carry=carry, auto_reset=auto)
    tb = m.rollout_batched(env, arena, S, carry=tb.carry, auto_reset=auto)       # steps 16..31 of a 24-step episode
    assert tb.boundary == T_ep - S
    return tb, arena


MODES = [("store", False), ("replay", False), ("store", True), ("auto_reset", False), ("auto_reset", True)]


@pytest.mark.parametrize("mode,shuffle", MODES, ids=[f"{m}{'-shuffle' if s else ''}" for m, s in MODES])
def test_train_stats_match_restatement_and_leave_training_unchanged(mode, shuffle):
    B, N, D, T_ep, mbs = 24, 8, 1, 24, 8
    m, env = _mappo(B, N, D, T_ep, mbs)
    tb, _arena = _batch(mode, m, env)
    torch.cuda.synchronize()
    opt, u = m.ac_optimizer, m.critic.Mean
    start = [t.clone() for t in (opt.flat_param, opt.exp_avg, opt.exp_avg_sq, u.weight_u, u.weight_v)]
    runs = []
    for stats in (False, True, False, True):                # two epochs each way, every one from the same state
        for t, s0 in zip((opt.flat_param, opt.exp_avg, opt.exp_avg_sq, u.weight_u, u.weight_v), start):
            t.copy_(s0)
        opt.step_count = 0
        trace = {}
        m.last_train_stats = None
        out = m.train(tb, B * T_ep, return_numpy=False, trace=trace, shuffle=shuffle, shuffle_seed=4, stats=stats)
        st = m.last_train_stats
        m.update(B * T_ep)
        torch.cuda.synchronize()
        runs.append(dict(out=out[:2], st=st, trace=trace, state=[t.clone() for t in (opt.flat_param, opt.exp_avg, opt.exp_avg_sq)]))
    off, on = runs[0], runs[1]
    assert off["st"] is None and on["st"] is not None
    assert on["out"] == off["out"]
    for a, b in zip(on["state"], off["state"]):
        assert torch.equal(a, b)                             # parameters and both Adam moments, bit for bit
    assert torch.equal(runs[1]["st"].sums, runs[3]["st"].sums)
    perm = on["trace"].get("permutation")
    want = _restated(on["trace"], tb, perm, mbs, m.epsilon, 5.0, m.use_value_clip)
    _assert_stats_close(on["st"], want)
    assert on["st"].rows == int(tb.active.sum()) and on["st"].minibatches == B // mbs
    assert on["st"].sums.is_cuda and on["st"].sums.dtype == torch.float64


def test_train_stats_do_not_depend_on_minibatches_in_flight(monkeypatch):
    from distributed_multi_agent_reinforcement_learning_b200 import mappo_parallel
    B, N, T_ep, mbs = 24, 8, 24, 4
    m, env = _mappo(B, N, 1, T_ep, mbs)
    tb, _arena = _batch("store", m, env)
    u = m.critic.Mean
    sn = (u.weight_u.clone(), u.weight_v.clone())
    sums = []
    for k in (1, 3):
        monkeypatch.setattr(mappo_parallel, "CONCURRENT_MINIBATCHES", k)
        u.weight_u.copy_(sn[0])
        u.weight_v.copy_(sn[1])
        m.train(tb, B * T_ep, return_numpy=False, stats=True)
        sums.append(m.last_train_stats.sums.clone())
    assert torch.equal(sums[0], sums[1])


def test_train_stats_without_value_clip_or_gradient_clip():
    B, N, T_ep, mbs = 24, 8, 24, 8
    m, env = _mappo(B, N, 1, T_ep, mbs, algo__use_value_clip=False, algo__use_grad_clip=False)
    tb, _arena = _batch("store", m, env)
    trace = {}
    m.train(tb, B * T_ep, return_numpy=False, trace=trace, stats=True)
    st = m.last_train_stats
    assert st.value_clip_frac is None and st.adv_mean is None and st.grad_norm_max is None and st.clipped_minibatches is None
    _assert_stats_close(st, _restated(trace, tb, None, mbs, m.epsilon, None, False))


def test_three_hop_train_stats(monkeypatch):
    """mappo_3hop.MAPPO.train(stats=True) on the golden batch: training is unchanged, and the statistics equal a float64 restatement
    from the per-minibatch logp / ent / val that `ppo_head` returned, the batch's own old log-probs, v_old and active mask (sliced here,
    independently of train()), the GAE targets and the pre-clip norms that `clip_grad_norm_` returned."""
    import glob
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    from distributed_multi_agent_reinforcement_learning_b200.train_stats import TrainStats
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_gpu_gnn3hop import _Big, _build
    fx = np.load(sorted(glob.glob(os.path.join(GOLDEN_DIR, "gnn3hop_*.npz")))[0])
    m, (N, O, B, T, mb, emb) = _build(fx)
    buf = {k[4:]: torch.from_numpy(fx[k]) for k in fx.files if k.startswith("buf.")}
    heads, norms = [], []
    head, clip = ops.ppo_head, ops.clip_grad_norm_

    def rec_head(*a, **kw):
        out = head(*a, **kw)
        heads.append(tuple(t.detach().clone() for t in out[2:5]))
        return out

    def rec_clip(*a, **kw):
        out = clip(*a, **kw)
        norms.append(float(out))
        return out
    monkeypatch.setattr(ops, "ppo_head", rec_head)
    monkeypatch.setattr(ops, "clip_grad_norm_", rec_clip)
    opt, u = m.ac_optimizer, m.critic.Mean
    sn = (u.weight_u.clone(), u.weight_v.clone())
    res = []
    for stats in (False, True):
        u.weight_u.copy_(sn[0])
        u.weight_v.copy_(sn[1])
        heads.clear()
        norms.clear()
        out = m.train(_Big(buf, T), 1000, stats=stats)
        res.append((out[:2], opt.flat_grad.clone(), m.last_train_stats))
    assert res[0][0] == res[1][0] and torch.equal(res[0][1], res[1][1]) and res[0][2] is None
    st = res[1][2]
    batch = {k: v.cuda() for k, v in buf.items()}
    _adv, vt = m.gae(batch, T)
    starts = list(range(0, B, mb))
    assert len(heads) == len(starts) == len(norms) and st.minibatches == len(starts)
    total = np.zeros(24)
    total[5], total[6] = -np.inf, np.inf
    for (logp, ent, val), lo in zip(heads, starts):
        idx = slice(lo, min(lo + mb, B))
        sl = lambda k: batch[k][idx, :T].cpu().numpy()           # noqa: E731
        s, _ = np_sums(logp.cpu().numpy(), sl("a_logprob_n"), ent.cpu().numpy(), val.cpu().numpy(), sl("v_n"), vt[idx].cpu().numpy(),
                       sl("active"), np.float32(m.epsilon))
        for j in range(16):
            total[j] = max(total[j], s[j]) if j == 5 else (min(total[j], s[j]) if j == 6 else total[j] + s[j])
    nh = np.array(norms)
    total[16:21] = len(starts), len(starts), nh.max(), nh[-1], (nh > 10.0).sum()
    _assert_stats_close(st, TrainStats.from_sums(total, m.epsilon, 10.0))
    assert st.rows == int((batch["active"][:, :T] != 0).sum())


# ------------------------------------------------------------------------------------------------ 5: the reference's values
def test_statistics_match_the_reference_per_minibatch_values():
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.train_stats import TrainStats
    fx = AlgoFixture(os.path.join(GOLDEN_DIR, "algo_d1_n8_e128.npz"))
    depth, n_def, T, episodes, mb, seed, emb = (int(v) for v in fx["meta"])
    cfg = default_config(env__num_defender=n_def, env__max_steps=T, algo__depth=depth, algo__embedding_dim=emb, algo__rnn_hidden_dim=emb,
                         algo__learner_device="cuda", algo__worker_device="cuda")
    m = MAPPO(cfg, episodes, mb, "Learner")
    for net, mod in (("actor", m.actor), ("critic", m.critic)):
        mod.load_state_dict({k[len("w." + net + "."):]: torch.from_numpy(fx[k]) for k in fx.files if k.startswith("w." + net + ".")})
    buf = {k[4:]: torch.from_numpy(fx[k]).cuda() for k in fx.files if k.startswith("buf.")}
    m.train(buf, int(fx["total_steps"]), return_numpy=False, stats=True)
    st = m.last_train_stats
    total = np.zeros(24)
    total[5], total[6] = -np.inf, np.inf
    n_mb = int(fx["n_mb"])
    for i in range(n_mb):
        idx = np.asarray(fx[f"mb{i}.index"]).reshape(-1)
        sel = lambda k: np.asarray(fx[k])[idx]                    # noqa: E731
        s, _ = np_sums(fx[f"mb{i}.logp"], sel("buf.a_logprob_n"), fx[f"mb{i}.ent"], fx[f"mb{i}.val"], sel("buf.v_n")[:, :T],
                       np.asarray(fx["v_target"])[idx], sel("buf.active"), np.float32(m.epsilon))
        for j in range(16):
            total[j] = max(total[j], s[j]) if j == 5 else (min(total[j], s[j]) if j == 6 else total[j] + s[j])
    total[16] = n_mb
    ref = TrainStats.from_sums(total, m.epsilon, None)
    n = st.rows
    assert n == ref.rows
    for k in KEYS[:12]:
        a, b = getattr(st, k), getattr(ref, k)
        tol = 2.0 / n if k.endswith("clip_frac") else 1e-5 * max(1.0, abs(b))      # a count may flip at a rounding tie
        assert abs(a - b) <= tol, (k, a, b)


# ------------------------------------------------------------------------------------------------ 6: two ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank_worker(rank, world, port, backend, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, rank=rank, world_size=world, **(dict(device_id=dev) if backend == "nccl" else {}))
    try:
        m, env = _mappo(16, 8, 1, 24, 8, seed=3 + rank)
        tb, _arena = _batch("store", m, env)
        m.train(tb, 1000, return_numpy=False, stats=True)
        st = m.last_train_stats
        own = st.sums.cpu().numpy().copy()
        st.allreduce_()
        out[rank] = (own, st.sums.cpu().numpy().copy(), {k: getattr(st, k) for k in KEYS})
    finally:
        dist.destroy_process_group()


def test_two_ranks_hold_identical_global_statistics():
    import torch.multiprocessing as mp
    backend = "nccl" if torch.cuda.device_count() >= 2 else "gloo"
    out = mp.Manager().dict()
    mp.spawn(_rank_worker, args=(2, _free_port(), backend, out), nprocs=2, join=True)
    (own0, g0, d0), (own1, g1, d1) = out[0], out[1]
    assert np.array_equal(g0, g1) and repr(d0) == repr(d1)
    for j in range(24):
        if j in (5, 18, 19):
            assert g0[j] == max(own0[j], own1[j]), j
        elif j == 6:
            assert g0[j] == min(own0[j], own1[j])
        else:
            assert g0[j] == own0[j] + own1[j], j
    assert not np.array_equal(own0, own1)


# ------------------------------------------------------------------------------------------------ 7: the driver
def _train_loop(*args):
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.join(ROOT, "tools", "train_loop.py"), "--envs", "64",
                                                                         "--steps", "30", "--maps", "4"] + list(args)
    out = subprocess.run(cmd, check=True, cwd=ROOT, timeout=900, capture_output=True, text=True).stdout
    lines = out.splitlines()
    col = lambda tag, key: {int(ln.split(key)[1].split()[0]): ln.split(key)[1] for ln in lines if ln.startswith(tag)}     # noqa: E731
    return col("iter", "exact "), col("stats", "hex "), col("kl_stop", "hex ")


@pytest.mark.parametrize("mode", [[], ["--segment", "20", "--auto-reset"]], ids=["plain", "auto_reset"])
def test_train_loop_stats_leave_the_exact_columns(mode):
    plain, no_stats, _ = _train_loop("--iters", "3", *mode)
    with_stats, stats, _ = _train_loop("--iters", "3", "--stats", *mode)
    assert plain == with_stats and not no_stats and sorted(stats) == [0, 1, 2]
    assert all(len(v.split()) == 3 + len(KEYS) + 1 for v in stats.values())     # + minibatches


def test_train_loop_target_kl_is_reproducible_and_resumable(tmp_path):
    args = ("--stats", "--epochs", "2", "--target-kl", "1e-12")
    a, sa, _ = _train_loop("--iters", "3", *args)
    b, sb, _ = _train_loop("--iters", "3", *args)
    assert a == b and sa == sb
    assert any(v.split()[2] == "2" for v in sa.values()), sa          # at least one update stopped at epoch 2
    _train_loop("--iters", "2", "--save-dir", str(tmp_path), *args)
    c, sc, _ = _train_loop("--iters", "3", "--resume", str(tmp_path), *args)
    assert c == {2: a[2]} and sc == {2: sa[2]}
    _, none, stops = _train_loop("--iters", "2", "--epochs", "2", "--target-kl", "1e-12")
    assert not none and stops and all(v.split()[1] == "2" for v in stops.values())
