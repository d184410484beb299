"""Bit-reproducible training and exact resume.

The message-layer weight gradients and the PPO loss sums are reduced through per-CTA partials in a fixed order
(marl_dhgn_message_bwd_det, marl_ppo_head_det), so every training step is a deterministic function of its inputs.  Checked here:
the two entry points against themselves and against the atomic ones, a whole epoch on a stored vs a replay-mode batch, two fresh
runs, and "stop, save, reload in another process, continue" against "never stopped" (one rank and two ranks).

Run as a script, this file is the resumed half of the resume test (see _resume_main)."""
import ctypes
import os
import socket
import subprocess
import sys

import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
E = 128
FULL_GRID_SAMPLES = 8 * 148 * 8           # >= 8 x the grouped backward's capped grid: every CTA of every launch has work


def _cfg(depth, n_def, T, **over):
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    return default_config(env__num_defender=n_def, env__max_steps=T, algo__depth=depth, algo__learner_device="cuda",
                          algo__worker_device="cuda", **over)


# ------------------------------------------------------------------------------------------------ 1: message backward
def _graph(S, N, O, all_ones, g):
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    dev = "cuda"
    Bo = 7
    p = torch.rand(S, N, 4, device=dev, generator=g) * 40
    e = torch.rand(S, 4, device=dev, generator=g) * 40
    oxy = torch.randint(0, 60, (Bo, O, 2), device=dev, generator=g).float()
    o_index = torch.randint(0, Bo, (S,), device=dev, generator=g, dtype=torch.int32)
    o_count = torch.randint(O // 2, O + 1, (Bo,), device=dev, generator=g, dtype=torch.int32)
    p_adj = ops.pack_bits(torch.rand(S, N, N, device=dev, generator=g) < 0.5)
    e_adj = (torch.rand(S, N, device=dev, generator=g) < 0.5).to(torch.uint8)
    o_adj = ops.pack_bits(torch.rand(S, N, O, device=dev, generator=g) < 0.3)
    return ops.GraphBatch(p, e, oxy, o_index, o_count, p_adj, e_adj, o_adj)


@pytest.mark.parametrize("all_ones", [False, True], ids=["actor_adjacency", "all_ones"])
@pytest.mark.parametrize("N,E_", [(8, 128), (20, 64), (64, 128)], ids=["grouped-N8-E128", "rows-N20-E64", "rows-N64-E128"])
def test_message_bwd_det_is_bit_reproducible(N, E_, all_ones):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    L = _lib.lib()
    g = torch.Generator(device="cuda").manual_seed(N * 1000 + E_)
    S, O = FULL_GRID_SAMPLES, 176
    graph = _graph(S, N, O, all_ones, g)
    ws = []                                                  # W0 [E,8], b0, W1 [E,4], b1, W2 [E,4], b2
    for k in (8, 4, 4):
        ws += [0.2 * torch.randn(E_, k, device="cuda", generator=g), 0.1 * torch.randn(E_, device="cuda", generator=g)]
    d_agg = torch.randn(S, N, 3, E_, device="cuda", generator=g)
    part = torch.empty(int(L.marl_dhgn_message_bwd_workspace_bytes(N, O, E_)), dtype=torch.uint8, device="cuda")

    def run(det):
        grads = [torch.zeros_like(w) for w in ws]
        args = (*graph._args(E_, all_ones), *[w.data_ptr() for w in ws], d_agg.data_ptr(), *[t.data_ptr() for t in grads])
        if det:
            part.fill_(0xFF)                                 # NaN garbage: every partial must be written
            rc = L.marl_dhgn_message_bwd_det(*args, part.data_ptr(), _lib.stream_ptr())
        else:
            rc = L.marl_dhgn_message_bwd(*args, _lib.stream_ptr())
        _lib.check(rc, "message bwd")
        torch.cuda.synchronize()
        return grads

    a, b, ref = run(True), run(True), run(False)
    for x, y, r in zip(a, b, ref):
        assert torch.isfinite(x).all()
        assert torch.equal(x, y)
        torch.testing.assert_close(x, r, rtol=1e-5, atol=1e-5 * float(r.abs().max()))


# ------------------------------------------------------------------------------------------------ 2: PPO head
def test_ppo_head_det_sums_are_bit_reproducible_and_exact():
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    L = _lib.lib()
    g = torch.Generator(device="cuda").manual_seed(11)
    R, A, eps, ent_coef = 60_000, 9, 0.2, 0.01
    f = lambda *s: torch.randn(*s, device="cuda", generator=g)       # noqa: E731
    feat_a, feat_c, Wa, ba, wc, bc = f(R, E), f(R, E), 0.1 * f(A, E), 0.1 * f(A), 0.1 * f(E), 0.1 * f(1)
    action = torch.randint(0, A, (R,), device="cuda", generator=g).float()
    old_logp = -2.2 + 0.3 * f(R)
    adv = f(R).abs() + 0.1                                   # one sign: the sum is well conditioned, so 1e-6 is meaningful
    v_old, v_target = f(R), f(R)
    active = (torch.rand(R, device="cuda", generator=g) < 0.9).float()
    part = torch.empty(int(L.marl_ppo_head_workspace_bytes(R)), dtype=torch.uint8, device="cuda")

    def run():
        logp, ent, val, dv = (torch.empty(R, device="cuda") for _ in range(4))
        dlog, sums = torch.empty(R, A, device="cuda"), torch.zeros(3, device="cuda")
        part.fill_(0xFF)
        _lib.check(L.marl_ppo_head_det(R, E, A, *[t.data_ptr() for t in (feat_a, feat_c, Wa, ba, wc, bc, action, old_logp, adv, v_old,
                                                                         v_target, active)],
                                       ctypes.c_float(eps), ctypes.c_float(ent_coef), *[t.data_ptr() for t in (logp, ent, val, dlog, dv, sums)],
                                       part.data_ptr(), _lib.stream_ptr()), "marl_ppo_head_det")
        torch.cuda.synchronize()
        return sums, logp, ent, val

    s1, logp, ent, val = run()
    s2 = run()[0]
    assert torch.equal(s1, s2)
    # the per-row terms in fp64 from the kernel's own per-row outputs
    d = lambda t: t.double()                                 # noqa: E731
    ratio = torch.exp(d(logp) - d(old_logp))
    a_term = -torch.minimum(ratio * d(adv), ratio.clamp(1 - eps, 1 + eps) * d(adv)) - ent_coef * d(ent)
    c1 = (torch.clamp(d(val) - d(v_old), -eps, eps) + d(v_old) - d(v_target)) ** 2
    c_term = torch.maximum(c1, (d(val) - d(v_target)) ** 2)
    ref = torch.stack([(a_term * d(active)).sum(), (c_term * d(active)).sum(), d(active).sum()])
    assert float(s1[2]) == float(ref[2])
    for j in range(2):
        assert abs(float(s1[j]) - float(ref[j])) <= 1e-6 * abs(float(ref[j])), (j, float(s1[j]), float(ref[j]))


# ------------------------------------------------------------------------------------------------ 3: store vs replay epoch
def _setup(B, N, D, T, mbs=None, M=4, seed=3):
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    cfg = _cfg(D, N, T)
    torch.manual_seed(seed)
    m = MAPPO(cfg, B, mbs or max(1, B // 4), "Learner")
    with torch.no_grad():                                    # biases are zero-initialised: make them matter
        for p in m.ac_parameters:
            if p.dim() == 1:
                p.add_(0.05 * torch.randn_like(p))
    env = BatchedPursuitEnv(cfg, B, num_maps=M)
    env.reset_device(seed=seed + 10, tape_len=32)
    return m, env, env.snapshot()


@pytest.mark.parametrize("in_flight", [1, 3])
@pytest.mark.parametrize("shuffle", [False, True], ids=["sequential", "shuffled"])
@pytest.mark.parametrize("D", [1, 3])
def test_epoch_on_replay_batch_equals_store_batch_bit_for_bit(D, shuffle, in_flight, monkeypatch):
    """The whole flat gradient (message layers included) and both losses of every minibatch are bit-identical, over two rounds with
    an update in between."""
    from distributed_multi_agent_reinforcement_learning_b200 import mappo_parallel
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import RolloutArena
    monkeypatch.setattr(mappo_parallel, "CONCURRENT_MINIBATCHES", in_flight)
    B, N, T = 48, 8, 24
    m, env, snap = _setup(B, N, D, T, mbs=16)
    tbs = []
    for mode in ("store", "replay"):
        env.restore(snap)
        arena = RolloutArena(env.params, B, T, env.device)
        tbs.append((m.rollout_batched(env, arena, T, seed=5, history=mode), arena))
    torch.cuda.synchronize()
    u = m.critic.Mean
    for rnd in range(2):
        traces, flats = [], []
        sn0 = (u.weight_u.clone(), u.weight_v.clone())
        for tb, _ in tbs:
            u.weight_u.copy_(sn0[0])                         # the spectral-norm power iteration advances on every forward
            u.weight_v.copy_(sn0[1])
            tr = {}
            m.train(tb, B * T * (rnd + 1), return_numpy=False, trace=tr, shuffle=shuffle, shuffle_seed=4)
            torch.cuda.synchronize()
            traces.append(tr)
            flats.append(m.ac_optimizer.flat_grad.clone())
        ts, tr_ = traces
        assert torch.equal(ts["mb_grads"], tr_["mb_grads"])
        assert torch.equal(flats[0], flats[1])
        for a, b in zip(ts["mb"], tr_["mb"]):
            assert a["actor_loss"] == b["actor_loss"] and a["critic_loss"] == b["critic_loss"]
        m.update(B * T * (rnd + 1))


# ------------------------------------------------------------------------------------------------ 4, 5: whole iterations
B_RUN, N_RUN, T_RUN, M_RUN, D_RUN = 32, 8, 30, 8, 1


def _build(history, seed=0, world=1):
    from distributed_multi_agent_reinforcement_learning_b200.evaluator import Evaluator
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena
    cfg = _cfg(D_RUN, N_RUN, T_RUN, algo__use_lr_decay=True)
    torch.manual_seed(seed)
    m = MAPPO(cfg, B_RUN, B_RUN // 4, "Learner")
    env = BatchedPursuitEnv(cfg, B_RUN, num_maps=M_RUN)
    arena = RolloutArena(env.params, B_RUN, T_RUN, env.device)
    ev = Evaluator(cfg, 4, m, seed=7)
    if world > 1:
        m.sync_weights(0)
    return dict(m=m, env=env, arena=arena, ev=ev, history=history)


def _iterate(run, its, rank=0, world=1):
    """tools/train_loop.py's iteration: device reset, rollout, one epoch, update (+ an evaluator row).  Returns the last iteration's
    losses and per-env episode rewards, and every iteration's losses."""
    m, env, arena = run["m"], run["env"], run["arena"]
    out = dict(losses=[])
    for it in its:
        env.reset_device(seed=1000 * rank + it)
        tb = m.rollout_batched(env, arena, T_RUN, seed=it * world + rank, history=run["history"])
        total = (it + 1) * world * B_RUN * T_RUN
        obj_c, obj_a, _, _ = m.train(tb, total, return_numpy=False)
        m.update(total)
        run["ev"].evaluate_and_save(total, 0.0, (obj_c, obj_a))
        torch.cuda.synchronize()
        out["losses"].append((obj_c, obj_a))
        out["ep_reward"] = arena.raw_reward[:T_RUN].sum(dim=(0, 2)).cpu()
    return out


def _final_state(run):
    m, env = run["m"], run["env"]
    opt = m.ac_optimizer
    return dict(flat_param=opt.flat_param.cpu(), exp_avg=opt.exp_avg.cpu(), exp_avg_sq=opt.exp_avg_sq.cpu(), step=opt.step_count,
                lr=opt.param_groups[0]["lr"], total_step=m.total_step, wf={k: getattr(env, k).cpu() for k in ("wf_n", "wf_mean", "wf_S", "wf_std")},
                sn=(m.critic.Mean.weight_u.cpu(), m.critic.Mean.weight_v.cpu()), recorder=list(run["ev"].recorder), max_r=run["ev"].max_r)


def _assert_same_state(a, b):
    for k in ("flat_param", "exp_avg", "exp_avg_sq"):
        assert torch.equal(a[k], b[k]), k
    assert a["step"] == b["step"] and a["lr"] == b["lr"] and a["total_step"] == b["total_step"]
    for k in a["wf"]:
        assert torch.equal(a["wf"][k], b["wf"][k]), k
    assert all(torch.equal(x, y) for x, y in zip(a["sn"], b["sn"]))
    assert a["recorder"] == b["recorder"] and a["max_r"] == b["max_r"]


def test_two_fresh_runs_are_bit_identical():
    results = []
    for _ in range(2):
        run = _build("store")
        out = _iterate(run, range(3))
        results.append((out, _final_state(run)))
    (o1, s1), (o2, s2) = results
    assert o1["losses"] == o2["losses"]
    assert torch.equal(o1["ep_reward"], o2["ep_reward"])
    _assert_same_state(s1, s2)


def _resume_main(path, history, out_path):
    """The resumed half: fresh objects in a new process, load, iterations 2 and 3."""
    from distributed_multi_agent_reinforcement_learning_b200.checkpoint import load_training_state
    run = _build(history, seed=123)                          # other initial weights: everything must come from the file
    extra = load_training_state(path, run["m"], run["env"], run["ev"])
    out = _iterate(run, range(int(extra["next_iter"]), 4))
    torch.save(dict(out=out, state=_final_state(run)), out_path)


@pytest.mark.parametrize("history", ["store", "replay"])
def test_resume_in_a_new_process_equals_uninterrupted_run(history, tmp_path):
    from distributed_multi_agent_reinforcement_learning_b200.checkpoint import save_training_state
    run_a = _build(history)
    out_a = _iterate(run_a, range(4))
    state_a = _final_state(run_a)
    del run_a

    run_b = _build(history)
    _iterate(run_b, range(2))
    path = str(tmp_path / "state.pt")
    save_training_state(path, run_b["m"], run_b["env"], run_b["ev"], extra=dict(next_iter=2))
    del run_b
    out_path = str(tmp_path / "resumed.pt")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), path, history, out_path]
    subprocess.run(cmd, check=True, cwd=ROOT, timeout=900)
    res = torch.load(out_path, weights_only=False)
    assert res["out"]["losses"][-1] == out_a["losses"][-1]
    assert torch.equal(res["out"]["ep_reward"], out_a["ep_reward"])
    _assert_same_state(res["state"], state_a)


# ------------------------------------------------------------------------------------------------ 6: rejected loads
def test_mismatched_loads_are_rejected_and_change_nothing(tmp_path):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.checkpoint import load_training_state, save_training_state
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv
    src = _build("store")
    _iterate(src, range(1))
    path = str(tmp_path / "state.pt")
    save_training_state(path, src["m"], src["env"])

    def target(N=N_RUN, D=D_RUN, B=B_RUN):
        cfg = _cfg(D, N, T_RUN)
        torch.manual_seed(5)
        return MAPPO(cfg, B, B // 4, "Learner"), BatchedPursuitEnv(cfg, B, num_maps=M_RUN)

    for kw, what in ((dict(N=4), "N"), (dict(D=3), "depth"), (dict(B=16), "B")):
        m, env = target(**kw)
        env.wf_mean.fill_(0.5)
        before = (m.ac_optimizer.flat_param.clone(), m.ac_optimizer.exp_avg.clone(), env.wf_mean.clone(), env.grid_bits.clone())
        with pytest.raises(_lib.MarlError, match=what):
            load_training_state(path, m, env)
        after = (m.ac_optimizer.flat_param, m.ac_optimizer.exp_avg, env.wf_mean, env.grid_bits)
        assert all(torch.equal(x, y) for x, y in zip(before, after)), what
        assert m.ac_optimizer.step_count == 0
    m, env = target()
    load_training_state(path, m, env)
    opt = m.ac_optimizer
    assert torch.equal(opt.flat_param, src["m"].ac_optimizer.flat_param)
    base, end = opt.flat_param.data_ptr(), opt.flat_param.data_ptr() + 4 * opt.flat_param.numel()
    for p, (off, k) in zip(m.ac_parameters, opt._views):
        assert p.data_ptr() == base + 4 * off and p.data_ptr() < end


# ------------------------------------------------------------------------------------------------ 7: two ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank_worker(rank, world, port, folder, out):
    import torch.distributed as dist
    from distributed_multi_agent_reinforcement_learning_b200.checkpoint import load_training_state, save_training_state
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        straight = _build("store", world=world)
        _iterate(straight, range(4), rank, world)
        ref = _final_state(straight)
        del straight
        first = _build("store", world=world)
        _iterate(first, range(2), rank, world)
        path = os.path.join(folder, f"rank{rank}.pt")
        save_training_state(path, first["m"], first["env"], first["ev"], extra=dict(next_iter=2))
        del first
        resumed = _build("store", seed=99, world=world)
        extra = load_training_state(path, resumed["m"], resumed["env"], resumed["ev"])
        _iterate(resumed, range(extra["next_iter"], 4), rank, world)
        try:
            _assert_same_state(_final_state(resumed), ref)
            out[rank] = "ok"
        except AssertionError as e:                          # noqa: PERF203
            out[rank] = f"differs: {e}"
    finally:
        dist.destroy_process_group()


def test_two_rank_resume_equals_straight_run(tmp_path):
    import torch.multiprocessing as mp
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    from distributed_multi_agent_reinforcement_learning_b200.checkpoint import load_training_state
    out = mp.Manager().dict()
    mp.spawn(_rank_worker, args=(2, _free_port(), str(tmp_path), out), nprocs=2, join=True)
    assert dict(out) == {0: "ok", 1: "ok"}
    run = _build("store")
    with pytest.raises(_lib.MarlError, match="world_size"):
        load_training_state(str(tmp_path / "rank0.pt"), run["m"], run["env"], run["ev"])


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    _resume_main(*sys.argv[1:4])
