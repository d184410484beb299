"""Teams of 17 to 128 pursuers: the DHGN network kernels against a float64 evaluation of oracle/policy_ref.py.

Paths that only large teams reach: adjacency rows of 2 to 4 words (NW = ceil(N/32)), tiles that hold a non-dividing number of envs
(33 -> 99 rows, 48 -> 96) or one env with 128 - N padded MMA rows (65 <= N <= 128), and the message backward's rows path (N > 16)
with its long per-warp fp32 chains.  Inputs are synthetic, so placement rules do not limit N, and they include the adjacency edges:
rows with no neighbour, full rows, rows whose only neighbours sit in words >= 1 (and >= 3), obstacle bits in the last word, maps
with o_count < O and o_count == O.

Tolerances (north_star, as in test_gpu_policy.py): 1e-5 relative + 2e-5 absolute for forward activations, values and log-probs;
1e-4 of the tensor's max for losses and gradients.  Every case prints its measured error; the negative controls show that each
comparison fails when the kernels see only the first adjacency word, or the reference a history shifted by one step."""
from types import SimpleNamespace

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEV = "cuda"
E = 128
O_CELLS = 110                   # configs[4]'s boundary slots: 4 obstacle words, the last one partial
FWD = dict(rtol=1e-5, atol=2e-5)


@pytest.fixture
def log(capsys):
    """Prints past pytest's capture, so the measured errors appear in the log of a passing run."""
    def emit(line):
        with capsys.disabled():
            print(line)
    return emit


def _fwd_err(log, name, got, ref, rtol=FWD["rtol"], atol=FWD["atol"]):
    """Worst |got - ref| / (atol + rtol |ref|): <= 1 is within the forward tolerance."""
    got, ref = got.detach().double(), ref.detach().double()
    d = (got - ref).abs()
    ratio = float((d / (atol + rtol * ref.abs())).max())
    ratio = float("inf") if ratio != ratio else ratio                    # a NaN output fails
    log(f"  {name:<28s} max abs err {float(d.max()):.3e}   err/tol {ratio:.3f}")
    return ratio


def _grad_err(log, name, got, ref):
    """max |got - ref| / (1e-4 max |ref|): <= 1 is within the loss / gradient tolerance."""
    got, ref = got.detach().double(), ref.detach().double()
    d = float((got - ref).abs().max())
    scale = float(ref.abs().max())
    ratio = d / (1e-4 * scale) if scale > 0 else (0.0 if d == 0 else float("inf"))
    ratio = float("inf") if ratio != ratio else ratio
    log(f"  {name:<28s} max abs err {d:.3e}   of max {scale:.3e}   err/tol {ratio:.3f}")
    return ratio


def _cfg(N, T=4, D=1):
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    return default_config(env__num_defender=N, env__max_steps=T, algo__depth=D, algo__learner_device=DEV,
                          algo__worker_device=DEV)


def _model(N, D, seed=5, T=4, **kw):
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    torch.manual_seed(seed)
    m = MAPPO(_cfg(N, T, D), kw.pop("batch", None), kw.pop("mini_batch", None), "Learner", **kw)
    with torch.no_grad():                                    # biases are zero-initialised: make them matter
        for p in m.ac_parameters:
            if p.dim() == 1:
                p.add_(0.05 * torch.randn_like(p))
    return m


def _weights64(m):
    """policy_ref's weight dict in float64, keyed "actor." / "critic." + the module names.  The encoder is one module under both
    networks: its parameters map to one leaf, so float64 autograd sums both networks' gradients into it as the model does."""
    leaves, w = {}, {}
    for net, mod in (("actor", m.actor), ("critic", m.critic)):
        for name, p in mod.named_parameters():
            if id(p) not in leaves:
                leaves[id(p)] = p.detach().double().requires_grad_(True)
            w[f"{net}.{name}"] = leaves[id(p)]
        for name, b in mod.named_buffers():
            w[f"{net}.{name}"] = b.detach().double()
    return w, [leaves[id(p)] for p in m.ac_parameters]


def _team(S, N, O=O_CELLS, M=3, seed=0, map_id=None):
    """Synthetic observations of S samples of N pursuers on M maps of O boundary slots.  Map 0 fills all O slots (o_count == O),
    the others fewer; sample 0 (on map 0) carries the adjacency edge rows."""
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    dev = DEV
    g = torch.Generator(device=dev).manual_seed(seed)
    rnd = lambda *s: torch.rand(*s, device=dev, generator=g)             # noqa: E731
    scale = torch.tensor([60.0, 55.0, 4.0, 4.0], device=dev)
    shift = torch.tensor([0.0, 0.0, 2.0, 2.0], device=dev)
    p = (rnd(S, N, 4) * scale - shift).contiguous()
    e = (rnd(S, 4) * scale - shift).contiguous()
    oxy = torch.randint(0, 55, (M, O, 2), device=dev, generator=g, dtype=torch.int32)
    o_count = torch.tensor([O, O - 17, 23, O - 1][:M] + [O // 2] * max(0, M - 4), dtype=torch.int32, device=dev)
    map_id = (torch.arange(S, device=dev) % M).to(torch.int32) if map_id is None else map_id.to(torch.int32).contiguous()
    real = torch.arange(O, device=dev)[None, :] < o_count[map_id.long()][:, None]          # [S, O]
    p_adj = (rnd(S, N, N) < 0.5).float()
    e_adj = (rnd(S, N) < 0.5).float()
    o_adj = ((rnd(S, N, O) < 0.15) & real[:, None, :]).float()
    assert int(map_id[0]) == 0 and int(o_count[0]) == O
    p_adj[0, 0], o_adj[0, 0] = 0, 0                                       # no neighbour, no obstacle
    p_adj[0, 1 % N], o_adj[0, 1 % N] = 1, 1                               # every pursuer, every slot
    if N > 32:                                                            # neighbours only in words >= 1
        p_adj[0, 2, :32] = 0
        p_adj[0, 2, 32 + (N - 32) // 2] = 1
    if N >= 97:                                                           # ... only in word 3
        p_adj[0, 3, :96] = 0
        p_adj[0, 3, 96:] = 1
    last = 32 * ((O - 1) // 32)
    o_adj[0, 2 % N] = 0                                                   # obstacle bits only in the last word
    o_adj[0, 2 % N, last:] = 1
    return SimpleNamespace(S=S, N=N, O=O, M=M, p=p, e=e, oxy=oxy, o_count=o_count, map_id=map_id, p_adj=p_adj, e_adj=e_adj,
                           o_adj=o_adj, p_adj_bits=ops.pack_bits(p_adj), e_adj_u8=(e_adj != 0).to(torch.uint8).contiguous(),
                           o_adj_bits=ops.pack_bits(o_adj))


def _first_word_only(bits):
    """The adjacency words a kernel would read if it never looked past word 0."""
    out = bits.clone()
    out[..., 1:] = 0
    return out


def _graph(team, p_adj_bits=None):
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    return ops.GraphBatch(team.p, team.e, team.oxy.float().contiguous(), team.map_id, team.o_count,
                          team.p_adj_bits if p_adj_bits is None else p_adj_bits, team.e_adj_u8, team.o_adj_bits)


def _ref_message_agg(team, all_ones, w, lo=0, hi=None):
    """float64 policy_ref message (DHGN.message) + L1-normalised mean aggregation of samples [lo, hi): [S, N, 3, E]."""
    import torch.nn.functional as F
    from oracle import policy_ref
    hi = team.S if hi is None else hi
    p, e = team.p[lo:hi].double(), team.e[lo:hi].double().unsqueeze(1)
    mid = team.map_id[lo:hi].long()
    o4 = torch.cat([team.oxy.double(), torch.zeros_like(team.oxy, dtype=torch.float64)], -1)[mid]
    S, N, O = p.shape[0], team.N, team.O
    if all_ones:
        real = (torch.arange(O, device=DEV)[None, :] < team.o_count[mid][:, None]).double()
        p_adj, e_adj = torch.ones(S, N, N, dtype=torch.float64, device=DEV), torch.ones(S, N, 1, dtype=torch.float64, device=DEV)
        o_adj = real[:, None, :].expand(S, N, O)
    else:
        p_adj, e_adj, o_adj = team.p_adj[lo:hi].double(), team.e_adj[lo:hi].double().unsqueeze(-1), team.o_adj[lo:hi].double()
    rel_pp = p.unsqueeze(-2) - p.unsqueeze(-3)
    rel_pe = p.unsqueeze(-2) - e.unsqueeze(-3)
    rel_po = p.unsqueeze(-2) - o4.unsqueeze(-3)
    a0 = torch.cat([rel_pp, rel_pe.expand(*rel_pp.shape[:-1], 4)], -1)
    outs = []
    for r, (attr, adj) in enumerate(((a0, p_adj), (rel_pe, e_adj), (rel_po, o_adj))):
        msg = torch.relu(policy_ref._lin(w, f"MSG_layers.{r}", attr))
        outs.append(torch.matmul(F.normalize(adj.unsqueeze(-2), p=1, dim=-1), msg).squeeze(-2))
    return torch.stack(outs, dim=2)


def _msg_weights(Ew, seed=1):
    g = torch.Generator(device=DEV).manual_seed(seed)
    W = []
    for r, k in enumerate((8, 4, 4)):
        W += [torch.randn(Ew, k, device=DEV, generator=g) * 0.3, torch.randn(Ew, device=DEV, generator=g) * 0.1]
    return W


def _msg_case(log, team, all_ones, Ew, p_adj_bits=None):
    """Kernel forward / backward of message_agg against float64 autograd; returns (forward err/tol, worst gradient err/tol)."""
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    W = _msg_weights(Ew)
    leaves = [t.clone().requires_grad_(True) for t in W]
    out = ops.message_agg(_graph(team, p_adj_bits), all_ones, *leaves)
    ref_leaves = [t.double().requires_grad_(True) for t in W]
    names = ("MSG_layers.0.weight", "MSG_layers.0.bias", "MSG_layers.1.weight", "MSG_layers.1.bias", "MSG_layers.2.weight",
             "MSG_layers.2.bias")
    ref = _ref_message_agg(team, all_ones, dict(zip(names, ref_leaves)))
    fwd = _fwd_err(log, "message_agg forward", out, ref)
    dout = torch.randn(out.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2))
    out.backward(dout)
    ref.backward(dout.double())
    bwd = max(_grad_err(log, f"d {n}", a.grad, b.grad) for n, a, b in zip(names, leaves, ref_leaves))
    return fwd, bwd


# ------------------------------------------------------------------------------------------------------------ 1. message layer
@pytest.mark.parametrize("N,S,Ew", [(17, 9, 32), (31, 7, 64), (32, 7, 128), (33, 5, 128), (48, 5, 32), (63, 4, 128), (64, 4, 64),
                                    (65, 3, 128), (100, 3, 128), (127, 3, 32), (128, 3, 128)])
@pytest.mark.parametrize("all_ones", [False, True], ids=["actor_adjacency", "all_ones"])
def test_message_agg_large_teams_vs_fp64(log, N, S, Ew, all_ones):
    """marl_dhgn_message_fwd / marl_dhgn_message_bwd_det (N > 16: the rows path) against float64 autograd of the policy_ref message
    and mean aggregation, on 2- to 4-word adjacency rows."""
    team = _team(S, N, seed=N)
    log(f"\n[message_agg] N={N} S={S} E={Ew} {'all_ones' if all_ones else 'actor'}")
    fwd, bwd = _msg_case(log, team, all_ones, Ew)
    assert fwd <= 1.0 and bwd <= 1.0, (fwd, bwd)


def test_message_agg_first_word_only_fails_at_64(log):
    """Negative control: a kernel that saw only adjacency word 0 would fail the comparison above at N = 64."""
    team = _team(4, 64, seed=64)
    log("\n[message_agg control] N=64, kernel given word 0 only")
    fwd, _ = _msg_case(log, team, False, E, p_adj_bits=_first_word_only(team.p_adj_bits))
    assert fwd > 1.0, fwd


# ------------------------------------------------------------------------------------------------------------ 2. FCRA aggregation
@pytest.mark.parametrize("N", [33, 64, 65, 100, 128])
def test_fcra_agg_multiword_strided_history_vs_fp64(log, N):
    """marl_fcra_agg over the [T+D, B, N, E] history arena addressed in place (sample stride N*E, agent stride E), 2 to 4 adjacency
    words, against L1norm(adj) @ hist in float64; all_ones is the critic's mean over the team."""
    import torch.nn.functional as F
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    T, B, D = 3, 2, 3
    team = _team(T * B, N, seed=100 + N)
    g = torch.Generator(device=DEV).manual_seed(3)
    arena = torch.randn(T + D, B, N, E, device=DEV, generator=g)
    adj = team.p_adj.double()
    log(f"\n[fcra_agg] N={N} words={(N + 31) // 32}")
    worst = 0.0
    for k in range(D):
        hist = arena[D - 1 - k: D - 1 - k + T].reshape(T * B, N, E).double()
        got = ops.fcra_agg(arena[D - 1 - k:], team.p_adj_bits, False, T * B, N, E, N * E, E)
        worst = max(worst, _fwd_err(log, f"k={k} adjacency", got, torch.matmul(F.normalize(adj, p=1, dim=-1), hist)))
        got1 = ops.fcra_agg(arena[D - 1 - k:], team.p_adj_bits, True, T * B, N, E, N * E, E)
        worst = max(worst, _fwd_err(log, f"k={k} all_ones", got1, hist.mean(1, keepdim=True).expand(-1, N, -1)))
    assert worst <= 1.0, worst


# ------------------------------------------------------------------------------------------------------------ 3. fused rollout step
def _step_inputs(team, D, seed=4):
    g = torch.Generator(device=DEV).manual_seed(seed)
    B, N = team.S, team.N
    hist = [0.3 * torch.randn(B, N, E, device=DEV, generator=g) for _ in range(D + 1)]   # one extra, older slab (control)
    ha = 0.1 * torch.randn(2, B * N, E, device=DEV, generator=g)
    hc = 0.1 * torch.randn(2, B * N, E, device=DEV, generator=g)
    action = torch.randint(0, 9, (B, N), device=DEV, generator=g, dtype=torch.int32)
    return hist, ha, hc, action


def _engine(team, p_adj_bits=None, f32=False, lo=0, hi=None):
    """What FusedRolloutStep.step reads from an engine, for envs [lo, hi)."""
    sl = slice(lo, team.S if hi is None else hi)
    p, e = (team.p, team.e) if f32 else (team.p.double(), team.e.double())
    bits = team.p_adj_bits if p_adj_bits is None else p_adj_bits
    return SimpleNamespace(B=sl.stop - sl.start, N=team.N, O=team.O, p_state=p[sl].contiguous(), e_state=e[sl].contiguous(),
                           map_id=team.map_id[sl].contiguous(), p_adj_bits=bits[sl].contiguous(), e_adj=team.e_adj_u8[sl].contiguous(),
                           o_adj_bits=team.o_adj_bits[sl].contiguous())


def _ref_step(m, team, hist, ha, hc, D):
    """float64 policy_ref.rollout_step (one aliased history list for both networks, the critic over the map's real cells):
    emb_a, emb_c, ha, hc, value and the actor's logits (its head applied to the last GRU layer's new state)."""
    import torch.nn.functional as F
    from oracle import policy_ref
    w, _ = _weights64(m)
    w = {k: v.detach() for k, v in w.items()}
    mid = team.map_id.long()
    B, N, O = team.S, team.N, team.O
    obs = dict(p=team.p.double(), e=team.e.double().unsqueeze(1),
               o=torch.cat([team.oxy.double(), torch.zeros_like(team.oxy, dtype=torch.float64)], -1)[mid],
               p_adj=team.p_adj.double(), e_adj=team.e_adj.double().unsqueeze(-1), o_adj=team.o_adj.double(),
               o_real=(torch.arange(O, device=DEV)[None, :] < team.o_count[mid][:, None]).double())
    with torch.no_grad():
        _, _, val, emb_a, emb_c, ha2, hc2 = policy_ref.rollout_step(
            w, obs, [h.double() for h in hist[:D]], ha.double(), hc.double(), D,
            generator=torch.Generator(device=DEV).manual_seed(0))
        logits = F.linear(ha2[-1], w["actor.Mean.weight"], w["actor.Mean.bias"]).view(B, N, -1)
    return dict(emb_a=emb_a, emb_c=emb_c, ha=ha2, hc=hc2, value=val, logits=logits)


def _fused(m):
    from distributed_multi_agent_reinforcement_learning_b200.fused_policy import FusedRolloutStep
    w_eff, _ = m.critic.head_weight()
    return FusedRolloutStep(m, w_eff)


def _launch(fused, eng, team, hist, ha, hc, action=None, force=True, deterministic=False, seed=77, t=5, nets=("actor", "critic"),
            **kw):
    """One fused step with fresh outputs; hidden states are copied (the kernel updates them in place)."""
    B, N = eng.B, eng.N
    out = dict(emb_a=torch.full((B, N, E), float("nan"), device=DEV), emb_c=torch.full((B, N, E), float("nan"), device=DEV),
               ha=ha.clone(), hc=hc.clone(), logp=torch.full((B, N), float("nan"), device=DEV),
               value=torch.full((B, N), float("nan"), device=DEV),
               action=action.clone() if action is not None else torch.full((B, N), -1, dtype=torch.int32, device=DEV))
    actor = "actor" in nets
    fused.step(eng, team.oxy, team.o_count, t, seed, deterministic, hist, hist, out["emb_a"], out["emb_c"],
               out["ha"] if actor else None, out["hc"], out["action"] if actor else None, out["logp"] if actor else None,
               out["value"], nets=nets, force_action=force, **kw)
    torch.cuda.synchronize()
    return out


def _compare_step(log, label, out, ref, action, keys=("emb_a", "emb_c", "ha", "hc", "value", "logp")):
    B, N = action.shape
    logp_ref = torch.log_softmax(ref["logits"], -1).gather(-1, action.long().unsqueeze(-1)).squeeze(-1)
    full = dict(ref, logp=logp_ref, value=ref["value"].view(B, N))
    log(f"  -- {label}")
    return max(_fw(log, k, out[k], full[k]) for k in keys)


def _fw(log, k, got, ref):
    return _fwd_err(log, k, got.reshape(ref.shape), ref)


def _full_tile(N):
    return (128 // N) * N         # what the env-group pipelines request (MappoParallel rollout), whole envs of one MMA tile


STEP_CASES = [(17, 15, 1, 3), (31, 9, 2, 1), (32, 5, 3, 3), (33, 4, 1, 1), (33, 7, 3, 3), (48, 3, 2, 3), (63, 3, 1, 1), (64, 3, 1, 3),
              (64, 5, 3, 1), (65, 2, 2, 3), (100, 3, 3, 1), (100, 2, 1, 3), (127, 2, 2, 3), (128, 3, 3, 3), (128, 2, 1, 1)]


@pytest.mark.parametrize("N,B,D,variant", STEP_CASES)
def test_fused_step_large_teams_vs_fp64(log, N, B, D, variant):
    """marl_policy_rollout_step against float64 policy_ref.rollout_step at the same inputs: the teacher-forced step (both
    embeddings, both hidden states, value, log-prob), the critic-only launch, MARL_POLICY_STATE_F32, MARL_POLICY_EMBED_ONLY and the
    arg-max launch.  B is chosen so that the last tile is partial (N <= 64) or one env fills a tile (N >= 65)."""
    from distributed_multi_agent_reinforcement_learning_b200.fused_policy import STATE_F32, EMBED_ONLY
    tile = _full_tile(N)
    assert (B * N) % tile != 0 or tile == N
    m = _model(N, D)
    fused = _fused(m)
    team = _team(B, N, seed=7 * N + D)
    hist, ha, hc, action = _step_inputs(team, D)
    ref = _ref_step(m, team, hist, ha, hc, D)
    log(f"\n[fused step] N={N} B={B} D={D} variant={variant} words={(N + 31) // 32} tile={tile}")
    kw = dict(variant=variant, tile_rows=tile)
    worst = _compare_step(log, "teacher-forced", _launch(fused, _engine(team), team, hist[:D], ha, hc, action, **kw), ref, action)
    crit = _launch(fused, _engine(team), team, hist[:D], ha, hc, nets=("critic",), variant=1, tile_rows=tile)
    worst = max(worst, _compare_step(log, "critic only", crit, ref, action, keys=("emb_c", "hc", "value")))
    f32 = _launch(fused, _engine(team, f32=True), team, hist[:D], ha, hc, action, flags=STATE_F32, **kw)
    worst = max(worst, _compare_step(log, "STATE_F32", f32, ref, action))
    emb = _launch(fused, _engine(team), team, hist[:D], ha, hc, action, flags=EMBED_ONLY, **kw)
    worst = max(worst, _compare_step(log, "EMBED_ONLY", emb, ref, action, keys=("emb_a", "emb_c")))
    assert torch.isnan(emb["value"]).all() and torch.equal(emb["ha"], ha)          # nothing past the embeddings is written
    # arg-max launch: the kernel's action is the reference's arg-max wherever the top-two logits are apart by more than the
    # logits' tolerance
    am = _launch(fused, _engine(team), team, hist[:D], ha, hc, force=False, deterministic=True, **kw)
    top2 = ref["logits"].topk(2, dim=-1).values
    clear = (top2[..., 0] - top2[..., 1]) > 1e-4
    assert float(clear.float().mean()) > 0.9
    assert torch.equal(am["action"].long()[clear], ref["logits"].argmax(-1)[clear])
    worst = max(worst, _compare_step(log, "arg-max", am, ref, am["action"], keys=("logp",)))
    assert worst <= 1.0, worst


@pytest.mark.parametrize("N,B", [(33, 7), (48, 5), (17, 13)])
def test_fused_step_every_tile_size_vs_fp64(log, N, B):
    """Every legal tile_rows (whole envs, at most 128 rows) gives the reference's outputs, partial last tiles included."""
    m = _model(N, 2)
    fused = _fused(m)
    team = _team(B, N, seed=N + 1)
    hist, ha, hc, action = _step_inputs(team, 2)
    ref = _ref_step(m, team, hist, ha, hc, 2)
    log(f"\n[fused step tiles] N={N} B={B}")
    worst = 0.0
    for rows in range(N, 129, N):
        for variant in (1, 3):
            out = _launch(fused, _engine(team), team, hist[:2], ha, hc, action, variant=variant, tile_rows=rows)
            worst = max(worst, _compare_step(log, f"tile_rows={rows} variant={variant}", out, ref, action))
    assert worst <= 1.0, worst


@pytest.mark.parametrize("N,B,lo", [(33, 7, 1), (64, 5, 2), (100, 3, 1), (128, 3, 1)])
def test_fused_step_sub_batch_row_offset_bit_identical(N, B, lo):
    """A launch over envs [lo, B) with row_offset = lo*N (an env-group pipeline's launch) equals the whole-batch launch bit for bit,
    sampled actions included: the sampling key follows the global row."""
    m = _model(N, 3)
    fused = _fused(m)
    team = _team(B, N, seed=N + 2)
    hist, ha, hc, _ = _step_inputs(team, 3)
    for variant in (1, 3):
        kw = dict(force=False, deterministic=False, variant=variant, tile_rows=_full_tile(N))
        whole = _launch(fused, _engine(team), team, hist[:3], ha, hc, **kw)
        rows = slice(lo * N, B * N)
        sub = _launch(fused, _engine(team, lo=lo), team, [h[lo:].contiguous() for h in hist[:3]], ha[:, rows].contiguous(),
                      hc[:, rows].contiguous(), row_offset=lo * N, **kw)
        for k in ("emb_a", "emb_c", "logp", "value", "action"):
            assert torch.equal(sub[k], whole[k][lo:]), (variant, k)
        for k in ("ha", "hc"):
            assert torch.equal(sub[k], whole[k][:, rows]), (variant, k)
        assert len(torch.unique(whole["action"])) > 1


def test_fused_step_controls_fail(log):
    """Negative controls: the fused-step comparison fails at N = 64 when the kernel sees adjacency word 0 only, and at D = 3 when
    the reference is given the history one step older."""
    N, B, D = 64, 3, 3
    m = _model(N, D)
    fused = _fused(m)
    team = _team(B, N, seed=9)
    hist, ha, hc, action = _step_inputs(team, D)
    ref = _ref_step(m, team, hist, ha, hc, D)
    log("\n[fused step controls] N=64 D=3")
    cut = _launch(fused, _engine(team, p_adj_bits=_first_word_only(team.p_adj_bits)), team, hist[:D], ha, hc, action, variant=3)
    assert _compare_step(log, "kernel given word 0 only", cut, ref, action, keys=("emb_a",)) > 1.0
    good = _launch(fused, _engine(team), team, hist[:D], ha, hc, action, variant=3)
    shifted = _ref_step(m, team, hist[1:], ha, hc, D)
    assert _compare_step(log, "reference history shifted", good, shifted, action, keys=("emb_a",)) > 1.0
    assert _compare_step(log, "unshifted", good, ref, action, keys=("emb_a",)) <= 1.0


# ------------------------------------------------------------------------------------------------------------ 4. training
class _KinkFree:
    """`torch` as policy_ref sees it, whose ReLUs after the GEMM layers (AGG, FCRA) move the layer's bias by 1e-3 in every channel
    with a float64 pre-activation within fp32 rounding of 0 (REL times the largest magnitude in its row).  There the fp32 kernels
    may legitimately take the other branch, and one flipped row moves a gradient by ~1/rows of its size, far beyond 1e-4 of its
    max at test sizes.  The message ReLUs need no such care: the training tests feed dyadic states and message weights, for which
    the kernel's fp32 message pre-activations are exact."""
    REL = 2e-6

    def __init__(self, w):
        self.w, self.moved = w, 0

    def __getattr__(self, name):
        return getattr(torch, name)

    def relu(self, x):
        import sys
        f = sys._getframe(1)
        if f.f_code.co_name == "_mean_op":                               # AGG layers
            key = f.f_locals["name"] + ".bias"
        elif f.f_code.co_name == "dhgn_fcra":
            key = f"{f.f_locals['pre']}FCRA_layers.{f.f_locals['k']}.bias"
        else:                                                            # DHGN.message (dhgn_encoder)
            return torch.relu(x)
        xd = x.detach()
        near = (xd.abs() <= self.REL * xd.abs().amax(-1, keepdim=True)).flatten(0, -2).any(0)
        if near.any():
            self.moved += int(near.sum())
            with torch.no_grad():
                self.w[key][near] += 1e-3
        return torch.relu(x)


def _clear_relu_kinks(m, minibatches, D):
    """Moves the model's AGG / FCRA biases until no float64 pre-activation of any minibatch sits at a ReLU kink (_KinkFree)."""
    from oracle import policy_ref
    for _ in range(6):
        w, leaves = _weights64(m)
        kf = _KinkFree(w)
        saved = policy_ref.torch
        policy_ref.torch = kf
        try:
            with torch.no_grad():
                for mb in minibatches:
                    policy_ref.train_forward(w, mb, D)
        finally:
            policy_ref.torch = saved
        if kf.moved == 0:
            return
        with torch.no_grad():
            for p, leaf in zip(m.ac_parameters, leaves):
                p.copy_(leaf)
    raise AssertionError("ReLU kinks did not clear")


class _Big:
    def __init__(self, d):
        self.buffer = d

    def get_training_data(self, device):
        return {k: v.to(device) for k, v in self.buffer.items()}


def _train_buffer(B, T, N, D, seed):
    """A reference-layout buffer ([B, T, ...]) of synthetic observations; o_state holds each env's map in every step."""
    dev = DEV
    team = _team(B * T, N, M=B, seed=seed, map_id=torch.arange(B, device=dev).repeat_interleave(T))
    team.p, team.e = (team.p * 16).round() / 16, (team.e * 16).round() / 16      # dyadic states (see _KinkFree)
    g = torch.Generator(device=dev).manual_seed(seed + 1)
    rn = lambda *s: torch.randn(*s, device=dev, generator=g)             # noqa: E731
    o4 = torch.cat([team.oxy.float(), torch.zeros(B, team.O, 2, device=dev)], -1)
    buf = dict(p_state=team.p.view(B, T, N, 4), e_state=team.e.view(B, T, 1, 4),
               o_state=o4.unsqueeze(1).expand(B, T, team.O, 4).contiguous(), p_adj=team.p_adj.view(B, T, N, N),
               e_adj=team.e_adj.view(B, T, N, 1), o_adj=team.o_adj.view(B, T, N, team.O),
               actor_historical_embedding=0.3 * rn(B, T + D, N, E), critic_historical_embedding=0.3 * rn(B, T + D, N, E),
               v_n=0.2 * rn(B, T + 1, N), a_n=torch.randint(0, 9, (B, T, N), device=dev, generator=g).float(),
               a_logprob_n=float(np.log(1.0 / 9)) + 0.05 * rn(B, T, N), r=rn(B, T, N),
               active=(torch.rand(B, T, N, device=dev, generator=g) < 0.9).float())
    return {k: v.contiguous() for k, v in buf.items()}


def _train_case(log, monkeypatch, N, D, kernel_p_adj=None):
    """MAPPO.train on a shuffled synthetic batch; each minibatch's log-probs, entropies, values, losses and gradients against
    float64 autograd of policy_ref.train_forward + ppo_losses on the same minibatch (the traced advantages, value targets and
    permutation; the stored history embeddings the batch trains on).  Returns (forward err/tol, loss and gradient err/tol)."""
    from distributed_multi_agent_reinforcement_learning_b200 import mappo_parallel as mp, policy_ops as ops
    from oracle import policy_ref
    monkeypatch.setattr(ops, "ROWGEMM_MIN_ROWS", 1)          # performance thresholds only: run the production kernels
    monkeypatch.setattr(ops, "WGRAD_MIN_ROWS", 1)
    monkeypatch.setattr(mp, "CONCURRENT_MINIBATCHES", 2)
    B, T, mbs = 4, 3, 2
    m = _model(N, D, T=T, batch=B, mini_batch=mbs)
    with torch.no_grad():                                    # dyadic message weights: exact fp32 message pre-activations
        for p in m.actor.shared_net.MSG_layers.parameters():
            p.copy_((p * 256).round() / 256)
    buf = _train_buffer(B, T, N, D, seed=N + D)
    feed = dict(buf) if kernel_p_adj is None else dict(buf, p_adj=kernel_p_adj(buf["p_adj"]))
    perm = [2, 0, 3, 1]
    index = [torch.tensor(perm[lo:lo + mbs], device=DEV) for lo in range(0, B, mbs)]
    _clear_relu_kinks(m, [{k: v[idx].double() for k, v in buf.items()} for idx in index], D)
    w, leaves = _weights64(m)
    trace = {}
    m.train(_Big(feed), B * T * N, return_numpy=False, trace=trace, permutation=perm)
    torch.cuda.synchronize()
    names = [f"{pre}.{n}" for pre, mod in (("shared_net", m.actor.shared_net), ("actor.GRU", m.actor.GRU), ("critic.GRU", m.critic.GRU),
                                           ("critic.Mean", m.critic.Mean), ("actor.Mean", m.actor.Mean)) for n, _ in mod.named_parameters()]
    assert len(names) == len(m.ac_parameters)
    sizes = [p.numel() for p in m.ac_parameters]
    fwd = bwd = 0.0
    for i, idx in enumerate(index):
        mb = {k: v[idx].double() for k, v in buf.items()}
        adv = trace["adv"].transpose(0, 1)[idx].double()
        vt = trace["v_target"].transpose(0, 1)[idx].double()
        logp, ent, val = policy_ref.train_forward(w, mb, D)
        la, lc = policy_ref.ppo_losses(logp, ent, val, mb, adv, vt, epsilon=m.epsilon, entropy_coef=m.entropy_coef,
                                       use_value_clip=m.use_value_clip)
        grads = torch.autograd.grad(la + lc, leaves, allow_unused=True)
        rec = trace["mb"][i]
        log(f"  -- minibatch {i}")
        tm = lambda x: x.transpose(0, 1)                 # noqa: E731
        fwd = max(fwd, _fwd_err(log, "logp", tm(rec["logp"]), logp), _fwd_err(log, "entropy", tm(rec["ent"]), ent),
                  _fwd_err(log, "value", tm(rec["val"]), val))
        for name, got, want in (("actor_loss", rec["actor_loss"], float(la)), ("critic_loss", rec["critic_loss"], float(lc))):
            r = abs(got - want) / (1e-4 * max(1.0, abs(want)))
            r = float("inf") if r != r else r
            log(f"  {name:<28s} {got:.8f} vs {want:.8f}   err/tol {r:.3f}")
            bwd = max(bwd, r)
        flat = trace["mb_grads"][i]
        off, worst_name, worst, worst_d, worst_scale = 0, None, 0.0, 0.0, 0.0
        for j, (k, g) in enumerate(zip(sizes, grads)):
            want = torch.zeros(k, dtype=torch.float64, device=DEV) if g is None else g.reshape(-1)
            d = float((flat[off:off + k].double() - want).abs().max())
            scale = float(want.abs().max())
            r = d / (1e-4 * scale) if scale > 0 else (0.0 if d == 0 else float("inf"))
            r = float("inf") if r != r else r
            if r >= worst:
                worst, worst_name, worst_d, worst_scale = r, names[j], d, scale
            off += k
        log(f"  {'gradients (worst tensor)':<28s} {worst_name}: max abs err {worst_d:.3e} of max {worst_scale:.3e}   err/tol {worst:.3f}")
        bwd = max(bwd, worst)
    return fwd, bwd


@pytest.mark.parametrize("D", [1, 3])
@pytest.mark.parametrize("N", [33, 64, 128])
def test_train_minibatches_large_teams_vs_fp64(log, monkeypatch, N, D):
    """Training forward and backward (message_agg + fcra_agg + GRU sequence + PPO head kernels) with reference_quirks on: the
    critic runs over all padded obstacle slots, as policy_ref.train_forward restates."""
    log(f"\n[train] N={N} D={D}")
    fwd, bwd = _train_case(log, monkeypatch, N, D)
    assert fwd <= 1.0 and bwd <= 1.0, (fwd, bwd)


def test_train_first_word_only_fails_at_64(log, monkeypatch):
    """Negative control: training on adjacency without words >= 1 fails the comparison against the full adjacency at N = 64."""
    def cut(p_adj):
        out = p_adj.clone()
        out[..., 32:] = 0
        return out
    log("\n[train control] N=64, kernels given word 0 only")
    fwd, _ = _train_case(log, monkeypatch, 64, 1, kernel_p_adj=cut)
    assert fwd > 1.0, fwd


# ------------------------------------------------------------------------------------------------------------ 5. rollout = training
@pytest.mark.parametrize("N,B,T", [(64, 4, 6), (100, 3, 5)])
def test_rollout_equals_training_forward_without_quirks(log, N, B, T):
    """With reference_quirks=False the training forward reproduces the rollout's log-probs and values (the N = 8 check of
    test_gpu_policy.py at large teams).  Pursuers and evader sit on random free cells: the reference's placement rule cannot seat
    this many pursuers on the default map."""
    from distributed_multi_agent_reinforcement_learning_b200 import maps
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena
    D, M = 2, 2
    m = _model(N, D, T=T, batch=B, mini_batch=B // 2 or 1, reference_quirks=False)
    cfg = m.cfg
    env = BatchedPursuitEnv(cfg, B, num_maps=M)
    rng = maps.GenRng(N)
    grids = np.stack([maps.make_obstacle_grid(cfg.map, rng) for _ in range(M)])
    infl = maps.dilate(grids, 2)
    env.set_maps(grids, infl)
    W, H = cfg.map.map_size
    g = np.random.default_rng(N)
    mid = (np.arange(B) % M).astype(np.int32)
    ps, es = np.zeros((B, N, 4)), np.zeros((B, 4))
    for b in range(B):
        free = np.argwhere(infl[mid[b]] == 0)
        cells = free[g.choice(len(free), N + 1, replace=False)]
        ps[b, :, :2], es[b, :2] = cells[:N], cells[N]
    tg = np.stack([maps.draw_target(infl[mid[b]], rng) for b in range(B)]).astype(np.int32)
    env.set_state(ps, es, tg, mid, time_step=0)
    env.set_target_tape(np.stack([g.integers(0, W, (B, 16)), g.integers(0, H, (B, 16))], axis=-1).astype(np.int32))
    env.start_episode()
    arena = RolloutArena(env.params, B, T, env.device)
    tb = m.rollout_batched(env, arena, T, seed=3)
    trace = {}
    m.train(tb, B * T * N, return_numpy=False, trace=trace)
    torch.cuda.synchronize()
    logp = torch.cat([t["logp"] for t in trace["mb"]], dim=1)
    val = torch.cat([t["val"] for t in trace["mb"]], dim=1)
    log(f"\n[rollout = training forward] N={N} B={B} T={T} D={D}")
    worst = max(_fwd_err(log, "logp", logp, tb.logp), _fwd_err(log, "value", val, tb.v[:-1]))
    assert worst <= 1.0, worst


# ------------------------------------------------------------------------------------------------------------ 6. configs[4] backward
@pytest.mark.parametrize("all_ones", [False, True], ids=["actor_adjacency", "all_ones"])
def test_message_bwd_precision_at_configs4_minibatch(log, all_ones):
    """marl_dhgn_message_bwd_det at configs[4]'s minibatch (32 envs x 250 steps x 64 pursuers: 8 000 samples, 512 000 rows, O = 110,
    E = 128): every weight and bias gradient within 1e-4 of its max of a float64 reference accumulated in sample chunks."""
    from distributed_multi_agent_reinforcement_learning_b200 import policy_ops as ops
    S, N, CH = 8000, 64, 80
    team = _team(S, N, M=32, seed=64)
    # dyadic states (1/16) and weights (1/256) make every fp32 pre-activation exact, so the kernel and the float64 reference take
    # the same ReLU branch everywhere: what remains is the rounding of the accumulation
    team.p, team.e = (team.p * 16).round() / 16, (team.e * 16).round() / 16
    W = [(t * 256).round() / 256 for t in _msg_weights(E, seed=11)]
    leaves = [t.clone().requires_grad_(True) for t in W]
    graph = _graph(team)
    out = ops.message_agg(graph, all_ones, *leaves)
    d_agg = torch.randn(out.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(12))
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(3):
        for t in leaves:
            t.grad = None
        start.record()
        torch.autograd.grad(out, leaves, d_agg, retain_graph=True)
        stop.record()
        torch.cuda.synchronize()
        times.append(start.elapsed_time(stop))
    out.backward(d_agg)
    names = ("MSG_layers.0.weight", "MSG_layers.0.bias", "MSG_layers.1.weight", "MSG_layers.1.bias", "MSG_layers.2.weight",
             "MSG_layers.2.bias")
    ref_leaves = [t.double().requires_grad_(True) for t in W]
    w = dict(zip(names, ref_leaves))
    fwd = 0.0
    for lo in range(0, S, CH):
        ref = _ref_message_agg(team, all_ones, w, lo, lo + CH)
        d = (out[lo:lo + CH].double() - ref.detach()).abs()
        fwd = max(fwd, float((d / (FWD["atol"] + FWD["rtol"] * ref.detach().abs())).max()))
        ref.backward(d_agg[lo:lo + CH].double())
        del ref, d
    log(f"\n[message backward, configs[4] minibatch] S={S} N={N} O={team.O} {'all_ones' if all_ones else 'actor'}: "
        f"backward {min(times):.2f} ms (best of 3, with its autograd glue); forward err/tol {fwd:.3f}")
    bwd = max(_grad_err(log, f"d {n}", a.grad, b.grad) for n, a, b in zip(names, leaves, ref_leaves))
    assert fwd <= 1.0 and bwd <= 1.0, (fwd, bwd)
