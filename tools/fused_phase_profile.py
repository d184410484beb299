"""Profiling aid: per-phase cycle counters of the fused policy step kernel (marl_policy_step.d_debug) at the bench shape.
MARL_VARIANT=3 (default: the pair kernel the bench runs) or 1 (one (tile, network) chain per CTA)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.fused_policy import FusedRolloutStep  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv  # noqa: E402

VARIANT = {"1": 1, "3": 3}.get(os.environ.get("MARL_VARIANT", "3"))
if VARIANT is None:
    sys.exit(f"MARL_VARIANT={os.environ['MARL_VARIANT']!r}: 1 (one chain per CTA) or 3 (pair kernel)")
if VARIANT == 3:
    os.environ["MARL_POLICY_PROFILE"] = "1"
cfg = bench.make_cfg()
B, M, N, E = bench.B_PER_GPU, 32, bench.N_AGENTS, 128
wl = bench.host_workload(cfg, B, M, seed=1)
env = BatchedPursuitEnv(cfg, B, num_maps=M)
env.set_maps(wl["grids"], wl["inflated"])
env.set_state(wl["p_state"], wl["e_state"], wl["target"], wl["map_id"], time_step=0)
env.set_target_tape(wl["tape"])
env.start_episode()
torch.manual_seed(0)
m = MAPPO(cfg, B, B // 10, "Learner")
w, _ = m.critic.head_weight()
fused = FusedRolloutStep(m, w.reshape(E).contiguous())
dev = env.device
oxy_i = env.boundary_xy.contiguous()
o_count = torch.clamp(env.boundary_count, max=env.O).contiguous()
ha, hc = torch.zeros(2, B * N, E, device=dev), torch.zeros(2, B * N, E, device=dev)
emb_a, emb_c = torch.empty(B, N, E, device=dev), torch.empty(B, N, E, device=dev)
act, logp, val = torch.zeros(B, N, dtype=torch.int32, device=dev), torch.empty(B, N, device=dev), torch.empty(B, N, device=dev)
hist = [0.1 * torch.randn(B, N, E, device=dev)]
env.observe()
n_tiles = (B * N + 127) // 128   # upper bound is 4/3 of this (the kernel may pick tiles down to 96 rows)
dbg = torch.zeros(24 * ((4 * n_tiles + 2) // 3), 16, dtype=torch.int64, device=dev)
for it in range(3):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    fused.step(env, oxy_i, o_count, it, 1, False, hist, hist, emb_a, emb_c, ha, hc, act, logp, val, debug=dbg, variant=VARIANT)
    e.record()
    e.synchronize()
    print("launch ms", s.elapsed_time(e))
d = dbg.cpu().numpy().astype(np.float64)
if VARIANT == 3:
    d_all = d
    d = d[: int((d[:, 13] > 1e15).sum())]
# wall-clock schedule of the launch: effective SM clock, gaps between consecutive CTAs of one SM
g0, g1, sm = d[:, 13], d[:, 14], d[:, 15].astype(int)
ok = d[:, 12] > 0
print(f"effective clock: {np.median(d[ok, 12] / (g1[ok] - g0[ok])):.3f} GHz; launch span {(g1[ok].max() - g0[ok].min()) / 1e3:.1f} us")
gaps = []
for s_ in np.unique(sm[ok]):
    idx = np.where(ok & (sm == s_))[0]
    idx = idx[np.argsort(g0[idx])]
    gaps += list(g0[idx][1:] - g1[idx][:-1])
    if s_ == 0:
        print("SM 0 schedule (start us, dur us):", [(round((g0[i] - g0[ok].min()) / 1e3, 1), round((g1[i] - g0[i]) / 1e3, 1)) for i in idx])
print(f"gap between consecutive CTAs on an SM: median {np.median(gaps) / 1e3:.2f} us, max {np.max(gaps) / 1e3:.2f} us; CTAs per SM: {ok.sum() / len(np.unique(sm[ok])):.2f}")
if VARIANT == 3:
    grid = len(d)                                 # CTA rows carry a %globaltimer stamp; the per-step rows follow them
    d = d[:grid]
    tot = d[:, 12]
    print(f"pair items {len(d)}; per-item worker cycles: mean {tot.mean():.0f} min {tot.min():.0f} max {tot.max():.0f}; sum/148 = {tot.sum() / 148:.0f}")
    for i, n in ((0, "messages"), (1, "epi_store"), (2, "fcra"), (3, "fill_x"), (4, "cell halves"), (5, "head"), (15, "loop back-edge"), (9, "dispatch+prefetch"), (10, "signal"), (11, "wait mma")):
        print(f"   {n:14s} {d[:, i].mean():10.0f} cycles ({100 * d[:, i].mean() / tot.mean():5.1f}%)")
    print(f"   issuer: waiting for the workers {d[:, 6].mean():.0f}, for weights {d[:, 7].mean():.0f}, total {d[:, 8].mean():.0f} -> issuing / idle in MMA queue {d[:, 8].mean() - d[:, 6].mean() - d[:, 7].mean():.0f}")
    sys.exit(0)
names = ["msg0", "msg1", "msg2", "epi_av(x3)", "epi_sem", "fcra", "epi_aggf", "epi_f", "load_hidden(x2)", "epi_cell(x2)", "head",
         "wait_mma(all)", "total"]
d = d[d[:, 12] > 0]            # CTAs that ran (critic items first, then the actor's)
n_tiles = len(d) // 2
print("items", len(d), "rows per tile ~", -(-B * N // max(n_tiles, 1)))
tot = d[:, 12]
print(f"per-item worker cycles: mean {tot.mean():.0f} min {tot.min():.0f} max {tot.max():.0f} std {tot.std():.0f}; sum/148 SMs = {tot.sum() / 148:.0f} cycles")
for label, rows in (("critic", d[:n_tiles]), ("actor", d[n_tiles:])):
    print(label, "tiles", len(rows))
    for i, n in enumerate(names):
        print(f"   {n:18s} {rows[:, i].mean():10.0f} cycles  ({100 * rows[:, i].mean() / rows[:, 12].mean():5.1f}%)")
