#!/usr/bin/env python
"""bench.py — headline benchmark of the rollout hot path (driver contract: see the task statement).

Workload (BASELINE.json configs[1]): pursuit-evasion with obstacles, 8 pursuers + 1 A*-driven evader, 60x55 map,
O=176, T=150 steps, 4096 batched envs per B200.  One bench "step" = one whole closed-loop episode of all envs:
per env step  evader A* / waypoint step -> observe (comm adjacency, LoS, obstacle visibility) -> pursuer step ->
actor encoder -> critic encoder -> GRU -> heads (sample / log-prob / value) -> reward-norm -> store into the time-major
rollout arena, i.e. MAPPO.run_episode (DHGN/mappo_parallel.py:742-827) for all envs at once.

metric = agent-env-steps/s = B*N*T / time, whole job (all ranks).
  value : episode replayed from HBM-resident initial state (one CUDA graph of the whole episode).
  env_only / train : secondary numbers (env-only closed loop with scripted random actions; one PPO epoch).
  e2e   : same episode through the public per-iteration call `MAPPO.explore_batched(engine, arena, host_state=..., host_out=...)`
          with HOST buffers: pinned initial states/targets H2D + per-env episode reward sums / collision flags D2H inside the
          timed region.
--impl reference : the CPU port of the same loop (oracle/marl_oracle.c env with OpenMP + the torch-CPU restatement of
          the networks, all host threads) on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "agent_env_steps_per_sec"
UNIT = "agent-env-steps/s"
N_AGENTS, B_PER_GPU, T_STEPS, N_MAPS = 8, 4096, 150, 256
STREAM_GROUPS = 16   # independent env sub-batches on separate streams inside the episode graph
SURVEY_BYTES_PER_AGENT_STEP = 118.0   # SURVEY.md §8(d): 72 state r/w + 22 raser row + 1 p_adj + 1 e_adj + 22 o_adj (N=8, O=176)


def workload_config(n_gpus):
    return {"workload": "pursuit_evasion_obstacles_8p_gru_c2", "num_pursuers": N_AGENTS, "envs_per_gpu": B_PER_GPU,
            "global_envs": B_PER_GPU * n_gpus, "max_steps": T_STEPS, "map": "60x55", "num_max_obstacle": 176,
            "map_pool_per_gpu": N_MAPS, "evader": "gpu A* (replan every 10 steps)",
            "policy": "DHGN actor + critic (embedding 128, depth 1, 2-layer GRU) in the loop, random-init weights, fp32-level arithmetic "
                      "(fp32 SIMT + tensor-core GEMMs on two-term fp16 / 3xTF32 operand splits with fp32 accumulation)",
            "parallelism": f"dp{n_gpus} (independent env shards, no data-path collective)",
            "l2": "flushed between timed iterations (256 MiB write)"}


def make_cfg():
    from distributed_multi_agent_reinforcement_learning_b200 import default_config
    return default_config(env__num_defender=N_AGENTS, env__max_steps=T_STEPS)


def host_workload(cfg, B, M, seed):
    """Synthetic initial conditions generated on the host with the reference's placement rules (untimed set-up)."""
    import numpy as np
    from distributed_multi_agent_reinforcement_learning_b200 import maps
    rng = maps.GenRng(seed)
    W, H = cfg.map.map_size
    grids = np.zeros((M, W, H), np.uint8)
    infl = np.zeros_like(grids)
    for m in range(M):
        grids[m] = maps.make_obstacle_grid(cfg.map, rng)
    infl = maps.dilate(grids, 2)
    N = cfg.env.num_defender
    ps = np.zeros((B, N, 4))
    es = np.zeros((B, 4))
    tg = np.zeros((B, 2), np.int32)
    mid = (np.arange(B) % M).astype(np.int32)
    for b in range(B):
        work = infl[mid[b]].copy()
        tg[b] = maps.draw_target(infl[mid[b]], rng)
        pxy, cells = maps.place_pursuers(work, N, float(cfg.defender.comm_range), rng)
        ps[b, :, :2] = pxy
        es[b, :2] = maps.place_evader(work, cells, float(cfg.defender.sen_range), rng)
    tape = np.stack([rng.g.integers(0, W, (B, 16)), rng.g.integers(0, H, (B, 16))], axis=-1).astype(np.int32)
    return dict(grids=grids, inflated=infl, p_state=ps, e_state=es, target=tg, map_id=mid, tape=tape)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index, self.t0 = [], None, index, None

    def start(self):
        """Launched BEFORE the warm-up (nvidia-smi needs a few hundred ms to print its first row); `mark()` opens the timed region."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def mark(self):
        self.t0 = time.monotonic()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)                                   # the row that covers the end of the timed region
        self.proc.terminate()
        t0 = self.t0 if self.t0 is not None else 0.0
        rows = [r for t, r in self.rows if t >= t0]        # rows printed inside the timed region (+ the one right after it)
        scope = "timed region"
        if not any(r and r[0].isdigit() for r in rows):    # a very short region: fall back to the warm-up + timed region
            rows, scope = [r for _, r in self.rows], "warm-up + timed region"
        sm = sorted(int(r[0]) for r in rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].startswith("Active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "sampled_over": scope}


def policy_flops_per_agent(N, O, D, head=2304):
    """SURVEY.md 8(d): forward FLOPs per agent per network (mult-add = 2)."""
    return 2048 * N + 1024 + 1024 * O + 256 * (N + 1 + O) + 3 * 32768 + 99328 + D * (256 * N + 98304) + 393216 + head


def measured_tensor_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1500.0)))
    return 1500.0


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------ CPU reference
def cpu_rollout(cfg, wl, n_envs, steps_T, seed):
    """The oracle port of the same closed loop on `n_envs` envs of the workload, all host threads.
    Returns (seconds, agent_env_steps)."""
    import numpy as np
    from oracle import oracle as orc
    from distributed_multi_agent_reinforcement_learning_b200 import env_params_dict, maps
    p = orc.EnvParams.from_dict(env_params_dict(cfg))
    B, N, O, M = n_envs, p.N, p.O, wl["grids"].shape[0]
    # per-map sensor tables with the oracle itself (untimed set-up, like reset in the reference)
    beam = maps.beam_directions(p.sensor_beams)
    used = sorted(set(int(m) for m in wl["map_id"][:B]))
    raser = np.zeros((M, p.W * p.H, O), np.uint8)
    ob_count = np.zeros(M, np.int32)
    for m in used:
        b_, xy, n = orc.boundary_map(p, wl["grids"][m])
        ob_count[m] = min(n, O)
        raser[m, :, :min(n, O)] = orc.raser_map(p, b_, xy, beam).reshape(p.W * p.H, -1)[:, :O]
    st = dict(p_state=wl["p_state"][:B].copy(), e_state=wl["e_state"][:B].copy(), target=wl["target"][:B].copy(),
              path=np.zeros((B, 512, 2), np.int16), path_len=np.zeros(B, np.int32),
              grid=np.ascontiguousarray(wl["grids"]), inflated=np.ascontiguousarray(wl["inflated"]), raser=raser,
              ob_count=ob_count, map_id=wl["map_id"][:B].copy(), action_table=maps.action_table(cfg.defender.vmax),
              tape=np.ascontiguousarray(wl["tape"][:B]), tape_pos=np.zeros(B, np.int32),
              p_adj=np.zeros((B, N, N), np.uint8), o_adj=np.zeros((B, N, O), np.uint8), e_adj=np.zeros((B, N), np.uint8),
              reward=np.zeros((B, N), np.int32), can_apply=np.zeros((B, N), np.uint8), collision=np.zeros(B, np.uint8),
              time_step=np.zeros(B, np.int32), done=np.zeros(B, np.uint8), wf_n=np.zeros(B, np.int64),
              wf_mean=np.zeros((B, N)), wf_S=np.zeros((B, N)), wf_std=np.zeros((B, N)),
              r_norm=np.zeros((B, N), np.float32), status=np.zeros(B, np.int32))
    rng = np.random.default_rng(seed)
    actions = rng.integers(0, 9, (steps_T, B, N)).astype(np.int32)
    t0 = time.perf_counter()
    for t in range(steps_T):
        st["action"] = actions[t]
        orc.rollout_iteration_closed(p, st)
    dt = time.perf_counter() - t0
    assert not st["status"].any(), "oracle evader reported an error"
    return dt, B * N * steps_T


def _reference_weights(cfg, seed=0xB200):
    """Random-init weights of the reference architecture as a name->tensor dict (same initialisers and order as the
    reference: orthogonal Linear layers, default nn.GRU init, spectral-norm buffers)."""
    import torch
    import torch.nn as nn
    a = cfg.algo
    E, D = a.embedding_dim, a.depth
    torch.manual_seed(seed)

    def lin(i, o):
        layer = nn.Linear(i, o)
        nn.init.orthogonal_(layer.weight)
        nn.init.constant_(layer.bias, 0)
        return layer

    w = {}

    def put(prefix, layer):
        w[prefix + ".weight"], w[prefix + ".bias"] = layer.weight.detach(), layer.bias.detach()

    enc = {"semantic_layer": lin(3 * E + 4, E)}
    for r in range(3):
        enc[f"MSG_layers.{r}"] = lin(8 if r == 0 else 4, E)
    for k in range(D):
        enc[f"FCRA_layers.{k}"] = lin(2 * E, E)
    enc["AGG_layers.AGG_vertex_0"] = lin(E, E)
    for k in range(D):
        enc[f"AGG_layers.AGG_fcra_{k}"] = lin(E, E)
    for net in ("actor", "critic"):
        for name, layer in enc.items():
            put(f"{net}.shared_net.{name}", layer)
        gru = nn.GRU(E, E, a.num_layers)
        for k, v in gru.state_dict().items():
            w[f"{net}.GRU.{k}"] = v
        if net == "actor":
            put("actor.Mean", lin(E, cfg.env.action_dim))
        else:
            head = lin(E, 1)
            w["critic.Mean.weight_orig"], w["critic.Mean.bias"] = head.weight.detach(), head.bias.detach()
            w["critic.Mean.weight_u"] = torch.nn.functional.normalize(torch.randn(1), dim=0)
    return w


def cpu_policy_rollout(cfg, wl, n_envs, steps_T, seed=0):
    """The reference rollout body (DHGN/mappo_parallel.py:758-801) on the host: oracle C env (observe, A* evader, step,
    reward-norm; OpenMP) + the torch-CPU restatement of both networks (oracle/policy_ref.py), dense tensors as in the
    reference.  Returns (seconds, agent_env_steps)."""
    import numpy as np
    import torch
    from oracle import oracle as orc, policy_ref
    from distributed_multi_agent_reinforcement_learning_b200 import env_params_dict, maps
    p = orc.EnvParams.from_dict(env_params_dict(cfg))
    B, N, O, M = n_envs, p.N, p.O, wl["grids"].shape[0]
    E, D, L = cfg.algo.embedding_dim, cfg.algo.depth, cfg.algo.num_layers
    beam = maps.beam_directions(p.sensor_beams)
    raser = np.zeros((M, p.W * p.H, O), np.uint8)
    ob_count = np.zeros(M, np.int32)
    oxy = np.zeros((M, O, 4), np.float32)
    for m in sorted(set(int(v) for v in wl["map_id"][:B])):
        b_, xy, n = orc.boundary_map(p, wl["grids"][m])
        n = min(n, O)
        ob_count[m] = n
        raser[m, :, :n] = orc.raser_map(p, b_, xy[:n], beam).reshape(p.W * p.H, -1)
        oxy[m, :n, :2] = xy[:n]
    st = dict(p_state=wl["p_state"][:B].copy(), e_state=wl["e_state"][:B].copy(), target=wl["target"][:B].copy(),
              path=np.zeros((B, 512, 2), np.int16), path_len=np.zeros(B, np.int32),
              grid=np.ascontiguousarray(wl["grids"]), inflated=np.ascontiguousarray(wl["inflated"]), raser=raser,
              ob_count=ob_count, map_id=wl["map_id"][:B].copy(), action_table=maps.action_table(cfg.defender.vmax),
              tape=np.ascontiguousarray(wl["tape"][:B]), tape_pos=np.zeros(B, np.int32),
              p_adj=np.zeros((B, N, N), np.uint8), o_adj=np.zeros((B, N, O), np.uint8), e_adj=np.zeros((B, N), np.uint8),
              reward=np.zeros((B, N), np.int32), can_apply=np.zeros((B, N), np.uint8), collision=np.zeros(B, np.uint8),
              time_step=np.zeros(B, np.int32), done=np.zeros(B, np.uint8), wf_n=np.zeros(B, np.int64),
              wf_mean=np.zeros((B, N)), wf_S=np.zeros((B, N)), wf_std=np.zeros((B, N)),
              r_norm=np.zeros((B, N), np.float32), status=np.zeros(B, np.int32))
    w = _reference_weights(cfg)
    mid = torch.from_numpy(st["map_id"]).long()
    o_ten = torch.from_numpy(oxy)[mid]                                                     # [B,O,4]
    o_real = (torch.arange(O)[None, :] < torch.from_numpy(ob_count)[mid][:, None]).float()   # [B,O]
    gen = torch.Generator().manual_seed(seed)
    ha, hc = torch.zeros(L, B * N, E), torch.zeros(L, B * N, E)
    emb_a_prev, emb_c_prev = [], []
    zero = torch.zeros(B, N, E)
    t0 = time.perf_counter()
    with torch.no_grad():
        for t in range(steps_T):
            orc.observe_batch(p, st)
            obs = dict(p=torch.from_numpy(st["p_state"]).float(), e=torch.from_numpy(st["e_state"]).float().unsqueeze(1),
                       o=o_ten, p_adj=torch.from_numpy(st["p_adj"]).float(), e_adj=torch.from_numpy(st["e_adj"]).float().unsqueeze(-1),
                       o_adj=torch.from_numpy(st["o_adj"]).float(), o_real=o_real)
            hist = []
            for k in range(D):          # aliased history list: C(t-1), A(t-1), C(t-2), ...
                back, src = k // 2 + 1, (emb_c_prev if k % 2 == 0 else emb_a_prev)
                hist.append(src[-back] if len(src) >= back else zero)
            a, lp, val, ea, ec, ha, hc = policy_ref.rollout_step(w, obs, hist, ha, hc, D, L, generator=gen)
            emb_a_prev.append(ea)
            emb_c_prev.append(ec)
            emb_a_prev, emb_c_prev = emb_a_prev[-(D // 2 + 1):], emb_c_prev[-(D // 2 + 1):]
            st["action"] = np.ascontiguousarray(a.numpy().astype(np.int32))
            orc.rollout_iteration_closed(p, st)
    dt = time.perf_counter() - t0
    assert not st["status"].any(), "oracle evader reported an error"
    return dt, B * N * steps_T


def use_all_host_threads():
    """The CPU arm runs on every host thread this process may use.  torchrun exports OMP_NUM_THREADS=1 to its workers when the
    variable is unset, which would silently make the N > 1 reference arm a one-thread run: set the count explicitly in the
    environment (for runtimes not initialised yet), in the GNU OpenMP runtime the C oracle links, and in torch."""
    import ctypes
    import torch
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    os.environ["OMP_NUM_THREADS"] = str(n)
    try:
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(n)
    except OSError:
        pass
    torch.set_num_threads(n)
    return n


def cpu_policy_baseline(cfg, wl, steps_T, budget_s):
    """Bounded sample of the same workload on the host: sized from a short calibration so one pass is ~budget_s."""
    import torch
    from oracle import oracle as orc
    orc.build()
    use_all_host_threads()
    cores = orc.num_threads()
    torch.set_num_threads(cores)
    n0 = min(32, len(wl["map_id"]))
    dt, n = cpu_policy_rollout(cfg, wl, n0, 5)
    per_env_step = dt / (n0 * 5)
    n_envs = int(max(8, min(len(wl["map_id"]), budget_s / (per_env_step * steps_T))))
    dt, n = cpu_policy_rollout(cfg, wl, n_envs, steps_T)
    return {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"first {n_envs} of {B_PER_GPU} envs x {steps_T} steps: oracle/marl_oracle.c env (OpenMP) + torch-CPU "
                      f"restatement of actor/critic (oracle/policy_ref.py), {cores} threads, {dt:.1f} s"}, n_envs


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = make_cfg()
    wl = host_workload(cfg, 512, min(N_MAPS, 512), seed=0xB200 + 1)
    base, n_envs = cpu_policy_baseline(cfg, wl, steps_T=30, budget_s=2.0)      # calibration + warm-up
    for _ in range(max(0, args.warmup - 1)):
        cpu_policy_rollout(cfg, wl, n_envs, 10)
    # size the per-step sample so that the whole run stays within a few minutes
    per_env_step = 1.0 / (base["value"] / N_AGENTS)
    n_envs = int(max(8, min(512, 8.0 / (per_env_step * T_STEPS))))
    tot_t, tot_n = 0.0, 0
    for k in range(args.steps):
        dt, n = cpu_policy_rollout(cfg, wl, n_envs, T_STEPS, seed=2 + k)
        tot_t += dt
        tot_n += n
    value = tot_n / tot_t
    from oracle import oracle as orc
    desc = (f"{n_envs} of {B_PER_GPU} envs x {T_STEPS} steps per step: oracle C env (A* evader, OpenMP) + torch-CPU actor/critic "
            f"restatement, {orc.num_threads()} threads")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64 env / f32 networks", "data": "synthetic", "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": orc.num_threads(), "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ------------------------------------------------------------------------------------------------ our arm
def policy_flops_split(N, O_actor, O_critic, D, head=2304):
    """SURVEY 8(d) per-agent forward FLOPs, split: (gemm-only per network [the 128-wide dense layers + heads: what the tensor
    cores execute], actor messages / aggregation with O_actor obstacle slots, same for the critic with O_critic)."""
    gemm = 3 * 32768 + 99328 + D * 98304 + 393216 + head
    msg = lambda O: 2048 * N + 1024 + 1024 * O + 256 * (N + 1 + O) + D * 256 * N
    return gemm, msg(O_actor), msg(O_critic)


def train_bytes_per_sample(D):
    """Algorithmic HBM bytes of one PPO training sample (one agent-step, BOTH networks) for the layer-by-layer schedule that
    `MAPPO.train` runs (DESIGN.md section 5): every layer reads its input rows once and writes its output rows once in the forward
    pass; the backward pass reads each saved activation and each upstream gradient once and writes each downstream gradient once
    (dX and dW share one read of dY only inside the GRU sequence kernel).  Unit = one 128-float row (512 B), per network:
      forward : messages 3 w | AGG_vertex 3 r + 3 w | semantic 3 r + 1 w (+ 2 for the state term) | per depth: neighbour mean 1 r + 1 w,
                AGG_fcra 1 r + 1 w, FCRA 2 r + 1 w | per GRU layer: input projection 1 r + 3 w, recurrence 3 r + 1 w + 4 saves | head 1 r
      backward: 2 x forward (dX pass + dW pass over the same rows)."""
    fwd_rows = 3 + 6 + 6 + D * 7 + 2 * 12 + 1
    return 2 * 3 * fwd_rows * 512


DUMP_ENVS, DUMP_SEED = 32, 0    # 32 of 4096 envs keep the dump at ~41 MiB, most of it the two [T+D,B,N,128] embedding histories


def dump_outputs(batch, out_dir):
    """Writes the TrainBatch that `MAPPO.explore_batched` returned for the last timed episode as <out_dir>/<key>.npy, restricted to
    a fixed, seeded sample of DUMP_ENVS envs (axis 1 of every key, in ascending env order).  float32, except the bit-packed
    adjacency words (int32), which are written as float64 so that they stay exact."""
    import numpy as np
    import torch
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import TrainBatch
    envs = np.sort(np.random.default_rng(DUMP_SEED).choice(batch.B, size=min(DUMP_ENVS, batch.B), replace=False))
    idx = torch.from_numpy(envs).to(batch.p.device)
    out = {}
    for k in TrainBatch.KEYS:
        a = getattr(batch, k).index_select(1, idx).cpu().numpy()
        out[k] = a.astype(np.float64 if a.dtype == np.int32 else np.float32)
    assert sum(a.nbytes for a in out.values()) <= 64e6
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def _popcount_mean(torch, words):
    """Mean number of set bits per row of a packed int32 [..., W] tensor."""
    w = words.to(torch.int64) & 0xFFFFFFFF
    cnt = torch.zeros(w.shape[:-1], dtype=torch.float64, device=w.device)
    for b in range(32):
        cnt += ((w >> b) & 1).sum(-1)
    return cnt.mean().item()


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from distributed_multi_agent_reinforcement_learning_b200 import _lib, parallel
    from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO
    from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, EpisodeGraph, RolloutArena

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — this arm has no CPU fallback")
    _lib.lib()   # fail loudly if the CUDA library is missing
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    cfg = make_cfg()
    B, N, T, M = B_PER_GPU, N_AGENTS, T_STEPS, N_MAPS
    wl = host_workload(cfg, B, M, seed=0xB200 + 1 + 7919 * rank)
    env = BatchedPursuitEnv(cfg, B, device=dev, num_maps=M)
    env.set_maps(wl["grids"], wl["inflated"])
    env.set_state(wl["p_state"], wl["e_state"], wl["target"], wl["map_id"], time_step=0)
    env.set_target_tape(wl["tape"])
    env.start_episode()
    arena = RolloutArena(env.params, B, T, dev)
    snap = env.snapshot()
    torch.manual_seed(0xB200)
    mappo = MAPPO(cfg, B, max(1, round(B / 10)), "Learner")      # mini_batch = round(workers/10) (main.py:48)
    mappo.sync_weights(0)
    SEED = 0xB200 + rank
    mappo.explore_batched(env, arena, T, seed=SEED)                # the public call; its first use captures the episode graph
    torch.cuda.synchronize()
    env.restore(snap)
    pol = mappo._episode_graphs[(id(env), id(arena), T, SEED)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def per_rank(ms):
        """[rank 0 .. rank N-1] of a per-rank time: the whole-job number is quoted on the slowest one."""
        t = torch.tensor([float(ms)], dtype=torch.float64, device=dev)
        if world == 1:
            return [float(ms)]
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [float(x.item()) for x in out]

    def timed(fn, n_iter, before=None):
        total = 0.0
        for _ in range(n_iter):
            if before is not None:
                before()
            flush.fill_(1)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            e.synchronize()
            total += s.elapsed_time(e)
        return total

    # ---- value: whole episode with the networks in the loop, HBM-resident -----------------------------------
    restore = lambda: env.restore(snap)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    timed(pol.replay, args.warmup, restore)
    barrier()
    sampler.mark()
    ms_total = timed(pol.replay, args.steps, restore)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    status = int(env.evader_status.max().item())
    assert status == 0, f"evader status {status}: search overflow or target tape exhausted"
    if args.dump_outputs and rank == 0:
        dump_outputs(pol.batch, args.dump_outputs)      # before e2e: it replays the same graph into the same buffers
    per_rank_ms = {"value": [x / args.steps for x in per_rank(ms_total)]}
    ms_total = parallel.max_over_ranks(ms_total, dev)
    value = world * B * N * T * args.steps / (ms_total * 1e-3)

    # ---- e2e: host buffers in, host metrics out ----------------------------------------------------------------
    pin = {k: torch.from_numpy(np.ascontiguousarray(wl[k])).pin_memory() for k in ("p_state", "e_state", "target")}
    ep_reward_host = torch.zeros(B, dtype=torch.int64).pin_memory()
    coll_host = torch.zeros(B, dtype=torch.uint8).pin_memory()
    h2d = sum(v.numel() * v.element_size() for v in pin.values())
    d2h = ep_reward_host.numel() * 8 + coll_host.numel()

    host_state = {k: pin[k] for k in ("p_state", "e_state", "target")}
    host_out = {"episode_reward": ep_reward_host, "collision": coll_host}

    def e2e_episode():
        # the public per-iteration call with HOST buffers: H2D of the initial state, the whole episode, D2H of the per-env results
        mappo.explore_batched(env, arena, T, seed=SEED, host_state=host_state, host_out=host_out, reset_reward_norm=True)

    timed(e2e_episode, args.warmup)
    barrier()
    e2e_ms = timed(e2e_episode, args.steps)
    barrier()
    per_rank_ms["e2e"] = [x / args.steps for x in per_rank(e2e_ms)]
    e2e_value = world * B * N * T * args.steps / (parallel.max_over_ranks(e2e_ms, dev) * 1e-3)

    # ---- secondary: env-only closed loop (scripted random policy), as in the survey's env-only probe ------------
    env.restore(snap)
    env_graph = EpisodeGraph(env, arena, T, seed=0xB200 + rank, groups=STREAM_GROUPS)
    timed(env_graph.replay, 2, restore)
    barrier()
    env_ms_local = timed(env_graph.replay, max(3, args.steps // 2), restore) / max(3, args.steps // 2)
    per_rank_ms["env_only"] = per_rank(env_ms_local)
    env_ms = parallel.max_over_ranks(env_ms_local, dev)
    env_only = {"value": world * B * N * T / (env_ms * 1e-3), "unit": UNIT, "ms_per_episode": env_ms,
                "policy": "uniform random actions (device counter RNG)", "stream_groups": STREAM_GROUPS}

    # ---- secondary: MAPPO training samples/s (GAE + 10 sequential minibatches fwd/bwd/clip + all-reduce + Adam) ---
    env.restore(snap)
    pol.replay()
    torch.cuda.synchronize()
    tb = pol.batch

    def train_epoch():
        mappo.train(tb, total_steps=B * T, return_numpy=False)
        mappo.update(B * T)

    train_epoch()
    barrier()
    n_train = max(1, min(3, args.steps))
    tr_ms_local = timed(train_epoch, n_train) / n_train
    per_rank_ms["train"] = per_rank(tr_ms_local)
    tr_ms = parallel.max_over_ranks(tr_ms_local, dev)
    hbm_peak, peak_src = measured_peaks()
    tensor_peak = measured_tensor_peak()
    D = int(cfg.algo.depth)
    o_b = float(torch.clamp(env.boundary_count, max=env.O).float()[env.map_id.long()].mean())      # real boundary cells per env
    gemm_f, msg_a_all, msg_c_all = policy_flops_split(N, env.O, env.O, D)
    tr_bytes = train_bytes_per_sample(D) * B * T * N
    tr_flops = 3 * (2 * gemm_f + msg_a_all + msg_c_all) * B * T * N            # forward + dX + dW passes; training pads to all O slots
    train = {"samples_per_sec": world * B * T * N / (tr_ms * 1e-3), "unit": "samples/s", "ms_per_epoch": tr_ms,
             "minibatches": -(-B // mappo.mini_batch_size), "dtype": "f32 (TF32 off)",
             "allreduce": "1 x SUM over the flat gradient arena (%d floats) per update; train(allreduce='minibatch') = 1 per PPO minibatch"
                          % mappo.ac_optimizer.flat_grad.numel(),
             "roofline": {"bound": "hbm", "achieved": tr_bytes / (tr_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                          "frac": tr_bytes / (tr_ms * 1e-3) / 1e9 / hbm_peak, "traffic": None,
                          "algorithmic_bytes_per_sample": train_bytes_per_sample(D),
                          "bytes_model": "layer-by-layer schedule: each layer reads its input rows and writes its output rows once "
                                         "forward, twice that backward (bench.train_bytes_per_sample; DESIGN.md section 5)",
                          "tensor_TFLOPs": tr_flops / (tr_ms * 1e-3) / 1e12, "tensor_frac": tr_flops / (tr_ms * 1e-3) / 1e12 / tensor_peak,
                          "peak_source": peak_src}}

    # ---- per-kernel durations (1): CUDA events around every launch of ONE eager, single-pipeline episode (same stream) -----
    env.restore(snap)
    timers = {}
    mappo.rollout_batched(env, arena, T, seed=SEED, timers=timers)
    torch.cuda.synchronize()
    kernel_table = {k: {"launches": len(v), "total_ms": sum(a.elapsed_time(b) for a, b in v)} for k, v in timers.items()}
    for v in kernel_table.values():
        v["avg_us"] = 1e3 * v["total_ms"] / v["launches"]
    # ---- per-kernel durations (2): the same events inside the schedule that `value` times - G env-group pipelines on G streams.
    # A group's policy launch is timed on its own stream; launches of different groups overlap, so the kernel's time per episode
    # is the UNION of its launch intervals (<= the episode's wall time by construction).
    G = MAPPO.default_pipelines(B, N)
    pk = kernel_table["policy_step_kernel"]
    pipe = None
    if G > 1:
        # The SAME graph-captured pipelined schedule once more, every policy launch writing its per-CTA %globaltimer start / end
        # and SM id (the kernel's profiling record): a launch's interval is [first CTA start, last CTA end]; launches of different
        # env groups overlap, so the kernel's time per episode is the UNION of the intervals (<= the episode's wall time).
        from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import RolloutGraph
        full_tile = (128 // N) * N
        ctas = 2 * (-(-(B // G) * N // full_tile) + 1)
        dbg = torch.zeros(T, G, ctas, 16, dtype=torch.int64, device=dev)
        env.restore(snap)
        ig = RolloutGraph(mappo, env, arena, T, SEED, policy_dbg=dbg)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(2):
            env.restore(snap)
            dbg.zero_()
            flush.fill_(1)
            ev0.record()
            ig.replay()
            ev1.record()
            torch.cuda.synchronize()
        wall = ev0.elapsed_time(ev1)
        rec = dbg.cpu().numpy()
        if os.environ.get("MARL_BENCH_TIMELINE"):          # tools: per-CTA (cycles, start ns, end ns, SM id) of every policy launch
            np.savez_compressed(os.environ["MARL_BENCH_TIMELINE"], rec=rec[..., 12:16], wall_ms=wall)
        used = rec[..., 14] > 0
        starts = np.where(used, rec[..., 13], np.iinfo(np.int64).max).min(axis=2)      # [T, G] ns
        ends = np.where(used, rec[..., 14], 0).max(axis=2)
        iv = sorted(zip(starts.reshape(-1).tolist(), ends.reshape(-1).tolist()))
        union, cs, ce = 0, None, None
        for a_, b_ in iv:
            if ce is None or a_ > ce:
                union += (ce - cs) if ce is not None else 0
                cs, ce = a_, b_
            else:
                ce = max(ce, b_)
        union += (ce - cs) if ce is not None else 0
        cta_busy_ns = float(np.where(used, rec[..., 14] - rec[..., 13], 0).sum())
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        pipe = {"pipelines": G, "instrumented_graph_episode_ms": wall, "policy_launches": int(starts.size),
                "policy_group_launch_avg_us": float((ends - starts).mean()) * 1e-3,
                "policy_union_ms": union * 1e-6, "policy_share_of_episode": union * 1e-6 / wall,
                "policy_sm_busy_ms": cta_busy_ns * 1e-6 / n_sm,
                "note": "per-CTA %globaltimer records written by policy_step_kernel inside the graph-captured pipelined schedule; "
                        "union = time during which at least one policy launch is executing; sm_busy = sum of CTA lifetimes / SMs"}
    env.restore(snap)
    ms_episode = ms_total / args.steps
    flops_pp = policy_flops_per_agent(N, env.O, D)
    flops_launch = 2 * flops_pp * B * N                                       # actor + critic, SURVEY 8(d) upper bound (all O slots)
    # executed obstacle work: the actor touches only visible cells, the critic the O_b real boundary cells of the map
    o_vis = float(_popcount_mean(torch, pol.batch.o_adj_bits))
    _, msg_a_exec, msg_c_exec = policy_flops_split(N, o_vis, o_b, D)
    flops_exec_launch = (2 * gemm_f + msg_a_exec + msg_c_exec) * B * N
    # headline rate: on the timed region itself - the episode's policy FLOPs over the driver-timed episode (a lower bound of the
    # kernel's own rate: the episode also contains the env / A* kernels), and over the union of the kernel's launch intervals
    policy_ms = pipe["policy_union_ms"] * min(1.0, ms_episode / pipe["instrumented_graph_episode_ms"]) if pipe else pk["total_ms"]
    policy_ms = min(policy_ms, ms_episode)
    achieved = flops_launch * (T + 1.0 / 2) / (policy_ms * 1e-3) / 1e12       # T two-network launches + the bootstrap critic launch
    achieved_step = flops_launch * (T + 1.0 / 2) / (ms_episode * 1e-3) / 1e12
    # HBM traffic the fused kernel needs per launch: state/adjacency in, history in, embedding + hidden (r/w) + heads out
    bytes_launch = B * N * (32 + 4 + 1 + 24 + 2 * (D * 512 + 512 + 4 * 512) + 12)
    roofline = {"kernel": "policy_step_kernel (DHGN encoder + 2-layer GRU + heads of actor AND critic, one launch per env step and env group; "
                          "tcgen05 kind::f16 on a two-term fp16 split of both operands, 3 products per K step for fp32-level accuracy, "
                          "accumulators in TMEM)",
                "bound": "tensor", "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s", "frac": achieved / tensor_peak,
                "traffic": None,
                "traffic_note": "not measured in this run; profiles/ holds the dram bytes of one launch from the ncu --set full capture",
                "timing": "in-kernel %globaltimer records of every policy launch inside the graph-captured pipelined schedule that `value` "
                          "times (a second, instrumented capture of the same schedule); kernel time per episode = union of the launch "
                          "intervals",
                "policy_ms_per_episode": policy_ms, "ms_per_step": ms_episode,
                "frac_on_timed_episode": achieved_step / tensor_peak,
                "frac_gemm_only": (2 * gemm_f * B * N) * (T + 0.5) / (policy_ms * 1e-3) / 1e12 / tensor_peak,
                "frac_executed": flops_exec_launch * (T + 0.5) / (policy_ms * 1e-3) / 1e12 / tensor_peak,
                "executed_obstacle_slots": {"actor_visible_mean": o_vis, "critic_boundary_mean": o_b, "survey_upper_bound": env.O},
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (dense bf16 = the kind::f16 rate; the split issues 3 MMAs "
                               "per algorithmic product, so this kernel's ceiling is frac = 1/3)",
                "algorithmic_flops_per_launch": flops_launch, "flops_per_agent_per_network": flops_pp,
                "gemm_flops_per_agent_per_network": gemm_f,
                "single_pipeline_avg_launch_us": pk["avg_us"], "pipelined": pipe,
                "hbm_bytes_per_launch_algorithmic": bytes_launch,
                "hbm_GBps_at_this_duration": bytes_launch * (T + 0.5) / (policy_ms * 1e-3) / 1e9, "hbm_peak_GBps": hbm_peak,
                "note": "SURVEY 8(d) FLOP count per agent and network (obstacle messages counted for all O slots: upper bound; "
                        "frac_executed counts the slots really evaluated, frac_gemm_only the dense layers only) x B*N rows x 2 networks"}

    if rank == 0:
        # ---- CPU baseline: oracle port (C env + torch-CPU network restatement) on the host cores, bounded sample ----
        cpu, _ = cpu_policy_baseline(cfg, wl, steps_T=T, budget_s=12.0)
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 env / f32 networks", "data": "synthetic", "config": workload_config(world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": pol.our_launches * args.steps, "clocks": clocks, "roofline": roofline,
            "cpu_baseline": cpu, "env_only": env_only, "train": train, "per_rank_ms": per_rank_ms,
            "kernel_ms_per_episode": kernel_table}))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last timed episode's rollout batch (a fixed sample of envs) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
