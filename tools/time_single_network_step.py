"""Times the fused policy step's single-network launches and the evaluator's episode:
  - the critic-only bootstrap launch at the bench's env-group shape (1024 envs x 8 agents, tile_rows 128);
  - an actor-only launch at 4096 x 8 (whole bench batch) and at the evaluator's 16 x 8;
  - Evaluator.get_rewards_and_step end to end (16 envs, T = 150).
Kernel times are CUDA events around --launches back-to-back launches (after a warm-up), in ms per launch; the evaluator episode is a
host clock around work that ends in a device synchronise.  MARL_AB_LIB=<libmarl_b200.so> times another build (tools/ab.py), so two
builds can be compared by alternating runs:

    for i in 1 2 3 4; do for lib in base.so new.so; do MARL_AB_LIB=$lib python tools/time_single_network_step.py; done; done

Prints one JSON line, with the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import ab  # noqa: E402,F401  (MARL_AB_LIB)
import bench  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200 import _lib  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.evaluator import Evaluator  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.fused_policy import FusedRolloutStep  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv  # noqa: E402

E = 128


def gpu_info():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, timeout=30).stdout.strip()
    name, power = (s.strip() for s in out.split(",", 1))
    return {"name": name, "power_limit": power}


def launch_ms(fn, launches, warmup=20):
    for _ in range(warmup):
        fn()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for _ in range(launches):
        fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) / launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=500)
    ap.add_argument("--episodes", type=int, default=10)
    args = ap.parse_args()
    cfg = bench.make_cfg()
    N = bench.N_AGENTS
    torch.manual_seed(0)
    m = MAPPO(cfg, bench.B_PER_GPU, bench.B_PER_GPU // 10, "Learner")
    w_eff, _ = m.critic.head_weight(update_buffers=False)
    fused = FusedRolloutStep(m, w_eff.reshape(E).contiguous())
    res = {}
    for name, B, nets, tile in (("critic_only_1024x8_tile128_ms", 1024, ("critic",), 128), ("actor_only_4096x8_ms", 4096, ("actor",), 0),
                                ("actor_only_16x8_ms", 16, ("actor",), 0)):
        wl = bench.host_workload(cfg, B, 32, seed=1)
        env = BatchedPursuitEnv(cfg, B, num_maps=32)
        env.set_maps(wl["grids"], wl["inflated"])
        env.set_state(wl["p_state"], wl["e_state"], wl["target"], wl["map_id"], time_step=0)
        env.set_target_tape(wl["tape"])
        env.start_episode()
        env.observe()
        oxy, oc = env.boundary_xy.contiguous(), torch.clamp(env.boundary_count, max=env.O).contiguous()
        hist = [0.1 * torch.randn(B, N, E, device=env.device)]
        emb = torch.empty(B, N, E, device=env.device)
        h = torch.zeros(2, B * N, E, device=env.device)
        act, logp, val = (torch.zeros(B, N, dtype=torch.int32, device=env.device), torch.empty(B, N, device=env.device),
                          torch.empty(B, N, device=env.device))
        if nets == ("critic",):
            fn = lambda: fused.step(env, oxy, oc, 3, 1, False, hist, hist, None, emb, None, h, None, None, val, nets=nets, tile_rows=tile)  # noqa: E731
        else:
            fn = lambda: fused.step(env, oxy, oc, 3, 1, True, hist, hist, emb, None, h, None, act, logp, None, nets=nets, tile_rows=tile)  # noqa: E731
        res[name] = launch_ms(fn, args.launches)
    torch.manual_seed(3)
    ev = Evaluator(cfg, 16, MAPPO(cfg, None, None, "Evaluator"), seed=3)
    ev.get_rewards_and_step()                                   # warm-up: env, arena, kernel attributes
    ts = []
    for _ in range(args.episodes):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ev.get_rewards_and_step()
        torch.cuda.synchronize()
        ts.append(1e3 * (time.perf_counter() - t0))
    res["evaluator_16x8_T150_ms"] = sorted(ts)[len(ts) // 2]
    res["evaluator_episode_ms_all"] = [round(t, 3) for t in ts]
    print(json.dumps({"lib": _lib.LIB_PATH, **res, "gpu": gpu_info()}))


if __name__ == "__main__":
    main()
