"""Episode time of the bench workload (graph-captured pipelined rollout) for a few env-group pipeline counts.
usage: python tools/sweep_pipelines.py [G ...]   (default 1 4 8)"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ab  # noqa: E402,F401  (MARL_AB_LIB=<alternative libmarl_b200.so> for A/B runs)
import bench  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO, RolloutGraph  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena  # noqa: E402


def main():
    cfg = bench.make_cfg()
    B, N, T, M = bench.B_PER_GPU, bench.N_AGENTS, bench.T_STEPS, bench.N_MAPS
    wl = bench.host_workload(cfg, B, M, seed=0xB200 + 1)
    env = BatchedPursuitEnv(cfg, B, num_maps=M)
    env.set_maps(wl["grids"], wl["inflated"])
    env.set_state(wl["p_state"], wl["e_state"], wl["target"], wl["map_id"], time_step=0)
    env.set_target_tape(wl["tape"])
    env.start_episode()
    arena = RolloutArena(env.params, B, T, env.device)
    snap = env.snapshot()
    torch.manual_seed(0xB200)
    mappo = MAPPO(cfg, B, max(1, round(B / 10)), "Learner")
    for pipes in [int(a) for a in sys.argv[1:]] or [1, 4, 8]:
        os.environ["MARL_PIPELINES"] = str(pipes)
        env.restore(snap)
        g = RolloutGraph(mappo, env, arena, T, 0xB200)
        ts = []
        for _ in range(6):
            env.restore(snap)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            g.replay()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        print(f"pipelines {pipes}: {min(ts[1:]):.2f} ms per episode (median {sorted(ts[1:])[2]:.2f})", flush=True)
        del g


if __name__ == "__main__":
    main()
