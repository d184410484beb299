"""The A* replanning launch of one env group (1024 envs) and of the whole batch at the bench shape, on mid-episode states: event
timings here, and the launch to capture under ncu:

    python tools/profile_evader.py [--map-size W H] [--envs B]
    ncu --set full --import-source on --clock-control none -k regex:evader_kernel -s 3 -c 1 -o gpurun_out/evader python tools/profile_evader.py

The states come from 40 closed-loop env steps with scripted random actions (env time_step 40: a replan is due).  --map-size runs the
same on another map (blocks centred on it; 60 55 is the bench map), e.g. 128 128 for the two-word column search.  The last line is
JSON: the whole-batch launch's event times (min and median of --reps), the map, the library and the GPU's name and power limit."""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ab  # noqa: E402,F401  (MARL_AB_LIB)
import bench  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200 import _lib  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena  # noqa: E402
from train_large import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--map-size", type=int, nargs=2, default=None, metavar=("W", "H"))
    ap.add_argument("--envs", type=int, default=bench.B_PER_GPU)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    cfg = bench.make_cfg()
    if args.map_size:
        cfg.map.map_size = list(args.map_size)
        cfg.map.center = [args.map_size[0] // 2, args.map_size[1] // 2]
    B, M, T = args.envs, bench.N_MAPS, bench.T_STEPS
    wl = bench.host_workload(cfg, B, M, seed=0xB200 + 1 + 7919 * int(os.environ.get("EVADER_RANK", "0")))      # bench.py's per-rank workload
    env = BatchedPursuitEnv(cfg, B, device=dev, num_maps=M)
    env.set_maps(wl["grids"], wl["inflated"])
    env.set_state(wl["p_state"], wl["e_state"], wl["target"], wl["map_id"], time_step=0)
    env.set_target_tape(wl["tape"])
    env.start_episode()
    arena = RolloutArena(env.params, B, T, dev)
    K = int(os.environ.get("EVADER_T0", "40"))
    env.rollout_closed(arena, K, seed=7)
    torch.cuda.synchronize()
    assert int(env.time_step[0]) == K
    G = min(B, int(os.environ.get("EVADER_GROUP", "1024")))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for lo, hi, name in ((0, G, f"group of {G}"), (0, B, f"all {B}")):
        ts = []
        for _ in range(args.reps):
            ev[0].record()
            env.evader_replan(lo, hi)
            ev[1].record()
            torch.cuda.synchronize()
            ts.append(ev[0].elapsed_time(ev[1]) * 1e3)
        print(f"replan {name}: {min(ts):.1f} us (min of {len(ts)}), path_len mean {float(env.path_len[lo:hi].float().mean()):.2f}, "
              f"status {int(env.evader_status.max())}")
    assert int(env.evader_status.max()) == 0
    W, H = cfg.map.map_size
    print(json.dumps({"replan_all_envs_us": {"min": min(ts), "median": statistics.median(ts), "reps": len(ts)}, "envs": B,
                      "pursuers": env.N, "map": f"{W}x{H}", "maps": M, "time_step": K,
                      "path_len_mean": float(env.path_len.float().mean()), "lib": os.path.relpath(_lib.LIB_PATH, ROOT),
                      "gpu": gpu_info()}))


if __name__ == "__main__":
    main()
