"""Cost of the PPO diagnostics (MAPPO.train(stats=True)) at the bench shape: 4096 envs x 8 pursuers, T 150, depth 1, stored history.
One rollout, then --reps rounds of one epoch with stats off and one with stats on, alternating (train() computes gradients without an
optimizer step, so every epoch sees the same weights and batch); the medians of both arms.  Then marl_ppo_stats on its own, timed with
CUDA events over --kernel-reps launches: once on all 4.9 M rows of the update and once per minibatch (the shape train() launches).

    python tools/bench_train_stats.py [--reps 7] [--out profiles/r9_train_stats_bench_shape.json]

Prints one JSON line, with the GPU's name and power limit read in the same run.  Epoch times are host clocks around work that ends in a
device synchronise."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from distributed_multi_agent_reinforcement_learning_b200 import default_config, mappo_parallel, policy_ops as ops  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        name, power = (s.strip() for s in out.split(",", 1))
        return {"name": name, "power_limit": power}
    except Exception as e:                                  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def time_kernel(args_list, reps):
    """Mean device time (s) of one round of marl_ppo_stats calls (one per entry of args_list), over `reps` rounds."""
    for a in args_list:
        ops.ppo_stats(*a)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(reps):
        for a in args_list:
            ops.ppo_stats(*a)
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--pursuers", type=int, default=8)
    ap.add_argument("--steps", type=int, default=150)
    ap.add_argument("--depth", type=int, default=1)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--kernel-reps", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, N, T = args.envs, args.pursuers, args.steps
    cfg = default_config(env__num_defender=N, env__max_steps=T, algo__depth=args.depth, algo__learner_device=str(dev),
                         algo__worker_device=str(dev))
    env = BatchedPursuitEnv(cfg, B, device=dev, num_maps=32)
    env.reset_device(seed=1)
    torch.manual_seed(0)
    mappo = MAPPO(cfg, B, max(1, round(B / 10)), "Learner")
    arena = RolloutArena(env.params, B, T, dev)
    mappo_parallel.STORE_HISTORY_SHARE = 1.0                # the stored history, as the issue's shape asks
    tb = mappo.rollout_batched(env, arena, T, seed=3)
    torch.cuda.synchronize()
    history = "replay" if tb.replay is not None else "store"

    def epoch(stats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mappo.train(tb, B * N * T, return_numpy=False, stats=stats)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    epoch(False)                                            # warm-up of both arms
    epoch(True)
    off, on = [], []
    for _ in range(args.reps):
        off.append(epoch(False))
        on.append(epoch(True))
    s = mappo.last_train_stats

    # the kernel alone on the batch's own rows: all of them in one call, and one call per minibatch as train() does
    R = T * B * N
    g = torch.Generator(device=dev).manual_seed(0)
    f = lambda: torch.randn(R, device=dev, generator=g)     # noqa: E731
    logp, old, ent, val, v_old, vt = (f() for _ in range(6))
    logp = old + 0.05 * logp
    active = (torch.rand(R, device=dev, generator=g) < 0.9).float()
    eps = mappo.epsilon
    whole = [(logp, old, ent, val, v_old, vt, active, eps)]
    mbs = mappo.mini_batch_size * T * N
    per_mb = [tuple(x[lo:lo + mbs] for x in (logp, old, ent, val, v_old, vt, active)) + (eps,) for lo in range(0, R, mbs)]
    t_whole = time_kernel(whole, args.kernel_reps)
    t_mb = time_kernel(per_mb, args.kernel_reps)
    nbytes = 7 * 4 * R
    med_off, med_on = statistics.median(off), statistics.median(on)
    out = {"shape": {"envs": B, "pursuers": N, "steps": T, "depth": args.depth, "mini_batch_size": mappo.mini_batch_size,
                     "minibatches": -(-B // mappo.mini_batch_size), "rows": R},
           "history": history,
           "epoch_s": {"stats_off": off, "stats_on": on, "median_off": med_off, "median_on": med_on,
                       "median_delta_s": med_on - med_off, "median_delta_pct": 100.0 * (med_on - med_off) / med_off},
           "kernel": {"bytes_read": nbytes, "one_call_all_rows_s": t_whole, "one_call_all_rows_GBps": nbytes / t_whole / 1e9,
                      "calls_per_minibatch": len(per_mb), "per_minibatch_calls_total_s": t_mb,
                      "per_minibatch_calls_GBps": nbytes / t_mb / 1e9},
           "last_stats": {k: v for k, v in s.as_dict().items()},
           "gpu": gpu_info(),
           "note": "arms alternate (stats off, then on) on the same batch and weights after one warm-up epoch of each; kernel times are "
                   "CUDA events over --kernel-reps rounds on synthetic rows of the update's size (7 fp32 arrays, larger than the L2)"}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
