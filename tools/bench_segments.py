"""Whole-episode vs segmented rollouts at the bench shape (4096 envs x 8 pursuers, T 150, depth 1): per episode, either one rollout of
150 steps and one epoch on it, or three segments of 50 steps (rollout_batched with a RolloutCarry) with one epoch on each.  The two
arms alternate, each from the same env state, for --reps rounds.

    python tools/bench_segments.py [--segment 50] [--reps 3] [--out profiles/r6_segments_bench_shape.json]

Prints one JSON line: per arm and round the rollout time per episode (sum over its segments), the epoch time per segment, the peak
allocation of the round (torch.cuda.max_memory_allocated, reset before each round), the history mode, and the GPU's name and power
limit read in the same run.  Times are host clocks around work that ends in a device synchronise."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from distributed_multi_agent_reinforcement_learning_b200 import default_config  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO, RolloutCarry  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        name, power = (s.strip() for s in out.split(",", 1))
        return {"name": name, "power_limit": power}
    except Exception as e:                                  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--pursuers", type=int, default=8)
    ap.add_argument("--steps", type=int, default=150)
    ap.add_argument("--segment", type=int, default=50)
    ap.add_argument("--depth", type=int, default=1)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.segment < 1 or args.steps % args.segment:
        ap.error("--segment must be a positive divisor of --steps")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, N, T, S = args.envs, args.pursuers, args.steps, args.segment
    cfg = default_config(env__num_defender=N, env__max_steps=T, algo__depth=args.depth, algo__learner_device=str(dev),
                         algo__worker_device=str(dev))
    env = BatchedPursuitEnv(cfg, B, device=dev, num_maps=32)
    env.reset_device(seed=1)
    snap = env.snapshot()
    torch.manual_seed(0)
    mappo = MAPPO(cfg, B, max(1, round(B / 10)), "Learner")
    arenas = {T: RolloutArena(env.params, B, T, dev), S: RolloutArena(env.params, B, S, dev)}

    def run(seg):
        """One episode as T / seg segments (seg = T: the whole episode, carry=None); returns rollout seconds and epoch seconds per segment."""
        env.restore(snap)
        carry = None if seg == T else RolloutCarry.zeros(mappo, B, N)
        roll, epochs, modes = 0.0, [], set()
        for k in range(T // seg):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            tb = mappo.rollout_batched(env, arenas[seg], seg, seed=3, carry=carry)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            mappo.train(tb, B * N * seg * (k + 1), return_numpy=False)     # gradients only: the weights stay those of the first round
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            roll += t1 - t0
            epochs.append(t2 - t1)
            modes.add("replay" if tb.replay is not None else "store")
            carry = tb.carry
            del tb
        return roll, epochs, sorted(modes)

    run(T)                                                  # warm-up of both shapes
    run(S)
    rounds = {str(T): [], str(S): []}
    for _ in range(args.reps):
        for seg in (T, S):
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            roll, epochs, modes = run(seg)
            rounds[str(seg)].append({"rollout_s_per_episode": roll, "epoch_s_per_segment": epochs,
                                     "max_memory_allocated": torch.cuda.max_memory_allocated(), "history": modes})
    out = {"shape": {"envs": B, "pursuers": N, "steps": T, "segment": S, "depth": args.depth,
                     "mini_batch_size": mappo.mini_batch_size},
           "arena_bytes": {str(T): arenas[T].nbytes(), str(S): arenas[S].nbytes()},
           "rounds": rounds, "gpu": gpu_info(),
           "note": "arms alternate (whole episode, then segments) from the same env state; the first round of each is a separate "
                   "warm-up; train() computes gradients without an optimizer step, so every round uses the same weights"}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
