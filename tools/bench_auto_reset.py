"""Rollout time of auto-reset segment streams at the bench shape (4096 envs x 8 pursuers, T_ep 150, depth 1, eager).  Every arm
collects the same 32 episodes (4800 env steps, 32 device resets, the last one after the final episode) as
  * "S50_host_reset": segments of 50 steps (divisors of the episode), the envs reset by the caller after every third segment,
  * "S50_auto": the same segments with auto_reset (the reset inside the rollout, at the end of every third segment),
  * "S64_auto": 75 segments of 64 steps with auto_reset (the boundary inside the segment, except after the last episode),
  * "S64_auto_device_tape": the same with the target tape drawn on the device (AutoReset(tape="device")), still eager,
  * "S50_auto_graph" / "S64_auto_graph": the device-tape streams of 50 / 64 steps replayed from CUDA graphs (MAPPO.explore_batched).
32 episodes are the fewest whose length is a multiple of 64, so the arms do the same env steps and the same resets.  The arms alternate,
each from the same env state, for --reps rounds after one warm-up round of two episodes each; before that, each graph arm runs one full
cycle of its segment starts (3 for S = 50, 75 for S = 64), which captures its graphs.  Reports the rollout milliseconds per 150 env steps
(host clock around work that ends in a device synchronise, resets included), the wall time of that first cycle (captures included), the
device memory (max_memory_allocated since the arm started, memory_reserved) after the eager S = 64 stream's warm-up and after the S = 64
graph cycle, and the GPU's name and power limit read in the same run.

    python tools/bench_auto_reset.py [--reps 3] [--out profiles/r7_auto_reset_bench_shape.json]"""
import argparse
import json
import math
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_segments import gpu_info  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200 import default_config  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO, AutoReset, RolloutCarry  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena  # noqa: E402

EPISODES = 32


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--pursuers", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, N, T = args.envs, args.pursuers, 150
    cfg = default_config(env__num_defender=N, env__max_steps=T, algo__depth=1, algo__learner_device=str(dev), algo__worker_device=str(dev))
    env = BatchedPursuitEnv(cfg, B, device=dev, num_maps=32)
    wf0 = {k: getattr(env, k).clone() for k in ("wf_n", "wf_mean", "wf_S", "wf_std")}
    torch.manual_seed(0)
    mappo = MAPPO(cfg, B, max(1, round(B / 10)), "Learner")
    arenas = {S: RolloutArena(env.params, B, S, dev) for S in (50, 64)}
    auto = AutoReset(reset_seed=lambda e: 1000 + e, sample_seed=lambda e: e)
    auto_dev = AutoReset(reset_seed=auto.reset_seed, sample_seed=auto.sample_seed, tape="device")

    def run(arm, episodes=None, calls=None):
        """`episodes` episodes (or `calls` segments) of `arm`; returns (seconds, env steps, rollout calls, resets)."""
        a = auto_dev if "device_tape" in arm or "graph" in arm else auto
        env.restore(wf0)
        env.reset_device(seed=a.reset_seed(0), tape_len=a.tape_len, tape=a.tape)
        carry = RolloutCarry.zeros(mappo, B, N)
        S = 64 if arm.startswith("S64") else 50
        calls = calls or episodes * T // S
        resets = 0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(calls):
            if arm == "S50_host_reset":
                e, seg = divmod(i, T // S)
                tb = mappo.rollout_batched(env, arenas[S], S, seed=auto.sample_seed(e), carry=carry)
                carry = tb.carry
                if seg == T // S - 1:
                    env.reset_device(seed=auto.reset_seed(e + 1), tape_len=auto.tape_len)
                    carry = RolloutCarry.zeros(mappo, B, N)
                    resets += 1
            elif "graph" in arm:
                tb = mappo.explore_batched(env, arenas[S], S, carry=carry, auto_reset=a)
                carry = tb.carry
                resets += tb.ended_collision is not None
            else:
                tb = mappo.rollout_batched(env, arenas[S], S, carry=carry, auto_reset=a)
                carry = tb.carry
                resets += tb.ended_collision is not None
            del tb
        torch.cuda.synchronize()
        return time.perf_counter() - t0, calls * S, calls, resets

    arms = ("S50_host_reset", "S50_auto", "S64_auto", "S64_auto_device_tape", "S50_auto_graph", "S64_auto_graph")
    gb = lambda x: round(x / 1e9, 3)                        # noqa: E731
    memory = {}
    for arm in arms[:4]:                                    # warm-up of the eager arms
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        run(arm, 2)
        if arm == "S64_auto_device_tape":
            memory["eager_S64"] = {"max_allocated_GB": gb(torch.cuda.max_memory_allocated(dev)),
                                   "reserved_GB": gb(torch.cuda.memory_reserved(dev))}
    capture = {}
    # one full cycle of segment starts captures every graph of a stream; S = 64 first, so that its memory holds no other graph stream
    for arm in ("S64_auto_graph", "S50_auto_graph"):
        S = 64 if arm.startswith("S64") else 50
        cycle = T // math.gcd(S, T)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        s, steps, calls, _ = run(arm, calls=cycle)
        capture[arm] = {"starts": cycle, "first_cycle_s": round(s, 3), "env_steps": steps}
        if S == 64:
            memory["graph_S64_cycle"] = {"graphs": cycle, "max_allocated_GB": gb(torch.cuda.max_memory_allocated(dev)),
                                         "reserved_GB": gb(torch.cuda.memory_reserved(dev))}
        run(arm, 2)
    rounds = {a: [] for a in arms}
    for _ in range(args.reps):
        for arm in arms:
            s, steps, calls, resets = run(arm, EPISODES)
            rounds[arm].append({"ms_per_150_steps": 1e3 * s * T / steps, "env_steps": steps, "rollout_calls": calls, "resets": resets})
    med = {a: sorted(r["ms_per_150_steps"] for r in rounds[a])[len(rounds[a]) // 2] for a in arms}
    out = {"shape": {"envs": B, "pursuers": N, "steps": T, "depth": 1, "episodes": EPISODES, "history": mappo.history_mode(64, B, N)},
           "rounds": rounds, "median_ms_per_150_steps": med, "graph_capture": capture, "memory": memory, "gpu": gpu_info(),
           "note": "rollout only (no training); every arm collects the same episodes with the same number of resets; arms alternate "
                   "from the same env state after one warm-up round each; first_cycle_s is the wall time of the first cycle of segment "
                   "starts, every capture (eager warm-up segment + capture) and replay included; memory is device memory of the whole "
                   "process (engine, networks, both arenas, earlier arms' cached blocks in reserved)"}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
