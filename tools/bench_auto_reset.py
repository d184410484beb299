"""Rollout time of auto-reset segment streams at the bench shape (4096 envs x 8 pursuers, T_ep 150, depth 1, eager).  Every arm
collects the same 32 episodes (4800 env steps, 32 device resets, the last one after the final episode) as
  * "S50_host_reset": segments of 50 steps (divisors of the episode), the envs reset by the caller after every third segment,
  * "S50_auto": the same segments with auto_reset (the reset inside the rollout, at the end of every third segment),
  * "S64_auto": 75 segments of 64 steps with auto_reset (the boundary inside the segment, except after the last episode),
  * "S64_auto_device_tape": the same with the target tape drawn on the device (AutoReset(tape="device")), still eager,
  * "S50_auto_graph" / "S64_auto_graph": the device-tape streams of 50 / 64 steps replayed from CUDA graphs (MAPPO.explore_batched),
  * "S64_auto_pool" / "S64_auto_graph_pool": the S = 64 device-tape streams, eager and from graphs, on a second engine that holds a map
    pool of --pool-maps maps (generated on the device, installed with MapPool.install): every reset keeps the pool and draws each env's
    map from it (AutoReset(maps="draw")) instead of generating 32 new maps and their sensor tables.
32 episodes are the fewest whose length is a multiple of 64, so the arms do the same env steps and the same resets.  The arms alternate,
each from the same env state, for --reps rounds after one warm-up round of two episodes each; before that, each graph arm runs one full
cycle of its segment starts (3 for S = 50, 75 for S = 64), which captures its graphs.  Reports the rollout milliseconds per 150 env steps
(host clock around work that ends in a device synchronise, resets included), the wall time of that first cycle (captures included), the
device memory (max_memory_allocated since the arm started, memory_reserved) after the eager S = 64 stream's warm-up and after the S = 64
graph cycle, and the GPU's name and power limit read in the same run.

For the pool it also reports: `reset_device` alone at the bench's env count, timed with CUDA events (median of --reset-reps calls per
mode, the modes alternating, device tape in all): "generate" with one map per env (M = envs) against "draw" and "keep" on the pool; the
wall time of MapPool.install(verify=True) of the whole pool (host-side verification included); the peak device memory after the pool's
graph cycle; and the size of a training-state file (checkpoint.save_training_state) of the pool engine, which holds all M maps' tables.

    python tools/bench_auto_reset.py [--reps 3] [--pool-maps 2000] [--out profiles/r8_map_pool_bench_shape.json]"""
import argparse
import json
import math
import os
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_segments import gpu_info  # noqa: E402
from make_map_pool import make_pool  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200 import default_config  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.checkpoint import save_training_state  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO, AutoReset, RolloutCarry  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena  # noqa: E402

EPISODES = 32


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--pursuers", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--pool-maps", type=int, default=2000)
    ap.add_argument("--reset-reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, N, T = args.envs, args.pursuers, 150
    cfg = default_config(env__num_defender=N, env__max_steps=T, algo__depth=1, algo__learner_device=str(dev), algo__worker_device=str(dev))
    env_gen = BatchedPursuitEnv(cfg, B, device=dev, num_maps=32)
    wf0 = {k: getattr(env_gen, k).clone() for k in ("wf_n", "wf_mean", "wf_S", "wf_std")}
    torch.manual_seed(0)
    mappo = MAPPO(cfg, B, max(1, round(B / 10)), "Learner")
    arenas = {S: RolloutArena(env_gen.params, B, S, dev) for S in (50, 64)}
    auto = AutoReset(reset_seed=lambda e: 1000 + e, sample_seed=lambda e: e)
    auto_dev = AutoReset(reset_seed=auto.reset_seed, sample_seed=auto.sample_seed, tape="device")
    auto_pool = AutoReset(reset_seed=auto.reset_seed, sample_seed=auto.sample_seed, tape="device", maps="draw")
    gb = lambda x: round(x / 1e9, 3)                        # noqa: E731
    t_make = time.perf_counter()
    pool = make_pool(cfg, args.pool_maps, seed=7, device=dev)
    t_make = time.perf_counter() - t_make
    pool_env = BatchedPursuitEnv(cfg, B, device=dev, num_maps=args.pool_maps)
    t_inst = time.perf_counter()
    pool.install(pool_env, verify=True)
    t_inst = time.perf_counter() - t_inst
    table_bytes = sum(getattr(pool_env, k).numel() * getattr(pool_env, k).element_size()
                      for k in ("grid_bits", "inflated_bits", "boundary_bits", "boundary_count", "boundary_xy", "raser_bits"))
    pool_info = {"maps": args.pool_maps, "generate_on_device_s": round(t_make, 3), "install_verify_s": round(t_inst, 3),
                 "device_table_MB": round(table_bytes / 1e6, 1)}
    del pool

    def run(arm, episodes=None, calls=None):
        """`episodes` episodes (or `calls` segments) of `arm`; returns (seconds, env steps, rollout calls, resets)."""
        a = auto_pool if "pool" in arm else auto_dev if "device_tape" in arm or "graph" in arm else auto
        env = pool_env if "pool" in arm else env_gen
        env.restore(wf0)
        env.reset_device(seed=a.reset_seed(0), tape_len=a.tape_len, tape=a.tape, maps=a.maps)
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

    arms = ("S50_host_reset", "S50_auto", "S64_auto", "S64_auto_device_tape", "S50_auto_graph", "S64_auto_graph", "S64_auto_pool",
            "S64_auto_graph_pool")
    memory = {}
    for arm in arms[:4] + ("S64_auto_pool",):               # warm-up of the eager arms
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        run(arm, 2)
        if arm == "S64_auto_device_tape":
            memory["eager_S64"] = {"max_allocated_GB": gb(torch.cuda.max_memory_allocated(dev)),
                                   "reserved_GB": gb(torch.cuda.memory_reserved(dev))}
    capture = {}
    # one full cycle of segment starts captures every graph of a stream; S = 64 first, so that its memory holds no other graph stream
    for arm in ("S64_auto_graph", "S50_auto_graph", "S64_auto_graph_pool"):
        S = 64 if arm.startswith("S64") else 50
        cycle = T // math.gcd(S, T)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        s, steps, calls, _ = run(arm, calls=cycle)
        capture[arm] = {"starts": cycle, "first_cycle_s": round(s, 3), "env_steps": steps}
        if S == 64:
            memory["graph_S64_cycle" + ("_pool" if "pool" in arm else "")] = {
                "graphs": cycle, "max_allocated_GB": gb(torch.cuda.max_memory_allocated(dev)), "reserved_GB": gb(torch.cuda.memory_reserved(dev))}
        run(arm, 2)
    reset_ms = time_resets(cfg, B, pool_env, args.reset_reps, dev)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "training_state.pt")
        save_training_state(path, mappo, pool_env)
        pool_info["training_state_file_MB"] = round(os.path.getsize(path) / 1e6, 1)
    rounds = {a: [] for a in arms}
    for _ in range(args.reps):
        for arm in arms:
            s, steps, calls, resets = run(arm, EPISODES)
            rounds[arm].append({"ms_per_150_steps": 1e3 * s * T / steps, "env_steps": steps, "rollout_calls": calls, "resets": resets})
    med = {a: sorted(r["ms_per_150_steps"] for r in rounds[a])[len(rounds[a]) // 2] for a in arms}
    out = {"shape": {"envs": B, "pursuers": N, "steps": T, "depth": 1, "episodes": EPISODES, "history": mappo.history_mode(64, B, N)},
           "rounds": rounds, "median_ms_per_150_steps": med, "graph_capture": capture, "memory": memory, "pool": pool_info,
           "reset_device_ms": reset_ms, "gpu": gpu_info(),
           "note": "rollout only (no training); every arm collects the same episodes with the same number of resets; arms alternate "
                   "from the same env state after one warm-up round each; first_cycle_s is the wall time of the first cycle of segment "
                   "starts, every capture (eager warm-up segment + capture) and replay included; memory is device memory of the whole "
                   "process (engine, networks, both arenas, earlier arms' cached blocks in reserved); the pool arms run on a second "
                   "engine (same envs, --pool-maps maps); reset_device_ms: CUDA events around one reset_device call (device tape), "
                   "median and min over reset_reps calls per mode"}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


def time_resets(cfg, B, pool_env, reps, dev):
    """reset_device alone: "generate" on an engine with one map per env against "draw" / "keep" on the pool engine, CUDA events around
    each call, the modes alternating after two warm-up calls each."""
    gen_env = BatchedPursuitEnv(cfg, B, device=dev, num_maps=B)
    modes = {"generate_M%d" % B: (gen_env, "generate"), "draw_M%d" % pool_env.M: (pool_env, "draw"),
             "keep_M%d" % pool_env.M: (pool_env, "keep")}
    times = {k: [] for k in modes}
    for i in range(reps + 2):
        for k, (e, mode) in modes.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            e.reset_device(seed=5000 + i, tape_len=16, tape="device", maps=mode)
            b.record()
            torch.cuda.synchronize()
            assert int(e.reset_fail.sum()) == 0, k
            if i >= 2:
                times[k].append(a.elapsed_time(b))
    del gen_env
    return {k: {"median": round(sorted(v)[len(v) // 2], 4), "min": round(min(v), 4), "calls": len(v)} for k, v in times.items()}


if __name__ == "__main__":
    main()
