"""One training iteration at configs[4]'s per-GPU shape (conf/*.yaml: 64 pursuers, 32 768 envs, T 250, O 110, 60x60 map, depth 3) on
one GPU: device reset -> rollout_batched (history replay: the stored history would take 543 GB) -> one train epoch -> update.

    python tools/train_large.py [--envs 32768] [--mini-batch 32] [--out profiles/r3_train_configs4.json]

mini_batch_size: the reference's B/10 would be 3 277 envs = 52 M rows per minibatch, ~27 GB per 128-wide activation.  The default
is 32 envs = 512 K rows (0.26 GB per 128-wide activation; a minibatch keeps a few dozen of them for the backward pass, and
CONCURRENT_MINIBATCHES = 3 are in flight), next to the 30 GB arena and the D+1-slab history ring.

Prints one JSON line: per-phase wall times (reset, rollout, a replay-only pass over the epoch's minibatches, the epoch, the update),
torch.cuda.max_memory_allocated, agent-env-steps/s of the rollout, training samples/s of the epoch, and the GPU's name and power
limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from distributed_multi_agent_reinforcement_learning_b200 import default_config, mappo_parallel  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO, history_bytes  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        name, power = (s.strip() for s in out.split(",", 1))
        return {"name": name, "power_limit": power}
    except Exception as e:                                  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def replay_pass(tb, mbs):
    """Regenerates every minibatch's history the way `train` does (minibatch m on stream pair m % CONCURRENT_MINIBATCHES)."""
    P = mappo_parallel.CONCURRENT_MINIBATCHES
    streams = [torch.cuda.Stream() for _ in range(P)]
    main = torch.cuda.current_stream()
    for m, lo in enumerate(range(0, tb.B, mbs)):
        st = streams[m % P]
        st.wait_stream(main)
        with torch.cuda.stream(st):
            mb = tb.minibatch(lo, min(lo + mbs, tb.B))
            del mb
    for st in streams:
        main.wait_stream(st)


def progress(msg):
    print(f"[train_large] {msg}", file=sys.stderr, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=32768)
    ap.add_argument("--pursuers", type=int, default=64)
    ap.add_argument("--steps", type=int, default=250)
    ap.add_argument("--depth", type=int, default=3)
    ap.add_argument("--maps", type=int, default=64)
    ap.add_argument("--mini-batch", type=int, default=32)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, N, T, D, mbs = args.envs, args.pursuers, args.steps, args.depth, args.mini_batch
    cfg = default_config(env__num_defender=N, env__max_steps=T, algo__depth=D, map__map_size=[60, 60], map__num_max_obstacle=110,
                         algo__learner_device=str(dev), algo__worker_device=str(dev))
    env = BatchedPursuitEnv(cfg, B, device=dev, num_maps=args.maps)
    arena = RolloutArena(env.params, B, T, dev)
    torch.manual_seed(0)
    mappo = MAPPO(cfg, B, mbs, "Learner")
    mode = mappo.history_mode(T, B, N)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    env.reset_device(seed=1, tape_len=32)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    progress(f"reset {t1 - t0:.2f} s; history mode {mode}")
    tb = mappo.rollout_batched(env, arena, T, seed=1)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    assert int(env.evader_status.max()) == 0, "evader search overflow / target tape exhausted"
    peak_rollout = torch.cuda.max_memory_allocated()
    progress(f"rollout {t2 - t1:.2f} s, peak {peak_rollout / 1e9:.1f} GB")
    replay_s = None
    if tb.replay is not None:
        replay_pass(tb, mbs)
        torch.cuda.synchronize()
        replay_s = time.perf_counter() - t2
        progress(f"replay pass {replay_s:.2f} s")
    t3 = time.perf_counter()
    obj_c, obj_a, _, _ = mappo.train(tb, B * T * N, return_numpy=False)
    torch.cuda.synchronize()
    t4 = time.perf_counter()
    progress(f"epoch {t4 - t3:.2f} s")
    mappo.update(B * T * N)
    torch.cuda.synchronize()
    t5 = time.perf_counter()
    rows = B * N * T
    out = {
        "shape": {"envs": B, "pursuers": N, "steps": T, "depth": D, "obstacle_slots": env.O, "map": "60x60", "maps": args.maps,
                  "mini_batch_size": mbs, "minibatches": -(-B // mbs), "concurrent_minibatches": mappo_parallel.CONCURRENT_MINIBATCHES},
        "history": mode, "history_bytes_if_stored": history_bytes(T, B, N, mappo.embedding_dim, D),
        "arena_bytes": arena.nbytes(), "reset_fail_envs": int((env.reset_fail != 0).sum()),
        "s": {"reset": t1 - t0, "rollout": t2 - t1, "replay_pass": replay_s, "epoch": t4 - t3, "update": t5 - t4},
        "replay_share_of_epoch": None if replay_s is None else replay_s / (t4 - t3),
        "max_memory_allocated": torch.cuda.max_memory_allocated(), "max_memory_allocated_rollout": peak_rollout,
        "agent_env_steps_per_s": rows / (t2 - t1), "train_samples_per_s": rows / (t4 - t3),
        "losses": {"critic": obj_c, "actor": obj_a},
        "gpu": gpu_info(),
        "note": "wall times of one iteration after a fresh process start (first launches included); replay_pass is a separate "
                "replay-only pass over the epoch's minibatches on the epoch's stream layout, before the epoch (which replays again)",
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
