"""History replay at the bench shape (4096 envs x 8 pursuers, T 150, depth 1, minibatch round(B/10)): the cost of regenerating the
epoch's history against the epoch, and the embeddings-only fused step (MARL_POLICY_EMBED_ONLY) against the full step for the replay.
Alternating A/B in one process; wall times of work that ends in a device synchronise.

    python tools/bench_replay.py [--reps 5] [--out profiles/r3_replay_bench_shape.json]"""
import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from distributed_multi_agent_reinforcement_learning_b200 import default_config, mappo_parallel  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena  # noqa: E402
from train_large import gpu_info, replay_pass  # noqa: E402


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--pursuers", type=int, default=8)
    ap.add_argument("--steps", type=int, default=150)
    ap.add_argument("--depth", type=int, default=1)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    B, N, T, D = args.envs, args.pursuers, args.steps, args.depth
    mbs = max(1, round(B / 10))
    cfg = default_config(env__num_defender=N, env__max_steps=T, algo__depth=D, algo__learner_device=str(dev), algo__worker_device=str(dev))
    env = BatchedPursuitEnv(cfg, B, device=dev, num_maps=64)
    env.reset_device(seed=3)
    snap = env.snapshot()
    torch.manual_seed(0)
    m = MAPPO(cfg, B, mbs, "Learner")
    batches = {}
    for mode in ("store", "replay"):
        env.restore(snap)
        arena = RolloutArena(env.params, B, T, dev)
        batches[mode] = (m.rollout_batched(env, arena, T, seed=1, history=mode), arena)
    tb_s, tb_r = batches["store"][0], batches["replay"][0]
    res = {"replay_ms": {"embed_only": [], "full_step": []}, "epoch_ms": {"store": [], "replay": []}}
    for embed in (True, False):                                 # warm-up of both kernels and of the epoch on both batches
        mappo_parallel.REPLAY_EMBED_ONLY = embed
        replay_pass(tb_r, mbs)
    mappo_parallel.REPLAY_EMBED_ONLY = True
    for tb in (tb_s, tb_r):
        m.train(tb, 1, return_numpy=False)
    for _ in range(args.reps):
        for embed in (True, False):
            mappo_parallel.REPLAY_EMBED_ONLY = embed
            res["replay_ms"]["embed_only" if embed else "full_step"].append(timed(lambda: replay_pass(tb_r, mbs)))
    mappo_parallel.REPLAY_EMBED_ONLY = True
    for _ in range(args.reps):
        for mode, tb in (("store", tb_s), ("replay", tb_r)):
            res["epoch_ms"][mode].append(timed(lambda: m.train(tb, 1, return_numpy=False)))
    med = {k: {kk: statistics.median(vv) for kk, vv in v.items()} for k, v in res.items()}
    out = {"shape": {"envs": B, "pursuers": N, "steps": T, "depth": D, "mini_batch_size": mbs,
                     "concurrent_minibatches": mappo_parallel.CONCURRENT_MINIBATCHES},
           "median_ms": med, "samples_ms": res,
           "replay_share_of_replay_epoch": med["replay_ms"]["embed_only"] / med["epoch_ms"]["replay"],
           "embed_only_speedup": med["replay_ms"]["full_step"] / med["replay_ms"]["embed_only"],
           "gpu": gpu_info(),
           "note": "replay_ms: a replay-only pass over the epoch's minibatches (stream layout of train); epoch_ms: MAPPO.train "
                   "(GAE + minibatches + clip), store vs replay batch of the same episode; A and B alternate"}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
