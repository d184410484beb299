"""End-to-end driver on one GPU (or one per rank under torchrun): what main.py + runner.py do with Ray actors
(main.py:79-129: broadcast weights -> workers explore -> learners train -> gradient sum -> Adam), here as
reset -> batched rollout (all envs, networks in the loop) -> MAPPO.train -> all-reduce + Adam, per iteration.

    python tools/train_loop.py --envs 512 --iters 10
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/train_loop.py --envs 512

Prints one line per iteration: mean episode reward per env (sum over pursuers and steps, the quantity the reference's
evaluator tracks), fraction of envs with a collision, losses, rollout / train wall times, then after "exact" the iteration, the step
count, and the reward and losses as float.hex.  Training is bit-reproducible, so two runs with the same arguments print the same exact
columns:  diff <(grep -o 'exact.*' a.log) <(grep -o 'exact.*' b.log)

    python tools/train_loop.py --envs 512 --iters 3 --save-dir ck       # saves ck/training_state_rank0.pt after every iteration
    python tools/train_loop.py --envs 512 --iters 6 --resume ck         # continues with iteration 3, as if never stopped"""
import argparse
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from distributed_multi_agent_reinforcement_learning_b200 import default_config, parallel  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.checkpoint import load_training_state, save_training_state  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=512)
    ap.add_argument("--maps", type=int, default=32)
    ap.add_argument("--pursuers", type=int, default=8)
    ap.add_argument("--steps", type=int, default=150)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--depth", type=int, default=1)
    ap.add_argument("--allreduce", default=None, choices=[None, "update", "minibatch"],
                    help="gradient exchange: once per update (reference, default) or once per PPO minibatch")
    ap.add_argument("--host-reset", action="store_true", help="generate episodes on the host with the reference's generators (slow)")
    ap.add_argument("--save-dir", default=None, help="write the training state (one file per rank) to this directory")
    ap.add_argument("--save-every", type=int, default=1, help="iterations between saves (the last iteration is always saved)")
    ap.add_argument("--resume", default=None, help="continue from the training state in this directory")
    args = ap.parse_args()
    if args.save_every < 1:
        ap.error("--save-every must be >= 1")
    rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("WORLD_SIZE", 1), ("LOCAL_RANK", 0)))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=dev)
    cfg = default_config(env__num_defender=args.pursuers, env__max_steps=args.steps, algo__depth=args.depth,
                         algo__learner_device=str(dev), algo__worker_device=str(dev))
    B, T, N = args.envs, args.steps, args.pursuers
    env = BatchedPursuitEnv(cfg, B, device=dev, num_maps=args.maps)
    arena = RolloutArena(env.params, B, T, dev)
    torch.manual_seed(0)
    mappo = MAPPO(cfg, B, max(1, round(B / 10)), "Learner")
    mappo.sync_weights(0)
    total_steps, start = 0, 0
    state_file = lambda d: os.path.join(d, f"training_state_rank{rank}.pt")     # noqa: E731  (env shards and reward statistics are per rank)
    if args.resume:
        extra = load_training_state(state_file(args.resume), mappo, env)
        start, total_steps = int(extra["next_iter"]), int(extra["total_steps"])
    W, H = cfg.map.map_size
    for it in range(start, args.iters):
        t0 = time.perf_counter()
        if args.host_reset:
            env.reset(seed=1000 * rank + it)                   # host generation with the reference's placement rules
            g = np.random.default_rng(7 + 1000 * rank + it)
            env.set_target_tape(np.stack([g.integers(0, W, (B, 16)), g.integers(0, H, (B, 16))], -1).astype(np.int32))
        else:
            env.reset_device(seed=1000 * rank + it)            # same rules, generated on the GPU (csrc/reset_kernels.cu)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        if not args.host_reset:
            assert int(env.reset_fail.sum()) == 0, "device reset could not place every pursuer / evader"
        tb = mappo.rollout_batched(env, arena, T, seed=it * world + rank)     # distinct sampling streams per replica and iteration
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        assert int(env.evader_status.max()) == 0, "evader search overflow / target tape exhausted"
        ep_reward = float(arena.raw_reward.sum(dim=(0, 2)).float().mean())
        collided = float(env.collision.float().mean())
        total_steps += world * B * T
        for _ in range(int(cfg.algo.epochs)):                       # main.py:99: K epochs over the same buffers, one Adam step each
            obj_c, obj_a, _, _ = mappo.train(tb, total_steps, return_numpy=False, allreduce=args.allreduce)
            mappo.update(total_steps)
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        stats = torch.tensor([ep_reward, collided, obj_c, obj_a], device=dev, dtype=torch.float64)
        if world > 1:
            torch.distributed.all_reduce(stats)
            stats /= world
        if args.save_dir and ((it + 1) % args.save_every == 0 or it + 1 == args.iters):
            save_training_state(state_file(args.save_dir), mappo, env, extra=dict(next_iter=it + 1, total_steps=total_steps))
        if rank == 0:
            s = [float(x) for x in stats.cpu()]
            print(f"iter {it:3d}  steps {total_steps:9d}  ep_reward {s[0]:9.2f}  collided {s[1]:5.2f}  objC {s[2]:8.4f}  "
                  f"objA {s[3]:8.4f}  reset {t1 - t0:5.2f}s  rollout {1e3 * (t2 - t1):7.1f}ms  train {1e3 * (t3 - t2):7.1f}ms  "
                  f"exact {it} {total_steps} {s[0].hex()} {s[2].hex()} {s[3].hex()}", flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
