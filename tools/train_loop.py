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
    python tools/train_loop.py --envs 512 --iters 6 --resume ck         # continues with iteration 3, as if never stopped

--segment S (a divisor of --steps; default: the whole episode) makes one iteration one rollout segment of S env steps followed by the
epoch and update on it; the GRU hidden states and the history embeddings carry over to the next segment of the same episode, and envs
are reset only at episode starts.  The episode reward is printed on the iteration that ends an episode ("-" on the others), and
--save-dir / --resume work at any segment boundary.

    python tools/train_loop.py --envs 512 --steps 150 --segment 50 --iters 6      # two episodes, three updates each

--auto-reset lets the segments run across episode boundaries (MAPPO.rollout_batched(auto_reset=...)): --segment may then be any
1 <= S <= --steps, and the rollout resets the envs on the device itself when an episode ends inside a segment.  The episodes and their
seeds are the ones the loop uses without it, so for an S that divides --steps both print the same exact columns.  The iteration that
finishes an episode prints its reward.

    python tools/train_loop.py --envs 512 --steps 150 --segment 64 --auto-reset --iters 7

--device-tape draws the evader's candidate-target tape on the device (reset_device(tape="device")) instead of with a torch.Generator.
--graph (needs --auto-reset, implies --device-tape) replays each segment from the CUDA graphs of MAPPO.explore_batched; it prints the same
exact columns as --device-tape without it.

    python tools/train_loop.py --envs 512 --steps 150 --segment 64 --auto-reset --graph --iters 7

--map-pool DIR trains on the maps of a map pool (MapPool files, e.g. the authors' or one written by tools/make_map_pool.py) instead of
generated ones: the pool's first M - K maps are installed into the engine once (verified against the files), and every reset of the
plain, --auto-reset and --graph loops keeps them and draws each env's map from them (reset_device(maps="draw")).  --held-out K keeps
the pool's last K maps out of training and evaluates the policy on them every --eval-every iterations (an Evaluator with the held-out
maps: --eval-envs arg-max episodes, env b on held-out map b % K, the same maps every time); rank 0 prints the result on an "eval" line,
whose float.hex columns follow "hex".  The evaluation does not change the training: the exact columns are those of a run on a pool of
the first M - K maps alone.

    python tools/make_map_pool.py --maps 2000 --seed 0 --out pool
    python tools/train_loop.py --envs 512 --steps 150 --segment 64 --auto-reset --map-pool pool --held-out 100 --eval-every 5

--stats has every epoch reduce the PPO diagnostics of MAPPO.train(stats=True) on the device (a TrainStats, all-reduced over the ranks);
rank 0 prints them on a "stats" line after the iteration's line: the epoch they belong to (the last one trained), the epoch at which
--target-kl stopped the update ("-" if it did not), entropy, approx_kl (k3), approx_kl_k1, clip_frac, ratio_min / ratio_max,
value_clip_frac, explained_variance, rollout_explained_variance, adv_mean / adv_std (raw advantage), return_mean, grad_norm_max /
grad_norm_last (pre-clip), clipped_minibatches, rows, then their float.hex after "hex" ("-" for a value the configuration does not
have).  The statistics change nothing in the training: the exact columns are those of a run without --stats.
--epochs K overrides algo.epochs (K epochs per update, one Adam step each).  --target-kl X (needs K >= 2) stops an update early: when
the approx_kl of epoch k >= 2 exceeds X, that epoch's gradient is dropped (no Adam step) and the update's remaining epochs are skipped.
The losses on the iteration's line are then those of the last epoch that stepped.  The decision comes from bit-reproducible statistics, so such runs stay reproducible and resumable; without --stats a "kl_stop" line
reports each stop.

    python tools/train_loop.py --envs 512 --iters 5 --stats --epochs 4 --target-kl 0.02"""
import argparse
import math
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from distributed_multi_agent_reinforcement_learning_b200 import default_config, parallel  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.checkpoint import load_training_state, save_training_state  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.evaluator import Evaluator  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.map_pool import MapPool, MapPoolError  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.mappo_parallel import MAPPO, AutoReset, RolloutCarry  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv, RolloutArena  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=512)
    ap.add_argument("--maps", type=int, default=None, help="maps generated per reset (default 32); not with --map-pool")
    ap.add_argument("--map-pool", default=None, help="train on the maps of the MapPool in this directory (resets draw from them)")
    ap.add_argument("--held-out", type=int, default=0, help="--map-pool: keep the pool's last K maps for evaluation")
    ap.add_argument("--eval-every", type=int, default=1, help="--held-out: iterations between evaluations")
    ap.add_argument("--eval-envs", type=int, default=None, help="--held-out: episodes per evaluation (default: K)")
    ap.add_argument("--pursuers", type=int, default=8)
    ap.add_argument("--steps", type=int, default=150)
    ap.add_argument("--segment", type=int, default=None, help="env steps per iteration, a divisor of --steps (default: --steps)")
    ap.add_argument("--auto-reset", action="store_true",
                    help="segments may cross episode boundaries: any --segment in [1, --steps], envs reset inside the rollout")
    ap.add_argument("--device-tape", action="store_true", help="--auto-reset: draw the target tape on the device")
    ap.add_argument("--graph", action="store_true", help="--auto-reset: replay the segments from CUDA graphs (implies --device-tape)")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--depth", type=int, default=1)
    ap.add_argument("--allreduce", default=None, choices=[None, "update", "minibatch"],
                    help="gradient exchange: once per update (reference, default) or once per PPO minibatch")
    ap.add_argument("--host-reset", action="store_true", help="generate episodes on the host with the reference's generators (slow)")
    ap.add_argument("--save-dir", default=None, help="write the training state (one file per rank) to this directory")
    ap.add_argument("--save-every", type=int, default=1, help="iterations between saves (the last iteration is always saved)")
    ap.add_argument("--resume", default=None, help="continue from the training state in this directory")
    ap.add_argument("--stats", action="store_true", help="print the PPO diagnostics of every update on a 'stats' line")
    ap.add_argument("--epochs", type=int, default=None, help="PPO epochs per update (default: algo.epochs)")
    ap.add_argument("--target-kl", type=float, default=None,
                    help="stop an update after epoch k >= 2 whose approx_kl exceeds this, dropping that epoch's gradient")
    args = ap.parse_args()
    if args.epochs is None:
        args.epochs = int(default_config().algo.epochs)
    if args.epochs < 1:
        ap.error("--epochs must be >= 1")
    if args.target_kl is not None:
        if args.epochs < 2:
            ap.error(f"--target-kl needs at least 2 epochs per update (--epochs; now {args.epochs}): the first epoch always steps")
        if not math.isfinite(args.target_kl) or args.target_kl < 0:
            ap.error("--target-kl must be a finite number >= 0")
    if args.save_every < 1:
        ap.error("--save-every must be >= 1")
    pool = None
    if args.map_pool is None:
        if args.held_out:
            ap.error("--held-out needs --map-pool")
        args.maps = 32 if args.maps is None else args.maps
    else:
        if args.host_reset:
            ap.error("--map-pool draws the envs' maps on the device; it does not combine with --host-reset")
        if args.maps is not None:
            ap.error("--map-pool sets the maps (the pool's size less --held-out); it does not combine with --maps")
        if args.held_out < 0 or args.eval_every < 1 or (args.eval_envs is not None and args.eval_envs < 1):
            ap.error("--held-out must be >= 0, --eval-every and --eval-envs >= 1")
        try:
            pool = MapPool.load(args.map_pool, mmap=True)
        except MapPoolError as e:
            ap.error(f"--map-pool: {e}")
        if args.held_out >= len(pool):
            ap.error(f"--held-out {args.held_out} leaves no training map of the pool's {len(pool)}")
        args.maps = len(pool) - args.held_out
    S = args.steps if args.segment is None else args.segment
    if (args.graph or args.device_tape) and not args.auto_reset:
        ap.error("--graph / --device-tape need --auto-reset")
    if args.auto_reset:
        if args.host_reset:
            ap.error("--auto-reset resets the envs on the device; it does not combine with --host-reset")
        if S < 1 or S > args.steps:
            ap.error(f"--segment {S} must lie in [1, --steps {args.steps}] with --auto-reset")
    elif S < 1 or args.steps % S:
        ap.error(f"--segment {S} must be a positive divisor of --steps {args.steps}")
    n_seg = args.steps // S
    rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("WORLD_SIZE", 1), ("LOCAL_RANK", 0)))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=dev)
    cfg = default_config(env__num_defender=args.pursuers, env__max_steps=args.steps, algo__depth=args.depth, algo__epochs=args.epochs,
                         algo__learner_device=str(dev), algo__worker_device=str(dev))
    B, T, N = args.envs, args.steps, args.pursuers
    env = BatchedPursuitEnv(cfg, B, device=dev, num_maps=args.maps)
    if pool is not None:
        pool.install(env, np.arange(args.maps), verify=True)
    arena = RolloutArena(env.params, B, S, dev)
    torch.manual_seed(0)
    mappo = MAPPO(cfg, B, max(1, round(B / 10)), "Learner")
    mappo.sync_weights(0)
    args.reset_maps = "generate" if pool is None else "draw"
    args.evaluator = None
    if pool is not None and args.held_out and rank == 0:
        with torch.random.fork_rng(devices=[dev]):      # the evaluator's networks do not draw from the training's RNG streams
            agent = MAPPO(cfg, None, None, "Evaluator")
        # its seed and recorder are part of the training state, so a resumed run evaluates as if never stopped
        args.evaluator = Evaluator(cfg, args.eval_envs or args.held_out, agent, device=dev, pool=pool,
                                   pool_indices=np.arange(args.maps, len(pool)))
    args.mappo = mappo
    total_steps, start = 0, 0
    carry = RolloutCarry.zeros(mappo, B, N) if n_seg > 1 else None     # where the next segment of the current episode starts
    ep_sum = torch.zeros(B, dtype=torch.int64, device=dev)              # raw reward of the current episode so far, per env
    state_file = lambda d: os.path.join(d, f"training_state_rank{rank}.pt")     # noqa: E731  (env shards and reward statistics are per rank)
    if args.auto_reset:
        return auto_reset_loop(args, rank, world, dev, cfg, env, arena, mappo, state_file)
    if args.resume:
        extra = load_training_state(state_file(args.resume), mappo, env, evaluator=args.evaluator, carry=carry)
        start, total_steps = int(extra["next_iter"]), int(extra["total_steps"])
        if carry is not None:
            ep_sum = extra["ep_reward_so_far"].to(dev)
            if carry.t0 != (start % n_seg) * S:
                raise SystemExit(f"--resume: the file continues at step {carry.t0} of an episode, iteration {start} of --segment {S} "
                                 f"starts at step {(start % n_seg) * S}")
    W, H = cfg.map.map_size
    for it in range(start, args.iters):
        ep, seg = divmod(it, n_seg)                    # episode and segment index (one segment per episode by default: ep == it)
        t0 = time.perf_counter()
        if seg == 0:
            if args.host_reset:
                env.reset(seed=1000 * rank + ep)                   # host generation with the reference's placement rules
                g = np.random.default_rng(7 + 1000 * rank + ep)
                env.set_target_tape(np.stack([g.integers(0, W, (B, 16)), g.integers(0, H, (B, 16))], -1).astype(np.int32))
            else:                                              # same rules, generated on the GPU (csrc/reset_kernels.cu)
                env.reset_device(seed=1000 * rank + ep, maps=args.reset_maps)
            if carry is not None:
                carry = RolloutCarry.zeros(mappo, B, N)
            ep_sum.zero_()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        if not args.host_reset and seg == 0:
            assert int(env.reset_fail.sum()) == 0, "device reset could not place every pursuer / evader"
        # distinct sampling streams per replica and episode; the segments of an episode share one (keyed by the episode's step)
        tb = mappo.rollout_batched(env, arena, S, seed=ep * world + rank, carry=carry)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        assert int(env.evader_status.max()) == 0, "evader search overflow / target tape exhausted"
        ep_sum += arena.raw_reward.sum(dim=(0, 2))
        ep_end = seg == n_seg - 1
        ep_reward = float(ep_sum.float().mean())
        collided = float(env.collision.float().mean())
        total_steps += world * B * S
        if carry is not None:
            carry = tb.carry
        obj_c, obj_a, stats_line = run_epochs(args, mappo, tb, total_steps, it)     # main.py:99: K epochs, one Adam step each
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        stats = torch.tensor([ep_reward, collided, obj_c, obj_a], device=dev, dtype=torch.float64)
        if world > 1:
            torch.distributed.all_reduce(stats)
            stats /= world
        s = [float(x) for x in stats.cpu()]
        evaluation = evaluate(args, it, total_steps, s)
        if args.save_dir and ((it + 1) % args.save_every == 0 or it + 1 == args.iters):
            extra = dict(next_iter=it + 1, total_steps=total_steps)
            if carry is not None:
                extra["ep_reward_so_far"] = ep_sum.cpu()
            save_training_state(state_file(args.save_dir), mappo, env, evaluator=args.evaluator, extra=extra,
                                carry=None if ep_end else carry)
        if rank == 0:
            rew, rew_hex = (f"{s[0]:9.2f}", s[0].hex()) if ep_end else (f"{'-':>9}", "-")
            print(f"iter {it:3d}  steps {total_steps:9d}  ep_reward {rew}  collided {s[1]:5.2f}  objC {s[2]:8.4f}  "
                  f"objA {s[3]:8.4f}  reset {t1 - t0:5.2f}s  rollout {1e3 * (t2 - t1):7.1f}ms  train {1e3 * (t3 - t2):7.1f}ms  "
                  f"exact {it} {total_steps} {rew_hex} {s[2].hex()} {s[3].hex()}", flush=True)
            if stats_line:
                print(stats_line, flush=True)
            if evaluation:
                print(evaluation, flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


def run_epochs(args, mappo, tb, total_steps, it):
    """The update on one batch: --epochs epochs of MAPPO.train, each followed by one Adam step (main.py:99), with the statistics of
    every epoch reduced on the device when --stats or --target-kl needs them.  --target-kl: an epoch k >= 2 whose all-reduced approx_kl
    exceeds the target gets no Adam step, and the update ends there (every rank takes the same decision from the same global numbers).
    Returns the losses of the last epoch that stepped (a stopped epoch's losses are dropped with its gradient) and the line to print
    after the iteration's (or None)."""
    want = args.stats or args.target_kl is not None
    stopped, st = None, None
    for k in range(1, args.epochs + 1):
        losses = mappo.train(tb, total_steps, return_numpy=False, allreduce=args.allreduce, stats=want)[:2]
        if want:
            st = mappo.last_train_stats.allreduce_()
            if args.target_kl is not None and k >= 2 and st.approx_kl > args.target_kl:
                stopped = k
                break
        mappo.update(total_steps)
        obj_c, obj_a = losses
    line = None
    if args.stats:
        fmt = lambda v: "-" if v is None else (str(v) if isinstance(v, int) else f"{v:.6g}")          # noqa: E731
        hx = lambda v: "-" if v is None else float(v).hex()                                             # noqa: E731
        vals = st.as_dict()
        line = (f"stats {it:3d}  epoch {k}  kl_stop {stopped or '-'}  " + "  ".join(f"{f} {fmt(v)}" for f, v in vals.items())
                + f"  hex {it} {k} {stopped or '-'} " + " ".join(hx(v) for v in vals.values()))
    elif stopped:
        line = f"kl_stop {it:3d}  epoch {stopped}  approx_kl {st.approx_kl:.6g}  target_kl {args.target_kl:g}  hex {it} {stopped} {st.approx_kl.hex()}"
    return obj_c, obj_a, line


def evaluate(args, it, total_steps, s):
    """--held-out, every --eval-every iterations: arg-max episodes of the current policy on the held-out maps (rank 0 only).  Returns
    the "eval" line, or None.  It runs before the iteration's save, so the saved evaluator continues where a resumed run expects it."""
    ev = args.evaluator
    if ev is None or (it + 1) % args.eval_every:
        return None
    t0 = time.perf_counter()
    weights = lambda net: {k: v.detach().clone() for k, v in net.state_dict().items()}     # noqa: E731
    with torch.random.fork_rng(devices=[args.mappo.device]):        # leaves the training's RNG streams as they were
        ev.run(weights(args.mappo.actor), weights(args.mappo.critic), total_steps, s[0], (s[2], s[3]))
    r = ev.last
    return (f"eval {it:3d}  steps {total_steps:9d}  held-out maps {args.held_out}  episodes {ev.num_cpus_eval}  avg_r {r['avg_r']:9.2f}  "
            f"std_r {r['std_r']:8.2f}  time {time.perf_counter() - t0:5.2f}s  hex {it} {float(r['avg_r']).hex()} {float(r['std_r']).hex()}")


def auto_reset_loop(args, rank, world, dev, cfg, env, arena, mappo, state_file):
    """The loop of --auto-reset: one segment of S steps per iteration, episode e reset on the device with seed 1000*rank + e and sampled
    with seed e*world + rank (the seeds of the loop without --auto-reset), the resets inside the rollout."""
    B, N, S, T_ep = args.envs, args.pursuers, args.segment or args.steps, args.steps
    auto = AutoReset(reset_seed=lambda e: 1000 * rank + e, sample_seed=lambda e: e * world + rank,
                     tape="device" if args.device_tape or args.graph else "torch", maps=args.reset_maps)
    carry = RolloutCarry.zeros(mappo, B, N)
    ep_sum = torch.zeros(B, dtype=torch.int64, device=dev)
    total_steps, start = 0, 0
    if args.resume:
        extra = load_training_state(state_file(args.resume), mappo, env, evaluator=args.evaluator, carry=carry)
        start, total_steps = int(extra["next_iter"]), int(extra["total_steps"])
        ep_sum = extra["ep_reward_so_far"].to(dev)
        if divmod(start * S, T_ep) != (carry.episode, carry.t0):
            raise SystemExit(f"--resume: the file continues at step {carry.t0} of episode {carry.episode}, iteration {start} of "
                             f"--segment {S} starts at step {start * S % T_ep} of episode {start * S // T_ep}")
    else:
        env.reset_device(seed=auto.reset_seed(0), tape_len=auto.tape_len, tape=auto.tape, maps=auto.maps)
        torch.cuda.synchronize()
        assert int(env.reset_fail.sum()) == 0, "device reset could not place every pursuer / evader"
    for it in range(start, args.iters):
        t1 = time.perf_counter()
        if args.graph:
            tb = mappo.explore_batched(env, arena, S, carry=carry, auto_reset=auto)
        else:
            tb = mappo.rollout_batched(env, arena, S, carry=carry, auto_reset=auto)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        assert int(env.evader_status.max()) == 0, "evader search overflow / target tape exhausted"
        ep_end = tb.ended_collision is not None     # an episode ended inside or at the end of this segment and the envs were reset
        k = S if tb.boundary is None else tb.boundary
        ep_sum += arena.raw_reward[:k].sum(dim=(0, 2))
        ep_reward = float(ep_sum.float().mean())
        if ep_end:
            assert int(tb.ended_evader_status.max()) == 0, "evader search overflow / target tape exhausted"
            assert int(env.reset_fail.sum()) == 0, "device reset could not place every pursuer / evader"
            collided = float(tb.ended_collision.float().mean())
            ep_sum = arena.raw_reward[k:S].sum(dim=(0, 2))
        else:
            collided = float(env.collision.float().mean())
        total_steps += world * B * S
        carry = tb.carry
        obj_c, obj_a, stats_line = run_epochs(args, mappo, tb, total_steps, it)
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        stats = torch.tensor([ep_reward, collided, obj_c, obj_a], device=dev, dtype=torch.float64)
        if world > 1:
            torch.distributed.all_reduce(stats)
            stats /= world
        s = [float(x) for x in stats.cpu()]
        evaluation = evaluate(args, it, total_steps, s)
        if args.save_dir and ((it + 1) % args.save_every == 0 or it + 1 == args.iters):
            save_training_state(state_file(args.save_dir), mappo, env, evaluator=args.evaluator,
                                extra=dict(next_iter=it + 1, total_steps=total_steps, ep_reward_so_far=ep_sum.cpu()), carry=carry)
        if rank == 0:
            rew, rew_hex = (f"{s[0]:9.2f}", s[0].hex()) if ep_end else (f"{'-':>9}", "-")
            print(f"iter {it:3d}  steps {total_steps:9d}  ep_reward {rew}  collided {s[1]:5.2f}  objC {s[2]:8.4f}  "
                  f"objA {s[3]:8.4f}  reset {0.0:5.2f}s  rollout {1e3 * (t2 - t1):7.1f}ms  train {1e3 * (t3 - t2):7.1f}ms  "
                  f"exact {it} {total_steps} {rew_hex} {s[2].hex()} {s[3].hex()}", flush=True)
            if stats_line:
                print(stats_line, flush=True)
            if evaluation:
                print(evaluation, flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
