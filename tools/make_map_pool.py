"""Writes a map pool (the seven MapPool .npy files) of M maps generated on the device: `BatchedPursuitEnv.reset_device` draws the
maps with the reference's obstacle rules and builds their sensor tables, and `MapPool.from_engine(...).save` writes them out in the
authors' file layout.  So a pool can be used (`tools/train_loop.py --map-pool`) and measured without the authors' files.

    python tools/make_map_pool.py --maps 2000 --seed 0 --out pool"""
import argparse
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from distributed_multi_agent_reinforcement_learning_b200 import default_config  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.map_pool import MapPool  # noqa: E402
from distributed_multi_agent_reinforcement_learning_b200.pursuit_env import BatchedPursuitEnv  # noqa: E402


def make_pool(cfg, M, seed, device="cuda"):
    """The MapPool of the M maps that reset_device(seed) generates on `device`."""
    env = BatchedPursuitEnv(cfg, M, device=device, num_maps=M)
    env.reset_device(seed=seed)
    return MapPool.from_engine(env)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--maps", type=int, required=True)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", required=True, help="directory to write the pool's .npy files to")
    args = ap.parse_args()
    if args.maps < 1:
        ap.error("--maps must be >= 1")
    t0 = time.perf_counter()
    pool = make_pool(default_config(), args.maps, args.seed)
    pool.save(args.out)
    M, W, H, O = pool.shape
    size = sum(os.path.getsize(os.path.join(args.out, f)) for f in os.listdir(args.out) if f.endswith(".npy"))
    print(f"wrote {M} maps of {W}x{H} (O = {O}) to {args.out}: {size / 1e6:.1f} MB in {time.perf_counter() - t0:.1f}s", flush=True)


if __name__ == "__main__":
    main()
