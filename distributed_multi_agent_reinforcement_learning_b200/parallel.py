"""Data-parallel plumbing: one process per GPU, `torch.distributed` (NCCL over NVLink/NVSwitch on the GPU box, gloo in
the CPU tests).  Replaces the Ray learner/worker protocol of the reference (runner.py:28-47,72-78; main.py:73-75,99-129):

  * envs are independent, so the rollout shards by env index with NO data-path collective (`shard_range`);
  * all replicas start from rank 0's weights (`broadcast_` — main.py:73-75);
  * per update the accumulated-and-clipped gradients are SUMMED across replicas (`allreduce_sum_` on the single flat
    gradient arena — main.py:121-126 sums, it does not average) and every replica applies the same Adam step.
"""
import torch
import torch.distributed as dist


def world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_range(n_global, rank=None, world_size=None):
    """Contiguous [lo, hi) block of env indices owned by `rank` (sizes differ by at most one)."""
    if rank is None or world_size is None:
        rank, world_size = world()
    base, rem = divmod(int(n_global), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def allreduce_sum_(flat, mean=False):
    """In-place all-reduce of one flat tensor (the whole gradient arena is ONE ~2 MB message: latency-bound, so a single
    collective per update).  `mean=True` divides by the world size (not the reference's semantics)."""
    rank, ws = world()
    if ws > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        if mean:
            flat.div_(ws)
    return flat


def allreduce_max_(t):
    """In-place element-wise maximum of one tensor over the ranks."""
    rank, ws = world()
    if ws > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t


def broadcast_(flat, src=0):
    rank, ws = world()
    if ws > 1:
        dist.broadcast(flat, src=src)
    return flat


def max_over_ranks(value, device):
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    rank, ws = world()
    if ws > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())
