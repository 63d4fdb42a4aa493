"""Multi-GPU plumbing of the rollout path: contiguous sharding of start states, the two
Allreduce steps of `mpi_statistics_scalar` (utilities/mpi_tools.py:71-92) and the batch-wide
rules of a sharded rollout block (`ModelSampler.distribute`).

Paths are independent units: every rank rolls out its own block of start states (Philox counters
use GLOBAL path ids, so results do not depend on the sharding).  Across ranks go the five running
sums (n, sum adv, sum cadv, sum ret, sum cret) and then the sum of squared deviations; with
`ModelSampler.distribute`, also small all-gathers of counts and sums (shard sizes, length histograms,
per-step statistics, diagnostics) and, in `ModelBuffer.get`, the populated rows to one rank.
One process per GPU, `torch.distributed` (NCCL on GPUs, gloo in the CPU tests).

The rollout block has one code path for any number of ranks: a process on its own is the one-rank case
(`Ranks()`), whose gathers return its own vector without touching `torch.distributed`.
"""
from typing import Any, NamedTuple

import numpy as np


def shard_bounds(n, rank, world):
    """Contiguous block partition [lo, hi) of n items; sizes differ by at most one."""
    base, rem = divmod(int(n), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def make_reduce_fn(group=None):
    """In-place SUM all-reduce of a small tensor, or None for a single process."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return None

    def reduce_fn(t):
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        return t
    return reduce_fn


def is_multi_rank(group=None):
    import torch.distributed as dist
    return dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1


def all_gather_host(vec, group=None, device=None):
    """All-gather of a small numpy vector of the same shape on every rank -> numpy [world, ...] in rank
    order.  `device`: where the collective runs (the rank's GPU for NCCL; the host for gloo)."""
    import torch
    import torch.distributed as dist
    if dist.get_backend(group) != "nccl":
        device = "cpu"
    a = np.ascontiguousarray(vec)
    x = torch.from_numpy(a.reshape(-1)).to(device)
    out = torch.empty(dist.get_world_size(group) * x.numel(), dtype=x.dtype, device=x.device)
    dist.all_gather_into_tensor(out, x, group=group)
    return out.cpu().numpy().reshape((-1,) + a.shape)


class Ranks(NamedTuple):
    """The ranks of a rollout block and this process's place among them.  `Ranks()` is a process on its own:
    one rank, no group.  `sharded` marks a block that `ModelSampler.distribute` set up (its `group` None is the
    default process group), even one of world size 1."""
    group: Any = None
    rank: int = 0
    world: int = 1
    root: int = 0
    sharded: bool = False

    @classmethod
    def of(cls, group=None, root=0):
        import torch.distributed as dist
        return cls(group, dist.get_rank(group), dist.get_world_size(group), int(root), True)

    def gather(self, vec, device=None):
        """all_gather_host over these ranks; one rank gathers its own vector and issues no collective."""
        if self.world == 1:
            return np.asarray(vec)[None]
        return all_gather_host(vec, self.group, device)


def rank_order_sum(gathered):
    """Sum of the rows of an all-gathered [world, ...] array, rank 0 first.  Every rank adds the same
    numbers in the same order, so float sums are bit-identical on every rank (an all-reduce does not
    promise that)."""
    acc = gathered[0].copy()
    for row in gathered[1:]:
        acc = acc + row
    return acc


def cap_split(n, survivors):
    """The max_samples cap of a sharded batch: the reference cuts the first n surviving paths of the whole
    batch by path index.  Shards are contiguous in path order, so rank r cuts its first
    clamp(n - sum_{g<r} s_g, 0, s_r) survivors, where s_g = survivors of rank g.  Returns the per-rank cuts."""
    cuts, before = [], 0
    for s in survivors:
        cuts.append(int(min(max(int(n) - before, 0), int(s))))
        before += int(s)
    return cuts


def combine_pass1(sums):
    """sums = (n, sum_adv, sum_cadv, sum_ret, sum_cret) after the first all-reduce ->
    float32 means exactly as mpi_statistics_scalar forms them (sum and n cast to float32 first)."""
    n = np.float32(sums[0])
    if sums[0] == 0:
        z = np.float32(0)
        return dict(n=0, adv_mean=z, cadv_mean=z, ret_mean=z, cret_mean=z)
    return dict(n=int(sums[0]), adv_mean=np.float32(sums[1]) / n, cadv_mean=np.float32(sums[2]) / n,
                ret_mean=np.float32(np.float32(sums[3]) / n), cret_mean=np.float32(np.float32(sums[4]) / n))


def combine_pass2(ssq, n):
    """Population std from the all-reduced sum of squared deviations (mpi_tools.py:85-86)."""
    return np.sqrt(np.float32(ssq) / np.float32(n))
