"""Data-parallel host logic for the hot path (SURVEY.md section 8e).

The batch shards naturally: every loss term is a sum over pixels and no stencil crosses a sample,
so rank r processes samples [r*N/G, (r+1)*N/G) with NO collective inside the data path.  The only
exchange is ONE all-reduce of the 8-float loss vector, replacing the reference's per-scalar
`dist.all_reduce` in Trainer.sync (src/trainer.py:381-386).

Two reduction conventions are offered:

* `reference`  -- each rank normalises by its LOCAL batch (what src/trainer.py:248-256 does) and
  sync() averages the per-rank means: identical to the reference under DDP.
* `global`     -- each rank passes `global_batch` to the kernels (vlg_problem_t.global_N), so local
  loss vectors and gradients are already divided by the GLOBAL pixel count and simply ADD: the
  G-GPU result equals the 1-GPU result up to summation order.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
import torch.distributed as dist

# slots of the loss vector (mirror of VLG_LOSS_* in include/vlg_b200.h)
N_SLOTS, SLOT_NVALID, SLOT_MAXDISP = 8, 6, 7


def shard_bounds(n_samples: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous, balanced split of the batch (the first `n % world` ranks get one extra sample);
    with n divisible by world this is the reference's `batch_size // gpus` (src/trainer.py:148)."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of {world}")
    base, extra = divmod(n_samples, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def shard_batch(tensors, rank: int, world: int):
    """Slice every tensor of a (src_rgb, src_layout, flow, tgt_rgb, tgt_label) tuple along dim 0."""
    n = tensors[0].shape[0]
    lo, hi = shard_bounds(n, rank, world)
    return tuple(t[lo:hi] for t in tensors)


def sync_loss_vector(vec: torch.Tensor, convention: str = "global",
                     group: Optional[dist.ProcessGroup] = None) -> torch.Tensor:
    """ONE collective for all loss scalars.  `vec` is the [8] fp32 loss vector of the local shard.

    convention='global'   : vec was computed with global_batch divisors -> SUM.
    convention='reference': vec holds local means -> SUM then / world (Trainer.sync mean=True).
    The max-displacement slot is a maximum, not a sum; it is reduced with MAX in the same call by
    packing it into a second tensor only when a caller asks for it (see `sync_max_disp`).
    """
    if convention not in ("global", "reference"):
        raise ValueError(convention)
    if not (dist.is_available() and dist.is_initialized()):
        return vec
    out = vec.clone()
    dist.all_reduce(out, op=dist.ReduceOp.SUM, group=group)
    if convention == "reference":
        world = dist.get_world_size(group)
        keep = out[SLOT_NVALID].clone()
        out /= world
        out[SLOT_NVALID] = keep           # counts add, they are not averaged
    out[SLOT_MAXDISP] = vec[SLOT_MAXDISP]  # local value; use sync_max_disp for the global maximum
    return out


def sync_counts(counts: torch.Tensor, group: Optional[dist.ProcessGroup] = None) -> torch.Tensor:
    """ONE all-reduce (SUM) of int64 counts, e.g. the confusion counts of `metrics.LayoutIoU`: integer sums, so the
    result equals the single-process counts bit for bit whatever the sharding.  Identity without a process group."""
    if not (dist.is_available() and dist.is_initialized()):
        return counts
    out = counts.clone()
    dist.all_reduce(out, op=dist.ReduceOp.SUM, group=group)
    return out


def sync_max_disp(vec: torch.Tensor, group: Optional[dist.ProcessGroup] = None) -> torch.Tensor:
    m = vec[SLOT_MAXDISP].clone()
    if dist.is_available() and dist.is_initialized():
        dist.all_reduce(m, op=dist.ReduceOp.MAX, group=group)
    return m
