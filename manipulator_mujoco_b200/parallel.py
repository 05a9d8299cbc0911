"""Host-side plumbing of the sample-sharded CEM (SURVEY.md section 8e).

Samples are independent through sampling, projection, rollout and cost, so a global batch of B
samples is split contiguously: rank r owns global indices [r*B/G, (r+1)*B/G).  Per iteration each
rank keeps its own k' = min(k, B/G) best (cost, global index, xi) triples, one all-gather (NCCL on
the GPUs, gloo in the CPU tests) concatenates them rank-major, and every rank selects the k best of
the G*k' candidates by (cost, row).  Because each rank's block is already (cost, index)-sorted and
blocks arrive in rank order, the row number orders equal costs exactly like the global sample index
does -- i.e. like the reference's stable ``jnp.argsort`` over the whole batch (mjx_planner.py:307).
Every rank therefore holds the identical elite list and computes the identical mean / covariance;
no broadcast is needed.

Exchange record (what ``cemk_topk_pack`` writes and ``cemk_merge_sorted_lists`` reads): ``[k'][nvar + 2]`` float32 =
xi[nvar], cost, global sample index (exact in float32 below 2^24, checked once at construction).
"""
from __future__ import annotations

import torch


def shard_bounds(num_batch: int, world: int, rank: int):
    if num_batch % world:
        raise ValueError("num_batch must be divisible by the number of ranks")
    bl = num_batch // world
    return rank * bl, (rank + 1) * bl


def local_topk_size(k: int, batch_local: int) -> int:
    return min(k, batch_local)


def check_index_range(num_batch: int):
    if num_batch > 1 << 24:
        raise ValueError("global sample index does not fit a float32 mantissa (num_batch > 2^24)")


def gather_elites(pack: torch.Tensor, world: int, group=None, out: torch.Tensor | None = None) -> torch.Tensor:
    import torch.distributed as dist
    if out is None:
        out = torch.empty(world * pack.shape[0], pack.shape[1], dtype=pack.dtype, device=pack.device)
    dist.all_gather_into_tensor(out, pack, group=group)
    return out


def exchange_owned_row(row: torch.Tensor, own, group=None) -> torch.Tensor:
    """Sum-all-reduce in which exactly one rank (``own`` true) contributes ``row`` and every other rank contributes
    exact zeros.  ``torch.where`` rather than a 0/1 multiplication: a non-owning rank's ``row`` is an arbitrary local
    sample and may hold NaN / Inf (diverged rollout), and NaN * 0 = NaN would poison the sum on every rank.
    ``own`` None: ``row`` is already the owner's values or exact zeros (``cemk_tick_record`` writes it that way) and is
    reduced in place."""
    import torch.distributed as dist
    out = row if own is None else torch.where(own.reshape(-1)[0], row, torch.zeros_like(row))
    dist.all_reduce(out, group=group)
    return out
