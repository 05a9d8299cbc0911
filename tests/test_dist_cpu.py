"""world_size-2 (and 4) gloo tests of the sample-sharded CEM plumbing (manipulator_mujoco_b200/parallel.py), on the exchange
record layout the kernels use (cemk_topk_pack -> all-gather -> cemk_merge_sorted_lists; tests/pack_ref.py restates the
two in numpy and tests/test_gpu_kernels.py checks the kernels against that restatement bit for bit):
local top-k' + all-gather + merge of the per-rank sorted blocks == the reference's global stable argsort top-k, including
cost ties across ranks and NaN costs; the best-sample exchange survives NaN rows on non-owning ranks."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from manipulator_mujoco_b200 import parallel
from pack_ref import merge_sorted_lists_ref, stable_order, topk_pack_ref

NVAR = 66


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _make(B, seed):
    rng = np.random.default_rng(seed)
    cost = rng.uniform(100, 200, B).astype(np.float32)
    cost[rng.integers(0, B, B // 4)] = 123.0          # many exact ties, spread over all ranks
    cost[[5, B - 3]] = np.nan                         # NaN sorts last in jnp.argsort
    cost[1], cost[B - 10] = 0.0, -0.0                 # the two best, on the first and the last rank: -0.0 ties with +0.0
    xi = rng.normal(size=(B, NVAR)).astype(np.float32)
    return cost, xi


def _worker(rank, world, port, B, k, seed, ret):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    cost, xi = _make(B, seed)
    lo, hi = parallel.shard_bounds(B, world, rank)
    kl = parallel.local_topk_size(k, hi - lo)
    cost4 = np.zeros((hi - lo, 4), np.float32)
    cost4[:, 0] = cost[lo:hi]                                                        # the rollout kernel's [B][4] cost record
    pack = torch.from_numpy(topk_pack_ref(cost4[:, 0], lo, kl, xi[lo:hi]))           # cemk_topk_pack
    gathered = parallel.gather_elites(pack, world, out=torch.empty(world * kl, NVAR + 2))     # the planner's call (persistent buffer)
    assert torch.equal(gathered[rank * kl:(rank + 1) * kl].view(torch.int32), pack.view(torch.int32))
    xi_e, cost_e, gidx_e = merge_sorted_lists_ref(gathered.numpy(), world, kl, k)     # cemk_merge_sorted_lists
    # best-sample exchange (planner._cem_device): the owner of the global best contributes its row, every other
    # rank's candidate row is an arbitrary local sample -- here NaN / Inf on purpose
    gbest = int(gidx_e[0])
    own = torch.tensor([lo <= gbest < hi])
    row = torch.full((9,), float("nan"))
    row[3] = float("inf")
    if bool(own):
        row = torch.from_numpy(np.concatenate([xi[gbest, :8], cost[gbest:gbest + 1]]))
    best = parallel.exchange_owned_row(row, own)
    # the pre-masked form the planner uses (cemk_tick_record writes the owner's row or exact zeros)
    masked = row.clone() if bool(own) else torch.zeros_like(row)
    assert torch.equal(parallel.exchange_owned_row(masked, None).view(torch.int32), best.view(torch.int32))
    ret[rank] = (gidx_e.copy(), xi_e.copy(), cost_e.copy(), best.numpy().copy())
    dist.destroy_process_group()


@pytest.mark.parametrize("world,B,k", [(2, 256, 12), (4, 256, 12), (2, 64, 40)])
def test_sharded_merge_equals_global_stable_topk(world, B, k):
    port = _free_port()
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, port, B, k, 7, ret), nprocs=world, join=True)
    cost, xi = _make(B, 7)
    ref = stable_order(cost)[:k]
    for r in range(world):
        gidx, gxi, gcost, best = ret[r]
        np.testing.assert_array_equal(gidx, ref)                      # bit-identical elite index lists on every rank
        np.testing.assert_array_equal(gxi, xi[ref])
        np.testing.assert_array_equal(gcost, cost[ref])
        # NaN rows of the non-owning ranks did not leak into the exchanged best sample
        np.testing.assert_array_equal(best, np.concatenate([xi[ref[0], :8], cost[ref[0]:ref[0] + 1]]))


def test_index_range_check():
    parallel.check_index_range(1 << 24)
    with pytest.raises(ValueError):
        parallel.check_index_range((1 << 24) + 1)


def test_shard_bounds():
    assert parallel.shard_bounds(65536, 8, 3) == (24576, 32768)
    with pytest.raises(ValueError):
        parallel.shard_bounds(100, 8, 0)
