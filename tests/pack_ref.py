"""numpy restatement of the elite exchange (test infrastructure; csrc/cemk.cu behind cemk_topk_pack and
cemk_merge_sorted_lists), at any width nvar.  Used by the gloo tests on the CPU and compared bit for bit with the CUDA
kernels in tests/test_gpu_kernels.py and tests/test_gpu_dof.py."""
import numpy as np


def stable_order(cost):
    """jnp.argsort semantics (mjx_planner.py:307): ascending, stable, NaN last."""
    cost = np.asarray(cost)
    key = np.where(np.isnan(cost), np.inf, cost)
    return np.lexsort((np.arange(len(cost)), np.isnan(cost), key))


def topk_pack_ref(cost, idx_base, k, xi):
    """cemk_topk_pack: records [k][nvar + 2] = xi, cost, global index (as float32) of the k best local samples."""
    nv = xi.shape[1]
    loc = stable_order(cost)[:k]
    out = np.empty((k, nv + 2), np.float32)
    out[:, :nv] = xi[loc]
    out[:, nv] = np.asarray(cost, np.float32)[loc]
    out[:, nv + 1] = (loc + idx_base).astype(np.float32)
    return out


def _order_key(cost):
    """float_order in csrc/cemk.cu: float32 bits mapped to an ascending unsigned key, every NaN last, -0.0 tied with +0.0
    (jnp.argsort's order; subnormals stay apart from zero)."""
    u = np.asarray(cost, np.float32).view(np.uint32)
    u = np.where(u << np.uint32(1) == 0, np.uint32(0), u).astype(np.uint32)
    key = np.where(u & 0x80000000, ~u, u | 0x80000000)
    return np.where(np.isnan(cost), np.uint32(0xffffffff), key).astype(np.uint32)


def merge_sorted_lists_ref(packed, nlist, kl, k):
    """cemk_merge_sorted_lists: `nlist` blocks of `kl` (cost, index)-sorted records -> the k best by (cost, row) as xi_elite,
    cost_elite, gidx_elite.  k_merge_lists' rule: a record's position is its position in its own block plus, for every other
    block, the number of records with a smaller key; blocks before its own also count equal keys."""
    nv = packed.shape[1] - 2
    key = _order_key(packed[:, nv]).reshape(nlist, kl)
    pos = np.tile(np.arange(kl), (nlist, 1))
    for a in range(nlist):
        for b in range(nlist):
            if b != a:
                pos[a] += np.searchsorted(key[b], key[a], side="right" if b < a else "left")
    pos = pos.ravel()
    win = np.flatnonzero(pos < k)
    sel = np.empty(k, np.int64)
    sel[pos[win]] = win
    return packed[sel, :nv].copy(), packed[sel, nv].copy(), packed[sel, nv + 1].astype(np.int32)
