"""Event-timed launches of the small kernels around k_rollout (one GPU), for A/B of library variants:
    [CEMK_LIB_PATH=<another build>/libcemk.so] python tools/time_small_kernels.py
sample (k_chol66 + k_sample), k_project, local top-k (argsort / pack), the merge of 8 gathered elite lists, mean / cov."""
import contextlib
import io
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from manipulator_mujoco_b200 import _lib, cem_planner, jax_prng  # noqa: E402
from manipulator_mujoco_b200.planner import _ptr  # noqa: E402

dev = torch.device("cuda:0")
B, T = int(os.environ.get("BL", 4096)), 100
with contextlib.redirect_stdout(io.StringIO()):
    pl = cem_planner(num_dof=6, num_batch=B, num_steps=T, timestep=0.05, maxiter_cem=1, num_elite=0.05, w_pos=20.0, w_rot=3.0, w_col=80.0,
                     maxiter_projection=10, device=dev)
lib, h, nv = pl._lib, pl._h, pl.nvar
z6 = torch.zeros(6, device=dev)
q0 = torch.tensor([1.5, -1.8, 1.75, -1.25, -1.6, 0.0], device=dev)
st = torch.cat([q0, z6, z6, z6, z6]).unsqueeze(0).expand(B, 30).contiguous()
mean0, cov0 = torch.zeros(nv, device=dev), 10 * torch.eye(nv, device=dev)
key1 = jax_prng.split(pl.key)[0]
flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)


REPS = int(os.environ.get("REPS", 20))          # REPS=1 under ncu: one launch of everything


def timed(fn, reps=REPS):
    for _ in range(3 if REPS > 1 else 0):
        fn()
    ts = []
    for _ in range(reps):
        flush.fill_(1.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    return float(np.median(ts))


xi, _ = pl.compute_xi_samples(key1, mean0, cov0)
print(f"sample (chol + sample)   {timed(lambda: pl.compute_xi_samples(key1, mean0, cov0)):7.1f} us")
print(f"project                  {timed(lambda: pl._project(xi, st, True)):7.1f} us")
g = torch.Generator(device="cpu").manual_seed(3)
cost4 = torch.rand(B, 4, generator=g).to(dev) * 50
print(f"argsort_topk n={B} k=204 {timed(lambda: pl._argsort_topk(cost4, 4, B, 204, xi)):7.1f} us")
for kl in (204, 1638):
    pack = torch.empty(kl, nv + 2, device=dev)
    keys = torch.empty(1 << (B - 1).bit_length(), dtype=torch.int64, device=dev)
    print(f"topk_pack n={B} k={kl:5d} {timed(lambda: _lib.check(lib.cemk_topk_pack(h, B, _ptr(cost4), 4, 0, _ptr(keys), kl, _ptr(xi), _ptr(pack), pl._stream()), lib)):7.1f} us")
for nlist, kl in ((2, 409), (8, 1638), (8, 3276)):
    k = kl
    packed = torch.empty(nlist * kl, nv + 2, device=dev)
    for a in range(nlist):
        c = torch.sort(torch.rand(kl, generator=g) * 50)[0]
        packed[a * kl:(a + 1) * kl, :nv] = torch.randn(kl, nv, generator=g).to(dev)
        packed[a * kl:(a + 1) * kl, nv] = c.to(dev)
        packed[a * kl:(a + 1) * kl, nv + 1] = torch.arange(a * B, a * B + kl, dtype=torch.float32, device=dev)
    xe, ce, gi = torch.empty(k, nv, device=dev), torch.empty(k, device=dev), torch.empty(k, dtype=torch.int32, device=dev)
    print(f"merge {nlist} lists x {kl:5d}     {timed(lambda: _lib.check(lib.cemk_merge_sorted_lists(h, nlist, kl, _ptr(packed), k, _ptr(xe), _ptr(ce), _ptr(gi), pl._stream()), lib)):7.1f} us")
    print(f"mean_cov k={k:5d}          {timed(lambda: pl.compute_mean_cov(ce, mean0, cov0, xe)):7.1f} us")
xe, ce = torch.randn(204, nv, device=dev), torch.rand(204, device=dev) * 5
print(f"mean_cov k=  204          {timed(lambda: pl.compute_mean_cov(ce, mean0, cov0, xe)):7.1f} us")
