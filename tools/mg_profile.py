"""Where a multi-GPU CEM iteration spends its time: CUDA events between the stages of cem_iter, stream-ordered (no host
synchronisation inside an iteration), averaged over 20 iterations, per rank.  Run under torchrun on N GPUs of one box:
    timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29544 tools/mg_profile.py
The all-gather stage of a rank includes its wait for the slowest rank's rollout.
DUMP=<file.npz> (one GPU): also save every stage's outputs of one iteration, for bitwise A/B of library variants
(CEMK_LIB_PATH=<another build>/libcemk.so; compare with tools/mg_profile.py --compare a.npz b.npz)."""
import contextlib
import io
import os
import sys

if len(sys.argv) == 4 and sys.argv[1] == "--compare":
    import numpy as np
    a, b = np.load(sys.argv[2]), np.load(sys.argv[3])
    for name in a.files:
        same = a[name].shape == b[name].shape and np.array_equal(a[name].view(np.int32) if a[name].dtype == np.float32 else a[name],
                                                                 b[name].view(np.int32) if b[name].dtype == np.float32 else b[name])
        print(f"{name:10s} {'bit-identical' if same else 'DIFFERENT  max |d| = %g' % float(np.nanmax(np.abs(a[name].astype(np.float64) - b[name].astype(np.float64))))}")
    sys.exit(0)

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from manipulator_mujoco_b200 import _lib, cem_planner, jax_prng, parallel  # noqa: E402
from manipulator_mujoco_b200.planner import _ptr  # noqa: E402

rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dev = torch.device(f"cuda:{local}")
pg = None
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
    pg = dist.group.WORLD
Bl, T = int(os.environ.get("BL", 4096)), 100
B = Bl * world
with contextlib.redirect_stdout(io.StringIO()):
    pl = cem_planner(num_dof=6, num_batch=B, num_steps=T, timestep=0.05, maxiter_cem=1, num_elite=0.05, w_pos=20.0, w_rot=3.0,
                     w_col=80.0, maxiter_projection=10, device=dev, process_group=pg)
z6 = torch.zeros(6, device=dev)
q0 = torch.tensor([1.5, -1.8, 1.75, -1.25, -1.6, 0.0], device=dev)
tp = torch.tensor([-0.3, -0.3, 0.5], device=dev)
tr = torch.tensor([0.0, 1.0, 0.0, 0.0], device=dev)
st = torch.cat([q0, z6, z6, z6, z6]).unsqueeze(0).expand(Bl, 30).contiguous()
mean0, cov0 = torch.zeros(pl.nvar, device=dev), 10 * torch.eye(pl.nvar, device=dev)
key1 = jax_prng.split(pl.key)[0]
lib, h, nv = pl._lib, pl._h, pl.nvar
k = pl.ellite_num
kl = min(k, Bl)
n = world * kl
np2l, np2 = 1 << max(0, (Bl - 1).bit_length()), 1 << max(0, (n - 1).bit_length())
flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
names = ["sample", "project", "rollout", "topk_pack", "all_gather", "merge", "mean_cov"]


def iteration(rec):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
    ev[0].record()
    xi, _ = pl.compute_xi_samples(key1, mean0, cov0); ev[1].record()
    xf, td = pl._project(xi, st, True); ev[2].record()
    theta, cost4, _, _, _ = pl._rollout(td, q0, z6, tp, tr, False); ev[3].record()
    if world == 1:
        xi_e, idx, cost_e = pl._argsort_topk(cost4, 4, Bl, kl, xi); ev[4].record(); ev[5].record(); ev[6].record()
    else:
        pack = pl._buf("elite_pack", (kl, nv + 2))
        _lib.check(lib.cemk_topk_pack(h, Bl, _ptr(cost4), 4, rank * Bl, _ptr(pl._buf("keys", (np2l,), torch.int64)), kl, _ptr(xi), _ptr(pack), pl._stream()), lib)
        ev[4].record()
        gathered = pl._buf("elite_gathered", (n, nv + 2))
        parallel.gather_elites(pack, world, pg, out=gathered); ev[5].record()
        xi_e, cost_e, gi = torch.empty(k, nv, device=dev), torch.empty(k, device=dev), torch.empty(k, dtype=torch.int32, device=dev)
        _lib.check(lib.cemk_merge_sorted_lists(h, world, kl, _ptr(gathered), k, _ptr(xi_e), _ptr(cost_e), _ptr(gi), pl._stream()), lib)
        ev[6].record()
    mc = pl.compute_mean_cov(cost_e, mean0, cov0, xi_e); ev[7].record()
    rec.append(ev)
    return dict(xi=xi, xi_f=xf, thetadot=td, theta=theta, cost4=cost4, xi_elite=xi_e, cost_elite=cost_e, mean=mc[0], cov=mc[1],
                chol=pl._buf("chol", (nv * nv,)), **({"idx": idx} if world == 1 else {"gidx": gi}))


for _ in range(5):
    iteration([])
torch.cuda.synchronize()
if world > 1:
    dist.barrier()
rec = []
for _ in range(20):
    flush.fill_(1.0)
    iteration(rec)
torch.cuda.synchronize()
tot = {nm: sum(ev[i].elapsed_time(ev[i + 1]) for ev in rec) / len(rec) for i, nm in enumerate(names)}
whole = sum(ev[0].elapsed_time(ev[-1]) for ev in rec) / len(rec)
line = f"rank {rank} (B/GPU {Bl}, k {k}, exchange {n} x {nv + 2} floats): " + "  ".join(f"{nm} {1e3 * v:.0f} us" for nm, v in tot.items()) + f"  | iteration {whole:.3f} ms"
if world > 1:
    out = [None] * world
    dist.all_gather_object(out, line)
    if rank == 0:
        print("\n".join(out), flush=True)
    pl.close()
    torch.cuda.synchronize()
    dist.destroy_process_group()
else:
    print(line)
    if os.environ.get("DUMP"):
        import numpy as np
        out = iteration([])
        torch.cuda.synchronize()
        np.savez(os.environ["DUMP"], **{k_: v.detach().cpu().numpy() for k_, v in out.items()})
