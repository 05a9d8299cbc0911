"""Event-timed planner algebra of BASELINE config 4 (dual_arm_scene.xml: two UR5e = 12 DOF, 16 384 samples, a sweep over Bernstein
orders) on one GPU:
    python tools/time_dof_algebra.py [--out FILE]
B = 16 384, num_dof = 12, k = 819 elites (num_elite 0.05), 10 projection iterations.  Config 4 does not state a horizon; T = 100
is config 2's.  Per order 5, 8, 10, 12, 15 (nvar = 12 (order + 1) = 72 .. 192): sample (normal draws + Cholesky + sampling),
projection + Bernstein evaluation, elite selection (bitonic path: n > 8192) and mean / covariance, each the median of 20 CUDA-event
timed calls with the L2 cache overwritten before every call.  The rollout of the dual-arm scene is not built, so a CEM
iteration of config 4 is not timed here."""
import argparse
import contextlib
import io
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from manipulator_mujoco_b200 import cem_planner, jax_prng  # noqa: E402

B, ND, T, ELITE, REPS = 16384, 12, 100, 0.05, 20
ORDERS = (5, 8, 10, 12, 15)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the table to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_dof_algebra.py needs a CUDA device")
    dev = torch.device("cuda:0")
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)          # 256 MB > the 126 MB L2

    def timed(fn):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(REPS):
            flush.fill_(1.0)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e3)
        return float(np.median(ts))

    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:                                                   # noqa: BLE001 (the table is still valid without it)
        q = torch.cuda.get_device_name(dev) + ", power limit not read"
    lines = [f"# planner algebra of BASELINE config 4 on one GPU: {q}",
             f"# B={B} num_dof={ND} T={T} (config 2's horizon; config 4 states none) k={int(ELITE * B)} maxiter_projection=10; "
             f"median of {REPS} CUDA-event timed calls, L2 overwritten before each; microseconds",
             f"{'order':>5} {'nvar':>4} {'sample':>9} {'project':>9} {'select':>9} {'mean_cov':>9}"]
    print("\n".join(lines), flush=True)
    g = torch.Generator(device="cpu").manual_seed(3)
    for order in ORDERS:
        with contextlib.redirect_stdout(io.StringIO()):
            pl = cem_planner(num_dof=ND, num_batch=B, num_steps=T, timestep=0.05, maxiter_cem=1, num_elite=ELITE, w_pos=20.0,
                             w_rot=3.0, w_col=80.0, maxiter_projection=10, device=dev, bernstein_order=order)
        pl.cache_normal_draws = False                                   # the draws are part of the sampling stage
        nv, k = pl.nvar, pl.ellite_num
        mean0, cov0 = torch.zeros(nv, device=dev), 10 * torch.eye(nv, device=dev)
        key = jax_prng.split(pl.key)[0]
        q0 = torch.tensor(np.tile([1.5, -1.8, 1.75, -1.25, -1.6, 0.0], 2), dtype=torch.float32, device=dev)
        zero = torch.zeros(ND, device=dev)
        st = torch.cat([q0, zero, zero, zero, zero]).unsqueeze(0).expand(B, 5 * ND).contiguous()
        xi, _ = pl.compute_xi_samples(key, mean0, cov0)
        t_s = timed(lambda: pl.compute_xi_samples(key, mean0, cov0))
        t_p = timed(lambda: pl._project(xi, st, True))
        cost4 = (torch.rand(B, 4, generator=g) * 50).to(dev)
        t_e = timed(lambda: pl._argsort_topk(cost4, 4, B, k, xi))        # what cem_iter runs on one GPU (_select_elites)
        xe, _, ce = pl._argsort_topk(cost4, 4, B, k, xi)
        t_m = timed(lambda: pl.compute_mean_cov(ce, mean0, cov0, xe))
        row = f"{order:>5} {nv:>4} {t_s:9.1f} {t_p:9.1f} {t_e:9.1f} {t_m:9.1f}"
        print(row, flush=True)
        lines.append(row)
        pl.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
