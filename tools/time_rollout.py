"""Time the fused rollout+cost kernel alone (GPU box only).

usage: python tools/time_rollout.py [--batch 4096] [--horizon 100] [--reps 5]
Also checks that every timed run returns costs bit-identical to the warm-up run's.
"""
import argparse
import contextlib
import io
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from manipulator_mujoco_b200 import cem_planner  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", default="4096")
    ap.add_argument("--horizon", type=int, default=100)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    for B in [int(b) for b in args.batch.split(",")]:
        with contextlib.redirect_stdout(io.StringIO()):
            pl = cem_planner(num_dof=6, num_batch=B, num_steps=args.horizon, timestep=0.05, maxiter_cem=1, num_elite=0.05, w_pos=20.0,
                             w_rot=3.0, w_col=80.0, maxiter_projection=10, device=dev)
        z6 = torch.zeros(6, device=dev)
        q0 = torch.tensor([1.5, -1.8, 1.75, -1.25, -1.6, 0.0], device=dev)
        tp = torch.tensor([-0.3, 0.3, 0.4], device=dev)
        tr = torch.tensor([0.0, 0.7071, -0.7071, 0.0], device=dev)
        state_term = torch.cat([q0, z6, z6, z6, z6]).unsqueeze(0).expand(B, 30).contiguous()
        xi, _ = pl.compute_xi_samples(pl.key, torch.zeros(pl.nvar, device=dev), 10 * torch.eye(pl.nvar, device=dev))
        _, thetadot = pl._project(xi, state_term, True)
        for _ in range(2):
            out = pl._rollout(thetadot, q0, z6, tp, tr, False)
        ref = out[1].detach().cpu().numpy().view(np.int32).copy()
        ms, same = [], True
        for _ in range(args.reps):
            flush.fill_(1.0)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = pl._rollout(thetadot, q0, z6, tp, tr, False)
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
            same = same and np.array_equal(ref, out[1].detach().cpu().numpy().view(np.int32))
        print(f"B={B} T={args.horizon}: {np.mean(ms):7.3f} ms (min {np.min(ms):.3f})  {B * args.horizon / np.mean(ms) * 1e3:.3e} env-steps/s"
              f"  {'bit-identical' if same else 'RESULTS DIFFER'}", flush=True)
        del pl


if __name__ == "__main__":
    main()
