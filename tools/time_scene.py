"""What scene and start records cost, on one GPU, each pair of calls alternating in one session:
    python tools/time_scene.py [--out FILE]
  * planner rollout, B = 4096, T = 100: cemk_rollout_cost_scene with a shared moved scene and a start record against
    cemk_rollout_cost (no record);
  * a closed-loop tick, B = 1000, T = 16, 3 CEM iterations: compute_cem(scene=, state=) against compute_cem (CUDA graphs on,
    host clock around the synchronising call);
  * step_batch, N = 16 384, T = 1: one scene per environment (cemk_step_states_scene, stride 160) against none.
CUDA events for the kernels (median of REPS rounds, the L2 cache overwritten before every call)."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from manipulator_mujoco_b200 import cem_planner  # noqa: E402
from manipulator_mujoco_b200.planner import _ptr  # noqa: E402

Q0 = np.array([1.5, -1.8, 1.75, -1.25, -1.6, 0.0])
TP, TR = np.array([-0.3, -0.3, 0.5]), np.array([0.0, 1.0, 0.0, 0.0])
REPS = 30
KW = dict(num_dof=6, timestep=0.05, num_elite=0.05, w_pos=20.0, w_rot=3.0, w_col=80.0, maxiter_projection=10)


def timed(calls, reps, flush=None):
    times = {k: [] for k in calls}
    for rnd in range(reps + 3):
        for k, fn in calls.items():
            if flush is not None:
                flush.fill_(1.0)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            assert fn() == 0, k
            b.record()
            torch.cuda.synchronize()
            if rnd >= 3:
                times[k].append(a.elapsed_time(b))
    return times


def report(lines, times, base, unit="ms"):
    for k, v in times.items():
        med = np.median(v)
        lines.append(f"  {k:28s} {med:.4f} {unit} (spread {np.percentile(v, 90) - np.percentile(v, 10):.4f}), ratio {med / np.median(times[base]):.4f}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the result lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_scene.py needs a CUDA device")
    dev = torch.device("cuda:0")
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)          # 256 MB > the 126 MB L2
    rng = np.random.default_rng(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    lines = [f"# one GPU: {smi}; CUDA events unless noted, median of {REPS} alternating rounds"]

    # (1) planner rollout 4096 x 100
    B, T = 4096, 100
    pl = cem_planner(num_batch=B, num_steps=T, maxiter_cem=1, **KW)
    moves = {"obstacle_1": (np.array([-0.1, -0.25, 0.55]), np.array([0.9, 0.2, -0.3, 0.25])),
             "obstacle_3": (np.array([0.3, -0.35, 0.3]), np.array([0.5, 0.5, -0.5, 0.5]))}
    scene = pl.make_scene(moves)
    state = dict(qpos=np.concatenate([Q0, np.array(pl.mjx_model.qpos0[6:13])]), qvel=np.zeros(12),
                 qacc_warmstart=np.array(pl.mjx_model.warm0[:12]))
    start = torch.as_tensor(pl.start_record(state), device=dev)
    xi = torch.randn(B, pl.nvar, device=dev) * 3
    st_term = torch.zeros(B, 30, device=dev)
    st_term[:, :6] = torch.as_tensor(Q0, dtype=torch.float32, device=dev)
    _, td = pl._project(xi, st_term, True)
    q0, v0 = torch.as_tensor(Q0, dtype=torch.float32, device=dev), torch.zeros(6, device=dev)
    tp, tr = torch.as_tensor(TP, dtype=torch.float32, device=dev), torch.as_tensor(TR, dtype=torch.float32, device=dev)
    theta, cost4 = torch.empty(B, 6 * T, device=dev), torch.empty(B, 4, device=dev)
    flags = torch.empty(B, dtype=torch.int32, device=dev)
    common = [pl._h, B, T, _ptr(td), _ptr(q0), _ptr(v0), _ptr(tp), _ptr(tr), 20.0, 3.0, 80.0, _ptr(theta), _ptr(cost4), None, None, None,
              None, _ptr(flags)]
    st = pl._stream()
    times = timed({"rollout_cost (no record)": lambda: pl._lib.cemk_rollout_cost(*common, st),
                   "rollout_cost_scene (scene+start)": lambda: pl._lib.cemk_rollout_cost_scene(*common, _ptr(scene), 0, _ptr(start), st)},
                  REPS, flush)
    lines.append(f"planner rollout B = {B}, T = {T} (one launch):")
    report(lines, times, "rollout_cost (no record)")
    pl.close()

    # (2) closed-loop tick, B = 1000, T = 16, 3 iterations (host clock around compute_cem, which synchronises)
    pa = cem_planner(num_batch=1000, num_steps=16, maxiter_cem=3, **KW)
    pb = cem_planner(num_batch=1000, num_steps=16, maxiter_cem=3, **KW)
    scene_h = pb.make_scene(moves).cpu().numpy()
    ticks = {"tick (no record)": [], "tick (scene+state)": []}
    xa = xb = np.zeros(pa.nvar)
    for rnd in range(REPS * 4 + 3):
        t0 = time.perf_counter()
        xa = pa.compute_cem(xa, Q0, np.zeros(6), np.zeros(6), TP, TR)[6]
        t1 = time.perf_counter()
        xb = pb.compute_cem(xb, Q0, np.zeros(6), np.zeros(6), TP, TR, scene=scene_h, state=state)[6]
        t2 = time.perf_counter()
        if rnd >= 3:
            ticks["tick (no record)"].append((t1 - t0) * 1e3)
            ticks["tick (scene+state)"].append((t2 - t1) * 1e3)
    lines.append(f"closed-loop tick B = 1000, T = 16, 3 iterations (CUDA graph, host clock, {REPS * 4} alternating ticks):")
    report(lines, ticks, "tick (no record)")
    pa.close()
    pb.close()

    # (3) step_batch, N = 16 384, T = 1, one scene per environment
    N = 16384
    ps = cem_planner(num_batch=100, num_steps=16, maxiter_cem=1, **KW)
    km = ps.mjx_model
    qpos = np.tile(np.concatenate([Q0, np.array(km.qpos0[6:13])]), (N, 1))
    qpos[:, :6] += rng.uniform(-0.6, 0.6, size=(N, 6))
    qvel, warm = np.zeros((N, 12)), np.tile(np.array(km.warm0[:12]), (N, 1))
    scenes = ps.make_scene({"obstacle_1": (np.array([-0.2, -0.15, 0.5]) + rng.uniform(-0.1, 0.1, size=(N, 3)), rng.normal(size=(N, 4)))})
    out = ps.step_batch(qpos, qvel, warm, thetadot=rng.uniform(-0.8, 0.8, size=(N, 6 * 8)), scene=scenes)
    qp, qv, wm = (out[k].contiguous() for k in ("qpos", "qvel", "qacc_warmstart"))
    qo, vo, wo = torch.empty_like(qp), torch.empty_like(qv), torch.empty_like(wm)
    fl = torch.empty(N, dtype=torch.int32, device=dev)
    sst = [_ptr(x) for x in (qp, qv, wm)] + [None] + [_ptr(x) for x in (qo, vo, wo)] + [None] * 5 + [_ptr(fl)]
    st = ps._stream()
    times = timed({"step_states (no record)": lambda: ps._lib.cemk_step_states(ps._h, N, 1, *sst, st),
                   "step_states_scene (per env)": lambda: ps._lib.cemk_step_states_scene(ps._h, N, 1, *sst, None, None, None, None, None,
                                                                                        _ptr(scenes), 160, st)},
                  REPS, flush)
    lines.append(f"step_batch N = {N}, T = 1, one scene per environment (one launch):")
    report(lines, times, "step_states (no record)")
    ps.close()
    print("\n".join(lines))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
