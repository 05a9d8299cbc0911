"""Timing of per-environment stepping (cemk_step_states / cem_planner.step_batch) on one GPU:
    python tools/time_step_states.py [--out FILE]
1. cemk_step_states against cemk_rollout_cost at 4096 x 100 (bench.py's rollout: the planner's projected samples from the
   snapshot state), alternating in one session: the same step body runs in both, one without the cost and with state rows.
2. One step (T = 1, thetadot NULL: plain mjx.step) of N = 1, 1000, 4096, 16384 perturbed states: time per call, env-steps/s.
3. 1000 states stepped by a loop of jit_step calls (one library handle and one B = 1 rollout per call, float64 Euler on the
   host) against one step_batch call, host wall clock from numpy inputs to results synchronised on the device.
CUDA-event timings are medians of REPS calls with the L2 cache overwritten before every call."""
import argparse
import contextlib
import ctypes as C
import io
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from manipulator_mujoco_b200 import cem_planner, jax_prng  # noqa: E402

Q0 = np.array([1.5, -1.8, 1.75, -1.25, -1.6, 0.0])
REPS = 20


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the table to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_step_states.py needs a CUDA device")
    dev = torch.device("cuda:0")
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)          # 256 MB > the 126 MB L2
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())

    def event_ms(fn):
        flush.fill_(1.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:                                                   # noqa: BLE001 (the table is still valid without it)
        q = torch.cuda.get_device_name(dev) + ", power limit not read"
    lines = [f"# per-environment stepping on one GPU: {q}",
             f"# CUDA events, median of {REPS} calls (alternating where two entries are compared), L2 overwritten before each call"]
    out = lambda s: (print(s, flush=True), lines.append(s))

    B, T = 4096, 100
    with contextlib.redirect_stdout(io.StringIO()):
        pl = cem_planner(num_dof=6, num_batch=B, num_steps=T, timestep=0.05, maxiter_cem=1, num_elite=0.05, w_pos=20.0, w_rot=3.0,
                         w_col=80.0, maxiter_projection=10, device=dev)
    lib, h, st = pl._lib, pl._h, pl._stream()
    km = pl.mjx_model
    key = jax_prng.split(jax_prng.split(pl.key)[0])[0]
    xi, _ = pl.compute_xi_samples(key, torch.zeros(66, device=dev), 10 * torch.eye(66, device=dev))
    zero = torch.zeros(6, device=dev)
    q0 = torch.tensor(Q0, dtype=torch.float32, device=dev)
    state = torch.cat([q0, zero, zero, zero, zero]).unsqueeze(0).expand(B, 30).contiguous()
    _, td = pl._project(xi, state, True)
    tp, tr = torch.tensor([-0.3, -0.3, 0.5], device=dev), torch.tensor([0.0, 1.0, 0.0, 0.0], device=dev)
    theta, cost4 = torch.empty(B, 6 * T, device=dev), torch.empty(B, 4, device=dev)

    def snapshot(n):
        qp = np.tile(np.concatenate([Q0, np.array(km.qpos0[6:13])]), (n, 1))
        qv = np.tile(np.concatenate([np.zeros(6), np.array(km.qvel0[6:12])]), (n, 1))
        wm = np.tile(np.array(km.warm0[:12]), (n, 1))
        return qp, qv, wm

    dv = lambda a: torch.as_tensor(a, dtype=torch.float32, device=dev).contiguous()
    qp, qv, wm = (dv(a) for a in snapshot(B))
    qo, vo, wo = torch.empty_like(qp), torch.empty_like(qv), torch.empty_like(wm)
    roll = lambda: lib.cemk_rollout_cost(h, B, T, p(td), p(q0), p(zero), p(tp), p(tr), 20.0, 3.0, 80.0, p(theta), p(cost4),
                                         None, None, None, None, None, st)
    step = lambda: lib.cemk_step_states(h, B, T, p(qp), p(qv), p(wm), p(td), p(qo), p(vo), p(wo), p(theta), None, None, None,
                                        None, None, st)
    for _ in range(3):
        assert roll() == 0 and step() == 0
    torch.cuda.synchronize()
    tr_, ts_ = [], []
    for _ in range(REPS):
        tr_.append(event_ms(roll)); ts_.append(event_ms(step))
    r, s = np.median(tr_), np.median(ts_)
    out(f"4096 x 100 from the snapshot: cemk_rollout_cost {r:.3f} ms (spread {np.ptp(tr_):.3f}), cemk_step_states {s:.3f} ms "
        f"(spread {np.ptp(ts_):.3f}), ratio {s / r:.4f}; {B * T / s * 1e3:.3e} env-steps/s")

    out(f"{'N':>6} {'T':>3} {'ms/call':>9} {'env-steps/s':>12}")
    rng = np.random.default_rng(0)
    for n in (1, 1000, 4096, 16384):
        a, b, c = snapshot(n)
        a[:, :6] += rng.uniform(-0.4, 0.4, size=(n, 6))
        b[:, :6] = rng.uniform(-0.8, 0.8, size=(n, 6))
        a, b, c = dv(a), dv(b), dv(c)
        o1, o2, o3 = torch.empty_like(a), torch.empty_like(b), torch.empty_like(c)
        one = lambda: lib.cemk_step_states(h, n, 1, p(a), p(b), p(c), None, p(o1), p(o2), p(o3), None, None, None, None, None, None, st)
        for _ in range(3):
            assert one() == 0
        t = float(np.median([event_ms(one) for _ in range(REPS)]))
        out(f"{n:>6} {1:>3} {t:9.4f} {n / t * 1e3:12.3e}")

    n = 1000
    a, b, c = snapshot(n)
    a[:, :6] += rng.uniform(-0.4, 0.4, size=(n, 6))
    b[:, :6] = rng.uniform(-0.8, 0.8, size=(n, 6))
    pl.jit_step(km, dict(qpos=a[0], qvel=b[0], qacc_warmstart=c[0]))
    pl.step_batch(a, b, c)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(n):
        pl.jit_step(km, dict(qpos=a[i], qvel=b[i], qacc_warmstart=c[i]))
    t_loop = time.perf_counter() - t0
    tb = []
    for _ in range(5):
        t0 = time.perf_counter()
        res = pl.step_batch(a, b, c)
        torch.cuda.synchronize()
        tb.append(time.perf_counter() - t0)
    assert res["qpos"].shape == (n, 13)
    t_batch = float(np.median(tb))
    out(f"1000 states, one step each: jit_step loop {t_loop * 1e3:.1f} ms, step_batch {t_batch * 1e3:.3f} ms "
        f"(host wall clock, median of 5), {t_loop / t_batch:.0f}x")
    pl.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
