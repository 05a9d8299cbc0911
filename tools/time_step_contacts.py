"""What the contact outputs cost: one step (T = 1) of 16 384 states in contact on one GPU,
    python tools/time_step_contacts.py [--parent-lib PATH] [--out FILE]
timed as cemk_step_states and as cemk_step_states_contacts, and, with --parent-lib (a libcemk.so built from the parent
commit), as that library's cemk_step_states, the calls alternating in one session.  CUDA events, median of REPS rounds,
the L2 cache overwritten before every call."""
import argparse
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from manipulator_mujoco_b200 import cem_planner  # noqa: E402
from manipulator_mujoco_b200.planner import _ptr  # noqa: E402

Q0 = np.array([1.5, -1.8, 1.75, -1.25, -1.6, 0.0])
N, REPS = 16384, 30


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", default=None, help="libcemk.so of the parent commit, timed alternately with this one")
    ap.add_argument("--out", default=None, help="also write the result lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_step_contacts.py needs a CUDA device")
    dev = torch.device("cuda:0")
    pl = cem_planner(num_dof=6, num_batch=100, num_steps=16, timestep=0.05, maxiter_cem=1, num_elite=0.05,
                     w_pos=20.0, w_rot=3.0, w_col=80.0, maxiter_projection=10)
    km = pl.mjx_model
    rng = np.random.default_rng(0)
    qpos = np.tile(np.concatenate([Q0, np.array(km.qpos0[6:13])]), (N, 1))
    qpos[:, :6] += rng.uniform(-0.6, 0.6, size=(N, 6))
    qvel = np.tile(np.concatenate([np.zeros(6), np.array(km.qvel0[6:12])]), (N, 1))
    warm = np.tile(np.array(km.warm0[:12]), (N, 1))
    # eight planner-like steps first: the box lands on the table (four contacts) and some arms touch something
    out = pl.step_batch(qpos, qvel, warm, thetadot=rng.uniform(-0.8, 0.8, size=(N, 6 * 8)))
    qp, qv, wm = (out[k].contiguous() for k in ("qpos", "qvel", "qacc_warmstart"))
    qo, vo, wo = torch.empty_like(qp), torch.empty_like(qv), torch.empty_like(wm)
    key = torch.as_tensor(pl._key_slot, dtype=torch.int32, device=dev)
    qfrc, ncon = torch.empty(N, 12, device=dev), torch.empty(N, dtype=torch.int32, device=dev)
    slot, rec = torch.empty(N, 48, dtype=torch.int32, device=dev), torch.empty(N, 48, 12, device=dev)
    st = pl._stream()
    state = [_ptr(x) for x in (qp, qv, wm)] + [None] + [_ptr(x) for x in (qo, vo, wo)] + [None] * 6

    calls = {
        "step_states": lambda: pl._lib.cemk_step_states(pl._h, N, 1, *state, st),
        "step_states_contacts": lambda: pl._lib.cemk_step_states_contacts(pl._h, N, 1, *state, _ptr(key), _ptr(qfrc), _ptr(ncon),
                                                                          _ptr(slot), _ptr(rec), st),
    }
    if args.parent_lib:
        par = C.CDLL(args.parent_lib)
        vp = C.c_void_p
        par.cemk_create.argtypes, par.cemk_create.restype = [vp, C.c_int, C.c_int, C.POINTER(vp)], C.c_int
        par.cemk_step_states.argtypes, par.cemk_step_states.restype = [vp, C.c_int, C.c_int] + [vp] * 14, C.c_int
        ph = vp()
        assert par.cemk_create(C.byref(km), C.sizeof(km), 0, C.byref(ph)) == 0
        calls["parent step_states"] = lambda: par.cemk_step_states(ph, N, 1, *state, st)

    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)          # 256 MB > the 126 MB L2
    times = {k: [] for k in calls}
    for rnd in range(REPS + 3):
        for k, fn in calls.items():
            flush.fill_(1.0)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            assert fn() == 0, k
            b.record()
            torch.cuda.synchronize()
            if rnd >= 3:
                times[k].append(a.elapsed_time(b))
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    lines = [f"# one step (T = 1) of {N} states (perturbed arms, 8 steps after the snapshot) on one GPU: {smi}",
             f"# CUDA events, median of {REPS} alternating rounds, L2 overwritten before each call"]
    base = np.median(times["step_states"])
    for k, v in times.items():
        med = np.median(v)
        lines.append(f"{k:22s} {med:.4f} ms (spread {np.percentile(v, 90) - np.percentile(v, 10):.4f}), "
                     f"ratio to step_states {med / base:.4f}, {N / med * 1e3:.3e} env-steps/s")
    lines.append(f"contacts per state: mean {ncon.float().mean().item():.2f}, max {int(ncon.max().item())}")
    print("\n".join(lines))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    pl.close()


if __name__ == "__main__":
    main()
