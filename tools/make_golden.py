"""Generate the committed golden fixtures under tests/golden/ from the reference checkout.

Needs a checkout of the upstream project alinjar1996/manipulator_mujoco; the tests only read what this writes:
    MANIPULATOR_MUJOCO_REFERENCE=<checkout> python tools/make_golden.py
Produces
  bernstein.npz        P, Pdot, Pddot of the reference's own bernstein_coeff_ordern_new for the
                       horizons used by the tests (imported from the reference, not restated);
  closed_loop_kat.npz  the recorded closed-loop run of the reference (data/theta.csv, data/thetadot.csv:
                       897 ticks of the C-MuJoCo plant at dt = 0.05) used as the smooth-dynamics
                       known-answer test, plus the per-tick best costs of the same run (data/cost_c.csv, cost_g.csv,
                       cost_r.csv, costs.csv) that pin the capsule-box far-field semantics;
  scene_ids.json       geom ids recorded in view_traj_mjx.py:54 and the FK pins of SURVEY.md section 4.
"""
import json
import os
import sys

import numpy as np

REF = os.path.join(os.environ["MANIPULATOR_MUJOCO_REFERENCE"], "sampling_based_planner")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")


def main():
    sys.path.insert(0, REF)
    import bernstein_coeff_ordern_arbitinterval as ref_b
    import bernstein_coeff_order10_arbitinterval as ref_b10
    os.makedirs(OUT, exist_ok=True)
    out = {}
    for T, dt in [(16, 0.05), (100, 0.05), (10, 0.04), (50, 0.05)]:
        tt = np.linspace(0, T * dt, T).reshape(T, 1)
        P, Pd, Pdd = ref_b.bernstein_coeff_ordern_new(10, tt[0], tt[-1], tt)
        out[f"P_{T}_{dt}"], out[f"Pdot_{T}_{dt}"], out[f"Pddot_{T}_{dt}"] = P, Pd, Pdd
        P10, Pd10, Pdd10 = ref_b10.bernstein_coeff_order10_new(10, tt[0], tt[-1], tt)
        out[f"P10_{T}_{dt}"], out[f"Pdot10_{T}_{dt}"], out[f"Pddot10_{T}_{dt}"] = P10, Pd10, Pdd10
    # other orders (SURVEY 8 f.4: order-n sweep) from the same reference function
    for n in (5, 8, 12, 15):
        T, dt = 16, 0.05
        tt = np.linspace(0, T * dt, T).reshape(T, 1)
        P, Pd, Pdd = ref_b.bernstein_coeff_ordern_new(n, tt[0], tt[-1], tt)
        out[f"P_n{n}"], out[f"Pdot_n{n}"], out[f"Pddot_n{n}"] = P, Pd, Pdd
    np.savez_compressed(os.path.join(OUT, "bernstein.npz"), **out)
    theta = np.loadtxt(os.path.join(REF, "data", "theta.csv"), delimiter=",")
    thetadot = np.loadtxt(os.path.join(REF, "data", "thetadot.csv"), delimiter=",")
    rec = {n: np.loadtxt(os.path.join(REF, "data", n + ".csv"), delimiter=",") for n in ("cost_c", "cost_g", "cost_r", "costs")}
    np.savez_compressed(os.path.join(OUT, "closed_loop_kat.npz"), theta=theta, thetadot=thetadot.astype(np.float32), **rec)
    with open(os.path.join(OUT, "scene_ids.json"), "w") as f:
        json.dump({
            "robot_geom_ids": [33, 7, 12, 13, 18, 19, 23, 27, 28, 30],          # view_traj_mjx.py:54
            "ncon": 215, "nrobot_slots": 187, "npair": 114, "nq": 13, "nv": 12, "nbody": 18, "ngeom": 42,
            "tcp_at_zero": [0.017, 0.817, 0.624],
            "init_pos": [1.5, -1.8, 1.75, -1.25, -1.6, 0],
            "tcp_at_init_pos": [0.04936, -0.10358, 0.90439],
            "xquat_hande_at_init_pos": [0.08889, 0.72357, 0.67677, 0.10259],
        }, f, indent=1)
    print("wrote", sorted(os.listdir(OUT)))


if __name__ == "__main__":
    main()
