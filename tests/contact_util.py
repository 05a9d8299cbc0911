"""Contact states and the checks of the contact outputs of cemk_step_states_contacts against the float64 oracle, shared by
tests/test_emu_step_contacts.py (CPU emulation) and tests/test_gpu_step_contacts.py.  Test infrastructure."""
import ctypes as C
import os
import subprocess

import numpy as np

from conftest import Q0, ROOT, planner_inputs

COL_TOL = 1e-5          # the teacher-forced collision tolerance of test_gpu_step.py (dist, and here pos and normal)

_SRC = os.path.join(ROOT, "tests", "oracle_constraint.c")
_DEPS = [_SRC, os.path.join(ROOT, "oracle", "mjstep.c")]
_LIB = None


def _constraint_lib():
    """tests/oracle_constraint.c (the float64 oracle plus oracle_forward_constraint), built like the oracle's f64 library."""
    global _LIB
    if _LIB is None:
        out = os.path.join(ROOT, "tests", "_emu_build", "liboracle_constraint.so")
        if not (os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in _DEPS)):
            os.makedirs(os.path.dirname(out), exist_ok=True)
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
            subprocess.run([cc, "-O2", "-fPIC", "-shared", "-fopenmp", "-o", out, _SRC, "-lm"], check=True, capture_output=True)
        _LIB = C.CDLL(out)
    return _LIB


def forward_constraint(oracle64, qpos, qvel, warm, qacc_at=None):
    """One float64 ``mjx.forward`` of `oracle64`'s model with the constraint part of its Data at the accepted qacc, or at
    ``qacc_at`` [nv] when given (oracle_forward_constraint): qacc, per slot con_dist / con_pos / con_frame [ncon, 9] /
    con_force [ncon, 3] (contact frame, decoded pyramid), efc_force [nefc] (limit rows, then four rows per active slot in
    slot order), qfrc_constraint [nv], nlim."""
    from oracle.oracle import MAXCON, MAXJ
    mc = oracle64.mc
    lib = _constraint_lib()
    assert lib.oracle_sizeof_model() == C.sizeof(oracle64.m)
    f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    qpos, qvel, warm = f64(qpos), f64(qvel), np.zeros(mc.nv) if warm is None else f64(warm)
    out = dict(qacc=np.zeros(mc.nv), con_dist=np.zeros(mc.ncon), con_pos=np.zeros((mc.ncon, 3)), con_frame=np.zeros((mc.ncon, 9)),
               efc_force=np.zeros(MAXJ + 4 * MAXCON), qfrc_constraint=np.zeros(mc.nv), con_force=np.zeros((mc.ncon, 3)))
    nefc, nlim = C.c_int(0), C.c_int(0)
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    qa = None if qacc_at is None else f64(qacc_at)
    lib.oracle_forward_constraint(C.byref(oracle64.m), p(qpos), p(qvel), p(warm), p(qa), p(out["qacc"]), p(out["con_dist"]),
                                  p(out["con_pos"]), p(out["con_frame"]), p(out["efc_force"]), p(out["qfrc_constraint"]),
                                  p(out["con_force"]), C.byref(nefc), C.byref(nlim))
    out["efc_force"] = out["efc_force"][:nefc.value]
    out["nlim"] = nlim.value
    return out


def harvest_contact_states(oracle64):
    """The teacher-forced contact states of test_gpu_step.py / test_gpu_step_states.py: every 4th step with a robot contact
    of 12 contact-rich planner samples (oracle float64 rollout), qvel[:6] = the commanded velocity of that step."""
    T, B = 100, 64
    td = planner_inputs(T, B, seed=1)[5]
    oth, oep, oer, ocol, oqp, oqa = oracle64.rollout(td, Q0, np.zeros(6), want_state=True)
    has = np.where((ocol < 0).any(axis=(1, 2)))[0]
    warm0 = oracle64.initial_warmstart()
    qps, qvs, wms = [], [], []
    for s in has[:12]:
        qvbox = np.zeros(6)
        for t in range(T):
            qpos = np.concatenate([Q0, oracle64.mc.qpos0[6:]]) if t == 0 else oqp[s, t - 1]
            warm = warm0 if t == 0 else oqa[s, t - 1]
            qvel = np.zeros(12); qvel[6:] = qvbox; qvel[:6] = td[s].reshape(6, T)[:, t]
            qvbox = qvbox + 0.05 * oqa[s, t, 6:]
            if not (ocol[s, t] < 0).any() or t % 4:
                continue
            qps.append(qpos); qvs.append(qvel); wms.append(warm)
    return _r32(qps), _r32(qvs), _r32(wms)


def deep_states(oracle64, n, seed=0, draws=20000):
    """Start states deep in collision: of `draws` random states (arm configurations far around Q0, links through the
    table, the floor, the box and each other; the box anywhere above the floor around the robot), the n with the most
    active contacts (more than the 20 a sample keeps in shared memory for the first few), small random velocities, the
    initial warm start."""
    mc = oracle64.mc
    rng = np.random.default_rng(seed)
    warm0 = oracle64.initial_warmstart()
    cand = []
    for _ in range(draws):
        qpos = np.concatenate([Q0 + rng.uniform(-2.5, 2.5, 6), mc.qpos0[6:]])
        qpos[6:9] = rng.uniform([-0.6, -0.6, -0.05], [0.6, 0.6, 0.6])
        qvel = np.concatenate([rng.uniform(-0.5, 0.5, 6), np.zeros(6)])
        cand.append(((oracle64.forward(qpos, qvel, warm0)["con_dist"] < 0).sum(), qpos, qvel))
    cand.sort(key=lambda c: -c[0])
    return _r32([c[1] for c in cand[:n]]), _r32([c[2] for c in cand[:n]]), _r32([warm0] * n)


def _r32(a):
    return np.array(a, dtype=np.float32).astype(np.float64)       # the states as the kernel sees them


def box_box_slots(mc):
    """The slots of the model's box-box pairs (the free box against a static box)."""
    from manipulator_mujoco_b200.mjcf import GEOM_BOX
    out = set()
    for (g1, g2), a, n in zip(mc.pair_geom, mc.pair_slotadr, mc.pair_nslot):
        if mc.geom_type[g1] == GEOM_BOX and mc.geom_type[g2] == GEOM_BOX:
            out.update(range(a, a + n))
    return out


def _match_box_box(mc, bb, ks, pos, nrm, o):
    """Oracle slot of each kernel contact.  The kernel's box-box manifold (box_box_warp) numbers the points of a pair in
    another order than the oracle and places each one on the other box's face (the positions differ by dist along the
    normal), so a box-box contact is matched to the oracle point of its pair nearest in the plane of the contact."""
    out = ks.copy()
    for j, k in enumerate(ks):
        if k not in bb:
            continue
        pair = [p for p, (a, n) in enumerate(zip(mc.pair_slotadr, mc.pair_nslot)) if a <= k < a + n][0]
        a, n = mc.pair_slotadr[pair], mc.pair_nslot[pair]
        cands = [c for c in range(a, a + n) if o["con_dist"][c] < 0]
        tang = lambda c: np.linalg.norm((pos[j] - o["con_pos"][c]) - np.dot(pos[j] - o["con_pos"][c], nrm[j]) * nrm[j])
        out[j] = min(cands, key=tang)
    return out


def check_against_oracle(oracle64, qpos, qvel, warm, got, mu, nrm_tol=100 * COL_TOL, pos_tol=COL_TOL, forces=True):
    """Every state: the slot set, dist / pos / normal of each contact, and the forces and qfrc_constraint against the oracle
    evaluated at the kernel's own qacc (forces=False: not the forces, for states whose contact positions are ill-conditioned);
    physics invariants on every contact.  got: numpy qacc [N, 12], flags [N], ncon [N],
    slot [N, 48], rec [N, 48, 12], qfrc [N, 12].  Returns the number of contacts checked."""
    mc = oracle64.mc
    bb = box_box_slots(mc)
    ncheck = 0
    for i in range(len(qpos)):
        o = forward_constraint(oracle64, qpos[i], qvel[i], warm[i], qacc_at=got["qacc"][i].astype(np.float64))
        nc = int(got["ncon"][i])
        slots, rec = got["slot"][i], got["rec"][i].astype(np.float64)
        assert (slots[nc:] == -1).all() and (rec[nc:] == 0).all(), i
        ks = slots[:nc]
        assert (np.diff(ks) > 0).all(), (i, ks)
        active = set(np.nonzero(o["con_dist"] < 0)[0])
        # a slot within the collision tolerance of dist = 0 may fall on either side in float32
        edge = set(np.nonzero(np.abs(o["con_dist"]) < COL_TOL)[0])
        if not got["flags"][i] & 1:
            assert set(ks) ^ active <= edge, (i, sorted(set(ks) ^ active))
        dist, pos, nrm, frc = rec[:nc, 0], rec[:nc, 1:4], rec[:nc, 4:7], rec[:nc, 7:10]
        # invariants: listed slots are penetrating, forces inside the friction pyramid
        assert (dist < 0).all(), i
        assert (frc[:, 0] >= 0).all(), i
        assert (np.abs(frc[:, 1]) + np.abs(frc[:, 2]) <= mu * frc[:, 0] * (1 + 1e-5) + 1e-6).all(), i
        om = _match_box_box(mc, bb, ks, pos, nrm, o)
        isbb = np.array([k in bb for k in ks], dtype=bool)
        np.testing.assert_allclose(dist, o["con_dist"][om], rtol=0, atol=COL_TOL)
        # a normal is the unit vector of a difference of float32 points (closest points of capsule axes, box edges): its
        # error is the points' error over their separation (up to 3e-4 on the contact states with the GPU's contracted
        # arithmetic, 6e-5 in the emulation), which is small for deeply interpenetrating geoms, whose closest
        # points (and so contact positions) are then ill-conditioned too, most of all for near-parallel capsule axes, whose
        # closest points slide along the overlap at the same distance (by centimetres, for the same dist): deep states take
        # looser nrm_tol and pos_tol, and their forces, whose Jacobians follow the positions, are not compared
        np.testing.assert_allclose(nrm, o["con_frame"][om, :3], rtol=0, atol=nrm_tol)
        dpos = pos - o["con_pos"][om]
        along = np.einsum("ij,ij->i", dpos, nrm)
        np.testing.assert_allclose(np.where(isbb[:, None], dpos - along[:, None] * nrm, dpos), 0, rtol=0, atol=pos_tol)
        assert (np.abs(along[isbb]) <= np.abs(dist[isbb]) + pos_tol).all(), i
        # forces at the same qacc: f_r = -D_r (J_r qacc - aref_r) with J, D, aref from float32 geometry.  The collision
        # tolerance moves aref by k imp COL_TOL and a Jacobian entry by |J| COL_TOL (lever arm), so a row force by D times
        # that; the bound below is that sensitivity over the rows, estimated from the oracle's own forces.
        ncheck += nc
        if not forces:
            continue
        scale = max(1.0, np.abs(o["efc_force"]).max() if len(o["efc_force"]) else 0.0)
        np.testing.assert_allclose(frc, o["con_force"][om], rtol=0, atol=2e-3 * scale, err_msg=str(i))
        np.testing.assert_allclose(got["qfrc"][i], o["qfrc_constraint"], rtol=0, atol=2e-3 * scale, err_msg=str(i))
    return ncheck
