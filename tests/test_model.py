"""MJCF compiler + model tables: ids / counts pinned by the reference, consistency of derived tables."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN
from manipulator_mujoco_b200 import kmodel as KM
from manipulator_mujoco_b200.mjcf import compile_mjcf, host_kinematics, host_mass_matrix

IDS = json.load(open(os.path.join(GOLDEN, "scene_ids.json")))
# checkout of the upstream project alinjar1996/manipulator_mujoco: its MJCF files are not part of this repository, so the
# tests that compile them run only where MANIPULATOR_MUJOCO_REFERENCE names such a checkout
REFERENCE = os.environ.get("MANIPULATOR_MUJOCO_REFERENCE", "")
REF_XML = os.path.join(REFERENCE, "sampling_based_planner", "ur5e_hande_mjx", "scene.xml")
NO_REFERENCE = "needs the upstream checkout named by MANIPULATOR_MUJOCO_REFERENCE"


def test_counts_and_ids(mc):
    assert [mc.geom_id(f"robot_{i}") for i in range(10)] == IDS["robot_geom_ids"]      # view_traj_mjx.py:54
    assert (mc.nq, mc.nv, mc.nbody, mc.ngeom) == (IDS["nq"], IDS["nv"], IDS["nbody"], IDS["ngeom"])
    assert mc.ncon == IDS["ncon"] and len(mc.pair_geom) == IDS["npair"]
    from oracle.oracle import robot_slot_mask
    assert robot_slot_mask(mc).sum() == IDS["nrobot_slots"]                             # mask.sum() of mjx_planner.py:115
    assert mc.opt["iterations"] == 1 and mc.opt["ls_iterations"] == 5 and mc.opt["eulerdamp"] == 0


def test_forward_kinematics_pins(mc):
    tcp = mc.site_id("tcp")
    q = mc.qpos0.copy()
    xpos, xquat, xmat = host_kinematics(mc, q)
    b = mc.site_body[tcp]
    np.testing.assert_allclose(xpos[b] + xmat[b] @ mc.site_pos[tcp], IDS["tcp_at_zero"], atol=1e-9)
    q[:6] = IDS["init_pos"]
    xpos, xquat, xmat = host_kinematics(mc, q)
    np.testing.assert_allclose(xpos[b] + xmat[b] @ mc.site_pos[tcp], IDS["tcp_at_init_pos"], atol=1e-5)
    np.testing.assert_allclose(xquat[mc.body_id("hande")], IDS["xquat_hande_at_init_pos"], atol=1e-5)


@pytest.mark.skipif(not REFERENCE or not os.path.exists(REF_XML), reason=NO_REFERENCE)
def test_packaged_constants_match_the_xml(mc):
    fresh = compile_mjcf(REF_XML)
    for k, v in fresh.d.items():
        if k not in mc.d:
            # fields of the loader extensions (equalities, tendons, actuators, keyframes, unknown pair types): scene A has
            # none of them, and the packaged table predates them
            assert (v == 0 if isinstance(v, int) else len(v) == 0), k
        elif isinstance(v, np.ndarray):
            np.testing.assert_allclose(v, mc.d[k], rtol=0, atol=1e-12, err_msg=k)
        elif k != "xml":
            assert v == mc.d[k], k


def test_hande_inertia_from_geoms(mc):
    """No <inertial> on `hande`: mass from coupler + hande meshes + robot_0 capsule at density 1000 (SURVEY A.2)."""
    m = mc.body_mass[mc.body_id("hande")]
    cap = 1000 * (np.pi * 0.04 ** 2 * 0.14 + 4 / 3 * np.pi * 0.04 ** 3)
    assert abs(cap - 0.9718) < 1e-3
    assert 1.30 < m < 1.40 and m > cap


def test_mass_matrix_spd_and_invweights(mc):
    q = mc.qpos0.copy()
    q[:6] = IDS["init_pos"]
    M, _, _ = host_mass_matrix(mc, q)
    np.testing.assert_allclose(M, M.T, atol=1e-12)
    assert np.linalg.eigvalsh(M).min() > 0
    assert abs(mc.body_invweight0[mc.body_id("target_0"), 0] - 1 / 0.064) < 1e-9      # free box: 1/m
    assert np.all(mc.dof_invweight0 > 0)


def test_kmodel_flattening(mc):
    km, info = KM.build_kmodel(mc, 0.05)
    assert km.nl == 6 and km.ncap == 10 and km.nsbox == 6 and km.has_box == 1
    assert km.nrpair == 107 and km.nbpair == 7 and km.nslot_robot == 187
    # merged link masses == sum of the bodies welded to each link
    masses = [km.l_inertia[i][6] for i in range(6)]
    assert abs(sum(masses) - mc.body_mass[3:12].sum()) < 1e-5
    # the pass-major pair table covers every robot slot exactly once
    seen = np.zeros(187, dtype=int)
    for e in range(KM.MAXRPAIR):
        x = km.rp[e]
        ty, a, b, sl = (x & 15) - 1, (x >> 4) & 15, (x >> 8) & 15, x >> 16
        if ty == KM.KP_NONE:
            continue
        n = 1 if ty == KM.KP_CAP_CAP else 2
        seen[sl:sl + n] += 1
        if ty == KM.KP_CAP_BOX:                       # pass = box, lane = capsule
            assert e // KM.LANE_GROUP == b and e % KM.LANE_GROUP == a and e // KM.LANE_GROUP < km.ncbpass
        else:
            assert e // KM.LANE_GROUP >= km.ncbpass
    assert (seen == 1).all()
    assert km.ncbpass == 7
    assert C.sizeof(km) % 4 == 0


def test_unsupported_models_are_refused(mc):
    import copy
    bad = copy.deepcopy(mc)
    bad.d["opt"] = dict(mc.opt, iterations=4)
    with pytest.raises(NotImplementedError):
        KM.build_kmodel(bad, 0.05)


class _MockMjModel:
    """An object with mujoco.MjModel's attribute names (the subset ModelConsts.from_mjmodel reads), filled from a compiled
    ModelConsts: stands in for MuJoCo, which cannot be installed here."""

    def __init__(self, mc):
        import types
        n = types.SimpleNamespace
        self.nq, self.nv, self.nbody, self.njnt, self.ngeom, self.nsite = mc.nq, mc.nv, mc.nbody, mc.njnt, mc.ngeom, len(mc.site_names)
        self.body_parentid, self.body_pos, self.body_quat, self.body_mass, self.body_ipos = mc.body_parent, mc.body_pos, mc.body_quat, mc.body_mass, mc.body_ipos
        # MuJoCo stores principal inertias + their frame: diagonalise our full tensors
        iq, diag = [], []
        for I in mc.body_inertia:
            w, V = np.linalg.eigh(I)
            if np.linalg.det(V) < 0:
                V[:, 0] = -V[:, 0]
            tr = np.trace(V)                                      # rotation matrix -> quaternion (w, x, y, z)
            qw = np.sqrt(max(0.0, 1 + tr)) / 2
            if qw > 1e-6:
                q = np.array([qw, (V[2, 1] - V[1, 2]) / (4 * qw), (V[0, 2] - V[2, 0]) / (4 * qw), (V[1, 0] - V[0, 1]) / (4 * qw)])
            else:                                                 # 180 degree turns: fall back to the axis with the largest diagonal
                i = int(np.argmax(np.diag(V))); j, k = (i + 1) % 3, (i + 2) % 3
                s = np.sqrt(max(0.0, 1 + V[i, i] - V[j, j] - V[k, k])) * 2
                q = np.zeros(4); q[1 + i] = s / 4; q[1 + j] = (V[j, i] + V[i, j]) / s; q[1 + k] = (V[k, i] + V[i, k]) / s; q[0] = (V[k, j] - V[j, k]) / s
            iq.append(q / np.linalg.norm(q)); diag.append(w)
        self.body_iquat, self.body_inertia = np.array(iq), np.array(diag)
        self.body_gravcomp, self.body_weldid, self.body_rootid = mc.body_gravcomp, mc.body_weldid, mc.body_rootid
        self.body_jntadr, self.body_dofadr, self.body_dofnum = mc.body_jntadr, mc.body_dofadr, mc.body_dofnum
        self.body_jntnum = (mc.body_jntadr >= 0).astype(np.int32)
        self.body_invweight0 = mc.body_invweight0
        self.jnt_type, self.jnt_bodyid, self.jnt_axis, self.jnt_pos, self.jnt_range = mc.jnt_type, mc.jnt_body, mc.jnt_axis, mc.jnt_pos, mc.jnt_range
        self.jnt_limited, self.jnt_margin, self.jnt_qposadr, self.jnt_dofadr = mc.jnt_limited, mc.jnt_margin, mc.jnt_qposadr, mc.jnt_dofadr
        arm, damp = np.zeros(mc.nv), np.zeros(mc.nv)
        for j in range(mc.njnt):
            w = 6 if mc.jnt_type[j] == 0 else 1
            arm[mc.jnt_dofadr[j]:mc.jnt_dofadr[j] + w] = mc.jnt_armature[j]
            damp[mc.jnt_dofadr[j]:mc.jnt_dofadr[j] + w] = mc.jnt_damping[j]
        self.dof_armature, self.dof_damping, self.dof_invweight0 = arm, damp, mc.dof_invweight0
        self.geom_type, self.geom_bodyid, self.geom_pos, self.geom_quat, self.geom_size = mc.geom_type, mc.geom_body, mc.geom_pos, mc.geom_quat, mc.geom_size
        self.geom_friction, self.geom_solref, self.geom_solimp, self.geom_margin, self.geom_condim = mc.geom_friction, mc.geom_solref, mc.geom_solimp, mc.geom_margin, mc.geom_condim
        self.geom_contype = mc.geom_collides.copy()
        self.geom_conaffinity = mc.geom_collides.copy()
        self.site_bodyid, self.site_pos = mc.site_body, mc.site_pos
        self.qpos0 = mc.qpos0
        self.exclude_signature = np.zeros(0, dtype=np.int64)
        o = mc.opt
        self.opt = n(timestep=o["timestep"], iterations=o["iterations"], ls_iterations=o["ls_iterations"], tolerance=o["tolerance"],
                     ls_tolerance=o["ls_tolerance"], impratio=o["impratio"], gravity=np.array(o["gravity"]), integrator=0,
                     disableflags=((1 << 14) if not o.get("eulerdamp", 1) else 0) | ((1 << 10) if not o.get("actuation", 1) else 0))
        self.stat = n(meaninertia=mc.meaninertia)
        self._names = dict(body=mc.body_names, joint=mc.jnt_names, geom=mc.geom_names, site=mc.site_names)

    def body(self, i):
        import types
        return types.SimpleNamespace(name=self._names["body"][i])

    def joint(self, i):
        import types
        return types.SimpleNamespace(name=self._names["joint"][i])

    def geom(self, i):
        import types
        return types.SimpleNamespace(name=self._names["geom"][i])

    def site(self, i):
        import types
        return types.SimpleNamespace(name=self._names["site"][i])


def test_from_mjmodel_reproduces_the_compiled_model(mc):
    """ModelConsts.from_mjmodel on an MjModel-shaped object carrying scene A gives back the same model: the same kernel
    table (KModel bytes) and the same oracle behaviour, pair list and slot order included."""
    import ctypes as C
    from manipulator_mujoco_b200.kmodel import build_kmodel
    from manipulator_mujoco_b200.mjcf import ModelConsts
    mc2 = ModelConsts.from_mjmodel(_MockMjModel(mc))
    assert mc2.nq == 13 and mc2.nv == 12 and mc2.ncon == mc.ncon == 215
    np.testing.assert_array_equal(mc2.pair_geom, mc.pair_geom)
    np.testing.assert_array_equal(mc2.pair_slotadr, mc.pair_slotadr)
    np.testing.assert_allclose(mc2.body_inertia, mc.body_inertia, atol=1e-12)
    k1, _ = build_kmodel(mc, 0.05)
    k2, _ = build_kmodel(mc2, 0.05)
    a = np.frombuffer(bytes(k1), dtype=np.float32)
    b = np.frombuffer(bytes(k2), dtype=np.float32)
    np.testing.assert_allclose(a, b, rtol=0, atol=1e-6)


SCENE_B = os.path.join(REFERENCE, "universal_robots_ur5e", "scene_mjx.xml")
DUAL_ARM = os.path.join(REFERENCE, "universal_robots_ur5e", "dual_arm_scene.xml")


@pytest.mark.skipif(not REFERENCE or not os.path.exists(SCENE_B), reason=NO_REFERENCE)
def test_scene_b_loads_with_the_counts_of_the_survey(tmp_path):
    """universal_robots_ur5e/scene_mjx.xml (the file BASELINE.json names; the planner itself loads scene A): slide joints of the
    two Hand-E fingers, their joint equality and fixed tendon, two contact excludes, one free box.  Counts: SURVEY.md A.3."""
    from collections import Counter
    from manipulator_mujoco_b200.mjcf import GEOM_BOX, GEOM_CAPSULE, GEOM_PLANE, JNT_SLIDE, ModelConsts
    mb = compile_mjcf(SCENE_B)
    assert (mb.nq, mb.nv, mb.njnt) == (15, 14, 9)
    assert list(mb.jnt_type).count(JNT_SLIDE) == 2 and (mb.neq, mb.ntendon, mb.nexclude, mb.nu) == (1, 1, 2, 0)
    assert mb.opt["iterations"] == 1 and mb.opt["ls_iterations"] == 5 and mb.opt["eulerdamp"] == 0 and mb.opt["integrator"] == "Euler"
    assert not np.any(mb.body_gravcomp)                                              # no gravity compensation in this scene
    pairs = Counter((int(a), int(b)) for a, b in mb.pair_type)
    assert pairs == {(GEOM_PLANE, GEOM_CAPSULE): 10, (GEOM_CAPSULE, GEOM_BOX): 20, (GEOM_CAPSULE, GEOM_CAPSULE): 27,
                     (GEOM_PLANE, GEOM_BOX): 1, (GEOM_BOX, GEOM_BOX): 1}
    assert mb.ncon == 95
    robot = [mb.geom_id(f"robot_{i}") for i in range(10)]
    nrob = sum(int(n) for (g1, g2), n in zip(mb.pair_geom, mb.pair_nslot) if g1 in robot or g2 in robot)
    assert nrob == 87                                                                # robot-involving contact slots
    assert int(mb.jnt_limited.sum()) == 8 and mb.neq + int(mb.jnt_limited.sum()) + 4 * mb.ncon == 389     # nefc
    e = 0
    assert mb.jnt_names[mb.eq_joint1[e]] == "hande_left_finger_joint" and mb.jnt_names[mb.eq_joint2[e]] == "hande_right_finger_joint"
    np.testing.assert_array_equal(mb.eq_polycoef[e], [0, 1, 0, 0, 0])
    assert mb.tendon_coefs[0] == [0.5, 0.5]
    np.testing.assert_allclose(mb.geom_size[mb.geom_id("robot_0")][:2], [0.03, 0.015])
    # host kinematics / dynamics understand the slide joints: opening a finger moves its body along the joint axis, and its
    # generalized inertia is the finger's mass
    q = mb.qpos0.copy()
    x0, _, xm = host_kinematics(mb, q)
    jl = mb.jnt_names.index("hande_left_finger_joint")
    q[mb.jnt_qposadr[jl]] = 0.02
    x1, _, _ = host_kinematics(mb, q)
    b = mb.jnt_body[jl]
    np.testing.assert_allclose(x1[b] - x0[b], 0.02 * xm[b] @ mb.jnt_axis[jl], atol=1e-12)
    M, _, _ = host_mass_matrix(mb, mb.qpos0)
    assert M.shape == (14, 14) and np.linalg.eigvalsh(M).min() > 0
    np.testing.assert_allclose(M[mb.jnt_dofadr[jl], mb.jnt_dofadr[jl]], mb.body_mass[b] + mb.jnt_armature[jl], rtol=1e-12)
    # the table survives the JSON round trip the package ships scene A through
    path = str(tmp_path / "scene_b.json")
    mb.to_json(path)
    back = ModelConsts.from_json(path)
    assert back.neq == 1 and back.tendon_joints == mb.tendon_joints and np.array_equal(back.pair_geom, mb.pair_geom)
    # ... and the rollout kernel says exactly what it lacks for it
    with pytest.raises(NotImplementedError, match=r"2 slide joint\(s\), 1 equality constraint\(s\), 1 tendon\(s\)"):
        KM.build_kmodel(mb, 0.05)


@pytest.mark.skipif(not REFERENCE or not os.path.exists(DUAL_ARM), reason=NO_REFERENCE)
def test_dual_arm_scene_loads_and_is_refused_by_the_kernel():
    """universal_robots_ur5e/dual_arm_scene.xml (BASELINE config 4, an extension: the reference planner cannot load it either,
    SURVEY.md finding 0.4 / A.4): 12 hinges, 12 position servos, implicitfast, cylinder end-effector geoms, keyframe `home`."""
    from manipulator_mujoco_b200.mjcf import GEOM_CYLINDER
    md = compile_mjcf(DUAL_ARM)
    assert (md.nq, md.nv, md.njnt, md.nu) == (12, 12, 12, 12) and md.opt["integrator"] == "implicitfast"
    cyl = [g for g in range(md.ngeom) if md.geom_type[g] == GEOM_CYLINDER and md.geom_collides[g]]
    assert len(cyl) == 2
    np.testing.assert_allclose(md.actuator_gainprm[0], [2000, 0, 0]); np.testing.assert_allclose(md.actuator_biasprm[0], [0, -2000, -400])
    assert md.key_names == ["home"] and len(md.key_qpos[0]) == 12
    # pairs with a cylinder have no slot count in the MJX table this package restates: listed, not guessed
    assert len(md.pair_unknown) > 0 and all(md.geom_type[g1] == GEOM_CYLINDER or md.geom_type[g2] == GEOM_CYLINDER for g1, g2 in md.pair_unknown)
    M, _, _ = host_mass_matrix(md, np.array(md.key_qpos[0]))
    assert M.shape == (12, 12) and np.linalg.eigvalsh(M).min() > 0
    assert np.allclose(M[:6, 6:], 0)                                                 # two independent chains
    with pytest.raises(NotImplementedError, match="12 hinge joints"):
        KM.build_kmodel(md, 0.05)
