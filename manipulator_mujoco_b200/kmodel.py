"""ModelConsts -> KModel (the float32 table of csrc/kmodel.h consumed by the rollout kernel).

The kernel is specialised to the topology of the scene the reference planner loads
(``mjx_planner.py:100``): a serial chain of 6 hinge joints on a static base, bodies welded behind a
joint merged into that joint's link, one free box, capsules on the chain, static planes / boxes.
``build_kmodel`` verifies every assumption and raises ``NotImplementedError`` otherwise -- there is
no fallback path.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from .mjcf import GEOM_BOX, GEOM_CAPSULE, GEOM_PLANE, JNT_FREE, JNT_HINGE, ModelConsts, quat_mul, quat_normalize, quat_to_mat

NL, NV, NQ, MAXCAP, MAXSBOX, MAXRPAIR, MAXBPAIR, MAXNEAR = 6, 12, 13, 12, 8, 160, 8, 96
LANE_GROUP = 16          # lanes per sample in the rollout kernel (csrc/warp_dsl.h KW); one collider pass = 16 pair entries
KP_NONE, KP_PLANE_CAP, KP_CAP_CAP, KP_CAP_BOX = -1, 0, 1, 2
KB_PLANE_BOX, KB_BOX_BOX, KB_BOX_BOX_SWAP = 0, 1, 2
_f, _i = C.c_float, C.c_int


class KModel(C.Structure):
    _fields_ = [
        ("nl", _i), ("ncap", _i), ("nsbox", _i), ("has_box", _i),
        ("nrpair", _i), ("nbpair", _i), ("nslot_robot", _i), ("ls_iterations", _i),
        ("dt", _f), ("tolerance", _f), ("ls_tolerance", _f), ("meaninertia", _f),
        ("impratio", _f), ("mu", _f), ("pad0", _f), ("pad1", _f),
        ("grav", _f * 4),
        ("solref", _f * 2), ("solimp", _f * 5), ("pad2", _f),
        ("refpt", _f * 4),
        ("base_pos", _f * 4), ("base_quat", _f * 4),
        ("l_pos", _f * 4 * NL), ("l_quat", _f * 4 * NL), ("l_axis", _f * 4 * NL), ("l_com", _f * 4 * NL),
        ("l_inertia", _f * 8 * NL),
        ("l_armature", _f * NL), ("l_damping", _f * NL), ("l_lo", _f * NL), ("l_hi", _f * NL),
        ("l_invw", _f * NL), ("l_margin", _f * NL),
        ("l_limited", _i * NL),
        ("ncbpass", _i), ("pad3", _i),
        ("tcp_pos", _f * 4), ("hande_quat", _f * 4),
        ("cap_link", _i * MAXCAP),
        ("cap_pos", _f * 4 * MAXCAP), ("cap_axis", _f * 4 * MAXCAP),
        ("cap_r", _f * MAXCAP), ("cap_hl", _f * MAXCAP), ("cap_invw", _f * MAXCAP),
        ("plane_pos", _f * 4), ("plane_n", _f * 4),
        ("sb_pos", _f * 4 * MAXSBOX), ("sb_mat", _f * 12 * MAXSBOX), ("sb_size", _f * 4 * MAXSBOX),
        ("fb_size", _f * 4), ("fb_inertia", _f * 4),
        ("fb_mass", _f), ("fb_damping", _f), ("fb_invw", _f), ("pad4", _f),
        ("rp", _i * MAXRPAIR),
        ("bp_type", _i * MAXBPAIR), ("bp_a", _i * MAXBPAIR),
        ("qpos0", _f * 16), ("warm0", _f * 12), ("qvel0", _f * 12),
    ]


# The records a rollout may take per call instead of the table's blocks (csrc/kmodel.h): a scene record is the
# sb_pos | sb_mat | sb_size block, a start record the qpos0 | warm0 | qvel0 block, in floats.
SCENE_FLOATS = MAXSBOX * (4 + 12 + 4)
START_FLOATS = 16 + 12 + 12
assert KModel.sb_mat.offset == KModel.sb_pos.offset + 4 * 4 * MAXSBOX and KModel.sb_size.offset == KModel.sb_pos.offset + 4 * 16 * MAXSBOX
assert KModel.fb_size.offset == KModel.sb_pos.offset + 4 * SCENE_FLOATS
assert KModel.warm0.offset == KModel.qpos0.offset + 4 * 16 and KModel.qvel0.offset == KModel.qpos0.offset + 4 * 28
assert C.sizeof(KModel) == KModel.qpos0.offset + 4 * START_FLOATS


def _set(dst, src):
    a = np.asarray(src, dtype=np.float64)
    flat = np.ctypeslib.as_array(dst).reshape(-1)
    flat[:a.size] = a.reshape(-1)


def _set_rows(dst, src, width):
    """Copy rows of ``src`` ([n, k], k <= width) into a padded [N][width] C array."""
    a = np.asarray(src, dtype=np.float64)
    arr = np.ctypeslib.as_array(dst)
    arr[:a.shape[0], :a.shape[1]] = a


def _static_pose(mc, body):
    """World pose (pos, quat) of a body whose whole ancestor chain is jointless."""
    chain = []
    b = body
    while b != 0:
        if mc.body_jntadr[b] >= 0:
            raise NotImplementedError(f"body {mc.body_names[body]} is not static")
        chain.append(b)
        b = mc.body_parent[b]
    pos, quat = np.zeros(3), np.array([1.0, 0, 0, 0])
    for b in reversed(chain):
        pos = pos + quat_to_mat(quat) @ mc.body_pos[b]
        quat = quat_mul(quat, mc.body_quat[b])
    return pos, quat


def _quat_to_mat_n(q):
    """mjcf.quat_to_mat over [N, 4] -> [N, 3, 3], the same float64 arithmetic per row."""
    w, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    return np.stack([
        np.stack([w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y)], -1),
        np.stack([2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x)], -1),
        np.stack([2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z], -1)], -2)


def _quat_mul_n(a, b):
    """mjcf.quat_mul over [N, 4] (b may be [4])."""
    b = np.broadcast_to(b, a.shape)
    aw, ax, ay, az = a[:, 0], a[:, 1], a[:, 2], a[:, 3]
    bw, bx, by, bz = b[:, 0], b[:, 1], b[:, 2], b[:, 3]
    return np.stack([aw * bw - ax * bx - ay * by - az * bz, aw * bx + ax * bw + ay * bz - az * by,
                     aw * by - ax * bz + ay * bw + az * bx, aw * bz + ax * by - ay * bx + az * bw], -1)


def _mat_vec_n(R, v):
    """R [N, 3, 3] @ v [3], one row at a time in a fixed order (the result of a row does not depend on N)."""
    return R[:, :, 0] * v[0] + R[:, :, 1] * v[1] + R[:, :, 2] * v[2]


def static_box_fields(body_pos, body_quat, geom_pos, geom_quat, size):
    """World pose of the body carrying a static box geom -> that box's rows of the scene record, for N poses at once, in
    float64: body_pos [N, 3], body_quat [N, 4] (unit), the geom's pose in the body and its half sizes [3] -> sb_pos [N, 4],
    sb_mat [N, 12], sb_size [N, 4] (csrc/kmodel.h).  An axis-aligned box (frame = signed permutation of the world axes, in
    float32) gets its half sizes along the world axes in sb_mat[9:12] and the flag sb_size[3] = 1: its far-field test runs
    on world coordinates with the permuted half sizes, no change of frame (rollout_core.h N1)."""
    body_pos, body_quat = np.asarray(body_pos, dtype=np.float64), np.asarray(body_quat, dtype=np.float64)
    geom_pos, size = np.asarray(geom_pos, dtype=np.float64), np.asarray(size, dtype=np.float64)
    n = body_pos.shape[0]
    gp = body_pos + _mat_vec_n(_quat_to_mat_n(body_quat), geom_pos)
    gm = _quat_to_mat_n(_quat_mul_n(body_quat, np.asarray(geom_quat, dtype=np.float64)))
    sb_pos, sb_mat, sb_size = np.zeros((n, 4)), np.zeros((n, 12)), np.zeros((n, 4))
    sb_pos[:, :3] = gp
    sb_mat[:, :9] = gm.reshape(n, 9)
    sb_size[:, :3] = size
    gm32 = gm.astype(np.float32)
    aligned = np.all((gm32 == 0) | (np.abs(gm32) == 1), axis=(1, 2))
    sb_mat[aligned, 9:12] = _mat_vec_n(np.abs(gm32[aligned].astype(np.float64)), size)
    sb_size[aligned, 3] = 1.0
    return sb_pos, sb_mat, sb_size


def _static_box_geoms(mc):
    """Collision box geoms on static bodies, in the kernel's static-box order (sb_* rows)."""
    free = {int(mc.jnt_body[j]) for j in range(mc.njnt) if mc.jnt_type[j] == JNT_FREE}
    return [g for g in range(mc.ngeom) if mc.geom_collides[g] and int(mc.geom_type[g]) == GEOM_BOX and int(mc.geom_body[g]) not in free
            and int(mc.body_weldid[mc.geom_body[g]]) == 0]


def movable_bodies(mc):
    """Names of the bodies a scene record can move: static children of the world that carry static box geoms."""
    bodies = sorted({int(mc.geom_body[g]) for g in _static_box_geoms(mc)})
    # a body whose static descendants carry boxes too is not movable: a record moves only the boxes of the named body
    nested = set()
    for b in bodies:
        c = int(mc.body_parent[b])
        while c != 0:
            nested.add(c)
            c = int(mc.body_parent[c])
    return [mc.body_names[b] for b in bodies if mc.body_parent[b] == 0 and mc.body_jntadr[b] < 0 and b not in nested]


def scene_records(mc, body_pose):
    """Scene records (csrc/kmodel.h, SCENE_FLOATS float32) with bodies moved: body_pose = {name: (pos [3], quat [4])}, either
    array with a leading [N] allowed (broadcast against the others).  Bodies not named keep their model pose, so
    ``scene_records(mc, {})`` is the table's own block.  Quaternions are normalised as the model compiler does.  Returns [N,
    SCENE_FLOATS], N = 1 without a leading dimension.  ValueError for a body that is not movable, a non-finite pose or a
    zero quaternion."""
    movable = movable_bodies(mc)
    poses, n = {}, 1
    for name, pq in body_pose.items():
        if name not in movable:
            raise ValueError(f"{name!r} is not a movable body; the movable bodies are {movable}")
        pos, quat = (np.asarray(a, dtype=np.float64) for a in pq)
        if pos.shape[-1:] != (3,) or quat.shape[-1:] != (4,) or pos.ndim > 2 or quat.ndim > 2:
            raise ValueError(f"{name}: pose must be pos [3] or [N, 3] and quat [4] or [N, 4], got {pos.shape} and {quat.shape}")
        if not (np.all(np.isfinite(pos)) and np.all(np.isfinite(quat))):
            raise ValueError(f"{name}: non-finite pose")
        pos, quat = pos.reshape(-1, 3), quat.reshape(-1, 4)
        if np.any(np.all(quat == 0, axis=1)):
            raise ValueError(f"{name}: zero quaternion")
        quat = np.array([quat_normalize(q) for q in quat])
        poses[mc.body_id(name)] = (pos, quat)
        n = max(n, pos.shape[0], quat.shape[0])
    for b, (pos, quat) in poses.items():
        if pos.shape[0] not in (1, n) or quat.shape[0] not in (1, n):
            raise ValueError(f"{mc.body_names[b]}: leading dimensions of the poses disagree (N = {n})")
        poses[b] = (np.broadcast_to(pos, (n, 3)), np.broadcast_to(quat, (n, 4)))
    rec = np.zeros((n, SCENE_FLOATS), dtype=np.float32)
    view = (rec[:, :4 * MAXSBOX].reshape(n, MAXSBOX, 4), rec[:, 4 * MAXSBOX:16 * MAXSBOX].reshape(n, MAXSBOX, 12),
            rec[:, 16 * MAXSBOX:].reshape(n, MAXSBOX, 4))
    for k, g in enumerate(_static_box_geoms(mc)):
        b = int(mc.geom_body[g])
        pos, quat = poses[b] if b in poses else (np.broadcast_to(p, (n, len(p))) for p in _static_pose(mc, b))
        for dst, f in zip(view, static_box_fields(pos, quat, mc.geom_pos[g], mc.geom_quat[g], mc.geom_size[g])):
            dst[:, k] = f
    return rec


def build_kmodel(mc: ModelConsts, timestep: float, robot_geom_names=None, tcp_site="tcp",
                 hande_body="hande", warm0=None):
    """Flatten the compiled scene.  Returns (KModel, info dict with the slot bookkeeping)."""
    if robot_geom_names is None:
        robot_geom_names = [f"robot_{i}" for i in range(10)]
    hinge = [j for j in range(mc.njnt) if mc.jnt_type[j] == JNT_HINGE]
    free = [j for j in range(mc.njnt) if mc.jnt_type[j] == JNT_FREE]
    # The loader (mjcf.compile_mjcf / from_mjmodel) accepts every scene the reference ships; the rollout kernel implements the
    # topology of the scene the planner loads (mjx_planner.py:100).  Say exactly what a refused model asks for.
    missing = []
    nslide = int(np.sum(np.asarray(mc.jnt_type) == 2))
    if nslide:
        missing.append(f"{nslide} slide joint(s)")
    if mc.d.get("neq", 0):
        missing.append(f"{mc.d['neq']} equality constraint(s)")
    if mc.d.get("ntendon", 0):
        missing.append(f"{mc.d['ntendon']} tendon(s)")
    if mc.d.get("nu", 0) and mc.opt.get("actuation", 1):
        missing.append(f"{mc.d['nu']} actuator(s)")
    if mc.opt.get("integrator", "Euler") != "Euler":
        missing.append(f"the {mc.opt['integrator']} integrator")
    if len(hinge) > NL:
        missing.append(f"{len(hinge)} hinge joints (a second arm; the kernel has one chain of {NL})")
    ncyl = int(np.sum((np.asarray(mc.geom_type) == 5) & (np.asarray(mc.geom_collides) != 0)))
    if ncyl:
        missing.append(f"{ncyl} cylinder collision geom(s)")
    if missing:
        raise NotImplementedError("the rollout kernel does not implement " + ", ".join(missing)
                                  + " of this model (it loads: see mjcf.compile_mjcf; the kernel's scope is DESIGN.md section 8)")
    if len(hinge) != NL or len(free) > 1 or len(hinge) + len(free) != mc.njnt:
        raise NotImplementedError("kernel supports exactly 6 hinge joints and at most one free joint")
    if free and (mc.jnt_dofadr[free[0]] != NL or mc.jnt_qposadr[free[0]] != NL):
        raise NotImplementedError("free joint must follow the robot joints")
    links = [int(mc.jnt_body[j]) for j in hinge]
    for i, (j, b) in enumerate(zip(hinge, links)):
        if mc.jnt_dofadr[j] != i or mc.jnt_qposadr[j] != i:
            raise NotImplementedError("robot dofs must be 0..5")
        if i and mc.body_parent[b] != links[i - 1]:
            raise NotImplementedError("robot must be a serial chain of directly nested bodies")
        if np.any(mc.jnt_pos[j] != 0):
            raise NotImplementedError("joint anchors must sit at the body origin")
    opt = mc.opt
    if opt["iterations"] != 1:
        raise NotImplementedError("kernel implements MJX's single Newton iteration (option iterations=1)")
    if opt.get("eulerdamp", 1) != 0:
        raise NotImplementedError("kernel implements Euler with eulerdamp disabled")

    m = KModel()
    m.nl, m.has_box = NL, int(bool(free))
    m.dt, m.tolerance, m.ls_tolerance = timestep, opt["tolerance"], opt["ls_tolerance"]
    m.meaninertia, m.impratio, m.ls_iterations = mc.meaninertia, opt["impratio"], opt["ls_iterations"]
    _set(m.grav, opt["gravity"])
    base_pos, base_quat = _static_pose(mc, mc.body_parent[links[0]])
    _set(m.base_pos, base_pos)
    _set(m.base_quat, base_quat)
    _set(m.refpt, base_pos + quat_to_mat(base_quat) @ mc.body_pos[links[0]])

    # pose of every robot-attached body relative to the link it is welded to
    rel = {}
    for b in range(1, mc.nbody):
        if mc.body_weldid[b] in links:
            li = links.index(int(mc.body_weldid[b]))
            pos, quat = np.zeros(3), np.array([1.0, 0, 0, 0])
            chain, c = [], b
            while c != links[li]:
                chain.append(c)
                c = mc.body_parent[c]
            for c in reversed(chain):
                pos = pos + quat_to_mat(quat) @ mc.body_pos[c]
                quat = quat_mul(quat, mc.body_quat[c])
            rel[b] = (li, pos, quat)
    for i, (j, b) in enumerate(zip(hinge, links)):
        m.l_pos[i][:3] = list(mc.body_pos[b])
        m.l_quat[i][:] = list(mc.body_quat[b])
        m.l_axis[i][:3] = list(mc.jnt_axis[j])
        # merge the inertia of all bodies welded to this link (same rigid body => same dynamics)
        parts = []
        for wb, (li, p, q) in rel.items():
            if li != i or mc.body_mass[wb] == 0:
                continue
            Rw = quat_to_mat(q)
            parts.append((mc.body_mass[wb], p + Rw @ mc.body_ipos[wb], Rw @ mc.body_inertia[wb] @ Rw.T))
        M = sum(p[0] for p in parts)
        com = sum(p[0] * p[1] for p in parts) / M
        I = np.zeros((3, 3))
        for ms, c, Ic in parts:
            d = c - com
            I += Ic + ms * (d @ d * np.eye(3) - np.outer(d, d))
        m.l_com[i][:3] = list(com)
        m.l_inertia[i][:] = [I[0, 0], I[1, 1], I[2, 2], I[0, 1], I[0, 2], I[1, 2], M, 0.0]
        m.l_armature[i], m.l_damping[i] = mc.jnt_armature[j], mc.jnt_damping[j]
        m.l_lo[i], m.l_hi[i] = mc.jnt_range[j]
        m.l_limited[i], m.l_margin[i] = int(mc.jnt_limited[j]), mc.jnt_margin[j]
        m.l_invw[i] = mc.dof_invweight0[i]
    sid = mc.site_id(tcp_site)
    li, p, q = rel[int(mc.site_body[sid])]
    if li != NL - 1:
        raise NotImplementedError("tcp site must be welded to the last link")
    _set(m.tcp_pos, p + quat_to_mat(q) @ mc.site_pos[sid])
    li, p, q = rel[mc.body_id(hande_body)]
    if li != NL - 1:
        raise NotImplementedError("hande body must be welded to the last link")
    _set(m.hande_quat, q)

    # ---- collision geoms ----
    col = [g for g in range(mc.ngeom) if mc.geom_collides[g]]
    par = np.array([[mc.geom_friction[g][0], *mc.geom_solref[g], *mc.geom_solimp[g], mc.geom_margin[g]] for g in col])
    if not np.all(par == par[0]):
        raise NotImplementedError("kernel assumes identical friction/solref/solimp/margin on all collision geoms")
    if par[0][-1] != 0 or any(mc.geom_condim[g] != 3 for g in col):
        raise NotImplementedError("kernel assumes margin 0 and condim 3")
    m.mu = par[0][0]
    _set(m.solref, par[0][1:3])
    _set(m.solimp, par[0][3:8])
    caps, sboxes, planes, fbox = {}, {}, {}, None
    for g in col:
        b, ty = int(mc.geom_body[g]), int(mc.geom_type[g])
        if ty == GEOM_CAPSULE:
            if b not in rel:
                raise NotImplementedError("capsules must be attached to the robot chain")
            li, p, q = rel[b]
            k = len(caps)
            if k >= MAXCAP:
                raise NotImplementedError("too many capsules")
            caps[g] = k
            m.cap_link[k] = li
            gq = quat_mul(q, mc.geom_quat[g])
            m.cap_pos[k][:3] = list(p + quat_to_mat(q) @ mc.geom_pos[g])
            m.cap_axis[k][:3] = list(quat_to_mat(gq)[:, 2])
            m.cap_r[k], m.cap_hl[k] = mc.geom_size[g][0], mc.geom_size[g][1]
            m.cap_invw[k] = mc.body_invweight0[b, 0]
        elif free and b == mc.jnt_body[free[0]]:
            if ty != GEOM_BOX or fbox is not None or np.any(mc.geom_pos[g] != 0) or not np.allclose(mc.geom_quat[g], [1, 0, 0, 0]):
                raise NotImplementedError("free body must carry exactly one centred box geom")
            fbox = g
        else:
            pos, quat = _static_pose(mc, b)
            gp = pos + quat_to_mat(quat) @ mc.geom_pos[g]
            gm = quat_to_mat(quat_mul(quat, mc.geom_quat[g]))
            if ty == GEOM_PLANE:
                if planes:
                    raise NotImplementedError("at most one plane")
                planes[g] = 0
                _set(m.plane_pos, gp)
                _set(m.plane_n, gm[:, 2])
            elif ty == GEOM_BOX:
                k = len(sboxes)
                if k >= MAXSBOX:
                    raise NotImplementedError("too many static boxes")
                sboxes[g] = k
                sp, sm, ss = static_box_fields(pos[None], quat[None], mc.geom_pos[g], mc.geom_quat[g], mc.geom_size[g])
                m.sb_pos[k][:] = list(sp[0])
                m.sb_mat[k][:] = list(sm[0])
                m.sb_size[k][:] = list(ss[0])
            else:
                raise NotImplementedError("static geoms must be planes or boxes")
    m.ncap, m.nsbox = len(caps), len(sboxes)
    if free:
        fb = int(mc.jnt_body[free[0]])
        I = mc.body_inertia[fb]
        if fbox is None or np.any(mc.body_ipos[fb] != 0) or not np.allclose(I, np.diag(np.diag(I)), atol=1e-12):
            raise NotImplementedError("free body needs a centred COM and principal-axis inertia")
        _set(m.fb_size, mc.geom_size[fbox])
        _set(m.fb_inertia, np.diag(I))
        m.fb_mass, m.fb_damping = mc.body_mass[fb], mc.jnt_damping[free[0]]
        m.fb_invw = mc.body_invweight0[fb, 0]

    # ---- pairs ----
    robot_ids = {mc.geom_id(n) for n in robot_geom_names if n in mc.geom_names}
    rpairs, bpairs, slot = [], [], 0
    robot_slots, box_slots = [], []           # the model's contact slot of each robot slot / free-box pair slot
    for (g1, g2), ns, adr in zip(mc.pair_geom, mc.pair_nslot, mc.pair_slotadr):
        g1, g2 = int(g1), int(g2)
        is_robot = g1 in robot_ids or g2 in robot_ids
        if g1 in caps or g2 in caps:
            robot_slots.extend(range(int(adr), int(adr) + int(ns)))
            if not is_robot:
                raise NotImplementedError("every capsule pair must be robot-involving (cost mask)")
            if g1 in planes:
                rpairs.append((KP_PLANE_CAP, 0, caps[g2], slot))
            elif g1 in caps and g2 in caps:
                rpairs.append((KP_CAP_CAP, caps[g1], caps[g2], slot))
            elif g2 in sboxes:
                rpairs.append((KP_CAP_BOX, caps[g1], sboxes[g2], slot))
            elif g2 == fbox:
                rpairs.append((KP_CAP_BOX, caps[g1], m.nsbox, slot))
            else:
                raise NotImplementedError("unsupported capsule pair")
            slot += int(ns)
        else:
            if is_robot:
                raise NotImplementedError("robot geoms must be capsules")
            other = g1 if g2 == fbox else g2
            box_slots.extend(int(adr) + k if k < ns else -1 for k in range(4))     # the kernel stages four slots per pair
            if fbox not in (g1, g2):
                raise NotImplementedError("non-robot pair without the free box")
            if other in planes:
                bpairs.append((KB_PLANE_BOX, 0))
            elif other in sboxes:
                bpairs.append((KB_BOX_BOX if g2 == fbox else KB_BOX_BOX_SWAP, sboxes[other]))
            else:
                raise NotImplementedError("unsupported free-box pair")
    if len(rpairs) > MAXRPAIR or len(bpairs) > MAXBPAIR:
        raise NotImplementedError("too many pairs")
    m.nrpair, m.nbpair, m.nslot_robot = len(rpairs), len(bpairs), slot
    # Table layout (csrc/kmodel.h): passes 0 .. ncbpass-1 = capsule-box, pass p = box p, lane l = capsule l; then
    # plane-capsule and capsule-capsule, each type starting on a pass boundary (lanes of a pass run one collider).
    by = lambda ty: [i for i in range(len(rpairs)) if rpairs[i][0] == ty]
    table = {}
    cb = by(KP_CAP_BOX)
    if len(cb) > MAXNEAR or m.ncap > LANE_GROUP:
        raise NotImplementedError("too many capsule-box pairs")
    m.ncbpass = (max(rpairs[i][2] for i in cb) + 1) if cb else 0
    for i in cb:
        _, cap, box, _ = rpairs[i]
        table[box * LANE_GROUP + cap] = i
    e = m.ncbpass * LANE_GROUP
    for ty in (KP_PLANE_CAP, KP_CAP_CAP):
        for i in by(ty):
            table[e] = i
            e += 1
        e += (-e) % LANE_GROUP
    if e > MAXRPAIR:
        raise NotImplementedError("pair table too small")
    for e in range(MAXRPAIR):
        m.rp[e] = 0
    for e, i in table.items():
        ty, a, b, sl = rpairs[i]
        m.rp[e] = (ty + 1) | (a << 4) | (b << 8) | (sl << 16)
    for e, (ty, a) in enumerate(bpairs):
        m.bp_type[e], m.bp_a[e] = ty, a
    _set(m.qpos0, mc.qpos0)
    if warm0 is not None:
        _set(m.warm0, warm0)
    # contact_key_slot: the model's contact slot of each contact key of the kernel (cemk_step_states_contacts' slot_map):
    # key k < nslot_robot is robot slot k, key nslot_robot + 4 q + j is slot j of free-box pair q
    info = dict(links=links, nslot_robot=slot, robot_ids=sorted(robot_ids),
                contact_key_slot=np.array(robot_slots + box_slots, dtype=np.int32))
    return m, info
