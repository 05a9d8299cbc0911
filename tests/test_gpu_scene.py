"""Scenes and start states given per call on the GPU (cemk_rollout_cost_scene, cemk_step_states_scene, and the keywords
scene= / state= of compute_cem, compute_rollout_batch and step_batch): NULL records give the old exports' bits, a moved
scene on a handle gives the bits of a handle built from the moved model, a start state gives the bits of a table holding it,
a captured tick replays changed records, the big-capacity rerun agrees, and the contacts on a moved box agree with the
float64 oracle of the moved model."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import Q0, TARGET_POS, TARGET_ROT, planner_inputs
from contact_util import check_against_oracle, harvest_contact_states
from test_emu_scene import ROT_GENERAL, ROT_PERM, moved_model

pytestmark = pytest.mark.gpu

KW = dict(num_dof=6, timestep=0.05, maxiter_cem=1, num_elite=0.05, w_pos=20.0, w_rot=3.0, w_col=80.0, maxiter_projection=10)


@pytest.fixture(scope="module")
def planner():
    from manipulator_mujoco_b200 import cem_planner
    return cem_planner(num_batch=100, num_steps=16, **KW)


@pytest.fixture(scope="module")
def moves(planner):
    """obstacle_1 on the TCP path (sample 0 halfway through the horizon), obstacle_3 moved and turned."""
    td = planner_inputs(16, 100, seed=3)[5]
    tcp = planner.compute_rollout_batch(td, Q0, np.zeros(6))[1][0, 8].cpu().numpy().astype(np.float64)
    return lambda rot: {"obstacle_1": (tcp, rot), "obstacle_3": (np.array([0.3, -0.35, 0.3]), ROT_PERM)}


def _bits(a):
    a = a.cpu().numpy() if torch.is_tensor(a) else a
    return a.view(np.int32) if a.dtype == np.float32 else a


class Handle:
    """A library handle of its own on a model table (the planner's warm start unless the table says otherwise)."""

    def __init__(self, pl, km):
        from manipulator_mujoco_b200 import _lib
        self.pl, self.lib, self.h = pl, pl._lib, C.c_void_p()
        _lib.check(self.lib.cemk_create(C.byref(km), C.sizeof(km), pl.device.index or 0, C.byref(self.h)), self.lib)

    def close(self):
        self.lib.cemk_destroy(self.h)


def table(pl, mc=None, start=None):
    """The planner's table, or the table of model `mc` with the planner's warm start, optionally holding a start record."""
    from manipulator_mujoco_b200.kmodel import build_kmodel
    km = type(pl.mjx_model)()
    C.memmove(C.byref(km), C.byref(pl.mjx_model), C.sizeof(km))
    if mc is not None:
        km = build_kmodel(mc, pl.t)[0]
        for i in range(12):
            km.warm0[i] = pl.mjx_model.warm0[i]
    if start is not None:
        C.memmove(C.addressof(km) + type(km).qpos0.offset, np.ascontiguousarray(start, np.float32).ctypes.data, 160)
    return km


def rollout(pl, h, td, scene=None, stride=0, start=None, old=False):
    """One planner rollout with every dump on a handle -> host arrays (theta, cost4, eef_pos, eef_rot, collision, qacc, flags)."""
    from manipulator_mujoco_b200 import _lib
    from manipulator_mujoco_b200.planner import _ptr
    dev = pl.device
    td = torch.as_tensor(td, dtype=torch.float32, device=dev).contiguous()
    B, T = td.shape[0], td.shape[1] // 6
    q0, v0 = torch.as_tensor(Q0, dtype=torch.float32, device=dev), torch.zeros(6, device=dev)
    tp, tr = torch.as_tensor(TARGET_POS, dtype=torch.float32, device=dev), torch.as_tensor(TARGET_ROT, dtype=torch.float32, device=dev)
    o = [torch.empty(B, 6 * T, device=dev), torch.empty(B, 4, device=dev), torch.empty(B, T, 3, device=dev), torch.empty(B, T, 4, device=dev),
         torch.empty(B, T, pl.nslot, device=dev), torch.empty(B, T, 12, device=dev), torch.empty(B, dtype=torch.int32, device=dev)]
    args = [h, B, T, _ptr(td), _ptr(q0), _ptr(v0), _ptr(tp), _ptr(tr), 20.0, 3.0, 80.0] + [_ptr(x) for x in o]
    if old:
        _lib.check(pl._lib.cemk_rollout_cost(*args, pl._stream()), pl._lib)
    else:
        sc = None if scene is None else torch.as_tensor(scene, dtype=torch.float32, device=dev).contiguous()
        st = None if start is None else torch.as_tensor(start, dtype=torch.float32, device=dev).contiguous()
        _lib.check(pl._lib.cemk_rollout_cost_scene(*args, _ptr(sc), stride, _ptr(st), pl._stream()), pl._lib)
    torch.cuda.synchronize()
    return [x.cpu().numpy() for x in o]


def _same(a, b):
    for i, (x, y) in enumerate(zip(a, b)):
        assert np.array_equal(_bits(x), _bits(y)), i


def test_null_records_give_the_old_exports(planner):
    from manipulator_mujoco_b200 import _lib
    from manipulator_mujoco_b200.planner import _ptr
    td = planner_inputs(16, 1000, seed=5)[5]
    _same(rollout(planner, planner._h, td, old=True), rollout(planner, planner._h, td))
    rng = np.random.default_rng(1)
    N = 500
    qpos = np.tile(np.concatenate([Q0, np.array(planner.mjx_model.qpos0[6:13])]), (N, 1))
    qpos[:, :6] += rng.uniform(-0.6, 0.6, size=(N, 6))
    qvel, warm = np.zeros((N, 12)), np.tile(np.array(planner.mjx_model.warm0[:12]), (N, 1))
    a = planner.step_batch(qpos, qvel, warm, contacts=True)
    dev = planner.device
    f = lambda x: torch.as_tensor(x, dtype=torch.float32, device=dev).contiguous()
    io = [f(qpos), f(qvel), f(warm)]
    out = [torch.empty(N, 13, device=dev), torch.empty(N, 12, device=dev), torch.empty(N, 12, device=dev)]
    flags, qfrc, ncon = torch.empty(N, dtype=torch.int32, device=dev), torch.empty(N, 12, device=dev), torch.empty(N, dtype=torch.int32, device=dev)
    slot, rec = torch.empty(N, 48, dtype=torch.int32, device=dev), torch.empty(N, 48, 12, device=dev)
    key = torch.as_tensor(planner._key_slot, dtype=torch.int32, device=dev)
    _lib.check(planner._lib.cemk_step_states_scene(planner._h, N, 1, *map(_ptr, io), None, *map(_ptr, out), None, None, None, None, None,
                                                   _ptr(flags), _ptr(key), _ptr(qfrc), _ptr(ncon), _ptr(slot), _ptr(rec), None, 0,
                                                   planner._stream()), planner._lib)
    _same([a["qpos"], a["qvel"], a["qacc_warmstart"], a["qfrc_constraint"], a["ncon"], a["contact_slot"], a["contact_dist"]],
          [out[0], out[1], out[2], qfrc, ncon, slot, rec[:, :, 0]])


def test_refusals(planner):
    from manipulator_mujoco_b200.planner import _ptr
    lib = planner._lib
    td = torch.zeros(4, 96, device=planner.device)
    v = torch.zeros(64, device=planner.device)
    scene = planner.make_scene({})
    for stride in (1, 159, 161, -160):
        assert lib.cemk_rollout_cost_scene(planner._h, 4, 16, _ptr(td), _ptr(v), _ptr(v), _ptr(v), _ptr(v), 1.0, 1.0, 1.0, _ptr(td),
                                           _ptr(v), None, None, None, None, None, _ptr(scene), stride, None, planner._stream()) == -1
        assert b"scene_stride" in lib.cemk_last_error()
        assert lib.cemk_step_states_scene(planner._h, 4, 1, _ptr(v), _ptr(v), _ptr(v), None, _ptr(v), _ptr(v), _ptr(v), None, None, None,
                                          None, None, None, None, None, None, None, None, _ptr(scene), stride, planner._stream()) == -1
    assert lib.cemk_rollout_cost_scene(planner._h, 0, 16, _ptr(td), _ptr(v), _ptr(v), _ptr(v), _ptr(v), 1.0, 1.0, 1.0, _ptr(td),
                                       _ptr(v), None, None, None, None, None, _ptr(scene), 0, None, planner._stream()) == -1
    assert lib.cemk_step_states_scene(planner._h, 4, 2, _ptr(v), _ptr(v), _ptr(v), None, _ptr(v), _ptr(v), _ptr(v), None, None, None,
                                      None, None, None, None, None, None, None, None, _ptr(scene), 0, planner._stream()) == -1
    with pytest.raises(ValueError, match="scene"):
        planner.step_batch(np.zeros((3, 13)), np.zeros((3, 12)), np.zeros((3, 12)), scene=torch.zeros(2, 160))
    with pytest.raises(ValueError, match="obstacle_1"):
        planner.make_scene({"target_0": (np.zeros(3), np.array([1.0, 0, 0, 0]))})
    assert planner.scene_bodies == ("table_1", "target_1", "target_2", "obstacle_1", "obstacle_2", "obstacle_3")


@pytest.mark.parametrize("B,T", [(1, 16), (29, 16), (1000, 16), (4096, 100)])
def test_moved_scene_equals_moved_handle(planner, moves, B, T):
    m = moves(ROT_GENERAL)
    h2 = Handle(planner, table(planner, moved_model(planner._mc, m)))
    try:
        td = planner_inputs(T, B, seed=B)[5]
        scene = planner.make_scene(m)
        a = rollout(planner, h2.h, td, old=True)
        b = rollout(planner, planner._h, td, scene=scene)
        _same(a, b)
        assert b[1][:, 3].max() > rollout(planner, planner._h, td, old=True)[1][:, 3].max()     # the moved obstacle is hit
        if T == 16:
            c = planner.compute_rollout_batch(td, Q0, np.zeros(6), scene=scene)
            _same([a[0], a[2], a[3], a[4]], c)
        # force_rerun (the 48-contact instantiation) with the scene agrees bit for bit
        from manipulator_mujoco_b200 import _lib
        _lib.check(planner._lib.cemk_set_option(planner._h, b"force_rerun", 1), planner._lib)
        try:
            _same(b[:6], rollout(planner, planner._h, td, scene=scene)[:6])
        finally:
            _lib.check(planner._lib.cemk_set_option(planner._h, b"force_rerun", 0), planner._lib)
    finally:
        h2.close()


def test_planner_rollout_per_sample_scenes(planner, moves):
    """Stride 160: adjacent samples -- the two lane groups of a warp -- with different scenes each give the bits of the
    shared-scene run of their own scene (B = 29 and 1000: one and several samples per CTA slot)."""
    scenes = [planner.make_scene(moves(ROT_GENERAL)), planner.make_scene(moves(ROT_PERM)), planner.make_scene({})]
    for B in (29, 1000):
        td = planner_inputs(16, B, seed=B + 1)[5]
        idx = np.arange(B) % 3
        per = torch.stack([scenes[i] for i in idx])
        got = rollout(planner, planner._h, td, scene=per, stride=160)
        for j in range(3):
            one = rollout(planner, planner._h, td, scene=scenes[j])
            for x, y in zip(got, one):
                assert np.array_equal(_bits(x[idx == j]), _bits(y[idx == j])), (B, j)
        c = planner.compute_rollout_batch(td, Q0, np.zeros(6), scene=per)
        assert np.array_equal(_bits(c[0]), _bits(got[0]))


@pytest.mark.parametrize("contacts", [False, True])
def test_step_batch_per_environment_scenes(planner, moves, contacts):
    rng = np.random.default_rng(4)
    N, T = 256, 8
    base = moves(ROT_GENERAL)["obstacle_1"][0]
    pos = base + rng.uniform(-0.08, 0.08, size=(N, 3))
    quat = rng.normal(size=(N, 4))
    scenes = planner.make_scene({"obstacle_1": (pos, quat)})
    assert scenes.shape == (N, 160)
    qpos = np.tile(np.concatenate([Q0, np.array(planner.mjx_model.qpos0[6:13])]), (N, 1))
    qpos[:, :6] += rng.uniform(-0.3, 0.3, size=(N, 6))
    qvel, warm = np.zeros((N, 12)), np.tile(np.array(planner.mjx_model.warm0[:12]), (N, 1))
    td = rng.uniform(-0.8, 0.8, size=(N, 6 * T))
    got = planner.step_batch(qpos, qvel, warm, thetadot=td, contacts=contacts, scene=scenes)
    keys = ("qpos", "qvel", "qacc_warmstart", "theta") + (("qfrc_constraint", "ncon", "contact_slot", "contact_dist", "contact_force")
                                                          if contacts else ())
    for i in (0, 1, 77, N - 1):
        h2 = Handle(planner, table(planner, moved_model(planner._mc, {"obstacle_1": (pos[i], quat[i])})))
        try:
            saved, planner._h = planner._h, h2.h
            try:
                one = planner.step_batch(qpos[i:i + 1], qvel[i:i + 1], warm[i:i + 1], thetadot=td[i:i + 1], contacts=contacts)
            finally:
                planner._h = saved
        finally:
            h2.close()
        for k in keys:
            assert np.array_equal(_bits(got[k][i:i + 1]), _bits(one[k])), (i, k)
    # a shared scene [160] is the per-environment form with every row equal
    shared = planner.step_batch(qpos, qvel, warm, thetadot=td, contacts=contacts, scene=scenes[5])
    rows = planner.step_batch(qpos, qvel, warm, thetadot=td, contacts=contacts, scene=scenes[5].expand(N, 160).contiguous())
    for k in keys:
        assert np.array_equal(_bits(shared[k]), _bits(rows[k])), k
    # the moved obstacle matters: some environment ends elsewhere than in the model's scene
    plain = planner.step_batch(qpos, qvel, warm, thetadot=td, contacts=contacts)
    assert not np.array_equal(_bits(plain["qpos"]), _bits(got["qpos"]))


def _state(pl, rng):
    qpos = np.concatenate([Q0, np.array(pl.mjx_model.qpos0[6:13])])
    qpos[6:9] += rng.uniform(-0.1, 0.1, size=3)
    qpos[9:13] = rng.normal(size=4)
    qpos[9:13] /= np.linalg.norm(qpos[9:13])
    return dict(qpos=qpos, qvel=rng.uniform(-0.5, 0.5, size=12), qacc_warmstart=rng.uniform(-1, 1, size=12))


def test_compute_cem_state_equals_a_table_holding_it():
    from manipulator_mujoco_b200 import _lib, cem_planner
    rng = np.random.default_rng(9)
    pl, pl2 = cem_planner(num_batch=200, num_steps=16, **KW), cem_planner(num_batch=200, num_steps=16, **KW)
    s = _state(pl, rng)
    km = table(pl2, start=pl2.start_record(s))
    _lib.check(pl2._lib.cemk_set_model(pl2._h, C.byref(km), C.sizeof(km)), pl2._lib)
    for _ in range(3):                                               # eager ticks, then a captured one
        a = pl.compute_cem(np.zeros(pl.nvar), Q0, np.zeros(6), np.zeros(6), TARGET_POS, TARGET_ROT, state=s)
        b = pl2.compute_cem(np.zeros(pl.nvar), Q0, np.zeros(6), np.zeros(6), TARGET_POS, TARGET_ROT)
        for x, y in zip(a, b):
            assert np.array_equal(_bits(x), _bits(y))
    c = pl.compute_cem(np.zeros(pl.nvar), Q0, np.zeros(6), np.zeros(6), TARGET_POS, TARGET_ROT)
    assert not np.array_equal(_bits(a[8]), _bits(c[8]))          # the start state (its warm start) matters, and nothing was kept
    pl.close()
    pl2.close()


def test_graph_replays_changed_scenes_and_states(moves):
    from manipulator_mujoco_b200 import cem_planner
    rng = np.random.default_rng(2)
    graph = cem_planner(num_batch=1000, num_steps=16, **dict(KW, maxiter_cem=3))
    eager = cem_planner(num_batch=1000, num_steps=16, **dict(KW, maxiter_cem=3))
    eager.use_cuda_graph = False
    ticks = []
    for i in range(6):
        m = moves(ROT_GENERAL if i % 2 else ROT_PERM)
        m["obstacle_1"] = (m["obstacle_1"][0] + rng.uniform(-0.05, 0.05, size=3), m["obstacle_1"][1])
        ticks.append((graph.make_scene(m), _state(graph, rng)))
    xa = xb = np.zeros(graph.nvar)
    g0 = None
    for i, (scene, s) in enumerate(ticks):
        a = graph.compute_cem(xa, Q0, np.zeros(6), np.zeros(6), TARGET_POS, TARGET_ROT, scene=scene, state=s)
        b = eager.compute_cem(xb, Q0, np.zeros(6), np.zeros(6), TARGET_POS, TARGET_ROT, scene=scene.cpu().numpy(), state=s)
        for x, y in zip(a, b):
            assert np.array_equal(_bits(x), _bits(y)), i
        xa, xb = a[6], b[6]
        if i == 2:
            g0 = graph._graph
        assert (graph._graph is not None) == (i >= 2)
    assert graph._graph is g0                                         # captured once, replayed with three new records
    graph.close()
    eager.close()


@pytest.mark.parametrize("rot", ["perm", "general"])
def test_moved_scene_rollouts_against_the_oracle(planner, oracle64, rot):
    """Planner rollouts (T = 100) through obstacle_1 moved into the arm's reach -- at the TCP position of sample 12 at step
    40, clear of every arm at the start -- against the float64 oracle of the moved model: the first four steps to 2e-6,
    every sample up to its first contact (all of it when it never touches) to the trajectory tolerance of
    test_gpu_rollout.py, collision distances before the first contact to 1e-3, and the samples the oracle sees touching
    the moved obstacle touch it in the kernel too.  "general" is an arbitrary rotation (the far test's change of frame),
    "perm" a signed permutation (its axis-aligned path)."""
    from oracle.oracle import Oracle
    td = planner_inputs(100, 64, seed=1)[5]
    base = oracle64.rollout(td, Q0, np.zeros(6))
    m = {"obstacle_1": (base[1][12, 40], ROT_GENERAL if rot == "general" else ROT_PERM)}
    ora = Oracle(moved_model(planner._mc, m), 0.05, dtype="f64")
    # the rollouts start from the handle's warm start (a forward of the model's own scene), not from one of the moved scene
    oth, oep, oer, ocol = ora.rollout(td, Q0, np.zeros(6), warm=oracle64.initial_warmstart())
    theta, _, eef_pos, _, col, _, _ = rollout(planner, planner._h, td, scene=planner.make_scene(m))
    touch = (ocol < 0).any(axis=2)
    first = np.where(touch.any(axis=1), touch.argmax(axis=1), 100)
    newly = touch.any(axis=1) & ~(base[3] < 0).any(axis=(1, 2))
    assert touch[:, 0].sum() == 0 and newly.sum() >= 10
    th, ot = theta.reshape(64, 6, 100), oth.reshape(64, 6, 100)
    assert np.abs(th[:, :, :4] - ot[:, :, :4]).max() < 2e-6
    dc = []
    for b in range(64):
        k = first[b]
        assert np.abs(th[b, :, :k] - ot[b, :, :k]).max() < 5e-4, b
        assert np.abs(eef_pos[b, :k] - oep[b, :k]).max() < 5e-4, b
        dc.append(np.abs(col[b, :k] - ocol[b, :k]).ravel())
    assert (np.concatenate(dc) > 1e-3).mean() < 1e-4
    assert (col[newly] < 0).any(axis=(1, 2)).all()


def test_contacts_on_the_moved_box_against_the_oracle(planner, moves):
    from oracle.oracle import Oracle
    m = moves(ROT_GENERAL)
    mc2 = moved_model(planner._mc, m)
    ora = Oracle(mc2, 0.05, dtype="f64")
    qpos, qvel, warm = harvest_contact_states(ora)
    got = planner.step_batch(qpos, qvel, warm, contacts=True, scene=planner.make_scene(m))
    h = {k: v.cpu().numpy() for k, v in got.items()}
    rec = np.concatenate([h["contact_dist"][..., None], h["contact_pos"], h["contact_normal"], h["contact_force"],
                          np.zeros(h["contact_dist"].shape + (2,), np.float32)], axis=-1)
    g = dict(qacc=h["qacc"], flags=h["overflow"].astype(np.int32), ncon=h["ncon"], slot=h["contact_slot"], rec=rec, qfrc=h["qfrc_constraint"])
    n = check_against_oracle(ora, qpos, qvel, warm, g, float(planner.mjx_model.mu))
    assert n > 0
    geoms = planner.contact_slot_geoms
    ob = planner._mc.geom_id("obstacle_1")
    slots = h["contact_slot"][h["contact_slot"] >= 0]
    assert (geoms[slots] == ob).any(), "no contact on the moved box"
