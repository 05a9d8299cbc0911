"""Scenes and start states given per call (rollout_sample<.., SCENE = true>, behind cemk_rollout_cost_scene and
cemk_step_states_scene) on the CPU emulation of the rollout core (tests/emu/emu_scene.cpp): the model's own records give the
bits of the existing entries, a moved scene gives the bits of a table built from the moved model, per-sample scenes give
each sample's single run, and the race-checking build finds no conflict.  Also the scene records themselves
(kmodel.scene_records) against build_kmodel of the moved model, and their refusals."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

from conftest import Q0, ROOT, TARGET_POS, TARGET_ROT, planner_inputs
from emu_util import Emu
from test_emu_step_contacts import ContactsEmu
from test_emu_step_states import snapshot_states

SRCS = [os.path.join(ROOT, "tests", "emu", "emu_scene.cpp")] + [os.path.join(ROOT, "manipulator_mujoco_b200", "csrc", n)
                                                                for n in ("rollout_core.h", "warp_dsl.h", "kmodel.h")]
# sha256 of bytes(build_kmodel(scene A, 0.05)[0]) before the static-box derivation moved into kmodel.static_box_fields
KMODEL_SHA256 = "85441cb320842c3c3973568fe35e616a73106fda3cd844c9c1d50796e4823c4d"
ROT_GENERAL = np.array([0.9, 0.2, -0.3, 0.25])         # not a signed permutation: the general far-test path
ROT_PERM = np.array([0.5, 0.5, -0.5, 0.5])             # 120 degrees about (1, -1, 1): a signed permutation


def _bits(a):
    return a.view(np.int32) if a.dtype == np.float32 else a


def own_records(km):
    from manipulator_mujoco_b200.kmodel import KModel, SCENE_FLOATS, START_FLOATS
    raw = np.frombuffer(bytes(km), dtype=np.float32)
    s, q = KModel.sb_pos.offset // 4, KModel.qpos0.offset // 4
    return raw[s:s + SCENE_FLOATS].copy(), raw[q:q + START_FLOATS].copy()


def moved_model(mc, moves):
    """ModelConsts with the named bodies at the given poses (quaternions normalised as the compiler does)."""
    from manipulator_mujoco_b200.mjcf import ModelConsts, quat_normalize
    bp, bq = mc.body_pos.copy(), mc.body_quat.copy()
    for name, (p, q) in moves.items():
        bp[mc.body_id(name)], bq[mc.body_id(name)] = p, quat_normalize(q)
    return ModelConsts(d=dict(mc.d, body_pos=bp, body_quat=bq))


class SceneEmu:
    """The emulation of the SCENE instantiations, plain or race-checking (-DCEMK_EMU_RACE)."""

    def __init__(self, km, key_slot, race=False):
        from manipulator_mujoco_b200.kmodel import KModel
        out = os.path.join(ROOT, "tests", "_emu_build", "libcemk_emu_scene" + ("_race" if race else "") + ".so")
        if not (os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in SRCS)):
            os.makedirs(os.path.dirname(out), exist_ok=True)
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            subprocess.run([cxx, "-O2", "-fPIC", "-shared", "-fopenmp", "-std=c++17", "-Wno-unknown-pragmas"]
                           + (["-DCEMK_EMU_RACE"] if race else []) + ["-o", out, SRCS[0]], check=True, capture_output=True)
        self.lib = C.CDLL(out)
        assert self.lib.emu_scene_race_enabled() == int(race)
        assert self.lib.emu_scene_sizeof_kmodel() == C.sizeof(KModel)
        self.km, self.key_slot = km, np.ascontiguousarray(key_slot, dtype=np.int32)

    def _call(self, states, B, T, td, q0, v0, warm, scene, start, nc, outs, contacts=False):
        f = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float32)
        scene = f(scene)
        stride = 0 if scene.ndim == 1 else scene.shape[1]
        p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        g = outs.get
        keep = [f(td), f(q0), f(v0), f(warm), f(TARGET_POS), f(TARGET_ROT), scene, f(start)]
        self.lib.emu_scene_rollout(C.byref(self.km), int(states), B, T, *map(p, keep[:4]), p(keep[4]), p(keep[5]), C.c_float(20.0),
                                   C.c_float(3.0), C.c_float(80.0), p(g("theta")), p(g("cost4")), p(g("qacc")), p(g("qpos")), p(g("qvel")),
                                   p(g("warm")), p(g("flags")), p(self.key_slot if contacts else None), p(g("qfrc")), p(g("ncon")),
                                   p(g("slot")), p(g("rec")), p(scene), stride, p(keep[7]), int(nc))
        return outs

    def rollout(self, td, scene, start, nc=20):
        B, T = td.shape[0], td.shape[1] // 6
        outs = dict(theta=np.zeros((B, 6 * T), np.float32), cost4=np.zeros((B, 4), np.float32), qacc=np.zeros((B, T, 12), np.float32),
                    flags=np.zeros(B, np.int32))
        return self._call(0, B, T, td, Q0, np.zeros(6), None, scene, start, nc, outs)

    def states(self, qpos, qvel, warm, scene, td=None, nc=20, contacts=False):
        N = qpos.shape[0]
        T = 1 if td is None else td.shape[1] // 6
        outs = dict(qpos=np.zeros((N, 13), np.float32), qvel=np.zeros((N, 12), np.float32), warm=np.zeros((N, 12), np.float32),
                    flags=np.zeros(N, np.int32))
        if contacts:
            outs.update(qfrc=np.zeros((N, 12), np.float32), ncon=np.zeros(N, np.int32), slot=np.zeros((N, 48), np.int32),
                        rec=np.zeros((N, 48, 12), np.float32))
        return self._call(1, N, T, td, qpos, qvel, warm, scene, None, nc, outs, contacts)

    def race_stats(self):
        out = (C.c_longlong * 2)()
        self.lib.emu_scene_race_stats(out)
        return int(out[0]), int(out[1])


@pytest.fixture(scope="module")
def setup(mc, oracle64):
    from manipulator_mujoco_b200.kmodel import build_kmodel
    warm0 = oracle64.initial_warmstart()
    km, info = build_kmodel(mc, 0.05, warm0=warm0)
    _, _, _, _, _, td = planner_inputs(16, 24, seed=3)
    # obstacle_1 on the TCP path of the rollouts: where sample 0's TCP is halfway through the horizon
    tcp = Emu(km).rollout(td, Q0, np.zeros(6), TARGET_POS, TARGET_ROT, nc=48)["eef_pos"][0, 8].astype(np.float64)
    return dict(mc=mc, km=km, info=info, warm0=warm0, td=td, tcp=tcp, emu=SceneEmu(km, info["contact_key_slot"]))


def _moves(s, rot):
    return {"obstacle_1": (s["tcp"], rot), "obstacle_3": (np.array([0.3, -0.35, 0.3]), ROT_PERM)}


def _kmodel_of(s, moves):
    from manipulator_mujoco_b200.kmodel import build_kmodel
    return build_kmodel(moved_model(s["mc"], moves), 0.05, warm0=s["warm0"])[0]


def test_build_kmodel_bytes_unchanged(mc):
    from manipulator_mujoco_b200.kmodel import build_kmodel
    assert hashlib.sha256(bytes(build_kmodel(mc, 0.05)[0])).hexdigest() == KMODEL_SHA256


@pytest.mark.parametrize("nc", [20, 48])
def test_own_records_give_the_existing_entries(setup, nc):
    s = setup
    scene, start = own_records(s["km"])
    a = Emu(s["km"]).rollout(s["td"], Q0, np.zeros(6), TARGET_POS, TARGET_ROT, nc=nc)
    b = s["emu"].rollout(s["td"], scene, start, nc=nc)
    for k in ("theta", "cost4", "qacc", "flags"):
        assert np.array_equal(_bits(a[k]), _bits(b[k])), k
    qpos, qvel, warm = snapshot_states(s["km"], 24)
    qpos[:, :6] += np.random.default_rng(nc).uniform(-0.5, 0.5, size=(24, 6))
    c = ContactsEmu(s["km"], s["info"]["contact_key_slot"]).step(qpos, qvel, warm, s["td"], nc=nc)
    d = s["emu"].states(qpos, qvel, warm, scene, s["td"], nc=nc, contacts=True)
    for k in ("qpos", "qvel", "warm", "flags", "qfrc", "ncon", "slot", "rec"):
        assert np.array_equal(_bits(c[k]), _bits(d[k])), k


@pytest.mark.parametrize("nc", [20, 48])
@pytest.mark.parametrize("rot", ["general", "perm"])
def test_moved_scene_equals_moved_model(setup, nc, rot):
    from manipulator_mujoco_b200.kmodel import scene_records
    s = setup
    moves = _moves(s, ROT_GENERAL if rot == "general" else ROT_PERM)
    km2 = _kmodel_of(s, moves)
    scene = scene_records(s["mc"], moves)[0]
    _, start = own_records(s["km"])
    a = Emu(km2).rollout(s["td"], Q0, np.zeros(6), TARGET_POS, TARGET_ROT, nc=nc)
    b = s["emu"].rollout(s["td"], scene, start, nc=nc)
    for k in ("theta", "cost4", "qacc", "flags"):
        assert np.array_equal(_bits(a[k]), _bits(b[k])), k
    base = Emu(s["km"]).rollout(s["td"], Q0, np.zeros(6), TARGET_POS, TARGET_ROT, nc=nc)
    assert b["cost4"][:, 3].max() > base["cost4"][:, 3].max(), "the moved obstacle must add collision cost"
    qpos, qvel, warm = snapshot_states(s["km"], 24)
    c = ContactsEmu(km2, s["info"]["contact_key_slot"]).step(qpos, qvel, warm, s["td"], nc=nc)
    d = s["emu"].states(qpos, qvel, warm, scene, s["td"], nc=nc, contacts=True)
    for k in ("qpos", "qvel", "warm", "flags", "qfrc", "ncon", "slot", "rec"):
        assert np.array_equal(_bits(c[k]), _bits(d[k])), k


def test_start_record_equals_the_table_snapshot(setup):
    s = setup
    scene, start = own_records(s["km"])
    start = start.copy()
    start[6:9] += np.float32([0.05, -0.04, 0.1])                      # the free box lifted and shifted, spinning
    start[16:28] = np.float32(np.linspace(-0.3, 0.4, 12))
    start[28 + 6:28 + 12] = np.float32([0.1, 0.0, -0.2, 0.5, -0.3, 0.2])
    km2 = _kmodel_of(s, {})
    C.memmove(C.addressof(km2) + type(km2).qpos0.offset, start.ctypes.data, start.nbytes)
    a = Emu(km2).rollout(s["td"], Q0, np.zeros(6), TARGET_POS, TARGET_ROT, nc=20)
    b = s["emu"].rollout(s["td"], scene, start, nc=20)
    for k in ("theta", "cost4", "qacc"):
        assert np.array_equal(_bits(a[k]), _bits(b[k])), k


def test_adjacent_samples_with_different_scenes(setup):
    from manipulator_mujoco_b200.kmodel import scene_records
    s = setup
    scenes = np.concatenate([scene_records(s["mc"], _moves(s, r)) for r in (ROT_GENERAL, ROT_PERM)] + [own_records(s["km"])[0][None]])
    idx = np.arange(24) % 3
    per = scenes[idx]
    _, start = own_records(s["km"])
    b = s["emu"].rollout(s["td"], per, start)
    qpos, qvel, warm = snapshot_states(s["km"], 24)
    d = s["emu"].states(qpos, qvel, warm, per, s["td"], contacts=True)
    for j in range(3):
        rows = idx == j
        a = s["emu"].rollout(s["td"][rows], scenes[j], start)
        c = s["emu"].states(qpos[rows], qvel[rows], warm[rows], scenes[j], s["td"][rows], contacts=True)
        for k in ("theta", "cost4", "qacc"):
            assert np.array_equal(_bits(a[k]), _bits(b[k][rows])), (j, k)
        for k in ("qpos", "qvel", "warm", "qfrc", "ncon", "slot", "rec"):
            assert np.array_equal(_bits(c[k]), _bits(d[k][rows])), (j, k)


@pytest.mark.parametrize("nc", [20, 48])
def test_race_build_finds_no_conflict(setup, nc):
    from manipulator_mujoco_b200.kmodel import scene_records
    s = setup
    race = SceneEmu(s["km"], s["info"]["contact_key_slot"], race=True)
    race.race_stats()
    scene = scene_records(s["mc"], _moves(s, ROT_GENERAL))[0]
    _, start = own_records(s["km"])
    a, b = s["emu"].rollout(s["td"], scene, start, nc=nc), race.rollout(s["td"], scene, start, nc=nc)
    qpos, qvel, warm = snapshot_states(s["km"], 24)
    c = s["emu"].states(qpos, qvel, warm, scene, s["td"], nc=nc, contacts=True)
    d = race.states(qpos, qvel, warm, scene, s["td"], nc=nc, contacts=True)
    waw, blocks = race.race_stats()
    assert waw == 0 and blocks > 0
    for k in ("theta", "cost4", "qacc"):
        assert np.array_equal(_bits(a[k]), _bits(b[k])), k
    for k in ("qpos", "qvel", "warm", "qfrc", "ncon", "slot", "rec"):
        assert np.array_equal(_bits(c[k]), _bits(d[k])), k


@pytest.mark.parametrize("rot", ["general", "perm", "unnormalised"])
def test_scene_records_equal_build_kmodel_of_the_moved_model(setup, rot):
    from manipulator_mujoco_b200.kmodel import scene_records
    s = setup
    q = {"general": ROT_GENERAL, "perm": ROT_PERM, "unnormalised": 3.0 * ROT_GENERAL}[rot]
    moves = {"obstacle_2": (np.array([0.1, 0.45, 0.62]), q), "table_1": (np.array([0.02, -0.01, 0.38]), np.array([1.0, 0, 0, 0]))}
    rec = scene_records(s["mc"], moves)
    assert rec.shape == (1, 160)
    assert np.array_equal(_bits(rec[0]), _bits(own_records(_kmodel_of(s, moves))[0]))
    flags = rec[0, 128:].reshape(8, 4)[:, 3]                  # sb_size[.][3]; obstacle_2 is static box 4
    assert flags[4] == (1.0 if rot == "perm" else 0.0) and flags[0] == 1.0
    # vectorised: N poses at once give the N single records
    rng = np.random.default_rng(7)
    pos = rng.uniform(-0.5, 0.5, size=(5, 3))
    quat = np.concatenate([rng.normal(size=(3, 4)), [ROT_PERM, [0.0, 0.0, 0.0, -2.0]]])
    many = scene_records(s["mc"], {"obstacle_1": (pos, quat), "target_2": (np.array([0.1, 0.1, 0.45]), ROT_PERM)})
    assert many.shape == (5, 160)
    for i in range(5):
        one = {"obstacle_1": (pos[i], quat[i]), "target_2": (np.array([0.1, 0.1, 0.45]), ROT_PERM)}
        assert np.array_equal(_bits(many[i]), _bits(scene_records(s["mc"], one)[0]))
        assert np.array_equal(_bits(many[i]), _bits(own_records(_kmodel_of(s, one))[0])), i


def test_scene_record_refusals(mc):
    from manipulator_mujoco_b200.kmodel import movable_bodies, scene_records
    assert movable_bodies(mc) == ["table_1", "target_1", "target_2", "obstacle_1", "obstacle_2", "obstacle_3"]
    one = (np.zeros(3), np.array([1.0, 0, 0, 0]))
    for name in ("target_0", "world", "hande", "no_such_body"):
        with pytest.raises(ValueError, match="obstacle_1"):
            scene_records(mc, {name: one})
    with pytest.raises(ValueError, match="non-finite"):
        scene_records(mc, {"obstacle_1": (np.array([0, np.nan, 0]), one[1])})
    with pytest.raises(ValueError, match="non-finite"):
        scene_records(mc, {"obstacle_1": (np.zeros(3), np.array([np.inf, 0, 0, 0]))})
    with pytest.raises(ValueError, match="zero quaternion"):
        scene_records(mc, {"obstacle_1": (np.zeros(3), np.zeros(4))})
    with pytest.raises(ValueError, match="disagree"):
        scene_records(mc, {"obstacle_1": (np.zeros((3, 3)), one[1]), "obstacle_2": (np.zeros((2, 3)), one[1])})
