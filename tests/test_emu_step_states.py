"""Stepping per-environment states (rollout_sample<NC, true>, behind cemk_step_states) on the CPU emulation of the
rollout core (tests/emu/emu_states.cpp): from the planner's snapshot it gives the planner rollout's bits (tests/emu/emu.cpp),
a run split into chunks gives the bits of one call, and the race-checking build finds no conflict and agrees bit for bit."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import Q0, ROOT, TARGET_POS, TARGET_ROT, planner_inputs
from emu_util import Emu

SRCS = [os.path.join(ROOT, "tests", "emu", "emu_states.cpp")] + [os.path.join(ROOT, "manipulator_mujoco_b200", "csrc", n)
                                                                 for n in ("rollout_core.h", "warp_dsl.h", "kmodel.h")]


class StatesEmu:
    """The emulation of the per-environment stepping instantiation, plain or race-checking (-DCEMK_EMU_RACE)."""

    def __init__(self, km, race=False):
        from manipulator_mujoco_b200.kmodel import KModel
        out = os.path.join(ROOT, "tests", "_emu_build", "libcemk_emu_states" + ("_race" if race else "") + ".so")
        if not (os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in SRCS)):
            os.makedirs(os.path.dirname(out), exist_ok=True)
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            subprocess.run([cxx, "-O2", "-fPIC", "-shared", "-fopenmp", "-std=c++17", "-Wno-unknown-pragmas"]
                           + (["-DCEMK_EMU_RACE"] if race else []) + ["-o", out, SRCS[0]], check=True, capture_output=True)
        self.lib = C.CDLL(out)
        assert self.lib.emu_states_race_enabled() == int(race)
        assert self.lib.emu_states_sizeof_kmodel() == C.sizeof(KModel)
        self.km = km

    def race_stats(self):
        """(write-write conflicts, lane blocks checked) since the last call; race build only."""
        out = (C.c_longlong * 2)()
        self.lib.emu_states_race_stats(out)
        return int(out[0]), int(out[1])


@pytest.fixture(scope="module")
def emus(mc, oracle64):
    """(planner rollout emulation, states emulation, race-checking states emulation) of one model."""
    from manipulator_mujoco_b200.kmodel import build_kmodel
    km, _ = build_kmodel(mc, 0.05, warm0=oracle64.initial_warmstart())
    return Emu(km), StatesEmu(km), StatesEmu(km, race=True)


def step_states(emu, qpos, qvel, warm, td=None, T=1, nc=20, out=None):
    """emu_rollout_states; out = (qpos, qvel, warm) arrays to write (the inputs themselves for in-place stepping)."""
    f = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    qpos, qvel, warm = f(qpos), f(qvel), f(warm)
    N = qpos.shape[0]
    if td is not None:
        td = f(td)
        T = td.shape[1] // 6
    qo, vo, wo = out if out is not None else (np.zeros((N, 13), np.float32), np.zeros((N, 12), np.float32), np.zeros((N, 12), np.float32))
    r = dict(theta=np.zeros((N, 6 * T), np.float32), eef_pos=np.zeros((N, T, 3), np.float32), eef_rot=np.zeros((N, T, 4), np.float32),
             collision=np.zeros((N, T, emu.km.nslot_robot), np.float32), qacc=np.zeros((N, T, 12), np.float32), flags=np.zeros(N, np.int32))
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    emu.lib.emu_rollout_states(C.byref(emu.km), N, T, p(qpos), p(qvel), p(warm), p(td), p(qo), p(vo), p(wo), p(r["theta"]),
                               p(r["eef_pos"]), p(r["eef_rot"]), p(r["collision"]), p(r["qacc"]), p(r["flags"]), int(nc))
    r.update(qpos=qo, qvel=vo, warm=wo)
    return r


def snapshot_states(km, N):
    """The planner's start state of every sample: Q0, the box at the model's qpos0, zero velocity, the KModel warm start."""
    qpos = np.tile(np.concatenate([Q0, np.array(km.qpos0[6:13])]), (N, 1))
    qvel = np.tile(np.concatenate([np.zeros(6), np.array(km.qvel0[6:12])]), (N, 1))
    warm = np.tile(np.array(km.warm0[:12]), (N, 1))
    return qpos, qvel, warm


def _bits(a):
    return a.view(np.int32) if a.dtype == np.float32 else a


def test_snapshot_states_give_the_planner_rollout(emus):
    rollout, plain, _ = emus
    T, N = 16, 24
    td = planner_inputs(T, N, seed=2)[5]
    ref = rollout.rollout(td, Q0, np.zeros(6), TARGET_POS, TARGET_ROT, nc=20)
    got = step_states(plain, *snapshot_states(plain.km, N), td=td)
    for k in ("theta", "qacc", "collision", "eef_pos", "eef_rot", "flags"):
        assert np.array_equal(_bits(got[k]), _bits(ref[k])), k
    assert np.array_equal(got["warm"], got["qacc"][:, -1])           # the next warm start is the last step's qacc
    assert np.array_equal(got["qpos"][:, :6], got["theta"].reshape(N, 6, T)[:, :, -1])


def test_chunks_equal_one_call(emus):
    _, plain, _ = emus
    T, N = 24, 16
    td = planner_inputs(T, N, seed=3)[5]
    one = step_states(plain, *snapshot_states(plain.km, N), td=td)
    for chunks in ((1, 9, 14), (1,) * T):
        st = snapshot_states(plain.km, N)
        parts, t0 = [], 0
        tdr = td.reshape(N, 6, T)
        for c in chunks:
            r = step_states(plain, *st, td=tdr[:, :, t0:t0 + c].reshape(N, 6 * c))
            parts.append(r)
            st = (r["qpos"], r["qvel"], r["warm"])
            t0 += c
        assert t0 == T
        theta = np.concatenate([p["theta"].reshape(N, 6, -1) for p in parts], axis=2).reshape(N, 6 * T)
        qacc = np.concatenate([p["qacc"] for p in parts], axis=1)
        col = np.concatenate([p["collision"] for p in parts], axis=1)
        assert np.array_equal(_bits(theta), _bits(one["theta"])), chunks
        assert np.array_equal(_bits(qacc), _bits(one["qacc"])), chunks
        assert np.array_equal(_bits(col), _bits(one["collision"])), chunks
        for k in ("qpos", "qvel", "warm"):
            assert np.array_equal(_bits(st[("qpos", "qvel", "warm").index(k)]), _bits(one[k])), (chunks, k)


def test_in_place_and_without_thetadot(emus):
    """Outputs written over the inputs give the bits of separate outputs; thetadot = NULL keeps each env's own qvel[:6]."""
    _, plain, _ = emus
    N = 29
    rng = np.random.default_rng(5)
    qpos, qvel, warm = snapshot_states(plain.km, N)
    qpos[:, :6] += rng.uniform(-0.3, 0.3, size=(N, 6))
    qvel[:, :6] = rng.uniform(-0.8, 0.8, size=(N, 6))
    sep = step_states(plain, qpos, qvel, warm)
    forced = step_states(plain, qpos, qvel, warm, td=qvel[:, :6])
    for k in ("qpos", "qvel", "warm", "qacc", "theta"):
        assert np.array_equal(_bits(sep[k]), _bits(forced[k])), k
    f = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    io = (f(qpos), f(qvel), f(warm))
    step_states(plain, *io, out=io)
    for a, k in zip(io, ("qpos", "qvel", "warm")):
        assert np.array_equal(_bits(a), _bits(sep[k])), k


def test_race_build_agrees_without_conflicts(emus):
    _, plain, race = emus
    T, N = 12, 12
    td = planner_inputs(T, N, seed=1)[5]
    st = snapshot_states(plain.km, N)
    a = step_states(plain, *st, td=td)
    race.race_stats()
    b = step_states(race, *st, td=td)
    waw, blocks = race.race_stats()
    assert waw == 0 and blocks > 100 * N
    for k in a:
        assert np.array_equal(_bits(a[k]), _bits(b[k])), k
