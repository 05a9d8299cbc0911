"""The contact outputs of stepping per-environment states (rollout_sample<NC, true, true>, behind
cemk_step_states_contacts) on the CPU emulation of the rollout core (tests/emu/emu_contacts.cpp): the state is the bits of
the stepping without contacts (tests/emu/emu_states.cpp), the contacts and forces agree with the float64 oracle on contact
states and deep-collision states, with the record in shared memory and spilled, and the race-checking build finds no
conflict."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from contact_util import check_against_oracle, deep_states, harvest_contact_states
from test_emu_step_states import StatesEmu, step_states

SRCS = [os.path.join(ROOT, "tests", "emu", "emu_contacts.cpp")] + [os.path.join(ROOT, "manipulator_mujoco_b200", "csrc", n)
                                                                   for n in ("rollout_core.h", "warp_dsl.h", "kmodel.h")]


class ContactsEmu:
    """The emulation of the contacts instantiation, plain or race-checking (-DCEMK_EMU_RACE)."""

    def __init__(self, km, key_slot, race=False):
        from manipulator_mujoco_b200.kmodel import KModel
        out = os.path.join(ROOT, "tests", "_emu_build", "libcemk_emu_contacts" + ("_race" if race else "") + ".so")
        if not (os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in SRCS)):
            os.makedirs(os.path.dirname(out), exist_ok=True)
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            subprocess.run([cxx, "-O2", "-fPIC", "-shared", "-fopenmp", "-std=c++17", "-Wno-unknown-pragmas"]
                           + (["-DCEMK_EMU_RACE"] if race else []) + ["-o", out, SRCS[0]], check=True, capture_output=True)
        self.lib = C.CDLL(out)
        assert self.lib.emu_contacts_race_enabled() == int(race)
        assert self.lib.emu_contacts_sizeof_kmodel() == C.sizeof(KModel)
        self.km, self.key_slot = km, np.ascontiguousarray(key_slot, dtype=np.int32)

    def step(self, qpos, qvel, warm, td=None, nc=20):
        f = lambda a: np.ascontiguousarray(a, dtype=np.float32)
        qpos, qvel, warm = f(qpos), f(qvel), f(warm)
        N = qpos.shape[0]
        T = 1 if td is None else td.shape[1] // 6
        td = None if td is None else f(td)
        r = dict(qpos=np.zeros((N, 13), np.float32), qvel=np.zeros((N, 12), np.float32), warm=np.zeros((N, 12), np.float32),
                 flags=np.zeros(N, np.int32), qfrc=np.zeros((N, 12), np.float32), ncon=np.zeros(N, np.int32),
                 slot=np.zeros((N, 48), np.int32), rec=np.zeros((N, 48, 12), np.float32))
        p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        self.lib.emu_rollout_states_contacts(C.byref(self.km), N, T, p(qpos), p(qvel), p(warm), p(td), p(r["qpos"]), p(r["qvel"]),
                                             p(r["warm"]), p(r["flags"]), p(self.key_slot), p(r["qfrc"]), p(r["ncon"]), p(r["slot"]),
                                             p(r["rec"]), int(nc))
        r["qacc"] = r["warm"]
        return r

    def race_stats(self):
        out = (C.c_longlong * 2)()
        self.lib.emu_contacts_race_stats(out)
        return int(out[0]), int(out[1])


@pytest.fixture(scope="module")
def emus(mc, oracle64):
    """(states emulation, contacts emulation, race-checking contacts emulation) of one model."""
    from manipulator_mujoco_b200.kmodel import build_kmodel
    km, info = build_kmodel(mc, 0.05, warm0=oracle64.initial_warmstart())
    return StatesEmu(km), ContactsEmu(km, info["contact_key_slot"]), ContactsEmu(km, info["contact_key_slot"], race=True)


@pytest.fixture(scope="module")
def states(oracle64):
    """The teacher-forced contact states (every 3rd, for time), then 12 deep-collision start states."""
    qp, qv, wm = harvest_contact_states(oracle64)
    dq, dv, dw = deep_states(oracle64, 12)
    return np.concatenate([qp[::3], dq]), np.concatenate([qv[::3], dv]), np.concatenate([wm[::3], dw])


def _bits(a):
    return a.view(np.int32) if a.dtype == np.float32 else a


@pytest.mark.parametrize("nc", [20, 48])
def test_contacts_against_the_oracle(emus, states, oracle64, mc, nc):
    plain, con, _ = emus
    qpos, qvel, warm = states
    got = con.step(qpos, qvel, warm, nc=nc)
    ref = step_states(plain, qpos, qvel, warm, nc=nc)
    for k in ("qpos", "qvel", "warm", "flags"):
        assert np.array_equal(_bits(got[k]), _bits(ref[k])), k
    assert got["ncon"].max() > 20                    # the spill area is exercised with nc = 20
    sub = lambda d, sl: {k: v[sl] for k, v in d.items()}
    mu = float(con.km.mu)
    n = check_against_oracle(oracle64, qpos[:-12], qvel[:-12], warm[:-12], sub(got, slice(None, -12)), mu)
    n += check_against_oracle(oracle64, qpos[-12:], qvel[-12:], warm[-12:], sub(got, slice(-12, None)), mu, nrm_tol=5e-3, pos_tol=5e-2, forces=False)
    assert n > 100


def test_chained_steps_report_the_last_step(emus, states, oracle64):
    """With thetadot over T = 4 steps, the outputs describe the last step: they equal those of one step from the state
    three chained steps reached."""
    plain, con, _ = emus
    qpos, qvel, warm = (a[:8] for a in states)
    rng = np.random.default_rng(3)
    td = rng.uniform(-0.5, 0.5, size=(8, 24)).astype(np.float32)
    four = con.step(qpos, qvel, warm, td=td)
    three = step_states(plain, qpos, qvel, warm, td=td.reshape(8, 6, 4)[:, :, :3].reshape(8, 18))
    last = con.step(three["qpos"], three["qvel"], three["warm"], td=td.reshape(8, 6, 4)[:, :, 3:].reshape(8, 6))
    for k in ("qpos", "qvel", "warm", "flags", "qfrc", "ncon", "slot", "rec"):
        assert np.array_equal(_bits(four[k]), _bits(last[k])), k


def test_race_checking_build_finds_no_conflict(emus, states):
    _, con, race = emus
    qpos, qvel, warm = (a[-10:] for a in states)
    race.race_stats()
    for nc in (20, 48):
        a, b = con.step(qpos, qvel, warm, nc=nc), race.step(qpos, qvel, warm, nc=nc)
        for k in a:
            assert np.array_equal(_bits(a[k]), _bits(b[k])), (nc, k)
    waw, blocks = race.race_stats()
    assert waw == 0 and blocks > 1000
