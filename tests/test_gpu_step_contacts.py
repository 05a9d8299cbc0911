"""Contacts and constraint forces from batched stepping (cemk_step_states_contacts, step_batch(..., contacts=True)): the
state is the bits of contacts=False, the contacts and forces agree with the float64 oracle, a box resting on the table
carries its weight, and the refusals."""
import numpy as np
import pytest
import torch

from conftest import Q0
from contact_util import check_against_oracle, deep_states, harvest_contact_states

pytestmark = pytest.mark.gpu

STATE_KEYS = ("qpos", "qvel", "qacc", "qacc_warmstart", "overflow")


@pytest.fixture(scope="module")
def planner():
    from manipulator_mujoco_b200 import cem_planner
    return cem_planner(num_dof=6, num_batch=100, num_steps=16, timestep=0.05, maxiter_cem=1, num_elite=0.05,
                       w_pos=20.0, w_rot=3.0, w_col=80.0, maxiter_projection=10)


def snapshot_states(pl, N):
    km = pl.mjx_model
    qpos = np.tile(np.concatenate([Q0, np.array(km.qpos0[6:13])]), (N, 1))
    qvel = np.tile(np.concatenate([np.zeros(6), np.array(km.qvel0[6:12])]), (N, 1))
    warm = np.tile(np.array(km.warm0[:12]), (N, 1))
    return qpos, qvel, warm


def _host(out):
    return {k: v.cpu().numpy() for k, v in out.items()}


def _eq(a, b):
    return np.array_equal(a.view(np.int32), b.view(np.int32)) if a.dtype == np.float32 else np.array_equal(a, b)


@pytest.mark.parametrize("N", [1, 29, 4096])
@pytest.mark.parametrize("T", [1, 16])
def test_contacts_leave_the_state_bits(planner, N, T):
    rng = np.random.default_rng(N + T)
    qpos, qvel, warm = snapshot_states(planner, N)
    qpos[:, :6] += rng.uniform(-0.6, 0.6, size=(N, 6))
    td = None if T == 1 else rng.uniform(-0.8, 0.8, size=(N, 6 * T))
    a = _host(planner.step_batch(qpos, qvel, warm, thetadot=td))
    b = _host(planner.step_batch(qpos, qvel, warm, thetadot=td, contacts=True))
    for k in STATE_KEYS + (("theta",) if T > 1 else ()):
        assert _eq(a[k], b[k]), k
    assert b["contact_slot"].shape == (N, 48) and b["contact_force"].shape == (N, 48, 3) and b["qfrc_constraint"].shape == (N, 12)
    # in place: the state tensors are the inputs (contact outputs are separate)
    dev = planner.device
    io = [torch.as_tensor(x, dtype=torch.float32, device=dev).contiguous() for x in (qpos, qvel, warm)]
    from manipulator_mujoco_b200 import _lib
    from manipulator_mujoco_b200.planner import _ptr
    tdd = None if td is None else torch.as_tensor(td, dtype=torch.float32, device=dev).contiguous()
    key = torch.as_tensor(planner._key_slot, dtype=torch.int32, device=dev)
    qfrc, ncon = torch.empty(N, 12, device=dev), torch.empty(N, dtype=torch.int32, device=dev)
    slot, rec = torch.empty(N, 48, dtype=torch.int32, device=dev), torch.empty(N, 48, 12, device=dev)
    _lib.check(planner._lib.cemk_step_states_contacts(planner._h, N, T, *map(_ptr, io), _ptr(tdd), *map(_ptr, io), None, None, None,
                                                      None, None, None, _ptr(key), _ptr(qfrc), _ptr(ncon), _ptr(slot), _ptr(rec),
                                                      planner._stream()), planner._lib)
    torch.cuda.synchronize()
    assert _eq(io[0].cpu().numpy(), a["qpos"]) and _eq(io[1].cpu().numpy(), a["qvel"]) and _eq(io[2].cpu().numpy(), a["qacc"])
    assert _eq(qfrc.cpu().numpy(), b["qfrc_constraint"]) and _eq(slot.cpu().numpy(), b["contact_slot"])
    assert _eq(rec[:, :, 7:10].cpu().numpy(), b["contact_force"]) and _eq(ncon.cpu().numpy(), b["ncon"])


def _got(out):
    h = _host(out)
    rec = np.concatenate([h["contact_dist"][..., None], h["contact_pos"], h["contact_normal"], h["contact_force"],
                          np.zeros(h["contact_dist"].shape + (2,), np.float32)], axis=-1)
    return dict(qacc=h["qacc"], flags=h["overflow"].astype(np.int32), ncon=h["ncon"], slot=h["contact_slot"], rec=rec,
                qfrc=h["qfrc_constraint"])


def test_contacts_against_the_oracle(planner, oracle64):
    """The teacher-forced contact states in one launch, and deep-collision start states (more than the 20 contacts a sample
    keeps in shared memory for the first ones): tolerances in contact_util.check_against_oracle."""
    mu = float(planner.mjx_model.mu)
    qpos, qvel, warm = harvest_contact_states(oracle64)
    n = check_against_oracle(oracle64, qpos, qvel, warm, _got(planner.step_batch(qpos, qvel, warm, contacts=True)), mu)
    assert n > 150
    qpos, qvel, warm = deep_states(oracle64, 12)
    got = _got(planner.step_batch(qpos, qvel, warm, contacts=True))
    assert got["ncon"].max() > 20
    check_against_oracle(oracle64, qpos, qvel, warm, got, mu, nrm_tol=5e-3, pos_tol=5e-2, forces=False)


def test_box_at_rest_carries_its_weight(planner):
    """The planner's snapshot state: target_0 drops onto the table in its first steps.  Once it rests, the normal forces of
    its table contacts and the z component of its qfrc_constraint both equal m g."""
    mc = planner._mc
    geoms = planner.contact_slot_geoms
    box, table = mc.geom_id("target_0"), mc.geom_id("table_geom_1")
    qpos, qvel, warm = snapshot_states(planner, 1)
    td = np.zeros((1, 6 * 16))
    for _ in range(20):
        out = planner.step_batch(qpos, qvel, warm, thetadot=td)
        qpos, qvel, warm = out["qpos"], out["qvel"], out["qacc_warmstart"]
        if float(qvel[0, 6:].abs().max()) < 1e-5:
            break
    assert float(qvel[0, 6:].abs().max()) < 1e-5
    h = _host(planner.step_batch(qpos, qvel, warm, thetadot=np.zeros((1, 6)), contacts=True))
    mg = float(mc.body_mass[mc.body_id("target_0")]) * 9.81
    nc = int(h["ncon"][0])
    slots = h["contact_slot"][0, :nc]
    on_table = np.array([set(geoms[s]) == {box, table} for s in slots])
    assert on_table.sum() >= 3
    assert abs(h["contact_force"][0, :nc, 0][on_table].sum() - mg) < 1e-3 * mg
    assert abs(h["qfrc_constraint"][0, 8] - mg) < 1e-3 * mg
    assert geoms.flags.writeable is False and geoms.shape == (mc.ncon, 2)


def test_refusals(planner):
    from manipulator_mujoco_b200.planner import _ptr
    lib, h, dev = planner._lib, planner._h, planner.device
    N = 4
    qp, qv, wm = (torch.as_tensor(a, dtype=torch.float32, device=dev).contiguous() for a in snapshot_states(planner, N))
    qo, vo, wo = torch.empty_like(qp), torch.empty_like(qv), torch.empty_like(wm)
    key = torch.as_tensor(planner._key_slot, dtype=torch.int32, device=dev)
    outs = [key, torch.empty(N, 12, device=dev), torch.empty(N, dtype=torch.int32, device=dev),
            torch.empty(N, 48, dtype=torch.int32, device=dev), torch.empty(N, 48, 12, device=dev)]
    st = planner._stream()

    def call(n=N, T=1, a=(qp, qv, wm), o=(qo, vo, wo), c=outs, handle=h):
        return lib.cemk_step_states_contacts(handle, n, T, *map(_ptr, a), None, *map(_ptr, o), None, None, None, None, None, None,
                                             *map(_ptr, c), st)

    assert call() == 0 and call(c=[None] * 5) == 0
    torch.cuda.synchronize()
    for i in range(5):
        c = list(outs); c[i] = None
        assert call(c=c) == -1 and b"all given or all NULL" in lib.cemk_last_error()
    assert call(n=0) == -1 and call(T=0) == -1 and call(T=2) == -1 and call(handle=None) == -1
    for i in range(3):
        a = [qp, qv, wm]; a[i] = None
        assert call(a=tuple(a)) == -1
        o = [qo, vo, wo]; o[i] = None
        assert call(o=tuple(o)) == -1
