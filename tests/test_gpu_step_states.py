"""Stepping many environments from their own states in one launch (cemk_step_states, cem_planner.step_batch): the planner
rollout's bits from its snapshot, chunked runs equal to one call, the oracle and jit_step on contact states, in-place
outputs, no effect on planning, and the refusals."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import Q0, TARGET_POS, TARGET_ROT, planner_inputs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def planner():
    from manipulator_mujoco_b200 import cem_planner
    return cem_planner(num_dof=6, num_batch=100, num_steps=16, timestep=0.05, maxiter_cem=1, num_elite=0.05,
                       w_pos=20.0, w_rot=3.0, w_col=80.0, maxiter_projection=10)


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _dev(pl, a):
    return torch.as_tensor(np.asarray(a), dtype=torch.float32, device=pl.device).contiguous()


def rollout_cost(pl, td):
    """cemk_rollout_cost from the planner's snapshot (arm at Q0 at rest) with every dump."""
    from manipulator_mujoco_b200 import _lib
    td = _dev(pl, td)
    N, T = td.shape[0], td.shape[1] // 6
    dev = pl.device
    q0, v0, tp, tr = _dev(pl, Q0), torch.zeros(6, device=dev), _dev(pl, TARGET_POS), _dev(pl, TARGET_ROT)
    r = dict(theta=torch.empty(N, 6 * T, device=dev), cost4=torch.empty(N, 4, device=dev), eef_pos=torch.empty(N, T, 3, device=dev),
             eef_rot=torch.empty(N, T, 4, device=dev), collision=torch.empty(N, T, pl.nslot, device=dev), qacc=torch.empty(N, T, 12, device=dev),
             flags=torch.empty(N, dtype=torch.int32, device=dev))
    _lib.check(pl._lib.cemk_rollout_cost(pl._h, N, T, _p(td), _p(q0), _p(v0), _p(tp), _p(tr), 20.0, 3.0, 80.0, _p(r["theta"]), _p(r["cost4"]),
                                         _p(r["eef_pos"]), _p(r["eef_rot"]), _p(r["collision"]), _p(r["qacc"]), _p(r["flags"]), pl._stream()), pl._lib)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in r.items()}


def step_states(pl, qpos, qvel, warm, td=None, out=None):
    """cemk_step_states with every dump; `out` = (qpos, qvel, warm) device tensors to write (the inputs for in place)."""
    from manipulator_mujoco_b200 import _lib
    qpos, qvel, warm = (a if torch.is_tensor(a) else _dev(pl, a) for a in (qpos, qvel, warm))
    N = qpos.shape[0]
    td = None if td is None else (td if torch.is_tensor(td) else _dev(pl, td))
    T = 1 if td is None else td.shape[1] // 6
    dev = pl.device
    qo, vo, wo = out if out is not None else (torch.empty(N, 13, device=dev), torch.empty(N, 12, device=dev), torch.empty(N, 12, device=dev))
    r = dict(theta=torch.empty(N, 6 * T, device=dev), eef_pos=torch.empty(N, T, 3, device=dev), eef_rot=torch.empty(N, T, 4, device=dev),
             collision=torch.empty(N, T, pl.nslot, device=dev), qacc=torch.empty(N, T, 12, device=dev), flags=torch.empty(N, dtype=torch.int32, device=dev))
    _lib.check(pl._lib.cemk_step_states(pl._h, N, T, _p(qpos), _p(qvel), _p(warm), _p(td), _p(qo), _p(vo), _p(wo), _p(r["theta"]),
                                        _p(r["eef_pos"]), _p(r["eef_rot"]), _p(r["collision"]), _p(r["qacc"]), _p(r["flags"]), pl._stream()), pl._lib)
    torch.cuda.synchronize()
    res = {k: v.cpu().numpy() for k, v in r.items()}
    res.update(qpos=qo.cpu().numpy(), qvel=vo.cpu().numpy(), warm=wo.cpu().numpy())
    return res


def snapshot_states(pl, N):
    """The start state of every planner rollout: Q0, the box at the model's qpos0, zero velocity, the KModel warm start."""
    km = pl.mjx_model
    qpos = np.tile(np.concatenate([Q0, np.array(km.qpos0[6:13])]), (N, 1))
    qvel = np.tile(np.concatenate([np.zeros(6), np.array(km.qvel0[6:12])]), (N, 1))
    warm = np.tile(np.array(km.warm0[:12]), (N, 1))
    return qpos, qvel, warm


def _eq(a, b):
    return np.array_equal(a.view(np.int32), b.view(np.int32)) if a.dtype == np.float32 else np.array_equal(a, b)


@pytest.mark.parametrize("N,T", [(100, 16), (4096, 100)])
def test_snapshot_states_give_the_planner_rollout(planner, N, T):
    td = planner_inputs(T, N, seed=7)[5]
    ref = rollout_cost(planner, td)
    got = step_states(planner, *snapshot_states(planner, N), td=td)
    for k in ("theta", "qacc", "collision", "eef_pos", "eef_rot", "flags"):
        assert _eq(got[k], ref[k]), k
    assert _eq(got["warm"], got["qacc"][:, -1])
    assert _eq(got["qpos"][:, :6], got["theta"].reshape(N, 6, T)[:, :, -1])


def _chunked(pl, td, chunks):
    N, T = td.shape[0], td.shape[1] // 6
    st = snapshot_states(pl, N)
    tdr = td.reshape(N, 6, T)
    parts, t0 = [], 0
    for c in chunks:
        r = step_states(pl, *st, td=tdr[:, :, t0:t0 + c].reshape(N, 6 * c))
        parts.append(r)
        st = (r["qpos"], r["qvel"], r["warm"])
        t0 += c
    assert t0 == T
    theta = np.concatenate([p["theta"].reshape(N, 6, -1) for p in parts], axis=2).reshape(N, 6 * T)
    qacc = np.concatenate([p["qacc"] for p in parts], axis=1)
    return st, theta, qacc


@pytest.mark.parametrize("N,T,chunks", [(512, 100, (1, 36, 63)), (512, 16, (1,) * 16)])
def test_chunks_equal_one_call(planner, N, T, chunks):
    td = planner_inputs(T, N, seed=8)[5]
    one = step_states(planner, *snapshot_states(planner, N), td=td)
    (qp, qv, wm), theta, qacc = _chunked(planner, td, chunks)
    assert _eq(theta, one["theta"]) and _eq(qacc, one["qacc"])
    assert _eq(qp, one["qpos"]) and _eq(qv, one["qvel"]) and _eq(wm, one["warm"])


@pytest.fixture(scope="module")
def contact_states(oracle64):
    """The teacher-forced contact states of test_gpu_step.py: every 4th step with a robot contact of 12 contact-rich
    planner samples (oracle float64 rollout), qvel[:6] = the commanded velocity of that step."""
    T, B = 100, 64
    td = planner_inputs(T, B, seed=1)[5]
    oth, oep, oer, ocol, oqp, oqa = oracle64.rollout(td, Q0, np.zeros(6), want_state=True)
    has = np.where((ocol < 0).any(axis=(1, 2)))[0]
    assert len(has) >= 8
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
    r32 = lambda a: np.array(a, dtype=np.float32).astype(np.float64)       # the states as the kernel sees them
    return r32(qps), r32(qvs), r32(wms)


def test_contact_states_in_one_launch_against_the_oracle(planner, contact_states, oracle64, oracle32):
    qpos, qvel, warm = contact_states
    n = len(qpos)
    assert n > 30
    got = step_states(planner, qpos, qvel, warm)
    worst_col, devs = 0.0, []
    for i in range(n):
        r64, r32 = oracle64.forward(qpos[i], qvel[i], warm[i]), oracle32.forward(qpos[i], qvel[i], warm[i])
        worst_col = max(worst_col, np.abs(got["collision"][i, 0] - r64["con_dist"][oracle64.mask]).max())
        scale = max(1.0, np.abs(r64["qacc"]).max())
        if np.abs(r32["qacc"] - r64["qacc"]).max() < 1e-3 * scale:
            devs.append(np.abs(got["qacc"][i, 0] - r64["qacc"]).max() / scale)
    assert worst_col < 1e-5
    dev = np.array(devs)
    assert len(dev) > 0.3 * n
    # the bracket-end rule of test_gpu_step.py (DESIGN.md section 3)
    assert (dev < 5e-2).all(), np.sort(dev)[-5:]
    assert (dev < 1e-3).mean() >= 0.85, np.sort(dev)[-10:]


def test_step_batch_equals_jit_step(planner, contact_states):
    qpos, qvel, warm = contact_states
    out = planner.step_batch(qpos, qvel, warm)
    assert set(out) == {"qpos", "qvel", "qacc", "qacc_warmstart", "overflow"}
    got = {k: v.cpu().numpy() for k, v in out.items()}
    assert not got["overflow"].any()
    for i in range(len(qpos)):
        ref = planner.jit_step(planner.mjx_model, dict(qpos=qpos[i], qvel=qvel[i], qacc_warmstart=warm[i]))
        assert _eq(got["qacc"][i], ref["qacc"].astype(np.float32)), i
        assert _eq(got["qacc_warmstart"][i], got["qacc"][i])
        np.testing.assert_allclose(got["qvel"][i], ref["qvel"], rtol=1e-6, atol=1e-6)
        np.testing.assert_allclose(got["qpos"][i], ref["qpos"], rtol=1e-6, atol=1e-6)
        assert abs(np.linalg.norm(got["qpos"][i, 9:13].astype(np.float64)) - 1.0) < 1e-6


@pytest.mark.parametrize("N", [1, 29, 1000])
def test_in_place_outputs_equal_separate_outputs(planner, N):
    T = 8
    rng = np.random.default_rng(N)
    qpos, qvel, warm = snapshot_states(planner, N)
    qpos[:, :6] += rng.uniform(-0.4, 0.4, size=(N, 6))
    td = rng.uniform(-0.8, 0.8, size=(N, 6 * T))
    sep = step_states(planner, qpos, qvel, warm, td=td)
    io = tuple(_dev(planner, a) for a in (qpos, qvel, warm))
    inp = step_states(planner, *io, td=td, out=io)
    for k in sep:
        assert _eq(inp[k], sep[k]), k
    pub = planner.step_batch(qpos, qvel, warm, thetadot=torch.as_tensor(td, dtype=torch.float32))
    assert _eq(pub["theta"].cpu().numpy(), sep["theta"]) and _eq(pub["qpos"].cpu().numpy(), sep["qpos"])
    assert _eq(pub["qacc"].cpu().numpy(), sep["qacc"][:, -1]) and _eq(pub["qvel"].cpu().numpy(), sep["qvel"])


@pytest.mark.parametrize("ticks", [1, 3])
def test_step_batch_leaves_planning_unchanged(ticks):
    """Before and after a step_batch call, compute_cem returns the same bits; with 3 ticks the tick runs as a captured
    CUDA graph and step_batch grows the library's rollout scratch past the planner's batch."""
    from manipulator_mujoco_b200 import cem_planner
    pl = cem_planner(num_dof=6, num_batch=100, num_steps=16, timestep=0.05, maxiter_cem=2, num_elite=0.05,
                     w_pos=20.0, w_rot=3.0, w_col=80.0, maxiter_projection=10)
    tp, tr = np.array([-0.3, -0.3, 0.5]), np.array([0.0, 1.0, 0.0, 0.0])
    host = lambda out: [o.cpu().numpy() if torch.is_tensor(o) else np.asarray(o) for o in out]
    for _ in range(ticks):
        before = host(pl.compute_cem(np.zeros(66), Q0, np.zeros(6), np.zeros(6), tp, tr))
    assert (pl._graph is not None) == (ticks == 3 and pl.use_cuda_graph)
    qpos, qvel, warm = snapshot_states(pl, 300)
    qpos[:, :6] += 0.3
    pl.step_batch(qpos, qvel, warm, thetadot=np.full((300, 6 * 5), 0.4))
    after = host(pl.compute_cem(np.zeros(66), Q0, np.zeros(6), np.zeros(6), tp, tr))
    for i, (a, b) in enumerate(zip(after, before)):
        assert np.array_equal(a, b), i
    pl.close()


def test_refusals(planner):
    from manipulator_mujoco_b200 import cem_planner
    lib, h, dev = planner._lib, planner._h, planner.device
    N = 4
    qp, qv, wm = (_dev(planner, a) for a in snapshot_states(planner, N))
    qo, vo, wo = torch.empty_like(qp), torch.empty_like(qv), torch.empty_like(wm)
    td = torch.zeros(N, 12, device=dev)
    st = planner._stream()

    def call(n=N, T=1, a=(qp, qv, wm), tdd=None, o=(qo, vo, wo), handle=h):
        return lib.cemk_step_states(handle, n, T, *map(_p, a), _p(tdd), *map(_p, o), None, None, None, None, None, None, st)

    assert call() == 0 and call(T=2, tdd=td) == 0
    torch.cuda.synchronize()
    assert call(n=0) == -1 and call(n=-3) == -1
    assert call(T=0) == -1 and call(T=0, tdd=td) == -1
    for i in range(3):
        a = [qp, qv, wm]; a[i] = None
        assert call(a=tuple(a)) == -1
        o = [qo, vo, wo]; o[i] = None
        assert call(o=tuple(o)) == -1
    assert call(T=2) == -1 and b"NULL" in lib.cemk_last_error()
    assert call(handle=None) == -1
    with pytest.raises(ValueError):
        planner.step_batch(np.zeros((N, 12)), np.zeros((N, 12)), np.zeros((N, 12)))
    with pytest.raises(ValueError):
        planner.step_batch(np.zeros((N, 13)), np.zeros((N, 12)), np.zeros((N + 1, 12)))
    with pytest.raises(ValueError):
        planner.step_batch(np.zeros((0, 13)), np.zeros((0, 12)), np.zeros((0, 12)))
    with pytest.raises(ValueError):
        planner.step_batch(np.zeros((N, 13)), np.zeros((N, 12)), np.zeros((N, 12)), thetadot=np.zeros((N, 7)))
    with pytest.raises(ValueError):
        planner.step_batch(np.zeros((N, 13)), np.zeros((N, 12)), np.zeros((N, 12)), thetadot=np.zeros((N + 1, 6)))
    pl7 = cem_planner(num_dof=7, num_batch=64, num_steps=16, timestep=0.05, maxiter_cem=1, num_elite=0.1,
                      w_pos=20.0, w_rot=3.0, w_col=80.0, maxiter_projection=5)
    try:
        assert call(handle=pl7._h) == -1 and b"DOF mismatch" in lib.cemk_last_error()
        with pytest.raises(NotImplementedError):
            pl7.step_batch(np.zeros((N, 13)), np.zeros((N, 12)), np.zeros((N, 12)))
    finally:
        pl7.close()
