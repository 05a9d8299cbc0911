"""The planner algebra at DOF counts other than 6 (cem_planner(num_dof=n), 1 <= n <= 12, nvar up to 12 x 16 = 192): sampling,
projection filter + Bernstein evaluation, elite selection (rank-select and bitonic paths, the multi-GPU pack / merge records) and
mean / covariance (two-pass and blocked forms) against oracle/planner_ref.py built with the same num_dof and order.  The rollout
models scene A's 6-DOF arm only: the methods that need it refuse other DOF counts."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from pack_ref import stable_order, topk_pack_ref

pytestmark = pytest.mark.gpu

DOFS = [12, 7, 1]
ORDERS = [5, 10, 15]
B, T = 16384, 16
GRID = [(nd, o) for nd in DOFS for o in ORDERS]


@functools.lru_cache(maxsize=None)
def _pair(nd, order):
    import contextlib
    import io
    from manipulator_mujoco_b200 import cem_planner
    from oracle.planner_ref import PlannerRef
    with contextlib.redirect_stdout(io.StringIO()):
        pl = cem_planner(num_dof=nd, num_batch=B, num_steps=T, timestep=0.05, maxiter_cem=1, num_elite=0.05, w_pos=20.0, w_rot=3.0,
                         w_col=80.0, maxiter_projection=10, bernstein_order=order)
    pr = PlannerRef(nd, B, T, 0.05, 0.05, 20.0, 3.0, 80.0, 10, order=order)
    return pl, pr


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


@pytest.mark.parametrize("nd,order", GRID)
def test_constants_and_structure(nd, order):
    pl, pr = _pair(nd, order)
    nv = nd * (order + 1)
    assert pl.nvar == nv == pr.nvar
    assert tuple(pl.Q_inv.shape) == (nv + 5 * nd,) * 2 and tuple(pl.A_eq.shape) == (5 * nd, nv)
    # (the planner's basis and the restatement's agree to ~1e-16 relative, Q_inv to ~4e-8 of its largest entry)
    for name in ("A_theta", "A_thetadot", "A_thetaddot", "A_v_ineq", "A_a_ineq", "A_p_ineq", "A_eq"):
        ref = getattr(pr, name)
        np.testing.assert_allclose(getattr(pl, name).cpu().numpy(), ref, rtol=0, atol=1e-6 * np.abs(ref).max(), err_msg=name)
    np.testing.assert_allclose(pl.Q_inv.cpu().numpy(), pr.Q_inv, rtol=0, atol=1e-6 * np.abs(pr.Q_inv).max())
    rng = np.random.default_rng(nd)
    st = rng.normal(size=(3, 5 * nd)).astype(np.float32)
    np.testing.assert_array_equal(pl.compute_boundary_vec_batch(st).cpu().numpy(), pr.boundary_vec(st))
    np.testing.assert_array_equal(pl.compute_boundary_vec_single(st[1]).cpu().numpy(), pr.boundary_vec(st[1:2])[0])
    diffs, d = rng.normal(size=(4, nv)).astype(np.float32), rng.uniform(size=4).astype(np.float32)
    np.testing.assert_allclose(pl.vec_product(diffs, d).cpu().numpy(), d[:, None, None] * diffs[:, :, None] * diffs[:, None, :], rtol=1e-6)
    np.testing.assert_allclose(pl.comp_prod(diffs[0], float(d[0])).cpu().numpy(), d[0] * np.outer(diffs[0], diffs[0]), rtol=1e-6)


@pytest.mark.parametrize("nd,order", GRID)
def test_sampling(nd, order):
    """compute_xi_samples = mean + z L^T with the planner's own draws (k_chol66 up to nvar 96, k_chol_wide above)."""
    pl, pr = _pair(nd, order)
    nv = pl.nvar
    rng = np.random.default_rng(100 + nv)
    A = rng.normal(size=(nv, nv))
    cov = (A @ A.T / nv + np.eye(nv)).astype(np.float32)
    mean = rng.normal(size=nv).astype(np.float32)
    xi, key = pl.compute_xi_samples(3, mean, cov)
    assert tuple(xi.shape) == (B, nv)
    z = pl._normal(key).cpu().numpy().astype(np.float64)
    ref = pr.compute_xi_samples(z, mean.astype(np.float64), cov.astype(np.float64))
    err = np.abs(xi.cpu().numpy() - ref).max()
    print(f"[dof-errors] sampling nd={nd} order={order}: {err:.2e}")
    assert err < 3e-5, f"sampling max error {err:.3e} (nvar {nv})"


@pytest.mark.parametrize("nd,order", GRID)
def test_projection_and_bernstein(nd, order):
    """k_project with the DOF count at run time: the full batch (16 384 samples, rows checked on a fixed subset: every row is an
    independent problem) and a ragged batch of 1001, against the dense float64 restatement; thetadot = xi_f A_thetadot^T
    (layout dof * T + t) and the boundary rows A_eq xi_f = boundary_vec(state_term)."""
    pl, pr = _pair(nd, order)
    nv = pl.nvar
    rng = np.random.default_rng(200 + 16 * nd + order)
    st = pr.state_term(rng.uniform(-1.5, 1.5, nd), 0.1 * rng.normal(size=nd), 0.1 * rng.normal(size=nd), B)
    st = st.astype(np.float32)
    xs = (3 * rng.normal(size=(B, nv))).astype(np.float32)
    for nb, rows in ((B, np.sort(rng.choice(B, 512, replace=False))), (1001, np.arange(1001))):
        xf, td = pl._project(xs[:nb], st[:nb], True)
        assert tuple(td.shape) == (nb, nd * T)
        xf, td = xf.cpu().numpy(), td.cpu().numpy()
        np.testing.assert_array_equal(pl.compute_projection_filter(xs[:nb], st[:nb]).cpu().numpy(), xf)
        ref = pr.compute_projection_filter(xs[rows].astype(np.float64), st[rows].astype(np.float64))
        e_x = np.abs(xf[rows] - ref).max()
        assert e_x < 1e-4, f"B={nb}: xi_f max error {e_x:.3e}"
        x64 = xf.astype(np.float64)
        # thetadot from the kernel's own xi_f: an (order + 1)-term float32 dot product per entry, so its error is bounded by
        # (order + 2) 2^-24 times the summed magnitude of the terms (2e-6 covers order 15)
        tscale = np.abs(x64) @ np.abs(pr.A_thetadot.T)
        e_td = (np.abs(td - x64 @ pr.A_thetadot.T) / np.maximum(1.0, tscale)).max()
        assert e_td < 2e-6, f"B={nb}: thetadot relative error {e_td:.3e}"
        e_ref = np.abs(td[rows] - ref @ pr.A_thetadot.T).max()
        assert e_ref < 1e-4, f"B={nb}: thetadot vs reference max error {e_ref:.3e}"
        # the boundary rows hold up to float32 rounding, relative to the summed magnitude of the terms of A_eq xi_f (Pddot[0] of
        # order 15 sums to ~750); measured on a B200: at most 4e-8
        bscale = np.abs(x64) @ np.abs(pr.A_eq.T)
        e_b = (np.abs(x64 @ pr.A_eq.T - pr.boundary_vec(st[:nb].astype(np.float64))) / np.maximum(1.0, bscale)).max()
        assert e_b < 1e-6, f"B={nb}: boundary rows relative error {e_b:.3e}"
        print(f"[dof-errors] projection nd={nd} order={order} B={nb}: xi_f {e_x:.2e} thetadot(rel) {e_td:.2e} "
              f"thetadot(ref) {e_ref:.2e} boundary(rel) {e_b:.2e}")


@pytest.mark.parametrize("n", [8192, 16384])            # counting-rank kernel / bitonic network
@pytest.mark.parametrize("nd,order", [(12, 15), (12, 10), (7, 5), (1, 5)])
def test_elite_selection_is_stable_with_nan_last(nd, order, n):
    pl, _ = _pair(nd, order)
    nv = pl.nvar
    rng = np.random.default_rng(n + nv)
    cost = rng.uniform(0, 1000, n).astype(np.float32)
    cost[rng.integers(0, n, n // 5)] = 77.0                            # ties
    cost[[3, n // 2]] = np.nan
    cost[7], cost[11] = -5.0, np.inf
    xi = rng.normal(size=(n, nv)).astype(np.float32)
    xe, idx, ce = pl.compute_ellite_samples(cost, xi)
    ref = stable_order(cost)
    k = pl.ellite_num
    np.testing.assert_array_equal(idx.cpu().numpy(), ref)
    np.testing.assert_array_equal(xe.cpu().numpy(), xi[ref[:k]])
    np.testing.assert_array_equal(ce.cpu().numpy().view(np.int32), cost[ref[:k]].view(np.int32))


@pytest.mark.parametrize("nd,order", [(12, 10), (12, 15)])                # nvar 132, 192
def test_topk_pack_and_merge_of_sorted_lists(nd, order):
    """cemk_topk_pack on three shards (rank-select and bitonic paths) + cemk_merge_sorted_lists, bit-exact against the global
    stable top-k by (cost, global index), ties across shards and NaNs included."""
    from manipulator_mujoco_b200 import _lib
    pl, _ = _pair(nd, order)
    lib, h, nv = pl._lib, pl._h, pl.nvar
    rng = np.random.default_rng(nv)
    sizes, k = (3000, 9000, 5000), 700
    n = sum(sizes)
    cost = np.round(rng.uniform(0, 100, n), 1).astype(np.float32)        # one decimal: many ties
    cost[[7, 4000, 16000]] = np.nan
    xi = rng.normal(size=(n, nv)).astype(np.float32)
    packs, lo = [], 0
    for m in sizes:
        c, x = torch.tensor(cost[lo:lo + m], device="cuda"), torch.tensor(xi[lo:lo + m], device="cuda")
        keys = torch.empty(1 << (m - 1).bit_length(), dtype=torch.int64, device="cuda")
        pack = torch.empty(k, nv + 2, device="cuda")
        _lib.check(lib.cemk_topk_pack(h, m, _p(c), 1, lo, _p(keys), k, _p(x), _p(pack), None), lib)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(pack.cpu().numpy().view(np.int32), topk_pack_ref(cost[lo:lo + m], lo, k, xi[lo:lo + m]).view(np.int32))
        packs.append(pack)
        lo += m
    gathered = torch.cat(packs).contiguous()
    xe, ce = torch.empty(k, nv, device="cuda"), torch.empty(k, device="cuda")
    ge = torch.empty(k, dtype=torch.int32, device="cuda")
    _lib.check(lib.cemk_merge_sorted_lists(h, len(sizes), k, _p(gathered), k, _p(xe), _p(ce), _p(ge), None), lib)
    torch.cuda.synchronize()
    ref = stable_order(cost)[:k]
    np.testing.assert_array_equal(ge.cpu().numpy(), ref)
    np.testing.assert_array_equal(xe.cpu().numpy(), xi[ref])
    np.testing.assert_array_equal(ce.cpu().numpy().view(np.int32), cost[ref].view(np.int32))


@pytest.mark.parametrize("k", [819, 1638])                               # two-pass kernel / blocked update
@pytest.mark.parametrize("nd,order", GRID)
def test_mean_cov(nd, order, k):
    pl, pr = _pair(nd, order)
    nv = pl.nvar
    rng = np.random.default_rng(k + nv)
    ce = np.sort(rng.uniform(200, 260, k)).astype(np.float32)
    mp_ = rng.normal(size=nv).astype(np.float32)
    xe = (mp_ + rng.normal(size=(k, nv))).astype(np.float32)
    A = rng.normal(size=(nv, nv)).astype(np.float32)
    cp_ = (A @ A.T / nv + 10 * np.eye(nv)).astype(np.float32)
    mean, cov = pl.compute_mean_cov(ce, mp_, cp_, xe)
    mean2, cov2 = pl.compute_mean_cov(ce, mp_, cp_, xe)
    assert torch.equal(mean, mean2) and torch.equal(cov, cov2)            # fixed summation order
    rm, rc = pr.compute_mean_cov(ce.astype(np.float64), mp_.astype(np.float64), cp_.astype(np.float64), xe.astype(np.float64))
    e_m, e_c = np.abs(mean.cpu().numpy() - rm).max(), np.abs(cov.cpu().numpy() - rc).max()
    print(f"[dof-errors] mean_cov nd={nd} order={order} k={k}: mean {e_m:.2e} cov {e_c:.2e}")
    assert e_m < 3e-5 and e_c < 1e-4, f"k={k} nvar={nv}: mean error {e_m:.3e}, covariance error {e_c:.3e}"


def test_constructor_range_and_rollout_refusal():
    from manipulator_mujoco_b200 import cem_planner
    pl, _ = _pair(12, 10)
    assert pl.num_dof == 12 and pl.nvar == 132 and pl.ellite_num == 819
    assert pl.model.nq == 13 and pl.nslot == 187 and callable(pl.jit_step)      # scene A, as the reference loads it
    td = torch.zeros(4, 12 * T, device="cuda")
    for call in (lambda: pl.compute_rollout_batch(td, np.zeros(6), np.zeros(6)),
                 lambda: pl.cem_iter((None,) * 8, None),
                 lambda: pl.compute_cem(np.zeros(132))):
        with pytest.raises(NotImplementedError, match="6-DOF"):
            call()
    # the library refuses the rollout on a 12-DOF handle by itself
    with pytest.raises(RuntimeError, match="DOF mismatch"):
        pl._rollout(td, np.zeros(6), np.zeros(6), np.zeros(3), np.array([1.0, 0, 0, 0]), False)
    for bad in (0, 13):
        with pytest.raises(ValueError):
            cem_planner(num_dof=bad, num_batch=8, num_steps=8, timestep=0.05, maxiter_cem=1, num_elite=0.5,
                        w_pos=1.0, w_rot=1.0, w_col=1.0, maxiter_projection=1)
    for bad in (3, 16):                         # order 3: four coefficients for five boundary conditions (singular KKT matrix)
        with pytest.raises(ValueError, match="bernstein_order"):
            cem_planner(num_dof=6, num_batch=8, num_steps=8, timestep=0.05, maxiter_cem=1, num_elite=0.5,
                        w_pos=1.0, w_rot=1.0, w_col=1.0, maxiter_projection=1, bernstein_order=bad)
