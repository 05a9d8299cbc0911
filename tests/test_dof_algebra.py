"""Host-side algebra at DOF counts other than 6: what k_project relies on at num_dof = 12 (Q_inv block diagonal per DOF, the
structured per-DOF projection equal to the reference's dense iteration), and the planner's num_dof range check."""
import numpy as np
import pytest

from oracle.planner_ref import PlannerRef
from test_planner_algebra import structured_projection


@pytest.mark.parametrize("order", [5, 10, 15])
def test_q_inv_is_block_diagonal_per_dof_at_12_dof(order):
    nd, n1 = 12, order + 1
    pr = PlannerRef(nd, 8, 16, 0.05, 0.05, 20, 3, 80, 10, order=order)
    nv = nd * n1
    assert pr.nvar == nv and pr.Q_inv.shape == (nv + 5 * nd,) * 2
    scale = np.abs(pr.Q_inv).max()
    for d in range(nd):
        blk = pr.Q_inv[d * n1:(d + 1) * n1]
        assert np.abs(blk[:, d * n1:(d + 1) * n1] - pr.Q_inv[:n1, :n1]).max() < 1e-7 * scale
        assert np.abs(blk[:, nv + 5 * d:nv + 5 * d + 5] - pr.Q_inv[:n1, nv:nv + 5]).max() < 1e-7 * scale
        mask = np.ones(nv + 5 * nd, bool); mask[d * n1:(d + 1) * n1] = False; mask[nv + 5 * d:nv + 5 * d + 5] = False
        assert np.abs(blk[:, mask]).max() < 1e-7 * scale


@pytest.mark.parametrize("order", [5, 10, 15])
def test_structured_projection_equals_dense_reference_at_12_dof(order):
    nd, B, T = 12, 24, 16
    pr = PlannerRef(nd, B, T, 0.05, 0.05, 20, 3, 80, 10, order=order)
    rng = np.random.default_rng(order)
    xi = rng.normal(size=(B, pr.nvar)) * np.sqrt(10)
    st = pr.state_term(rng.uniform(-1.5, 1.5, nd), rng.normal(size=nd) * 0.1, rng.normal(size=nd) * 0.1, B)
    dense = pr.compute_projection_filter(xi, st)
    fast = structured_projection(pr, xi, st, 10)
    np.testing.assert_allclose(fast, dense, rtol=0, atol=2e-8 * max(1.0, np.abs(dense).max()))
    np.testing.assert_allclose(dense @ pr.A_eq.T, pr.boundary_vec(st), atol=1e-6 * max(1.0, np.abs(pr.A_eq).max()))


@pytest.mark.parametrize("num_dof", [0, 13, -6, 6.0, True])
def test_planner_refuses_dof_counts_outside_1_to_12(num_dof):
    """Checked before anything else (no device needed)."""
    from manipulator_mujoco_b200 import cem_planner
    with pytest.raises(ValueError, match="num_dof"):
        cem_planner(num_dof=num_dof, num_batch=8, num_steps=8, timestep=0.05, maxiter_cem=1, num_elite=0.5,
                    w_pos=1.0, w_rot=1.0, w_col=1.0, maxiter_projection=1)
