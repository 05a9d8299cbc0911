"""Every compiled variant and size switch of the planner algebra against the float64 restatement (oracle/planner_ref.py):
all 26 k_project instantiations (NC = 4 .. 16, product path ND = 6 and run-time DOF count ND = 0) with one- and seven-warp CTAs,
the longest horizon cemk_set_horizon accepts per NC and its refusals, sampling across the k_chol66 / k_chol_wide switch,
mean / covariance across every kernel switch, elite selection on the product call's strided cost record, and the cost
(standalone and fused into the rollout) against the formula of mjx_planner.py:277-303.

Tolerances come from float32 arithmetic: either the same restatement run in float32, or an explicit error bound written next
to the check.  Every check prints its worst error on a `[variant-errors]` line."""
import contextlib
import copy
import ctypes as C
import functools
import io

import numpy as np
import pytest
import torch

from conftest import Q0, TARGET_POS, TARGET_ROT, planner_inputs
from pack_ref import stable_order

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                          # float32 unit roundoff
ERR_ARG = -1
PROJ_THREADS = 224                      # 32 PROJ_WARPS: the block size project_smem is checked for in cemk_set_horizon


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _hp(a):
    return a.ctypes.data_as(C.c_void_p)


def project_warps(nprob):
    """cemk.cu project_warps: warps per CTA of k_project (8 problems per warp, 148 SMs x 3 CTAs)."""
    warps = -(-nprob // 8)
    return min(7, max(1, -(-warps // (148 * 3))))


def t_max(nc):
    """The longest horizon cemk_set_horizon accepts: T <= 1024 and project_smem<NC>(T, 224) <= 227 KB."""
    pc, kpad = -(-nc // 4) * 4, (5 * nc + 6) // 4 * 4
    return min(1024, (227 * 1024 // 4 - nc * pc - kpad - 3 * nc * PROJ_THREADS) // (3 * pc))


@functools.lru_cache(maxsize=None)
def _pair(nd, order, T, num_batch=64):
    """A planner and the restatement at (nd, order, T).  Order 3 (nc = 4) is refused by cem_planner: four coefficients cannot
    meet the five boundary conditions of mjx_planner.py:163-164 (the KKT matrix is singular).  k_project<4, .> runs on the
    well-posed problem that keeps the three initial conditions (position, velocity, acceleration; one free coefficient per
    DOF): the handle of an order-4 planner is switched to nc = 4 and given that problem's tables (Kpe's last two columns zero),
    and the restatement keeps the same three conditions."""
    from manipulator_mujoco_b200 import _lib, cem_planner
    from oracle.planner_ref import PlannerRef
    with contextlib.redirect_stdout(io.StringIO()):
        pl = cem_planner(num_dof=nd, num_batch=num_batch, num_steps=T, timestep=0.05, maxiter_cem=1, num_elite=0.05, w_pos=20.0,
                         w_rot=3.0, w_col=80.0, maxiter_projection=10, bernstein_order=max(order, 4))
    pr = PlannerRef(nd, num_batch, T, 0.05, 0.05, 20.0, 3.0, 80.0, 10, order=order, boundary=5 if order > 3 else 3)
    if order == 3:
        n1, nv = 4, pr.nvar
        kpe = np.zeros((n1, 5))
        kpe[:, :3] = pr.Q_inv[:n1, nv:nv + 3]
        c32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
        tables = (c32(np.stack((pr.Pdot, pr.Pddot, pr.P))), c32(pr.Q_inv[:n1, :n1]), c32(kpe), c32([pr.v_max, pr.a_max, pr.p_max]))
        _lib.check(pl._lib.cemk_set_order(pl._h, 4), pl._lib)
        _lib.check(pl._lib.cemk_set_horizon(pl._h, T, *map(_hp, tables)), pl._lib)
        pl._nc4_tables = tables
    return pl, pr


def _project(pl, xs, st, iters, want_td, T):
    """cemk_project through the C ABI (thetadot NULL when not wanted)."""
    from manipulator_mujoco_b200 import _lib
    nd, B = pl.num_dof, xs.shape[0]
    xi, s = torch.tensor(xs, device="cuda"), torch.tensor(st, device="cuda")
    xf = torch.empty(B, xs.shape[1], device="cuda")
    td = torch.empty(B, nd * T, device="cuda") if want_td else None
    _lib.check(pl._lib.cemk_project(pl._h, B, iters, _p(xi), _p(s), _p(xf), _p(td), None), pl._lib)
    torch.cuda.synchronize()
    return xf.cpu().numpy(), (td.cpu().numpy() if want_td else None)


def _inputs(pr, B, seed):
    nd = pr.num_dof
    rng = np.random.default_rng(seed)
    st = pr.state_term(rng.uniform(-1.5, 1.5, nd), 0.1 * rng.normal(size=nd), 0.1 * rng.normal(size=nd), B).astype(np.float32)
    xs = (3 * rng.normal(size=(B, pr.nvar))).astype(np.float32)
    return xs, st, rng


def _check_projection(tag, pl, pr, xs, st, rows, iters, T):
    """xi_f on `rows` against the dense float64 restatement, thetadot and the boundary rows from the kernel's own xi_f, and the
    thetadot-free launch bit-equal.  xi_f tolerance: the restatement run in float32 (PlannerRef.astype) does the same
    iteration in float32 with sums of the same lengths; the kernel may round differently, so 4x its error, plus a floor of
    64 float32 ulps of the largest entry for rows where the float32 restatement happens to be near-exact."""
    xf, td = _project(pl, xs, st, iters, True, T)
    xf_only, _ = _project(pl, xs, st, iters, False, T)
    np.testing.assert_array_equal(xf_only.view(np.int32), xf.view(np.int32))
    ref_pr = copy.copy(pr)
    ref_pr.maxiter_projection = iters
    ref = ref_pr.compute_projection_filter(xs[rows].astype(np.float64), st[rows].astype(np.float64))
    r32 = ref_pr.astype(np.float32).compute_projection_filter(xs[rows], st[rows])
    scale = max(1.0, float(np.abs(ref).max()))
    e_x, e32 = np.abs(xf[rows] - ref).max(), np.abs(r32 - ref).max()
    tol = 4 * e32 + 64 * U * scale
    # thetadot = xi_f A_thetadot^T: an NC-term float32 dot product per entry, error <= (NC + 2) 2^-24 sum |terms| (test_gpu_dof)
    x64 = xf[rows].astype(np.float64)
    tscale = np.abs(x64) @ np.abs(pr.A_thetadot.T)
    e_td = (np.abs(td[rows] - x64 @ pr.A_thetadot.T) / np.maximum(1.0, tscale)).max()
    # boundary rows A_eq xi_f = b_eq hold to float32 rounding relative to the summed magnitude of the terms (test_gpu_dof)
    bscale = np.abs(x64) @ np.abs(pr.A_eq.T)
    e_b = (np.abs(x64 @ pr.A_eq.T - pr.boundary_vec(st[rows].astype(np.float64))) / np.maximum(1.0, bscale)).max()
    print(f"[variant-errors] projection {tag}: xi_f {e_x:.2e} (float32 restatement {e32:.2e}, tol {tol:.2e}) "
          f"thetadot(rel) {e_td:.2e} boundary(rel) {e_b:.2e}")
    assert e_x <= tol, f"{tag}: xi_f max error {e_x:.3e} > {tol:.3e}"
    assert e_td < 2e-6, f"{tag}: thetadot relative error {e_td:.3e}"
    assert e_b < 1e-6, f"{tag}: boundary rows relative error {e_b:.3e}"


# NC = order + 1 = 4 .. 16; ND = 6 (product path) and one other DOF count: 12 at odd orders (nvar up to 192), 5 at even ones
# (odd widths)
PROJ = [(nd, order, T) for order in range(3, 16) for nd in (6, 12 if order % 2 else 5) for T in (7, 50)]


@pytest.mark.parametrize("nd,order,T", PROJ)
def test_projection_every_instantiation(nd, order, T):
    """k_project<order + 1, 6 or 0> at T = 7 (not a multiple of four, below NC for NC > 7) and T = 50, with a ragged batch of 37
    (one warp per CTA) and a batch of B nd > 21 312 problems (seven warps per CTA, last warp partly idle)."""
    pl, pr = _pair(nd, order, T)
    big = 21312 // nd + 3
    assert project_warps(37 * nd) == 1 and project_warps(big * nd) == 7
    for B in (37, big):
        xs, st, rng = _inputs(pr, B, 1000 * order + 10 * nd + T + B)
        rows = np.unique(np.concatenate([rng.choice(B, 24, replace=False), [0, B - 1]]))
        _check_projection(f"nd={nd} nc={order + 1} T={T} B={B}", pl, pr, xs, st, rows, 10, T)


@pytest.mark.parametrize("nd,order", [(6, 8), (12, 13)])                 # ND = 6 at NC = 9, ND = 0 at NC = 14
@pytest.mark.parametrize("iters", [1, 25])
def test_projection_iteration_counts(nd, order, iters):
    pl, pr = _pair(nd, order, 50)
    for B in (37, 21312 // nd + 3):
        xs, st, rng = _inputs(pr, B, 77 + iters + B)
        rows = np.unique(np.concatenate([rng.choice(B, 16, replace=False), [B - 1]]))
        _check_projection(f"nd={nd} nc={order + 1} T=50 B={B} iters={iters}", pl, pr, xs, st, rows, iters, 50)


def _set_horizon(pl, T):
    """cemk_set_horizon with tables of the right size for T (the values do not matter for a refusal)."""
    nc = pl.nvar_single if not hasattr(pl, "_nc4_tables") else 4
    G = np.zeros((3, T, nc), np.float32)
    Kpp, Kpe, bnd = np.eye(nc, dtype=np.float32), np.zeros((nc, 5), np.float32), np.ones(3, np.float32)
    return pl._lib.cemk_set_horizon(pl._h, T, _hp(G), _hp(Kpp), _hp(Kpe), _hp(bnd))


@pytest.mark.parametrize("order", range(3, 16))
def test_longest_horizon(order):
    """The largest T cemk_set_horizon accepts for NC = order + 1 (1024, or the 227 KB shared-memory limit for NC >= 13) on the
    product path with seven warps per CTA; T_max + 1, 1 and 1025 are refused.  Nobody measured the error at these horizons
    before: the tolerance is the float32 restatement's (see _check_projection)."""
    T = t_max(order + 1)
    pl, pr = _pair(6, order, T)
    B = 21312 // 6 + 3
    xs, st, rng = _inputs(pr, B, 5000 + order)
    rows = np.unique(np.concatenate([rng.choice(B, 6, replace=False), [B - 1]]))
    _check_projection(f"longest horizon nd=6 nc={order + 1} T={T} B={B}", pl, pr, xs, st, rows, 10, T)
    for bad in (T + 1, 1, 1025):
        assert _set_horizon(pl, bad) == ERR_ARG, f"cemk_set_horizon accepted T = {bad} at nc = {order + 1}"


def test_refused_horizon_changes_nothing():
    """A refused cemk_set_horizon leaves the handle as it was: at NC = 16, T_max = 979, the same projection before and after a
    refused T_max + 1 (small batch, thetadot NULL)."""
    T = t_max(16)
    assert T == 979
    pl, pr = _pair.__wrapped__(6, 15, T)                  # a handle of its own: no earlier refusal has touched it
    xs, st, _ = _inputs(pr, 37, 99)
    before, _ = _project(pl, xs, st, 10, False, T)
    assert _set_horizon(pl, T + 1) == ERR_ARG
    after, _ = _project(pl, xs, st, 10, False, T)
    np.testing.assert_array_equal(after.view(np.int32), before.view(np.int32))


# ---------------------------------------------------------------------------------------------- sampling
@pytest.mark.parametrize("nd,order", [(6, 15), (12, 7), (7, 13), (9, 10)])      # nvar 96, 96 (k_chol66), 98, 99 (k_chol_wide)
@pytest.mark.parametrize("kind", ["well", "cem"])
def test_sampling_at_the_cholesky_switch(nd, order, kind):
    """compute_xi_samples on the planner's own draws for B = 1, 28, 29, 55 (SAMPLE_TILE = 28), with a well-conditioned covariance
    and with a CEM-like one: compute_mean_cov's output from fewer elites than nvar (rank-deficient elite part over a small
    cov_prev), which the sampler's 0.003 I makes positive definite.
    Bounds: L from k_chol66 / k_chol_wide (read back from the workspace) satisfies L L^T = cov + 0.003 I to the Cholesky backward
    error (nvar + 2) 2^-24 |L| |L^T| (x2), cov taken from its lower triangle, the only one the kernel (and np.linalg.cholesky)
    reads -- compute_mean_cov's two halves differ in rounding; xi = mean + z L^T with the kernel's L to (nvar + 2) 2^-24 (|mean| + |z| |L|^T) (x2);
    xi against the float64 reference within 4x the error of the same computation in float32 (float32 Cholesky of the float32
    matrix, float32 product), and never tighter than the existing tests' 3e-5."""
    from manipulator_mujoco_b200 import _lib
    pl, pr = _pair(nd, order, 16)
    nv = pl.nvar
    rng = np.random.default_rng(nv + (kind == "cem"))
    mean = rng.normal(size=nv).astype(np.float32)
    if kind == "well":
        A = rng.normal(size=(nv, nv))
        cov = (A @ A.T / nv + np.eye(nv)).astype(np.float32)
    else:
        k = nv // 3
        ce = np.sort(rng.uniform(200, 230, k)).astype(np.float32)
        xe = (mean + rng.normal(size=(k, nv))).astype(np.float32)
        _, c = pl.compute_mean_cov(ce, mean, (1e-3 * np.eye(nv)).astype(np.float32), xe)
        cov = c.cpu().numpy()
    z = pl._normal(pl._split0(3))[:55].contiguous()
    zn = z.cpu().numpy().astype(np.float64)
    low = np.tril(cov.astype(np.float64))
    c64 = low + np.tril(low, -1).T + 0.003 * np.eye(nv)
    ref = pr.compute_xi_samples(zn, mean.astype(np.float64), cov.astype(np.float64))
    L32 = np.linalg.cholesky(cov + np.float32(0.003) * np.eye(nv, dtype=np.float32))
    x32 = mean + z.cpu().numpy() @ L32.T
    dm, dc = torch.tensor(mean, device="cuda"), torch.tensor(cov, device="cuda")
    for B in (1, 28, 29, 55):
        ws, xi = torch.empty(nv * nv, device="cuda"), torch.empty(B, nv, device="cuda")
        _lib.check(pl._lib.cemk_sample(pl._h, B, _p(z), _p(dm), _p(dc), _p(ws), _p(xi), None), pl._lib)
        torch.cuda.synchronize()
        L = ws.cpu().numpy().reshape(nv, nv).astype(np.float64)
        assert not np.triu(L, 1).any()
        e_l = (np.abs(L @ L.T - c64) / (np.abs(L) @ np.abs(L.T))).max()
        x = xi.cpu().numpy()
        own = mean + zn[:B] @ L.T
        e_own = (np.abs(x - own) / (np.abs(mean) + np.abs(zn[:B]) @ np.abs(L.T))).max()
        e_ref, e32 = np.abs(x - ref[:B]).max(), np.abs(x32[:B] - ref[:B]).max()
        tol = max(3e-5, 4 * e32)                          # 3e-5: the bound of the existing well-conditioned tests
        print(f"[variant-errors] sampling nvar={nv} {kind} B={B}: L backward(rel) {e_l:.2e} xi vs own L(rel) {e_own:.2e} "
              f"xi vs reference {e_ref:.2e} (float32 restatement {e32:.2e}, tol {tol:.2e})")
        assert e_l <= 2 * (nv + 2) * U, f"B={B}: Cholesky backward error {e_l:.3e}"
        assert e_own <= 2 * (nv + 2) * U, f"B={B}: sample error with the kernel's own L {e_own:.3e}"
        assert e_ref <= tol, f"B={B}: xi max error {e_ref:.3e} > {tol:.3e}"


# ---------------------------------------------------------------------------------------------- mean / covariance
MC_SIZES = {96: (6, 15), 98: (7, 13), 126: (9, 13), 128: (8, 15), 192: (12, 15)}
MC_KS = [1, 1023, 1024, 1025, 8192, 8193, 12000]
MC_CASES = [(nv, k, "spread") for nv in MC_SIZES for k in MC_KS] + [(128, k, c) for k in MC_KS for c in ("equal", "wide")]


@pytest.mark.parametrize("nv,k,costs", MC_CASES)
def test_mean_cov_at_every_switch(nv, k, costs):
    """k_mean_cov (k < 1024 and k > 8192; weights recomputed past 4096), k_mc_partial / _wide (nvar <= 96 / above) +
    k_mc_finish<128 / 256> (nvar < 128 / above) for 1024 <= k <= 8192, at both sides of every switch and block remainder.
    Costs: spread over a few lambda, all equal, or over more than 100 lambda (most weights underflow to zero in float32).
    Bound: every sum of the update is a float32 chain of at most m = (elites per thread group) + (groups) terms (two-pass:
    G = 512 // nvar groups; blocked: 32 per block + the blocks), so its error is <= m 2^-24 times the sum of the magnitudes of its
    terms; with the division by the weight sum and the final blend that gives, per entry,
      mean: 2 (m + 8) 2^-24 am (sum w |x|) / sum w,   cov: 2 (m + 8) 2^-24 ac (sum w (|x_r - a_r| + |d_r|)(|x_c - a_c| + |d_c|)) / sum w
    (a = mean_prev, d = new mean - a: the blocked form sums about a), on top of the tolerances of the existing tests."""
    nd, order = MC_SIZES[nv]
    pl, pr = _pair(nd, order, 16)
    assert pl.nvar == nv
    rng = np.random.default_rng(k + nv + len(costs))
    if costs == "spread":
        ce = np.sort(rng.uniform(200, 260, k))
    elif costs == "equal":
        ce = np.full(k, 231.5)
    else:
        ce = np.sort(rng.uniform(200, 200 + 150 * pl.lamda, k))
    ce = ce.astype(np.float32)
    mp_ = rng.normal(size=nv).astype(np.float32)
    xe = (mp_ + rng.normal(size=(k, nv))).astype(np.float32)
    A = rng.normal(size=(nv, nv)).astype(np.float32)
    cp_ = (A @ A.T / nv + 10 * np.eye(nv)).astype(np.float32)
    mean, cov = pl.compute_mean_cov(ce, mp_, cp_, xe)
    mean2, cov2 = pl.compute_mean_cov(ce, mp_, cp_, xe)
    assert torch.equal(mean, mean2) and torch.equal(cov, cov2)                     # fixed summation order
    c64, m64, x64 = ce.astype(np.float64), mp_.astype(np.float64), xe.astype(np.float64)
    rm, rc = pr.compute_mean_cov(c64, m64, cp_.astype(np.float64), x64)
    blocked = 1024 <= k <= 8192
    m = (32 + -(-k // 32) + 16) if blocked else (-(-k // (512 // nv)) + 512 // nv)
    w = np.exp(-(c64 - c64.min()) / pr.lamda)
    sw = w.sum()
    tol_m = 3e-5 + 2 * (m + 8) * U * pr.alpha_mean * (w @ np.abs(x64)) / sw
    dev = np.abs(x64 - m64) + np.abs(rm - m64)
    tol_c = 1e-4 + 2 * (m + 8) * U * pr.alpha_cov * (dev.T * w) @ dev / sw
    e_m, e_c = np.abs(mean.cpu().numpy() - rm), np.abs(cov.cpu().numpy() - rc)
    print(f"[variant-errors] mean_cov nvar={nv} k={k} {costs}: mean {e_m.max():.2e} (worst err/tol {(e_m / tol_m).max():.2f}) "
          f"cov {e_c.max():.2e} (worst err/tol {(e_c / tol_c).max():.2f})")
    assert (e_m <= tol_m).all(), f"mean error {e_m.max():.3e}"
    assert (e_c <= tol_c).all(), f"covariance error {e_c.max():.3e}"
    if blocked:
        # the elite part of the blocked update is exactly symmetric (one value written to both halves)
        c = cov.cpu().numpy()
        np.testing.assert_allclose(c - 0.4 * cp_, (c - 0.4 * cp_).T, rtol=0, atol=1e-5)


# ---------------------------------------------------------------------------------------------- elite selection
@pytest.mark.parametrize("n", [5000, 20000])                     # counting-rank kernel / bitonic network
def test_argsort_topk_on_the_cost_record(n):
    """The single-GPU product call (planner._select_elites): cost read from column 0 of the [n][4] cost record (stride 4, the
    other columns NaN), idx_base != 0; k = n // 20, k = n, and k = 0 with idx_sorted only.  Bit-exact."""
    from manipulator_mujoco_b200 import _lib
    pl, _ = _pair(6, 10, 16)
    rng = np.random.default_rng(n)
    cost = np.round(rng.uniform(0, 50, n), 1).astype(np.float32)
    cost[[3, n // 3]] = np.nan
    cost[[5, 6, n - 2]] = (-0.0, 0.0, -0.0)
    rec = np.full((n, 4), np.nan, np.float32)
    rec[:, 0] = cost
    xi = rng.normal(size=(n, 66)).astype(np.float32)
    base = 123457
    d_rec, d_xi = torch.tensor(rec, device="cuda"), torch.tensor(xi, device="cuda")
    keys = torch.empty(1 << (n - 1).bit_length(), dtype=torch.int64, device="cuda")
    ref = stable_order(cost)
    for k in (n // 20, n, 0):
        idx = torch.empty(n, dtype=torch.int32, device="cuda")
        xe = torch.empty(max(k, 1), 66, device="cuda") if k else None
        ce = torch.empty(max(k, 1), device="cuda") if k else None
        _lib.check(pl._lib.cemk_argsort_topk(pl._h, n, _p(d_rec), 4, base, _p(keys), _p(idx), k, _p(d_xi) if k else None,
                                             _p(xe), _p(ce), None), pl._lib)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(idx.cpu().numpy(), ref + base)
        if k:
            np.testing.assert_array_equal(xe.cpu().numpy().view(np.int32), xi[ref[:k]].view(np.int32))
            np.testing.assert_array_equal(ce.cpu().numpy().view(np.int32), cost[ref[:k]].view(np.int32))


# ---------------------------------------------------------------------------------------------- cost
def _cost_bounds(eef_pos, eef_rot, col, tp, tr, w):
    """Float64 formula (PlannerRef.compute_cost_single) and float32 error bounds of one sample's cost4.
    cost_g: T square roots of 3-term sums (relative error <= 4 2^-24 each) summed in a chain of <= T + 5 terms.
    cost_r: 2 acos(dp) per step; dp = |q . t| / (|q| |t|) carries a float32 error delta <= 16 2^-24, and acos turns it into
      |acos(dp +- delta) - acos(dp)| (<= sqrt(2 delta) at dp = 1, where acos is ill-conditioned), plus acosf's own error (8 ulps allowed).
    cost_c: the per-term errors 3 2^-24 (|c_t| + |c_t+1|) (the float32 constant 1 - 0.005 included) and a chain of at most
      T nslot terms, all non-negative: T nslot 2^-24 cost_c (the counts of c < 0 are exact)."""
    T, ns = col.shape
    cg = np.linalg.norm(eef_pos - tp, axis=1)
    dp = np.clip(np.abs((eef_rot / np.linalg.norm(eef_rot, axis=1)[:, None]) @ (tr / np.linalg.norm(tr))), 0.0, 1.0)
    d = 16 * U
    e_r = 2 * np.maximum(np.arccos(np.clip(dp - d, 0, 1)) - np.arccos(dp), np.arccos(dp) - np.arccos(np.clip(dp + d, 0, 1)))
    ar = 2 * np.arccos(dp)
    tol_g = 4 * U * cg.sum() + (T + 5) * U * cg.sum() + 1e-7
    tol_r = e_r.sum() + 8 * U * ar.sum() + (T + 5) * U * ar.sum() + 1e-7
    g = np.maximum(-col[1:] + col[:-1] - 0.005 * col[:-1], 0)
    cc = g.sum() + (col < 0).sum()
    tol_c = 3 * U * (np.abs(col[1:]) + np.abs(col[:-1])).sum() + T * ns * U * cc + 1e-7
    tol = w[0] * tol_g + w[1] * tol_r + w[2] * tol_c + 3 * U * (w[0] * cg.sum() + w[1] * ar.sum() + w[2] * cc)
    return np.array([tol, tol_g, tol_r, tol_c]), np.array([(dp > 1 - 1e-6).sum(), (dp > 1 - 1e-3).sum()])


@pytest.mark.parametrize("T", [1, 31, 32, 33, 100])
@pytest.mark.parametrize("nslot", [1, 33, 187])
def test_cost_batch_against_formula(T, nslot):
    """cemk_cost_batch (a warp per sample, the time loop strided over 32 lanes, 4 samples per CTA) with per-sample targets,
    B = 37: negative distances, +1 sentinels switching to small values, non-unit eef and target quaternions, and eef
    orientations equal to +-target (dp = 1, where acos is ill-conditioned)."""
    from oracle.planner_ref import PlannerRef
    pl, _ = _pair(6, 10, 16)
    B = 37
    rng = np.random.default_rng(T * 1000 + nslot)
    ep = rng.uniform(-1, 1, (B, T, 3)).astype(np.float32)
    er = (rng.normal(size=(B, T, 4)) * rng.uniform(0.5, 2.0, (B, T, 1))).astype(np.float32)
    tp = rng.uniform(-1, 1, (B, 3)).astype(np.float32)
    tr = (rng.normal(size=(B, 4)) * rng.uniform(0.5, 2.0, (B, 1))).astype(np.float32)
    same = rng.random((B, T)) < 0.3                                   # eef orientation = +-target, scaled
    er[same] = (tr[:, None, :] * rng.choice([-2.5, -1.0, 0.7, 1.0], (B, T, 1))).astype(np.float32)[same]
    col = np.where(rng.random((B, T, nslot)) < 0.6, 1.0, rng.uniform(-0.05, 0.2, (B, T, nslot))).astype(np.float32)
    w = (20.0, 3.0, 80.0)
    pr = PlannerRef(6, B, max(T, 2), 0.05, 0.05, *w, 10)
    out = np.stack([c.cpu().numpy() for c in pl.compute_cost_batch(None, ep, er, col, tp, tr)], axis=1)
    worst, nnear = np.zeros(4), np.zeros(2, int)
    for b in range(B):
        ref = np.array(pr.compute_cost_single(*(a.astype(np.float64) for a in (ep[b], er[b], col[b], tp[b], tr[b]))))
        tol, nn = _cost_bounds(*(a.astype(np.float64) for a in (ep[b], er[b], col[b], tp[b], tr[b])), w)
        nnear += nn
        err = np.abs(out[b] - ref)
        worst = np.maximum(worst, err / tol)
        assert (err <= tol).all(), f"sample {b}: cost4 error {err} > {tol}"
    print(f"[variant-errors] cost_batch T={T} nslot={nslot}: worst err/tol cost {worst[0]:.2f} g {worst[1]:.2f} r {worst[2]:.2f} "
          f"c {worst[3]:.2f}; sample-steps with dp > 1 - 1e-6: {nnear[0]}, > 1 - 1e-3: {nnear[1]}")


@pytest.mark.parametrize("target", ["scene", "hand"])
def test_fused_cost_at_bench_size_against_formula(target):
    """cemk_rollout_cost at 4096 x 100 (the bench size) on planner-distributed samples: cost4 against the float64 formula on the
    kernel's own eef_pos / eef_rot / collision dumps, every sample whose dumps are finite, contact samples included (the
    near-pass booking feeds cost_c).  Bounds as in _cost_bounds.  `hand`: the target orientation is a hand pose from inside the
    batch -- the hand at t = 0, where every sample starts from the same state -- so that many sample-steps have dp close to 1."""
    pl, _ = _pair(6, 10, 100, num_batch=4096)
    B, T = 4096, 100
    pr, _z, _xi, _st, _xif, td = planner_inputs(T, B, seed=41)
    tp, tr = TARGET_POS, TARGET_ROT
    if target == "hand":
        er0 = pl._rollout(td, Q0, np.zeros(6), tp, tr, True)[3].cpu().numpy().astype(np.float64)
        tr = er0[0, 0] / np.linalg.norm(er0[0, 0])
    theta, cost4, ep, er, col = pl._rollout(td, Q0, np.zeros(6), tp, tr, True)
    c4, ep, er, col = (a.cpu().numpy() for a in (cost4, ep, er, col))
    ok = np.isfinite(ep).all(axis=(1, 2)) & np.isfinite(er).all(axis=(1, 2)) & np.isfinite(col).all(axis=(1, 2))
    assert ok.mean() > 0.9
    w = (20.0, 3.0, 80.0)
    tr32 = np.asarray(tr, np.float32).astype(np.float64)
    worst, nnear, ncontact = np.zeros(4), np.zeros(2, int), 0
    for b in np.flatnonzero(ok):
        args = (ep[b].astype(np.float64), er[b].astype(np.float64), col[b].astype(np.float64), np.asarray(tp, np.float64), tr32)
        ref = np.array(pr.compute_cost_single(*args))
        tol, nn = _cost_bounds(*args, w)
        nnear += nn
        ncontact += bool((col[b] < 0).any())
        err = np.abs(c4[b] - ref)
        worst = np.maximum(worst, err / tol)
        assert (err <= tol).all(), f"sample {b}: cost4 {c4[b]} vs formula {ref} (error {err}, bound {tol})"
    print(f"[variant-errors] fused cost 4096x100 target={target}: {ok.sum()} finite samples, {ncontact} with contacts, "
          f"sample-steps with dp > 1 - 1e-6: {nnear[0]}, > 1 - 1e-3: {nnear[1]}; "
          f"worst err/tol cost {worst[0]:.2f} g {worst[1]:.2f} r {worst[2]:.2f} c {worst[3]:.2f}")
