"""GPU parity of the planner-algebra kernels (through the C ABI) against oracle/planner_ref.py."""
import numpy as np
import pytest
import torch

from conftest import Q0, planner_inputs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def planner():
    from manipulator_mujoco_b200 import cem_planner
    return cem_planner(num_dof=6, num_batch=512, num_steps=50, timestep=0.05, maxiter_cem=1, num_elite=0.05,
                       w_pos=20.0, w_rot=3.0, w_col=80.0, maxiter_projection=10)


def test_constants_match_reference_shapes(planner):
    """Shapes recorded in the reference notebooks (SURVEY.md section 4)."""
    assert tuple(planner.Q_inv.shape) == (96, 96) and tuple(planner.A_eq.shape) == (30, 66)
    assert tuple(planner.A_theta.shape) == (300, 66) and planner.P.shape == (50, 11)
    assert planner.nvar == 66 and planner.ellite_num == 25 and planner.nslot == 187
    assert planner.hande_id == 9 and planner.tcp_id == planner._mc.site_id("tcp")
    np.testing.assert_array_equal(planner.geom_ids, [33, 7, 12, 13, 18, 19, 23, 27, 28, 30])
    assert int(planner.mask.sum()) == 187 and planner.mask.shape[0] == 215


def test_sample(planner):
    rng = np.random.default_rng(0)
    A = rng.normal(size=(66, 66))
    cov = (A @ A.T / 66 + np.eye(66)).astype(np.float32)
    mean = rng.normal(size=66).astype(np.float32)
    from manipulator_mujoco_b200 import jax_prng
    xi, key = planner.compute_xi_samples(5, mean, cov)                 # integer seed = PRNGKey(5)
    np.testing.assert_array_equal(key, jax_prng.split(jax_prng.PRNGKey(5))[0])
    z = planner._normal(key).cpu().numpy().astype(np.float64)
    L = np.linalg.cholesky(cov.astype(np.float64) + 0.003 * np.eye(66))
    np.testing.assert_allclose(xi.cpu().numpy(), mean + z @ L.T, rtol=0, atol=2e-5)
    # same key -> same draws (the reference never advances self.key, mjx_planner.py:388)
    xi2, _ = planner.compute_xi_samples(5, mean, cov)
    assert torch.equal(xi, xi2)


def test_projection_filter_and_bernstein(planner):
    pr, z, xi, st, xif, td = planner_inputs(50, 512)
    out = planner.compute_projection_filter(xi, st).cpu().numpy()
    # float32 structured kernel vs float64 dense reference iteration (10 ADMM steps)
    np.testing.assert_allclose(out, xif, rtol=0, atol=5e-5)
    xf, thetadot = planner._project(xi, st, True)
    np.testing.assert_allclose(thetadot.cpu().numpy(), xif @ pr.A_thetadot.T, rtol=0, atol=5e-5)
    # layout: index = dof * T + t (mjx_planner.py:144,271)
    np.testing.assert_allclose(thetadot.cpu().numpy().reshape(512, 6, 50)[:, 2, :], xf.cpu().numpy()[:, 22:33] @ pr.Pdot.T.astype(np.float32), atol=1e-4)


@pytest.mark.parametrize("T,B", [(7, 3), (16, 1000), (100, 37), (400, 9)])
def test_projection_filter_across_horizons_and_ragged_batches(T, B):
    """k_project deals 8 problems x 4 time slices to a warp: horizons that are not a multiple of four, batches that leave the last
    warp partly idle, a batch smaller than a warp's 8 problems / 6, and a long horizon (more shared memory per CTA)."""
    from manipulator_mujoco_b200 import cem_planner
    pl = cem_planner(num_dof=6, num_batch=B, num_steps=T, timestep=0.05, maxiter_cem=1, num_elite=0.5, w_pos=20.0, w_rot=3.0, w_col=80.0,
                     maxiter_projection=10)
    pr, z, xi, st, xif, td = planner_inputs(T, B, seed=T)
    xf, thetadot = pl._project(xi, st, True)
    scale = max(1.0, float(np.abs(xif).max()))
    np.testing.assert_allclose(xf.cpu().numpy(), xif, rtol=0, atol=5e-5 * scale)
    np.testing.assert_allclose(thetadot.cpu().numpy(), xif @ pr.A_thetadot.T, rtol=0, atol=5e-5 * max(1.0, float(np.abs(td).max())))


@pytest.mark.parametrize("n", [1, 5, 100, 1000, 4096, 5000, 8192, 8193, 20000])   # <= 8192: counting-rank kernel, above: bitonic network
def test_argsort_topk_is_stable_with_nan_last(planner, n):
    """jnp.argsort's order (mjx_planner.py:307): NaNs of any sign and payload last, -0.0 tied with +0.0 (lax's sort maps -0.0 to
    +0.0), subnormals apart from zero, ties by index; signed zeros straddle the top-k cut."""
    rng = np.random.default_rng(n)
    cost = rng.uniform(0, 1000, n).astype(np.float32)
    bits = lambda *u: np.array(u, np.uint32).view(np.float32)
    k = max(1, n // 20)
    if n == 1:
        cost[0] = -0.0
    elif n == 5:
        cost[:] = [0.0, -0.0, 1.0, -0.0, 0.0]                        # k = 1: the +0.0 at index 0 wins
    else:
        cost[rng.integers(0, n, n // 5)] = 77.0           # ties
        cost[[3, n // 2]] = np.nan
        cost[[7]] = -5.0
        cost[[11]] = np.inf
        cost[[13, 17, 19, 23]] = bits(0xffc00000, 0x7f800001, 0xffffffff, 0x7fc12345)   # -NaN, signalling and payload NaNs
        cost[[29, 31]] = -np.inf
        cost[[37, 41, 43, 47]] = bits(0x80000001, 0x00000001, 0x807fffff, 0x007fffff)   # -+ smallest and largest subnormals
        zeros = rng.choice(np.arange(50, n), 8, replace=False)
        cost[zeros] = np.where(np.arange(8) % 3 == 0, 0.0, -0.0).astype(np.float32)
        # negative costs in front, so that positions k - 4 .. k + 3 of the order are the eight signed zeros
        free = np.setdiff1d(np.arange(50, n), zeros)
        nneg = k - 4 - int((cost < 0).sum())
        if nneg > 0:
            cost[rng.choice(free, nneg, replace=False)] = -rng.uniform(1, 100, nneg).astype(np.float32)
    xi = rng.normal(size=(n, 66)).astype(np.float32)
    old = planner.ellite_num
    planner.ellite_num = max(1, n // 20)
    try:
        xe, idx, ce = planner.compute_ellite_samples(cost, xi)
    finally:
        planner.ellite_num = old
    key = np.where(np.isnan(cost), np.inf, cost)
    ref = np.lexsort((np.arange(n), np.isnan(cost), key))
    np.testing.assert_array_equal(idx.cpu().numpy(), ref)
    np.testing.assert_array_equal(xe.cpu().numpy(), xi[ref[:k]])
    np.testing.assert_array_equal(ce.cpu().numpy().view(np.int32), cost[ref[:k]].view(np.int32))


def test_mean_cov(planner):
    pr, *_ = planner_inputs(50, 512)
    rng = np.random.default_rng(2)
    k = 204
    ce = np.sort(rng.uniform(200, 260, k)).astype(np.float32)
    xe = rng.normal(size=(k, 66)).astype(np.float32)
    mp_, cp_ = rng.normal(size=66).astype(np.float32), (10 * np.eye(66)).astype(np.float32)
    mean, cov = planner.compute_mean_cov(ce, mp_, cp_, xe)
    rm, rc = pr.compute_mean_cov(ce.astype(np.float64), mp_.astype(np.float64), cp_.astype(np.float64), xe.astype(np.float64))
    np.testing.assert_allclose(mean.cpu().numpy(), rm, rtol=0, atol=2e-5)
    np.testing.assert_allclose(cov.cpu().numpy(), rc, rtol=0, atol=5e-5)


@pytest.mark.parametrize("k,case", [(1023, "far"), (1024, "first"), (1638, "far"), (1638, "near"), (3276, "near"), (3276, "first")])
def test_mean_cov_large_elite_sets(planner, k, case):
    """Elite sets of the multi-GPU configurations (k >= 1024 takes the blocked single-pass update about mean_prev; 1023 is the
    last size of the two-pass kernel): against the float64 restatement of mjx_planner.py:326-335, with mean_prev far from the
    elites, near them (later CEM iterations) and at the sampler's mean (first iteration); deterministic run to run."""
    pr, *_ = planner_inputs(50, 8)
    rng = np.random.default_rng(k)
    ce = np.sort(rng.uniform(200, 260, k)).astype(np.float32)
    if case == "far":
        xe, mp_ = rng.normal(size=(k, 66)).astype(np.float32), rng.normal(size=66).astype(np.float32)
    elif case == "near":
        mp_ = (3 * rng.normal(size=66)).astype(np.float32)
        xe = (mp_ + 0.3 * rng.normal(size=(k, 66))).astype(np.float32)
    else:
        mp_, xe = np.zeros(66, np.float32), (np.sqrt(10) * rng.normal(size=(k, 66))).astype(np.float32)
    A = rng.normal(size=(66, 66)).astype(np.float32)
    cp_ = (A @ A.T / 66 + 10 * np.eye(66)).astype(np.float32)
    mean, cov = planner.compute_mean_cov(ce, mp_, cp_, xe)
    mean2, cov2 = planner.compute_mean_cov(ce, mp_, cp_, xe)
    assert torch.equal(mean, mean2) and torch.equal(cov, cov2)
    rm, rc = pr.compute_mean_cov(ce.astype(np.float64), mp_.astype(np.float64), cp_.astype(np.float64), xe.astype(np.float64))
    np.testing.assert_allclose(mean.cpu().numpy(), rm, rtol=0, atol=2e-5)
    np.testing.assert_allclose(cov.cpu().numpy(), rc, rtol=0, atol=5e-5)
    c = cov.cpu().numpy()
    if k >= 1024:
        # the elite part of the blocked update is exactly symmetric (one value written to both halves)
        np.testing.assert_allclose(c - 0.4 * cp_, (c - 0.4 * cp_).T, rtol=0, atol=1e-5)


def test_compute_cem_end_to_end_against_oracle_pipeline(oracle64):
    """One CEM iteration (C1-like config, T=16) through the public API vs the same pipeline assembled
    from the oracle pieces with the *same* normal draws: costs, elite set, new mean."""
    from manipulator_mujoco_b200 import cem_planner
    from oracle.planner_ref import PlannerRef
    B, T = 200, 16
    pl = cem_planner(num_dof=6, num_batch=B, num_steps=T, timestep=0.05, maxiter_cem=1, num_elite=0.05,
                     w_pos=20.0, w_rot=3.0, w_col=80.0, maxiter_projection=10)
    tp, tr = np.array([-0.3, -0.3, 0.5]), np.array([0.0, 1.0, 0.0, 0.0])
    cost, bg, br, bc, best_vels, best_traj, xi_mean, thetadot, theta = pl.compute_cem(np.zeros(66), Q0, np.zeros(6), np.zeros(6), tp, tr)
    assert best_vels.shape == (T, 6) and best_traj.shape == (T, 6) and xi_mean.shape == (66,)
    assert tuple(thetadot.shape) == (1, B, 6 * T) and tuple(theta.shape) == (1, B, 6 * T)
    # oracle pipeline with the planner's own z (jax.random cannot be reproduced; samples are injected)
    pr = PlannerRef(6, B, T, 0.05, 0.05, 20.0, 3.0, 80.0, 10)
    from manipulator_mujoco_b200 import jax_prng
    k1 = jax_prng.split(pl.key)[0]                                     # compute_cem (:388)
    k2 = jax_prng.split(k1)[0]                                         # compute_xi_samples (:314)
    z = pl._normal(k2).cpu().numpy().astype(np.float64)
    xi_ref = pr.compute_xi_samples(z, np.zeros(66), 10 * np.eye(66))
    xi_gpu, _ = pl.compute_xi_samples(k1, np.zeros(66), 10 * np.eye(66))              # the draws compute_cem used
    xi = xi_gpu.cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(xi, xi_ref, atol=5e-5)
    xif = pr.compute_projection_filter(xi, pr.state_term(Q0, np.zeros(6), np.zeros(6), B))
    td = xif @ pr.A_thetadot.T
    np.testing.assert_allclose(thetadot[0].cpu().numpy(), td, atol=5e-5)
    oth, oep, oer, ocol = oracle64.rollout(thetadot[0].cpu().numpy().astype(np.float64), Q0, np.zeros(6))
    np.testing.assert_allclose(theta[0].cpu().numpy(), oth, atol=5e-4)
    oc, ocg, ocr, occ = pr.compute_cost_batch(oep, oer, ocol, tp, tr)
    order = np.argsort(oc, kind="stable")
    k = pr.ellite_num
    # elite index set: bit-exact wherever the sorted-cost gap around the cut exceeds the cost tolerance
    tol = 2e-3 * np.abs(oc[order[k]])
    xe, ce = pl._last_elite
    got = set(pl._last_elite[1].cpu().numpy().tolist())
    assert abs(float(cost[0]) - oc[order[0]]) < tol
    if oc[order[k]] - oc[order[k - 1]] > 2 * tol:
        assert got == set(order[:k].tolist())
    else:
        assert len(got & set(order[:k + 3].tolist())) >= k - 1
    if oc[order[1]] - oc[order[0]] > 2 * tol:
        np.testing.assert_allclose(best_traj, oth[order[0]].reshape(6, T).T, atol=5e-4)
        np.testing.assert_allclose(best_vels, td[order[0]].reshape(6, T).T, atol=3e-4)
    xe_ref, _, ce_ref = pr.compute_ellite_samples(oc, xi)
    m_ref, _ = pr.compute_mean_cov(ce_ref, np.zeros(66), 10 * np.eye(66), xe_ref)
    if got == set(order[:k].tolist()):
        np.testing.assert_allclose(xi_mean, m_ref, atol=5e-3)


def test_topk_pack_and_merge_of_sorted_lists_equal_global_stable_topk(planner):
    """cemk_topk_pack on three shards (two rank-select, one bitonic) + cemk_merge_sorted_lists (the multi-GPU elite exchange
    without NCCL in between) must give the global stable top-k, ties and NaNs included."""
    import ctypes as C
    from manipulator_mujoco_b200 import _lib
    from pack_ref import merge_sorted_lists_ref, topk_pack_ref
    lib, h = planner._lib, planner._h
    rng = np.random.default_rng(4)
    sizes, k, nv = (1500, 1500, 9000), 150, 66
    n = sum(sizes)
    cost = rng.uniform(0, 100, n).astype(np.float32)
    cost[rng.integers(0, n, n // 5)] = 1.0                             # ties across all shards, the k-th best among them
    cost[[7, 2000, 9000]] = np.nan
    cost[[40, 1700, 1701, 5000]] = (0.0, -0.0, 0.0, -0.0)              # -0.0 ties with +0.0, within and across shards
    xi = rng.normal(size=(n, nv)).astype(np.float32)
    p = lambda t: C.c_void_p(t.data_ptr())
    packs, lo = [], 0
    for m in sizes:
        c = torch.tensor(cost[lo:lo + m], device="cuda"); x = torch.tensor(xi[lo:lo + m], device="cuda")
        keys = torch.empty(1 << (m - 1).bit_length(), dtype=torch.int64, device="cuda")
        pack = torch.empty(k, nv + 2, device="cuda")
        _lib.check(lib.cemk_topk_pack(h, m, p(c), 1, lo, p(keys), k, p(x), p(pack), None), lib)
        packs.append(pack)
        # the numpy restatement the gloo tests run on (tests/pack_ref.py) is the kernel's record, bit for bit
        np.testing.assert_array_equal(pack.cpu().numpy().view(np.int32), topk_pack_ref(cost[lo:lo + m], lo, k, xi[lo:lo + m]).view(np.int32))
        lo += m
    gathered = torch.cat(packs).contiguous()
    xe = torch.empty(k, nv, device="cuda"); ce = torch.empty(k, device="cuda"); ge = torch.empty(k, dtype=torch.int32, device="cuda")
    _lib.check(lib.cemk_merge_sorted_lists(h, len(sizes), k, p(gathered), k, p(xe), p(ce), p(ge), None), lib)
    torch.cuda.synchronize()
    key = np.where(np.isnan(cost), np.inf, cost)
    ref = np.lexsort((np.arange(n), np.isnan(cost), key))[:k]
    np.testing.assert_array_equal(ge.cpu().numpy(), ref)
    np.testing.assert_array_equal(xe.cpu().numpy(), xi[ref])
    np.testing.assert_array_equal(ce.cpu().numpy().view(np.int32), cost[ref].view(np.int32))
    rx, rc, rg = merge_sorted_lists_ref(gathered.cpu().numpy(), len(sizes), k, k)
    np.testing.assert_array_equal(ge.cpu().numpy(), rg)
    np.testing.assert_array_equal(xe.cpu().numpy(), rx)
    np.testing.assert_array_equal(ce.cpu().numpy().view(np.int32), rc.view(np.int32))


@pytest.mark.parametrize("nlist,kl", [(8, 500), (3, 1638), (8, 6200)])      # the last one exceeds the shared-memory key staging
def test_merge_of_many_sorted_lists_with_ties_across_lists(planner, nlist, kl):
    """cemk_merge_sorted_lists (what the planner runs after the all-gather): global stable top-k of `nlist` per-rank sorted
    lists, bit-exact against a lexsort on (cost, global index), with cost ties inside and across lists and NaNs."""
    import ctypes as C
    from manipulator_mujoco_b200 import _lib
    lib, h = planner._lib, planner._h
    rng = np.random.default_rng(11 + nlist)
    nv, Bl = 66, 4 * kl
    k = kl
    recs, allc, allg = [], [], []
    for a in range(nlist):
        c = np.round(rng.uniform(0, 30, kl), 1).astype(np.float32)          # one decimal: many ties
        if a % 3 == 0:
            c[rng.integers(0, kl, 3)] = np.nan
        if a < 3:                                   # zeros of both signs: +0.0 in list 0, -0.0 in list 1, both in list 2 (a tie)
            c[:4] = (0.0, 0.0, -0.0, -0.0) if a == 2 else (0.0 if a == 0 else -0.0)
        gi = a * Bl + np.sort(rng.choice(Bl, kl, replace=False))
        o = np.lexsort((gi, np.isnan(c), np.where(np.isnan(c), np.inf, c)))
        c, gi = c[o], gi[o]
        x = rng.normal(size=(kl, nv)).astype(np.float32)
        recs.append(np.concatenate([x, c[:, None], gi[:, None].astype(np.float32)], axis=1))
        allc.append(c); allg.append(gi)
    packed = torch.tensor(np.concatenate(recs), device="cuda").contiguous()
    p = lambda t: C.c_void_p(t.data_ptr())
    xe = torch.empty(k, nv, device="cuda"); ce = torch.empty(k, device="cuda"); ge = torch.empty(k, dtype=torch.int32, device="cuda")
    _lib.check(lib.cemk_merge_sorted_lists(h, nlist, kl, p(packed), k, p(xe), p(ce), p(ge), None), lib)
    torch.cuda.synchronize()
    c, g = np.concatenate(allc), np.concatenate(allg)
    ref = np.lexsort((g, np.isnan(c), np.where(np.isnan(c), np.inf, c)))[:k]
    np.testing.assert_array_equal(ge.cpu().numpy(), g[ref])
    np.testing.assert_array_equal(ce.cpu().numpy().view(np.int32), c[ref].view(np.int32))
    np.testing.assert_array_equal(xe.cpu().numpy(), np.concatenate(recs)[ref, :nv])


def test_tick_record_packs_what_compute_cem_returns(planner):
    """cemk_tick_record: per-iteration minimum + overflow count, and at the last iteration the best sample's rows and the new
    mean; with a best_row buffer (several GPUs) the rows go there, exact zeros when the sample lives on another rank even if
    this rank's data is NaN."""
    import ctypes as C
    from manipulator_mujoco_b200 import _lib
    lib, h = planner._lib, planner._h
    rng = np.random.default_rng(8)
    B, T, nv, m = 37, planner.num, planner.nvar, 3
    nd = 6 * T
    td, th = rng.normal(size=(B, nd)).astype(np.float32), rng.normal(size=(B, nd)).astype(np.float32)
    c4 = rng.uniform(size=(B, 4)).astype(np.float32)
    td[5, 3] = np.nan
    mean = rng.normal(size=nv).astype(np.float32)
    dv = lambda a: torch.tensor(a, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    d_td, d_th, d_c4, d_mean = dv(td), dv(th), dv(c4), dv(mean)
    out = torch.full((m + 2 * nd + 3 + nv + 1,), -7.0, device="cuda")
    flags_all, cmin = [], []
    for i in range(m):
        flags = rng.integers(0, 4, B).astype(np.int32)
        ce = np.sort(rng.uniform(size=4).astype(np.float32)); gi = np.array([11, 2, 30, 4], np.int32)
        d_f, d_ce, d_gi = dv(flags), dv(ce), dv(gi)
        _lib.check(lib.cemk_tick_record(h, i, m, int(i == m - 1), B, T, p(d_ce), p(d_gi), 0, p(d_f), p(d_td), p(d_th), p(d_c4), p(d_mean), p(out), None, None), lib)
        torch.cuda.synchronize()
        flags_all.append(int((flags & 1).sum())); cmin.append(ce[0])
    o = out.cpu().numpy()
    np.testing.assert_array_equal(o[:m], np.array(cmin, np.float32))
    np.testing.assert_array_equal(o[m:m + nd], td[11]); np.testing.assert_array_equal(o[m + nd:m + 2 * nd], th[11])
    np.testing.assert_array_equal(o[m + 2 * nd:m + 2 * nd + 3], c4[11, 1:])
    np.testing.assert_array_equal(o[m + 2 * nd + 3:m + 2 * nd + 3 + nv], mean)
    assert o[-1] == sum(flags_all)
    # several GPUs: this rank holds rows [100, 100 + B); the best sample 105 is local row 5 (which has a NaN), 11 is elsewhere
    row = torch.full((2 * nd + 3,), 5.0, device="cuda")
    for best, owned in ((105, True), (11, False), (100 + B, False)):
        d_gi = dv(np.array([best, 0], np.int32))
        _lib.check(lib.cemk_tick_record(h, 0, 1, 1, B, T, p(d_ce), p(d_gi), 100, p(d_f), p(d_td), p(d_th), p(d_c4), p(d_mean), p(out), p(row), None), lib)
        torch.cuda.synchronize()
        r = row.cpu().numpy()
        if owned:
            np.testing.assert_array_equal(r[:nd].view(np.int32), td[5].view(np.int32)); np.testing.assert_array_equal(r[nd:2 * nd], th[5])
            np.testing.assert_array_equal(r[2 * nd:], c4[5, 1:])
        else:
            assert not r.any() and not np.signbit(r).any()


def test_normal_draw_cache_is_only_a_cache(planner):
    """cem_planner keeps the normal draws of a key (the reference restarts from the same key every call); switching the cache off
    (what bench.py times) must give the same samples."""
    mean, cov = np.zeros(planner.nvar, np.float32), 10 * np.eye(planner.nvar, dtype=np.float32)
    old = planner.cache_normal_draws
    try:
        planner.cache_normal_draws = True
        a1, k1 = planner.compute_xi_samples(planner.key, mean, cov)
        a2, _ = planner.compute_xi_samples(planner.key, mean, cov)
        planner.cache_normal_draws = False
        b1, k2 = planner.compute_xi_samples(planner.key, mean, cov)
        b2, _ = planner.compute_xi_samples(planner.key, mean, cov)
    finally:
        planner.cache_normal_draws = old
    assert torch.equal(a1, a2) and torch.equal(a1, b1) and torch.equal(b1, b2)
    assert np.array_equal(np.asarray(k1), np.asarray(k2))


def test_graph_replay_equals_eager_ticks_with_a_large_elite_set():
    """compute_cem runs two eager ticks, captures the tick into a CUDA graph and replays it: every tick must return the same
    tuple bit for bit (the reference restarts from the same key).  20 480 samples = 1024 elites, which takes the blocked
    mean / covariance update (two launches on a library-owned workspace) and cemk_tick_record through capture and replay."""
    from manipulator_mujoco_b200 import cem_planner
    pl = cem_planner(num_dof=6, num_batch=20480, num_steps=16, timestep=0.05, maxiter_cem=2, num_elite=0.05, w_pos=20.0, w_rot=3.0, w_col=80.0,
                     maxiter_projection=10)
    assert pl.ellite_num == 1024
    tp, tr = np.array([-0.3, -0.3, 0.5]), np.array([0.0, 1.0, 0.0, 0.0])
    outs = [pl.compute_cem(np.zeros(66), Q0, np.zeros(6), np.zeros(6), tp, tr) for _ in range(4)]
    assert pl._graph is not None
    host = lambda a: a.cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    for o in outs[1:]:
        for a, b in zip(outs[0], o):
            np.testing.assert_array_equal(host(a), host(b))
    assert np.all(np.isfinite(outs[0][0])) and pl.overflow_samples == 0


def test_notebook_attributes_jit_step_and_vec_product(planner, oracle64):
    """mjx_planner.py:98,108: `vec_product` (vmapped outer product) and `jit_step` (one mjx.step of one environment),
    touched by mpc_planning.ipynb."""
    rng = np.random.default_rng(2)
    diffs, d = rng.normal(size=(5, 66)).astype(np.float32), rng.uniform(size=5).astype(np.float32)
    vp = planner.vec_product(diffs, d).cpu().numpy()
    np.testing.assert_allclose(vp, d[:, None, None] * diffs[:, :, None] * diffs[:, None, :], rtol=1e-6)
    data = dict(planner.mjx_data)
    data["qpos"] = data["qpos"].copy()
    data["qpos"][:6] = Q0
    data["qvel"] = np.zeros(12)
    data["qvel"][:6] = [0.2, -0.1, 0.3, 0.0, 0.1, -0.2]
    out = planner.jit_step(planner.mjx_model, data)
    ref = oracle64.forward(data["qpos"], data["qvel"], data["qacc_warmstart"])
    np.testing.assert_allclose(out["qacc"], ref["qacc"], atol=2e-3 * max(1.0, np.abs(ref["qacc"]).max()))
    np.testing.assert_allclose(out["qvel"], data["qvel"] + 0.05 * out["qacc"], atol=1e-12)
    np.testing.assert_allclose(out["qpos"][:9], data["qpos"][:9] + 0.05 * out["qvel"][:9], atol=1e-12)


@pytest.mark.parametrize("order", [5, 8, 12, 15])
def test_order_n_bernstein_pipeline(order):
    """SURVEY 8 f.4 (order-n half): cem_planner(bernstein_order=n) -- sampling, projection filter + Bernstein evaluation,
    elite selection and mean / covariance at nvar = 6 (n + 1), against the dense float64 restatement built with the same
    order (oracle/planner_ref.py, whose basis is pinned to the reference's bernstein_coeff_ordern_new(n, ...) golden)."""
    from manipulator_mujoco_b200 import cem_planner
    from oracle.planner_ref import PlannerRef
    B, T = 96, 16
    nv = 6 * (order + 1)
    pl = cem_planner(num_dof=6, num_batch=B, num_steps=T, timestep=0.05, maxiter_cem=2, num_elite=0.1, w_pos=20.0, w_rot=3.0,
                     w_col=80.0, maxiter_projection=10, bernstein_order=order)
    pr = PlannerRef(6, B, T, 0.05, 0.1, 20.0, 3.0, 80.0, 10, order=order)
    assert pl.nvar == nv == pr.nvar and tuple(pl.A_thetadot.shape) == (6 * T, nv)
    rng = np.random.default_rng(order)
    A = rng.normal(size=(nv, nv))
    cov = (A @ A.T / nv + np.eye(nv)).astype(np.float32)
    mean = rng.normal(size=nv).astype(np.float32)
    xi, key = pl.compute_xi_samples(3, mean, cov)
    z = pl._normal(key).cpu().numpy().astype(np.float64)
    ref_xi = pr.compute_xi_samples(z, mean.astype(np.float64), cov.astype(np.float64))
    np.testing.assert_allclose(xi.cpu().numpy(), ref_xi, rtol=0, atol=3e-5)
    st = pr.state_term(Q0, np.zeros(6), np.zeros(6), B)
    xs = (rng.normal(size=(B, nv)) * 3).astype(np.float32)
    xf, td = pl._project(xs, st, True)
    ref_xf = pr.compute_projection_filter(xs.astype(np.float64), st)
    np.testing.assert_allclose(xf.cpu().numpy(), ref_xf, rtol=0, atol=1e-4)
    np.testing.assert_allclose(td.cpu().numpy(), ref_xf @ pr.A_thetadot.T, rtol=0, atol=1e-4)
    k = pl.ellite_num
    ce = np.sort(rng.uniform(200, 260, k)).astype(np.float32)
    xe = rng.normal(size=(k, nv)).astype(np.float32)
    m2, c2 = pl.compute_mean_cov(ce, mean, cov, xe)
    rm, rc = pr.compute_mean_cov(ce.astype(np.float64), mean.astype(np.float64), cov.astype(np.float64), xe.astype(np.float64))
    np.testing.assert_allclose(m2.cpu().numpy(), rm, rtol=0, atol=3e-5)
    np.testing.assert_allclose(c2.cpu().numpy(), rc, rtol=0, atol=1e-4)
    cost = rng.uniform(0, 10, B).astype(np.float32)
    xi_e, idx, cost_e = pl.compute_ellite_samples(cost, xs)
    order_ref = np.argsort(cost, kind="stable")
    np.testing.assert_array_equal(idx.cpu().numpy(), order_ref)
    np.testing.assert_array_equal(xi_e.cpu().numpy(), xs[order_ref[:k]])
    # and the whole tick runs (two CEM iterations, graph capture on the third call)
    for _ in range(3):
        out = pl.compute_cem(np.zeros(nv), Q0, np.zeros(6), np.zeros(6), np.array([-0.3, -0.3, 0.5]), np.array([0.0, 1.0, 0.0, 0.0]))
    assert out[6].shape == (nv,) and np.isfinite(out[0]).all() and out[4].shape == (T, 6)
