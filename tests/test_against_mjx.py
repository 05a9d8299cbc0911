"""Ready-made hook for the day a real MJX oracle is available (SURVEY.md section 8c).

`mujoco`, `mujoco.mjx` and `jax` cannot be installed in this environment, so every test here is
skipped; with them importable (and MANIPULATOR_MUJOCO_REFERENCE naming a checkout of the upstream project) the tests compare
  * the MJCF compiler's constants against `mujoco.MjModel`,
  * the C oracle's rollout against `jax.vmap(lax.scan(mjx.step))` exactly as the reference planner
    builds it (mjx_planner.py:251-274),
which would turn "parity unpinned" into a pinned statement.  Never run so far -- best effort."""
import os

import numpy as np
import pytest

mujoco = pytest.importorskip("mujoco")
jax = pytest.importorskip("jax")
mjx = pytest.importorskip("mujoco.mjx")

REFERENCE = os.environ.get("MANIPULATOR_MUJOCO_REFERENCE", "")
REF_XML = os.path.join(REFERENCE, "sampling_based_planner", "ur5e_hande_mjx", "scene.xml")
pytestmark = pytest.mark.skipif(not REFERENCE or not os.path.exists(REF_XML),
                                reason="needs the upstream checkout named by MANIPULATOR_MUJOCO_REFERENCE")


@pytest.fixture(scope="module")
def mj():
    model = mujoco.MjModel.from_xml_path(REF_XML)
    model.opt.timestep = 0.05
    return model


def test_model_constants(mj, mc):
    assert (mj.nq, mj.nv, mj.nbody, mj.ngeom) == (mc.nq, mc.nv, mc.nbody, mc.ngeom)
    np.testing.assert_allclose(mj.body_mass, mc.body_mass, rtol=2e-3, atol=1e-6)          # mesh-inertia mode may differ
    np.testing.assert_allclose(mj.body_pos, mc.body_pos, atol=1e-9)
    np.testing.assert_allclose(mj.body_quat, mc.body_quat, atol=1e-9)
    np.testing.assert_allclose(mj.jnt_range[:6], mc.jnt_range[:6], atol=1e-9)
    np.testing.assert_allclose(mj.dof_armature[:6], 0.1)
    np.testing.assert_allclose(mj.dof_invweight0, mc.dof_invweight0, rtol=5e-3)
    np.testing.assert_allclose(mj.body_invweight0[:, 0], mc.body_invweight0[:, 0], rtol=5e-3, atol=1e-9)
    np.testing.assert_allclose(mj.stat.meaninertia, mc.meaninertia, rtol=5e-3)
    for i in range(10):
        assert mujoco.mj_name2id(mj, mujoco.mjtObj.mjOBJ_GEOM, f"robot_{i}") == mc.geom_id(f"robot_{i}")


def test_contact_slots_and_mask(mj, mc):
    from oracle.oracle import robot_slot_mask
    mx = mjx.put_model(mj)
    dx = jax.jit(mjx.forward)(mx, mjx.put_data(mj, mujoco.MjData(mj)))
    geom = np.asarray(dx.contact.geom)
    assert geom.shape[0] == mc.ncon
    ids = np.array([mc.geom_id(f"robot_{i}") for i in range(10)])
    mask = np.any(np.isin(geom, ids), axis=1)
    assert mask.sum() == robot_slot_mask(mc).sum() == 187
    # slot order: same pair sequence as the compiled pair list (geom1 <= geom2 by type)
    mine = np.repeat(mc.pair_geom, mc.pair_nslot, axis=0)
    np.testing.assert_array_equal(np.sort(geom, axis=1), np.sort(mine, axis=1))


def test_rollout_against_mjx(mj, mc, oracle64):
    from conftest import Q0, planner_inputs
    import jax.numpy as jnp
    T, B = 16, 16
    pr, z, xi, st, xif, td = planner_inputs(T, B)
    mx = mjx.put_model(mj)
    dx0 = jax.jit(mjx.forward)(mx, mjx.put_data(mj, mujoco.MjData(mj)))
    hande, tcp = mj.body(name="hande").id, mj.site(name="tcp").id
    ids = np.array([mc.geom_id(f"robot_{i}") for i in range(10)])
    mask = np.any(np.isin(np.asarray(dx0.contact.geom), ids), axis=1)

    def step(d, v):
        d = d.replace(qvel=d.qvel.at[:6].set(v))
        d = mjx.step(mx, d)
        return d, (d.qpos[:6], d.site_xpos[tcp], d.xquat[hande], d.contact.dist[mask])

    def rollout(tdot):
        d = dx0.replace(qpos=dx0.qpos.at[:6].set(jnp.asarray(Q0)), qvel=dx0.qvel.at[:6].set(jnp.zeros(6)))
        _, out = jax.lax.scan(step, d, tdot.reshape(6, T).T)
        return out

    theta, eef_pos, eef_rot, col = jax.vmap(rollout)(jnp.asarray(td, dtype=jnp.float32))
    oth, oep, oer, ocol = oracle64.rollout(td, Q0, np.zeros(6))
    np.testing.assert_allclose(np.asarray(theta).transpose(0, 2, 1).reshape(B, -1), oth, atol=5e-4)
    np.testing.assert_allclose(np.asarray(eef_pos), oep, atol=5e-4)
    np.testing.assert_allclose(np.abs(np.asarray(eef_rot)), np.abs(oer), atol=5e-4)
    # the far-field convention of capsule_convex (SURVEY C.9) shows up here first
    assert (np.abs(np.asarray(col) - ocol) > 1e-3).mean() < 1e-3


def test_jax_random_stream_restatement():
    """The sampler's key chain and draws against jax.random itself (mjx_planner.py:80,314-315,388): would pin
    `jax_prng` / `oracle/jax_random_ref.py` for the counter layout of the installed jax (default config)."""
    import jax.numpy as jnp
    from manipulator_mujoco_b200 import jax_prng
    from oracle import jax_random_ref as ref
    part = bool(jax.config.jax_threefry_partitionable)
    key = jax.random.PRNGKey(0)
    np.testing.assert_array_equal(np.asarray(jax.random.key_data(key)), jax_prng.PRNGKey(0))
    k1, _ = jax.random.split(key)
    np.testing.assert_array_equal(np.asarray(jax.random.key_data(k1)), jax_prng.split(jax_prng.PRNGKey(0), 2, part)[0])
    k2, _ = jax.random.split(k1)
    mean = jnp.zeros(66)
    cov = 10 * jnp.identity(66) + 0.003 * jnp.identity(66)
    xi = np.asarray(jax.random.multivariate_normal(k2, mean, cov, (64,)))
    mine = ref.multivariate_normal(jax_prng.split(jax_prng.split(jax_prng.PRNGKey(0), 2, part)[0], 2, part)[0],
                                   np.zeros(66), np.asarray(cov, dtype=np.float64), 64, part)
    np.testing.assert_allclose(xi, mine, rtol=0, atol=2e-5)
