"""Drop-in ``cem_planner`` for the UR5e + Hand-E scene, backed by libcemk.so (sm_100a CUDA).

Mirrors the public surface of the reference class (``sampling_based_planner/mjx_planner.py:17-406``):
same constructor keywords, same attribute names read by ``mpc_planner.py`` (``nvar``, ``model``,
``data``, ``tcp_id``, ``hande_id``) and the notebooks, the same per-iteration methods with the
same argument order and shapes, and ``compute_cem`` returning the same 9-tuple.  JAX arrays become
torch CUDA tensors; the small results of ``compute_cem`` come back as numpy arrays because the
caller feeds them straight to ``np.mean`` / ``np.round`` (``mpc_planner.py:178,185``).

There is no CPU path: constructing the planner without a CUDA device or without libcemk.so raises.

Reference quirks kept on purpose (SURVEY.md appendix C): elites are taken from the *unprojected*
samples (:357); the PRNG key never advances across ``compute_cem`` calls (:80,:388) so the same
standard-normal draws are reused every tick; the covariance restarts at 10*I every call (:386);
``theta`` is the post-step joint angle while ``eef_pos`` / ``eef_rot`` / ``collision`` are pre-step.
``jax.random`` is restated: ``key`` is raw threefry key data (``PRNGKey(0)`` = two zero words), the
``split`` chain runs on the host (``jax_prng``) and the normal draws of ``multivariate_normal`` come
from the device generator ``cemk_jax_normal`` (same counters, bit -> uniform -> erf_inv mapping as
jax 0.5.3), so identical seeds give the reference's samples up to float32 rounding of the Cholesky.

Other DOF counts (``num_dof`` 1..12): the per-iteration algebra (sampling, projection filter + Bernstein evaluation,
elite selection, mean / covariance, the constant matrices) runs on the GPU at that width (nvar = num_dof * (order + 1)
<= 192).  The model is still scene A's 6-DOF UR5e, so the rollout and everything built on it (``compute_rollout_batch``,
``cem_iter``, ``compute_cem``) raise ``NotImplementedError`` there.

Multi-GPU (extension, SURVEY.md section 8e): pass ``process_group``; ``num_batch`` is then the global
batch, each rank rolls out ``num_batch / world`` samples, keeps its local top-k and one NCCL
all-gather merges the elite lists so every rank computes the identical mean / covariance.
"""
from __future__ import annotations

import ctypes as C
import os
import warnings

import numpy as np
import torch

from . import _lib, jax_prng, parallel
from .bernstein import bernstein_coeff_ordern_new
from .kmodel import build_kmodel
from .mjcf import ModelConsts, exclude_body_pairs, host_kinematics, load_model, quat_mul, quat_normalize

_VP = C.c_void_p


def _ptr(t):
    return None if t is None else _VP(t.data_ptr())


class _Named:
    def __init__(self, **kw):
        self.__dict__.update(kw)


class _ModelView:
    """Stand-in for the ``mujoco.MjModel`` attributes the callers touch (mpc_planner.py:109-124,231)."""

    def __init__(self, mc: ModelConsts, timestep):
        self._mc = mc
        self.opt = _Named(timestep=timestep)
        self.nq, self.nv, self.nbody, self.ngeom = mc.nq, mc.nv, mc.nbody, mc.ngeom
        self._body_pos = mc.body_pos.copy()
        self._body_quat = mc.body_quat.copy()

    def body(self, name=None):
        i = self._mc.body_id(name)
        return _Named(id=i, name=name, pos=self._body_pos[i], quat=self._body_quat[i])

    def site(self, name=None):
        return _Named(id=self._mc.site_id(name), name=name)

    def geom(self, name=None):
        return _Named(id=self._mc.geom_id(name), name=name)


class _DataView:
    """Stand-in for ``mujoco.MjData``: qpos/qvel/qacc plus kinematics refreshed by ``forward()``."""

    def __init__(self, mc: ModelConsts):
        self._mc = mc
        self.qpos = mc.qpos0.copy()
        self.qvel = np.zeros(mc.nv)
        self.qacc = np.zeros(mc.nv)
        self.forward()

    def forward(self):
        xpos, xquat, xmat = host_kinematics(self._mc, self.qpos)
        self.xpos, self.xquat, self.xmat = xpos, xquat, xmat
        sb = self._mc.site_body
        self.site_xpos = np.array([xpos[b] + xmat[b] @ p for b, p in zip(sb, self._mc.site_pos)])


class cem_planner:

    def __init__(self, num_dof=None, num_batch=None, num_steps=None, timestep=None, maxiter_cem=None, num_elite=None,
                 w_pos=None, w_rot=None, w_col=None, maxiter_projection=None, *, model_path=None, device=None,
                 process_group=None, seed=0, contact_exclude=None, threefry_partitionable=True, bernstein_order=10):
        if isinstance(num_dof, bool) or not isinstance(num_dof, (int, np.integer)) or not 1 <= num_dof <= 12:
            raise ValueError(f"num_dof must be an integer in [1, 12], got {num_dof!r}")
        num_dof = int(num_dof)
        if not torch.cuda.is_available():
            raise RuntimeError("cem_planner needs a CUDA device (B200 / sm_100a); there is no CPU fallback")
        self._lib = _lib.load()
        self.num_dof = num_dof
        self.num_batch = num_batch
        self.t = timestep
        self.num = num_steps
        self.num_elite = num_elite
        self.cost_weights = {'w_pos': w_pos, 'w_rot': w_rot, 'w_col': w_col}
        self.maxiter_projection = maxiter_projection
        self.maxiter_cem = maxiter_cem

        # ---- distributed layout: samples are sharded contiguously by rank ----
        self.process_group = process_group
        if process_group is not None:
            import torch.distributed as dist
            self._dist = dist
            self.world = dist.get_world_size(process_group)
            self.rank = dist.get_rank(process_group)
        else:
            self._dist, self.world, self.rank = None, 1, 0
        if num_batch % self.world:
            raise ValueError("num_batch must be divisible by the number of ranks")
        self.num_batch_local = num_batch // self.world
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        dev = self.device

        # ---- basis and constraint matrices (mjx_planner.py:34-76) ----
        self.t_fin = self.num * self.t
        tot_time = np.linspace(0, self.t_fin, self.num)
        self.tot_time = tot_time
        tc = tot_time.reshape(self.num, 1)
        # the reference hard-codes order 10 (mjx_planner.py:40); `bernstein_order` is the order-n extension of SURVEY 8 f.4
        # order 3 has four coefficients per DOF for the five boundary conditions of mjx_planner.py:163-164: its KKT matrix is
        # singular (np.linalg.inv fails or returns per-DOF blocks of rounding noise)
        if not 4 <= int(bernstein_order) <= 15:
            raise ValueError("bernstein_order must be in [4, 15]")
        self.bernstein_order = int(bernstein_order)
        self.P, self.Pdot, self.Pddot = bernstein_coeff_ordern_new(self.bernstein_order, tc[0], tc[-1], tc)
        f32 = lambda a: torch.as_tensor(np.asarray(a), dtype=torch.float32, device=dev)
        self.P_jax, self.Pdot_jax, self.Pddot_jax = f32(self.P), f32(self.Pdot), f32(self.Pddot)
        self.nvar_single = self.P.shape[1]
        self.nvar = self.nvar_single * self.num_dof
        self.A_projection = torch.eye(self.nvar, device=dev)
        self.rho_ineq = 1.0
        self.rho_projection = 1.0
        A_v_ineq, A_v = self.get_A_v()
        A_a_ineq, A_a = self.get_A_a()
        A_p_ineq, A_p = self.get_A_p()
        A_eq = self.get_A_eq()
        self._np = dict(A_v_ineq=A_v_ineq, A_a_ineq=A_a_ineq, A_p_ineq=A_p_ineq)
        Q_inv = self.get_Q_inv(A_eq)
        A_theta, A_thetadot, A_thetaddot = self.get_A_traj()
        self.A_v_ineq, self.A_v = f32(A_v_ineq), f32(A_v)
        self.A_a_ineq, self.A_a = f32(A_a_ineq), f32(A_a)
        self.A_p_ineq, self.A_p = f32(A_p_ineq), f32(A_p)
        self.A_eq, self.Q_inv = f32(A_eq), f32(Q_inv)
        self.A_theta, self.A_thetadot, self.A_thetaddot = f32(A_theta), f32(A_thetadot), f32(A_thetaddot)

        # jax.random.PRNGKey(0) (:80) as raw threefry key data; `seed` is a keyword-only extension.
        # threefry_partitionable selects the counter layout of jax >= 0.5 (the reference pins jax 0.5.3) or the older one.
        self.key = jax_prng.PRNGKey(seed)
        self._partitionable = bool(threefry_partitionable)
        self.v_max = 0.8
        self.a_max = 1.8
        self.p_max = 180 * np.pi / 180
        self.l_1 = self.l_2 = self.l_3 = 1.0
        self.ellite_num = int(self.num_elite * self.num_batch)
        self.alpha_mean = 0.6
        self.alpha_cov = 0.6
        self.lamda = 10
        self.g = 10

        # ---- model (mjx_planner.py:100-121) ----
        self.model_path = model_path if model_path is not None else "<packaged ur5e_hande_mjx/scene.xml constants>"
        self._mc = load_model(model_path)
        if contact_exclude:                 # [(body1, body2), ...] == MJCF <contact><exclude/> entries
            self._mc = exclude_body_pairs(self._mc, contact_exclude)
        self.model = _ModelView(self._mc, self.t)
        self.data = _DataView(self._mc)
        km, info = build_kmodel(self._mc, self.t)
        self.mjx_model = km
        self.geom_ids = np.array([self._mc.geom_id(f'robot_{i}') for i in range(10)])
        mask = np.zeros(self._mc.ncon, dtype=bool)
        for (g1, g2), a, n in zip(self._mc.pair_geom, self._mc.pair_slotadr, self._mc.pair_nslot):
            if g1 in self.geom_ids or g2 in self.geom_ids:
                mask[a:a + n] = True
        self.mask = torch.as_tensor(mask, device=dev)
        self.nslot = int(mask.sum())
        self.hande_id = self.model.body(name="hande").id
        self.tcp_id = self.model.site(name="tcp").id

        h = _VP()
        _lib.check(self._lib.cemk_create(C.byref(km), C.sizeof(km), dev.index or 0, C.byref(h)), self._lib)
        self._h = h
        # mjx.forward at qpos0 (:107): its qacc becomes the first warm start of every rollout (the model is 6-DOF whatever
        # num_dof is, so this runs while the handle still has its default 6 DOF)
        self.mjx_data = self._initial_forward()
        _lib.check(self._lib.cemk_set_dof(self._h, self.num_dof), self._lib)
        _lib.check(self._lib.cemk_set_order(self._h, self.nvar_single), self._lib)
        self._set_horizon(Q_inv)

        # attributes the notebooks touch (mjx_planner.py:98,108): the vmapped outer product and the jitted single step
        self.vec_product = lambda diffs, d: self._t(d).reshape(-1, 1, 1) * torch.einsum("ki,kj->kij", self._t(diffs), self._t(diffs))
        self.jit_step = self._single_step

        self._z_cache = {}
        self._split_cache = {}
        # compute_cem restarts from self.key on every call (mjx_planner.py:388 never stores the advanced key), so the closed
        # loop asks for the same maxiter_cem blocks of normal draws every tick: keep them.  False = draw on every call
        # (what bench.py times).
        self.cache_normal_draws = True
        parallel.check_index_range(self.num_batch)
        self._ws = {}
        self._iter_out = None
        self._key_seen, self._key_tuple = None, None
        self._graph, self._graph_out, self._graph_key, self._eager_ticks = None, None, None, 0
        self.overflow_samples, self._warned_overflow = 0, False
        self.use_cuda_graph = os.environ.get("CEMK_CUDA_GRAPH", "1") != "0"
        if self.world > 1 and os.environ.get("CEMK_CUDA_GRAPH_MULTI", "1") == "0":
            self.use_cuda_graph = False
        self.print_info()

    # ------------------------------------------------------------------ constants (mjx_planner.py:142-172)
    def get_A_traj(self):
        I = np.identity(self.num_dof)
        return np.kron(I, self.P), np.kron(I, self.Pdot), np.kron(I, self.Pddot)

    def get_A_p(self):
        A_p = np.vstack((self.P, -self.P))
        return np.kron(np.identity(self.num_dof), A_p), A_p

    def get_A_v(self):
        A_v = np.vstack((self.Pdot, -self.Pdot))
        return np.kron(np.identity(self.num_dof), A_v), A_v

    def get_A_a(self):
        A_a = np.vstack((self.Pddot, -self.Pddot))
        return np.kron(np.identity(self.num_dof), A_a), A_a

    def get_A_eq(self):
        return np.kron(np.identity(self.num_dof),
                       np.vstack((self.P[0], self.Pdot[0], self.Pddot[0], self.Pdot[-1], self.Pddot[-1])))

    def get_Q_inv(self, A_eq):
        # the reference forms the cost block from float32 arrays and inverts the KKT matrix in float64
        r = lambda a: a.astype(np.float32).astype(np.float64)
        Av, Aa, Ap = r(self._np["A_v_ineq"]), r(self._np["A_a_ineq"]), r(self._np["A_p_ineq"])
        Q = (np.identity(self.nvar) + self.rho_ineq * Av.T @ Av + self.rho_ineq * Aa.T @ Aa
             + self.rho_ineq * Ap.T @ Ap).astype(np.float32).astype(np.float64)
        ne = A_eq.shape[0]
        return np.linalg.inv(np.vstack((np.hstack((Q, A_eq.T)), np.hstack((A_eq, np.zeros((ne, ne)))))))

    def _set_horizon(self, Q_inv):
        """Per-DOF blocks of Q_inv (block diagonal: every DOF solves the same (order + 1)-variable problem)."""
        n1, nd, nv = self.nvar_single, self.num_dof, self.nvar
        Kpp = Q_inv[:n1, :n1]
        Kpe = Q_inv[:n1, nv:nv + 5]
        # verify the structure the kernel relies on
        scale = np.abs(Q_inv).max()
        for d in range(nd):
            blk = Q_inv[d * n1:(d + 1) * n1]
            if (np.abs(blk[:, d * n1:(d + 1) * n1] - Kpp).max() > 1e-6 * scale
                    or np.abs(blk[:, nv + 5 * d:nv + 5 * d + 5] - Kpe).max() > 1e-6 * scale):
                raise RuntimeError("Q_inv is not block diagonal per DOF")
        off = Q_inv[:n1, n1:nv]
        if off.size and np.abs(off).max() > 1e-6 * scale:
            raise RuntimeError("Q_inv couples different DOFs")
        c32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
        G, Kpp, Kpe = c32(np.stack((self.Pdot, self.Pddot, self.P))), c32(Kpp), c32(Kpe)
        bnd = c32([self.v_max, self.a_max, self.p_max])
        hp = lambda a: a.ctypes.data_as(_VP)
        _lib.check(self._lib.cemk_set_horizon(self._h, self.num, hp(G), hp(Kpp), hp(Kpe), hp(bnd)), self._lib)

    def _initial_forward(self):
        """One forward at qpos0 with zero velocity: qacc -> KModel.warm0 (mjx_planner.py:107)."""
        dev = self.device
        z6 = torch.zeros(6, device=dev)
        q0 = torch.as_tensor(self._mc.qpos0[:6], dtype=torch.float32, device=dev)
        td = torch.zeros(1, 6, device=dev)
        theta = torch.empty(1, 6, device=dev)
        cost4 = torch.empty(1, 4, device=dev)
        qacc = torch.empty(1, 1, 12, device=dev)
        tp = torch.zeros(3, device=dev)
        tr = torch.tensor([1.0, 0, 0, 0], device=dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(self._lib.cemk_rollout_cost(self._h, 1, 1, _ptr(td), _ptr(q0), _ptr(z6), _ptr(tp), _ptr(tr), 0.0, 0.0, 0.0,
                                               _ptr(theta), _ptr(cost4), None, None, None, _ptr(qacc), None, _VP(st)), self._lib)
        warm = qacc[0, 0].cpu().numpy()
        for i in range(12):
            self.mjx_model.warm0[i] = float(warm[i])
        _lib.check(self._lib.cemk_set_model(self._h, C.byref(self.mjx_model), C.sizeof(self.mjx_model)), self._lib)
        return dict(qpos=self._mc.qpos0.copy(), qvel=np.zeros(12), qacc=warm.copy(), qacc_warmstart=warm.copy())

    def _single_step(self, model, data):
        """``jax.jit(mjx.step)(mjx_model, mjx_data)`` (mjx_planner.py:108,256) for one environment: ``data`` is a dict with
        qpos[13], qvel[12], qacc_warmstart[12] (``self.mjx_data`` has that form); returns the stepped dict plus qacc.
        Runs the rollout kernel with B = 1, T = 1 from that state (the free box included), like the closed-loop plant."""
        km = type(self.mjx_model)()
        C.memmove(C.byref(km), C.byref(self.mjx_model), C.sizeof(km))
        qpos, qvel = np.asarray(data["qpos"], dtype=np.float64), np.asarray(data["qvel"], dtype=np.float64)
        warm = np.asarray(data.get("qacc_warmstart", np.zeros(12)), dtype=np.float64)
        for i in range(13):
            km.qpos0[i] = qpos[i]
        for i in range(12):
            km.qvel0[i], km.warm0[i] = qvel[i], warm[i]
        dev = self.device
        h = _VP()
        _lib.check(self._lib.cemk_create(C.byref(km), C.sizeof(km), dev.index or 0, C.byref(h)), self._lib)
        try:
            td = self._t(qvel[:6]).reshape(1, 6)
            q0, v0 = self._t(qpos[:6]), self._t(qvel[:6])
            tp, tr = torch.zeros(3, device=dev), torch.tensor([1.0, 0, 0, 0], device=dev)
            theta, cost4, qacc = torch.empty(1, 6, device=dev), torch.empty(1, 4, device=dev), torch.empty(1, 1, 12, device=dev)
            _lib.check(self._lib.cemk_rollout_cost(h, 1, 1, _ptr(td), _ptr(q0), _ptr(v0), _ptr(tp), _ptr(tr), 0.0, 0.0, 0.0, _ptr(theta),
                                                   _ptr(cost4), None, None, None, _ptr(qacc), None, self._stream()), self._lib)
            a = qacc[0, 0].cpu().numpy().astype(np.float64)
        finally:
            self._lib.cemk_destroy(h)
        dt = float(self.t)
        v = qvel + dt * a
        q = qpos.copy()
        q[:9] += dt * v[:9]
        w = v[9:12]
        n = np.linalg.norm(w)
        if n > 0:
            ang = dt * n
            b = np.concatenate([[np.cos(ang / 2)], np.sin(ang / 2) * w / n])
            p = q[9:13]
            q[9:13] = quat_normalize(quat_mul(p, b))
        return dict(qpos=q, qvel=v, qacc=a, qacc_warmstart=a.copy())

    def print_info(self):
        if self.rank == 0:
            print(
                f'\n Default backend: cuda ({torch.cuda.get_device_name(self.device)})'
                f'\n Model path: {self.model_path}',
                f'\n Timestep: {self.t}',
                f'\n CEM Iter: {self.maxiter_cem}',
                f'\n Number of batches: {self.num_batch}',
                f'\n Number of steps per trajectory: {self.num}',
                f'\n Time per trajectory: {self.t_fin}',
            )

    def close(self):
        """Release the captured CUDA graph and the library handle.  With several GPUs call this before
        ``torch.distributed.destroy_process_group()``: a live graph holds captured NCCL kernels, and tearing the
        communicator down under it blocks."""
        if getattr(self, "_graph", None) is not None:
            torch.cuda.current_stream(self.device).synchronize()
            self._graph, self._graph_out, self._graph_key = None, None, None
        if getattr(self, "_h", None):
            self._lib.cemk_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    def _t(self, a, shape=None):
        t = torch.as_tensor(np.asarray(a) if not torch.is_tensor(a) else a, dtype=torch.float32, device=self.device)
        t = t.contiguous()
        return t if shape is None else t.reshape(shape)

    def _require_rollout_dof(self, what):
        if self.num_dof != 6:
            raise NotImplementedError(
                f"{what} needs the rollout, which models scene A's 6-DOF UR5e arm; this planner has num_dof={self.num_dof} "
                "and the dual-arm model is not built (the planner algebra runs at any num_dof in [1, 12])")

    def _stream(self):
        return _VP(torch.cuda.current_stream(self.device).cuda_stream)

    def _buf(self, name, shape, dtype=torch.float32):
        key = (name, tuple(shape), dtype)
        b = self._ws.get(key)
        if b is None:
            b = torch.empty(shape, dtype=dtype, device=self.device)
            self._ws[key] = b
        return b

    def _const(self, name, make):
        """A device constant built once (read-only afterwards; CUDA graphs keep pointing at it)."""
        key = ("const", name)
        b = self._ws.get(key)
        if b is None:
            b = make()
            self._ws[key] = b
        return b

    def _split0(self, key):
        """``jax.random.split(key)[0]``; memoised, the reference walks the same key chain every tick (:80, :388)."""
        k = jax_prng.as_key(key)
        ck = (int(k[0]), int(k[1]))
        out = self._split_cache.get(ck)
        if out is None:
            out = jax_prng.split(k, 2, self._partitionable)[0]
            self._split_cache[ck] = out
        return out

    def _normal(self, key):
        """jax.random.normal(key, (num_batch, nvar)) rows [rank*Bl, (rank+1)*Bl): the draws behind
        jax.random.multivariate_normal (:315), generated on the device by cemk_jax_normal.  A function of
        (key, global sample index) only, so results do not depend on the number of GPUs."""
        k = jax_prng.as_key(key)
        ck = (int(k[0]), int(k[1]))
        z = self._z_cache.get(ck) if self.cache_normal_draws else None
        if z is None:
            Bl, nv = self.num_batch_local, self.nvar
            z = torch.empty(Bl, nv, device=self.device, dtype=torch.float32)
            _lib.check(self._lib.cemk_jax_normal(self._h, ck[0], ck[1], 0 if self._partitionable else 1, self.num_batch * nv,
                                                 self.rank * Bl * nv, Bl * nv, _ptr(z), self._stream()), self._lib)
            if self.cache_normal_draws:
                self._z_cache[ck] = z
        return z

    # ------------------------------------------------------------------ per-iteration methods
    def compute_boundary_vec_single(self, state_term):
        st = self._t(state_term)
        return st.reshape(5, self.num_dof).T.reshape(self.num_dof * 5)

    def compute_boundary_vec_batch(self, state_term):
        st = self._t(state_term)
        return st.reshape(-1, 5, self.num_dof).transpose(1, 2).reshape(-1, self.num_dof * 5)

    def compute_xi_samples(self, key, xi_mean, xi_cov):
        """mjx_planner.py:313-316.  ``key``: raw threefry key data (2 x uint32, what jax.random.key_data
        gives) or an integer seed; returns (xi_samples, new key)."""
        key = self._split0(key)                                # key, subkey = split(key); sample with key
        z = self._normal(key)
        B = z.shape[0]
        xi = torch.empty(B, self.nvar, device=self.device)
        ws = self._buf("chol", (self.nvar * self.nvar,))
        mean, cov = self._t(xi_mean), self._t(xi_cov)
        _lib.check(self._lib.cemk_sample(self._h, B, _ptr(z), _ptr(mean), _ptr(cov), _ptr(ws), _ptr(xi), self._stream()),
                   self._lib)
        self._keep_s = (mean, cov)
        return xi, key

    def _project(self, xi_samples, state_term, want_thetadot, out_thetadot=None):
        xi = self._t(xi_samples)
        st = self._t(state_term)
        B = xi.shape[0]
        xi_f = torch.empty(B, self.nvar, device=self.device)
        thetadot = None
        if want_thetadot:
            thetadot = out_thetadot if out_thetadot is not None else torch.empty(B, self.num_dof * self.num, device=self.device)
        _lib.check(self._lib.cemk_project(self._h, B, int(self.maxiter_projection), _ptr(xi), _ptr(st), _ptr(xi_f),
                                          _ptr(thetadot), self._stream()), self._lib)
        return xi_f, thetadot

    def compute_projection_filter(self, xi_samples, state_term):
        """mjx_planner.py:234-249 -> primal_sol [B, nvar]."""
        return self._project(xi_samples, state_term, False)[0]

    def _rollout(self, thetadot, init_pos, init_vel, target_pos, target_rot, dumps, out_theta=None):
        td = self._t(thetadot)
        B, T = td.shape[0], self.num
        dev = self.device
        theta = out_theta if out_theta is not None else torch.empty(B, self.num_dof * T, device=dev)
        cost4 = torch.empty(B, 4, device=dev)
        eef_pos = torch.empty(B, T, 3, device=dev) if dumps else None
        eef_rot = torch.empty(B, T, 4, device=dev) if dumps else None
        collision = torch.empty(B, T, self.nslot, device=dev) if dumps else None
        flags = self._buf("flags", (B,), torch.int32)
        w = self.cost_weights
        # keep every converted argument referenced until the launch is enqueued (a temporary tensor
        # would hand its storage to the next allocation before the kernel reads it)
        q0, v0, tp, tr = self._t(init_pos), self._t(init_vel), self._t(target_pos), self._t(target_rot)
        _lib.check(self._lib.cemk_rollout_cost(
            self._h, B, T, _ptr(td), _ptr(q0), _ptr(v0), _ptr(tp), _ptr(tr), float(w['w_pos']), float(w['w_rot']),
            float(w['w_col']), _ptr(theta), _ptr(cost4), _ptr(eef_pos), _ptr(eef_rot), _ptr(collision), None, _ptr(flags),
            self._stream()), self._lib)
        self._keep = (td, q0, v0, tp, tr)
        return theta, cost4, eef_pos, eef_rot, collision

    def compute_rollout_batch(self, thetadot, init_pos, init_vel):
        """mjx_planner.py:123,266-274 -> theta [B,6T], eef_pos [B,T,3], eef_rot [B,T,4], collision [B,T,187]."""
        self._require_rollout_dof("compute_rollout_batch")
        tp = torch.zeros(3, device=self.device)
        tr = torch.tensor([1.0, 0, 0, 0], device=self.device)
        theta, _c, eef_pos, eef_rot, collision = self._rollout(thetadot, init_pos, init_vel, tp, tr, True)
        return theta, eef_pos, eef_rot, collision

    def step_batch(self, qpos, qvel, qacc_warmstart, thetadot=None):
        """``jax.vmap(jit_step, in_axes=(None, 0))``: N environments, each stepped from its own state in one launch
        (``cemk_step_states``); the planner's model snapshot is not used or changed.  qpos [N, 13], qvel [N, 12],
        qacc_warmstart [N, 12] (numpy or torch).  ``thetadot`` [N, 6T] (dof-major, the rollout's layout) chains T steps with
        qvel[:6] set to thetadot[:, t] before step t (mjx_planner.py:254); without it each environment takes one plain step
        with its own qvel.  Returns CUDA tensors: qpos, qvel, qacc (last step), qacc_warmstart (= that qacc), overflow [N]
        (bool: more simultaneous contacts than the kernel keeps, extra ones dropped) and, with thetadot, theta [N, 6T]."""
        self._require_rollout_dof("step_batch")
        qp, qv, wm = self._t(qpos), self._t(qvel), self._t(qacc_warmstart)
        if qp.dim() != 2 or qp.shape[1] != 13 or qp.shape[0] == 0:
            raise ValueError(f"qpos must be [N, 13] with N >= 1, got {tuple(qp.shape)}")
        N = qp.shape[0]
        if tuple(qv.shape) != (N, 12) or tuple(wm.shape) != (N, 12):
            raise ValueError(f"qvel and qacc_warmstart must be [{N}, 12], got {tuple(qv.shape)} and {tuple(wm.shape)}")
        td, T, theta = None, 1, None
        if thetadot is not None:
            td = self._t(thetadot)
            if td.dim() != 2 or td.shape[0] != N or td.shape[1] == 0 or td.shape[1] % 6:
                raise ValueError(f"thetadot must be [{N}, 6T] with T >= 1, got {tuple(td.shape)}")
            T = td.shape[1] // 6
            theta = torch.empty(N, 6 * T, device=self.device)
        dev = self.device
        if self._graph is not None and N > self.num_batch_local:
            # the library grows its rollout scratch to N samples and frees the old one, which the captured tick points at
            torch.cuda.current_stream(dev).synchronize()
            self._graph, self._graph_out, self._eager_ticks = None, None, 0
        qpos_out, qvel_out, warm_out = torch.empty(N, 13, device=dev), torch.empty(N, 12, device=dev), torch.empty(N, 12, device=dev)
        flags = torch.empty(N, dtype=torch.int32, device=dev)
        _lib.check(self._lib.cemk_step_states(self._h, N, T, _ptr(qp), _ptr(qv), _ptr(wm), _ptr(td), _ptr(qpos_out), _ptr(qvel_out),
                                              _ptr(warm_out), _ptr(theta), None, None, None, None, _ptr(flags), self._stream()), self._lib)
        self._keep_sb = (qp, qv, wm, td)
        out = dict(qpos=qpos_out, qvel=qvel_out, qacc=warm_out.clone(), qacc_warmstart=warm_out, overflow=(flags & 1).bool())
        if theta is not None:
            out["theta"] = theta
        return out

    def compute_cost_batch(self, thetadot, eef_pos, eef_rot, collision, target_pos, target_rot):
        """mjx_planner.py:124,277-303 (thetadot is unused there too) -> cost, cost_g, cost_r, cost_c [B]."""
        ep, er, col = self._t(eef_pos), self._t(eef_rot), self._t(collision)
        B, T, ns = col.shape
        tp, tr = self._t(target_pos).reshape(-1, 3), self._t(target_rot).reshape(-1, 4)
        if tp.shape[0] == 1:
            tp, tr = tp.expand(B, 3).contiguous(), tr.expand(B, 4).contiguous()
        cost4 = torch.empty(B, 4, device=self.device)
        w = self.cost_weights
        _lib.check(self._lib.cemk_cost_batch(self._h, B, T, ns, _ptr(ep), _ptr(er), _ptr(col), _ptr(tp), _ptr(tr),
                                             float(w['w_pos']), float(w['w_rot']), float(w['w_col']), _ptr(cost4),
                                             self._stream()), self._lib)
        return cost4[:, 0], cost4[:, 1], cost4[:, 2], cost4[:, 3]

    def _argsort_topk(self, cost, stride, n, k, xi, idx_base=0):
        np2 = 1 << max(0, (n - 1).bit_length())
        keys = self._buf("keys", (np2,), torch.int64)
        idx = torch.empty(n, dtype=torch.int32, device=self.device)
        xi_e = torch.empty(k, self.nvar, device=self.device)
        cost_e = torch.empty(k, device=self.device)
        _lib.check(self._lib.cemk_argsort_topk(self._h, n, _ptr(cost), stride, idx_base, _ptr(keys), _ptr(idx), k, _ptr(xi),
                                               _ptr(xi_e), _ptr(cost_e), self._stream()), self._lib)
        return xi_e, idx, cost_e

    def compute_ellite_samples(self, cost_batch, xi_filtered):
        """mjx_planner.py:306-310 -> xi_ellite [k,nvar], idx_ellite [B] (stable argsort), cost_ellite [k]."""
        cost = self._t(cost_batch)
        xi = self._t(xi_filtered)
        n = cost.shape[0]
        k = min(self.ellite_num, n)
        return self._argsort_topk(cost, 1, n, k, xi)

    def comp_prod(self, diffs, d):
        diffs = self._t(diffs)
        return d * torch.outer(diffs, diffs)

    def compute_mean_cov(self, cost_ellite, mean_control_prev, cov_control_prev, xi_ellite):
        """mjx_planner.py:326-335."""
        ce, xe = self._t(cost_ellite), self._t(xi_ellite)
        mean = torch.empty(self.nvar, device=self.device)
        cov = torch.empty(self.nvar, self.nvar, device=self.device)
        mp, cp = self._t(mean_control_prev), self._t(cov_control_prev)
        _lib.check(self._lib.cemk_mean_cov(self._h, ce.shape[0], _ptr(ce), _ptr(xe), _ptr(mp), _ptr(cp), float(self.lamda),
                                           float(self.alpha_mean), float(self.alpha_cov), _ptr(mean), _ptr(cov),
                                           self._stream()), self._lib)
        self._keep_m = (ce, xe, mp, cp)
        return mean, cov

    # ------------------------------------------------------------------ elite selection across GPUs
    def _select_elites(self, cost4, xi_samples):
        """Local top-k, then (multi-GPU) one all-gather + merge.  Returns xi_e [k,nvar], cost_e [k], gidx_e [k]|None."""
        Bl = self.num_batch_local
        k = self.ellite_num
        kl = min(k, Bl)
        base = self.rank * Bl
        if self.world == 1:
            xi_e, idx, cost_e = self._argsort_topk(cost4, 4, Bl, kl, xi_samples, idx_base=base)
            return xi_e, cost_e, idx[:kl]
        # Two library calls around one all-gather, persistent buffers only: tensors handed to the collective
        # must not churn through the caching allocator, and nothing here reads device memory from the host.
        nv = self.nvar
        np2l = 1 << max(0, (Bl - 1).bit_length())
        pack = self._buf("elite_pack", (kl, nv + 2))
        c4, xs = self._t(cost4), self._t(xi_samples)
        _lib.check(self._lib.cemk_topk_pack(self._h, Bl, _ptr(c4), 4, base, _ptr(self._buf("keys", (np2l,), torch.int64)), kl,
                                            _ptr(xs), _ptr(pack), self._stream()), self._lib)
        gathered = self._buf("elite_gathered", (self.world * kl, nv + 2))
        parallel.gather_elites(pack, self.world, self.process_group, out=gathered)
        xi_m = torch.empty(k, nv, device=self.device)
        cost_m = torch.empty(k, device=self.device)
        gidx_m = torch.empty(k, dtype=torch.int32, device=self.device)
        _lib.check(self._lib.cemk_merge_sorted_lists(self._h, self.world, kl, _ptr(gathered), k, _ptr(xi_m), _ptr(cost_m), _ptr(gidx_m),
                                                     self._stream()), self._lib)
        self._keep_e = (c4, xs)
        return xi_m, cost_m, gidx_m

    # ------------------------------------------------------------------ cem_iter / compute_cem (mjx_planner.py:337-406)
    def cem_iter(self, carry, _):
        self._require_rollout_dof("cem_iter")
        init_pos, init_vel, target_pos, target_rot, xi_mean, xi_cov, key, state_term = carry
        xi_mean_prev, xi_cov_prev = xi_mean, xi_cov
        xi_samples, key = self.compute_xi_samples(key, xi_mean, xi_cov)
        out_td, out_th = self._iter_out if self._iter_out is not None else (None, None)      # compute_cem: rows of its [maxiter, B, 6T] results
        xi_filtered, thetadot = self._project(xi_samples, state_term, True, out_thetadot=out_td)
        tp = self._t(target_pos).reshape(-1, 3)[0]
        tr = self._t(target_rot).reshape(-1, 4)[0]
        theta, cost4, _, _, _ = self._rollout(thetadot, init_pos, init_vel, tp, tr, False, out_theta=out_th)
        xi_ellite, cost_ellite, gidx = self._select_elites(cost4, xi_samples)
        xi_mean, xi_cov = self.compute_mean_cov(cost_ellite, xi_mean_prev, xi_cov_prev, xi_ellite)
        self._last_elite = (cost_ellite, gidx)
        self._last_cost4 = cost4
        carry = (init_pos, init_vel, target_pos, target_rot, xi_mean, xi_cov, key, state_term)
        return carry, (cost4[:, 0], cost4[:, 1], cost4[:, 2], cost4[:, 3], thetadot, theta)

    def _cem_device(self, pin, pout):
        """Everything a planning tick does on the device: H2D of the packed inputs, maxiter_cem
        iterations, best-sample extraction, D2H of the packed results (stream-ordered, no sync).
        pin = [xi_mean | q0 v0 a0 0 0 (the state row, :374-384) | target_pos | target_rot]."""
        dev = self.device
        Bl, T, nd, nv, m = self.num_batch_local, self.num, self.num_dof, self.nvar, self.maxiter_cem
        d_in = self._buf("d_in", (pin.numel(),))
        d_in.copy_(pin, non_blocking=True)
        xi_mean_d = d_in[:nv]
        q0, v0 = d_in[nv:nv + 6], d_in[nv + 6:nv + 12]
        tp, tr = d_in[nv + 30:nv + 33], d_in[nv + 33:nv + 37]
        state_term = d_in[nv:nv + 30].unsqueeze(0).expand(Bl, 30).contiguous()             # :374-384
        xi_cov = self._const("cov0", lambda: 10 * torch.eye(nv, device=dev))               # :386 (read-only)
        key = self._split0(self.key)                                                       # :388
        carry = (q0, v0, tp, tr, xi_mean_d, xi_cov, key, state_term)
        both = torch.empty(2, m, Bl, nd * T, device=dev)
        thetadot_all, theta_all = both[0], both[1]
        out_d = self._buf("tick_out", (pout.numel(),))
        best_row = self._buf("best_row", (2 * nd * T + 3,)) if self.world > 1 else None
        flags = self._buf("flags", (Bl,), torch.int32)
        for i in range(m):                                                                 # :390-392
            self._iter_out = (thetadot_all[i], theta_all[i])
            try:
                carry, out = self.cem_iter(carry, None)
            finally:
                self._iter_out = None
            cost_e, gidx = self._last_elite
            # min over the (global) batch, overflow count, and (last iteration, :395-402) the best sample = head of the
            # (merged) sorted list and the new mean, straight into the packed result
            _lib.check(self._lib.cemk_tick_record(self._h, i, m, int(i == m - 1), Bl, T, _ptr(cost_e), _ptr(gidx), self.rank * Bl, _ptr(flags),
                                                  _ptr(out[4]), _ptr(out[5]), _ptr(self._last_cost4), _ptr(carry[4]), _ptr(out_d),
                                                  _ptr(best_row), self._stream()), self._lib)
            self._keep_t = (cost_e, gidx, carry[4])
        if self.world > 1:
            # only the owning rank wrote its row; the others contributed exact zeros (their clamped row may hold
            # NaN / Inf of a diverged sample, which a 0/1 multiplication would leak into the sum)
            out_d[m:m + 2 * nd * T + 3].copy_(parallel.exchange_owned_row(best_row, None, self.process_group))
        pout.copy_(out_d, non_blocking=True)
        return thetadot_all, theta_all

    def compute_cem(self, xi_mean, init_pos=np.array([1.5, -1.8, 1.75, -1.25, -1.6, 0]), init_vel=np.zeros(6),
                    init_acc=np.zeros(6), target_pos=np.zeros(3), target_rot=np.zeros(4)):
        self._require_rollout_dof("compute_cem")
        dev = self.device
        Bl, T, nd, nv = self.num_batch_local, self.num, self.num_dof, self.nvar
        # one packed host->device copy for the per-tick inputs
        pin = self._ws.get("pin_in")
        if pin is None:
            pin = torch.zeros(nv + 37, dtype=torch.float32).pin_memory()
            self._ws["pin_in"] = pin
            self._ws["pin_in_np"] = pin.numpy()                       # a view: written in place every tick
        host = self._ws["pin_in_np"]
        host[:nv] = np.asarray(xi_mean.detach().cpu() if torch.is_tensor(xi_mean) else xi_mean, dtype=np.float32).reshape(-1)
        host[nv:nv + 6], host[nv + 6:nv + 12], host[nv + 12:nv + 18] = np.asarray(init_pos).reshape(-1), np.asarray(init_vel).reshape(-1), np.asarray(init_acc).reshape(-1)
        host[nv + 30:nv + 33], host[nv + 33:nv + 37] = np.asarray(target_pos).reshape(-1), np.asarray(target_rot).reshape(-1)
        m = self.maxiter_cem
        nout = m + 2 * nd * T + 3 + self.nvar + 1
        # The device side of a tick is a fixed sequence of launches on fixed buffers: after two eager
        # ticks (allocations, caches) it is captured once into a CUDA graph and replayed, which removes
        # the per-launch CPU cost that dominates small batches (closed-loop config: 3 x 9 launches).  With
        # several GPUs the NCCL all-gather / all-reduce are captured with it (every rank captures at the same
        # tick).  The graph bakes in everything that reaches a kernel as a scalar or a host pointer, so it is
        # keyed on those and dropped when one of them changes.
        w = self.cost_weights
        if self._key_seen is not self.key:                              # (the reference never reassigns its key)
            self._key_seen, self._key_tuple = self.key, tuple(int(x) for x in jax_prng.as_key(self.key))
        gkey = (m, int(self.maxiter_projection), float(w['w_pos']), float(w['w_rot']), float(w['w_col']),
                self._key_tuple, self._partitionable, T, Bl, int(self.ellite_num), nv)
        if self._graph is not None and gkey != self._graph_key:
            torch.cuda.current_stream(dev).synchronize()
            self._graph, self._graph_out, self._eager_ticks = None, None, 0
        pout = self._ws.get("pin_out")
        if pout is None or pout.numel() != nout:          # (no graph is alive here: nout is a function of the key)
            pout = torch.empty(nout, dtype=torch.float32).pin_memory()
            self._ws["pin_out"] = pout
        if self._graph is not None:
            self._graph.replay()
            thetadot_all, theta_all = self._graph_out
        elif self.use_cuda_graph and self._eager_ticks >= 2:
            torch.cuda.current_stream(dev).synchronize()
            g = torch.cuda.CUDAGraph()
            # thread_local: NCCL's watchdog thread polls events while this thread captures
            with torch.cuda.graph(g, capture_error_mode="thread_local" if self.world > 1 else "global"):
                out = self._cem_device(pin, pout)
            self._graph, self._graph_out, self._graph_key = g, out, gkey
            g.replay()
            thetadot_all, theta_all = out
        else:
            thetadot_all, theta_all = self._cem_device(pin, pout)
            self._eager_ticks += 1
        torch.cuda.current_stream(dev).synchronize()
        res = pout.numpy().copy()
        cost = res[:m]
        best_vels = res[m:m + nd * T].reshape(nd, T).T.copy()
        best_traj = res[m + nd * T:m + 2 * nd * T].reshape(nd, T).T.copy()
        o = m + 2 * nd * T
        best_cost_g, best_cost_r, best_cost_c = res[o], res[o + 1], res[o + 2]
        xi_mean_out = res[o + 3:o + 3 + nv].copy()
        # Samples whose simultaneous contacts exceeded the kernel's capacity (KM_NC_TOT = 48) were rolled out with
        # the extra contacts dropped -- MJX never truncates.  Count of such (sample, iteration) pairs on this rank:
        self.overflow_samples = int(res[o + 3 + nv])
        if self.overflow_samples and not self._warned_overflow:
            self._warned_overflow = True
            warnings.warn(f"cem_planner: {self.overflow_samples} rollout(s) of this tick exceeded the contact capacity of the "
                          "rollout kernel (48 simultaneous contacts); their extra contacts were dropped", RuntimeWarning)
        self.h2d_bytes = host.size * 4
        self.d2h_bytes = nout * 4
        if self._graph is not None:          # graph outputs are static buffers: hand out copies (one launch for both)
            both = thetadot_all._base.clone()
            thetadot_all, theta_all = both[0], both[1]
        return cost, best_cost_g, best_cost_r, best_cost_c, best_vels, best_traj, xi_mean_out, thetadot_all, theta_all
