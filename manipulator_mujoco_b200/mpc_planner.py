"""Headless closed-loop MPC driver -- the reference's ``run_cem_planner``
(``sampling_based_planner/mpc_planner.py:14-254``) without the MuJoCo viewer.

Same keyword arguments, same control flow (warm-up call, per-tick ``compute_cem``, mean of the
planned velocities ``best_vels[1:num_steps-2]`` applied to the plant, target switching on the
position / rotation thresholds, ``home`` target, CSV files with the reference's names) and the same
return dict.  Differences, all forced by the environment:

* the reference steps a C-MuJoCo plant (``mujoco.mj_step``, mpc_planner.py:180) inside a passive
  viewer loop that ends when the window is closed.  Neither exists here, so the plant is one
  env-step of this package's own CUDA stepper (``PlantSim``: the planner's rollout kernel with
  B = 1, T = 1, i.e. MJX semantics) and the loop ends after ``max_ticks`` ticks or, with
  ``stop_at_final_target``, when the last target is reached;
* ``show_viewer=True`` raises (the reference's own no-viewer branch is unimplemented,
  mpc_planner.py:234-236);
* the loop does not sleep to real time unless ``realtime=True``.
"""
from __future__ import annotations

import ctypes as C
import os
import time

import numpy as np
import torch

from . import _lib
from .kmodel import SCENE_FLOATS, scene_records
from .planner import cem_planner


def quaternion_distance(q1, q2):
    """quat_math.py:3-6 of the reference."""
    d = np.clip(np.abs(np.dot(q1, q2)), -1.0, 1.0)
    return 2 * np.arccos(d)


class PlantSim:
    """Single-environment plant: one MJX-semantics env-step per call on the GPU stepper.

    State (qpos[13], qvel[12], qacc_warmstart[12]) lives on the host in float64; each step uploads it
    as the kernel's snapshot, runs a 1-sample / 1-step rollout that returns qacc, and integrates with
    the same semi-implicit Euler as the kernel (B.8 of SURVEY.md)."""

    def __init__(self, cem: cem_planner):
        self.cem = cem
        self.mc = cem._mc
        self.dt = float(cem.t)
        self.qpos = self.mc.qpos0.copy()
        self.qvel = np.zeros(self.mc.nv)
        self.qacc = np.zeros(self.mc.nv)
        self.warm = np.asarray(cem.mjx_data["qacc_warmstart"], dtype=np.float64).copy()
        self._km = type(cem.mjx_model)()
        C.memmove(C.byref(self._km), C.byref(cem.mjx_model), C.sizeof(cem.mjx_model))
        self._h = C.c_void_p()
        dev = cem.device
        _lib.check(cem._lib.cemk_create(C.byref(self._km), C.sizeof(self._km), dev.index or 0, C.byref(self._h)), cem._lib)
        f = lambda n: torch.zeros(n, device=dev)
        self._td, self._q0, self._v0 = f(6).reshape(1, 6), f(6), f(6)
        self._tp, self._tr = f(3), torch.tensor([1.0, 0, 0, 0], device=dev)
        self._theta, self._cost4, self._qacc = f(6).reshape(1, 6), f(4).reshape(1, 4), f(12).reshape(1, 1, 12)
        self._moves = {}
        self.scene = scene_records(self.mc, {})[0]           # the plant's scene record (its table's static box block)

    def set_body_pose(self, name, pos, quat):
        """Move a static body of the plant (one of ``cem.scene_bodies``): rewrites the static box block of the plant's own
        table with the derivation of the model table (kmodel.scene_records); ``self.scene`` is the new scene record."""
        self._moves[name] = (np.asarray(pos, dtype=np.float64), np.asarray(quat, dtype=np.float64))
        self.scene = scene_records(self.mc, self._moves)[0]
        C.memmove(C.addressof(self._km) + type(self._km).sb_pos.offset, self.scene.ctypes.data, 4 * SCENE_FLOATS)

    def state(self):
        """The plant's state as ``compute_cem(state=...)`` takes it."""
        return dict(qpos=self.qpos.copy(), qvel=self.qvel.copy(), qacc_warmstart=self.warm.copy())

    def close(self):
        if self._h:
            self.cem._lib.cemk_destroy(self._h)
            self._h = None

    def step(self, thetadot_cmd):
        """data.qvel[:6] = thetadot; mj_step (mpc_planner.py:179-180)."""
        lib, km = self.cem._lib, self._km
        self.qvel[:6] = np.asarray(thetadot_cmd, dtype=np.float64)
        for i in range(13):
            km.qpos0[i] = self.qpos[i]
        for i in range(12):
            km.qvel0[i], km.warm0[i] = self.qvel[i], self.warm[i]
        _lib.check(lib.cemk_set_model(self._h, C.byref(km), C.sizeof(km)), lib)
        dev = self.cem.device
        self._td.copy_(torch.as_tensor(self.qvel[:6], dtype=torch.float32).reshape(1, 6))
        self._q0.copy_(torch.as_tensor(self.qpos[:6], dtype=torch.float32))
        self._v0.copy_(torch.as_tensor(self.qvel[:6], dtype=torch.float32))
        p = lambda t: C.c_void_p(t.data_ptr())
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(lib.cemk_rollout_cost(self._h, 1, 1, p(self._td), p(self._q0), p(self._v0), p(self._tp), p(self._tr), 0.0, 0.0, 0.0,
                                         p(self._theta), p(self._cost4), None, None, None, p(self._qacc), None, st), lib)
        self.qacc = self._qacc[0, 0].cpu().numpy().astype(np.float64)
        self.warm = self.qacc.copy()
        dt = self.dt
        self.qvel = self.qvel + dt * self.qacc
        self.qpos[:9] += dt * self.qvel[:9]
        w = self.qvel[9:12]
        n = np.linalg.norm(w)
        if n > 0:
            ang = dt * n
            qr = np.concatenate([[np.cos(ang / 2)], np.sin(ang / 2) * w / n])
            a, b = self.qpos[9:13], qr
            q = np.array([a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3], a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
                          a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1], a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0]])
            self.qpos[9:13] = q / np.linalg.norm(q)


def run_cem_planner(num_dof=None, num_batch=None, num_steps=None, maxiter_cem=None, maxiter_projection=None, w_pos=None, w_rot=None,
                    w_col=None, num_elite=None, timestep=None, initial_qpos=None, target_names=None, show_viewer=None,
                    cam_distance=None, show_contact_points=None, position_threshold=None, rotation_threshold=None, save_data=None,
                    data_dir=None, stop_at_final_target=None, *, max_ticks=200, realtime=False, verbose=True, device=None,
                    contact_exclude=None, plan_from_plant=False, body_moves=None):
    """``body_moves`` = {tick: {body name: (pos, quat)}} moves static bodies of the plant at the start of those ticks
    (``PlantSim.set_body_pose``).  ``plan_from_plant=True`` plans every tick in the plant's scene from its full state
    (``compute_cem(scene=..., state=...)``): the free box where the plant has it, moved obstacles where they are.  With the
    default the planner plans in the model's scene from its snapshot, as the reference does."""
    if show_viewer:
        raise NotImplementedError("no MuJoCo viewer in this build: call with show_viewer=False (headless loop, max_ticks)")
    if save_data:
        os.makedirs(data_dir, exist_ok=True)
    start_time = time.time()
    cem = cem_planner(num_dof=num_dof, num_batch=num_batch, num_steps=num_steps, maxiter_cem=maxiter_cem, w_pos=w_pos, w_rot=w_rot,
                      w_col=w_col, num_elite=num_elite, timestep=timestep, maxiter_projection=maxiter_projection, device=device,
                      contact_exclude=contact_exclude)
    if verbose:
        print(f"Initialized CEM Planner: {round(time.time() - start_time, 2)}s")
    model, data = cem.model, cem.data
    plant = PlantSim(cem)
    plant.qpos[:num_dof] = np.asarray(initial_qpos, dtype=np.float64)
    data.qpos[:] = plant.qpos
    data.forward()                                                       # mujoco.mj_forward (mpc_planner.py:114)
    xi_mean = np.zeros(cem.nvar)
    init_position = data.site_xpos[cem.tcp_id].copy()
    init_rotation = data.xquat[cem.hande_id].copy()
    target_pos = model.body(name=target_names[0]).pos
    target_rot = model.body(name=target_names[0]).quat
    start_time = time.time()
    _ = cem.compute_cem(xi_mean, data.qpos[:num_dof], data.qvel[:num_dof], data.qacc[:num_dof], target_pos, target_rot)
    if verbose:
        print(f"Compute CEM: {round(time.time() - start_time, 2)}s")

    thetadot = np.zeros(num_dof)
    cost_g_list, cost_list, cost_r_list, cost_c_list, thetadot_list, theta_list, tick_ms = [], [], [], [], [], [], []
    dist_list, switch_ticks, plant_states = [], [], []
    target_idx = 0
    current_target = target_names[target_idx]
    reached_final = False
    for _tick in range(max_ticks):
        start_time = time.time()
        for name, (pos, quat) in (body_moves or {}).get(_tick, {}).items():
            plant.set_body_pose(name, pos, quat)
        plant_kw = dict(scene=plant.scene, state=plant.state()) if plan_from_plant else {}
        if current_target != "home":
            target_pos = model.body(name=current_target).pos
            target_rot = model.body(name=current_target).quat
        else:
            target_pos, target_rot = init_position, init_rotation
        if current_target == "target_1" and "target_0" in target_names:      # mpc_planner.py:164-166
            model.body(name="target_0").pos[:] = data.site_xpos[cem.tcp_id]
            model.body(name="target_0").quat[:] = data.xquat[cem.hande_id]
        cost, best_cost_g, best_cost_r, best_cost_c, best_vels, best_traj, xi_mean, _, _ = cem.compute_cem(
            xi_mean, data.qpos[:num_dof], data.qvel[:num_dof], data.qacc[:num_dof], target_pos, target_rot, **plant_kw)
        plan_ms = (time.time() - start_time) * 1e3
        if not reached_final:
            thetadot = np.mean(best_vels[1:num_steps - 2], axis=0)           # mpc_planner.py:178
        plant.step(thetadot)
        plant_states.append(plant.state())
        data.qpos[:], data.qvel[:], data.qacc[:] = plant.qpos, plant.qvel, plant.qacc
        data.forward()
        current_cost_g = np.linalg.norm(data.site_xpos[cem.tcp_id] - target_pos)
        current_cost_r = quaternion_distance(data.xquat[cem.hande_id], target_rot)
        current_cost = np.round(cost, 2)
        tick_ms.append(plan_ms)
        dist_list.append(float(current_cost_g))
        if verbose:
            print(f'Step Time: {"%.0f" % ((time.time() - start_time) * 1000)}ms | Cost g: {"%.2f" % float(current_cost_g)}'
                  f' | Cost r: {"%.2f" % float(current_cost_r)} | Cost c: {"%.2f" % float(best_cost_c)} | Cost: {current_cost}')
            print(f'target: {current_target}')
        if current_cost_g < position_threshold and current_cost_r < rotation_threshold:
            switch_ticks.append((_tick, current_target))
            if target_idx == len(target_names) - 1:
                if stop_at_final_target:
                    if verbose:
                        print(f"Reached final target: {current_target}. Stopping motion.")
                    thetadot = np.zeros(num_dof)
                    reached_final = True
                else:
                    target_idx = 0
                    current_target = target_names[target_idx]
            else:
                target_idx += 1
                current_target = target_names[target_idx]
                if verbose:
                    print(f"Moving to next target: {current_target}")
            if current_target == "home" and "target_0" in target_names:     # mpc_planner.py:217-220
                model.body(name="target_0").pos[:] = data.site_xpos[cem.tcp_id].copy()
                model.body(name="target_0").quat[:] = data.xquat[cem.hande_id].copy()
        cost_g_list.append(float(best_cost_g))
        cost_r_list.append(float(best_cost_r))
        cost_c_list.append(float(best_cost_c))
        thetadot_list.append(np.array(thetadot))
        theta_list.append(data.qpos[:num_dof].copy())
        cost_list.append(current_cost[-1] if isinstance(current_cost, np.ndarray) else current_cost)
        if reached_final:
            break
        if realtime:
            rest = model.opt.timestep - (time.time() - start_time)
            if rest > 0:
                time.sleep(rest)
    plant.close()
    if save_data:
        np.savetxt(f'{data_dir}/costs.csv', cost_list, delimiter=",")
        np.savetxt(f'{data_dir}/thetadot.csv', thetadot_list, delimiter=",")
        np.savetxt(f'{data_dir}/theta.csv', theta_list, delimiter=",")
        np.savetxt(f'{data_dir}/cost_g.csv', cost_g_list, delimiter=",")
        np.savetxt(f'{data_dir}/cost_r.csv', cost_r_list, delimiter=",")
        np.savetxt(f'{data_dir}/cost_c.csv', cost_c_list, delimiter=",")
    return {'cost_g': cost_g_list, 'cost_r': cost_r_list, 'cost_c': cost_c_list, 'cost': cost_list, 'thetadot': thetadot_list,
            'theta': theta_list, 'tick_ms': tick_ms, 'final_target': current_target, 'reached_final': reached_final,
            'dist': dist_list, 'switch_ticks': switch_ticks, 'cem': cem, 'plant_states': plant_states, 'plant_scene': plant.scene,
            'last': dict(xi_mean=xi_mean, qpos=data.qpos.copy(), qvel=data.qvel.copy(), qacc=data.qacc.copy(),
                         target_pos=np.array(target_pos), target_rot=np.array(target_rot))}
