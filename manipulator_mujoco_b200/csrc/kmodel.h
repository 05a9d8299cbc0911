// kmodel.h -- flat, float32 model table consumed by the rollout kernel.
//
// The rollout kernel is specialised to the topology of the planner scene
// (reference sampling_based_planner/ur5e_hande_mjx/scene.xml, loaded at mjx_planner.py:100):
//   * one serial chain of NL hinge joints on a static base (bodies welded behind the last joint are
//     merged into the last link by the host),
//   * at most one free-floating box (target_0),
//   * capsule collision geoms on the chain, static planes / boxes in the world.
// manipulator_mujoco_b200/kmodel.py builds this struct from ModelConsts and refuses any model that
// does not fit.  Plain POD: shared by the CUDA build, the host C-ABI and the CPU emulation build
// used by the no-GPU tests.
#pragma once

#define KM_NL 6          // robot links == robot dofs
#define KM_NV 12         // robot dofs + free box dofs
#define KM_NQ 13
#define KM_MAXCAP 12
#define KM_MAXSBOX 8
#define KM_MAXRPAIR 160  // robot pair table entries = KM_MAXRPAIR / KW collider passes of KW lanes (see warp_dsl.h)
#define KM_MAXNEAR 96    // capsule-box pairs a model may have (capacity of the per-step near list)
#define KM_MAXBPAIR 8    // free-box vs static pairs

// robot pair types; a table entry packs (type + 1) | a << 4 | b << 8 | first cost slot << 16  (0 = no pair)
#define KP_NONE (-1)
#define KP_PLANE_CAP 0
#define KP_CAP_CAP 1
#define KP_CAP_BOX 2
#define KP_TYPE(x) (((x) & 15) - 1)
#define KP_A(x) (((x) >> 4) & 15)
#define KP_B(x) (((x) >> 8) & 15)
#define KP_SLOT(x) ((x) >> 16)
// free-box pair types
#define KB_PLANE_BOX 0
#define KB_BOX_BOX 1        // static box is geom1, free box geom2
#define KB_BOX_BOX_SWAP 2   // free box is geom1 (lower geom id), static box geom2

struct KModel {
  int nl, ncap, nsbox, has_box;
  int nrpair, nbpair, nslot_robot, ls_iterations;
  float dt, tolerance, ls_tolerance, meaninertia;
  float impratio, mu, pad0, pad1;
  float grav[4];
  float solref[2], solimp[5], pad2;
  float refpt[4];                       // reference point of all spatial vectors
  float base_pos[4], base_quat[4];      // static parent frame of link 0
  float l_pos[KM_NL][4], l_quat[KM_NL][4], l_axis[KM_NL][4], l_com[KM_NL][4];
  float l_inertia[KM_NL][8];            // xx yy zz xy xz yz (link frame, about com), mass, 0
  float l_armature[KM_NL], l_damping[KM_NL], l_lo[KM_NL], l_hi[KM_NL], l_invw[KM_NL], l_margin[KM_NL];
  int l_limited[KM_NL];
  int ncbpass, pad3;                    // leading passes of the pair table that hold the capsule-box pairs (see rp)
  float tcp_pos[4], hande_quat[4];      // relative to the last link frame
  int cap_link[KM_MAXCAP];
  float cap_pos[KM_MAXCAP][4], cap_axis[KM_MAXCAP][4];
  float cap_r[KM_MAXCAP], cap_hl[KM_MAXCAP], cap_invw[KM_MAXCAP];
  float plane_pos[4], plane_n[4];
  float sb_pos[KM_MAXSBOX][4], sb_mat[KM_MAXSBOX][12], sb_size[KM_MAXSBOX][4];   // sb_size[.][3] = 1: axis-aligned box, sb_mat[.][9..11] = its half sizes along the world axes
  float fb_size[4], fb_inertia[4];      // free box half sizes; principal inertia (body frame)
  float fb_mass, fb_damping, fb_invw, pad4;
  // robot pairs, pass-major: entry p*KW + lane.  Passes 0 .. ncbpass-1 hold the capsule-box pairs with a fixed shape:
  // pass p = box p (static boxes 0 .. nsbox-1, then the free box), lane l = capsule l, so a lane keeps its capsule in
  // registers and a pass reads one box; missing (excluded) pairs are empty entries.  Plane-capsule and
  // capsule-capsule pairs follow, grouped by type.
  int rp[KM_MAXRPAIR];
  int bp_type[KM_MAXBPAIR], bp_a[KM_MAXBPAIR];
  float qpos0[16], warm0[12], qvel0[12];   // snapshot every rollout starts from (mjx_planner.py:267)
};

// The two pose blocks a rollout may take per call instead of the table's (cemk_rollout_cost_scene, cemk_step_states_scene):
// a scene record is exactly sb_pos | sb_mat | sb_size (static box poses, unused rows zero), a start record exactly
// qpos0 | warm0 | qvel0.  The table's own blocks are the default records.
#define KM_SCENE_FLOATS (KM_MAXSBOX * (4 + 12 + 4))   // 160
#define KM_START_FLOATS (16 + 12 + 12)                // 40
