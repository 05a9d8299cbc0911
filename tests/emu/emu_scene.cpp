// tests/emu/emu_scene.cpp -- CPU emulation of the rollout instantiations with scene / start records given per call
// (rollout_sample<NC, STATES, CONTACTS, SCENE = true>, behind cemk_rollout_cost_scene and cemk_step_states_scene) for the
// no-GPU tests (tests/test_emu_scene.py).
//
// Built like tests/emu/emu_contacts.cpp (-DCEMK_EMU, optionally -DCEMK_EMU_RACE for the race-checking emulation, see
// warp_dsl.h) into a library of its own.  Nothing in the package imports it; the product path is the CUDA build in
// csrc/cemk.cu.
#define CEMK_EMU 1
#include "../../manipulator_mujoco_b200/csrc/rollout_core.h"
#include <cstdlib>
#include <new>

extern "C" int emu_scene_sizeof_kmodel() { return (int)sizeof(KModel); }

// Race-checking build: write-write conflicts and lane blocks checked over all samples since the last read.
static long long g_race_waw = 0, g_race_blocks = 0;
extern "C" int emu_scene_race_enabled() {
#ifdef CEMK_EMU_RACE
  return 1;
#else
  return 0;
#endif
}
extern "C" void emu_scene_race_stats(long long* out2) {
  out2[0] = g_race_waw; out2[1] = g_race_blocks;
  g_race_waw = g_race_blocks = 0;
}

// One entry for both forms, as k_rollout<.., SCENE = true> runs them.  states = 0: a planner rollout (emu_rollout of
// emu.cpp) with q0 / v0 [6] shared, the cost to cost4 [B][4], theta [B][6T], qacc [B][T][12] and the start record `start`.
// states = 1: stepping per-environment state rows (emu_rollout_states_contacts of emu_contacts.cpp): q0 / v0 / warm are
// qpos [B][13] / qvel [B][12] / qacc_warmstart [B][12], the final state to qpos_out / qvel_out / warm_out, and the contact
// outputs when slot_map is given.  Sample s reads the scene record scene + s * scene_stride.  nc: shared-memory contact
// capacity of the emulated record (20 = the product instantiation, 48 = everything in the record).
extern "C" int emu_scene_rollout(const KModel* m, int states, int B, int T, const float* thetadot, const float* q0, const float* v0,
                                 const float* warm, const float* tpos, const float* trot, float w_pos, float w_rot, float w_col,
                                 float* theta, float* cost4, float* qacc_dbg, float* qpos_out, float* qvel_out, float* warm_out,
                                 int* flags, const int* slot_map, float* qfrc, int* ncon, int* con_slot, float* con_rec,
                                 const float* scene, int scene_stride, const float* start, int nc) {
#pragma omp parallel
  {
    Warp* W = new Warp();
    WarpSmemT<KM_NC_FAST>* S = new WarpSmemT<KM_NC_FAST>();
    WarpSmemT<KM_NC_BIG>* Sb = new WarpSmemT<KM_NC_BIG>();
    float* prevd = new float[2 * KM_NPASS * KW];
    float* ovf = new float[KM_NC_TOT * KM_OVF_STRIDE];
#pragma omp for schedule(dynamic, 4)
    for (int s = 0; s < B; ++s) {
      memset((void*)W, 0, sizeof(Warp));
      memset((void*)S, 0, sizeof(*S));
      memset((void*)Sb, 0, sizeof(*Sb));
      RolloutArgs A = {};
      A.T = T;
      A.live = true;
      A.thetadot = thetadot ? thetadot + (size_t)s * KM_NL * T : nullptr;
      A.theta = theta ? theta + (size_t)s * KM_NL * T : nullptr;
      A.qacc_dbg = qacc_dbg ? qacc_dbg + (size_t)s * T * KM_NV : nullptr;
      A.flags = flags ? flags + s : nullptr;
      A.prevd = prevd;
      A.ovf = ovf;
      if (states) {
        A.q0 = q0 + (size_t)s * KM_NQ; A.v0 = v0 + (size_t)s * KM_NV; A.warm0 = warm + (size_t)s * KM_NV;
        A.qpos_out = qpos_out + (size_t)s * KM_NQ; A.qvel_out = qvel_out + (size_t)s * KM_NV; A.warm_out = warm_out + (size_t)s * KM_NV;
        if (slot_map) {
          A.slot_map = slot_map;
          A.qfrc = qfrc + (size_t)s * KM_NV; A.ncon = ncon + s;
          A.con_slot = con_slot + (size_t)s * KM_NC_TOT; A.con_rec = con_rec + (size_t)s * KM_NC_TOT * KM_CON_REC;
        }
      } else {
        A.q0 = q0; A.v0 = v0; A.target_pos = tpos; A.target_rot = trot;
        A.w_pos = w_pos; A.w_rot = w_rot; A.w_col = w_col;
        A.cost4 = cost4 + (size_t)s * 4;
      }
      const float* sc = scene + (size_t)s * scene_stride;
#ifdef CEMK_EMU_RACE
      RaceState rs;                                   // this sample's record, scratch and outputs
      if (nc <= KM_NC_FAST) rs.add(S, sizeof(*S)); else rs.add(Sb, sizeof(*Sb));
      rs.add(prevd, sizeof(float) * 2 * KM_NPASS * KW);
      rs.add(ovf, sizeof(float) * KM_NC_TOT * KM_OVF_STRIDE);
      if (states && slot_map) {
        rs.add(A.qfrc, sizeof(float) * KM_NV);
        rs.add(A.con_slot, sizeof(int) * KM_NC_TOT);
        rs.add(A.con_rec, sizeof(float) * KM_NC_TOT * KM_CON_REC);
      }
      W->race = &rs;
      g_emu_race = &rs;
#endif
      if (!states) {
        if (nc <= KM_NC_FAST) rollout_sample<KM_NC_FAST, false, false, true>(*W, *m, *S, A, sc, start);
        else rollout_sample<KM_NC_BIG, false, false, true>(*W, *m, *Sb, A, sc, start);
      } else if (!slot_map) {
        if (nc <= KM_NC_FAST) rollout_sample<KM_NC_FAST, true, false, true>(*W, *m, *S, A, sc);
        else rollout_sample<KM_NC_BIG, true, false, true>(*W, *m, *Sb, A, sc);
      } else {
        if (nc <= KM_NC_FAST) rollout_sample<KM_NC_FAST, true, true, true>(*W, *m, *S, A, sc);
        else rollout_sample<KM_NC_BIG, true, true, true>(*W, *m, *Sb, A, sc);
      }
#ifdef CEMK_EMU_RACE
#pragma omp critical
      { g_race_waw += rs.waw; g_race_blocks += rs.blocks; }
      delete[] rs.snap; delete[] rs.pend; delete[] rs.owner;
#endif
    }
    delete W; delete S; delete Sb; delete[] prevd; delete[] ovf;
  }
  return 0;
}
