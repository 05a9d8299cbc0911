// tests/emu/emu_contacts.cpp -- CPU emulation of the per-environment stepping instantiation with the contact outputs
// (rollout_sample<NC, true, true>, behind cemk_step_states_contacts) for the no-GPU tests (tests/test_emu_step_contacts.py).
//
// Built like tests/emu/emu_states.cpp (-DCEMK_EMU, optionally -DCEMK_EMU_RACE for the race-checking emulation, see
// warp_dsl.h) into a library of its own.  Nothing in the package imports it; the product path is the CUDA build in
// csrc/cemk.cu.
#define CEMK_EMU 1
#include "../../manipulator_mujoco_b200/csrc/rollout_core.h"
#include <cstdlib>
#include <new>

extern "C" int emu_contacts_sizeof_kmodel() { return (int)sizeof(KModel); }

// Race-checking build: write-write conflicts and lane blocks checked over all samples since the last read.
static long long g_race_waw = 0, g_race_blocks = 0;
extern "C" int emu_contacts_race_enabled() {
#ifdef CEMK_EMU_RACE
  return 1;
#else
  return 0;
#endif
}
extern "C" void emu_contacts_race_stats(long long* out2) {
  out2[0] = g_race_waw; out2[1] = g_race_blocks;
  g_race_waw = g_race_blocks = 0;
}

// emu_rollout_states of emu_states.cpp plus the contact outputs of cemk_step_states_contacts: slot_map [nslot_robot +
// 4 nbpair], qfrc [B][12], ncon [B], con_slot [B][48], con_rec [B][48][KM_CON_REC].  nc: shared-memory contact capacity
// of the emulated record (20 = the product instantiation, 48 = everything in the record).
extern "C" int emu_rollout_states_contacts(const KModel* m, int B, int T, const float* qpos, const float* qvel, const float* warm,
                                           const float* thetadot, float* qpos_out, float* qvel_out, float* warm_out, int* flags,
                                           const int* slot_map, float* qfrc, int* ncon, int* con_slot, float* con_rec, int nc) {
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
      A.q0 = qpos + (size_t)s * KM_NQ; A.v0 = qvel + (size_t)s * KM_NV; A.warm0 = warm + (size_t)s * KM_NV;
      A.qpos_out = qpos_out + (size_t)s * KM_NQ; A.qvel_out = qvel_out + (size_t)s * KM_NV; A.warm_out = warm_out + (size_t)s * KM_NV;
      A.flags = flags ? flags + s : nullptr;
      A.prevd = prevd;
      A.ovf = ovf;
      A.slot_map = slot_map;
      A.qfrc = qfrc + (size_t)s * KM_NV; A.ncon = ncon + s;
      A.con_slot = con_slot + (size_t)s * KM_NC_TOT; A.con_rec = con_rec + (size_t)s * KM_NC_TOT * KM_CON_REC;
#ifdef CEMK_EMU_RACE
      RaceState rs;                                   // this sample's record, scratch and contact outputs
      if (nc <= KM_NC_FAST) rs.add(S, sizeof(*S)); else rs.add(Sb, sizeof(*Sb));
      rs.add(prevd, sizeof(float) * 2 * KM_NPASS * KW);
      rs.add(ovf, sizeof(float) * KM_NC_TOT * KM_OVF_STRIDE);
      rs.add(A.qfrc, sizeof(float) * KM_NV);
      rs.add(A.con_slot, sizeof(int) * KM_NC_TOT);
      rs.add(A.con_rec, sizeof(float) * KM_NC_TOT * KM_CON_REC);
      W->race = &rs;
      g_emu_race = &rs;
#endif
      if (nc <= KM_NC_FAST) rollout_sample<KM_NC_FAST, true, true>(*W, *m, *S, A);
      else rollout_sample<KM_NC_BIG, true, true>(*W, *m, *Sb, A);
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
