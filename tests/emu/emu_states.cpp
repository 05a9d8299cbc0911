// tests/emu/emu_states.cpp -- CPU emulation of the per-environment stepping instantiation of the rollout core
// (rollout_sample<NC, true>, behind cemk_step_states) for the no-GPU tests (tests/test_emu_step_states.py).
//
// Built like tests/emu/emu.cpp (-DCEMK_EMU, optionally -DCEMK_EMU_RACE for the race-checking emulation, see warp_dsl.h)
// into a library of its own.  Nothing in the package imports it; the product path is the CUDA build in csrc/cemk.cu.
#define CEMK_EMU 1
#include "../../manipulator_mujoco_b200/csrc/rollout_core.h"
#include <cstdlib>
#include <new>

extern "C" int emu_states_sizeof_kmodel() { return (int)sizeof(KModel); }

// Race-checking build: write-write conflicts and lane blocks checked over all samples since the last read.
static long long g_race_waw = 0, g_race_blocks = 0;
extern "C" int emu_states_race_enabled() {
#ifdef CEMK_EMU_RACE
  return 1;
#else
  return 0;
#endif
}
extern "C" void emu_states_race_stats(long long* out2) {
  out2[0] = g_race_waw; out2[1] = g_race_blocks;
  g_race_waw = g_race_blocks = 0;
}

// Every sample steps T times from its own qpos [13] / qvel [12] / warm [12] rows and writes its final state to the *_out
// rows (which may be the input rows); thetadot, theta, the dumps and flags may be null as in cemk_step_states.
extern "C" int emu_rollout_states(const KModel* m, int B, int T, const float* qpos, const float* qvel, const float* warm,
                                  const float* thetadot, float* qpos_out, float* qvel_out, float* warm_out, float* theta,
                                  float* eef_pos, float* eef_rot, float* collision, float* qacc_dbg, int* flags, int nc) {
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
      A.theta = theta ? theta + (size_t)s * KM_NL * T : nullptr;
      A.eef_pos = eef_pos ? eef_pos + (size_t)s * T * 3 : nullptr;
      A.eef_rot = eef_rot ? eef_rot + (size_t)s * T * 4 : nullptr;
      A.collision = collision ? collision + (size_t)s * T * m->nslot_robot : nullptr;
      A.qacc_dbg = qacc_dbg ? qacc_dbg + (size_t)s * T * KM_NV : nullptr;
      A.flags = flags ? flags + s : nullptr;
      A.prevd = prevd;
      A.ovf = ovf;
#ifdef CEMK_EMU_RACE
      RaceState rs;                                   // shared scratch of this sample: the record, the previous distances, the spill area
      if (nc <= KM_NC_FAST) rs.add(S, sizeof(*S)); else rs.add(Sb, sizeof(*Sb));
      rs.add(prevd, sizeof(float) * 2 * KM_NPASS * KW);
      rs.add(ovf, sizeof(float) * KM_NC_TOT * KM_OVF_STRIDE);
      W->race = &rs;
      g_emu_race = &rs;
#endif
      if (nc <= KM_NC_FAST) rollout_sample<KM_NC_FAST, true>(*W, *m, *S, A); else rollout_sample<KM_NC_BIG, true>(*W, *m, *Sb, A);
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
