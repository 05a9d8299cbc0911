// rollout_core.h -- one lane group (KW = 16 lanes: two samples per warp) rolls one CEM sample through the
// whole horizon.
//
// Replaces, for the planner scene, the reference's `vmap(scan(mjx.step))` + `vmap(compute_cost_single)`
// (reference sampling_based_planner/mjx_planner.py:251-303): forward kinematics, joint-space
// inertia, bias forces, primitive-geom narrow phase, MJX's soft-constraint Newton step with its
// bracketed line search, semi-implicit Euler, and the per-sample cost accumulated on the fly so the
// [B,T,187] distance tensor is never materialised.
//
// Formulation notes (all mathematically equivalent to the MJX algorithm restated in
// oracle/mjstep.c; only rounding differs):
//   * spatial vectors are [rot; lin] in world axes about the fixed point m.refpt (MJX uses the
//     subtree COM of the kinematic tree root; any fixed point gives the same joint-space result);
//   * gravity is dropped from the robot's recursive Newton-Euler pass because every robot body has
//     gravcomp = 1, so `qfrc_gravcomp - qfrc_bias(gravity)` cancels identically;
//   * the free box has its COM at the body origin and a principal-axis inertia, so its mass matrix
//     is constant and diagonal and its bias is  [-m g ; w x I w];
//   * only rows of active constraints (dist < 0, limit violated) are built: MJX multiplies the
//     Jacobian of every inactive row by zero, which leaves H, grad and the line search untouched;
//   * capsule-box evaluates MJX's `_capsule_convex` only inside its near zone (see capsule_box): outside it
//     both slots are the +1 sentinel by construction (has_support gate), which six min/max decide.
//
// Written against warp_dsl.h so that tests/emu can single-step it on the CPU.
#pragma once
#include "kmodel.h"
#include "warp_dsl.h"

#define KM_NC_FAST 20                     // active-contact capacity of the fast kernel (shared-memory budget per sample)
#define KM_NPASS (KM_MAXRPAIR / KW)         // collider passes over the robot pair table
#define KM_NC_TOT 48                      // contacts a sample can have in total: the ones beyond the shared-memory capacity
                                          // spill to a per-sample global (L2) area
#define KM_OVF_STRIDE 80                  // floats per spilled contact: geo 16, J 36, dots 2x3, rows 4x4
#define KM_NC_BIG 48                      // shared-memory capacity of the debug instantiation (everything in shared memory)
#define MJ_MINVAL 1e-15f
#define MJ_MINIMP 0.0001f
#define MJ_MAXIMP 0.9999f

struct LaneRegs {
  float cost_c;               // this lane's share of cost_c
  int nact, off;              // active contacts this lane will emit, and where
  int actmask;                // bit (2*pass + slot)
  int farprev;                // bit p: the previous step's distances of this lane's capsule-box pair of pass p were the (+1, +1) sentinel
  int tri;                    // (i, j), 4 bits each, of the 6x6 lower-triangle entries lane and lane + KW (8 bits per entry; 0xff = none)
  float acc[9];               // line-search partial sums (compile-time indices only)
  float h[KM_NV];             // row `lane` of the Newton Hessian / its Cholesky factor (compile-time indices only)
#ifdef CEMK_EMU
  float hrow[KM_NV];          // emulation build: chol_solve_rows' working copy (a plain local array on the GPU)
#endif
  float td;                   // next step's commanded joint velocity (lanes < 6), prefetched one step ahead
  float f0, f1, f2;
};

// Per-sample scratch in shared memory.  Unions reuse space between phases that never overlap: the
// spatial-dynamics arrays (P2-P5) vs the constraint rows (C1-S5), the capsule end points (P2-N2) vs the
// Newton Hessian (S3-S4), and the free-box contact staging (N1-N2) vs the contact Jacobians (C2-S5).
// With KW = 16 a CTA of 14 warps holds 28 of these next to the model table (227 KB per SM).
template <int NC>
struct WarpSmemT {
  static constexpr int NROW = KM_NL + 4 * NC;
  float qpos[16], qvel[12], warm[12];
  float lpos[KM_NL][4], lquat[KM_NL][4], lmat[KM_NL][12];
  float cdof[KM_NL][8];
  float bmat[12];
  float Mr[KM_NL][KM_NL];             // robot block of the joint-space inertia (box block is constant, diagonal)
  union {
    struct { float capA[KM_MAXCAP][4], capB[KM_MAXCAP][4]; };
    float H[KM_NV][KM_NV];
  };
  float fs[12], as[12], qacc[12], Ma[12], grad[12], search[12];
  int ncon, nrow, nlim, flags;
  union {
    struct { float cinert[KM_NL][12], crb[KM_NL][12], cvel[KM_NL][8], cdofdot[KM_NL][8], cfrc[KM_NL][8]; };
    struct { float rD[NROW], rAref[NROW], rJaref[NROW], rJv[NROW]; };   // rJv doubles as the smooth-start J.a - aref in S1
    struct {                            // N1 only: the near capsule-box pairs of this step (pair table entry | prefetched << 14 | was-far << 15)
      unsigned short nlist[KM_MAXNEAR]; //          and, per pair table entry, their previous distances fetched ahead by the owner lane
      float nprev[(KM_MAXSBOX + 1) * KW][2];
    };
  };
  float cgeo[NC][16];                 // pos3 n3 t1 3 t2 3 dist invw link1 link2
  union {
    float cJ[NC][36];                 // Jn[12] Jt1[12] Jt2[12] (tangents pre-multiplied by mu)
    struct {                          // free-box pair candidates (pos3, dist) + scratch of the cooperative box-box
      float bstage[KM_MAXBPAIR][4][4], bnrm[KM_MAXBPAIR][4];
      union {
        struct { float bbR[12], bbc[4], bbsz[2][4], bbrf[4][4], bben[4][4], bbpoly[2][8][4], bbpref[8][4]; };
        struct {                                            // near pass: box-frame geometry of the pairs in their edge stage (by list slot),
          float estage[KW][16], eres[KW][8];                // the result of the edge item each lane evaluated in this round,
          unsigned short eidx[KW * 12];                     // and the edge items of the group: list slot << 4 | edge
        };
      };
    };
  };
  float cd[2][NC][3];                 // per contact: Jn.v, mu*Jt1.v, mu*Jt2.v for up to two vectors v
  int limdof[KM_NL];
  float limsign[KM_NL];
  float* ovf;                         // spill area of this sample for contacts NC .. KM_NC_TOT-1: [KM_NC_TOT - NC][KM_OVF_STRIDE]
  float* ovf_pad;                     // (keeps the record a multiple of 16 bytes)

  // Per-contact / per-row storage: shared memory for the first NC contacts, the spill area beyond.  Samples
  // with more than NC simultaneous contacts are rare (deep-collision trajectories); they run in the same
  // kernel at the price of L2 accesses for the extra contacts instead of a serial re-run afterwards.
  // SP = false: the caller knows nothing is spilled -- plain shared-memory addressing (an address that may
  // point to either space would turn every access into a generic load).
  template <bool SP> KMEM float* geo(int c) const { return (!SP || c < NC) ? const_cast<float*>(cgeo[c]) : ovf + (c - NC) * KM_OVF_STRIDE; }
  template <bool SP> KMEM float* jac(int c) const { return (!SP || c < NC) ? const_cast<float*>(cJ[c]) : ovf + (c - NC) * KM_OVF_STRIDE + 16; }
  template <bool SP> KMEM float* dots(int set, int c) const {
    return (!SP || c < NC) ? const_cast<float*>(cd[set][c]) : ovf + (c - NC) * KM_OVF_STRIDE + 52 + 3 * set;
  }
  template <bool SP> KMEM float& row(const float* arr, int off, int r, int nl) const {
    const int rc = r - nl;              // rows nl + 4 c + q belong to contact c; limit rows (rc < 0) are always in shared memory
    return (!SP || rc < 4 * NC) ? const_cast<float*>(arr)[r] : ovf[((rc >> 2) - NC) * KM_OVF_STRIDE + off + (rc & 3)];
  }
  template <bool SP> KMEM float& D(int r, int nl) const { return row<SP>(rD, 58, r, nl); }
  template <bool SP> KMEM float& Aref(int r, int nl) const { return row<SP>(rAref, 62, r, nl); }
  template <bool SP> KMEM float& Jaref(int r, int nl) const { return row<SP>(rJaref, 66, r, nl); }
  template <bool SP> KMEM float& Jv(int r, int nl) const { return row<SP>(rJv, 70, r, nl); }
};

typedef WarpCtx<LaneRegs> Warp;

// the entries (i, j), j <= i, of a 6x6 lower triangle a lane owns: e = lane (and lane + 16 when KW = 16); 8 bits per entry
KFN int tri_entries(int lane) {
  int tri = 0;
  for (int q = 0; q < 32 / KW; ++q) {
    int e = lane + KW * q, i = 0, j = e;
    if (e < KM_NL * (KM_NL + 1) / 2) { while (j > i) { j -= i + 1; ++i; } } else { i = 15; j = 15; }
    tri |= (i | (j << 4)) << (8 * q);
  }
  return tri;
}
// A lane-group context of its own for an out-of-line (cold) routine.  Rare paths are real functions so that they do not
// sit inside the step loop, whose address span decides how well the instruction fetch of the lockstep warps works; a
// routine taking the caller's Warp by reference would force that struct (the per-lane state of the whole kernel) out of
// registers, so cold routines rebuild the few fields they need and exchange everything else through the sample's record.
KFN void cold_warp(Warp& W, int bar, int nthr) {
#ifdef CEMK_EMU
  std::memset((void*)&W, 0, sizeof(Warp));
  W.race = g_emu_race;
  for (int l = 0; l < KW; ++l) W.regs[l].tri = tri_entries(l);
  (void)bar; (void)nthr;
#else
  W.lane = threadIdx.x & (KW - 1);
  W.shift = (threadIdx.x & 31) & ~(KW - 1);
  W.mask = KW_FULL << W.shift;
  W.bar = bar; W.nthr = nthr;
  W.regs.tri = tri_entries(W.lane);
#ifdef CEMK_PHASE_TIMING
  W.phase = 0; W.t0 = clock64(); W.stepflag = 0; W.nflag = 0;
  for (int i = 0; i < 24; ++i) { W.ph[i] = 0; W.phs[i] = 0; W.phc[i] = 0; }
  for (int i = 0; i < 24; ++i) W.ev[i] = 0;
#endif
#endif
}

// ------------------------------------------------------------------------------------------ vec3
KFN float dot3(const float* a, const float* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
KFN void cross3(float* r, const float* a, const float* b) {
  float x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  r[0] = x; r[1] = y; r[2] = z;
}
KFN void sub3(float* r, const float* a, const float* b) { r[0] = a[0] - b[0]; r[1] = a[1] - b[1]; r[2] = a[2] - b[2]; }
KFN void add3(float* r, const float* a, const float* b) { r[0] = a[0] + b[0]; r[1] = a[1] + b[1]; r[2] = a[2] + b[2]; }
KFN void madd3(float* r, const float* a, const float* b, float s) { r[0] = a[0] + s * b[0]; r[1] = a[1] + s * b[1]; r[2] = a[2] + s * b[2]; }
KFN void copy3(float* r, const float* a) { r[0] = a[0]; r[1] = a[1]; r[2] = a[2]; }
KFN float normalize3(float* a) {
  float n = sqrtf(dot3(a, a));
  if (n > 0.f) { float i = 1.f / n; a[0] *= i; a[1] *= i; a[2] *= i; } else { a[0] = a[1] = a[2] = 0.f; }
  return n;
}
KFN void mat_vec(float* r, const float* m, const float* v) {      // row-major 3x3
  float x = m[0] * v[0] + m[1] * v[1] + m[2] * v[2], y = m[3] * v[0] + m[4] * v[1] + m[5] * v[2], z = m[6] * v[0] + m[7] * v[1] + m[8] * v[2];
  r[0] = x; r[1] = y; r[2] = z;
}
KFN void matT_vec(float* r, const float* m, const float* v) {
  float x = m[0] * v[0] + m[3] * v[1] + m[6] * v[2], y = m[1] * v[0] + m[4] * v[1] + m[7] * v[2], z = m[2] * v[0] + m[5] * v[1] + m[8] * v[2];
  r[0] = x; r[1] = y; r[2] = z;
}
KFN void quat_mul(float* r, const float* a, const float* b) {
  float w = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3];
  float x = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2];
  float y = a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1];
  float z = a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0];
  r[0] = w; r[1] = x; r[2] = y; r[3] = z;
}
KFN void quat_to_mat(float* m, const float* q) {
  float w = q[0], x = q[1], y = q[2], z = q[3];
  m[0] = w * w + x * x - y * y - z * z; m[1] = 2.f * (x * y - w * z);         m[2] = 2.f * (x * z + w * y);
  m[3] = 2.f * (x * y + w * z);         m[4] = w * w - x * x + y * y - z * z; m[5] = 2.f * (y * z - w * x);
  m[6] = 2.f * (x * z - w * y);         m[7] = 2.f * (y * z + w * x);         m[8] = w * w - x * x - y * y + z * z;
}
// sin/cos for |x| up to a few hundred: Cody-Waite reduction to [-pi/4, pi/4] + minimax polynomials
// (max error 7e-8 absolute for |x| <= 8, as good as sinf/cosf).  Replaces sincosf, whose slow path drags a large local-memory
// Payne-Hanek routine into the kernel.
KFN void k_sincos(float x, float* sn, float* cs) {
  const float k = rintf(x * 0.636619772367581343f);
  float r = fmaf(k, -1.5707963705062866f, x);          // pi/2 split in three float32 pieces
  r = fmaf(k, 4.371138828673793e-08f, r);
  r = fmaf(k, 1.7763568394002505e-15f, r);
  const float r2 = r * r;
  float sp = fmaf(r2, 2.724990382407328e-06f, -0.00019840086439758365f);
  sp = fmaf(sp, r2, 0.008333331873528407f);
  sp = fmaf(sp, r2, -0.16666666663842697f);
  sp = fmaf(sp * r2, r, r);
  float cp = fmaf(r2, -2.1011874848372744e-08f, 2.452856854478212e-05f);
  cp = fmaf(cp, r2, -0.0013888048639039594f);
  cp = fmaf(cp, r2, 0.041666660194519124f);
  cp = fmaf(cp, r2, -0.5f);
  cp = fmaf(cp, r2, 1.f);
  const int q = (int)k;
  const float s0 = (q & 1) ? cp : sp, c0 = (q & 1) ? sp : cp;
  *sn = (q & 2) ? -s0 : s0;
  *cs = ((q + 1) & 2) ? -c0 : c0;
}
// MJX math.make_frame: tangents for a unit normal (rows t1, t2)
KFN void make_tangents(const float* n, float* t1, float* t2) {
  float b[3] = {0.f, 0.f, 0.f};
  if (n[1] > -0.5f && n[1] < 0.5f) b[1] = 1.f; else b[2] = 1.f;
  float s = dot3(n, b);
  madd3(b, b, n, -s);
  normalize3(b);
  copy3(t1, b);
  cross3(t2, n, b);
}
// spatial algebra (BD.2, BD.4)
KFN void mul_inert(float* r, const float* i, const float* v) {
  r[0] = i[0] * v[0] + i[3] * v[1] + i[4] * v[2] - i[8] * v[4] + i[7] * v[5];
  r[1] = i[3] * v[0] + i[1] * v[1] + i[5] * v[2] + i[8] * v[3] - i[6] * v[5];
  r[2] = i[4] * v[0] + i[5] * v[1] + i[2] * v[2] - i[7] * v[3] + i[6] * v[4];
  r[3] = i[8] * v[1] - i[7] * v[2] + i[9] * v[3];
  r[4] = i[6] * v[2] - i[8] * v[0] + i[9] * v[4];
  r[5] = i[7] * v[0] - i[6] * v[1] + i[9] * v[5];
}
KFN float dot6(const float* a, const float* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3] + a[4] * b[4] + a[5] * b[5]; }
KFN void cross_motion(float* r, const float* v, const float* s) {
  float a[3], b[3], c[3];
  cross3(a, v, s); cross3(b, v, s + 3); cross3(c, v + 3, s);
  r[0] = a[0]; r[1] = a[1]; r[2] = a[2]; r[3] = b[0] + c[0]; r[4] = b[1] + c[1]; r[5] = b[2] + c[2];
}
KFN void cross_force(float* r, const float* v, const float* f) {
  float a[3], b[3], c[3];
  cross3(a, v, f); cross3(b, v + 3, f + 3); cross3(c, v, f + 3);
  r[0] = a[0] + b[0]; r[1] = a[1] + b[1]; r[2] = a[2] + b[2]; r[3] = c[0]; r[4] = c[1]; r[5] = c[2];
}

// ------------------------------------------------------------------------------------------ colliders
// Code-size note: the first build inlined every collider into four unrolled passes (670 KB of SASS)
// and spent 80 % of its issue slots waiting on instruction fetch (profiles/r1a).  Colliders are now
// real functions (KNOINLINE) called from rolled loops.

// MJX math.closest_segment_point_and_dist
KFN float closest_segment_point(float* res, const float* a, const float* b, const float* pt) {
  float ab[3], ap[3], d[3];
  sub3(ab, b, a); sub3(ap, pt, a);
  float t = dot3(ap, ab) / (dot3(ab, ab) + 1e-6f);
  t = fminf(fmaxf(t, 0.f), 1.f);
  madd3(res, a, ab, t);
  sub3(d, pt, res);
  return dot3(d, d);
}
// MJX math.closest_segment_to_segment_points; res = besta(3), bestb(3)
struct SegPair { float a[3], b[3]; };
KNOINLINE SegPair closest_seg_seg(float a0x, float a0y, float a0z, float a1x, float a1y, float a1z,
                                  float b0x, float b0y, float b0z, float b1x, float b1y, float b1z) {
  const float a0[3] = {a0x, a0y, a0z}, a1[3] = {a1x, a1y, a1z}, b0[3] = {b0x, b0y, b0z}, b1[3] = {b1x, b1y, b1z};
  float da[3], db[3], amid[3], bmid[3], tr[3];
  SegPair r;
  sub3(da, a1, a0); sub3(db, b1, b0);
  float ha = 0.5f * normalize3(da), hb = 0.5f * normalize3(db);
  madd3(amid, a0, da, ha); madd3(bmid, b0, db, hb);
  sub3(tr, amid, bmid);
  float dd = dot3(da, db), dat = dot3(da, tr), dbt = dot3(db, tr);
  float ta = (-dat + dd * dbt) / (1.f - dd * dd + 1e-6f);
  float tb = dbt + ta * dd;
  ta = fminf(fmaxf(ta, -ha), ha);
  tb = fminf(fmaxf(tb, -hb), hb);
  madd3(r.a, amid, da, ta); madd3(r.b, bmid, db, tb);
  float na[3], nb[3];
  float d1 = closest_segment_point(na, a0, a1, r.b);
  float d2 = closest_segment_point(nb, b0, b1, r.a);
  if (d1 < d2) copy3(r.a, na); else copy3(r.b, nb);
  return r;
}
KFN SegPair closest_seg_seg_v(const float* a0, const float* a1, const float* b0, const float* b1) {
  return closest_seg_seg(a0[0], a0[1], a0[2], a1[0], a1[1], a1[2], b0[0], b0[1], b0[2], b1[0], b1[1], b1[2]);
}

struct Contact2 { float dist[2], pos[2][3], nrm[2][3]; };
struct Dist2 { float d0, d1; };

// plane (geom1) vs capsule (geom2); B = centre + axis*hl is slot 0 (MJX plane_capsule offset order)
template <bool FULL>
KFN void plane_capsule(const float* ppos, const float* pn, const float* A, const float* B, float r, Contact2& c) {
  float t[3];
  sub3(t, B, ppos); c.dist[0] = dot3(t, pn) - r;
  sub3(t, A, ppos); c.dist[1] = dot3(t, pn) - r;
  if (FULL) {
    madd3(c.pos[0], B, pn, -(r + 0.5f * c.dist[0]));
    madd3(c.pos[1], A, pn, -(r + 0.5f * c.dist[1]));
    copy3(c.nrm[0], pn); copy3(c.nrm[1], pn);
  }
}
// capsule_capsule -> sphere_sphere on the closest segment points
template <bool FULL>
KFN void capsule_capsule(const float* a0, const float* a1, float r1, const float* b0, const float* b1, float r2, Contact2& c) {
  SegPair sp = closest_seg_seg_v(a0, a1, b0, b1);
  float n[3];
  sub3(n, sp.b, sp.a);
  float dn = normalize3(n);
  if (dn == 0.f) { n[0] = 1.f; n[1] = 0.f; n[2] = 0.f; }
  c.dist[0] = dn - (r1 + r2);
  c.dist[1] = 1.f;
  if (FULL) { madd3(c.pos[0], sp.a, n, r1 + 0.5f * c.dist[0]); copy3(c.nrm[0], n); }
}
// capsule (geom1) vs box (geom2): MJX collision_convex._capsule_convex for a box, restated in oracle/mjstep.c
// (capsule_box, mode 1).  Both slots are the "no contact" sentinel dist = +1 unless
//   * every face plane has an end point of the radius-inflated segment behind it (has_support) and the
//     segment clips against the side planes of the best face (then: face distances of the clipped points), or
//   * one of the 12 box edges is a shallow contact (closer than r, capsule point in front of both faces
//     adjacent to the edge), which replaces slot 0.
// Far field: if some box axis separates the segment's bounding interval from the box by >= r, has_support
// fails and no edge can be within r, so the pair costs one change of frame and six min/max (capbox_far).
// Otherwise (near path, = has_support): face part in registers; the edge stage is an out-of-line call taken only
// when the segment sticks out of the box on two axes.
KFN void capbox_local(const float* A, const float* B, const float* bpos, const float* bmat, float* a, float* b) {
  float t[3];
  sub3(t, A, bpos); matT_vec(a, bmat, t);
  sub3(t, B, bpos); matT_vec(b, bmat, t);
}
KFN bool capbox_far(const float* a, const float* b, float r, const float* s) {
  const float s0 = fmaxf(fminf(a[0], b[0]), -fmaxf(a[0], b[0])) - s[0];
  const float s1 = fmaxf(fminf(a[1], b[1]), -fmaxf(a[1], b[1])) - s[1];
  const float s2 = fmaxf(fminf(a[2], b[2]), -fmaxf(a[2], b[2])) - s[2];
  return !(fmaxf(fmaxf(s0, s1), s2) < r);
}
struct CapBoxOut { float dist[2], pos[2][3], nrm[2][3]; };     // box coordinates
// Shallow edge contact of the near path (rare: only when the segment's bounding box sticks out of the box on two
// axes).  Edge e = 4k + 2iu + iw runs along axis k at (u, w) = (+-s_u, +-s_w).  An edge can only win with a
// positive penetration, which needs a point of the segment in front of both faces adjacent to the edge and closer
// than r to it; the interval tests are necessary for that, so edges failing them skip the segment-segment routine
// without changing the result.  On a hit (pen > 0) the caller replaces slot 0 by the edge contact.  n = outward normal of the
// best face, minface = min(-dist[0], -dist[1]) of the face part.
struct CapBoxEdge { float pen, pos[3], nrm[3]; };            // pen <= 0: no edge contact
KNOINLINE CapBoxEdge capbox_edges(float ax, float ay, float az, float bx, float by, float bz, float r, float sx, float sy, float sz,
                                  float nx, float ny, float nz, float minface) {
  const float bsize[3] = {sx, sy, sz}, n[3] = {nx, ny, nz};
  float bpen = -1.f, beax[3] = {0.f, 0.f, 0.f}, bec[3] = {0.f, 0.f, 0.f}, bcc[3] = {0.f, 0.f, 0.f};
  bool bdeg = false;
  const float lo[3] = {fminf(ax, bx), fminf(ay, by), fminf(az, bz)}, hi[3] = {fmaxf(ax, bx), fmaxf(ay, by), fmaxf(az, bz)};
  // MJX math.closest_segment_to_segment_points(edge, capsule segment) with the edge-independent half hoisted out of the
  // loop and the edge half specialised to an axis-aligned edge (unit direction e_k, half length s_k, mid point (cu, cw, 0)):
  // the same formulas, a third of the instructions of the general routine, no call
  const float A0[3] = {ax, ay, az};
  float abb[3] = {bx - ax, by - ay, bz - az}, dbv[3] = {bx - ax, by - ay, bz - az}, bmid[3];
  const float den_abb = dot3(abb, abb) + 1e-6f;
  const float hb = 0.5f * normalize3(dbv);
  madd3(bmid, A0, dbv, hb);
  // axis k unrolled (compile-time component indices keep every array in registers), the four edges of an axis rolled
#pragma unroll
  for (int k = 0; k < 3; ++k)
#pragma unroll 1
  for (int e4 = 0; e4 < 4; ++e4) {
    const int u = (k + 1) % 3, w = (k + 2) % 3;
    const float eu = (e4 & 2) ? 1.f : -1.f, ew = (e4 & 1) ? 1.f : -1.f;
    const float cu = eu * bsize[u], cw = ew * bsize[w];
    // furthest the segment reaches in front of the two faces, measured from the edge (must be > 0), and its
    // nearest approach (must be < r)
    const float fu = eu > 0.f ? hi[u] - cu : cu - lo[u], fw = ew > 0.f ? hi[w] - cw : cw - lo[w];
    const float gu = eu > 0.f ? lo[u] - cu : cu - hi[u], gw = ew > 0.f ? lo[w] - cw : cw - hi[w];
    if (!(fu > 0.f && fw > 0.f && gu < r && gw < r && lo[k] < bsize[k] + r && hi[k] > -bsize[k] - r)) continue;
    SegPair sp;
    {
      const float sk = bsize[k];
      float tr[3];
      tr[k] = -bmid[k]; tr[u] = cu - bmid[u]; tr[w] = cw - bmid[w];
      const float dd = dbv[k], dat = tr[k], dbt = dot3(dbv, tr);
      float ta = (-dat + dd * dbt) / (1.f - dd * dd + 1e-6f);
      float tb = dbt + ta * dd;
      ta = fminf(fmaxf(ta, -sk), sk);
      tb = fminf(fmaxf(tb, -hb), hb);
      sp.a[k] = ta; sp.a[u] = cu; sp.a[w] = cw;
      madd3(sp.b, bmid, dbv, tb);
      // closest point of the edge to sp.b, of the capsule segment to sp.a (math.closest_segment_point_and_dist)
      float na[3], nb[3], dv[3], ap[3];
      float t1 = ((sp.b[k] + sk) * (2.f * sk)) / (4.f * sk * sk + 1e-6f);
      t1 = fminf(fmaxf(t1, 0.f), 1.f);
      na[k] = -sk + 2.f * sk * t1; na[u] = cu; na[w] = cw;
      sub3(dv, sp.b, na);
      const float d1 = dot3(dv, dv);
      sub3(ap, sp.a, A0);
      float t2 = dot3(ap, abb) / den_abb;
      t2 = fminf(fmaxf(t2, 0.f), 1.f);
      madd3(nb, A0, abb, t2);
      sub3(dv, sp.a, nb);
      const float d2 = dot3(dv, dv);
      if (d1 < d2) copy3(sp.a, na); else copy3(sp.b, nb);
    }
    float dir[3];
    sub3(dir, sp.a, sp.b);
    const bool deg = dot3(dir, dir) < 1e-6f;
    const float ed = normalize3(dir);
    const bool front = (eu * dir[u] < 0.f) && (ew * dir[w] < 0.f);
    const float epen = (!deg && front) ? r - ed : -1.f;
    if (epen > bpen) { bpen = epen; bdeg = deg; copy3(beax, dir); copy3(bec, sp.a); copy3(bcc, sp.b); }
  }
  const bool parallel = fabsf(dot3(beax, n)) > 0.99f && !bdeg;
  const bool has_edge = bpen > 0.f && (minface > 0.f ? bpen < minface : true) && !parallel;
  CapBoxEdge out;
  out.pen = has_edge ? bpen : 0.f;
#pragma unroll
  for (int q = 0; q < 3; ++q) { out.pos[q] = 0.5f * (bec[q] + bcc[q] + beax[q] * r); out.nrm[q] = beax[q]; }
  return out;
}
// Near path, in box coordinates; the caller has established has_support (= !capbox_far).  Face part in registers
// (no dynamic indexing); FULL also produces contact positions / normals.
// Returns the number of box axes on which the segment's bounding interval sticks out of the box (the edge stage can only
// matter when that is >= 2).  EDGES = false leaves the edge stage to the caller (the near pass deals the candidate edges of its
// pairs over lanes, see capbox_edge_mask) and also returns the outward normal of the best face in `nface`.
template <bool FULL, bool EDGES = true>
KFN int capsule_box_near(const float* a, const float* b, float r, const float* bsize, CapBoxOut& o, float* nface = nullptr) {
  // best face: first argmax over (+x,-x,+y,-y,+z,-z) of min over end points of the signed face distance
  float bests = fminf(a[0], b[0]) - bsize[0]; int bk = 0; float sg = 1.f;
  { float s = -fmaxf(a[0], b[0]) - bsize[0]; if (s > bests) { bests = s; sg = -1.f; } }
  { float s = fminf(a[1], b[1]) - bsize[1]; if (s > bests) { bests = s; bk = 1; sg = 1.f; } }
  { float s = -fmaxf(a[1], b[1]) - bsize[1]; if (s > bests) { bests = s; bk = 1; sg = -1.f; } }
  { float s = fminf(a[2], b[2]) - bsize[2]; if (s > bests) { bests = s; bk = 2; sg = 1.f; } }
  { float s = -fmaxf(a[2], b[2]) - bsize[2]; if (s > bests) { bests = s; bk = 2; sg = -1.f; } }
  // cyclic permutation into (k, u, w) coordinates without dynamic indexing
  float ak, au, aw, bk_, bu, bw, sk, su, sw;
  if (bk == 0)      { ak = a[0]; au = a[1]; aw = a[2]; bk_ = b[0]; bu = b[1]; bw = b[2]; sk = bsize[0]; su = bsize[1]; sw = bsize[2]; }
  else if (bk == 1) { ak = a[1]; au = a[2]; aw = a[0]; bk_ = b[1]; bu = b[2]; bw = b[0]; sk = bsize[1]; su = bsize[2]; sw = bsize[0]; }
  else              { ak = a[2]; au = a[0]; aw = a[1]; bk_ = b[2]; bu = b[0]; bw = b[1]; sk = bsize[2]; su = bsize[0]; sw = bsize[1]; }
  // clip the segment (parameter 0..1 from a to b) against the four side planes: closed form of MJX
  // _clip_edge_to_planes for a rectangular face
  float t0 = 0.f, t1 = 1.f; bool both = false;
  {
    const float Lu = 2.f * sw, Lw = 2.f * su;      // length of the edge each side plane is built on
#define CEMK_CLIP(pa, pb, s, tau, L) { \
      float na_ = ((tau) * (pa) - (s)) * (L), nb_ = ((tau) * (pb) - (s)) * (L); \
      bool fa = na_ > 1e-6f, fb = nb_ > 1e-6f; \
      float den = (tau) * ((pb) - (pa)) * (L); \
      float tt = (-na_) / (den + (den == 0.f ? 1e-6f : 0.f)); \
      tt = fminf(fmaxf(tt, 0.f), 1.f); \
      if (fa) t0 = fmaxf(t0, tt); \
      if (fb) t1 = fminf(t1, tt); \
      both = both || (fa && fb); }
    CEMK_CLIP(au, bu, su, -1.f, Lu)
    CEMK_CLIP(aw, bw, sw, -1.f, Lw)
    CEMK_CLIP(au, bu, su, 1.f, Lu)
    CEMK_CLIP(aw, bw, sw, 1.f, Lw)
#undef CEMK_CLIP
  }
  bool mask = !both;
  if (!mask) { t0 = 0.f; t1 = 1.f; }
  {
    const float dk = bk_ - ak, du = bu - au, dw = bw - aw;
    if ((t1 - t0) * (dk * dk + du * du + dw * dw) < 0.f) mask = false;
  }
  const float h0 = sg * (ak + t0 * (bk_ - ak)) - r - sk, h1 = sg * (ak + t1 * (bk_ - ak)) - r - sk;
  o.dist[0] = mask ? h0 : 1.f;
  o.dist[1] = mask ? h1 : 1.f;
  const float nx = bk == 0 ? sg : 0.f, ny = bk == 1 ? sg : 0.f, nz = bk == 2 ? sg : 0.f;
  // an edge needs the segment in front of two faces of different axes
  const int nout = ((fmaxf(a[0], b[0]) > bsize[0] || fminf(a[0], b[0]) < -bsize[0]) ? 1 : 0) +
                   ((fmaxf(a[1], b[1]) > bsize[1] || fminf(a[1], b[1]) < -bsize[1]) ? 1 : 0) +
                   ((fmaxf(a[2], b[2]) > bsize[2] || fminf(a[2], b[2]) < -bsize[2]) ? 1 : 0);
  if (FULL || nout >= 2) {
    // contact points / normals in (k,u,w) coordinates, rotated back to box axes
    const float l0[3] = {sg * (sk + 0.5f * h0), au + t0 * (bu - au), aw + t0 * (bw - aw)};
    const float l1[3] = {sg * (sk + 0.5f * h1), au + t1 * (bu - au), aw + t1 * (bw - aw)};
    if (bk == 0)      { o.pos[0][0] = l0[0]; o.pos[0][1] = l0[1]; o.pos[0][2] = l0[2]; o.pos[1][0] = l1[0]; o.pos[1][1] = l1[1]; o.pos[1][2] = l1[2]; }
    else if (bk == 1) { o.pos[0][1] = l0[0]; o.pos[0][2] = l0[1]; o.pos[0][0] = l0[2]; o.pos[1][1] = l1[0]; o.pos[1][2] = l1[1]; o.pos[1][0] = l1[2]; }
    else              { o.pos[0][2] = l0[0]; o.pos[0][0] = l0[1]; o.pos[0][1] = l0[2]; o.pos[1][2] = l1[0]; o.pos[1][0] = l1[1]; o.pos[1][1] = l1[2]; }
    o.nrm[0][0] = o.nrm[1][0] = -nx; o.nrm[0][1] = o.nrm[1][1] = -ny; o.nrm[0][2] = o.nrm[1][2] = -nz;
    if (EDGES && nout >= 2) {
      const CapBoxEdge e = capbox_edges(a[0], a[1], a[2], b[0], b[1], b[2], r, bsize[0], bsize[1], bsize[2], nx, ny, nz, fminf(-o.dist[0], -o.dist[1]));
      if (e.pen > 0.f) { o.dist[0] = -e.pen; copy3(o.pos[0], e.pos); copy3(o.nrm[0], e.nrm); }
    }
  }
  if (nface) { nface[0] = nx; nface[1] = ny; nface[2] = nz; }
  return nout;
}
// One of the 12 box edges against the capsule segment: the body of capbox_edges' loop for edge e = 4 k + 2 iu + iw, written in
// the edge's own (k, u, w) coordinates with component selects instead of indices (e is a lane number here, and a dynamic index
// would put the vectors in local memory).  epen = r - distance if the edge qualifies, -1 otherwise; pa / pb = closest points
// on the edge / on the segment, dir = normalised pa - pb, all in box coordinates.  TEST = false: the caller knows the edge passes the
// interval test (capbox_edge_mask), which is then not evaluated again.
struct EdgeEval { float epen, deg, dir[3], pa[3], pb[3]; };
KFN float pick3(const float* v, int k) { return k == 0 ? v[0] : (k == 1 ? v[1] : v[2]); }
KFN void unpick3(float* out, int k, int u, float vk, float vu, float vw) {
  out[0] = k == 0 ? vk : (u == 0 ? vu : vw); out[1] = k == 1 ? vk : (u == 1 ? vu : vw); out[2] = k == 2 ? vk : (u == 2 ? vu : vw);
}
template <bool TEST = true>
KFN EdgeEval capbox_edge_lane(int e, const float* a, const float* b, float r, const float* bsize) {
  EdgeEval out;
  out.epen = -1.f; out.deg = 0.f;
  out.dir[0] = out.dir[1] = out.dir[2] = 0.f; out.pa[0] = out.pa[1] = out.pa[2] = 0.f; out.pb[0] = out.pb[1] = out.pb[2] = 0.f;
  const int k = e >> 2, u = k == 2 ? 0 : k + 1, w = k == 0 ? 2 : k - 1;
  const float eu = (e & 2) ? 1.f : -1.f, ew = (e & 1) ? 1.f : -1.f;
  const float ak = pick3(a, k), au = pick3(a, u), aw = pick3(a, w), bk = pick3(b, k), bu = pick3(b, u), bw = pick3(b, w);
  const float sk = pick3(bsize, k), su = pick3(bsize, u), sw = pick3(bsize, w);
  const float lou = fminf(au, bu), hiu = fmaxf(au, bu), low = fminf(aw, bw), hiw = fmaxf(aw, bw), lok = fminf(ak, bk), hik = fmaxf(ak, bk);
  const float cu = eu * su, cw = ew * sw;
  const float fu = eu > 0.f ? hiu - cu : cu - lou, fw = ew > 0.f ? hiw - cw : cw - low;
  const float gu = eu > 0.f ? lou - cu : cu - hiu, gw = ew > 0.f ? low - cw : cw - hiw;
  if (TEST && !(fu > 0.f && fw > 0.f && gu < r && gw < r && lok < sk + r && hik > -sk - r)) return out;
  // closest points of the edge and the segment (same formulas as capbox_edges), vectors as (k, u, w) triples
  const float abk = bk - ak, abu = bu - au, abw = bw - aw;
  const float den = abk * abk + abu * abu + abw * abw + 1e-6f;
  float dv[3] = {abk, abu, abw};
  const float hb = 0.5f * normalize3(dv);
  const float mk = ak + dv[0] * hb, mu = au + dv[1] * hb, mw = aw + dv[2] * hb;
  const float trk = -mk, tru = cu - mu, trw = cw - mw;
  const float dd = dv[0], dat = trk, dbt = dv[0] * trk + dv[1] * tru + dv[2] * trw;
  float ta = (-dat + dd * dbt) / (1.f - dd * dd + 1e-6f);
  float tb = dbt + ta * dd;
  ta = fminf(fmaxf(ta, -sk), sk);
  tb = fminf(fmaxf(tb, -hb), hb);
  float pa[3] = {ta, cu, cw}, pb[3] = {mk + dv[0] * tb, mu + dv[1] * tb, mw + dv[2] * tb};
  float t1 = ((pb[0] + sk) * (2.f * sk)) / (4.f * sk * sk + 1e-6f);
  t1 = fminf(fmaxf(t1, 0.f), 1.f);
  const float na[3] = {-sk + 2.f * sk * t1, cu, cw};
  float d[3];
  sub3(d, pb, na);
  const float d1 = dot3(d, d);
  float t2 = ((pa[0] - ak) * abk + (pa[1] - au) * abu + (pa[2] - aw) * abw) / den;
  t2 = fminf(fmaxf(t2, 0.f), 1.f);
  const float nb[3] = {ak + abk * t2, au + abu * t2, aw + abw * t2};
  sub3(d, pa, nb);
  const float d2 = dot3(d, d);
  if (d1 < d2) copy3(pa, na); else copy3(pb, nb);
  float dir[3];
  sub3(dir, pa, pb);
  const bool deg = dot3(dir, dir) < 1e-6f;
  const float ed = normalize3(dir);
  const bool front = (eu * dir[1] < 0.f) && (ew * dir[2] < 0.f);
  out.epen = (!deg && front) ? r - ed : -1.f;
  out.deg = deg ? 1.f : 0.f;
  unpick3(out.dir, k, u, dir[0], dir[1], dir[2]);
  unpick3(out.pa, k, u, pa[0], pa[1], pa[2]);
  unpick3(out.pb, k, u, pb[0], pb[1], pb[2]);
  return out;
}
// The edges that pass capbox_edge_lane's interval test: bit e set iff edge e does (the others return epen = -1, which never
// becomes the contact).  The same comparisons, evaluated once per face: bit 2 j + (s > 0) of `face` says the segment reaches past
// face (j, s) and comes within r of its plane, bit j of `along` that it overlaps the r-inflated extent of axis j.
KFN int capbox_edge_mask(const float* a, const float* b, float r, const float* bsize) {
  int face = 0, along = 0;
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const float lo = fminf(a[j], b[j]), hi = fmaxf(a[j], b[j]), s = bsize[j], cn = -1.f * s;
    if (hi - s > 0.f && lo - s < r) face |= 2 << (2 * j);
    if (cn - lo > 0.f && cn - hi < r) face |= 1 << (2 * j);
    if (lo < s + r && hi > -s - r) along |= 1 << j;
  }
  int mask = 0;
#pragma unroll
  for (int e = 0; e < 12; ++e) {
    const int k = e >> 2, u = k == 2 ? 0 : k + 1, w = k == 0 ? 2 : k - 1;
    if (((along >> k) & 1) && ((face >> (2 * u + ((e >> 1) & 1))) & 1) && ((face >> (2 * w + (e & 1))) & 1)) mask |= 1 << e;
  }
  return mask;
}
template <bool FULL>
KFN void capsule_box(const float* A, const float* B, float r, const float* bpos, const float* bmat, const float* bsize, Contact2& c) {
  float a[3], b[3];
  capbox_local(A, B, bpos, bmat, a, b);
  c.dist[0] = 1.f; c.dist[1] = 1.f;
  if (capbox_far(a, b, r, bsize)) {
    if (FULL) { for (int j = 0; j < 2; ++j) { copy3(c.pos[j], bpos); c.nrm[j][0] = 1.f; c.nrm[j][1] = 0.f; c.nrm[j][2] = 0.f; } }
    return;
  }
  CapBoxOut o;
  capsule_box_near<FULL>(a, b, r, bsize, o);
  c.dist[0] = o.dist[0]; c.dist[1] = o.dist[1];
  if (FULL) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      float w[3];
      mat_vec(w, bmat, o.pos[j]); add3(c.pos[j], w, bpos);
      mat_vec(c.nrm[j], bmat, o.nrm[j]);
      normalize3(c.nrm[j]);
    }
  }
}

// ---- free-box colliders (lane-serial, rarely past the bounding-sphere test) -------------------
// 4-point manifold selection of MJX _manifold_points, with the oracle's distinct-point tie rule
KFN void manifold_points(int n, float poly[][3], const bool* mask, const float* nrm, int* idx) {
  float dm[16];
  for (int i = 0; i < n; ++i) dm[i] = mask[i] ? 0.f : -1e6f;
  int a = 0;
  for (int i = 1; i < n; ++i) if (dm[i] > dm[a]) a = i;
  int b = 0; float bv = 0.f;
  for (int i = 0; i < n; ++i) { float t[3]; sub3(t, poly[a], poly[i]); float v = dot3(t, t) + dm[i]; if (i == 0 || v > bv) { bv = v; b = i; } }
  float ab[3], t[3];
  sub3(t, poly[a], poly[b]); cross3(ab, nrm, t);
  int c = 0; float cv = 0.f;
  for (int i = 0; i < n; ++i) { float ap[3]; sub3(ap, poly[a], poly[i]); float v = fabsf(dot3(ap, ab)) + dm[i]; if (i == 0 || v > cv) { cv = v; c = i; } }
  float ac[3], bc[3];
  sub3(t, poly[a], poly[c]); cross3(ac, nrm, t);
  sub3(t, poly[b], poly[c]); cross3(bc, nrm, t);
  int dsel = 0; float dv = 0.f;
  for (int i = 0; i < n; ++i) {
    float bp[3], ap[3];
    sub3(bp, poly[b], poly[i]); sub3(ap, poly[a], poly[i]);
    float v = fmaxf(fabsf(dot3(bp, bc)), fabsf(dot3(ap, ac))) + dm[i] - ((i == a || i == b || i == c) ? 2e6f : 0.f);
    if (i == 0 || v > dv) { dv = v; dsel = i; }
  }
  idx[0] = a; idx[1] = b; idx[2] = c; idx[3] = dsel;
}
KFN void box_face(const float* s, int f, float v[4][3], float* n) {
  int k = f >> 1, u = (k + 1) % 3, w = (k + 2) % 3;
  float sg = (f & 1) ? -1.f : 1.f;
  n[0] = n[1] = n[2] = 0.f; n[k] = sg;
  const float su[4] = {-1.f, 1.f, 1.f, -1.f}, sw[4] = {-1.f, -1.f, 1.f, 1.f};
  for (int i = 0; i < 4; ++i) {
    int ii = (f & 1) ? 3 - i : i;
    v[i][k] = sg * s[k]; v[i][u] = su[ii] * s[u]; v[i][w] = sw[ii] * s[w];
  }
}
// plane (geom1) vs free box: out[k] = pos3, dist; normal = plane normal.  Only penetrating
// vertices matter (these slots never enter the cost), see oracle plane_box.
KNOINLINE int plane_box(const float* ppos, const float* pn, const float* bpos, const float* bmat, const float* bs, float out[4][4]) {
  float v[8][3], sup[8], t[3], pl[3], n[3], smax = -1e30f;
  bool mask[8]; int idx[4];
  sub3(t, ppos, bpos); matT_vec(pl, bmat, t); matT_vec(n, bmat, pn);
  for (int i = 0; i < 8; ++i) {
    v[i][0] = (i & 4 ? 1.f : -1.f) * bs[0]; v[i][1] = (i & 2 ? 1.f : -1.f) * bs[1]; v[i][2] = (i & 1 ? 1.f : -1.f) * bs[2];
    sub3(t, pl, v[i]); sup[i] = dot3(t, n); smax = fmaxf(smax, sup[i]);
  }
  float thr = fmaxf(0.f, smax - 1e-3f);
  for (int i = 0; i < 8; ++i) mask[i] = sup[i] > thr;
  manifold_points(8, v, mask, n, idx);
  int nact = 0;
  for (int k = 0; k < 4; ++k) {
    bool uniq = true;
    for (int q = 0; q < k; ++q) if (idx[q] == idx[k]) uniq = false;
    float w[3];
    mat_vec(w, bmat, v[idx[k]]); add3(w, w, bpos);
    float d = uniq ? -sup[idx[k]] : 1.f;
    madd3(out[k], w, pn, -0.5f * d);
    out[k][3] = d;
    nact += d < 0.f;
  }
  return nact;
}
// ---- rare parts of box_box_warp, out of line (they would otherwise sit, never executed, inside the step loop; each
//      builds a lane-group context of its own, see cold_warp).  `act`, `outside`, the polygon size and the results are
//      per sample (per lane group); everything else is read from the scratch the inlined part has filled. ----
// edge-edge contact: closest points of the two support edges
template <int NC>
KNOINLINE void bb_edge_edge(WarpSmemT<NC>& S, bool act, int slot, int bl, float bn0, float bn1, float bn2, const float* s1, const float* s2,
                            const float* m2, const float* p2) {
  Warp W;
  cold_warp(W, 0, 0);
  const float bn[3] = {bn0, bn1, bn2};
  float Rm[9], c[3];
#pragma unroll
  for (int k = 0; k < 9; ++k) Rm[k] = S.bbR[k];
  c[0] = S.bbc[0]; c[1] = S.bbc[1]; c[2] = S.bbc[2];
  const int be = bl >= 6 ? bl - 6 : 0;       // (a face-face sample of the same warp computes a dummy pair)
  const int bi = be / 3, bj = be % 3;
  float e1c[3] = {c[0], c[1], c[2]}, e2c[3] = {0.f, 0.f, 0.f};
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float Ak[3] = {Rm[k], Rm[3 + k], Rm[6 + k]};
    if (k != bi) { const float sg = dot3(Ak, bn) > 0.f ? 1.f : -1.f; madd3(e1c, e1c, Ak, sg * s1[k]); }
    if (k != bj) e2c[k] = (bn[k] > 0.f ? -1.f : 1.f) * s2[k];
  }
  const float Ab[3] = {S.bbR[bi], S.bbR[3 + bi], S.bbR[6 + bi]}, e2[3] = {bj == 0 ? 1.f : 0.f, bj == 1 ? 1.f : 0.f, bj == 2 ? 1.f : 0.f};
  float a0[3], a1[3], b0[3], b1[3];
  madd3(a0, e1c, Ab, -s1[bi]); madd3(a1, e1c, Ab, s1[bi]);
  madd3(b0, e2c, e2, -s2[bj]); madd3(b1, e2c, e2, s2[bj]);
  SegPair sp = closest_seg_seg_v(a0, a1, b0, b1);
  const float mid[3] = {0.5f * (sp.a[0] + sp.b[0]), 0.5f * (sp.a[1] + sp.b[1]), 0.5f * (sp.a[2] + sp.b[2])};
  float w[3], df[3];
  mat_vec(w, m2, mid); add3(w, w, p2);
  sub3(df, sp.b, sp.a);
  const float d = dot3(df, bn);
  UNIFORM_WRITE(W) { if (act && bl >= 6) { copy3(S.bstage[slot][0], w); S.bstage[slot][0][3] = d; } } END_UNIFORM_WRITE
}
// Sutherland-Hodgman of the incident face (S.bbpoly[0], four vertices) against the four side planes of the reference
// face, polygon edges on lanes; output slots by ballot (each edge emits its start vertex if inside, then the crossing
// point).  Returns (polygon size) | (buffer holding it) << 8.
template <int NC>
KNOINLINE int bb_clip(WarpSmemT<NC>& S, bool act, unsigned outside) {
  Warp W;
  cold_warp(W, 0, 0);
  int np = 4, cur = 0;
#pragma unroll 1
  for (int i = 0; i < 4; ++i) {
    const bool clip = act && np > 0 && outside != 0u;       // this sample still has something to clip
    if (!warp_any_groups(W, clip)) break;
    LANES(W, R)
      R.actmask = 0; R.f0 = 0.f;
      if (clip && lane < np) {
        const float* a = S.bbpoly[cur][lane]; const float* b = S.bbpoly[cur][lane + 1 == np ? 0 : lane + 1];
        float ta[3], tb[3];
        sub3(ta, a, S.bbrf[i]); sub3(tb, b, S.bbrf[i]);
        const float da = dot3(ta, S.bben[i]), db = dot3(tb, S.bben[i]);
        const bool keep = da <= 0.f, cross = (da < 0.f && db > 0.f) || (da > 0.f && db < 0.f);
        R.actmask = (keep ? 1 : 0) | (cross ? 2 : 0);
        R.f0 = cross ? da / (da - db) : 0.f;
      }
    END_LANES
    const unsigned mk = warp_ballot(W, [](int, LaneRegs& R) { return (R.actmask & 1) != 0; });
    const unsigned mx = warp_ballot(W, [](int, LaneRegs& R) { return (R.actmask & 2) != 0; });
    LANES(W, R)
      if (clip && lane < np && R.actmask) {
        const float* a = S.bbpoly[cur][lane]; const float* b = S.bbpoly[cur][lane + 1 == np ? 0 : lane + 1];
        const unsigned below = (1u << lane) - 1u;
        int o = KPOPC(mk & below) + KPOPC(mx & below);
        if (R.actmask & 1) { copy3(S.bbpoly[cur ^ 1][o], a); ++o; }
        if (R.actmask & 2) { float ab[3]; sub3(ab, b, a); madd3(S.bbpoly[cur ^ 1][o], a, ab, R.f0); }
      }
    END_LANES
    if (clip) { np = KPOPC(mk) + KPOPC(mx); cur ^= 1; }
  }
  return np | (cur << 8);
}
// MJX's 4-point manifold rule on a clipped polygon of more than four vertices (S.bbpref = the vertices projected on the
// reference face, [3] = height; negative = penetrating)
template <int NC>
KNOINLINE void bb_manifold(WarpSmemT<NC>& S, bool act, int slot, int np, bool swap, float rn0, float rn1, float rn2, const float* m2, const float* p2) {
  Warp W;
  cold_warp(W, 0, 0);
  const float rn[3] = {rn0, rn1, rn2};
  float Rm[9], c[3];
#pragma unroll
  for (int k = 0; k < 9; ++k) Rm[k] = S.bbR[k];
  c[0] = S.bbc[0]; c[1] = S.bbc[1]; c[2] = S.bbc[2];
  LANES(W, R)
    R.f0 = (lane < np && S.bbpref[lane < 8 ? lane : 0][3] < 0.f) ? 0.f : -1e6f;            // dm: only penetrating vertices compete
  END_LANES
  // lanes >= np must never win: give them -inf in every argmax
  const int ia = warp_argmax_first8(W, [&](int l, LaneRegs& R) { return l < np ? R.f0 : -INFINITY; });
  LANES(W, R)
    R.f1 = -INFINITY;
    if (lane < np) { float t[3]; sub3(t, S.bbpref[ia], S.bbpref[lane]); R.f1 = dot3(t, t) + R.f0; }
  END_LANES
  const int ib = warp_argmax_first8(W, [](int, LaneRegs& R) { return R.f1; });
  float ab[3];
  { float t[3]; sub3(t, S.bbpref[ia], S.bbpref[ib]); cross3(ab, rn, t); }
  LANES(W, R)
    R.f1 = -INFINITY;
    if (lane < np) { float ap[3]; sub3(ap, S.bbpref[ia], S.bbpref[lane]); R.f1 = fabsf(dot3(ap, ab)) + R.f0; }
  END_LANES
  const int ic = warp_argmax_first8(W, [](int, LaneRegs& R) { return R.f1; });
  float ac[3], bc[3];
  { float t[3]; sub3(t, S.bbpref[ia], S.bbpref[ic]); cross3(ac, rn, t); sub3(t, S.bbpref[ib], S.bbpref[ic]); cross3(bc, rn, t); }
  LANES(W, R)
    R.f1 = -INFINITY;
    if (lane < np) {
      float bp[3], ap[3];
      sub3(bp, S.bbpref[ib], S.bbpref[lane]); sub3(ap, S.bbpref[ia], S.bbpref[lane]);
      R.f1 = fmaxf(fabsf(dot3(bp, bc)), fabsf(dot3(ap, ac))) + R.f0 - ((lane == ia || lane == ib || lane == ic) ? 2e6f : 0.f);
    }
  END_LANES
  const int id = warp_argmax_first8(W, [](int, LaneRegs& R) { return R.f1; });
  const int idx[4] = {ia, ib, ic, id};
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    bool uniq = true;
#pragma unroll
    for (int z = 0; z < q; ++z) if (idx[z] == idx[q]) uniq = false;
    const float h = S.bbpref[idx[q]][3];
    const bool put = act && h < 0.f && uniq;
    float w[3];
    if (swap) { float u[3]; mat_vec(u, Rm, S.bbpref[idx[q]]); add3(u, u, c); mat_vec(w, m2, u); }
    else mat_vec(w, m2, S.bbpref[idx[q]]);
    add3(w, w, p2);
    UNIFORM_WRITE(W) { if (put) { copy3(S.bstage[slot][q], w); S.bstage[slot][q][3] = h; } } END_UNIFORM_WRITE
  }
}

// Warp-cooperative box (geom1) vs box (geom2).  Same algorithm, axis order and tie rules as the
// oracle's box_box (SAT over face2 x3, face1 x3, edge x edge 3x3; clipped face
// manifold reduced by the 4-point rule, or one edge-edge contact), with the 15 axes, the polygon edges
// and the polygon vertices spread over lanes: the resting target_0 / table pair is evaluated every
// step, and the scalar version on one lane was 30 % of all issued warp instructions (profiles/r1c).
// Called by the whole warp with warp-uniform control flow: both samples walk the same path (the union of
// what they need) and `act` switches a sample's result writes off once it is done or if it does not test
// this pair at all.  Writes S.bstage[slot][k] = pos3, dist (dist = 1: unused) and S.bnrm[slot].
template <int NC>
KFN void box_box_warp(Warp& W, WarpSmemT<NC>& S, bool act, int slot, const float* p1, const float* m1, const float* s1,
                      const float* p2, const float* m2, const float* s2) {
  LANES(W, R)
    if (lane < 9) { const int i = lane / 3, j = lane % 3; S.bbR[lane] = m2[i] * m1[j] + m2[3 + i] * m1[3 + j] + m2[6 + i] * m1[6 + j]; }
    else if (lane < 12) { const int i = lane - 9; S.bbc[i] = m2[i] * (p1[0] - p2[0]) + m2[3 + i] * (p1[1] - p2[1]) + m2[6 + i] * (p1[2] - p2[2]); }
    else if (lane < 16 && act) { float* o = S.bstage[slot][lane - 12]; o[0] = o[1] = o[2] = 0.f; o[3] = 1.f; }
  END_LANES
  // ---- separating axes, one per lane ----
  LANES(W, R)
    float cmp = -INFINITY, a0 = 0.f, a1 = 0.f, a2 = 1.f, sgn = 1.f;
    if (lane < 15) {
      const float* Rm = S.bbR; const float* c = S.bbc;
      bool ok = true;
      if (lane < 3) { a0 = lane == 0 ? 1.f : 0.f; a1 = lane == 1 ? 1.f : 0.f; a2 = lane == 2 ? 1.f : 0.f; }
      else if (lane < 6) { const int i = lane - 3; a0 = Rm[i]; a1 = Rm[3 + i]; a2 = Rm[6 + i]; }
      else {
        const int i = (lane - 6) / 3, j = (lane - 6) % 3;
        const float x = Rm[i], y = Rm[3 + i], z = Rm[6 + i];
        if (j == 0) { a0 = 0.f; a1 = z; a2 = -y; } else if (j == 1) { a0 = -z; a1 = 0.f; a2 = x; } else { a0 = y; a1 = -x; a2 = 0.f; }
        const float n = sqrtf(a0 * a0 + a1 * a1 + a2 * a2);
        if (n > 0.f) { const float in = 1.f / n; a0 *= in; a1 *= in; a2 *= in; } else { a0 = a1 = a2 = 0.f; }
        ok = !(n < 1e-6f);
      }
      float r1 = 0.f;
#pragma unroll
      for (int k = 0; k < 3; ++k) r1 += s1[k] * fabsf(Rm[k] * a0 + Rm[3 + k] * a1 + Rm[6 + k] * a2);
      const float r2 = s2[0] * fabsf(a0) + s2[1] * fabsf(a1) + s2[2] * fabsf(a2);
      const float dc = c[0] * a0 + c[1] * a1 + c[2] * a2;
      if (ok) cmp = fabsf(dc) - r1 - r2 - (lane >= 6 ? 1e-6f : 0.f);
      sgn = dc > 0.f ? -1.f : 1.f;          // contact normal points from box 1 (at c) to box 2 (origin)
    }
    R.f0 = cmp; R.f1 = a0 * sgn; R.f2 = a1 * sgn; R.acc[0] = a2 * sgn;
  END_LANES
  const int bl = warp_argmax_first(W, [](int, LaneRegs& R) { return R.f0; });
  const float bestsep = warp_bcast(W, bl, [](int, LaneRegs& R) { return R.f0; });
  act = act && !(bestsep > 0.f);             // separated: no slot can be active
  if (!warp_any_groups(W, act)) return;
  const float bn[3] = {warp_bcast(W, bl, [](int, LaneRegs& R) { return R.f1; }), warp_bcast(W, bl, [](int, LaneRegs& R) { return R.f2; }),
                       warp_bcast(W, bl, [](int, LaneRegs& R) { return R.acc[0]; })};
  {
    float nw[3];
    mat_vec(nw, m2, bn);
    normalize3(nw);
    UNIFORM_WRITE(W) { if (act) copy3(S.bnrm[slot], nw); } END_UNIFORM_WRITE
  }
  float Rm[9], c[3];
#pragma unroll
  for (int k = 0; k < 9; ++k) Rm[k] = S.bbR[k];
  c[0] = S.bbc[0]; c[1] = S.bbc[1]; c[2] = S.bbc[2];
  if (warp_any_groups(W, act && bl >= 6)) bb_edge_edge<NC>(S, act, slot, bl, bn[0], bn[1], bn[2], s1, s2, m2, p2);      // rare, out of line
  act = act && bl < 6;
  if (!warp_any_groups(W, act)) return;
  // ---- face-face: reference face on the box owning the axis, incident face on the other ----
  const bool swap = bl >= 3 && bl < 6;         // reference = box 1
  float rc[3], Rr[9], nref[3];
  if (!swap) {
    copy3(rc, c);
#pragma unroll
    for (int k = 0; k < 9; ++k) Rr[k] = Rm[k];
    nref[0] = -bn[0]; nref[1] = -bn[1]; nref[2] = -bn[2];
  } else {
    const float mc[3] = {-c[0], -c[1], -c[2]};
    matT_vec(rc, Rm, mc);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) Rr[3 * i + j] = Rm[3 * j + i];
    matT_vec(nref, Rm, bn);
  }
  const float* rs = swap ? s1 : s2; const float* is = swap ? s2 : s1;
  int rk = 0;
  if (fabsf(nref[1]) > fabsf(nref[0])) rk = 1;
  if (fabsf(nref[2]) > fabsf(rk == 0 ? nref[0] : nref[1])) rk = 2;
  const float rsg = (rk == 0 ? nref[0] : (rk == 1 ? nref[1] : nref[2])) > 0.f ? 1.f : -1.f;
  const float rn[3] = {rk == 0 ? rsg : 0.f, rk == 1 ? rsg : 0.f, rk == 2 ? rsg : 0.f};
  // incident face: most anti-parallel to rn (first minimum over +x,-x,+y,-y,+z,-z of the incident box)
  int inf = 0; float mind = 1e30f;
#pragma unroll
  for (int f = 0; f < 6; ++f) {
    const int kk = f >> 1; const float sg = (f & 1) ? -1.f : 1.f;
    const float dd = sg * (Rr[kk] * rn[0] + Rr[3 + kk] * rn[1] + Rr[6 + kk] * rn[2]);
    if (dd < mind) { mind = dd; inf = f; }
  }
  // box face f = 2*axis + (0:+, 1:-), vertices counter-clockwise seen from outside:
  // in-plane signs (u, w) = (-,-),(+,-),(+,+),(-,+) for +k, reversed for -k  (u = k+1, w = k+2 cyclic)
  LANES(W, R)
    if (lane < 8) {
      const bool ref = lane < 4;
      const int i = lane & 3;
      const int k = ref ? rk : (inf >> 1);
      const float sg = ref ? rsg : ((inf & 1) ? -1.f : 1.f);
      const float* sz = ref ? rs : is;
      const int ii = sg < 0.f ? 3 - i : i;
      const float su = (ii == 1 || ii == 2) ? 1.f : -1.f, sw = ii >= 2 ? 1.f : -1.f;
      const int u = (k + 1) % 3, w = (k + 2) % 3;
      float v[3];
      v[0] = k == 0 ? sg * sz[0] : (u == 0 ? su * sz[0] : sw * sz[0]);
      v[1] = k == 1 ? sg * sz[1] : (u == 1 ? su * sz[1] : sw * sz[1]);
      v[2] = k == 2 ? sg * sz[2] : (u == 2 ? su * sz[2] : sw * sz[2]);
      if (ref) copy3(S.bbrf[i], v);
      else { float t[3]; mat_vec(t, Rr, v); add3(S.bbpoly[0][i], t, rc); }
    }
  END_LANES
  LANES(W, R)
    if (lane < 4) {                            // outward side-plane normals of the reference face
      float e[3], en[3];
      sub3(e, S.bbrf[lane], S.bbrf[(lane + 3) & 3]);
      cross3(en, e, rn); normalize3(en);
      copy3(S.bben[lane], en);
    }
  END_LANES
  // ---- Sutherland-Hodgman against the four side planes, polygon edges on lanes; output slots by
  //      ballot (each edge emits its start vertex if inside, then the crossing point) ----
  int np = 4, cur = 0;
  // common case (a box resting on a larger one): every incident vertex is inside every side plane,
  // so clipping would return the polygon unchanged -- 16 tests on 16 lanes and one ballot
  const unsigned outside = warp_ballot(W, [&](int l, LaneRegs&) {
    if (l >= 16) return false;
    float t[3];
    sub3(t, S.bbpoly[0][l & 3], S.bbrf[l >> 2]);
    return dot3(t, S.bben[l >> 2]) > 0.f;
  });
  if (warp_any_groups(W, act && outside != 0u)) {                  // rare, out of line
    const int r = bb_clip<NC>(S, act, outside);
    if (act && outside != 0u) { np = r & 0xff; cur = r >> 8; }
  }
  act = act && np > 0;
  if (!warp_any_groups(W, act)) return;
  // ---- penetrating vertices projected on the reference face; 4-point manifold ----
  LANES(W, R)
    R.f0 = -1e6f; R.actmask = 0;
    if (lane < np) {
      float tt[3];
      sub3(tt, S.bbpoly[cur][lane], S.bbrf[0]);
      const float h = dot3(tt, rn);
      madd3(S.bbpref[lane], S.bbpoly[cur][lane], rn, -h);
      S.bbpref[lane][3] = h;
      R.actmask = h < 0.f;
      R.f0 = h < 0.f ? 0.f : -1e6f;            // dm
    }
  END_LANES
  if (warp_any_groups(W, act && np <= 4)) {
    // With at most four vertices MJX's 4-point rule returns exactly the penetrating ones (every
    // later pick prefers a not-yet-chosen vertex); emit them in polygon order.
    const unsigned pen = warp_ballot(W, [&](int l, LaneRegs& R) { return l < np && R.actmask != 0; });
    LANES(W, R)
      if (act && np <= 4 && (pen & (1u << lane))) {
        const int q = KPOPC(pen & ((1u << lane) - 1u));
        float w[3];
        if (swap) { float u[3]; mat_vec(u, Rm, S.bbpref[lane]); add3(u, u, c); mat_vec(w, m2, u); }
        else mat_vec(w, m2, S.bbpref[lane]);
        add3(w, w, p2);
        copy3(S.bstage[slot][q], w); S.bstage[slot][q][3] = S.bbpref[lane][3];
      }
    END_LANES
  }
  act = act && np > 4;
  if (!warp_any_groups(W, act)) return;
  bb_manifold<NC>(S, act, slot, np, swap, rn[0], rn[1], rn[2], m2, p2);             // more than four vertices: rare, out of line
}

// ------------------------------------------------------------------------------------------ constraints
KFN float pow_pos(float x, float p) { return p == 2.f ? x * x : (p == 1.f ? x : powf(x, p)); }
// MJX constraint._kbi + row regulariser (BD.8)
KNOINLINE void row_params(const KModel& m, float pos, float invw, float vel, float& D, float& aref) {
  float tc = fmaxf(m.solref[0], 2.f * m.dt), dr = m.solref[1];
  float dmin = fminf(fmaxf(m.solimp[0], MJ_MINIMP), MJ_MAXIMP), dmax = fminf(fmaxf(m.solimp[1], MJ_MINIMP), MJ_MAXIMP);
  float width = fmaxf(m.solimp[2], MJ_MINVAL), mid = fminf(fmaxf(m.solimp[3], MJ_MINIMP), MJ_MAXIMP), power = fmaxf(m.solimp[4], 1.f);
  float k = 1.f / (dmax * dmax * tc * tc * dr * dr), b = 2.f / (dmax * tc);
  if (m.solref[0] <= 0.f) k = -m.solref[0] / (dmax * dmax);
  if (m.solref[1] <= 0.f) b = -m.solref[1] / dmax;
  float x = fabsf(pos) / width, y;
  if (x < mid) y = pow_pos(x, power) / pow_pos(mid, power - 1.f);
  else y = 1.f - pow_pos(1.f - x, power) / pow_pos(1.f - mid, power - 1.f);
  float imp = fminf(fmaxf(dmin + y * (dmax - dmin), dmin), dmax);
  if (x > 1.f) imp = dmax;
  float R = fmaxf(invw * (1.f - imp) / imp, MJ_MINVAL);
  D = 1.f / R;
  aref = -b * vel - k * imp * pos;
}
// (M v)[d] and M[i][j] with the constant diagonal free-box block
template <int NC>
KFN float mul_M(const KModel& m, const WarpSmemT<NC>& S, int d, const float* v) {
  if (d < KM_NL) { float s = 0.f; for (int k = 0; k < KM_NL; ++k) s += S.Mr[d][k] * v[k]; return s; }
  return (d < KM_NL + 3 ? m.fb_mass : (d == KM_NL + 3 ? m.fb_inertia[0] : (d == KM_NL + 4 ? m.fb_inertia[1] : m.fb_inertia[2]))) * v[d];
}
// translational Jacobian column of world point p on `link` (0..5 robot link, 6 free box, <0 static)
template <int NC>
KFN void jac_col(const KModel& m, const WarpSmemT<NC>& S, const float* p, int link, int d, float* col) {
  col[0] = col[1] = col[2] = 0.f;
  if (link < 0) return;
  if (d < KM_NL) {
    if (link >= KM_NL || d > link) return;
    float off[3], t[3];
    sub3(off, p, m.refpt);
    cross3(t, S.cdof[d], off);
    add3(col, S.cdof[d] + 3, t);
  } else {
    if (link != KM_NL) return;
    int k = d - KM_NL;
    if (k < 3) { col[0] = k == 0 ? 1.f : 0.f; col[1] = k == 1 ? 1.f : 0.f; col[2] = k == 2 ? 1.f : 0.f; return; }   // (no dynamic index: keeps col in registers)
    k -= 3;
    float r[3] = {S.bmat[k], S.bmat[3 + k], S.bmat[6 + k]}, off[3];
    sub3(off, p, S.qpos + KM_NL);
    cross3(col, r, off);
  }
}

// Dense 6x6 SPD solve in registers, executed redundantly by every lane (uniform): for matrices this
// small a straight-line Cholesky beats a lane-distributed one, whose ~50 dependent shuffles cost more
// than the arithmetic (measured: profiles/README.md).  A: lower triangle read with row stride `ld`.
// The 4 pyramid rows of a contact are Jn +- mu*Jt1, Jn +- mu*Jt2: three dot products per contact (one
// (contact, component) item per lane) give all four J_r . v.
// which dof blocks a contact touches: bit 0 = robot (a link 0..5 on either side), bit 1 = free box.  Its Jacobian is
// identically zero in a block it does not touch; those entries are neither written (C2) nor read.
KFN int contact_blocks(const float* g) {
  const int l1 = (int)g[14], l2 = (int)g[15];
  return (((unsigned)l1 < (unsigned)KM_NL || (unsigned)l2 < (unsigned)KM_NL) ? 1 : 0) | ((l1 == KM_NL || l2 == KM_NL) ? 2 : 0);
}
template <int NC, bool SP>
KFN void contact_dots(Warp& W, WarpSmemT<NC>& S, int ncon, const float* v0, const float* v1) {
  LANES(W, R)
#pragma unroll 1
    for (int e = lane; e < 3 * ncon; e += KW) {
      const int c = e / 3, k = e - 3 * c;
      const int blk = contact_blocks(S.template geo<SP>(c));
      const float* J = S.template jac<SP>(c) + 12 * k;
      float s0 = 0.f, s1 = 0.f;
      if (blk != 3) {                               // one block (the usual case): six terms
        const int o = (blk & 1) ? 0 : KM_NL;
#pragma unroll
        for (int d = 0; d < KM_NL; ++d) { s0 += J[o + d] * v0[o + d]; if (v1) s1 += J[o + d] * v1[o + d]; }
      } else {
#pragma unroll
        for (int d = 0; d < KM_NV; ++d) { s0 += J[d] * v0[d]; if (v1) s1 += J[d] * v1[d]; }
      }
      S.template dots<SP>(0, c)[k] = s0;
      if (v1) S.template dots<SP>(1, c)[k] = s1;
    }
  END_LANES
}
template <int NC, bool SP>
KFN float row_val(const WarpSmemT<NC>& S, int set, int r, const float* v) {
  if (r < S.nlim) return S.limsign[r] * v[S.limdof[r]];
  const int c = (r - S.nlim) >> 2, q = (r - S.nlim) & 3;
  const float dn = S.template dots<SP>(set, c)[0], dt = S.template dots<SP>(set, c)[q < 2 ? 1 : 2];
  return (q & 1) ? dn - dt : dn + dt;
}

struct Vec6 { float v[6]; };
KNOINLINE Vec6 chol_solve6(const float* A, int ld, const float* rhs) {
  float L[6][6], y[6];
  Vec6 x;
#pragma unroll
  for (int i = 0; i < 6; ++i) {
#pragma unroll
    for (int j = 0; j <= i; ++j) {
      float s = A[i * ld + j];
#pragma unroll
      for (int k = 0; k < j; ++k) s -= L[i][k] * L[j][k];
      if (i == j) { const float d = sqrtf(s); L[i][i] = 1.f / d; }    // store the reciprocal of the diagonal
      else L[i][j] = s * L[j][j];
    }
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) { float s = rhs[i]; for (int k = 0; k < i; ++k) s -= L[i][k] * y[k]; y[i] = s * L[i][i]; }
#pragma unroll
  for (int i = 5; i >= 0; --i) { float s = y[i]; for (int k = i + 1; k < 6; ++k) s -= L[k][i] * x.v[k]; x.v[i] = s * L[i][i]; }
  return x;
}

// Cholesky solve with one matrix row per lane, all in registers.  N = 12: lanes 0..11 hold the
// rows of one 12x12 SPD matrix (R.h[k] = A[lane][k], k <= lane).  N = 6: two independent 6x6 systems
// at once, rows of the first on lanes 0..5 and of the second on lanes 6..11 (R.h[k] = A[lane][base+k]).
// In: R.h, R.f0 = right-hand side.  Out: R.f0 = A^-1 rhs.
template <int N>
KFN void chol_solve_rows(Warp& W) {
  static_assert(N == 6 || N == 12, "N");
  auto base = [](int l) { return (N == 6 && l >= 6 && l < 12) ? 6 : 0; };
  auto loc = [&](int l) { return l - base(l); };
  // The column loops below are too long for nvcc to unroll completely, so the row is indexed dynamically: work on
  // a copy (R.hrow) that only this rare path touches -- a dynamic index into LaneRegs::h itself would force the
  // whole per-lane state of the kernel out of registers into local memory.
#ifdef CEMK_EMU
#define CEMK_ROW(R) (R).hrow
#else
  float hrow_[N];
#define CEMK_ROW(R) hrow_
#endif
  RLANES(W, R)
#pragma unroll
    for (int k = 0; k < N; ++k) CEMK_ROW(R)[k] = R.h[k];
  END_RLANES
  for (int j = 0; j < N; ++j) {
    warp_shfl_each<true>(W, [&](int, LaneRegs& R) { return CEMK_ROW(R)[j]; }, [&](int l) { return base(l) + j; },
                   [&](int l, LaneRegs& R, float d) { const float dj = sqrtf(d); CEMK_ROW(R)[j] = (loc(l) == j) ? dj : CEMK_ROW(R)[j] / dj; });
    for (int k = j + 1; k < N; ++k)
      warp_shfl_each<true>(W, [&](int, LaneRegs& R) { return CEMK_ROW(R)[j]; }, [&](int l) { return base(l) + k; },
                     [&](int l, LaneRegs& R, float lkj) { if (loc(l) >= k) CEMK_ROW(R)[k] -= CEMK_ROW(R)[j] * lkj; });
  }
  for (int k = 0; k < N; ++k)                  // forward substitution L y = rhs
    warp_shfl_each<true>(W, [&](int, LaneRegs& R) { return R.f0 / CEMK_ROW(R)[k]; }, [&](int l) { return base(l) + k; },
                   [&](int l, LaneRegs& R, float yk) { if (loc(l) == k) R.f0 = yk; else if (loc(l) > k) R.f0 -= CEMK_ROW(R)[k] * yk; });
  for (int k = N - 1; k >= 0; --k) {           // back substitution L^T x = y, column k of L^T lives in lane base+k
    warp_shfl_each<true>(W, [&](int, LaneRegs& R) { return R.f0 / CEMK_ROW(R)[k]; }, [&](int l) { return base(l) + k; },
                   [&](int l, LaneRegs& R, float xk) { R.f1 = xk; if (loc(l) == k) R.f0 = xk; });
    for (int i = 0; i < k; ++i)
      warp_shfl_each<true>(W, [&](int, LaneRegs& R) { return CEMK_ROW(R)[i] * R.f1; }, [&](int l) { return base(l) + k; },
                     [&](int l, LaneRegs& R, float p) { if (loc(l) == i) R.f0 -= p; });
  }
#undef CEMK_ROW
}

// (Out of line like every routine with more than one call site: the address span of the step loop decides how well the
// instruction fetch of the lockstep warps works -- one inlined copy less of the box-box routine was worth 4 %.)
// sum over the contacts in `sel` (bit c = contact c; contacts >= 32 exist only for samples deep in collision and are
// tested one by one: `need` = the dof blocks of entry (i, j), 1 robot, 2 box, 3 cross) of the Hessian contribution of
// the four pyramid rows to entry (i, j)
template <int NC, bool SP>
KNOINLINE float hess_contacts(const WarpSmemT<NC>& S, unsigned sel, int need, int ncon, int i, int j) {
  float h = 0.f;
  auto term = [&](int c) {
    const float* g = S.template geo<SP>(c); const float* J = S.template jac<SP>(c);
    const float ni = J[i], nj = J[j], ai = J[12 + i], aj = J[12 + j], bi = J[24 + i], bj = J[24 + j];
    return g[3] * (ni + ai) * (nj + aj) + g[4] * (ni - ai) * (nj - aj) + g[5] * (ni + bi) * (nj + bj) + g[6] * (ni - bi) * (nj - bj);
  };
  if (sel != 0u && KPOPC(sel) <= 4) {
    // up to four contacts (the resting box): the four terms are independent, only their sum is ordered
    unsigned rem = sel;
    const int c0 = KFFS(rem) - 1; rem &= rem - 1u;
    const bool v1 = rem != 0u; const int c1 = v1 ? KFFS(rem) - 1 : c0; rem &= rem - 1u;
    const bool v2 = rem != 0u; const int c2 = v2 ? KFFS(rem) - 1 : c0; rem &= rem - 1u;
    const bool v3 = rem != 0u; const int c3 = v3 ? KFFS(rem) - 1 : c0;
    const float t0 = term(c0), t1 = term(c1), t2 = term(c2), t3 = term(c3);
    h = t0;
    if (v1) h += t1;
    if (v2) h += t2;
    if (v3) h += t3;
  } else {
#pragma unroll 1
    for (unsigned rem = sel; rem != 0u; rem &= rem - 1u) h += term(KFFS(rem) - 1);
  }
  if (KM_NC_TOT > 32) {
#pragma unroll 1
    for (int c = 32; c < ncon; ++c) {
      const float* g = S.template geo<SP>(c); const float* J = S.template jac<SP>(c);
      if ((__float_as_int(g[7]) & need) != need) continue;       // the Jacobian only exists in the blocks the contact touches
      const float ni = J[i], nj = J[j], ai = J[12 + i], aj = J[12 + j], bi = J[24 + i], bj = J[24 + j];
      h += g[3] * (ni + ai) * (nj + aj) + g[4] * (ni - ai) * (nj - aj) + g[5] * (ni + bi) * (nj + bj) + g[6] * (ni - bi) * (nj - bj);
    }
  }
  return h;
}

struct LSPoint { float alpha, cost, d0, d1; };
KFN bool in_bracket(const LSPoint& x, const LSPoint& y) {
  return ((x.d0 < y.d0) && (y.d0 < 0.f)) || ((x.d0 > y.d0) && (y.d0 > 0.f));
}

// write one contact record (position, frame, distance, weights, the two links); t1 = own first tangent or nullptr
template <int NC>
KFN void put_contact(WarpSmemT<NC>& S, int o, const float* pos, const float* nrm, const float* t1, float dist, float invw, int l1, int l2) {
  if (o >= KM_NC_TOT) return;
  float* g = S.template geo<true>(o);             // rare path: a pointer into either space is fine here
  copy3(g, pos); copy3(g + 3, nrm);
  if (t1) { copy3(g + 6, t1); cross3(g + 9, nrm, t1); }
  else make_tangents(nrm, g + 6, g + 9);
  g[12] = dist; g[13] = invw; g[14] = (float)l1; g[15] = (float)l2;
}
// emit the full contact records of one lane's active plane-capsule / capsule-capsule slots; rare path
// (capsule-box contacts are written by the near pass of the narrow phase itself)
template <int NC>
KNOINLINE void emit_robot_contacts(const KModel& m, WarpSmemT<NC>& S, int lane, int actmask, int o) {
#pragma unroll 1
  for (int p = m.ncbpass; p < KM_NPASS; ++p) {
    const int bits = (actmask >> (2 * p)) & 3;
    if (!bits) continue;
    const int x = m.rp[p * KW + lane], ty = KP_TYPE(x), a = KP_A(x), b = KP_B(x);
    Contact2 c;
    float invw; int l1, l2;
    float pt1[3]; bool own_t1 = false;
    if (ty == KP_CAP_CAP) {
      capsule_capsule<true>(S.capA[a], S.capB[a], m.cap_r[a], S.capA[b], S.capB[b], m.cap_r[b], c);
      invw = m.cap_invw[a] + m.cap_invw[b]; l1 = m.cap_link[a]; l2 = m.cap_link[b];
    } else {
      plane_capsule<true>(m.plane_pos, m.plane_n, S.capA[b], S.capB[b], m.cap_r[b], c);
      invw = m.cap_invw[b]; l1 = -1; l2 = m.cap_link[b];
      // MJX plane_capsule: first tangent = capsule axis projected on the plane
      float ax[3];
      sub3(ax, S.capB[b], S.capA[b]); normalize3(ax);
      madd3(pt1, ax, m.plane_n, -dot3(m.plane_n, ax));
      if (normalize3(pt1) < 0.5f) {
        pt1[0] = 0.f;
        if (m.plane_n[1] > -0.5f && m.plane_n[1] < 0.5f) { pt1[1] = 1.f; pt1[2] = 0.f; } else { pt1[1] = 0.f; pt1[2] = 1.f; }
      }
      own_t1 = true;
    }
#pragma unroll 1
    for (int k = 0; k < 2; ++k) {
      if (!((bits >> k) & 1)) continue;
      put_contact<NC>(S, o, c.pos[k], c.nrm[k], own_t1 ? pt1 : nullptr, c.dist[k], invw, l1, l2);
      ++o;
    }
  }
}
// per-step observation / cost hooks of the narrow phase
struct StepIO {
  bool first;                 // t == 0: no previous distance yet
  float* collision_row;       // optional dump of this step's robot-slot distances [nslot_robot]
  float* prevd;               // this sample's previous-step distances, [2 * KM_NPASS][KW] (global scratch, L2-resident)
  // step_forward<NC, true> only (null: not this step): per contact in list order, its key (robot slot, or nslot_robot +
  // 4 box pair + slot; RolloutArgs::slot_map) and a KM_CON_REC record with dist, pos and normal.  The solve overwrites the
  // position and frame in the contact record, so contact_outputs takes them from here.
  int* con_key;
  float* con_rec;
};
#define KM_CON_REC 12                     // floats per contact output record: dist, pos[3], normal[3], force[3], 2 unused

// search = -H^-1 grad for the full 12x12 system (a contact couples a robot link and the free box).  Cold: a real
// function with its own lane-group context; may be entered by one of the two samples of a warp (D-flavoured fences).
template <int NC>
KNOINLINE void coupled_solve(WarpSmemT<NC>& S) {
  Warp W;
  cold_warp(W, 0, 0);
  DLANES(W, R)
#pragma unroll
    for (int k = 0; k < KM_NV; ++k) R.h[k] = (lane < KM_NV && k <= lane) ? S.H[lane][k] : 0.f;
    R.f0 = lane < KM_NV ? S.grad[lane] : 0.f;
  END_DLANES
  chol_solve_rows<12>(W);
  DLANES(W, R)
    if (lane < KM_NV) S.search[lane] = -R.f0;
  END_DLANES
}

// ------------------------------------------------------------------------------------------ constraint solve
// C2 .. S5 of one forward(): rows of the active constraints, Newton direction, line search.  SP = true is
// the instantiation for a sample whose contact list does not fit shared memory (spill area, see WarpSmemT).
template <int NC, bool SP>
KFN void solve_rows(Warp& W, const KModel& m, WarpSmemT<NC>& S, const int ncon, const int nlim, const int nrow) {
  PHASE(W, 16);
  // ---- C2: contact Jacobians in the contact frame: Jn, mu*Jt1, mu*Jt2 ----
  LANES(W, R)
    // one (contact, dof of a block the contact touches) item per lane: six items per contact, twelve for a contact
    // between a robot link and the free box
#pragma unroll 1
    for (int e = lane; e < KM_NL * ncon; e += KW) {
      const int c = e / KM_NL, k = e - KM_NL * c;
      const float* g = S.template geo<SP>(c);
      const int blk = contact_blocks(g);
      float* J = S.template jac<SP>(c);
#pragma unroll 1
      for (int d = (blk & 1) ? k : KM_NL + k; d < KM_NV; d += KM_NL) {       // (the second trip only for blk == 3)
        float c1[3], c2[3], df[3];
        jac_col(m, S, g, (int)g[14], d, c1);
        jac_col(m, S, g, (int)g[15], d, c2);
        sub3(df, c2, c1);
        J[d] = dot3(g + 3, df);
        J[12 + d] = m.mu * dot3(g + 6, df);
        J[24 + d] = m.mu * dot3(g + 9, df);
        if (blk != 3) break;
      }
    }
  END_LANES
  PHASE(W, 17);
  // ---- C3: contact row parameters (the 4 pyramid edges share pos and D) ----
  contact_dots<NC, SP>(W, S, ncon, S.qvel, nullptr);
  LANES(W, R)
#pragma unroll 1
    for (int r = nlim + lane; r < nrow; r += KW) {
      const float* g = S.template geo<SP>((r - nlim) >> 2);
      float w = g[13];
      w = w + m.mu * m.mu * w;
      w = w * 2.f * m.mu * m.mu / m.impratio;
      float vel = row_val<NC, SP>(S, 0, r, S.qvel), D, aref;
      row_params(m, g[12], w, vel, D, aref);
      S.template D<SP>(r, nlim) = D; S.template Aref<SP>(r, nlim) = aref;
    }
    // does any active contact join a robot link and the free box?  (then H is a full 12x12)
    R.f2 = 0.f;
    for (int c = lane; c < ncon; c += KW) {
      const int l1 = (int)S.template geo<SP>(c)[14], l2 = (int)S.template geo<SP>(c)[15];
      if ((l1 == KM_NL && l2 >= 0 && l2 < KM_NL) || (l2 == KM_NL && l1 >= 0 && l1 < KM_NL)) R.f2 = 1.f;
    }
  END_LANES
  const bool coupled = warp_sum(W, [](int, LaneRegs& R) { return R.f2; }) > 0.f;
  PHASE(W, 8);
  // ---- S1: warm start vs smooth start (B.6) ----
  contact_dots<NC, SP>(W, S, ncon, S.warm, S.as);
  LANES(W, R)
    float cw = 0.f, cs = 0.f;
#pragma unroll 1
    for (int r = lane; r < nrow; r += KW) {
      const float ar = S.template Aref<SP>(r, nlim), Dr = S.template D<SP>(r, nlim);
      float jw = row_val<NC, SP>(S, 0, r, S.warm) - ar, js = row_val<NC, SP>(S, 1, r, S.as) - ar;
      S.template Jaref<SP>(r, nlim) = jw; S.template Jv<SP>(r, nlim) = js;
      if (jw < 0.f) cw += 0.5f * Dr * jw * jw;
      if (js < 0.f) cs += 0.5f * Dr * js * js;
    }
    R.f0 = cw; R.f1 = cs; R.f2 = 0.f;
    if (lane < KM_NV) {
      float ma = mul_M<NC>(m, S, lane, S.warm);
      S.Ma[lane] = ma;
      R.f2 = 0.5f * (ma - S.fs[lane]) * (S.warm[lane] - S.as[lane]);
    }
  END_LANES
  const float gauss_w = warp_sum(W, [](int, LaneRegs& R) { return R.f2; });
  const float cost_w = warp_sum(W, [](int, LaneRegs& R) { return R.f0; }) + gauss_w;
  const float cost_s = warp_sum(W, [](int, LaneRegs& R) { return R.f1; });
  const bool use_warm = cost_w < cost_s;
#ifdef CEMK_EMU_DEBUG
  printf("[emu] nrow %d nlim %d ncon %d cost_w %.9g cost_s %.9g use_warm %d\n", nrow, nlim, ncon, cost_w, cost_s, (int)use_warm);
#endif
  const float gauss = use_warm ? gauss_w : 0.f;
  LANES(W, R)
    if (!use_warm) {
      for (int r = lane; r < nrow; r += KW) S.template Jaref<SP>(r, nlim) = S.template Jv<SP>(r, nlim);
      if (lane < KM_NV) {
        S.Ma[lane] = mul_M<NC>(m, S, lane, S.as);
      }
    }
    if (lane < KM_NV) S.qacc[lane] = use_warm ? S.warm[lane] : S.as[lane];
  END_LANES
  PHASE(W, 9);
  // ---- S3: gradient and Hessian over the active rows (BD.9) ----
  // per contact: the pyramid-edge weights w_q = D [Jaref_q < 0] and the force sums that multiply
  // Jn, mu*Jt1, mu*Jt2; the contact position / frame slots of cgeo are dead after C2 and are reused.
  LANES(W, R)
#pragma unroll 1
    for (int c = lane; c < ncon; c += KW) {
      const int r0 = nlim + 4 * c;
      float w[4], f[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) { const float ja = S.template Jaref<SP>(r0 + q, nlim); w[q] = ja < 0.f ? S.template D<SP>(r0 + q, nlim) : 0.f; f[q] = -w[q] * ja; }
      float* g = S.template geo<SP>(c);
      const int l1 = (int)g[14], l2 = (int)g[15];
      g[0] = f[0] + f[1] + f[2] + f[3]; g[1] = f[0] - f[1]; g[2] = f[2] - f[3];
      g[3] = w[0]; g[4] = w[1]; g[5] = w[2]; g[6] = w[3];
      g[7] = __int_as_float((((l1 >= 0 && l1 < KM_NL) || (l2 >= 0 && l2 < KM_NL)) ? 1 : 0) | ((l1 == KM_NL || l2 == KM_NL) ? 2 : 0));
    }
  END_LANES
  // which contacts touch the robot block / the box block (ncon <= 32: one bit per contact); the loops
  // below then visit only the contacts that can contribute (typically: 4 box contacts, no robot contact)
  const unsigned mrob = warp_ballot32(W, [&](int l) { return l < ncon && (__float_as_int(S.template geo<SP>(l)[7]) & 1); });
  const unsigned mbox = warp_ballot32(W, [&](int l) { return l < ncon && (__float_as_int(S.template geo<SP>(l)[7]) & 2); });
  LANES(W, R)
    if (lane < KM_NV) {
      float fc = 0.f;
#pragma unroll 1
      for (int r = 0; r < nlim; ++r) { const float ja = S.rJaref[r]; if (ja < 0.f && S.limdof[r] == lane) fc += S.limsign[r] * (-S.rD[r] * ja); }
      {
        const unsigned sel = lane < KM_NL ? mrob : mbox;
        auto term = [&](int c) {
          const float* g = S.template geo<SP>(c); const float* J = S.template jac<SP>(c);
          return J[lane] * g[0] + J[12 + lane] * g[1] + J[24 + lane] * g[2];
        };
        if (sel != 0u && KPOPC(sel) <= 4) {
          unsigned rem = sel;
          const int c0 = KFFS(rem) - 1; rem &= rem - 1u;
          const bool v1 = rem != 0u; const int c1 = v1 ? KFFS(rem) - 1 : c0; rem &= rem - 1u;
          const bool v2 = rem != 0u; const int c2 = v2 ? KFFS(rem) - 1 : c0; rem &= rem - 1u;
          const bool v3 = rem != 0u; const int c3 = v3 ? KFFS(rem) - 1 : c0;
          const float t0 = term(c0), t1 = term(c1), t2 = term(c2), t3 = term(c3);
          fc += t0;
          if (v1) fc += t1;
          if (v2) fc += t2;
          if (v3) fc += t3;
        } else {
#pragma unroll 1
          for (unsigned rem = sel; rem != 0u; rem &= rem - 1u) fc += term(KFFS(rem) - 1);
        }
      }
      if (KM_NC_TOT > 32) {
#pragma unroll 1
        for (int c = 32; c < ncon; ++c) {        // more than 32 contacts: deep-collision samples only
          const float* g = S.template geo<SP>(c); const float* J = S.template jac<SP>(c);
          if (!(__float_as_int(g[7]) & (lane < KM_NL ? 1 : 2))) continue;
          fc += J[lane] * g[0] + J[12 + lane] * g[1] + J[24 + lane] * g[2];
        }
      }
      S.grad[lane] = S.Ma[lane] - S.fs[lane] - fc;
    }
  END_LANES
  // Hessian by blocks: lanes 0-20 own entry (i, j) of the 6x6 lower triangle and build it for the robot
  // block and for the box block; the 36 robot/box cross entries exist only when a contact couples the two
  // (otherwise the blocks are solved separately and the cross entries are never read).
  LANES(W, R)
#pragma unroll
   for (int q = 0; q < 32 / KW; ++q) {
    const int i = (R.tri >> (8 * q)) & 15, j = (R.tri >> (8 * q + 4)) & 15;
    if (i < KM_NL) {
      float hr = S.Mr[i][j];
#pragma unroll 1
      for (int r = 0; r < nlim; ++r) if (S.rJaref[r] < 0.f && S.limdof[r] == i && i == j) hr += S.rD[r];      // (rolled: limit rows are rare, their code must stay small)
      hr += hess_contacts<NC, SP>(S, mrob, 1, ncon, i, j);
      S.H[i][j] = hr;
      float hb = i != j ? 0.f : (i < 3 ? m.fb_mass : (i == 3 ? m.fb_inertia[0] : (i == 4 ? m.fb_inertia[1] : m.fb_inertia[2])));
      hb += hess_contacts<NC, SP>(S, mbox, 2, ncon, KM_NL + i, KM_NL + j);
      S.H[KM_NL + i][KM_NL + j] = hb;
    }
   }
    if (coupled) {
#pragma unroll 1
      for (int e = lane; e < KM_NL * KM_NL; e += KW) {
        const int i = KM_NL + e / KM_NL, j = e % KM_NL;
        S.H[i][j] = hess_contacts<NC, SP>(S, mrob & mbox, 3, ncon, i, j);
      }
    }
  END_LANES
  PHASE(W, 10);
  // ---- S4: search = -H^-1 grad, Cholesky with one row per lane in registers.  Robot and box
  //      blocks only couple through a robot/box contact; otherwise the two 6x6 blocks are factorised
  //      side by side (6 column steps instead of 12) ----
  {
    USYNC();
    const Vec6 xr = chol_solve6(&S.H[0][0], KM_NV, S.grad);
    const Vec6 xb = chol_solve6(&S.H[KM_NL][KM_NL], KM_NV, S.grad + KM_NL);
    UNIFORM_WRITE(W) {
      for (int i = 0; i < KM_NL; ++i) { S.search[i] = -xr.v[i]; S.search[KM_NL + i] = -xb.v[i]; }
    } END_UNIFORM_WRITE
  }
  EVENT(W, 7, coupled);
  if (coupled) coupled_solve<NC>(S);            // rare: full 12x12 system (replaces the block solution above); out of line
  REGROUP();
  PHASE_ALIGN();
  PHASE(W, 11);
  // ---- S5: line search (BD.10) ----
  // J.search per row, the Gauss-term sums and the constraint sums of the starting point alpha = 0
  // (MJX's p0) in one pass and one fused warp reduction
  contact_dots<NC, SP>(W, S, ncon, S.search, nullptr);
  LANES(W, R)
    float e0 = 0.f, e1 = 0.f, e2 = 0.f, a0 = 0.f, a1 = 0.f, a2 = 0.f;
    if (lane < KM_NV) {
      const float mv = mul_M<NC>(m, S, lane, S.search), s = S.search[lane];
      e0 = s * s; e1 = s * S.Ma[lane] - s * S.fs[lane]; e2 = 0.5f * s * mv;
    }
    // the lane's first row stays in registers for the line-search trips (R.h is free after the solve):
    // ja, jv and the three quadratic coefficients; an idle lane gets a row that is never active
    R.h[0] = 1.f; R.h[1] = 0.f; R.h[2] = 0.f; R.h[3] = 0.f; R.h[4] = 0.f;
#pragma unroll 1
    for (int r = lane; r < nrow; r += KW) {
      const float jv = row_val<NC, SP>(S, 0, r, S.search), ja = S.template Jaref<SP>(r, nlim), D = S.template D<SP>(r, nlim);
      S.template Jv<SP>(r, nlim) = jv;
      const float q0 = 0.5f * D * ja * ja, q1 = D * jv * ja, q2 = 0.5f * D * jv * jv;
      if (r == lane) { R.h[0] = ja; R.h[1] = jv; R.h[2] = q0; R.h[3] = q1; R.h[4] = q2; }
      if (ja < 0.f) { a0 += q0; a1 += q1; a2 += q2; }
    }
    R.acc[0] = e0; R.acc[1] = e1; R.acc[2] = e2; R.acc[3] = a0; R.acc[4] = a1; R.acc[5] = a2; R.acc[6] = R.acc[7] = R.acc[8] = 0.f;
  END_LANES
  float qg[3], gtol;
  LSPoint p0, lo, hi;
  {
    float sums[9];
    warp_sum9(W, sums);
    qg[0] = gauss; qg[1] = sums[1]; qg[2] = sums[2];
    gtol = m.tolerance * m.ls_tolerance * sqrtf(sums[0]) * m.meaninertia * (float)KM_NV;
    const float q2 = qg[2] + sums[5];
    p0.alpha = 0.f; p0.cost = qg[0] + sums[3]; p0.d0 = qg[1] + sums[4]; p0.d1 = 2.f * q2 + (q2 == 0.f ? MJ_MINVAL : 0.f);
    lo = p0; hi = p0;
  }
  PHASE(W, 19);
  // One rolled loop evaluates the piecewise quadratic at three step sizes per trip:
  //   trip -1: lo = point(-p0.d0/p0.d1); trips 0..ls_iterations-1: MJX bracket update.
  // The loop is warp-uniform: it runs until every sample of the warp is done; a sample that finished
  // earlier idles through the remaining trips with its bracket frozen.
  bool swapped = true, done = nrow == 0;
#pragma unroll 1
  for (int it = -1; it < m.ls_iterations; ++it) {
    float al0, al1, al2;
    if (it == -1) { al0 = al1 = al2 = p0.alpha - p0.d0 / p0.d1; }
    else {
      done = done || !swapped;
      done = done || ((lo.d0 < 0.f) && (lo.d0 > -gtol));
      done = done || ((hi.d0 > 0.f) && (hi.d0 < gtol));
      if (warp_all_groups(W, done)) break;
      EVENT(W, 6, 1); EVENT(W, 5, !done);
      al0 = lo.alpha - lo.d0 / lo.d1; al1 = hi.alpha - hi.d0 / hi.d1; al2 = 0.5f * (lo.alpha + hi.alpha);
    }
    // rows are read-only here and the sums live in registers: no fences inside the loop
    RLANES(W, R)
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, b0 = 0.f, b1 = 0.f, b2 = 0.f, c0 = 0.f, c1 = 0.f, c2 = 0.f;
      {
        const float ja = R.h[0], jv = R.h[1], q0 = R.h[2], q1 = R.h[3], q2 = R.h[4];
        if (ja + al0 * jv < 0.f) { a0 = q0; a1 = q1; a2 = q2; }
        if (ja + al1 * jv < 0.f) { b0 = q0; b1 = q1; b2 = q2; }
        if (ja + al2 * jv < 0.f) { c0 = q0; c1 = q1; c2 = q2; }
      }
#pragma unroll 1
      for (int r = lane + KW; r < nrow; r += KW) {             // more than KW rows: the rest from shared memory
        const float ja = S.template Jaref<SP>(r, nlim), jv = S.template Jv<SP>(r, nlim), D = S.template D<SP>(r, nlim);
        const float q0 = 0.5f * D * ja * ja, q1 = D * jv * ja, q2 = 0.5f * D * jv * jv;
        if (ja + al0 * jv < 0.f) { a0 += q0; a1 += q1; a2 += q2; }
        if (ja + al1 * jv < 0.f) { b0 += q0; b1 += q1; b2 += q2; }
        if (ja + al2 * jv < 0.f) { c0 += q0; c1 += q1; c2 += q2; }
      }
      R.acc[0] = a0; R.acc[1] = a1; R.acc[2] = a2; R.acc[3] = b0; R.acc[4] = b1; R.acc[5] = b2; R.acc[6] = c0; R.acc[7] = c1; R.acc[8] = c2;
    END_RLANES
    float sums[9];
    warp_sum9(W, sums);
    LSPoint pt[3];
    const float als[3] = {al0, al1, al2};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float q0 = qg[0] + sums[3 * k], q1 = qg[1] + sums[3 * k + 1], q2 = qg[2] + sums[3 * k + 2];
      const float a = als[k];
      pt[k].alpha = a;
      pt[k].cost = a * a * q2 + a * q1 + q0;
      pt[k].d0 = 2.f * a * q2 + q1;
      pt[k].d1 = 2.f * q2 + (q2 == 0.f ? MJ_MINVAL : 0.f);
    }
    if (it == -1) {
      if (pt[0].d0 < p0.d0) { lo = pt[0]; hi = p0; } else { hi = pt[0]; lo = p0; }
      continue;
    }
    if (done) continue;
    const LSPoint lo_next = pt[0], hi_next = pt[1], mid = pt[2];
    bool s1 = in_bracket(lo, lo_next); if (s1) lo = lo_next;
    bool s2 = in_bracket(lo, mid);     if (s2) lo = mid;
    bool s3 = in_bracket(lo, hi_next); if (s3) lo = hi_next;
    bool s4 = in_bracket(hi, hi_next); if (s4) hi = hi_next;
    bool s5 = in_bracket(hi, mid);     if (s5) hi = mid;
    bool s6 = in_bracket(hi, lo_next); if (s6) hi = lo_next;
    swapped = s1 || s2 || s3 || s4 || s5 || s6;
#ifdef CEMK_EMU_DEBUG
    printf("[emu]  it %d cand %.7g %.7g %.7g -> lo a %.7g d0 %.5g  hi a %.7g d0 %.5g swaps %d%d%d%d%d%d\n", it, al0, al1, al2, lo.alpha, lo.d0, hi.alpha, hi.d0, s1, s2, s3, s4, s5, s6);
#endif
  }
  const bool improved = (lo.cost < p0.cost) || (hi.cost < p0.cost);
#ifdef CEMK_EMU_DEBUG
  printf("[emu] p0 cost %.9g d0 %.6g d1 %.6g | lo a %.7g cost %.9g d0 %.6g | hi a %.7g cost %.9g d0 %.6g | gtol %.3g\n", p0.cost, p0.d0, p0.d1, lo.alpha, lo.cost, lo.d0, hi.alpha, hi.cost, hi.d0, gtol);
#endif
  const float alpha = improved ? (lo.cost < hi.cost ? lo.alpha : hi.alpha) : 0.f;
  LANES(W, R)
    if (lane < KM_NV) {
      float a = S.qacc[lane] + alpha * S.search[lane];
      if (nrow == 0) a = S.as[lane];
      S.qacc[lane] = a; S.warm[lane] = a;
    }
  END_LANES
}

// the spill-capable instantiation (a sample of the warp has more contacts than fit its shared-memory record): cold, out
// of line, with its own lane-group context (solve_rows leaves its results in the sample's record, nothing in registers)
template <int NC>
KNOINLINE void solve_rows_spilled(const KModel& m, WarpSmemT<NC>& S, int ncon, int nlim, int nrow, int bar, int nthr) {
  Warp W;
  cold_warp(W, bar, nthr);
  solve_rows<NC, true>(W, m, S, ncon, nlim, nrow);
}

// ------------------------------------------------------------------------------------------ one forward()
// Inputs: S.qpos, S.qvel, S.warm.  Outputs: S.qacc (= new warm start), link frames, and the
// collision-cost contribution of this step added to R.cost_c (mjx_planner.py:287-296).
// CON: also the contact keys and geometry of io.con_key / io.con_rec when they are set.
// SCENE: the static boxes' poses come from the sample's scene record `scene` (the table's sb_pos | sb_mat | sb_size block,
// KM_SCENE_FLOATS floats), not from the table.
template <int NC, bool CON = false, bool SCENE = false>
KFN void step_forward(Warp& W, const KModel& m, WarpSmemT<NC>& S, const StepIO& io, const float* scene = nullptr) {
  const float (*sb_pos)[4] = SCENE ? reinterpret_cast<const float (*)[4]>(scene) : m.sb_pos;
  const float (*sb_mat)[12] = SCENE ? reinterpret_cast<const float (*)[12]>(scene + 4 * KM_MAXSBOX) : m.sb_mat;
  const float (*sb_size)[4] = SCENE ? reinterpret_cast<const float (*)[4]>(scene + 16 * KM_MAXSBOX) : m.sb_size;
  PHASE(W, 1);
  // ---- P1: joint chain as a parallel prefix of rigid transforms.  Lane 0 holds the static base frame, lane
  //      i = 1..6 the local transform of link i-1 (body quat x joint rotation, body offset); composition
  //      (qa, pa) o (qb, pb) = (qa qb, pa + R(qa) pb) is associative, so three shuffle rounds replace the six
  //      dependent link-by-link products.  R.h[0..3] = quaternion, R.h[4..6] = position. ----
  LANES(W, R)
    R.h[0] = 1.f; R.h[1] = R.h[2] = R.h[3] = 0.f; R.h[4] = R.h[5] = R.h[6] = 0.f;
    if (lane == 0) {
      R.h[0] = m.base_quat[0]; R.h[1] = m.base_quat[1]; R.h[2] = m.base_quat[2]; R.h[3] = m.base_quat[3];
      R.h[4] = m.base_pos[0]; R.h[5] = m.base_pos[1]; R.h[6] = m.base_pos[2];
    } else if (lane <= KM_NL) {
      const int i = lane - 1;
      float sn, cs, qj[4], ql[4];
      k_sincos(0.5f * S.qpos[i], &sn, &cs);
      qj[0] = cs; qj[1] = sn * m.l_axis[i][0]; qj[2] = sn * m.l_axis[i][1]; qj[3] = sn * m.l_axis[i][2];
      quat_mul(ql, m.l_quat[i], qj);
      R.h[0] = ql[0]; R.h[1] = ql[1]; R.h[2] = ql[2]; R.h[3] = ql[3];
      R.h[4] = m.l_pos[i][0]; R.h[5] = m.l_pos[i][1]; R.h[6] = m.l_pos[i][2];
    } else if (lane == 8 && m.has_box) {
      float* q = S.qpos + KM_NL + 3;
      float inv = 1.f / sqrtf(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
      q[0] *= inv; q[1] *= inv; q[2] *= inv; q[3] *= inv;
      quat_to_mat(S.bmat, q);
    }
  END_LANES
#pragma unroll
  for (int o = 1; o < 8; o <<= 1) {
    // fetch the prefix that ends o lanes below (R.acc[0..6] as the receive buffer), then compose
#pragma unroll
    for (int k = 0; k < 7; ++k)
      warp_shfl_each(W, [&](int, LaneRegs& R) { return R.h[k]; }, [&](int l) { return l >= o ? l - o : l; },
                     [&](int, LaneRegs& R, float v) { R.acc[k] = v; });
    RLANES(W, R)
      if (lane >= o && lane <= KM_NL) {
        const float qa[4] = {R.acc[0], R.acc[1], R.acc[2], R.acc[3]}, qb[4] = {R.h[0], R.h[1], R.h[2], R.h[3]};
        const float pb[3] = {R.h[4], R.h[5], R.h[6]};
        float q[4], t[3], u[3];
        quat_mul(q, qa, qb);
        // R(qa) pb = pb + 2 w (v x pb) + 2 v x (v x pb),  qa = (w, v)
        cross3(t, qa + 1, pb);
        cross3(u, qa + 1, t);
        R.h[0] = q[0]; R.h[1] = q[1]; R.h[2] = q[2]; R.h[3] = q[3];
        R.h[4] = R.acc[4] + pb[0] + 2.f * (qa[0] * t[0] + u[0]);
        R.h[5] = R.acc[5] + pb[1] + 2.f * (qa[0] * t[1] + u[1]);
        R.h[6] = R.acc[6] + pb[2] + 2.f * (qa[0] * t[2] + u[2]);
      }
    END_RLANES
  }
  LANES(W, R)
    if (lane >= 1 && lane <= KM_NL) {
      const int i = lane - 1;
      const float q[4] = {R.h[0], R.h[1], R.h[2], R.h[3]};
      S.lpos[i][0] = R.h[4]; S.lpos[i][1] = R.h[5]; S.lpos[i][2] = R.h[6];
      for (int k = 0; k < 4; ++k) S.lquat[i][k] = q[k];
      quat_to_mat(S.lmat[i], q);
    }
  END_LANES
  PHASE(W, 2);
  // ---- P2: per-link spatial quantities, capsule end points, box frame ----
  LANES(W, R)
#pragma unroll 1
   for (int it = lane; it < KM_NL + m.ncap; it += KW) {
    if (it < KM_NL) {
      const int i = it;
      float a[3], off[3], com[3], d[3], t[3];
      mat_vec(a, S.lmat[i], m.l_axis[i]);
      sub3(off, m.refpt, S.lpos[i]);
      copy3(S.cdof[i], a);
      cross3(S.cdof[i] + 3, a, off);
      mat_vec(t, S.lmat[i], m.l_com[i]); add3(com, S.lpos[i], t);
      sub3(d, com, m.refpt);
      const float* I = m.l_inertia[i]; const float* Rm = S.lmat[i];
      float ms = I[6];
      float RI[9];
      for (int r = 0; r < 3; ++r) {
        RI[3 * r + 0] = Rm[3 * r] * I[0] + Rm[3 * r + 1] * I[3] + Rm[3 * r + 2] * I[4];
        RI[3 * r + 1] = Rm[3 * r] * I[3] + Rm[3 * r + 1] * I[1] + Rm[3 * r + 2] * I[5];
        RI[3 * r + 2] = Rm[3 * r] * I[4] + Rm[3 * r + 1] * I[5] + Rm[3 * r + 2] * I[2];
      }
      float T00 = RI[0] * Rm[0] + RI[1] * Rm[1] + RI[2] * Rm[2];
      float T11 = RI[3] * Rm[3] + RI[4] * Rm[4] + RI[5] * Rm[5];
      float T22 = RI[6] * Rm[6] + RI[7] * Rm[7] + RI[8] * Rm[8];
      float T01 = RI[0] * Rm[3] + RI[1] * Rm[4] + RI[2] * Rm[5];
      float T02 = RI[0] * Rm[6] + RI[1] * Rm[7] + RI[2] * Rm[8];
      float T12 = RI[3] * Rm[6] + RI[4] * Rm[7] + RI[5] * Rm[8];
      float* ci = S.cinert[i];
      ci[0] = T00 + ms * (d[1] * d[1] + d[2] * d[2]);
      ci[1] = T11 + ms * (d[0] * d[0] + d[2] * d[2]);
      ci[2] = T22 + ms * (d[0] * d[0] + d[1] * d[1]);
      ci[3] = T01 - ms * d[0] * d[1];
      ci[4] = T02 - ms * d[0] * d[2];
      ci[5] = T12 - ms * d[1] * d[2];
      ci[6] = ms * d[0]; ci[7] = ms * d[1]; ci[8] = ms * d[2]; ci[9] = ms;
    } else {
      const int j = it - KM_NL, L = m.cap_link[j];
      float cpos[3], ax[3], t[3];
      mat_vec(t, S.lmat[L], m.cap_pos[j]); add3(cpos, S.lpos[L], t);
      mat_vec(ax, S.lmat[L], m.cap_axis[j]);
      madd3(S.capA[j], cpos, ax, -m.cap_hl[j]);
      madd3(S.capB[j], cpos, ax, m.cap_hl[j]);
    }
   }
  END_LANES
  // ---- P3: composite inertias (suffix sums over the chain, one inertia component per lane 0-9) and link
  //      velocities (prefix sums, one spatial component per lane 10-15) (BD.3, BD.4) ----
  LANES(W, R)
    if (lane < 10) {
      float s = 0.f;
#pragma unroll
      for (int b = KM_NL - 1; b >= 0; --b) { s += S.cinert[b][lane]; S.crb[b][lane] = s; }
    } else if (lane < 16) {
      const int k = lane - 10;
      float v = 0.f;
#pragma unroll
      for (int b = 0; b < KM_NL; ++b) { v += S.cdof[b][k] * S.qvel[b]; S.cvel[b][k] = v; }
    }
  END_LANES
  // ---- P4: robot inertia matrix entries (lanes 0-20), cdof_dot (lanes 24-29) ----
  LANES(W, R)
#pragma unroll
    for (int q = 0; q < 32 / KW; ++q) {
      const int i = (R.tri >> (8 * q)) & 15, j = (R.tri >> (8 * q + 4)) & 15;
      if (i < KM_NL) {
        float buf[6];
        mul_inert(buf, S.crb[i], S.cdof[i]);
        float v = dot6(S.cdof[j], buf);
        if (i == j) v += m.l_armature[i];
        S.Mr[i][j] = v; S.Mr[j][i] = v;
      }
    }
    if (lane >= KW - KM_NL) {                  // the last six lanes (idle in the second pass above)
      const int i = lane - (KW - KM_NL);
      if (i == 0) { for (int k = 0; k < 6; ++k) S.cdofdot[0][k] = 0.f; }
      else cross_motion(S.cdofdot[i], S.cvel[i - 1], S.cdof[i]);
    }
  END_LANES
  // ---- P4b: per-link bias wrench (BD.5 without gravity) ----
  LANES(W, R)
    if (lane < KM_NL) {
      const int i = lane;
      float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, f[6], t[6], t2[6];
      for (int b = 1; b <= i; ++b) for (int k = 0; k < 6; ++k) acc[k] += S.cdofdot[b][k] * S.qvel[b];
      mul_inert(f, S.cinert[i], acc);
      mul_inert(t, S.cinert[i], S.cvel[i]);
      cross_force(t2, S.cvel[i], t);
      for (int k = 0; k < 6; ++k) S.cfrc[i][k] = f[k] + t2[k];
    }
  END_LANES
  // ---- P5: qfrc_smooth ----
  LANES(W, R)
    if (lane < KM_NL) {
      float f[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int b = lane; b < KM_NL; ++b) for (int k = 0; k < 6; ++k) f[k] += S.cfrc[b][k];
      S.fs[lane] = -dot6(S.cdof[lane], f) - m.l_damping[lane] * S.qvel[lane];
    } else if (lane < KM_NV) {
      const int k = lane - KM_NL;
      const float* w = S.qvel + KM_NL + 3;
      if (k < 3) S.fs[lane] = m.fb_mass * m.grav[k] - m.fb_damping * S.qvel[lane];
      else {
        float Iw[3] = {m.fb_inertia[0] * w[0], m.fb_inertia[1] * w[1], m.fb_inertia[2] * w[2]}, g[3];
        cross3(g, w, Iw);
        S.fs[lane] = -(k == 3 ? g[0] : (k == 4 ? g[1] : g[2])) - m.fb_damping * S.qvel[lane];
      }
    }
  END_LANES
  PHASE(W, 3);
  // ---- P6: qacc_smooth = M^-1 qfrc_smooth (robot block by a uniform 6x6 Cholesky; box block is diagonal) ----
  {
    USYNC();
    const Vec6 x = chol_solve6(&S.Mr[0][0], KM_NL, S.fs);
    UNIFORM_WRITE(W) {
      for (int i = 0; i < KM_NL; ++i) S.as[i] = x.v[i];
      for (int k = 0; k < 3; ++k) { S.as[KM_NL + k] = S.fs[KM_NL + k] / m.fb_mass; S.as[KM_NL + 3 + k] = S.fs[KM_NL + 3 + k] / m.fb_inertia[k]; }
    } END_UNIFORM_WRITE
  }
  PHASE(W, 4);
  // ---- N1: narrow phase + collision cost of this step (mjx_planner.py:287-296:
  //      cost_c = sum max(0, (1-y) c_t - c_{t+1}) + #(c < 0), y = 0.005) ----
  // Capsule-box (70 of the 107 pairs): lane l keeps capsule l in registers and walks the boxes; a pair is decided by
  // its far-field test (both slots = +1, see capsule_box) and then costs nothing -- not even its previous
  // distances are touched while it stays far (R.farprev).  The few pairs that are not far are *compacted* into a
  // per-sample list and evaluated densely by the first lanes, full contact records included, so a sample's narrow
  // phase costs one extra collider pass however its near pairs are spread over the table (the warps of a CTA
  // step in lockstep: the slowest one sets the pace).
  LANES(W, R)
    int nact = 0, actmask = 0, nearbits = 0, farbits = 0;
    float cc = 0.f;
    float* pd = io.prevd + lane;
    if (lane < m.ncap) {
      const float A[3] = {S.capA[lane][0], S.capA[lane][1], S.capA[lane][2]}, B[3] = {S.capB[lane][0], S.capB[lane][1], S.capB[lane][2]};
      const float r = m.cap_r[lane];
#pragma unroll 2
      for (int p = 0; p < m.ncbpass; ++p) {
        const bool st = p < m.nsbox;
        float la[3], lb[3];
        bool far;
        if (st && sb_size[p][3] != 0.f) {
          // axis-aligned static box: its frame is a signed permutation of the world axes, so the box coordinates are
          // the world offsets up to order and sign and the test is the same arithmetic on (A - c, B - c) with the
          // permuted half sizes -- bit-identical decision without the change of frame
          sub3(la, A, sb_pos[p]); sub3(lb, B, sb_pos[p]);
          far = capbox_far(la, lb, r, sb_mat[p] + 9);
        } else {
          capbox_local(A, B, st ? sb_pos[p] : S.qpos + KM_NL, st ? sb_mat[p] : S.bmat, la, lb);
          far = capbox_far(la, lb, r, st ? sb_size[p] : m.fb_size);
        }
        const bool valid = KP_TYPE(m.rp[p * KW + lane]) == KP_CAP_BOX;
        if (valid) { if (far) farbits |= 1 << p; else nearbits |= 1 << p; }
      }
    }
    // previous distances of the pairs that stay near (an L2 round trip): fetched here by the owner lane, handed to the
    // near pass through the sample's record at the end of this block, so the latency hides behind the other passes
    int pf = 0, pf0 = 0, pf1 = 0;
    float q00 = 0.f, q01 = 0.f, q10 = 0.f, q11 = 0.f;
    if (!io.first) {
      int rem = nearbits & ~R.farprev;
      if (rem) { pf0 = KFFS(rem) - 1; rem &= rem - 1; pf = 1; q00 = pd[(2 * pf0) * KW]; q01 = pd[(2 * pf0 + 1) * KW]; }
      if (rem) { pf1 = KFFS(rem) - 1; pf = 2; q10 = pd[(2 * pf1) * KW]; q11 = pd[(2 * pf1 + 1) * KW]; }
    }
    // a far pair whose previous distances were real: (1-y) c_t - 1 can only be positive for c_t > 1 / (1-y)
    if (!io.first) {
#pragma unroll 1
      for (int rem = farbits & ~R.farprev; rem; rem &= rem - 1) {
        const int p = KFFS(rem) - 1;
        cc += fmaxf((1.f - 0.005f) * pd[(2 * p) * KW] - 1.f, 0.f) + fmaxf((1.f - 0.005f) * pd[(2 * p + 1) * KW] - 1.f, 0.f);
      }
    }
    if (io.collision_row) {
#pragma unroll 1
      for (int rem = farbits; rem; rem &= rem - 1) {
        const int sl = KP_SLOT(m.rp[(KFFS(rem) - 1) * KW + lane]);
        io.collision_row[sl] = 1.f; io.collision_row[sl + 1] = 1.f;
      }
    }
    R.off = nearbits | ((nearbits & R.farprev) << 16);     // near pairs, and which of them were far one step ago
    R.farprev = farbits;
    // plane-capsule and capsule-capsule passes: previous distances of this lane's two slots, fetched one pass ahead
    // so the L2 latency hides behind the collider (asynchronous copies into the sample's record at the start of the step,
    // cp.async, were measured 3.7 % slower)
    float pv0 = 0.f, pv1 = 0.f;
    if (!io.first) { pv0 = pd[(2 * m.ncbpass) * KW]; pv1 = pd[(2 * m.ncbpass + 1) * KW]; }
#pragma unroll 1
    for (int p = m.ncbpass; p < KM_NPASS; ++p) {
      const int e = p * KW + lane;
      const int x = m.rp[e], ty = KP_TYPE(x);
      const float prev0 = pv0, prev1 = pv1;
      if (!io.first && p + 1 < KM_NPASS) { pv0 = pd[(2 * p + 2) * KW]; pv1 = pd[(2 * p + 3) * KW]; }
      if (ty == KP_NONE) continue;
      const int a = KP_A(x), b = KP_B(x);
      float d0, d1 = 1.f;
      Contact2 c;
      if (ty == KP_CAP_CAP) {
        capsule_capsule<false>(S.capA[a], S.capB[a], m.cap_r[a], S.capA[b], S.capB[b], m.cap_r[b], c);
        d0 = c.dist[0];
      } else {
        plane_capsule<false>(m.plane_pos, m.plane_n, S.capA[b], S.capB[b], m.cap_r[b], c);
        d0 = c.dist[0]; d1 = c.dist[1];
      }
      const int ns = ty == KP_CAP_CAP ? 1 : 2;
      if (d0 < 0.f) { ++nact; actmask |= 1 << (2 * p); cc += 1.f; }
      if (!io.first) cc += fmaxf((1.f - 0.005f) * prev0 - d0, 0.f);
      pd[(2 * p) * KW] = d0;
      if (ns == 2) {
        if (d1 < 0.f) { ++nact; actmask |= 1 << (2 * p + 1); cc += 1.f; }
        if (!io.first) cc += fmaxf((1.f - 0.005f) * prev1 - d1, 0.f);
        pd[(2 * p + 1) * KW] = d1;
      }
      if (io.collision_row) {
        io.collision_row[KP_SLOT(x)] = d0;
        if (ns == 2) io.collision_row[KP_SLOT(x) + 1] = d1;
      }
    }
    R.cost_c += cc;
    if (pf >= 1) { S.nprev[pf0 * KW + lane][0] = q00; S.nprev[pf0 * KW + lane][1] = q01; }
    if (pf >= 2) { S.nprev[pf1 * KW + lane][0] = q10; S.nprev[pf1 * KW + lane][1] = q11; }
    R.acc[6] = __int_as_float((pf >= 1 ? 1 << pf0 : 0) | (pf >= 2 ? 1 << pf1 : 0));     // which near pairs have their previous distances in S.nprev
    R.acc[7] = __int_as_float(actmask);        // parked: the near pass and the cooperative box colliders below reuse the scratch fields
    R.acc[8] = __int_as_float(nact);
  END_LANES
  PHASE(W, 20);
  int ncbcon = 0;                                  // capsule-box contacts: they open the contact list
  {
    // List position of a near pair: lane-major (capsule), pass-minor (box).
    int ntot = warp_excl_scan(W, [](int, LaneRegs& R) { return KPOPC(R.off & 0xffff); }, [](int, LaneRegs& R, int o) { R.actmask = o; });
    EVENT(W, 0, 1); EVENT(W, 1, ntot > 0); EVENT(W, 2, ntot); EVENT(W, 11, warp_any_groups(W, ntot > 0));
    // (Letting every warp walk this pass with a dummy pair, so that it runs in lockstep like the rest of the step, was
    //  measured: +1.4 %.)
    if (warp_any_groups(W, ntot > 0)) {
      LANES(W, R)
        int o = R.actmask;
#pragma unroll 1
        for (int rem = R.off & 0xffff; rem; rem &= rem - 1, ++o) {
          const int p = KFFS(rem) - 1;
          S.nlist[o] = (unsigned short)((p * KW + lane) | (((__float_as_int(R.acc[6]) >> p) & 1) << 14) | (((R.off >> (16 + p)) & 1) << 15));
                                                                   // bit 14: previous distances prefetched, bit 15: the pair was far one step ago
        }
      END_LANES
      PHASE(W, 21);
#pragma unroll 1
      for (int i0 = 0; warp_any_groups(W, i0 < ntot); i0 += KW) {
        const long long tk0 = TICK(); (void)tk0;
        // (1) one near pair per lane: the face part of the collider (both slots, in box coordinates; parked in R.h); the
        //     pairs that need the edge stage leave their box-frame geometry in S.estage and their candidate edges in R.off
        LANES(W, R)
          const int i = i0 + lane;
          R.off = 0;
          R.f2 = -1.f;                           // best edge penetration so far (only a positive one can become the contact)
          if (i < ntot) {
            const int e = S.nlist[i] & 0x3fff, x = m.rp[e], a = KP_A(x), b = KP_B(x);
            const bool st = b < m.nsbox;
            const float* bsz = st ? sb_size[b] : m.fb_size;
            // (the list holds exactly the pairs that failed the far test: straight to the near path)
            float la[3], lb[3], nf[3];
            CapBoxOut c;
            capbox_local(S.capA[a], S.capB[a], st ? sb_pos[b] : S.qpos + KM_NL, st ? sb_mat[b] : S.bmat, la, lb);
            const int nout = capsule_box_near<true, false>(la, lb, m.cap_r[a], bsz, c, nf);
#pragma unroll
            for (int k = 0; k < 3; ++k) { R.h[k] = c.pos[0][k]; R.h[3 + k] = c.nrm[0][k]; R.h[6 + k] = c.pos[1][k]; R.h[9 + k] = c.nrm[1][k]; }
            R.f0 = c.dist[0]; R.f1 = c.dist[1];
            if (nout >= 2) {
              R.off = capbox_edge_mask(la, lb, m.cap_r[a], bsz);
              float* g = S.estage[lane];
              g[0] = la[0]; g[1] = la[1]; g[2] = la[2]; g[3] = lb[0]; g[4] = lb[1]; g[5] = lb[2];
              g[6] = bsz[0]; g[7] = bsz[1]; g[8] = bsz[2]; g[9] = m.cap_r[a]; g[10] = nf[0]; g[11] = nf[1]; g[12] = nf[2];
            }
          }
        END_LANES
        // (2) the shallow edge contact of those pairs (MJX: closest box edge in front of two faces, see capbox_edges).  The
        //     candidate edges of all pairs of the group are items in (list slot, edge) order, dealt KW per round over the lanes,
        //     so a round serves every pair at once.  A pair's items are consecutive, in ascending edge order, and its owner folds
        //     them in that order keeping strictly greater penetrations: the first maximum, as capbox_edges and a lane argmax.
        const int nitem = warp_excl_scan(W, [](int, LaneRegs& R) { return KPOPC(R.off); }, [](int, LaneRegs& R, int o) { R.actmask = o; });
        if (warp_any_groups(W, nitem > 0)) {
          LANES(W, R)
            int it = R.actmask;
#pragma unroll 1
            for (int rem = R.off; rem; rem &= rem - 1, ++it) S.eidx[it] = (unsigned short)((lane << 4) | (KFFS(rem) - 1));
          END_LANES
#pragma unroll 1
          for (int base = 0; warp_any_groups(W, base < nitem); base += KW) {
            LANES(W, R)
              const int it = base + lane;
              if (it < nitem) {
                const int q = S.eidx[it] >> 4;
                const float* g = S.estage[q];
                const EdgeEval e1 = capbox_edge_lane<false>(S.eidx[it] & 15, g, g + 3, g[9], g + 6);
                float* o = S.eres[lane];
                o[0] = e1.epen;
                if (e1.epen > 0.f) {
                  o[1] = e1.dir[0]; o[2] = e1.dir[1]; o[3] = e1.dir[2];
                  o[4] = 0.5f * (e1.pa[0] + e1.pb[0] + e1.dir[0] * g[9]); o[5] = 0.5f * (e1.pa[1] + e1.pb[1] + e1.dir[1] * g[9]);
                  o[6] = 0.5f * (e1.pa[2] + e1.pb[2] + e1.dir[2] * g[9]);
                }
              }
            END_LANES
            // the owner folds its items of this round (parked in R.f2 / R.acc[0..5]); after its last one, edge contact or not
            LANES(W, R)
              const int lo = R.actmask > base ? R.actmask : base, end = R.actmask + KPOPC(R.off);
#pragma unroll 1
              for (int it = lo; it < end && it < base + KW; ++it) {
                const float* o = S.eres[it - base];
                if (o[0] > R.f2) {
                  R.f2 = o[0];
                  if (o[0] > 0.f) { R.acc[0] = o[1]; R.acc[1] = o[2]; R.acc[2] = o[3]; R.acc[3] = o[4]; R.acc[4] = o[5]; R.acc[5] = o[6]; }
                }
              }
              if (end > base && end <= base + KW && R.f2 > 0.f) {
                const float* nf = S.estage[lane] + 10;
                const float bpen = R.f2, minface = fminf(-R.f0, -R.f1);
                const bool parallel = fabsf(R.acc[0] * nf[0] + R.acc[1] * nf[1] + R.acc[2] * nf[2]) > 0.99f;
                if ((minface > 0.f ? bpen < minface : true) && !parallel) {
                  R.f0 = -bpen;
                  R.h[0] = R.acc[3]; R.h[1] = R.acc[4]; R.h[2] = R.acc[5]; R.h[3] = R.acc[0]; R.h[4] = R.acc[1]; R.h[5] = R.acc[2];
                }
              }
            END_LANES
          }
        }
        RLANES(W, R)
          R.nact = i0 + lane < ntot ? (R.f0 < 0.f ? 1 : 0) + (R.f1 < 0.f ? 2 : 0) : 0;
        END_RLANES
        const long long tk1 = TICK(); (void)tk1;
        EVENT(W, 14, (int)(tk1 - tk0));
        // (3) back on the pair's lane, its contacts' list positions known: the pair's share of the collision cost, its
        //     previous-distance record, world position and normal of the penetrating slots and their contact records
        const int nnew = warp_excl_scan(W, [](int, LaneRegs& R) { return (R.nact & 1) + (R.nact >> 1); }, [](int, LaneRegs& R, int o) { R.actmask = o; });
        LANES(W, R)
          const int i = i0 + lane;
          if (i < ntot) {
            const int e = S.nlist[i] & 0x3fff, x = m.rp[e], a = KP_A(x), b = KP_B(x);
            const bool wasfar = (S.nlist[i] >> 15) != 0, pref = ((S.nlist[i] >> 14) & 1) != 0, st = b < m.nsbox;
            const float* bpos = st ? sb_pos[b] : S.qpos + KM_NL;
            const float* bmat = st ? sb_mat[b] : S.bmat;
            const float d0 = R.f0, d1 = R.f1;
            float cc = (d0 < 0.f ? 1.f : 0.f) + (d1 < 0.f ? 1.f : 0.f);
            float* pd = io.prevd + (2 * (e / KW)) * KW + (e & (KW - 1));       // the owner's slots: pass e / KW, capsule lane e % KW
            if (!io.first) {
              const float prev0 = wasfar ? 1.f : (pref ? S.nprev[e][0] : pd[0]), prev1 = wasfar ? 1.f : (pref ? S.nprev[e][1] : pd[KW]);
              cc += fmaxf((1.f - 0.005f) * prev0 - d0, 0.f) + fmaxf((1.f - 0.005f) * prev1 - d1, 0.f);
            }
            pd[0] = d0; pd[KW] = d1;
            if (io.collision_row) { io.collision_row[KP_SLOT(x)] = d0; io.collision_row[KP_SLOT(x) + 1] = d1; }
            R.cost_c += cc;                        // (cost_c is summed over the lanes at the end of the rollout: any lane may book a pair)
            if (R.nact) {
              // world position and normal of both slots: box frame -> world
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                const float pj[3] = {R.h[6 * j], R.h[6 * j + 1], R.h[6 * j + 2]}, nj[3] = {R.h[6 * j + 3], R.h[6 * j + 4], R.h[6 * j + 5]};
                float w[3], nw[3];
                mat_vec(w, bmat, pj); add3(w, w, bpos);
                mat_vec(nw, bmat, nj);
                normalize3(nw);
                R.h[6 * j] = w[0]; R.h[6 * j + 1] = w[1]; R.h[6 * j + 2] = w[2];
                R.h[6 * j + 3] = nw[0]; R.h[6 * j + 4] = nw[1]; R.h[6 * j + 5] = nw[2];
              }
              const float invw = m.cap_invw[a] + (st ? 0.f : m.fb_invw);
              const int l1 = m.cap_link[a], l2 = st ? -1 : KM_NL;
              int o = ncbcon + R.actmask;
              if (CON && io.con_key) {
                if ((R.nact & 1) && o < KM_NC_TOT) io.con_key[o] = KP_SLOT(x);
                const int o1 = o + (R.nact & 1);
                if ((R.nact & 2) && o1 < KM_NC_TOT) io.con_key[o1] = KP_SLOT(x) + 1;
              }
              if (R.nact & 1) { put_contact<NC>(S, o, R.h, R.h + 3, nullptr, d0, invw, l1, l2); ++o; }
              if (R.nact & 2) put_contact<NC>(S, o, R.h + 6, R.h + 9, nullptr, d1, invw, l1, l2);
            }
          }
        END_LANES
        ncbcon += nnew;
        EVENT(W, 15, (int)(TICK() - tk1));
      }
      PHASE(W, 22);
    }
  }
  PHASE(W, 23);
  PHASE(W, 5);
  // free-box pairs: broad phase for all pairs at once (one lane per pair), then the cooperative
  // narrow phase only for the pairs that pass
  if (m.has_box) {
    const float* bp = S.qpos + KM_NL;
    LANES(W, R)
      for (int sl = lane; sl < 4 * m.nbpair; sl += KW) S.bstage[sl >> 2][sl & 3][3] = 1.f;
    END_LANES
    const unsigned cand = warp_ballot(W, [&](int q, LaneRegs&) {
      if (q >= m.nbpair) return false;
      if (m.bp_type[q] == KB_PLANE_BOX) {
        const float rb = sqrtf(m.fb_size[0] * m.fb_size[0] + m.fb_size[1] * m.fb_size[1] + m.fb_size[2] * m.fb_size[2]);
        float t[3]; sub3(t, bp, m.plane_pos);
        return dot3(t, m.plane_n) < rb;
      }
      // world AABBs (extent_i = sum_j |R_ij| size_j); disjoint boxes cannot have an active slot
      const int a = m.bp_a[q];
      bool overlap = true;
      // (the table's rows spelled out without SCENE: a closure that captured the views kept them in local memory)
      if constexpr (SCENE) {
        const float* ap = scene + 4 * a; const float* am = scene + 4 * KM_MAXSBOX + 12 * a; const float* as = scene + 16 * KM_MAXSBOX + 4 * a;
        for (int i = 0; i < 3; ++i) {
          const float ea = fabsf(am[3 * i]) * as[0] + fabsf(am[3 * i + 1]) * as[1] + fabsf(am[3 * i + 2]) * as[2];
          const float eb = fabsf(S.bmat[3 * i]) * m.fb_size[0] + fabsf(S.bmat[3 * i + 1]) * m.fb_size[1] + fabsf(S.bmat[3 * i + 2]) * m.fb_size[2];
          if (fabsf(bp[i] - ap[i]) > ea + eb) overlap = false;
        }
      } else {
        for (int i = 0; i < 3; ++i) {
          const float ea = fabsf(m.sb_mat[a][3 * i]) * m.sb_size[a][0] + fabsf(m.sb_mat[a][3 * i + 1]) * m.sb_size[a][1] + fabsf(m.sb_mat[a][3 * i + 2]) * m.sb_size[a][2];
          const float eb = fabsf(S.bmat[3 * i]) * m.fb_size[0] + fabsf(S.bmat[3 * i + 1]) * m.fb_size[1] + fabsf(S.bmat[3 * i + 2]) * m.fb_size[2];
          if (fabsf(bp[i] - m.sb_pos[a][i]) > ea + eb) overlap = false;
        }
      }
      return overlap;
    });
    // the loop runs over the pairs either sample of the warp has to test; a sample that does not need a
    // pair walks through it with its writes switched off, so all fences stay full-warp
#pragma unroll 1
    for (unsigned rem = warp_or_groups(W, cand); rem != 0u; rem &= rem - 1u) {
      EVENT(W, 10, 1);
      const int q = KFFS(rem) - 1;
      const bool mine = (cand >> q) & 1u;
      const int ty = m.bp_type[q], a = m.bp_a[q];
      if (ty == KB_PLANE_BOX) {
        LANES(W, R)
          if (mine && lane == q) { plane_box(m.plane_pos, m.plane_n, bp, S.bmat, m.fb_size, S.bstage[q]); copy3(S.bnrm[q], m.plane_n); }
        END_LANES
      } else {
        // one call site (the routine is large and inlined): geom1 is the static box, or the free box when it has the lower geom id
        const bool sw = ty == KB_BOX_BOX_SWAP;
        box_box_warp<NC>(W, S, mine, q, sw ? bp : sb_pos[a], sw ? S.bmat : sb_mat[a], sw ? m.fb_size : sb_size[a],
                         sw ? sb_pos[a] : bp, sw ? sb_mat[a] : S.bmat, sw ? sb_size[a] : m.fb_size);
      }
    }
  }
  LANES(W, R)
    R.actmask = __float_as_int(R.acc[7]);
    R.nact = __float_as_int(R.acc[8]);
  END_LANES
  // list positions: capsule-box contacts (written above, near-list order), then the other robot contacts
  // (lane-major), then the staged free-box contacts (pair-major)
  const int nrob = ncbcon + warp_excl_scan(W, [](int, LaneRegs& R) { return R.nact; }, [&](int, LaneRegs& R, int o) { R.off = ncbcon + o; });
  const unsigned bmask = m.has_box ? warp_ballot32(W, [&](int l) { return l < 4 * m.nbpair && S.bstage[l >> 2][l & 3][3] < 0.f; }) : 0u;
  const int ncon_all = nrob + KPOPC(bmask);
  const int ncon = ncon_all < KM_NC_TOT ? ncon_all : KM_NC_TOT;
  EVENT(W, 3, ncon); EVENT(W, 4, nrob > 0); EVENT(W, 12, warp_any_groups(W, nrob > 0));
  FLAGSTEP(W, warp_any_groups(W, nrob > 0));
  PHASE(W, 6);
  // ---- N2: full contact records for the active slots (divergent, rare for robot slots) ----
  LANES(W, R)
    if (R.nact > 0) emit_robot_contacts<NC>(m, S, lane, R.actmask, R.off);
    if (CON && io.con_key && R.nact > 0) {         // the keys of those contacts, in emit_robot_contacts' order
      int o = R.off;
#pragma unroll 1
      for (int p = m.ncbpass; p < KM_NPASS; ++p)
#pragma unroll 1
        for (int k = 0; k < 2; ++k)
          if ((R.actmask >> (2 * p + k)) & 1) { if (o < KM_NC_TOT) io.con_key[o] = KP_SLOT(m.rp[p * KW + lane]) + k; ++o; }
    }
    for (int sl = lane; sl < 32; sl += KW) {
      if (!(bmask & (1u << sl))) continue;
      const int o = nrob + KPOPC(bmask & ((1u << sl) - 1u)), q = sl >> 2;
      if (CON && io.con_key && o < KM_NC_TOT) io.con_key[o] = m.nslot_robot + sl;
      if (o < KM_NC_TOT) {
        const bool sw = m.bp_type[q] == KB_BOX_BOX_SWAP;
        const float* st = S.bstage[q][sl & 3];
        auto put = [&](float* g) {
          copy3(g, st); copy3(g + 3, S.bnrm[q]);
          make_tangents(S.bnrm[q], g + 6, g + 9);
          g[12] = st[3]; g[13] = m.fb_invw; g[14] = sw ? (float)KM_NL : -1.f; g[15] = sw ? -1.f : (float)KM_NL;
        };
        if (o < NC) put(S.cgeo[o]); else put(S.template geo<true>(o));      // every step: keep the common case in shared-memory addressing
      }
    }
  END_LANES
  if (CON && io.con_rec) {
    LANES(W, R)
#pragma unroll 1
      for (int c = lane; c < ncon; c += KW) {
        const float* g = S.template geo<true>(c);
        float* rec = io.con_rec + c * KM_CON_REC;
        rec[0] = g[12];
#pragma unroll
        for (int k = 0; k < 6; ++k) rec[1 + k] = g[k];
      }
    END_LANES
  }
  PHASE(W, 18);
  PHASE_ALIGN();
  PHASE(W, 7);
  // ---- C1: joint-limit rows ----
  LANES(W, R)
    R.nact = 0;
    if (lane < KM_NL && m.l_limited[lane]) {
      float q = S.qpos[lane], dlo = q - m.l_lo[lane], dhi = m.l_hi[lane] - q;
      float pos = fminf(dlo, dhi) - m.l_margin[lane];
      R.f0 = pos; R.f1 = dlo < dhi ? 1.f : -1.f;
      R.nact = pos < 0.f;
    }
  END_LANES
  const int nlim = warp_excl_scan(W, [](int, LaneRegs& R) { return R.nact; }, [](int, LaneRegs& R, int o) { R.off = o; });
  UNIFORM_WRITE(W) { S.ncon = ncon; S.nlim = nlim; S.nrow = nlim + 4 * ncon; if (ncon_all > KM_NC_TOT) S.flags |= 1; } END_UNIFORM_WRITE
  const int nrow = nlim + 4 * ncon;
  // No active row (the box in free fall, first steps of a rollout): qacc = qacc_smooth.  Such a sample
  // still runs through the solver below with empty loops and takes qacc_smooth at the end, which keeps
  // the fenced code and the CTA alignment points the same for every warp.
  LANES(W, R)
    if (R.nact) {
      const int r = R.off;
      S.limdof[r] = lane; S.limsign[r] = R.f1;
      float D, aref;
      row_params(m, R.f0, m.l_invw[lane], R.f1 * S.qvel[lane], D, aref);
      S.rD[r] = D; S.rAref[r] = aref;
    }
  END_LANES
  // contacts beyond the shared-memory capacity: both samples of the warp take the spill-capable instantiation
  // (same arithmetic, other addressing), so fences stay warp-uniform
  EVENT(W, 8, nrow == 0); EVENT(W, 9, !warp_all_groups(W, ncon <= NC)); EVENT(W, 13, nlim > 0);
  if (NC < KM_NC_TOT && !warp_all_groups(W, ncon <= NC)) solve_rows_spilled<NC>(m, S, ncon, nlim, nrow, WARP_BAR(W), WARP_NTHR(W));
  else solve_rows<NC, false>(W, m, S, ncon, nlim, nrow);
}

// B.8: semi-implicit Euler with eulerdamp disabled
template <int NC>
KFN void step_euler(Warp& W, const KModel& m, WarpSmemT<NC>& S) {
  LANES(W, R)
    if (lane < KM_NV) {
      float v = S.qvel[lane] + m.dt * S.qacc[lane];
      S.qvel[lane] = v;
      if (lane < KM_NL + 3) S.qpos[lane] += m.dt * v;
    }
  END_LANES
  LANES(W, R)
    if (lane == 0 && m.has_box) {
      float v[3] = {S.qvel[KM_NL + 3], S.qvel[KM_NL + 4], S.qvel[KM_NL + 5]};
      float nrm = normalize3(v), sn, cs;
      k_sincos(0.5f * m.dt * nrm, &sn, &cs);
      float qr[4] = {cs, sn * v[0], sn * v[1], sn * v[2]}, qn[4];
      float* q = S.qpos + KM_NL + 3;
      quat_mul(qn, q, qr);
      float inv = 1.f / sqrtf(qn[0] * qn[0] + qn[1] * qn[1] + qn[2] * qn[2] + qn[3] * qn[3]);
      q[0] = qn[0] * inv; q[1] = qn[1] * inv; q[2] = qn[2] * inv; q[3] = qn[3] * inv;
    }
  END_LANES
}

// ------------------------------------------------------------------------------------------ rollout + cost
struct RolloutArgs {
  int T;
  bool live;                  // false: padding warp of the last CTA (computes, writes nothing)
  const float* thetadot;      // this sample's [NL][T]
  const float* q0; const float* v0;
  const float* target_pos; const float* target_rot;     // uniform target (compute_cem tiles it, :380-381)
  float w_pos, w_rot, w_col;
  float* theta;               // [NL][T] post-step joint angles
  float* cost4;               // cost, cost_g, cost_r, cost_c
  float* eef_pos; float* eef_rot; float* collision;     // optional per-step dumps [T][3], [T][4], [T][nslot]
  float* qacc_dbg;            // optional [T][12]
  int* flags;
  float* prevd;               // scratch [2 * KM_NPASS][KW] of this sample (StepIO::prevd)
  float* ovf;                 // spill area [KM_NC_TOT - NC][KM_OVF_STRIDE] of this sample (WarpSmemT::ovf)
  // STATES only: q0 / v0 are this sample's qpos [13] / qvel [12] rows, warm0 its qacc_warmstart [12]; the state after the
  // last step goes to the *_out rows (they may be the input rows: a sample reads its rows before it writes them)
  const float* warm0;
  float* qpos_out; float* qvel_out; float* warm_out;
  // CONTACTS only: the last step's contacts and constraint forces (contact_outputs).  slot_map [nslot_robot + 4 nbpair]
  // maps a contact key to the model's contact slot; qfrc [12], ncon [1], con_slot [KM_NC_TOT], con_rec [KM_NC_TOT][KM_CON_REC]
  const int* slot_map;
  float* qfrc; int* ncon; int* con_slot; float* con_rec;
};

// The contact list and constraint forces of the last forward() (rollout_sample<.., CONTACTS>), after MJX's solver finish:
// at the accepted qacc, Jaref_r = J_r qacc - aref_r and f_r = -D_r Jaref_r where Jaref_r < 0 (SURVEY BD.10).  Reads the
// rows the last solve left in the sample's record and the keys and geometry step_forward<NC, true> put in A.con_slot /
// A.con_rec (list order); writes the contacts sorted by model slot, padded with slot -1 and zero records, and
// qfrc_constraint = sum_r J_r^T f_r, summed over the limit rows, then the contacts in slot order (the row order of
// oracle/mjstep.c make_constraint).  Per contact, force = (sum f, mu (f0 - f1), mu (f2 - f3)) of its four pyramid rows
// Jn + mu Jt1, Jn - mu Jt1, Jn + mu Jt2, Jn - mu Jt2 (mju_decodePyramid).
template <int NC>
KFN void contact_outputs(Warp& W, const KModel& m, WarpSmemT<NC>& S, const RolloutArgs& A) {
  const int ncon = A.live ? S.ncon : 0, nlim = S.nlim;       // (a padding sample wrote no keys)
  int* inv = reinterpret_cast<int*>(&S.H[0][0]);      // list position of the k-th contact in slot order (H is dead here)
  // (1) per contact: the force sums of its rows, which replace the contact record's dead fields with the geometry kept in
  //     A.con_rec (g[0..2] force sums, g[3..5] normal, g[6..8] position, g[13] model slot; g[12] dist and the links stay)
  LANES(W, R)
#pragma unroll 1
    for (int c = lane; c < ncon; c += KW) {
      float* g = S.template geo<true>(c);
      const float* J = S.template jac<true>(c);
      const int blk = contact_blocks(g), o = (blk & 1) ? 0 : KM_NL, nd = blk == 3 ? KM_NV : KM_NL;
      float dn = 0.f, d1 = 0.f, d2 = 0.f;
#pragma unroll 1
      for (int d = o; d < o + nd; ++d) { dn += J[d] * S.qacc[d]; d1 += J[12 + d] * S.qacc[d]; d2 += J[24 + d] * S.qacc[d]; }
      float f[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int r = nlim + 4 * c + q;
        const float dt = q < 2 ? d1 : d2;
        const float ja = ((q & 1) ? dn - dt : dn + dt) - S.template Aref<true>(r, nlim);
        f[q] = ja < 0.f ? -S.template D<true>(r, nlim) * ja : 0.f;
      }
      const float* rec = A.con_rec + c * KM_CON_REC;
      const int slot = A.slot_map[A.con_slot[c]];
      g[0] = f[0] + f[1] + f[2] + f[3]; g[1] = f[0] - f[1]; g[2] = f[2] - f[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) { g[3 + k] = rec[4 + k]; g[6 + k] = rec[1 + k]; }
      g[13] = __int_as_float(slot);
    }
  END_LANES
  // (2) ranks by model slot (the slots of a sample's contacts are distinct)
  LANES(W, R)
#pragma unroll 1
    for (int c = lane; c < ncon; c += KW) {
      const int s = __float_as_int(S.template geo<true>(c)[13]);
      int rank = 0;
#pragma unroll 1
      for (int c2 = 0; c2 < ncon; ++c2) rank += __float_as_int(S.template geo<true>(c2)[13]) < s ? 1 : 0;
      inv[rank] = c;
    }
  END_LANES
  // (3) the sorted outputs and qfrc_constraint
  LANES(W, R)
    if (A.live) {
#pragma unroll 1
      for (int k = lane; k < KM_NC_TOT; k += KW) {
        float* rec = A.con_rec + k * KM_CON_REC;
        if (k < ncon) {
          const float* g = S.template geo<true>(inv[k]);
          A.con_slot[k] = __float_as_int(g[13]);
          rec[0] = g[12];
          rec[1] = g[6]; rec[2] = g[7]; rec[3] = g[8];
          rec[4] = g[3]; rec[5] = g[4]; rec[6] = g[5];
          rec[7] = g[0]; rec[8] = m.mu * g[1]; rec[9] = m.mu * g[2];
          rec[10] = 0.f; rec[11] = 0.f;
        } else {
          A.con_slot[k] = -1;
#pragma unroll
          for (int i = 0; i < KM_CON_REC; ++i) rec[i] = 0.f;
        }
      }
      if (lane < KM_NV) {
        float fc = 0.f;
#pragma unroll 1
        for (int r = 0; r < nlim; ++r) {
          if (S.limdof[r] != lane) continue;
          const float ja = S.limsign[r] * S.qacc[lane] - S.rAref[r];
          if (ja < 0.f) fc += S.limsign[r] * (-S.rD[r] * ja);
        }
        const int need = lane < KM_NL ? 1 : 2;
#pragma unroll 1
        for (int k = 0; k < ncon; ++k) {
          const float* g = S.template geo<true>(inv[k]);
          if (!(contact_blocks(g) & need)) continue;        // the Jacobian only exists in the blocks the contact touches
          const float* J = S.template jac<true>(inv[k]);
          fc += J[lane] * g[0] + J[12 + lane] * g[1] + J[24 + lane] * g[2];
        }
        A.qfrc[lane] = fc;
      }
      if (lane == 0) *A.ncon = ncon;
    }
  END_LANES
}

// STATES = false: a planner rollout from the KModel snapshot (arm state q0 / v0, shared by all samples) with its cost.
// STATES = true: the same steps from the sample's own state rows, which it writes back after the last step; thetadot
// may be null with T = 1 (the sample keeps its own qvel[:6], a plain mjx.step), theta is optional, no cost, no target.
// CONTACTS (with STATES): also the contacts and constraint forces of the last step (contact_outputs).
// SCENE: the static boxes from the sample's scene record `scene` (KM_SCENE_FLOATS) and, without STATES, the snapshot
// from the start record `start` (qpos0 | warm0 | qvel0, KM_START_FLOATS) instead of the table's.
template <int NC, bool STATES = false, bool CONTACTS = false, bool SCENE = false>
KFN void rollout_sample(Warp& W, const KModel& m, WarpSmemT<NC>& S, const RolloutArgs& A, const float* scene = nullptr,
                        const float* start = nullptr) {
  const float* qpos0 = SCENE && !STATES ? start : m.qpos0;
  const float* warm0 = SCENE && !STATES ? start + 16 : m.warm0;
  const float* qvel0 = SCENE && !STATES ? start + 28 : m.qvel0;
  LANES(W, R)
    if (STATES) {
      if (lane < KM_NQ) S.qpos[lane] = A.q0[lane];
      if (lane < KM_NV) { S.qvel[lane] = A.v0[lane]; S.warm[lane] = A.warm0[lane]; }
    } else {
      if (lane < KM_NQ) S.qpos[lane] = lane < KM_NL ? A.q0[lane] : qpos0[lane];
      if (lane < KM_NV) { S.qvel[lane] = lane < KM_NL ? A.v0[lane] : qvel0[lane]; S.warm[lane] = warm0[lane]; }
    }
    R.tri = tri_entries(lane);
    if (lane == 0) { S.flags = 0; S.ovf = A.ovf; }
    R.cost_c = 0.f;
    R.farprev = 0;
    R.td = lane < KM_NL ? ((!STATES || A.thetadot) ? A.thetadot[lane * A.T] : A.v0[lane]) : 0.f;
  END_LANES
  const float tp[3] = {STATES ? 0.f : A.target_pos[0], STATES ? 0.f : A.target_pos[1], STATES ? 0.f : A.target_pos[2]};   // read once: the step loop only touches registers for the goal terms
  float tq[4] = {STATES ? 1.f : A.target_rot[0], STATES ? 0.f : A.target_rot[1], STATES ? 0.f : A.target_rot[2], STATES ? 0.f : A.target_rot[3]};
  {
    float inv = 1.f / sqrtf(tq[0] * tq[0] + tq[1] * tq[1] + tq[2] * tq[2] + tq[3] * tq[3]);
    tq[0] *= inv; tq[1] *= inv; tq[2] *= inv; tq[3] *= inv;
  }
  float cost_g = 0.f, cost_r = 0.f;
#pragma unroll 1
  for (int t = 0; t < A.T; ++t) {
    PHASE(W, 13);
    STEP_ALIGN();
    PHASE(W, 0);
    LANES(W, R)
      if (lane < KM_NL) {
        S.qvel[lane] = R.td;                                             // mjx_planner.py:254
        if (t + 1 < A.T) R.td = A.thetadot[lane * A.T + t + 1];          // consumed next step: latency hidden
      }
    END_LANES
    StepIO io;
    io.first = t == 0;
    io.collision_row = (A.collision && A.live) ? A.collision + (size_t)t * m.nslot_robot : nullptr;
    io.prevd = A.prevd;
    if (CONTACTS) {
      const bool last = A.live && t + 1 == A.T;
      io.con_key = last ? A.con_slot : nullptr;
      io.con_rec = last ? A.con_rec : nullptr;
    }
    step_forward<NC, CONTACTS, SCENE>(W, m, S, io, scene);
    PHASE(W, 12);
    // pre-step observations (mjx_planner.py:259-261) and running cost (:277-285)
    {
      float tcp[3], tv[3], eq[4];
      USYNC();
      mat_vec(tv, S.lmat[KM_NL - 1], m.tcp_pos); add3(tcp, S.lpos[KM_NL - 1], tv);
      quat_mul(eq, S.lquat[KM_NL - 1], m.hande_quat);
      float d[3]; sub3(d, tcp, tp);
      cost_g += sqrtf(dot3(d, d));
      float inv = 1.f / sqrtf(eq[0] * eq[0] + eq[1] * eq[1] + eq[2] * eq[2] + eq[3] * eq[3]);
      float dp = fabsf((eq[0] * tq[0] + eq[1] * tq[1] + eq[2] * tq[2] + eq[3] * tq[3]) * inv);
      dp = fminf(fmaxf(dp, -1.f), 1.f);
      cost_r += 2.f * acosf(dp);
      if (A.live && (A.eef_pos || A.eef_rot || A.qacc_dbg)) {
        LANES(W, R)
          if (A.eef_pos && lane < 3) A.eef_pos[t * 3 + lane] = lane == 0 ? tcp[0] : (lane == 1 ? tcp[1] : tcp[2]);
          if (A.eef_rot && lane < 4) A.eef_rot[t * 4 + lane] = lane == 0 ? eq[0] : (lane == 1 ? eq[1] : (lane == 2 ? eq[2] : eq[3]));
          if (A.qacc_dbg && lane < KM_NV) A.qacc_dbg[t * KM_NV + lane] = S.qacc[lane];
        END_LANES
      }
    }
    step_euler<NC>(W, m, S);
    LANES(W, R)
      if (A.live && lane < KM_NL && (!STATES || A.theta)) A.theta[lane * A.T + t] = S.qpos[lane];
    END_LANES
    PHASE(W, 12);
    STEPEND(W);
  }
  if (CONTACTS) contact_outputs<NC>(W, m, S, A);           // (step_euler changes nothing it reads)
  if (STATES) {
    LANES(W, R)
      if (A.live) {
        if (lane < KM_NQ) A.qpos_out[lane] = S.qpos[lane];
        if (lane < KM_NV) { A.qvel_out[lane] = S.qvel[lane]; A.warm_out[lane] = S.warm[lane]; }
        if (lane == 0 && A.flags) *A.flags = S.flags;
      }
    END_LANES
    return;
  }
  const float cost_c = warp_sum(W, [](int, LaneRegs& R) { return R.cost_c; });
  LANES(W, R)
    if (lane == 0 && A.live) {
      A.cost4[0] = A.w_pos * cost_g + A.w_rot * cost_r + A.w_col * cost_c;
      A.cost4[1] = cost_g; A.cost4[2] = cost_r; A.cost4[3] = cost_c;
      if (A.flags) *A.flags = S.flags;
    }
  END_LANES
}
