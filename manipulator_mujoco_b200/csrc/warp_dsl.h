// warp_dsl.h -- a tiny "one lane group = one sample" programming layer.
//
// A sample is owned by a group of KW = 16 lanes, two samples per warp.  The rollout core (rollout_core.h)
// is written once against these macros and compiled twice:
//   * by nvcc for sm_100a, where a LANES block is the body executed by each of the KW lanes of the
//     group, per-lane state lives in registers, collectives are shuffles / ballots restricted to the
//     group (member mask = the group's lanes, width = KW) and every block is fenced by
//     __syncwarp(group mask).  The two halves of a warp run the same instruction stream on
//     two samples: "uniform" scalar code (small dense solves, the serial joint chain, line-search control)
//     is issued once for both, and phases that only have 6..16 work items fill the warp twice as well.
//     Two flavours of every fence / collective exist.  The plain ones (LANES, UNIFORM_WRITE, warp_sum ...)
//     use the constant full-warp member mask and may only appear where both groups of the warp are on
//     the same path ("converged" code: the core keeps its sample-dependent control flow warp-uniform
//     there, e.g. the line search runs until both samples are done).  The D-flavours (DLANES,
//     DUNIFORM_WRITE, warp_sum<true> ...) use the group's own mask and are for the few regions where the
//     two samples may take different paths (free-box narrow phase, coupled 12x12 solve); a variable
//     member mask costs a MATCH/vote sequence per fence, which is why it is not used everywhere.
//     A divergent region ends with REGROUP(), a full-warp fence;
//   * by g++ with -DCEMK_EMU (tests/emu, no-GPU unit tests only), where a LANES block is a plain
//     `for (lane = 0..KW-1)` loop over an array of per-lane register structs.  This is a debugging
//     aid for kernel logic in a container without a GPU; it is never used by the product path.
//
// Rules the core follows so both builds mean the same thing:
//   1. inside one LANES block a lane reads only shared scratch written in *earlier* blocks (or by
//      itself) and writes only locations no other lane touches in that block;
//   2. code outside LANES blocks is group-uniform (every lane of the group computes the same scalars);
//      shared scratch is written there only through UNIFORM_WRITE, which is fenced on both sides.
#pragma once
#include <math.h>

#define KW 16
#define KW_FULL 0xffffu

#ifdef CEMK_EMU
#include <cstring>
#define KFN static inline
#define KMEM inline
#define KNOINLINE static
#define STEP_ALIGN()
#define PHASE_ALIGN()
#ifdef CEMK_EMU_RACE
// Race-checking emulation (tests/test_emu_race.py): every lane of a LANES block runs against the scratch as it was when
// the block started (plus its own writes); the lanes' writes are merged when the block ends.  That is exactly what rule 1
// below promises the GPU build, so a kernel that obeys the rule computes bit-identical results in this mode and in the
// plain lane-after-lane emulation, while a block in which a lane consumes another lane's write of the same block (a
// missing fence) gives that lane the stale value here and the results differ.  Two lanes writing different values to
// the same scratch byte in one block are counted directly (RaceState::waw).
struct RaceState {
  struct Region { unsigned char* p; size_t n; } reg[8];
  int nreg = 0, open = -1, line = 0;
  long long waw = 0, blocks = 0;
  int first_line = 0, first_word = 0, first_lanes = 0;      // where the first write-write conflict was seen (source line of the block)
  size_t total = 0;
  unsigned char* snap = nullptr; unsigned char* pend = nullptr; signed char* owner = nullptr;
  void add(void* p, size_t n) { reg[nreg].p = (unsigned char*)p; reg[nreg].n = n & ~size_t(3); total += reg[nreg].n; ++nreg; }
  void gather(unsigned char* dst) { size_t o = 0; for (int i = 0; i < nreg; ++i) { std::memcpy(dst + o, reg[i].p, reg[i].n); o += reg[i].n; } }
  void scatter(const unsigned char* src) { size_t o = 0; for (int i = 0; i < nreg; ++i) { std::memcpy(reg[i].p, src + o, reg[i].n); o += reg[i].n; } }
  void begin_block() {
    if (!snap) { snap = new unsigned char[total]; pend = new unsigned char[total]; owner = new signed char[total]; }
    gather(snap); std::memcpy(pend, snap, total); std::memset(owner, -1, total); open = -1; ++blocks;
  }
  void close_lane() {                          // byte granularity: lanes may own different bytes of one word (S.nlist)
    if (open < 0) return;
    size_t o = 0;
    for (int i = 0; i < nreg; ++i) {
      for (size_t w = 0; w < reg[i].n; ++w, ++o) {
        const unsigned char v = reg[i].p[w];
        if (v == snap[o]) continue;            // not written (or rewritten with the old value)
        if (owner[o] >= 0 && owner[o] != open && v != pend[o]) {
          if (!waw) { first_line = line; first_word = (int)(o / 4); first_lanes = owner[o] * 100 + open; }
          ++waw;
        }
        owner[o] = (signed char)open;
        pend[o] = v;
      }
    }
    open = -1;
  }
  void begin_lane(int lane) { close_lane(); scatter(snap); open = lane; }
  void end_block() { close_lane(); scatter(pend); }
};
struct RaceBlock {
  RaceState* rs;
  RaceBlock(void* p, int line) : rs((RaceState*)p) { if (rs) { rs->line = line; rs->begin_block(); } }
  void lane(int l) { if (rs) rs->begin_lane(l); }
  ~RaceBlock() { if (rs) rs->end_block(); }
};
#define LANES(W, R) { RaceBlock race_blk_((W).race, __LINE__); for (int lane = 0; lane < KW; ++lane) { race_blk_.lane(lane); auto& R = (W).regs[lane]; (void)R;
#define END_LANES } }
#define DLANES(W, R) LANES(W, R)
#define END_DLANES } }
#else
#define LANES(W, R) for (int lane = 0; lane < KW; ++lane) { auto& R = (W).regs[lane]; (void)R;
#define END_LANES }
#define DLANES(W, R) LANES(W, R)
#define END_DLANES }
#endif
#define RLANES(W, R) for (int lane = 0; lane < KW; ++lane) { auto& R = (W).regs[lane]; (void)R;
#define END_RLANES }
#define UNIFORM_WRITE(W) if (true)
#define END_UNIFORM_WRITE
#define DUNIFORM_WRITE(W) if (true)
#define END_DUNIFORM_WRITE
#define USYNC()
#define REGROUP()
#define KRSQRT(x) (1.0f / sqrtf(x))
#define WARP_BAR(W) 0
#define WARP_NTHR(W) 0
#define KPOPC(x) __builtin_popcount(x)
#define KFFS(x) __builtin_ffs((int)(x))
static inline float __int_as_float(int i) { float f; std::memcpy(&f, &i, 4); return f; }
static inline int __float_as_int(float f) { int i; std::memcpy(&i, &f, 4); return i; }
#else
#define KFN __device__ __forceinline__
#define KMEM __device__ __forceinline__
#define KNOINLINE __device__ __noinline__
// Keep the live warps of a CTA on the same code (instruction-cache locality): named barrier 1 with the
// live thread count of this CTA (a CTA may run fewer samples than its launch width, see
// cemk_rollout_cost).  The two groups of a warp re-converge first (bar.sync is a per-warp instruction).
#define CTA_ALIGN(W) do { __syncwarp(); asm volatile("bar.sync %0, %1;" :: "r"((W).bar), "r"((W).nthr) : "memory"); } while (0)
// STEP_ALIGN: once per env-step.  PHASE_ALIGN: inside a step, only at points every group reaches (before the
// constraint rows and before the line search)
#define STEP_ALIGN() CTA_ALIGN(W)
#define PHASE_ALIGN() CTA_ALIGN(W)
#define LANES(W, R) { __syncwarp(); const int lane = (W).lane; auto& R = (W).regs; (void)R;
#define END_LANES } __syncwarp();
#define DLANES(W, R) { __syncwarp((W).mask); const int lane = (W).lane; auto& R = (W).regs; (void)R;
#define END_DLANES } __syncwarp((W).mask);
// register-only lane block: touches no shared scratch, so no fences
#define RLANES(W, R) { const int lane = (W).lane; auto& R = (W).regs; (void)R; (void)lane;
#define END_RLANES }
#define UNIFORM_WRITE(W) __syncwarp(); if ((W).lane == 0)
#define END_UNIFORM_WRITE __syncwarp();
#define DUNIFORM_WRITE(W) __syncwarp((W).mask); if ((W).lane == 0)
#define END_DUNIFORM_WRITE __syncwarp((W).mask);
#define USYNC() __syncwarp()
#define REGROUP() __syncwarp()
#define KRSQRT(x) rsqrtf(x)
#define WARP_BAR(W) ((W).bar)
#define WARP_NTHR(W) ((W).nthr)
#define KPOPC(x) __popc(x)
#define KFFS(x) __ffs((int)(x))
#endif

// member mask of a collective: the group's own lanes in divergent regions, the whole warp otherwise
#define KMASK(w) (DIV ? (w).mask : 0xffffffffu)

#ifdef CEMK_EMU
inline thread_local void* g_emu_race = nullptr;      // RaceState of the sample being emulated (race-checking build), for cold_warp()
#endif

template <class LR>
struct WarpCtx {
#ifdef CEMK_EMU
  LR regs[KW];
  void* race;        // RaceState* of the race-checking emulation (null otherwise)
#else
  LR regs;
  int lane;          // lane within the group, 0..KW-1
  int shift;         // first lane of the group within the warp (0 or 16)
  unsigned mask;     // member mask of the group
  int nthr;          // threads of the CTA's live warps (barrier width of CTA_ALIGN)
  int bar;           // named barrier of CTA_ALIGN (1)
#ifdef CEMK_PHASE_TIMING
  long long t0; int phase; long long ph[24];
  long long phs[24], phc[24]; int stepflag, nflag;   // this step's clocks; clocks of the steps with stepflag set (conditional profile)
  int ev[24];        // event counters (tools/phase_timing.py)
#endif
#endif
};

// Debug build only (-DCEMK_PHASE_TIMING): per-phase SM-clock accounting of one group's step, summed
// into a global table by the kernel wrapper (tools/phase_timing.py).  No-op otherwise.
#if !defined(CEMK_EMU) && defined(CEMK_PHASE_TIMING)
#define PHASE(W, id) do { long long now_ = clock64(); (W).ph[(W).phase] += now_ - (W).t0; (W).phs[(W).phase] += now_ - (W).t0; (W).t0 = now_; (W).phase = (id); } while (0)
// conditional profile: FLAGSTEP marks the current step, STEPEND books the step's clocks under the flag
#define FLAGSTEP(W, cond) do { if (cond) (W).stepflag = 1; } while (0)
#define STEPEND(W) do { for (int i_ = 0; i_ < 24; ++i_) { if ((W).stepflag) (W).phc[i_] += (W).phs[i_]; (W).phs[i_] = 0; } (W).nflag += (W).stepflag; (W).stepflag = 0; } while (0)
#define EVENT(W, id, n) do { (W).ev[(id)] += (n); } while (0)
#define TICK() clock64()
#else
#define PHASE(W, id) do { } while (0)
#define EVENT(W, id, n) do { } while (0)
#define TICK() 0LL
#define FLAGSTEP(W, cond) do { } while (0)
#define STEPEND(W) do { } while (0)
#endif

// sum over the group's lanes of f(lane, regs); result is group-uniform
template <bool DIV = false, class W, class F>
KFN float warp_sum(W& w, F f) {
#ifdef CEMK_EMU
  float s = 0.f;
  for (int l = 0; l < KW; ++l) s += f(l, w.regs[l]);
  return s;
#else
  float v = f(w.lane, w.regs);
#pragma unroll
  for (int o = KW / 2; o; o >>= 1) v += __shfl_xor_sync(KMASK(w), v, o, KW);
  return v;
#endif
}

// exclusive prefix sum of small non-negative ints; set(lane, regs, offset) receives each lane's
// offset; returns the group total
template <bool DIV = false, class W, class G, class S>
KFN int warp_excl_scan(W& w, G get, S set) {
#ifdef CEMK_EMU
  int run = 0;
  for (int l = 0; l < KW; ++l) { int v = get(l, w.regs[l]); set(l, w.regs[l], run); run += v; }
  return run;
#else
  int v = get(w.lane, w.regs), inc = v;
#pragma unroll
  for (int o = 1; o < KW; o <<= 1) { int t = __shfl_up_sync(KMASK(w), inc, o, KW); if (w.lane >= o) inc += t; }
  set(w.lane, w.regs, inc - v);
  return __shfl_sync(KMASK(w), inc, KW - 1, KW);
#endif
}

// value of f(src, regs[src]) broadcast to every lane of the group
template <bool DIV = false, class W, class F>
KFN float warp_bcast(W& w, int src, F f) {
#ifdef CEMK_EMU
  return f(src, w.regs[src]);
#else
  return __shfl_sync(KMASK(w), f(w.lane, w.regs), src, KW);
#endif
}

// lane index of the maximum of f(lane, regs) over the group; ties -> lowest lane ("first max");
// lanes whose value is NaN never win against a number
template <bool DIV = false, class W, class F>
KFN int warp_argmax_first(W& w, F f) {
#ifdef CEMK_EMU
  int best = 0; float bv = f(0, w.regs[0]);
  for (int l = 1; l < KW; ++l) { float v = f(l, w.regs[l]); if (v > bv || (bv != bv && v == v)) { bv = v; best = l; } }
  return best;
#else
  float v = f(w.lane, w.regs); int idx = w.lane;
#pragma unroll
  for (int o = KW / 2; o; o >>= 1) {
    const float ov = __shfl_xor_sync(KMASK(w), v, o, KW);
    const int oi = __shfl_xor_sync(KMASK(w), idx, o, KW);
    if (ov > v || (ov == v && oi < idx) || (v != v && ov == ov)) { v = ov; idx = oi; }
  }
  return idx;
#endif
}

// per-lane-source shuffle: lane l receives get(src(l), regs[src(l)]) through set(l, regs[l], value)
template <bool DIV = false, class W, class G, class SRC, class SET>
KFN void warp_shfl_each(W& w, G get, SRC src, SET set) {
#ifdef CEMK_EMU
  float vals[KW];
  for (int l = 0; l < KW; ++l) vals[l] = get(l, w.regs[l]);
  for (int l = 0; l < KW; ++l) set(l, w.regs[l], vals[src(l) & (KW - 1)]);
#else
  const float v = __shfl_sync(KMASK(w), get(w.lane, w.regs), src(w.lane), KW);
  set(w.lane, w.regs, v);
#endif
}

// bit l of the result is set iff pred(l, regs[l]) holds, l = 0..KW-1
template <bool DIV = false, class W, class F>
KFN unsigned warp_ballot(W& w, F pred) {
#ifdef CEMK_EMU
  unsigned m = 0;
  for (int l = 0; l < KW; ++l) if (pred(l, w.regs[l])) m |= 1u << l;
  return m;
#else
  return (__ballot_sync(KMASK(w), pred(w.lane, w.regs)) >> w.shift) & KW_FULL;
#endif
}
// ballot over 32 items: bit i of the result is pred(i), evaluated by lane i % KW
template <bool DIV = false, class W, class F>
KFN unsigned warp_ballot32(W& w, F pred) {
#ifdef CEMK_EMU
  unsigned m = 0;
  for (int i = 0; i < 32; ++i) if (pred(i)) m |= 1u << i;
  return m;
#else
  unsigned m = 0;
#pragma unroll
  for (int q = 0; q < 32 / KW; ++q) {
    const int i = q * KW + w.lane;
    m |= ((__ballot_sync(KMASK(w), pred(i)) >> w.shift) & KW_FULL) << (q * KW);
  }
  return m;
#endif
}
// warp_argmax_first restricted to lanes 0..7 (three exchange rounds); other lanes' values are ignored
template <bool DIV = false, class W, class F>
KFN int warp_argmax_first8(W& w, F f) {
#ifdef CEMK_EMU
  int best = 0; float bv = f(0, w.regs[0]);
  for (int l = 1; l < 8; ++l) { float v = f(l, w.regs[l]); if (v > bv || (bv != bv && v == v)) { bv = v; best = l; } }
  return best;
#else
  float v = f(w.lane, w.regs); int idx = w.lane;
#pragma unroll
  for (int o = 4; o; o >>= 1) {
    const float ov = __shfl_xor_sync(KMASK(w), v, o, KW);
    const int oi = __shfl_xor_sync(KMASK(w), idx, o, KW);
    if (ov > v || (ov == v && oi < idx) || (v != v && ov == ov)) { v = ov; idx = oi; }
  }
  return __shfl_sync(KMASK(w), idx, 0, KW);
#endif
}

#ifndef CEMK_EMU
// one round of the transposed butterfly: a lane carrying N values keeps ceil(N/2) of them (the low ones
// if its `bit` is clear, the high ones otherwise) and adds the partner's copy of the same values
template <int N, bool DIV, class W>
KFN void fold_round(W& w, const float* in, float* out, bool hi, int xor_lanes) {
  constexpr int H = (N + 1) / 2;
#pragma unroll
  for (int k = 0; k < H; ++k) {
    const float upper = H + k < N ? in[H + k] : 0.f;
    const float mine = hi ? upper : in[k];
    const float send = hi ? in[k] : upper;
    out[k] = mine + __shfl_xor_sync(KMASK(w), send, xor_lanes, KW);
  }
}
#endif

// Sums of nine per-lane values (regs.acc[0..8]) over the group, all nine results to every lane.
// GPU: transposed butterfly -- each exchange round halves the number of values a lane still carries
// (9 -> 5 -> 3 -> 2 -> 1), then nine broadcasts: 20 shuffles for 16 lanes (36 if summed one by one).
template <bool DIV = false, class W>
KFN void warp_sum9(W& w, float* out) {
#ifdef CEMK_EMU
  for (int k = 0; k < 9; ++k) { float s = 0.f; for (int l = 0; l < KW; ++l) s += w.regs[l].acc[k]; out[k] = s; }
#else
  const int lane = w.lane;
  float v[9], u[5], t[3], s2[2], r[1];
#pragma unroll
  for (int k = 0; k < 9; ++k) v[k] = w.regs.acc[k];
  fold_round<9, DIV>(w, v, u, lane & 8, 8);
  fold_round<5, DIV>(w, u, t, lane & 4, 4);
  fold_round<3, DIV>(w, t, s2, lane & 2, 2);
  fold_round<2, DIV>(w, s2, r, lane & 1, 1);
  // lane holding the total of value k: bit 3 adds 5, bit 2 adds 3, bit 1 adds 2, bit 0 adds 1 to the index
  out[0] = __shfl_sync(KMASK(w), r[0], 0, KW); out[1] = __shfl_sync(KMASK(w), r[0], 1, KW);  out[2] = __shfl_sync(KMASK(w), r[0], 2, KW);
  out[3] = __shfl_sync(KMASK(w), r[0], 4, KW); out[4] = __shfl_sync(KMASK(w), r[0], 5, KW);  out[5] = __shfl_sync(KMASK(w), r[0], 8, KW);
  out[6] = __shfl_sync(KMASK(w), r[0], 9, KW); out[7] = __shfl_sync(KMASK(w), r[0], 10, KW); out[8] = __shfl_sync(KMASK(w), r[0], 12, KW);
#endif
}

// true iff pred holds for every sample of the warp (both lane groups); converged code only
template <class W>
KFN bool warp_all_groups(W& w, bool pred) {
#ifdef CEMK_EMU
  (void)w;
  return pred;
#else
  (void)w;
  return __all_sync(0xffffffffu, pred);
#endif
}

// true iff pred holds for some sample of the warp; converged code only
template <class W>
KFN bool warp_any_groups(W& w, bool pred) {
#ifdef CEMK_EMU
  (void)w;
  return pred;
#else
  (void)w;
  return __any_sync(0xffffffffu, pred);
#endif
}
// bitwise OR of a group-uniform mask over the samples of the warp; converged code only
template <class W>
KFN unsigned warp_or_groups(W& w, unsigned m) {
#ifdef CEMK_EMU
  (void)w;
  return m;
#else
  (void)w;
  return __reduce_or_sync(0xffffffffu, m);
#endif
}

