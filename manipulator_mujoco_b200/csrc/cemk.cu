// cemk.cu -- sm_100a kernels + the C ABI declared in include/cemk.h.
//
// Kernels (one per stage of cem_planner.cem_iter, reference mjx_planner.py:337-362):
//   k_jax_normal / k_chol66 | k_chol_wide / k_sample   compute_xi_samples  (:313-316)
//   k_project                compute_projection_filter + A_thetadot @ xi   (:181-249, :348)
//   k_rollout                vmap(scan(mjx.step)) + compute_cost_batch     (:251-303)   <- hot kernel
//   k_rollout<.., STATES>    vmap(mjx.step) over per-environment states, chained T steps (cemk_step_states)
//   k_cost_batch             compute_cost_batch on materialised trajectories (:277-303)
//   k_rank_select (n <= 8192) | k_make_keys / k_bitonic* / k_gather_sorted    compute_ellite_samples   (:306-310)
//   k_merge_lists            the same selection over the per-rank sorted lists of several GPUs
//   k_mean_cov | k_mc_partial[_wide] + k_mc_finish (k >= 1024)             compute_mean_cov (:326-335)
//   k_tick_record            what compute_cem keeps of an iteration        (:390-404)
// The rollout core lives in rollout_core.h (shared with the CPU emulation used by the no-GPU tests).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/cemk.h"
#include "rollout_core.h"

// Bernstein order n (mjx_planner.py:40 hard-codes 10; SURVEY 8 f.4 asks for order n): ncoef = n + 1 coefficients per DOF,
// nvar = ndof ncoef decision variables, chosen per handle by cemk_set_dof / cemk_set_order (default 6 DOF x 11 = 66).  The
// planner algebra runs at any ndof <= MAXDOF; the rollout models the 6-DOF (KM_NL) arm only.
#define MINCOEF 4
#define MAXCOEF 16
#define MAXDOF 12
#define MAXVAR (MAXDOF * MAXCOEF)      // 192
#ifndef ROLLOUT_WARPS
#define ROLLOUT_WARPS 14      // warps per CTA (28 samples with two samples per warp: all the shared memory of an SM); they
                              // step in lockstep (STEP_ALIGN) to share the instruction cache
#endif
#ifndef ROLLOUT_SETS
#define ROLLOUT_SETS 1        // independent lockstep sets per CTA (named barriers 1 .. ROLLOUT_SETS)
#endif
#ifndef ROLLOUT_MINB
#define ROLLOUT_MINB 1
#endif

static thread_local char g_err[256] = "";
static int set_err(int code, const char* msg) { snprintf(g_err, sizeof g_err, "%s", msg); return code; }
static int cuda_err(cudaError_t e, const char* where) {
  snprintf(g_err, sizeof g_err, "%s: %s", where, cudaGetErrorString(e));
  return CEMK_ERR_CUDA;
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return cuda_err(e_, #call); } while (0)

// Every entry point runs on its handle's device and leaves the caller's current device as it found it (a planner on
// cuda:1 next to one on cuda:0, or torch code that never set a device, must not notice the library).
struct DevGuard {
  int prev = -1; bool switched = false;
  explicit DevGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DevGuard() { if (switched) cudaSetDevice(prev); }
};

struct cemk_handle {
  int device;
  KModel* d_model;
  int ndof, ncoef, nvar;           // DOF of the planner algebra, Bernstein coefficients per DOF, decision variables (ndof ncoef)
  int T;
  float* d_G;      // [3][T][11]
  float* d_K;      // Kpp[ncoef^2] Kpe[ncoef*5] bounds[3]
  long long launches;
  int* d_flags; int flags_cap; int num_sms;
  float* d_prevd; int prevd_cap;   // previous-step slot distances of every sample (rollout scratch, stays in L2)
  float* d_ovf;                    // contact spill area of every sample (same capacity as d_prevd)
  int force_rerun;               // debug option: recompute every sample with the all-in-shared-memory instantiation
  int cta_samples;                 // debug option "cta_samples": fixed number of samples per CTA (0 = see cemk_rollout_cost)
  float* d_mc;                     // block sums of the blocked mean / covariance update (k_mc_partial -> k_mc_finish)
};

// ---------------------------------------------------------------------------------------------- rollout
#ifdef CEMK_PHASE_TIMING
__device__ unsigned long long g_phase[24];
__device__ unsigned long long g_event[24];
__device__ unsigned long long g_phase_cond[25];
#endif
struct RolloutBatch {
  int B, T;
  const float* thetadot; const float* q0; const float* v0; const float* target_pos; const float* target_rot;
  float w_pos, w_rot, w_col;
  float* theta; float* cost4; float* eef_pos; float* eef_rot; float* collision; float* qacc; int* flags;
  float* prevd;                  // [B][2 * KM_NPASS][KW] previous-step slot distances (library scratch)
  float* ovf;                    // [B][KM_NC_TOT - KM_NC_FAST][KM_OVF_STRIDE] contact spill area (library scratch)
  // CTA -> samples: the first n_hi CTAs run w_hi samples each, the others w_lo (both <= the launch width);
  // warps beyond a CTA's share exit at once
  int n_hi, w_hi, w_lo;
  // cemk_step_states (STATES): q0 / v0 are then qpos [B][13] / qvel [B][12], and warm [B][12] is the third state input
  const float* warm;
  float* qpos_out; float* qvel_out; float* warm_out;
};

// NC = contacts of a sample kept in shared memory (the rest, up to KM_NC_TOT, in the global spill area),
// WARPS = warps per CTA; a warp carries 32 / KW samples (one per lane group, warp_dsl.h).  The fast
// instantiation (NC = KM_NC_FAST) is the product path.  ONLY_FLAGGED is the debug instantiation behind
// cemk_set_option("force_rerun"): NC = 48 (no spill area), one warp per CTA, samples whose flag bit 0 is set.
// STATES: every sample steps from its own state rows and writes its final state (cemk_step_states, rollout_sample).
#define GPW (32 / KW)                                     // lane groups (samples) per warp
template <int NC, int WARPS, bool ONLY_FLAGGED, bool STATES = false>
__global__ void __launch_bounds__(WARPS * 32, ROLLOUT_MINB) k_rollout(const KModel* __restrict__ gm, RolloutBatch a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  KModel* sm = reinterpret_cast<KModel*>(smem_raw);
  WarpSmemT<NC>* ws = reinterpret_cast<WarpSmemT<NC>*>(smem_raw + ((sizeof(KModel) + 15) & ~size_t(15)));
  const int group = threadIdx.x / KW;                     // sample slot within the CTA
  const int cta = blockIdx.x;
  const int share = cta < a.n_hi ? a.w_hi : a.w_lo;
  const int base = cta < a.n_hi ? cta * a.w_hi : a.n_hi * a.w_hi + (cta - a.n_hi) * a.w_lo;
  const int nlive = min(share, a.B - base);               // samples this CTA rolls out (<= 0: nothing left)
  const int s = base + group;
  bool mine = group < nlive;
  if (ONLY_FLAGGED) {
    mine = mine && (a.flags[s] & 1);
    if (!__any_sync(0xffffffffu, mine)) return;           // WARPS == 1: the whole CTA leaves together
  }
  if (nlive <= 0) return;
  {
    const int* src = reinterpret_cast<const int*>(gm);
    int* dst = reinterpret_cast<int*>(sm);
    for (int i = threadIdx.x; i < (int)(sizeof(KModel) / 4); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  if (!mine) return;                                       // idle group of a partly filled warp: exits (full-mask fences skip exited lanes)
  Warp W;
  W.lane = threadIdx.x & (KW - 1);
  W.shift = (threadIdx.x & 31) & ~(KW - 1);
  W.mask = KW_FULL << W.shift;
  {
    // alignment sets: the live warps of the CTA step in lockstep within ROLLOUT_SETS sets (warp w -> set w % SETS)
    const int nw = ONLY_FLAGGED ? 1 : (nlive + GPW - 1) / GPW, w = threadIdx.x >> 5;
    const int sets = nw < ROLLOUT_SETS ? 1 : ROLLOUT_SETS, set = w % sets;
    W.bar = 1 + set;
    W.nthr = ((nw - set + sets - 1) / sets) * 32;
  }
#ifdef CEMK_PHASE_TIMING
  W.phase = 14; W.t0 = clock64();
  for (int i = 0; i < 24; ++i) { W.ph[i] = 0; W.phs[i] = 0; W.phc[i] = 0; }
  W.stepflag = 0; W.nflag = 0;
  for (int i = 0; i < 24; ++i) W.ev[i] = 0;
#endif
  RolloutArgs A;
  const size_t row = (size_t)s * KM_NL * a.T;
  A.T = a.T;
  A.live = true;
  A.thetadot = (STATES && !a.thetadot) ? nullptr : a.thetadot + row;
  if (STATES) {
    A.q0 = a.q0 + (size_t)s * KM_NQ; A.v0 = a.v0 + (size_t)s * KM_NV; A.warm0 = a.warm + (size_t)s * KM_NV;
    A.qpos_out = a.qpos_out + (size_t)s * KM_NQ; A.qvel_out = a.qvel_out + (size_t)s * KM_NV; A.warm_out = a.warm_out + (size_t)s * KM_NV;
  } else {
    A.q0 = a.q0; A.v0 = a.v0;
  }
  A.target_pos = a.target_pos; A.target_rot = a.target_rot;
  A.w_pos = a.w_pos; A.w_rot = a.w_rot; A.w_col = a.w_col;
  A.theta = (STATES && !a.theta) ? nullptr : a.theta + row;
  A.cost4 = STATES ? nullptr : a.cost4 + (size_t)s * 4;
  A.eef_pos = a.eef_pos ? a.eef_pos + (size_t)s * a.T * 3 : nullptr;
  A.eef_rot = a.eef_rot ? a.eef_rot + (size_t)s * a.T * 4 : nullptr;
  A.collision = a.collision ? a.collision + (size_t)s * a.T * sm->nslot_robot : nullptr;
  A.qacc_dbg = a.qacc ? a.qacc + (size_t)s * a.T * KM_NV : nullptr;
  A.flags = a.flags + s;
  A.prevd = a.prevd + (size_t)s * (2 * KM_NPASS * KW);
  A.ovf = a.ovf + (size_t)s * ((KM_NC_TOT - KM_NC_FAST) * KM_OVF_STRIDE);
  rollout_sample<NC, STATES>(W, *sm, ws[group], A);
#ifdef CEMK_PHASE_TIMING
  PHASE(W, 15);
  if (W.lane == 0 && !ONLY_FLAGGED) for (int i = 0; i < 24; ++i) atomicAdd(&g_phase[i], (unsigned long long)W.ph[i]);
  if (W.lane == 0 && !ONLY_FLAGGED) for (int i = 0; i < 24; ++i) atomicAdd(&g_event[i], (unsigned long long)W.ev[i]);
  if (W.lane == 0 && !ONLY_FLAGGED) { for (int i = 0; i < 24; ++i) atomicAdd(&g_phase_cond[i], (unsigned long long)W.phc[i]); atomicAdd(&g_phase_cond[24], (unsigned long long)W.nflag); }
#endif
}
template <int NC, int WARPS>
static size_t rollout_smem() { return ((sizeof(KModel) + 15) & ~size_t(15)) + WARPS * GPW * sizeof(WarpSmemT<NC>); }
static_assert(((sizeof(KModel) + 15) & ~size_t(15)) + ROLLOUT_WARPS * GPW * sizeof(WarpSmemT<KM_NC_FAST>) <= 227 * 1024,
              "rollout scratch exceeds the 227 KB of shared memory a CTA can have");

// ---------------------------------------------------------------------------------------------- sampling
// L = chol(cov + 0.003 I), lower, row-major [n][n] (n = nvar <= MAXVAR); one CTA of 256 threads.  Right-looking on the
// unscaled columns: A[i][k] -= (A[i][j] / A[j][j]) A[k][j] for j = 0 .. k-1 in this order for every element, column j is
// final after step j, scaled by 1 / sqrt(A[j][j]) in a last pass.  The updates are applied in panels of CHOL_NB columns:
// inside a panel every column step touches only the panel's columns (at most 2 elements per thread, one barrier), then
// one pass applies the panel's CHOL_NB updates to every trailing element -- the same operations on the same operands in
// the same order per element as the column-at-a-time loop (bit-identical, 33 us), with the long per-column trailing
// sweep off the barrier chain.  (A left-looking variant with four lanes per row dot product was slower: 43 us.)
// N = largest n of the instantiation: k_chol66 (n <= 96, the matrix in static shared memory) and k_chol_wide (n <= 192, the
// matrix in dynamic shared memory: 148 KB at 192).  Both run this body with the same operations in the same order.
#define CHOL_NB 8
#define CHOL_SMALL_N 96
static_assert(CHOL_NB == 8, "chol_body deals the panel columns with threadIdx.x & 7");
template <int N>
__device__ __forceinline__ void chol_body(int n, const float* __restrict__ cov, float* __restrict__ L, float (*A)[N + 1], float* P) {
  constexpr int KU = (N + 15) / 16, RM = (N + 31) / 32;   // trailing elements of a row per thread; panel rows per thread
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  for (int i = ty; i < n; i += 16)
    for (int j = tx; j < n; j += 16) A[i][j] = cov[i * n + j] + (i == j ? 0.003f : 0.f);
  __syncthreads();
  const int pc = threadIdx.x & (CHOL_NB - 1), pr = threadIdx.x >> 3;      // panel steps: thread = (row offset, panel column)
  for (int j0 = 0; j0 < n - 1; j0 += CHOL_NB) {
    const int je = j0 + CHOL_NB < n ? j0 + CHOL_NB : n;
    for (int j = j0; j < je && j < n - 1; ++j) {
      // every load of the step is issued before the first dependent instruction (rows i0, i0 + 32, ...)
      const int k = j + 1 + pc, i0 = j + 1 + pr;
      const bool kon = k < je;
      const float ajj = A[j][j], akj = kon ? A[k][j] : 0.f;
      float aij[RM], aik[RM]; bool on[RM];
#pragma unroll
      for (int m = 0; m < RM; ++m) {
        const int i = i0 + 32 * m;
        on[m] = kon && i < n && k <= i;
        aij[m] = on[m] ? A[i][j] : 0.f; aik[m] = on[m] ? A[i][k] : 0.f;
      }
      const float p = __frcp_rn(ajj);                    // (the library is built with -use_fast_math for k_rollout; the small
                                                         //  kernels spell out IEEE division / sqrt / exp so the flag does not touch them)
      if (threadIdx.x == 0) P[j] = p;
#pragma unroll
      for (int m = 0; m < RM; ++m) {
        const float s = aij[m] * p;
        aik[m] -= s * akj;
        if (on[m]) A[i0 + 32 * m][k] = aik[m];
      }
      __syncthreads();
    }
    if (je < n) {
      float pp[CHOL_NB];
#pragma unroll
      for (int q = 0; q < CHOL_NB; ++q) pp[q] = P[j0 + q];
      for (int i = je + ty; i < n; i += 16) {
        float ai[CHOL_NB];
#pragma unroll
        for (int q = 0; q < CHOL_NB; ++q) ai[q] = A[i][j0 + q] * pp[q];
        // up to KU elements of row i per thread, their CHOL_NB-long chains interleaved
        float a[KU], ak[KU][CHOL_NB]; bool on[KU];
#pragma unroll
        for (int u = 0; u < KU; ++u) {
          const int k = je + tx + 16 * u;
          on[u] = k <= i;
          a[u] = on[u] ? A[i][k] : 0.f;
#pragma unroll
          for (int q = 0; q < CHOL_NB; ++q) ak[u][q] = on[u] ? A[k][j0 + q] : 0.f;
        }
#pragma unroll
        for (int q = 0; q < CHOL_NB; ++q)
#pragma unroll
          for (int u = 0; u < KU; ++u) a[u] -= ai[q] * ak[u][q];
#pragma unroll
        for (int u = 0; u < KU; ++u) if (on[u]) A[i][je + tx + 16 * u] = a[u];
      }
    }
    __syncthreads();
  }
  for (int i = ty; i < n; i += 16)
    for (int j = tx; j < n; j += 16) {
      const float d = __fsqrt_rn(A[j][j]);
      L[i * n + j] = j > i ? 0.f : (i == j ? d : __fdiv_rn(A[i][j], d));
    }
}
__global__ void __launch_bounds__(256) k_chol66(int n, const float* __restrict__ cov, float* __restrict__ L) {
  __shared__ float A[CHOL_SMALL_N][CHOL_SMALL_N + 1];
  __shared__ float P[CHOL_SMALL_N];
  chol_body<CHOL_SMALL_N>(n, cov, L, A, P);
}
__global__ void __launch_bounds__(256) k_chol_wide(int n, const float* __restrict__ cov, float* __restrict__ L) {
  extern __shared__ float chol_sm[];                     // A[MAXVAR][MAXVAR + 1], P[MAXVAR]
  chol_body<MAXVAR>(n, cov, L, reinterpret_cast<float (*)[MAXVAR + 1]>(chol_sm), chol_sm + MAXVAR * (MAXVAR + 1));
}
static size_t chol_wide_smem() { return sizeof(float) * ((size_t)MAXVAR * (MAXVAR + 1) + MAXVAR); }
// xi[b][i] = mean[i] + sum_{j<=i} L[i][j] z[b][j] (the sum runs j = 0 .. i in this order).  One CTA per SAMPLE_TILE
// consecutive samples: L and the tile's draws in shared memory, a warp works on one row i for different samples (L[i][j]
// is a broadcast, the triangular trip count is uniform in the warp), results leave through a shared tile so that the
// global reads and writes are contiguous.
#define SAMPLE_TILE 28
#define SAMPLE_THREADS 1024      // the kernel is a few dependent memory round trips long: many threads = few loads per thread
__global__ void __launch_bounds__(SAMPLE_THREADS) k_sample(int B, int n, const float* __restrict__ z, const float* __restrict__ mean,
                                                           const float* __restrict__ L, float* __restrict__ xi) {
  extern __shared__ float ssm[];
  const int ld = n + 1, zs = n | 1;                // odd strides: rows i / samples bl fall on different banks
  float* sL = ssm;                                 // [n][ld]
  float* sz = sL + n * ld;                         // [SAMPLE_TILE][zs]
  float* sx = sz + SAMPLE_TILE * zs;               // [SAMPLE_TILE][n]
  float* smu = sx + SAMPLE_TILE * n;               // [n]
  const int b0 = blockIdx.x * SAMPLE_TILE, nb = B - b0 < SAMPLE_TILE ? B - b0 : SAMPLE_TILE;
#pragma unroll 5
  for (int e = threadIdx.x; e < n * n; e += SAMPLE_THREADS) { const int i = e / n; sL[i * ld + (e - i * n)] = L[e]; }
#pragma unroll 2
  for (int e = threadIdx.x; e < nb * n; e += SAMPLE_THREADS) { const int bl = e / n; sz[bl * zs + (e - bl * n)] = z[(size_t)b0 * n + e]; }
  if (threadIdx.x < n) smu[threadIdx.x] = mean[threadIdx.x];
  __syncthreads();
  for (int e = threadIdx.x; e < SAMPLE_TILE * n; e += SAMPLE_THREADS) {
    const int i = e / SAMPLE_TILE, bl = e - i * SAMPLE_TILE;
    if (bl >= nb) continue;
    const float* Li = sL + i * ld; const float* zb = sz + bl * zs;
    float s = 0.f;
    for (int j = 0; j <= i; ++j) s += Li[j] * zb[j];
    sx[bl * n + i] = smu[i] + s;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < nb * n; e += SAMPLE_THREADS) xi[(size_t)b0 * n + e] = sx[e];
}
static size_t sample_smem(int n) { return sizeof(float) * ((size_t)n * (n + 1) + SAMPLE_TILE * (size_t)(n | 1) + SAMPLE_TILE * (size_t)n + n); }

// ---------------------------------------------------------------------------------------------- jax.random stream
// Threefry-2x32 (20 rounds) as used by jax.random (jax/_src/prng.py, pinned jax==0.5.3 in the reference's
// requirements.txt:9); known answers in tests/test_jax_prng.py.
__device__ __forceinline__ void threefry2x32(uint32_t k0, uint32_t k1, uint32_t& x0, uint32_t& x1) {
  const uint32_t ks[3] = {k0, k1, k0 ^ k1 ^ 0x1BD11BDAu};
  x0 += ks[0]; x1 += ks[1];
#define TF_R(r) { x0 += x1; x1 = (x1 << (r)) | (x1 >> (32 - (r))); x1 ^= x0; }
#define TF_A TF_R(13) TF_R(15) TF_R(26) TF_R(6)
#define TF_B TF_R(17) TF_R(29) TF_R(16) TF_R(24)
  TF_A x0 += ks[1]; x1 += ks[2] + 1u;
  TF_B x0 += ks[2]; x1 += ks[0] + 2u;
  TF_A x0 += ks[0]; x1 += ks[1] + 3u;
  TF_B x0 += ks[1]; x1 += ks[2] + 4u;
  TF_A x0 += ks[2]; x1 += ks[0] + 5u;
#undef TF_A
#undef TF_B
#undef TF_R
}
// XLA's float32 erf_inv (Giles' polynomial, xla/client/lib/math.cc ErfInv32)
__device__ __forceinline__ float xla_erfinv32(float x) {
  float w = -log1pf(-x * x);
  const bool lt = w < 5.f;
  w = lt ? w - 2.5f : __fsqrt_rn(w) - 3.f;
  float p = lt ? 2.81022636e-08f : -0.000200214257f;
  p = __fmaf_rn(p, w, lt ? 3.43273939e-07f : 0.000100950558f);
  p = __fmaf_rn(p, w, lt ? -3.5233877e-06f : 0.00134934322f);
  p = __fmaf_rn(p, w, lt ? -4.39150654e-06f : -0.00367342844f);
  p = __fmaf_rn(p, w, lt ? 0.00021858087f : 0.00573950773f);
  p = __fmaf_rn(p, w, lt ? -0.00125372503f : -0.0076224613f);
  p = __fmaf_rn(p, w, lt ? -0.00417768164f : 0.00943887047f);
  p = __fmaf_rn(p, w, lt ? 0.246640727f : 1.00167406f);
  p = __fmaf_rn(p, w, lt ? 1.50140941f : 2.83297682f);
  return fabsf(x) == 1.f ? x * INFINITY : p * x;
}
// out[i] = jax.random.normal(key, (total,), float32)[offset + i], i < count.
//   bits -> uniform in [nextafter(-1, 0), 1): jax/_src/random.py _uniform;  normal = sqrt(2) erfinv(u): _normal_real.
//   partitionable (jax >= 0.5 default): bits[e] = x0 ^ x1 of threefry(key, (0, e));
//   original: counters iota(total) padded to even and split in halves, bits = out0 | out1 concatenated.
__global__ void __launch_bounds__(256) k_jax_normal(uint32_t k0, uint32_t k1, int original, unsigned total, unsigned offset,
                                                    unsigned count, float* __restrict__ out) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const unsigned e = offset + i;
  uint32_t bits;
  if (!original) {
    uint32_t x0 = 0u, x1 = e;
    threefry2x32(k0, k1, x0, x1);
    bits = x0 ^ x1;
  } else {
    const unsigned half = (total + 1u) / 2u;
    const unsigned j = e < half ? e : e - half;
    uint32_t x0 = j, x1 = half + j < total ? half + j : 0u;
    threefry2x32(k0, k1, x0, x1);
    bits = e < half ? x0 : x1;
  }
  const float f = __uint_as_float((bits >> 9) | 0x3F800000u) - 1.f;
  const float lo = -0.99999994f;                                  // nextafter(-1, 0)
  const float u = fmaxf(lo, __fadd_rn(__fmul_rn(f, __fsub_rn(1.f, lo)), lo));
  out[i] = 1.41421354f * xla_erfinv32(u);
}

// ---------------------------------------------------------------------------------------------- projection
// Four lanes per (sample, dof) problem.  Q_inv of the reference is block
// diagonal per DOF, and with A_c = [G_c; -G_c] the slack / residual / multiplier updates of
// mjx_planner.py:196-223 collapse to
//   u_c   = G_c x                                  c in {velocity, acceleration, position}
//   e_c   = u_c - clip(u_c, -b_c, b_c)             (= res+ - res-; exactly 0 inside the bounds)
//   h_c   = u_c + clip(u_c, -b_c, b_c)             (= (b - s+) - (b - s-))
//   Lam  -= sum_c G_c^T e_c                        (the three multipliers only ever appear summed)
//   x'    = Kpp (Lam + xi + sum_c G_c^T h_c) + Kpe b_eq
// i.e. the reference iteration with s and res eliminated.  e_c is formed per time step *before* the
// transpose product -- forming G^T G x - G^T clip(.) instead cancels catastrophically in float32
// (|G^T G| ~ 1e6 at T = 16).
// Mapping: a warp holds 8 problems x 4 time slices (lane = 8 slice + problem); slice s walks the basis rows t = s, s + 4, ...
// A row (NC coefficients padded to PC floats) is read with PC / 4 128-bit shared-memory loads (four distinct rows per warp
// instruction, one per quarter warp) for 3 NC FMAs per lane.  The partial G^T e / G^T h of the four slices are exchanged with
// shuffles inside the quad and summed in slice order by every lane (so the four lanes of a problem carry identical iterates):
// no block barrier after the prologue, a CTA is just PROJ_WARPS independent warps sharing the basis in shared memory.
// One thread per problem alone gives a B200 only ~5 warps per SM on a 1e5-long dependent FMA chain; splitting a problem
// over more lanes runs into the shared-memory bandwidth.
// Occupancy decides this kernel: 6 B / 8 warps have to be resident at once or the tail wave runs the SMs nearly empty
// (4096 samples: 3072 warps; at 118 registers 16 warps fit an SM = 1.3 waves, 175 us).  Registers are
// allocated per SM quadrant, 16384 each: 3072 warps = 20.8 per SM means six warps in some quadrant = at most 80 registers,
// and a CTA size of 7 (or 3 or 1) warps so that 21 per SM is reachable.  The per-problem vectors that are touched once per
// iteration (xs, cst, the multiplier sum) sit in per-thread shared-memory columns, which brings the kernel to 80 registers:
// 3 CTAs of 7 warps per SM = 3108 warp slots, one wave.
#ifndef PROJ_UNROLL
#define PROJ_UNROLL 2
#endif
constexpr int kProjUnroll = PROJ_UNROLL;
#define PROJ_SLICES 4
#define PROJ_PPW (32 / PROJ_SLICES)      // problems per warp
#ifndef PROJ_WARPS
#define PROJ_WARPS 7
#endif
#ifndef PROJ_MINB
#define PROJ_MINB 3
#endif
// NC = Bernstein coefficients per DOF (order + 1), a template parameter so that the iterates stay in registers; a basis
// row is padded to PC = 4 ceil(NC / 4) floats.  nd = DOF per sample: B nd problems, xi / xi_f rows of nd NC, state_term rows of
// 5 nd, thetadot rows of nd T.  ND = KM_NL fixes it at compile time (the product path, the code the 6-DOF build always had);
// ND = 0 takes it from `ndof` at run time (any other DOF count; the per-problem arithmetic is the same).
template <int NC, int ND>
__global__ void __launch_bounds__(32 * PROJ_WARPS, NC <= 11 ? PROJ_MINB : 1) k_project(int B, int ndof, int T, int iters, const float* __restrict__ G,
                                                              const float* __restrict__ Kc, const float* __restrict__ xi,
                                                              const float* __restrict__ state_term, float* __restrict__ xi_f,
                                                              float* __restrict__ thetadot) {
  constexpr int PC = (NC + 3) / 4 * 4, KPAD = (5 * NC + 3 + 3) / 4 * 4;
  const int nd = ND ? ND : ndof, NV = nd * NC;
  extern __shared__ __align__(16) float sm[];
  float* sG = sm;                        // [3][T][PC]
  float* sKpp = sm + 3 * T * PC;         // [NC][PC]
  float* sK = sKpp + NC * PC;            // Kpe[5 NC] bounds[3], padded to KPAD
  float* sP = sK + KPAD;                 // [3 NC][blockDim.x] per-thread columns: xs, cst, lam
  for (int e = threadIdx.x; e < 3 * T * PC; e += blockDim.x) { const int r = e / PC, k = e % PC; sG[e] = k < NC ? G[r * NC + k] : 0.f; }
  for (int e = threadIdx.x; e < NC * PC; e += blockDim.x) { const int r = e / PC, k = e % PC; sKpp[e] = k < NC ? Kc[r * NC + k] : 0.f; }
  for (int e = threadIdx.x; e < 5 * NC + 3; e += blockDim.x) sK[e] = Kc[NC * NC + e];
  __syncthreads();
#ifndef PROJ_LANEMAP
#define PROJ_LANEMAP 1
#endif
#if PROJ_LANEMAP
  // lane = 8 slice + problem: the eight lanes of a quarter warp (one phase of a 128-bit shared-memory load) read the same row
  const int lane = threadIdx.x & 31, slice = lane >> 3, pl = lane & (PROJ_PPW - 1);
#define PROJ_SRC(q) ((q) * PROJ_PPW + pl)
#else
  const int lane = threadIdx.x & 31, slice = lane & (PROJ_SLICES - 1), pl = lane >> 2;
#define PROJ_SRC(q) ((lane & ~(PROJ_SLICES - 1)) | (q))
#endif
  int prob = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * PROJ_PPW + pl;
  const bool act = prob < B * nd;        // idle lanes still take part in the shuffles
  if (!act) prob = B * nd - 1;
  const int b = prob / nd, d = prob % nd;
  const float* Kpe = sK; const float* bnd = sK + 5 * NC;
  float* myxs = sP + threadIdx.x;
  float* mycst = sP + NC * blockDim.x + threadIdx.x;
  float* mylam = sP + 2 * NC * blockDim.x + threadIdx.x;
  const int cs = blockDim.x;
  auto rowp = [](const float* p, float* g) {
#pragma unroll
    for (int q = 0; q < PC / 4; ++q) {
      const float4 a = reinterpret_cast<const float4*>(p)[q];
      if (4 * q < NC) g[4 * q] = a.x;
      if (4 * q + 1 < NC) g[4 * q + 1] = a.y;
      if (4 * q + 2 < NC) g[4 * q + 2] = a.z;
      if (4 * q + 3 < NC) g[4 * q + 3] = a.w;
    }
  };
  float x[NC], rh[NC], re[NC];
  {
    float beq[5];
#pragma unroll
    for (int k = 0; k < NC; ++k) { myxs[k * cs] = xi[(size_t)b * NV + d * NC + k]; mylam[k * cs] = 0.f; x[k] = 0.f; rh[k] = 0.f; }
#pragma unroll
    for (int k = 0; k < 5; ++k) beq[k] = state_term[(size_t)b * 5 * nd + k * nd + d];
#pragma unroll
    for (int i = 0; i < NC; ++i) { float s = 0.f; for (int k = 0; k < 5; ++k) s += Kpe[i * 5 + k] * beq[k]; mycst[i * cs] = s; }
  }
  for (int it = 0; it < iters; ++it) {
    {
      float rhs[NC];
#pragma unroll
      for (int k = 0; k < NC; ++k) { rhs[k] = mylam[k * cs] + myxs[k * cs] + rh[k]; rh[k] = 0.f; re[k] = 0.f; }
#pragma unroll
      for (int i = 0; i < NC; ++i) { float kr[NC]; rowp(sKpp + i * PC, kr); float s = mycst[i * cs]; for (int k = 0; k < NC; ++k) s += kr[k] * rhs[k]; x[i] = s; }
    }
    for (int c = 0; c < 3; ++c) {
      const float bc = bnd[c];
      const float* Gc = sG + c * T * PC;
#pragma unroll(kProjUnroll)
      for (int t = slice; t < T; t += PROJ_SLICES) {
        float g[NC];
        rowp(Gc + t * PC, g);
        float u0 = 0.f, u1 = 0.f, u2 = 0.f;                            // three short chains instead of one of NC
#pragma unroll
        for (int k = 0; k < NC; ++k) { if (k % 3 == 0) u0 += g[k] * x[k]; else if (k % 3 == 1) u1 += g[k] * x[k]; else u2 += g[k] * x[k]; }
        const float u = (u0 + u1) + u2;
        const float cl = fminf(fmaxf(u, -bc), bc);
        const float e = u - cl, h = u + cl;
#pragma unroll
        for (int k = 0; k < NC; ++k) { re[k] += g[k] * e; rh[k] += g[k] * h; }
      }
    }
    // exchange the partial sums of the four slices of a problem; every lane adds them in slice order
#pragma unroll
    for (int k = 0; k < NC; ++k) {
      float se = 0.f, sh = 0.f;
#pragma unroll
      for (int q = 0; q < PROJ_SLICES; ++q) { se += __shfl_sync(0xffffffffu, re[k], PROJ_SRC(q)); sh += __shfl_sync(0xffffffffu, rh[k], PROJ_SRC(q)); }
      rh[k] = sh;
      mylam[k * cs] -= se;
    }
  }
  if (!act) return;
  if (slice == 0) {
#pragma unroll
    for (int k = 0; k < NC; ++k) xi_f[(size_t)b * NV + d * NC + k] = x[k];
  }
  if (thetadot) {
    const float* Gv = sG;    // Pdot
    float* out = thetadot + (size_t)b * nd * T + (size_t)d * T;
    for (int t = slice; t < T; t += PROJ_SLICES) {
      float g[NC];
      rowp(Gv + t * PC, g);
      float u = 0.f;
#pragma unroll
      for (int k = 0; k < NC; ++k) u += g[k] * x[k];
      out[t] = u;
    }
  }
}
template <int NC>
static int project_smem(int T, int threads) {
  constexpr int PC = (NC + 3) / 4 * 4, KPAD = (5 * NC + 3 + 3) / 4 * 4;
  return (3 * T * PC + NC * PC + KPAD + 3 * NC * threads) * (int)sizeof(float);
}
// warps per CTA: PROJ_WARPS when the nprob = B ndof problems fill the GPU, fewer (more CTAs) for small batches
static int project_warps(int nprob) {
  const int warps = (nprob + PROJ_PPW - 1) / PROJ_PPW;
  const int w = (warps + 148 * PROJ_MINB - 1) / (148 * PROJ_MINB);
  return w < 1 ? 1 : (w > PROJ_WARPS ? PROJ_WARPS : w);
}
// run `body` with NC = ncoef as a compile-time constant
#define CEMK_FOR_NCOEF(ncoef, body) switch (ncoef) { \
  case 4: { constexpr int NC = 4; body; } break;   case 5: { constexpr int NC = 5; body; } break;   case 6: { constexpr int NC = 6; body; } break; \
  case 7: { constexpr int NC = 7; body; } break;   case 8: { constexpr int NC = 8; body; } break;   case 9: { constexpr int NC = 9; body; } break; \
  case 10: { constexpr int NC = 10; body; } break; case 11: { constexpr int NC = 11; body; } break; case 12: { constexpr int NC = 12; body; } break; \
  case 13: { constexpr int NC = 13; body; } break; case 14: { constexpr int NC = 14; body; } break; case 15: { constexpr int NC = 15; body; } break; \
  case 16: { constexpr int NC = 16; body; } break; default: break; }

// ---------------------------------------------------------------------------------------------- standalone cost
__global__ void __launch_bounds__(128) k_cost_batch(int B, int T, int nslot, const float* __restrict__ eef_pos, const float* __restrict__ eef_rot,
                                                    const float* __restrict__ collision, const float* __restrict__ tpos, const float* __restrict__ trot,
                                                    float w_pos, float w_rot, float w_col, float* __restrict__ cost4) {
  const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (s >= B) return;
  float cg = 0.f, cr = 0.f, cc = 0.f;
  const float* tp = tpos + (size_t)s * 3; const float* tq = trot + (size_t)s * 4;
  const float tn = __frcp_rn(__fsqrt_rn(tq[0] * tq[0] + tq[1] * tq[1] + tq[2] * tq[2] + tq[3] * tq[3]));
  for (int t = lane; t < T; t += 32) {
    const float* p = eef_pos + ((size_t)s * T + t) * 3; const float* q = eef_rot + ((size_t)s * T + t) * 4;
    float dx = p[0] - tp[0], dy = p[1] - tp[1], dz = p[2] - tp[2];
    cg += __fsqrt_rn(dx * dx + dy * dy + dz * dz);
    float qn = __frcp_rn(__fsqrt_rn(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]));
    float dp = fabsf((q[0] * tq[0] + q[1] * tq[1] + q[2] * tq[2] + q[3] * tq[3]) * qn * tn);
    cr += 2.f * acosf(fminf(fmaxf(dp, -1.f), 1.f));
  }
  for (int k = lane; k < nslot; k += 32) {
    float prev = 0.f;
    for (int t = 0; t < T; ++t) {
      float c = collision[((size_t)s * T + t) * nslot + k];
      if (c < 0.f) cc += 1.f;
      if (t > 0) cc += fmaxf((1.f - 0.005f) * prev - c, 0.f);
      prev = c;
    }
  }
  for (int o = 16; o; o >>= 1) { cg += __shfl_xor_sync(0xffffffffu, cg, o); cr += __shfl_xor_sync(0xffffffffu, cr, o); cc += __shfl_xor_sync(0xffffffffu, cc, o); }
  if (lane == 0) {
    float* o4 = cost4 + (size_t)s * 4;
    o4[0] = w_pos * cg + w_rot * cr + w_col * cc; o4[1] = cg; o4[2] = cr; o4[3] = cc;
  }
}

// ---------------------------------------------------------------------------------------------- argsort / top-k
// Ascending unsigned key of a cost in jnp.argsort's order: NaN last, -0.0 ties with +0.0 (lax's sort canonicalises the
// zero's sign), every other value -- subnormals included -- in IEEE order.  The zero test looks at the bits: a float
// comparison would be flushed to zero by -use_fast_math and tie the subnormals with zero as well.
__device__ __forceinline__ unsigned int float_order(float f) {
  if (f != f) return 0xffffffffu;                       // NaN sorts last (jnp.argsort)
  unsigned int u = __float_as_uint(f);
  if ((u << 1) == 0u) u = 0u;                           // -0.0 -> +0.0
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__global__ void k_make_keys(int n, int npow2, const float* __restrict__ cost, int stride, unsigned long long* __restrict__ keys) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npow2) return;
  keys[i] = i < n ? (((unsigned long long)float_order(cost[(size_t)i * stride]) << 32) | (unsigned int)i) : ~0ull;
}
#define SORT_BLK 4096    // keys per CTA held in shared memory (32 KB)
// All stages with partner distance < SORT_BLK for merge size k_outer (full: the whole local sort, k = 2..SORT_BLK) on a block of
// SORT_BLK keys, four consecutive keys per thread in registers: partner distances 1, 2 stay inside a thread, 4 .. 64 inside a
// warp (shuffles), only distances >= 128 go through shared memory -- 15 of the 78 stages of a full 4096-key sort need a barrier
// pair instead of all of them (39 -> about 20 us).  Keys are unique (the low word is the index), so any correct sorting
// network gives the identical result.
__device__ __forceinline__ void bitonic_cas(unsigned long long& a, unsigned long long b, bool keep_min) {
  a = keep_min ? (a < b ? a : b) : (a > b ? a : b);
}
__global__ void __launch_bounds__(SORT_BLK / 4) k_bitonic_local4(unsigned long long* __restrict__ keys, int k_outer, int full) {
  __shared__ unsigned long long s[SORT_BLK];
  const int t = threadIdx.x, base = blockIdx.x * SORT_BLK, i0 = 4 * t;
  unsigned long long v[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) v[r] = keys[base + i0 + r];
  for (int k = full ? 2 : k_outer; k <= (full ? SORT_BLK : k_outer); k <<= 1) {
    for (int j = (k >> 1) < SORT_BLK ? (k >> 1) : (SORT_BLK >> 1); j > 0; j >>= 1) {
      if (j >= 128) {                                        // partner in another warp: through shared memory
#pragma unroll
        for (int r = 0; r < 4; ++r) s[i0 + r] = v[r];
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int i = i0 + r;
          const bool up = ((base + i) & k) == 0, lower = (i & j) == 0;
          bitonic_cas(v[r], s[i ^ j], lower == up);
        }
        __syncthreads();
      } else if (j >= 4) {                                   // partner thread in the same warp
        const int dl = j >> 2;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int i = i0 + r;
          const unsigned long long o = __shfl_xor_sync(0xffffffffu, v[r], dl);
          const bool up = ((base + i) & k) == 0, lower = (i & j) == 0;
          bitonic_cas(v[r], o, lower == up);
        }
      } else {                                               // partner in this thread (j = 2 or 1)
        if (j == 2) {
          const bool u0 = ((base + i0) & k) == 0;            // k >= 4 here: the four keys share the direction
          unsigned long long a0 = v[0], a1 = v[1], a2 = v[2], a3 = v[3];
          v[0] = u0 ? (a0 < a2 ? a0 : a2) : (a0 > a2 ? a0 : a2); v[2] = u0 ? (a0 < a2 ? a2 : a0) : (a0 > a2 ? a2 : a0);
          v[1] = u0 ? (a1 < a3 ? a1 : a3) : (a1 > a3 ? a1 : a3); v[3] = u0 ? (a1 < a3 ? a3 : a1) : (a1 > a3 ? a3 : a1);
        } else {                                             // j == 1: pairs (0,1) and (2,3); directions may differ when k == 2
          const bool u0 = ((base + i0) & k) == 0, u2 = ((base + i0 + 2) & k) == 0;
          unsigned long long a0 = v[0], a1 = v[1], a2 = v[2], a3 = v[3];
          v[0] = u0 ? (a0 < a1 ? a0 : a1) : (a0 > a1 ? a0 : a1); v[1] = u0 ? (a0 < a1 ? a1 : a0) : (a0 > a1 ? a1 : a0);
          v[2] = u2 ? (a2 < a3 ? a2 : a3) : (a2 > a3 ? a2 : a3); v[3] = u2 ? (a2 < a3 ? a3 : a2) : (a2 > a3 ? a3 : a2);
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) keys[base + i0 + r] = v[r];
}
__global__ void k_bitonic_global(unsigned long long* __restrict__ keys, int npow2, int k, int j) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= npow2 / 2) return;
  const int i = 2 * e - (e & (j - 1));
  const int p = i + j;
  const bool up = ((i & k) == 0);
  unsigned long long a = keys[i], b = keys[p];
  if ((a > b) == up) { keys[i] = b; keys[p] = a; }
}
// Small inputs (n <= RANK_MAXN, every per-GPU shard of the weak-scaling configurations): the sorted position of a key is the
// number of keys below it (keys are unique), so one launch does what key generation + 78 compare-exchange stages + the
// gather did: every CTA builds all n keys in shared memory, takes RANK_CAND candidates (one per lane), its warps count
// over disjoint parts of the key array (broadcast 64-bit loads), and the candidates whose position is below k copy their
// row straight to its place.  n^2 / 2 comparisons spread over the whole GPU (4096 keys: 1.7e7, a few microseconds)
// instead of a latency chain of barriers in one CTA (37 us).
#define RANK_CAND 32
#define RANK_MAXN 8192
#define RANK_THREADS 512
__global__ void __launch_bounds__(RANK_THREADS) k_rank_select(int NVAR, int n, const float* __restrict__ cost, int stride, int idx_base,
                                                              unsigned long long* __restrict__ keys_sorted, int* __restrict__ idx_sorted, int k,
                                                              const float* __restrict__ xi, float* __restrict__ xi_elite,
                                                              float* __restrict__ cost_elite, float* __restrict__ pack) {
  extern __shared__ unsigned long long rk_keys[];
  __shared__ int cnt[RANK_CAND];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = RANK_THREADS / 32;
  for (int e = tid; e < n; e += RANK_THREADS) rk_keys[e] = ((unsigned long long)float_order(cost[(size_t)e * stride]) << 32) | (unsigned int)e;
  if (tid < RANK_CAND) cnt[tid] = 0;
  __syncthreads();
  const int base = blockIdx.x * RANK_CAND, i = base + lane;
  const unsigned long long ki = i < n ? rk_keys[i] : 0ull;
  const int chunk = (n + nw - 1) / nw, j0 = warp * chunk, j1 = j0 + chunk < n ? j0 + chunk : n;
  int c = 0;
#pragma unroll 8
  for (int j = j0; j < j1; ++j) c += rk_keys[j] < ki ? 1 : 0;
  atomicAdd(&cnt[lane], c);
  __syncthreads();
  if (tid < RANK_CAND && i < n) {
    const int r = cnt[tid];
    if (idx_sorted) idx_sorted[r] = i + idx_base;
    if (keys_sorted) keys_sorted[r] = ki;
  }
  if (k <= 0) return;
  const int W = pack ? NVAR + 2 : NVAR;
  for (int e = tid; e < RANK_CAND * W; e += RANK_THREADS) {
    const int cnd = e / W, col = e - cnd * W, src = base + cnd;
    if (src >= n) break;
    const int r = cnt[cnd];
    if (r >= k) continue;
    if (pack) pack[(size_t)r * W + col] = col < NVAR ? xi[(size_t)src * NVAR + col] : (col == NVAR ? cost[(size_t)src * stride] : (float)(src + idx_base));
    else {
      xi_elite[(size_t)r * NVAR + col] = xi[(size_t)src * NVAR + col];
      if (col == 0) cost_elite[r] = cost[(size_t)src * stride];
    }
  }
}
static_assert(RANK_MAXN >= SORT_BLK, "the bitonic path (n > RANK_MAXN) assumes full SORT_BLK blocks");
// The gather after the bitonic sort, with k_rank_select's outputs: idx_sorted[n] when given, then the k best rows either as
// xi_elite / cost_elite or as the elite exchange records pack[k][nvar + 2] = xi[nvar], cost, global index (as float, exact
// below 2^24) that one rank contributes to the NCCL all-gather.
__global__ void k_gather_sorted(int NVAR, int n, const unsigned long long* __restrict__ keys, int idx_base, int* __restrict__ idx_sorted, int k,
                                const float* __restrict__ cost, int stride, const float* __restrict__ xi, float* __restrict__ xi_elite,
                                float* __restrict__ cost_elite, float* __restrict__ pack) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, W = pack ? NVAR + 2 : NVAR;
  if (idx_sorted && i < n) idx_sorted[i] = (int)(unsigned int)(keys[i] & 0xffffffffull) + idx_base;
  if (i >= k * W) return;
  const int e = i / W, c = i % W;
  const int src = (int)(unsigned int)(keys[e] & 0xffffffffull);
  if (pack) pack[i] = c < NVAR ? xi[(size_t)src * NVAR + c] : (c == NVAR ? cost[(size_t)src * stride] : (float)(src + idx_base));
  else {
    xi_elite[i] = xi[(size_t)src * NVAR + c];
    if (c == 0) cost_elite[e] = cost[(size_t)src * stride];
  }
}

// Merge of the gathered elite lists without sorting: the candidates arrive as `nlist` blocks of `kl` records, each block
// already (cost, index)-sorted by its rank, so the global position of a record is the number of records that precede it in
// (cost, row) order = its position in its own block + for every other block the count of records with a smaller key (blocks
// before it also count equal keys: rows there are lower).  One thread per record, a binary search per block; records whose
// position is below k are written straight to their place.  Replaces key generation + a bitonic sort of nlist * kl keys.
// STAGED: the (order-mapped) cost keys of all records are first copied to shared memory (nlist * kl <= MERGE_MAXKEYS), so
// the nlist - 1 binary searches of a record run at shared-memory instead of L2 latency.  The winners of a CTA are then
// compacted and their rows copied element-wise by all threads with several independent loads in flight per thread (a thread
// copying its own 68-float row alone was a chain of 68 L2 round trips: most of the 39 us at 8 lists of 1638).
#define MERGE_MAXKEYS (48 * 1024)
#define MERGE_THREADS 1024
template <bool STAGED>
__global__ void __launch_bounds__(MERGE_THREADS) k_merge_lists(int NVAR, int nlist, int kl, int k, const float* __restrict__ packed,
                                                               float* __restrict__ xi_elite, float* __restrict__ cost_elite, int* __restrict__ gidx_elite) {
  extern __shared__ unsigned mk[];
  __shared__ int wsrc[MERGE_THREADS], wpos[MERGE_THREADS], nwin;
  const int tid = threadIdx.x, n = nlist * kl, PACKW = NVAR + 2;
  if (tid == 0) nwin = 0;
  if (STAGED) {
#pragma unroll 8
    for (int e = tid; e < n; e += MERGE_THREADS) mk[e] = float_order(packed[(size_t)e * PACKW + NVAR]);
  }
  __syncthreads();
  const int r = blockIdx.x * MERGE_THREADS + tid;
  if (r < n) {
    const int a = r / kl, p = r - a * kl;
    const unsigned key = STAGED ? mk[r] : float_order(packed[(size_t)r * PACKW + NVAR]);
    int pos = p;
    for (int b = 0; b < nlist && pos < k; ++b) {
      if (b == a) continue;
      const float* blk = packed + (size_t)b * kl * PACKW + NVAR;
      int lo = 0, hi = kl;                              // first record of block b that does not precede this one
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const unsigned km = STAGED ? mk[b * kl + mid] : float_order(blk[(size_t)mid * PACKW]);
        if (km < key || (km == key && b < a)) lo = mid + 1; else hi = mid;
      }
      pos += lo;
    }
    if (pos < k) { const int w = atomicAdd(&nwin, 1); wsrc[w] = r; wpos[w] = pos; }
  }
  __syncthreads();
  const int tot = nwin * PACKW;
#pragma unroll 4
  for (int e = tid; e < tot; e += MERGE_THREADS) {
    const int w = e / PACKW, c = e - w * PACKW, ps = wpos[w];
    const float v = packed[(size_t)wsrc[w] * PACKW + c];
    if (c < NVAR) xi_elite[(size_t)ps * NVAR + c] = v;
    else if (c == NVAR) cost_elite[ps] = v;
    else gidx_elite[ps] = (int)v;
  }
}

// ---------------------------------------------------------------------------------------------- mean / covariance
__device__ __forceinline__ float precise_expf(float x) { return (float)exp((double)x); }     // -use_fast_math would turn expf into ex2.approx
// grid = nvar CTAs (one covariance row each) of MC_THREADS threads.  The k elites are dealt to G = MC_THREADS / nvar thread
// groups (thread = (group, column)); partial sums meet in shared memory and are added in group order, and the weights are
// reduced by a fixed tree: the summation order depends on (k, nvar) only, so every rank gets bit-identical mean / cov.
// (One thread per column walking all k elites took 0.67 ms at k = 1638, the 8-GPU weak-scaling configuration.)
#define MC_THREADS 512
#define MC_WCACHE 4096         // elite weights kept in shared memory (beyond that they are recomputed)
__global__ void __launch_bounds__(MC_THREADS) k_mean_cov(int NVAR, int k, const float* __restrict__ cost, const float* __restrict__ xi,
                                                         const float* __restrict__ mean_prev, const float* __restrict__ cov_prev, float lamda,
                                                         float am, float ac, float* __restrict__ mean_out, float* __restrict__ cov_out) {
  __shared__ float red[MC_THREADS];
  __shared__ float sw[MC_WCACHE];
  __shared__ float part[MC_THREADS];
  __shared__ float smean[MAXVAR];
  const int tid = threadIdx.x, row = blockIdx.x;
  const int G = MC_THREADS / NVAR, g = tid / NVAR, j = tid - g * NVAR;
  const bool on = g < G;
  // smallest cost
  float v = INFINITY;
  for (int i = tid; i < k; i += MC_THREADS) v = fminf(v, cost[i]);
  red[tid] = v; __syncthreads();
  for (int o = MC_THREADS / 2; o; o >>= 1) { if (tid < o) red[tid] = fminf(red[tid], red[tid + o]); __syncthreads(); }
  const float cmin = red[0], il = __frcp_rn(lamda);
  __syncthreads();
  // weights and their sum
  float ws = 0.f;
  for (int i = tid; i < k; i += MC_THREADS) { const float w = precise_expf(-il * (cost[i] - cmin)); if (i < MC_WCACHE) sw[i] = w; ws += w; }
  red[tid] = ws; __syncthreads();
  for (int o = MC_THREADS / 2; o; o >>= 1) { if (tid < o) red[tid] += red[tid + o]; __syncthreads(); }
  const float sumw = red[0];
  auto weight = [&](int i) { return i < MC_WCACHE ? sw[i] : precise_expf(-il * (cost[i] - cmin)); };
  // new mean (every CTA needs all of it)
  // (cached weights in a loop of their own: with the recomputing branch inside, the loop is not unrolled and runs at one
  //  L2 round trip per elite -- 127 us at k = 1638)
  const int kc = k < MC_WCACHE ? k : MC_WCACHE;
  float s = 0.f;
  if (on) {
#pragma unroll 8
    for (int i = g; i < kc; i += G) s += sw[i] * xi[(size_t)i * NVAR + j];
    for (int i = g + ((kc - g + G - 1) / G) * G; i < k; i += G) s += weight(i) * xi[(size_t)i * NVAR + j];
  }
  part[tid] = s; __syncthreads();
  if (tid < NVAR) {
    float t = 0.f;
    for (int q = 0; q < G; ++q) t += part[q * NVAR + tid];
    const float mnew = (1.f - am) * mean_prev[tid] + am * __fdiv_rn(t, sumw);
    smean[tid] = mnew;
    if (row == 0) mean_out[tid] = mnew;
  }
  __syncthreads();
  // covariance row
  s = 0.f;
  if (on) {
    const float mr = smean[row], mj = smean[j];
#pragma unroll 8
    for (int i = g; i < kc; i += G) s += sw[i] * (xi[(size_t)i * NVAR + row] - mr) * (xi[(size_t)i * NVAR + j] - mj);
    for (int i = g + ((kc - g + G - 1) / G) * G; i < k; i += G) s += weight(i) * (xi[(size_t)i * NVAR + row] - mr) * (xi[(size_t)i * NVAR + j] - mj);
  }
  part[tid] = s; __syncthreads();
  if (tid < NVAR) {
    float t = 0.f;
    for (int q = 0; q < G; ++q) t += part[q * NVAR + tid];
    cov_out[row * NVAR + tid] = (1.f - ac) * cov_prev[row * NVAR + tid] + ac * __fdiv_rn(t, sumw) + (row == tid ? 0.0001f : 0.f);
  }
}

// Large elite sets (k >= MC_BLOCKED_MINK: the 8-GPU configurations, where every rank redoes the update over all k global
// elites): k_mean_cov makes every one of its nvar CTAs stream the whole elite matrix twice (57 MB of L2 reads at k = 1638,
// 35 us; 67 us at k = 3276).  Here the elites are cut into blocks of MC_EB; a CTA reads its block once and writes the block's
// weighted sums about the shift a = mean_prev,
//   S0 = sum w,  S1[j] = sum w (x_j - a_j),  S2[r][c] = sum w (x_r - a_r)(x_c - a_c)   (c <= r),
// and a second launch adds the blocks in block order and forms, with delta = S1 / S0, the new mean m = (1 - am) a + am (a + delta)
// and the covariance about m:  S2 / S0 - delta D^T - D delta^T + D D^T,  D = m - a.  Fixed summation order (block by block,
// elite by elite) => bit-identical on every rank.  The shift keeps the single pass accurate: after the first iteration the
// elites sit around mean_prev (|delta| below one standard deviation), and in the first one mean_prev is the sampler's mean.
#define MC_EB 32
#define MC_BLOCKED_MINK 1024
#define MC_BLOCKED_MAXK 8192
#define MC_PAD 16                       // the number of blocks is padded to a multiple (zero blocks): no remainder loop in the sums
static int mc_blocks(int k) { return ((k + MC_EB - 1) / MC_EB + MC_PAD - 1) / MC_PAD * MC_PAD; }
static size_t mc_stride(int nvar) { return 1 + (size_t)nvar + (size_t)nvar * (nvar + 1) / 2; }
// The elite tiles x - a and w (x - a) of a block, rows of LD floats: k_mc_partial keeps them in static shared memory
// (LD = 97, nvar <= 96), k_mc_partial_wide in dynamic shared memory (LD = 193, nvar <= 192: 49 KB, above the static limit).
#define MC_LD_SMALL (CHOL_SMALL_N + 1)
#define MC_LD_WIDE (MAXVAR + 1)
template <int LD>
__device__ __forceinline__ void mc_partial_body(int NVAR, int k, const float* __restrict__ cost, const float* __restrict__ xi,
                                                const float* __restrict__ mean_prev, float lamda, float* __restrict__ part,
                                                float* red, float* sw, float (*sd)[LD], float (*swd)[LD]) {
  const int tid = threadIdx.x, e0 = blockIdx.x * MC_EB, ne = k - e0 < MC_EB ? (k - e0 > 0 ? k - e0 : 0) : MC_EB;
  const int npair = NVAR * (NVAR + 1) / 2;
  float* P = part + (size_t)blockIdx.x * (1 + NVAR + npair);
  if (ne == 0) {                                   // padding block
    for (int e = tid; e < 1 + NVAR + npair; e += 256) P[e] = 0.f;
    return;
  }
  float v = INFINITY;
  for (int i = tid; i < k; i += 256) v = fminf(v, cost[i]);
  red[tid] = v; __syncthreads();
  for (int o = 128; o; o >>= 1) { if (tid < o) red[tid] = fminf(red[tid], red[tid + o]); __syncthreads(); }
  const float cmin = red[0], il = __frcp_rn(lamda);
  if (tid < MC_EB) sw[tid] = tid < ne ? precise_expf(-il * (cost[e0 + tid] - cmin)) : 0.f;
  for (int idx = tid; idx < ne * NVAR; idx += 256) { const int e = idx / NVAR, j = idx - e * NVAR; sd[e][j] = xi[(size_t)(e0 + e) * NVAR + j] - mean_prev[j]; }
  __syncthreads();
  for (int idx = tid; idx < ne * NVAR; idx += 256) { const int e = idx / NVAR, j = idx - e * NVAR; swd[e][j] = sw[e] * sd[e][j]; }
  __syncthreads();
  if (tid == 0) { float t = 0.f; for (int e = 0; e < ne; ++e) t += sw[e]; P[0] = t; }
  if (tid < NVAR) { float t = 0.f; for (int e = 0; e < ne; ++e) t += swd[e][tid]; P[1 + tid] = t; }
  for (int p = tid; p < npair; p += 256) {
    int r = (int)((sqrtf(8.f * (float)p + 1.f) - 1.f) * 0.5f);
    while (r * (r + 1) / 2 > p) --r;
    while ((r + 1) * (r + 2) / 2 <= p) ++r;
    const int c = p - r * (r + 1) / 2;
    float t = 0.f;
#pragma unroll 8
    for (int e = 0; e < ne; ++e) t += sd[e][r] * swd[e][c];
    P[1 + NVAR + p] = t;
  }
}
__global__ void __launch_bounds__(256) k_mc_partial(int NVAR, int k, const float* __restrict__ cost, const float* __restrict__ xi,
                                                    const float* __restrict__ mean_prev, float lamda, float* __restrict__ part) {
  __shared__ float red[256];
  __shared__ float sw[MC_EB];
  __shared__ float sd[MC_EB][MC_LD_SMALL];         // x - a
  __shared__ float swd[MC_EB][MC_LD_SMALL];        // w (x - a)
  mc_partial_body<MC_LD_SMALL>(NVAR, k, cost, xi, mean_prev, lamda, part, red, sw, sd, swd);
}
__global__ void __launch_bounds__(256) k_mc_partial_wide(int NVAR, int k, const float* __restrict__ cost, const float* __restrict__ xi,
                                                         const float* __restrict__ mean_prev, float lamda, float* __restrict__ part) {
  __shared__ float red[256];
  __shared__ float sw[MC_EB];
  extern __shared__ float mc_tiles[];              // sd, swd [MC_EB][MC_LD_WIDE]
  float (*sd)[MC_LD_WIDE] = reinterpret_cast<float (*)[MC_LD_WIDE]>(mc_tiles);
  mc_partial_body<MC_LD_WIDE>(NVAR, k, cost, xi, mean_prev, lamda, part, red, sw, sd, sd + MC_EB);
}
static size_t mc_wide_smem() { return sizeof(float) * 2 * MC_EB * MC_LD_WIDE; }
// grid = nvar CTAs (covariance row r = blockIdx.x, entries c <= r and their mirror images), THREADS > nvar threads
// (128 for nvar <= 127, 256 above)
template <int THREADS>
__global__ void __launch_bounds__(THREADS) k_mc_finish(int NVAR, int nblk, const float* __restrict__ part, const float* __restrict__ mean_prev,
                                                   const float* __restrict__ cov_prev, float am, float ac, float* __restrict__ mean_out,
                                                   float* __restrict__ cov_out) {
  __shared__ float sdelta[MAXVAR], sD[MAXVAR], sS2[MAXVAR], sW;
  const int tid = threadIdx.x, r = blockIdx.x, npair = NVAR * (NVAR + 1) / 2;
  const size_t stride = 1 + (size_t)NVAR + npair;
  // one pass over the blocks: thread t < nvar adds S1[t] and S2[r][t]; thread THREADS - 1 adds S0
  {
    const bool w = tid == THREADS - 1, on = tid < NVAR, lo = on && tid <= r;
    const float* p1 = part + (w ? 0 : 1 + (on ? tid : 0));
    const float* p2 = part + 1 + NVAR + (size_t)r * (r + 1) / 2 + (lo ? tid : 0);
    float s1 = 0.f, s2 = 0.f;
    if (w || on) {
#pragma unroll 16
      for (int b = 0; b < nblk; ++b) { s1 += p1[b * stride]; s2 += p2[b * stride]; }
    }
    if (w) sW = s1;
    if (on) { sdelta[tid] = s1; sS2[tid] = s2; }
  }
  __syncthreads();
  const float W = sW;
  if (tid < NVAR) {
    const float a = mean_prev[tid], delta = __fdiv_rn(sdelta[tid], W);
    const float mnew = (1.f - am) * a + am * (a + delta);
    sdelta[tid] = delta; sD[tid] = mnew - a;
    if (r == 0) mean_out[tid] = mnew;
  }
  __syncthreads();
  if (tid <= r && tid < NVAR) {
    const int c = tid;
    const float cv = __fdiv_rn(sS2[c], W) - sdelta[r] * sD[c] - sD[r] * sdelta[c] + sD[r] * sD[c];
    cov_out[r * NVAR + c] = (1.f - ac) * cov_prev[r * NVAR + c] + ac * cv + (r == c ? 0.0001f : 0.f);
    if (c != r) cov_out[c * NVAR + r] = (1.f - ac) * cov_prev[c * NVAR + r] + ac * cv;
  }
}


// ---------------------------------------------------------------------------------------------- calibration
// FP32 FMA throughput of this GPU under the kernel's own conditions (register operands, 8 independent
// chains per thread): the measured denominator of the rollout kernel's FP32 roofline.
__global__ void __launch_bounds__(256) k_fma_peak(float* out, int iters, float a, float b) {
  float x0 = threadIdx.x, x1 = x0 + 1.f, x2 = x0 + 2.f, x3 = x0 + 3.f, x4 = x0 + 4.f, x5 = x0 + 5.f, x6 = x0 + 6.f, x7 = x0 + 7.f;
#pragma unroll 1
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
      x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

// ================================================================================================ C ABI
// block sums of the blocked mean / covariance update, sized for the handle's nvar (19 MB at nvar = 192, 2.3 MB at 66)
static int mc_alloc(cemk_handle* h) {
  if (h->d_mc) { CK(cudaFree(h->d_mc)); h->d_mc = nullptr; }
  CK(cudaMalloc(&h->d_mc, sizeof(float) * mc_blocks(MC_BLOCKED_MAXK) * mc_stride(h->nvar)));
  return CEMK_OK;
}
// the rollout models the KM_NL-DOF arm of the KModel; a handle planning for another DOF count cannot feed it
static int rollout_dof_check(const cemk_handle* h, const char* fn) {
  if (h->ndof == KM_NL) return CEMK_OK;
  snprintf(g_err, sizeof g_err, "%s: DOF mismatch: the rollout models a %d-DOF arm, this handle plans for %d DOF (cemk_set_dof)",
           fn, KM_NL, h->ndof);
  return CEMK_ERR_ARG;
}

// One launch of the product rollout over a.B samples (cemk_rollout_cost, and cemk_step_states with STATES): grows the
// library scratch to a.B samples (the flags when a.flags is null, the previous distances, the spill area), points `a` at it
// and chooses the CTA shares.
template <bool STATES>
static int launch_rollout(cemk_handle* h, RolloutBatch& a, cudaStream_t st) {
  const int B = a.B;
  if (!a.flags) {
    if (h->flags_cap < B) {
      if (h->d_flags) CK(cudaFree(h->d_flags));
      CK(cudaMalloc(&h->d_flags, sizeof(int) * B));
      h->flags_cap = B;
    }
    a.flags = h->d_flags;
  }
  if (h->prevd_cap < B) {
    if (h->d_prevd) CK(cudaFree(h->d_prevd));
    CK(cudaMalloc(&h->d_prevd, sizeof(float) * (size_t)B * 2 * KM_NPASS * KW));
    if (h->d_ovf) CK(cudaFree(h->d_ovf));
    CK(cudaMalloc(&h->d_ovf, sizeof(float) * (size_t)B * (KM_NC_TOT - KM_NC_FAST) * KM_OVF_STRIDE));
    h->prevd_cap = B;
  }
  a.prevd = h->d_prevd;
  a.ovf = h->d_ovf;
  // Samples per CTA (a warp carries GPW = 32 / KW of them).  One CTA is resident per SM and its warps step
  // in lockstep, so the time of a wave grows with the warps per SM sub-partition (4 schedulers):
  //  * up to 4 / 8 warps-worth of samples per SM: the 4- / 8-warp instantiations (more registers per
  //    thread, latency-bound regime, e.g. the closed-loop config B = 1000);
  //  * one wave: every SM gets ceil(B / SMs) samples;
  //  * several waves: the ceil(B / SMs) samples an SM has to run are split into `waves` shares counted in
  //    units of 4 warps where that fits the CTA capacity, otherwise evenly.
  const int nsm = h->num_sms > 0 ? h->num_sms : 148;
  const int cap = ROLLOUT_WARPS * GPW, unit = 4 * GPW;
  int grid;
#define CEMK_LAUNCH_ROLLOUT(W_) k_rollout<KM_NC_FAST, W_, false, STATES><<<grid, (W_) * 32, rollout_smem<KM_NC_FAST, W_>(), st>>>(h->d_model, a)
  const int need = (B + nsm - 1) / nsm;                            // samples per SM
  if (h->cta_samples > 0) {
    const int w = h->cta_samples < cap ? h->cta_samples : cap;
    a.n_hi = 0; a.w_hi = a.w_lo = w; grid = (B + w - 1) / w;
    CEMK_LAUNCH_ROLLOUT(ROLLOUT_WARPS);
  } else if (need <= cap) {
    a.n_hi = 0; a.w_hi = a.w_lo = need; grid = (B + need - 1) / need;
    if (need <= 4 * GPW) CEMK_LAUNCH_ROLLOUT(4);
    else if (need <= 8 * GPW) CEMK_LAUNCH_ROLLOUT(8);
    else CEMK_LAUNCH_ROLLOUT(ROLLOUT_WARPS);
  } else {
    const int waves = (need + cap - 1) / cap;
    const int units = (need + unit - 1) / unit, u_lo = units / waves, r = units % waves;
    a.w_lo = unit * u_lo; a.w_hi = unit * (u_lo + (r ? 1 : 0)); a.n_hi = r * nsm;
    if (a.w_hi > cap || a.w_lo == 0) { a.n_hi = 0; a.w_hi = a.w_lo = (need + waves - 1) / waves; }
    const int rest = B - a.n_hi * a.w_hi;
    grid = a.n_hi + (rest > 0 ? (rest + a.w_lo - 1) / a.w_lo : 0);
    CEMK_LAUNCH_ROLLOUT(ROLLOUT_WARPS);
  }
#undef CEMK_LAUNCH_ROLLOUT
  h->launches += 1;
  return CEMK_OK;
}

extern "C" {

int cemk_version(void) { return 4; }
const char* cemk_last_error(void) { return g_err; }
int cemk_sizeof_kmodel(void) { return (int)sizeof(KModel); }

int cemk_create(const void* kmodel, int kmodel_bytes, int device, cemk_handle** out) {
  if (!kmodel || !out) return set_err(CEMK_ERR_ARG, "cemk_create: null argument");
  if (kmodel_bytes != (int)sizeof(KModel)) return set_err(CEMK_ERR_MODEL, "cemk_create: KModel size mismatch");
  const KModel* km = (const KModel*)kmodel;
  if (km->nl != KM_NL || km->ncap > KM_MAXCAP || km->nsbox > KM_MAXSBOX || km->nrpair > KM_MAXRPAIR || km->nbpair > KM_MAXBPAIR)
    return set_err(CEMK_ERR_MODEL, "cemk_create: unsupported topology");
  DevGuard guard(device);
  cemk_handle* h = new cemk_handle();
  h->device = device; h->ndof = KM_NL; h->ncoef = 11; h->nvar = KM_NL * 11; h->T = 0; h->d_G = nullptr; h->d_K = nullptr; h->launches = 0; h->d_flags = nullptr; h->flags_cap = 0; h->force_rerun = 0; h->cta_samples = 0; h->d_prevd = nullptr; h->prevd_cap = 0; h->d_ovf = nullptr;
  { cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, device)); h->num_sms = prop.multiProcessorCount; }
  CK(cudaMalloc(&h->d_model, sizeof(KModel)));
  CK(cudaMemcpy(h->d_model, kmodel, sizeof(KModel), cudaMemcpyHostToDevice));
  CK(cudaMalloc(&h->d_K, (MAXCOEF * MAXCOEF + 5 * MAXCOEF + 3) * sizeof(float)));
  CK(cudaFuncSetAttribute(k_rollout<KM_NC_FAST, ROLLOUT_WARPS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)rollout_smem<KM_NC_FAST, ROLLOUT_WARPS>()));
  CK(cudaFuncSetAttribute(k_rollout<KM_NC_FAST, 8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rollout_smem<KM_NC_FAST, 8>()));
  CK(cudaFuncSetAttribute(k_rollout<KM_NC_FAST, 4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rollout_smem<KM_NC_FAST, 4>()));
  CK(cudaFuncSetAttribute(k_rollout<KM_NC_FAST, ROLLOUT_WARPS, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)rollout_smem<KM_NC_FAST, ROLLOUT_WARPS>()));
  CK(cudaFuncSetAttribute(k_rollout<KM_NC_FAST, 8, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rollout_smem<KM_NC_FAST, 8>()));
  CK(cudaFuncSetAttribute(k_rollout<KM_NC_FAST, 4, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rollout_smem<KM_NC_FAST, 4>()));
  CK(cudaFuncSetAttribute(k_rollout<KM_NC_BIG, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)rollout_smem<KM_NC_BIG, 1>()));
  h->d_mc = nullptr;
  { const int rc = mc_alloc(h); if (rc) return rc; }
  CK(cudaFuncSetAttribute(k_rank_select, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(unsigned long long) * RANK_MAXN)));
  CK(cudaFuncSetAttribute(k_sample, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sample_smem(MAXVAR)));
  CK(cudaFuncSetAttribute(k_chol_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)chol_wide_smem()));
  CK(cudaFuncSetAttribute(k_mc_partial_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mc_wide_smem()));
  CK(cudaFuncSetAttribute(k_merge_lists<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(unsigned) * MERGE_MAXKEYS)));
  *out = h;
  return CEMK_OK;
}
int cemk_destroy(cemk_handle* h) {
  if (!h) return CEMK_OK;
  DevGuard guard(h->device);
  cudaFree(h->d_model); cudaFree(h->d_G); cudaFree(h->d_K); cudaFree(h->d_flags); cudaFree(h->d_prevd); cudaFree(h->d_ovf); cudaFree(h->d_mc);
  delete h;
  return CEMK_OK;
}
int cemk_set_model(cemk_handle* h, const void* kmodel, int kmodel_bytes) {
  if (!h || !kmodel) return set_err(CEMK_ERR_ARG, "cemk_set_model: null argument");
  if (kmodel_bytes != (int)sizeof(KModel)) return set_err(CEMK_ERR_MODEL, "cemk_set_model: KModel size mismatch");
  DevGuard guard(h->device);
  CK(cudaMemcpy(h->d_model, kmodel, sizeof(KModel), cudaMemcpyHostToDevice));
  return CEMK_OK;
}
int cemk_set_dof(cemk_handle* h, int ndof) {
  if (!h) return set_err(CEMK_ERR_ARG, "cemk_set_dof: null handle");
  if (ndof < 1 || ndof > MAXDOF) return set_err(CEMK_ERR_ARG, "cemk_set_dof: DOF count out of range [1, 12]");
  DevGuard guard(h->device);
  if (h->d_G) { CK(cudaFree(h->d_G)); h->d_G = nullptr; }     // the horizon tables belong to the old width
  h->T = 0;
  h->ndof = ndof; h->nvar = ndof * h->ncoef;
  return mc_alloc(h);
}
int cemk_set_order(cemk_handle* h, int ncoef) {
  if (!h) return set_err(CEMK_ERR_ARG, "cemk_set_order: null handle");
  if (ncoef < MINCOEF || ncoef > MAXCOEF) return set_err(CEMK_ERR_ARG, "cemk_set_order: coefficients per DOF out of range [4, 16]");
  DevGuard guard(h->device);
  if (h->d_G) { CK(cudaFree(h->d_G)); h->d_G = nullptr; }     // the horizon tables belong to the old order
  h->T = 0;
  h->ncoef = ncoef; h->nvar = h->ndof * ncoef;
  return mc_alloc(h);
}
int cemk_set_horizon(cemk_handle* h, int T, const float* G, const float* Kpp, const float* Kpe, const float* bounds3) {
  if (!h || !G || !Kpp || !Kpe || !bounds3) return set_err(CEMK_ERR_ARG, "cemk_set_horizon: null argument");
  if (T < 2 || T > 1024) return set_err(CEMK_ERR_ARG, "cemk_set_horizon: T out of range [2, 1024]");
  const int nc = h->ncoef;
  // every check before the first change: a refused horizon leaves the handle's tables and T as they were
  int smem = 0;
  CEMK_FOR_NCOEF(nc, { smem = project_smem<NC>(T, 32 * PROJ_WARPS); });
  if (smem > 227 * 1024) return set_err(CEMK_ERR_ARG, "cemk_set_horizon: horizon too long for the projection kernel's shared memory");
  DevGuard guard(h->device);
  if (h->d_G) { CK(cudaFree(h->d_G)); h->d_G = nullptr; }
  CK(cudaMalloc(&h->d_G, sizeof(float) * 3 * T * nc));
  CK(cudaMemcpy(h->d_G, G, sizeof(float) * 3 * T * nc, cudaMemcpyHostToDevice));
  float kc[MAXCOEF * MAXCOEF + 5 * MAXCOEF + 3];
  memcpy(kc, Kpp, nc * nc * 4); memcpy(kc + nc * nc, Kpe, nc * 5 * 4); memcpy(kc + nc * nc + nc * 5, bounds3, 12);
  CK(cudaMemcpy(h->d_K, kc, (nc * nc + nc * 5 + 3) * sizeof(float), cudaMemcpyHostToDevice));
  h->T = T;
  const int carve = 100 * PROJ_MINB * smem / (228 * 1024) + 8;                       // room for PROJ_MINB CTAs per SM, in percent
  CEMK_FOR_NCOEF(nc, { CK(cudaFuncSetAttribute(k_project<NC, KM_NL>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
                       CK(cudaFuncSetAttribute(k_project<NC, KM_NL>, cudaFuncAttributePreferredSharedMemoryCarveout, carve > 100 ? 100 : carve));
                       CK(cudaFuncSetAttribute(k_project<NC, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
                       CK(cudaFuncSetAttribute(k_project<NC, 0>, cudaFuncAttributePreferredSharedMemoryCarveout, carve > 100 ? 100 : carve)); });
  return CEMK_OK;
}

int cemk_sample(cemk_handle* h, int B, const float* z, const float* mean, const float* cov, float* chol_ws, float* xi, void* stream) {
  if (!h || !z || !mean || !cov || !chol_ws || !xi || B <= 0) return set_err(CEMK_ERR_ARG, "cemk_sample: bad argument");
  DevGuard guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (h->nvar <= CHOL_SMALL_N) k_chol66<<<1, 256, 0, st>>>(h->nvar, cov, chol_ws);
  else k_chol_wide<<<1, 256, chol_wide_smem(), st>>>(h->nvar, cov, chol_ws);
  k_sample<<<(B + SAMPLE_TILE - 1) / SAMPLE_TILE, SAMPLE_THREADS, sample_smem(h->nvar), st>>>(B, h->nvar, z, mean, chol_ws, xi);
  h->launches += 2;
  CK(cudaPeekAtLastError());
  return CEMK_OK;
}

int cemk_jax_normal(cemk_handle* h, unsigned key0, unsigned key1, int original, unsigned total, unsigned offset, unsigned count,
                    float* out, void* stream) {
  if (!h || !out || count == 0 || offset > total || count > total - offset) return set_err(CEMK_ERR_ARG, "cemk_jax_normal: bad argument");
  DevGuard guard(h->device);
  k_jax_normal<<<(count + 255) / 256, 256, 0, (cudaStream_t)stream>>>(key0, key1, original, total, offset, count, out);
  h->launches += 1;
  CK(cudaPeekAtLastError());
  return CEMK_OK;
}

int cemk_project(cemk_handle* h, int B, int iters, const float* xi, const float* state_term, float* xi_f, float* thetadot, void* stream) {
  if (!h || !xi || !state_term || !xi_f || B <= 0 || iters < 1) return set_err(CEMK_ERR_ARG, "cemk_project: bad argument");
  DevGuard guard(h->device);
  if (!h->d_G) return set_err(CEMK_ERR_ARG, "cemk_project: cemk_set_horizon has not been called");
  const int T = h->T;
  const int nprob = B * h->ndof, wpc = project_warps(nprob), warps = (nprob + PROJ_PPW - 1) / PROJ_PPW;
  const int grid = (warps + wpc - 1) / wpc;
  if (h->ndof == KM_NL)
    CEMK_FOR_NCOEF(h->ncoef, (k_project<NC, KM_NL><<<grid, 32 * wpc, project_smem<NC>(T, 32 * wpc), (cudaStream_t)stream>>>(
                                  B, h->ndof, T, iters, h->d_G, h->d_K, xi, state_term, xi_f, thetadot)))
  else
    CEMK_FOR_NCOEF(h->ncoef, (k_project<NC, 0><<<grid, 32 * wpc, project_smem<NC>(T, 32 * wpc), (cudaStream_t)stream>>>(
                                  B, h->ndof, T, iters, h->d_G, h->d_K, xi, state_term, xi_f, thetadot)))
  h->launches += 1;
  CK(cudaPeekAtLastError());
  return CEMK_OK;
}

int cemk_rollout_cost(cemk_handle* h, int B, int T, const float* thetadot, const float* q0, const float* v0, const float* target_pos,
                      const float* target_rot, float w_pos, float w_rot, float w_col, float* theta, float* cost4, float* eef_pos,
                      float* eef_rot, float* collision, float* qacc, int* flags, void* stream) {
  if (!h || !thetadot || !q0 || !v0 || !target_pos || !target_rot || !theta || !cost4 || B <= 0 || T <= 0)
    return set_err(CEMK_ERR_ARG, "cemk_rollout_cost: bad argument");
  { const int rc = rollout_dof_check(h, "cemk_rollout_cost"); if (rc) return rc; }
  DevGuard guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  RolloutBatch a = {};
  a.B = B; a.T = T; a.thetadot = thetadot; a.q0 = q0; a.v0 = v0; a.target_pos = target_pos; a.target_rot = target_rot;
  a.w_pos = w_pos; a.w_rot = w_rot; a.w_col = w_col;
  a.theta = theta; a.cost4 = cost4; a.eef_pos = eef_pos; a.eef_rot = eef_rot; a.collision = collision; a.qacc = qacc; a.flags = flags;
  { const int rc = launch_rollout<false>(h, a, st); if (rc) return rc; }
  // debug option: recompute every sample with the all-in-shared-memory instantiation (no spill area)
  if (h->force_rerun) {
    CK(cudaMemsetAsync(a.flags, 1, sizeof(int) * B, st));                      // 0x01010101: bit 0 set
    a.n_hi = 0; a.w_hi = a.w_lo = GPW;
    k_rollout<KM_NC_BIG, 1, true><<<(B + GPW - 1) / GPW, 32, rollout_smem<KM_NC_BIG, 1>(), st>>>(h->d_model, a);
    h->launches += 1;
  }
  CK(cudaPeekAtLastError());
  return CEMK_OK;
}

// force_rerun does not apply here: it re-reads the samples' inputs after the product launch, and with in-place outputs
// those rows already hold the stepped states.
int cemk_step_states(cemk_handle* h, int N, int T, const float* qpos, const float* qvel, const float* warm, const float* thetadot,
                     float* qpos_out, float* qvel_out, float* warm_out, float* theta, float* eef_pos, float* eef_rot, float* collision,
                     float* qacc, int* flags, void* stream) {
  if (!h || !qpos || !qvel || !warm || !qpos_out || !qvel_out || !warm_out || N <= 0 || T <= 0)
    return set_err(CEMK_ERR_ARG, "cemk_step_states: bad argument");
  if (!thetadot && T > 1) return set_err(CEMK_ERR_ARG, "cemk_step_states: thetadot may only be NULL with T = 1");
  { const int rc = rollout_dof_check(h, "cemk_step_states"); if (rc) return rc; }
  DevGuard guard(h->device);
  RolloutBatch a = {};
  a.B = N; a.T = T; a.thetadot = thetadot; a.q0 = qpos; a.v0 = qvel; a.warm = warm;
  a.qpos_out = qpos_out; a.qvel_out = qvel_out; a.warm_out = warm_out;
  a.theta = theta; a.eef_pos = eef_pos; a.eef_rot = eef_rot; a.collision = collision; a.qacc = qacc; a.flags = flags;
  { const int rc = launch_rollout<true>(h, a, (cudaStream_t)stream); if (rc) return rc; }
  CK(cudaPeekAtLastError());
  return CEMK_OK;
}

int cemk_cost_batch(cemk_handle* h, int B, int T, int nslot, const float* eef_pos, const float* eef_rot, const float* collision,
                    const float* target_pos, const float* target_rot, float w_pos, float w_rot, float w_col, float* cost4, void* stream) {
  if (!h || !eef_pos || !eef_rot || !collision || !target_pos || !target_rot || !cost4 || B <= 0 || T <= 0 || nslot <= 0)
    return set_err(CEMK_ERR_ARG, "cemk_cost_batch: bad argument");
  DevGuard guard(h->device);
  k_cost_batch<<<(B * 32 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(B, T, nslot, eef_pos, eef_rot, collision, target_pos, target_rot, w_pos, w_rot, w_col, cost4);
  h->launches += 1;
  CK(cudaPeekAtLastError());
  return CEMK_OK;
}

// npow2 >= SORT_BLK: only called above RANK_MAXN
static void sort_keys(cemk_handle* h, int npow2, unsigned long long* keys, cudaStream_t st) {
  const int nblk = npow2 / SORT_BLK;
  k_bitonic_local4<<<nblk, SORT_BLK / 4, 0, st>>>(keys, 0, 1);
  h->launches += 1;
  for (int k = 2 * SORT_BLK; k <= npow2; k <<= 1) {
    for (int j = k >> 1; j >= SORT_BLK; j >>= 1) {
      k_bitonic_global<<<(npow2 / 2 + 255) / 256, 256, 0, st>>>(keys, npow2, k, j);
      h->launches += 1;
    }
    k_bitonic_local4<<<nblk, SORT_BLK / 4, 0, st>>>(keys, k, 0);
    h->launches += 1;
  }
}
static int next_pow2(int n) { int p = 1; while (p < n) p <<= 1; return p; }

// The stable top-k of cost behind cemk_argsort_topk (pack null) and cemk_topk_pack (pack given, xi_elite / cost_elite /
// idx_sorted null): one counting-rank launch up to RANK_MAXN keys, else key generation + the bitonic sort + the gather.
static int select_topk(cemk_handle* h, int n, const float* cost, int stride, int idx_base, unsigned long long* keys, int* idx_sorted, int k,
                       const float* xi, float* xi_elite, float* cost_elite, float* pack, cudaStream_t st) {
  const int NVAR = h->nvar;
  if (n <= RANK_MAXN) {
    k_rank_select<<<(n + RANK_CAND - 1) / RANK_CAND, RANK_THREADS, sizeof(unsigned long long) * n, st>>>(NVAR, n, cost, stride, idx_base, keys, idx_sorted,
                                                                                                       k, xi, xi_elite, cost_elite, pack);
    h->launches += 1;
  } else {
    const int np2 = next_pow2(n);
    k_make_keys<<<(np2 + 255) / 256, 256, 0, st>>>(n, np2, cost, stride, keys);
    h->launches += 1;
    sort_keys(h, np2, keys, st);
    const int work = pack ? k * (NVAR + 2) : (n > k * NVAR ? n : k * NVAR);
    k_gather_sorted<<<(work + 255) / 256, 256, 0, st>>>(NVAR, n, keys, idx_base, idx_sorted, k, cost, stride, xi, xi_elite, cost_elite, pack);
    h->launches += 1;
  }
  CK(cudaPeekAtLastError());
  return CEMK_OK;
}

int cemk_argsort_topk(cemk_handle* h, int n, const float* cost, int cost_stride, int idx_base, unsigned long long* keys_ws,
                      int* idx_sorted, int k, const float* xi, float* xi_elite, float* cost_elite, void* stream) {
  if (!h || !cost || !keys_ws || n <= 0 || k < 0 || k > n || cost_stride < 1) return set_err(CEMK_ERR_ARG, "cemk_argsort_topk: bad argument");
  DevGuard guard(h->device);
  if (k > 0 && (!xi || !xi_elite || !cost_elite)) return set_err(CEMK_ERR_ARG, "cemk_argsort_topk: elite buffers missing");
  return select_topk(h, n, cost, cost_stride, idx_base, keys_ws, idx_sorted, k, xi, xi_elite, cost_elite, nullptr, (cudaStream_t)stream);
}

int cemk_topk_pack(cemk_handle* h, int n, const float* cost, int cost_stride, int idx_base, unsigned long long* keys_ws, int k,
                   const float* xi, float* pack, void* stream) {
  if (!h || !cost || !keys_ws || !xi || !pack || n <= 0 || k <= 0 || k > n || cost_stride < 1)
    return set_err(CEMK_ERR_ARG, "cemk_topk_pack: bad argument");
  DevGuard guard(h->device);
  return select_topk(h, n, cost, cost_stride, idx_base, keys_ws, nullptr, k, xi, nullptr, nullptr, pack, (cudaStream_t)stream);
}

int cemk_merge_sorted_lists(cemk_handle* h, int nlist, int kl, const float* packed, int k, float* xi_elite, float* cost_elite,
                            int* gidx_elite, void* stream) {
  if (!h || !packed || !xi_elite || !cost_elite || !gidx_elite || nlist <= 0 || kl <= 0 || k <= 0 || k > nlist * kl)
    return set_err(CEMK_ERR_ARG, "cemk_merge_sorted_lists: bad argument");
  DevGuard guard(h->device);
  const int n = nlist * kl;
  if (n <= MERGE_MAXKEYS)
    k_merge_lists<true><<<(n + MERGE_THREADS - 1) / MERGE_THREADS, MERGE_THREADS, sizeof(unsigned) * n, (cudaStream_t)stream>>>(h->nvar, nlist, kl, k, packed, xi_elite, cost_elite, gidx_elite);
  else
    k_merge_lists<false><<<(n + MERGE_THREADS - 1) / MERGE_THREADS, MERGE_THREADS, 0, (cudaStream_t)stream>>>(h->nvar, nlist, kl, k, packed, xi_elite, cost_elite, gidx_elite);
  h->launches += 1;
  CK(cudaPeekAtLastError());
  return CEMK_OK;
}

int cemk_mean_cov(cemk_handle* h, int k, const float* cost_elite, const float* xi_elite, const float* mean_prev, const float* cov_prev,
                  float lamda, float alpha_mean, float alpha_cov, float* mean_out, float* cov_out, void* stream) {
  if (!h || !cost_elite || !xi_elite || !mean_prev || !cov_prev || !mean_out || !cov_out || k <= 0)
    return set_err(CEMK_ERR_ARG, "cemk_mean_cov: bad argument");
  DevGuard guard(h->device);
  if (k >= MC_BLOCKED_MINK && k <= MC_BLOCKED_MAXK) {
    const int nblk = mc_blocks(k);
    if (h->nvar < MC_LD_SMALL)
      k_mc_partial<<<nblk, 256, 0, (cudaStream_t)stream>>>(h->nvar, k, cost_elite, xi_elite, mean_prev, lamda, h->d_mc);
    else
      k_mc_partial_wide<<<nblk, 256, mc_wide_smem(), (cudaStream_t)stream>>>(h->nvar, k, cost_elite, xi_elite, mean_prev, lamda, h->d_mc);
    if (h->nvar < 128)
      k_mc_finish<128><<<h->nvar, 128, 0, (cudaStream_t)stream>>>(h->nvar, nblk, h->d_mc, mean_prev, cov_prev, alpha_mean, alpha_cov, mean_out, cov_out);
    else
      k_mc_finish<256><<<h->nvar, 256, 0, (cudaStream_t)stream>>>(h->nvar, nblk, h->d_mc, mean_prev, cov_prev, alpha_mean, alpha_cov, mean_out, cov_out);
    h->launches += 2;
    CK(cudaPeekAtLastError());
    return CEMK_OK;
  }
  k_mean_cov<<<h->nvar, MC_THREADS, 0, (cudaStream_t)stream>>>(h->nvar, k, cost_elite, xi_elite, mean_prev, cov_prev, lamda, alpha_mean, alpha_cov, mean_out, cov_out);
  h->launches += 1;
  CK(cudaPeekAtLastError());
  return CEMK_OK;
}

// ---------------------------------------------------------------------------------------------- tick record
// What compute_cem (mjx_planner.py:390-404) keeps of an iteration, written straight into the tick's packed result
//   out = [cost_min[n_iter] | best thetadot[6T] | best theta[6T] | cost_g, cost_r, cost_c | xi_mean[nvar] | overflow count]
// (one D2H copy at the end of the tick): iteration `iter` stores the smallest (global) cost and adds the number of samples whose
// contacts overflowed the rollout kernel's capacity (flags bit 0); the last iteration also stores the new mean and the best
// sample's rows -- the head of the sorted elite list, local row gbest - idx_base.  With several GPUs only the owning rank
// has that row: the segment then goes to `best_row` (6T + 6T + 3 floats), exact zeros on the other ranks, for the caller's
// all-reduce.  Replaces a dozen framework kernels (index, cat, reduce, copies) per tick.
__global__ void __launch_bounds__(256) k_tick_record(int NVAR, int iter, int n_iter, int last, int B, int T, const float* __restrict__ cost_elite,
                                                     const int* __restrict__ gidx_elite, int idx_base, const int* __restrict__ flags,
                                                     const float* __restrict__ thetadot, const float* __restrict__ theta,
                                                     const float* __restrict__ cost4, const float* __restrict__ xi_mean,
                                                     float* __restrict__ out, float* __restrict__ best_row) {
  __shared__ int red[256];
  const int tid = threadIdx.x, nd = KM_NL * T;
  int c = 0;
  for (int i = tid; i < B; i += 256) c += flags[i] & 1;
  red[tid] = c; __syncthreads();
  for (int o = 128; o; o >>= 1) { if (tid < o) red[tid] += red[tid + o]; __syncthreads(); }
  float* ovf = out + n_iter + 2 * nd + 3 + NVAR;
  if (tid == 0) {
    out[iter] = cost_elite[0];
    *ovf = (iter == 0 ? 0.f : *ovf) + (float)red[0];
  }
  if (!last) return;
  for (int e = tid; e < NVAR; e += 256) out[n_iter + 2 * nd + 3 + e] = xi_mean[e];
  const int li = gidx_elite[0] - idx_base;
  const bool own = li >= 0 && li < B;
  float* dst = best_row ? best_row : out + n_iter;
  for (int e = tid; e < 2 * nd + 3; e += 256) {
    float v = 0.f;
    if (own) v = e < nd ? thetadot[(size_t)li * nd + e] : (e < 2 * nd ? theta[(size_t)li * nd + (e - nd)] : cost4[(size_t)li * 4 + 1 + (e - 2 * nd)]);
    dst[e] = v;
  }
}
int cemk_tick_record(cemk_handle* h, int iter, int n_iter, int last, int B, int T, const float* cost_elite, const int* gidx_elite, int idx_base,
                     const int* flags, const float* thetadot, const float* theta, const float* cost4, const float* xi_mean, float* out,
                     float* best_row, void* stream) {
  if (!h || !cost_elite || !gidx_elite || !flags || !thetadot || !theta || !cost4 || !xi_mean || !out || iter < 0 || iter >= n_iter || B <= 0 || T <= 0)
    return set_err(CEMK_ERR_ARG, "cemk_tick_record: bad argument");
  { const int rc = rollout_dof_check(h, "cemk_tick_record"); if (rc) return rc; }
  DevGuard guard(h->device);
  k_tick_record<<<1, 256, 0, (cudaStream_t)stream>>>(h->nvar, iter, n_iter, last, B, T, cost_elite, gidx_elite, idx_base, flags, thetadot, theta, cost4,
                                                    xi_mean, out, best_row);
  h->launches += 1;
  CK(cudaPeekAtLastError());
  return CEMK_OK;
}

long long cemk_launch_count(cemk_handle* h) { return h ? h->launches : 0; }

int cemk_set_option(cemk_handle* h, const char* name, int value) {
  if (!h || !name) return set_err(CEMK_ERR_ARG, "cemk_set_option: null argument");
  if (!strcmp(name, "force_rerun")) { h->force_rerun = value != 0; return CEMK_OK; }
  if (!strcmp(name, "cta_samples")) { h->cta_samples = value > 0 ? value : 0; return CEMK_OK; }
  return set_err(CEMK_ERR_ARG, "cemk_set_option: unknown option");
}

int cemk_fp32_fma_peak(cemk_handle* h, double* tflops) {
  if (!h || !tflops) return set_err(CEMK_ERR_ARG, "cemk_fp32_fma_peak: null argument");
  DevGuard guard(h->device);
  const int nsm = h->num_sms > 0 ? h->num_sms : 148, blocks = nsm * 8, threads = 256, iters = 4096;
  float* d = nullptr;
  CK(cudaMalloc(&d, sizeof(float) * blocks * threads));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    CK(cudaEventRecord(e0));
    k_fma_peak<<<blocks, threads>>>(d, iters, 0.999f, 0.001f);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    const double fl = 2.0 * 8 * 16 * (double)iters * blocks * threads;
    if (rep > 0 && fl / (ms * 1e-3) / 1e12 > best) best = fl / (ms * 1e-3) / 1e12;
  }
  h->launches += 5;
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
  *tflops = best;
  return CEMK_OK;
}

#ifdef CEMK_PHASE_TIMING
/* debug builds only: copy out and clear the per-phase clock table */
int cemk_debug_phase_clocks(unsigned long long* out24) {
  unsigned long long z[24] = {0};
  if (cudaMemcpyFromSymbol(out24, g_phase, sizeof z) != cudaSuccess) return CEMK_ERR_CUDA;
  if (cudaMemcpyToSymbol(g_phase, z, sizeof z) != cudaSuccess) return CEMK_ERR_CUDA;
  return CEMK_OK;
}
int cemk_debug_phase_cond(unsigned long long* out25) {
  unsigned long long z[25] = {0};
  if (cudaMemcpyFromSymbol(out25, g_phase_cond, sizeof z) != cudaSuccess) return CEMK_ERR_CUDA;
  if (cudaMemcpyToSymbol(g_phase_cond, z, sizeof z) != cudaSuccess) return CEMK_ERR_CUDA;
  return CEMK_OK;
}
int cemk_debug_events(unsigned long long* out24) {
  unsigned long long z[24] = {0};
  if (cudaMemcpyFromSymbol(out24, g_event, sizeof z) != cudaSuccess) return CEMK_ERR_CUDA;
  if (cudaMemcpyToSymbol(g_event, z, sizeof z) != cudaSuccess) return CEMK_ERR_CUDA;
  return CEMK_OK;
}
#endif

}  // extern "C"
