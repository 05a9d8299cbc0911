/*
 * cemk.h -- C ABI of libcemk.so, the sm_100a CUDA library behind the drop-in `cem_planner`.
 *
 * The reference exposes this path only as a Python class (there is no FFI in the reference); each
 * entry point below replaces one jitted method of `cem_planner`
 * (reference sampling_based_planner/mjx_planner.py) and is what a ctypes / JAX-FFI / cffi binding of
 * that class would call.  Conventions:
 *   - every function returns 0 on success, a negative cemk_status otherwise; nothing throws;
 *     cemk_last_error() returns a static description of the last failure on the calling thread;
 *   - all buffers are caller-owned DEVICE pointers (float32 / int32, row-major, shapes as in the
 *     reference method), kernels are enqueued on `stream` (a cudaStream_t passed as void*) and the
 *     call returns without synchronising;
 *   - one handle per device, not thread-safe per handle;
 *   - B = num_batch (samples on this GPU), T = num_steps, nd = num_dof (cemk_set_dof, default 6),
 *     nc = Bernstein coefficients per DOF (cemk_set_order, default 11), NV = nvar = nd * nc decision variables.
 *     "66", "30" and "6T" in the shapes below are NV, 5 nd and nd T at the defaults.
 *   - The planner algebra (sampling, projection, elite selection, mean / covariance) runs at any
 *     1 <= nd <= 12 and 4 <= nc <= 16 (NV <= 192).  The rollout (cemk_rollout_cost, cemk_step_states[_contacts], cemk_tick_record)
 *     models the 6-DOF arm of the KModel only and returns CEMK_ERR_ARG on a handle with nd != 6.
 */
#ifndef CEMK_H
#define CEMK_H
#ifdef __cplusplus
extern "C" {
#endif

typedef struct cemk_handle cemk_handle;

enum cemk_status {
  CEMK_OK = 0,
  CEMK_ERR_ARG = -1,      /* bad argument (null pointer, size out of range) */
  CEMK_ERR_CUDA = -2,     /* a CUDA runtime call failed */
  CEMK_ERR_MODEL = -3     /* model table has the wrong size / unsupported topology */
};

int cemk_version(void);
const char* cemk_last_error(void);
/* sizeof(KModel) this library was built with (host bindings assert their mirror matches). */
int cemk_sizeof_kmodel(void);

/* `kmodel`: host pointer to a KModel (csrc/kmodel.h; built by manipulator_mujoco_b200/kmodel.py from
 * the compiled MJCF).  Replaces mjx.put_model / put_data in cem_planner.__init__ (mjx_planner.py:100-107). */
int cemk_create(const void* kmodel, int kmodel_bytes, int device, cemk_handle** out);
int cemk_destroy(cemk_handle* h);
/* Update the rollout snapshot (qpos0 / warm0 / qvel0 of the KModel) after construction. */
int cemk_set_model(cemk_handle* h, const void* kmodel, int kmodel_bytes);

/* Degrees of freedom of the planner algebra, 1 <= nd <= 12 (cem_planner(num_dof=nd); default 6, the UR5e of the KModel).
 * nvar = nd nc.  Call before cemk_set_horizon (it discards the horizon tables). */
int cemk_set_dof(cemk_handle* h, int ndof);

/* Bernstein coefficients per DOF, nc = order + 1 (mjx_planner.py:40 calls bernstein_coeff_ordern_new(10, ...), i.e. nc = 11, the
 * default; SURVEY.md 8 f.4: arbitrary order n).  4 <= nc <= 16; nvar = nd nc is the width of every xi / mean / cov / elite array
 * below ("66" in their descriptions is the default nvar).  Call before cemk_set_horizon (it discards the horizon tables). */
int cemk_set_order(cemk_handle* h, int ncoef);

/* Per-horizon constants, host pointers, float32:
 *   G [3][T][nc] = Pdot, Pddot, P (bernstein_coeff_ordern_new, mjx_planner.py:40);
 *   Kpp [nc][nc], Kpe [nc][5] = per-DOF blocks of Q_inv (mjx_planner.py:166-172, block diagonal per DOF);
 *   bounds = v_max, a_max, p_max (mjx_planner.py:84-86).
 * 2 <= T <= 1024, and the projection kernel's shared memory (3 T pc + nc pc + 4 ceil((5 nc + 3) / 4) + 672 nc floats,
 * pc = 4 ceil(nc / 4)) must fit 227 KB: T <= 979 at nc = 16.  CEMK_ERR_ARG otherwise, with the handle unchanged. */
int cemk_set_horizon(cemk_handle* h, int T, const float* G, const float* Kpp, const float* Kpe, const float* bounds3);

/* compute_xi_samples (mjx_planner.py:313-316) with the standard-normal draws injected:
 *   xi[B][66] = mean[66] + z[B][66] . chol(cov[66][66] + 0.003 I)^T.   `chol_ws` [66*66] scratch. */
int cemk_sample(cemk_handle* h, int B, const float* z, const float* mean, const float* cov, float* chol_ws, float* xi,
                void* stream);

/* The standard-normal draws of jax.random.multivariate_normal (mjx_planner.py:315; jax==0.5.3, requirements.txt:9):
 *   out[i] = jax.random.normal(key, (total,), float32)[offset + i], i < count, for the raw threefry key
 *   (key0, key1).  `original` = 0: jax_threefry_partitionable (default since jax 0.5), 1: the older layout.
 *   A [B][66] table is total = B*66, row-major; a rank fills its rows with offset = first_row*66. */
int cemk_jax_normal(cemk_handle* h, unsigned key0, unsigned key1, int original, unsigned total, unsigned offset,
                    unsigned count, float* out, void* stream);

/* compute_projection_filter (mjx_planner.py:234-249) + Bernstein evaluation (mjx_planner.py:348):
 *   xi[B][NV], state_term[B][5 nd] -> xi_f[B][NV]; thetadot[B][nd*T] (index dof*T + t) when non-null. */
int cemk_project(cemk_handle* h, int B, int maxiter_projection, const float* xi, const float* state_term, float* xi_f,
                 float* thetadot, void* stream);

/* compute_rollout_batch + compute_cost_batch fused (mjx_planner.py:251-303):
 *   thetadot[B][6T], q0[6], v0[6], target_pos[3], target_rot[4] (device) ->
 *   theta[B][6T] (post-step joint angles, dof-major), cost4[B][4] = (cost, cost_g, cost_r, cost_c).
 *   Optional per-step dumps (pass NULL to skip): eef_pos[B][T][3], eef_rot[B][T][4],
 *   collision[B][T][nslot_robot] (pre-step, mjx_planner.py:259-261), qacc[B][T][12],
 *   flags[B] (bit 0: more than 48 simultaneously active contacts, extra ones dropped; up to 20 contacts of
 *   a sample live in shared memory, contacts 21..48 in a library-owned global spill area). */
int cemk_rollout_cost(cemk_handle* h, int B, int T, const float* thetadot, const float* q0, const float* v0,
                      const float* target_pos, const float* target_rot, float w_pos, float w_rot, float w_col,
                      float* theta, float* cost4, float* eef_pos, float* eef_rot, float* collision, float* qacc,
                      int* flags, void* stream);

/* vmap(mjx.step) over N environments, each from its own state, chained over T steps (the rollout body of
 * cemk_rollout_cost without the cost and without the handle's KModel snapshot, which is neither read nor changed):
 *   qpos[N][13], qvel[N][12], warm[N][12] (qacc_warmstart) -> qpos_out, qvel_out, warm_out (same shapes) after T steps.
 *   thetadot[N][6T] (dof-major as in cemk_rollout_cost) overwrites qvel[:6] before each step (mjx_planner.py:254); NULL is
 *   allowed with T = 1 only, each environment then keeps its own qvel[:6] (a plain mjx.step).  Outputs may be the inputs
 *   (in-place stepping).  warm_out is the last step's qacc.  Optional (NULL to skip): theta[N][6T] and the dumps and flags
 *   of cemk_rollout_cost.  A run split into chunks, each fed the previous chunk's outputs, gives the same bits as one call.
 *   CEMK_ERR_ARG for N <= 0, T <= 0, a missing state pointer, NULL thetadot with T > 1, or a handle with nd != 6. */
int cemk_step_states(cemk_handle* h, int N, int T, const float* qpos, const float* qvel, const float* warm,
                     const float* thetadot, float* qpos_out, float* qvel_out, float* warm_out, float* theta,
                     float* eef_pos, float* eef_rot, float* collision, float* qacc, int* flags, void* stream);

/* Contacts a step keeps per environment, and floats per contact record of cemk_step_states_contacts. */
#define CEMK_MAX_CONTACTS 48
#define CEMK_CONTACT_REC 12

/* cemk_step_states, plus what mjx.step's Data holds about the constraints of the last step (at the accepted qacc, MJX's
 * solver finish: f_r = -D_r (J_r qacc - aref_r) where that is negative, else 0):
 *   qfrc_constraint[N][12] = sum_r J_r^T f_r over the joint-limit and contact rows;
 *   ncon[N] = contacts kept (<= 48; flags bit 0 reports dropped ones);
 *   con_slot[N][48] = the model's contact-slot index of each contact, ascending, padded with -1;
 *   con_rec[N][48][CEMK_CONTACT_REC] = dist, pos[3], normal[3] (first row of the contact frame), force[3] (contact frame:
 *   normal, tangent 1, tangent 2, decoded from the four pyramid rows as mju_decodePyramid does), 2 unused; zeros as padding.
 * slot_map (device, int): the model's contact slot of each contact key of the KModel, [nslot_robot + 4 nbpair]; key k <
 * nslot_robot is robot slot k (the cost slots of cemk_rollout_cost, in model order), key nslot_robot + 4 q + j is slot j of
 * free-box pair q (bp_type order).  The KModel numbers its pairs but not the model's slots, hence the map.
 * slot_map and the four outputs are all given or all NULL (then this is cemk_step_states); CEMK_ERR_ARG for some but not
 * all, and for everything cemk_step_states refuses. */
int cemk_step_states_contacts(cemk_handle* h, int N, int T, const float* qpos, const float* qvel, const float* warm,
                              const float* thetadot, float* qpos_out, float* qvel_out, float* warm_out, float* theta,
                              float* eef_pos, float* eef_rot, float* collision, float* qacc, int* flags, const int* slot_map,
                              float* qfrc_constraint, int* ncon, int* con_slot, float* con_rec, void* stream);

/* Scenes and start states given per call.  The model's topology, sizes, pairs, floor plane and robot stay the handle's;
 * only the poses of the static boxes and the free box's start state become inputs (float32, device):
 *   scene record [CEMK_SCENE_FLOATS] = the KModel's sb_pos[8][4] | sb_mat[8][12] | sb_size[8][4] block: per static box its
 *     world position, rotation matrix (row-major) with its half sizes along the world axes in [9..11] when the box is
 *     axis-aligned, half sizes with [3] = 1 for an axis-aligned box; unused rows zero.  Build it with
 *     manipulator_mujoco_b200.kmodel.scene_records (cem_planner.make_scene): a hand-made record whose flag and world half
 *     sizes disagree with its rotation gives wrong far-field tests.
 *   start record [CEMK_START_FLOATS] = the KModel's qpos0[16] | warm0[12] | qvel0[12] block: qpos[13] (3 unused), qacc_warmstart[12],
 *     qvel[12].  A planner rollout takes the free box (qpos[6:13], qvel[6:12]) and the warm start from it; the arm still
 *     comes from q0 / v0.
 * The handle's table holds the default records, so a NULL record and the table's own give the same bits; nothing is stored
 * in the handle.
 * cemk_rollout_cost_scene: cemk_rollout_cost with a scene (sample s reads scene + s * scene_stride; scene_stride 0 = one
 *   scene for all samples, or CEMK_SCENE_FLOATS) and a start record, each NULL for the handle's own.
 * cemk_step_states_scene: cemk_step_states_contacts with per-environment (scene_stride CEMK_SCENE_FLOATS) or shared (0)
 *   scenes, NULL for the handle's own.  The environments' state rows hold their start state.
 * Both refuse what the calls they extend refuse, and a scene_stride other than 0 or CEMK_SCENE_FLOATS (CEMK_ERR_ARG). */
#define CEMK_SCENE_FLOATS 160
#define CEMK_START_FLOATS 40
int cemk_rollout_cost_scene(cemk_handle* h, int B, int T, const float* thetadot, const float* q0, const float* v0,
                            const float* target_pos, const float* target_rot, float w_pos, float w_rot, float w_col,
                            float* theta, float* cost4, float* eef_pos, float* eef_rot, float* collision, float* qacc,
                            int* flags, const float* scene, int scene_stride, const float* start, void* stream);
int cemk_step_states_scene(cemk_handle* h, int N, int T, const float* qpos, const float* qvel, const float* warm,
                           const float* thetadot, float* qpos_out, float* qvel_out, float* warm_out, float* theta,
                           float* eef_pos, float* eef_rot, float* collision, float* qacc, int* flags, const int* slot_map,
                           float* qfrc_constraint, int* ncon, int* con_slot, float* con_rec, const float* scene, int scene_stride,
                           void* stream);

/* compute_cost_batch alone (mjx_planner.py:277-303), per-sample targets as in the reference method:
 *   eef_pos[B][T][3], eef_rot[B][T][4], collision[B][T][nslot], target_pos[B][3], target_rot[B][4] -> cost4[B][4]. */
int cemk_cost_batch(cemk_handle* h, int B, int T, int nslot, const float* eef_pos, const float* eef_rot,
                    const float* collision, const float* target_pos, const float* target_rot, float w_pos, float w_rot,
                    float w_col, float* cost4, void* stream);

/* compute_ellite_samples (mjx_planner.py:306-310): stable ascending argsort of cost (NaN last, -0.0 ties with
 * +0.0, ties by lower index).  cost is read with stride `cost_stride` floats.  keys_ws: [n_pow2] uint64 scratch
 * (n_pow2 = next power of two >= n).  idx_base is added to every index (global sample index of this
 * shard).  Outputs: idx_sorted[n] (int32, global indices), and when k > 0 the k best rows gathered:
 * xi_elite[k][66] from xi[n][66] (local rows), cost_elite[k]. */
int cemk_argsort_topk(cemk_handle* h, int n, const float* cost, int cost_stride, int idx_base, unsigned long long* keys_ws,
                      int* idx_sorted, int k, const float* xi, float* xi_elite, float* cost_elite, void* stream);

/* The two halves of the multi-GPU form of compute_ellite_samples without intermediate tensors.
 * cemk_topk_pack: this rank's k best samples, sorted as above, as exchange records pack[k][68] = xi[66], cost, global index
 * (idx_base + local row, stored as float: exact below 2^24) -- the send buffer of the NCCL all-gather, and what
 * cemk_merge_sorted_lists consumes.  keys_ws as above.
 * cemk_merge_sorted_lists: the all-gathered `nlist` blocks of `kl` such records (rank-major) -> the k best by (cost, row) =
 * (cost, global index).  No sort: every record finds its global position by binary searches in the other blocks (one launch). */
int cemk_topk_pack(cemk_handle* h, int n, const float* cost, int cost_stride, int idx_base, unsigned long long* keys_ws, int k,
                   const float* xi, float* pack, void* stream);
int cemk_merge_sorted_lists(cemk_handle* h, int nlist, int kl, const float* packed, int k, float* xi_elite, float* cost_elite,
                            int* gidx_elite, void* stream);

/* compute_mean_cov (mjx_planner.py:326-335): k elites -> mean_out[66], cov_out[66][66]. */
int cemk_mean_cov(cemk_handle* h, int k, const float* cost_elite, const float* xi_elite, const float* mean_prev,
                  const float* cov_prev, float lamda, float alpha_mean, float alpha_cov, float* mean_out, float* cov_out,
                  void* stream);

/* What compute_cem keeps of CEM iteration `iter` of `n_iter` (mjx_planner.py:390-404), written into the tick's packed result
 *   out = [cost_min[n_iter] | best thetadot[6T] | best theta[6T] | cost_g, cost_r, cost_c | xi_mean[nvar] | overflow count]
 * (floats; the planner copies it to the host once per tick): out[iter] = cost_elite[0], the overflow count grows by the number of
 * rollouts of this iteration whose contacts exceeded the kernel's capacity (flags bit 0), and when `last` is set the new mean and
 * the rows of the best sample -- local row gidx_elite[0] - idx_base of thetadot / theta [B][6T] and cost4 [B][4] -- are stored.
 * best_row != NULL (several GPUs): the 12T + 3 best-sample floats go there instead, exact zeros when the row is not on this
 * rank, for the caller's all-reduce. */
int cemk_tick_record(cemk_handle* h, int iter, int n_iter, int last, int B, int T, const float* cost_elite, const int* gidx_elite,
                     int idx_base, const int* flags, const float* thetadot, const float* theta, const float* cost4,
                     const float* xi_mean, float* out, float* best_row, void* stream);

/* Options.  "force_rerun" (0/1): recompute every sample with the rollout instantiation that keeps all 48
 * contacts in shared memory, used by the tests to check that it agrees bit for bit with the fast kernel
 * and its spill area.  Any other name returns CEMK_ERR_ARG. */
int cemk_set_option(cemk_handle* h, const char* name, int value);

/* Calibration: measured FP32 FMA throughput (TFLOP/s, register operands) of the handle's device; synchronous.
 * bench.py uses it as the measured denominator of the rollout kernel's FP32 roofline. */
int cemk_fp32_fma_peak(cemk_handle* h, double* tflops);

/* Number of kernels this library has launched since cemk_create (bench.py's gpu_launches). */
long long cemk_launch_count(cemk_handle* h);

#ifdef __cplusplus
}
#endif
#endif
