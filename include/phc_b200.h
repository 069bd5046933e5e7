/*
 * phc_b200.h — C ABI of the B200-native PHC step path (libphc_b200.so).
 *
 * The reference (howird/humanoid, packages/puffer-phc) has no FFI for this path: the
 * boundary is a set of plain Python call signatures (SURVEY.md §8(b)).  Each entry point
 * below is the native function the Python drop-in of one of those signatures binds with
 * ctypes; the reference interface it replaces is cited as file:line relative to
 * packages/puffer-phc/puffer_phc/.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name says host; fp32 unless typed;
 *     quaternions are xyzw;
 *   - nothing is allocated, retained or freed on behalf of the caller except the opaque
 *     handles (PhcLib borrows the motion tensors; the caller keeps them alive);
 *   - all functions return 0 on success and a negative PHC_ERR_* code otherwise, never
 *     throw, never synchronise (except phc_host_step and phc_host_step_wait, which return when
 *     the host buffers are filled) and launch on the stream passed last, so they can be captured
 *     in a CUDA graph;
 *   - views of rigid-body state carry element strides so that the reference's stride-13
 *     AoS views (envs/humanoid_phc.py:542-549) and contiguous tensors both work; the last
 *     dimension (3 or 4 floats) must be contiguous.
 */
#ifndef PHC_B200_H_
#define PHC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PHC_ABI_VERSION 6 /* 6: PhcHostResetArgs, phc_host_step_submit_reset / phc_host_reset_submit; 5: phc_host_step_submit / phc_host_step_wait, PHC_ERR_BUSY; 4: PhcResetArgs grew (initial_*, default_mask: StateInit.Default / Hybrid); 3: PhcStepArgs grew (rew_out, reset_out, terminate_out, auto_reset, ref_dof_pos, obs_flags), PhcResetArgs grew (obs_norm*, obs_moments*),
                              phc_action_to_pd_targets takes the action clip; 2: obs_moments_buckets, ep_*, phc_motion_build / phc_peer_reduce_* / phc_episode_fold */
#define PHC_NUM_BODIES 24      /* SMPL humanoid, body_sets.py:11-36 */
#define PHC_SELF_OBS_DIM 358   /* envs/humanoid_phc.py:461 */
#define PHC_TASK_OBS_DIM 576   /* per future step, envs/humanoid_phc.py:464 */
#define PHC_MAX_TIME_STEPS 16

typedef struct CUstream_st* phc_stream_t; /* == cudaStream_t */

#if defined(__GNUC__)
#define PHC_API __attribute__((visibility("default")))
#else
#define PHC_API
#endif

enum {
  PHC_OK = 0,
  PHC_ERR_NULL = -1,        /* required pointer is NULL */
  PHC_ERR_SHAPE = -2,       /* size / count out of range */
  PHC_ERR_ALIGN = -3,       /* pointer or stride not aligned as required */
  PHC_ERR_UNSUPPORTED = -4, /* valid in the reference, not implemented here */
  PHC_ERR_CUDA = -5,        /* CUDA runtime error (phc_last_cuda_error() has the code) */
  PHC_ERR_ALLOC = -6,
  PHC_PEER_TIMEOUT = -7,    /* a peer rank did not publish its partials within the timeout */
  PHC_ERR_BUSY = -8         /* the host-step slot already has a step in flight */
};

PHC_API const char* phc_strerror(int code);
PHC_API int phc_abi_version(void);
PHC_API int phc_last_cuda_error(void); /* cudaError_t of the last PHC_ERR_CUDA on this thread */

/* ------------------------------------------------------------------------------------
 * Motion library — the tensor set MotionLibBase.load_motions leaves on the device
 * (motion_lib.py:396-420).  F = total frames of all clips, M = clips.
 * ---------------------------------------------------------------------------------- */
typedef struct PhcLibDesc {
  const float* gts;   /* [F,24,3] global translation            motion_lib.py:407 */
  const float* grs;   /* [F,24,4] global rotation                motion_lib.py:408 */
  const float* lrs;   /* [F,24,4] local rotation (may be NULL if dof_pos is never asked) */
  const float* gvs;   /* [F,24,3] global linear velocity         motion_lib.py:413 */
  const float* gavs;  /* [F,24,3] global angular velocity        motion_lib.py:412 */
  const float* dvs;   /* [F,23,3] dof velocity (may be NULL)     motion_lib.py:414 */
  const float* motion_aa;           /* [F,72] (may be NULL)      motion_lib.py:399 */
  const float* motion_lengths;      /* [M] seconds               motion_lib.py:396 */
  const int64_t* motion_num_frames; /* [M]                       motion_lib.py:402 */
  const float* motion_dt;           /* [M]                       motion_lib.py:401 */
  const int64_t* length_starts;     /* [M] first frame of clip   motion_lib.py:416-419 */
  const float* motion_bodies;       /* [M,17] (may be NULL)      motion_lib.py:398 */
  const float* motion_limb_weights; /* [M,10] (may be NULL)      motion_lib.py:403 */
  int64_t total_frames;             /* F */
  int64_t num_motions;              /* M */
} PhcLibDesc;

typedef struct PhcLib PhcLib;
PHC_API int phc_lib_create(const PhcLibDesc* desc, PhcLib** out);
PHC_API void phc_lib_destroy(PhcLib* lib);
/* (Re)build the library's packed frame table on `stream`: one 1248-B row per frame,
 * [gts 72 | grs 96 | gvs 72 | gavs 72] floats, owned by the handle (1248 B x F of HBM).  The
 * fused step's TMA fast path reads it; without it phc_step_fused uses the generic kernel on
 * the four reference tensors.  Call once after phc_lib_create and again whenever the caller rewrites
 * ANY library tensor in place (frames or per-clip metadata): the fast step kernel overlaps its prologue
 * with the previous kernel on the stream and reads the library before that kernel has finished, so it
 * must know when the library changed.  The first phc_step_fused after phc_lib_create / phc_lib_pack
 * launches without that overlap and therefore sees every write ordered before it on the stream. */
PHC_API int phc_lib_pack(PhcLib* lib, phc_stream_t stream);

/* [n, J, C] fp32 view, innermost C contiguous; strides in elements. */
typedef struct PhcView {
  const float* ptr;
  int64_t stride_env;
  int64_t stride_body;
} PhcView;

/* The four views the env hands to the path (envs/humanoid_phc.py:546-549). */
typedef struct PhcBodyState {
  PhcView pos;     /* [n,J,3] */
  PhcView rot;     /* [n,J,4] */
  PhcView vel;     /* [n,J,3] */
  PhcView ang_vel; /* [n,J,3] */
  int32_t num_bodies; /* J */
} PhcBodyState;

/* MotionLibBase._calc_frame_blend(time, len, num_frames, dt)      motion_lib.py:655-665 */
PHC_API int phc_calc_frame_blend(const float* time, const float* len, const int64_t* num_frames, const float* dt,
                         int64_t n, int64_t* frame_idx0, int64_t* frame_idx1, float* blend,
                         phc_stream_t stream);

/* Outputs of get_motion_state; any pointer may be NULL (that output is skipped).  All are
 * dense row-major with the shapes of the reference's dict (motion_lib.py:611-626). */
typedef struct PhcMotionOut {
  float* root_pos;            /* [n,3]    */
  float* root_rot;            /* [n,4]    */
  float* dof_pos;             /* [n,69]   */
  float* root_vel;            /* [n,3]    */
  float* root_ang_vel;        /* [n,3]    */
  float* dof_vel;             /* [n,69]   */
  float* motion_aa;           /* [n,72]   frame f0, not blended */
  float* rg_pos;              /* [n,24,3] */
  float* rb_rot;              /* [n,24,4] */
  float* body_vel;            /* [n,24,3] */
  float* body_ang_vel;        /* [n,24,3] */
  float* motion_bodies;       /* [n,17]   */
  float* motion_limb_weights; /* [n,10]   */
  int64_t* frame_idx0;        /* [n] clip-local, extra (for parity tests) */
  int64_t* frame_idx1;        /* [n] */
  float* blend;               /* [n] */
} PhcMotionOut;

/* MotionLibBase.get_motion_state(motion_ids, motion_times, offset=None)  motion_lib.py:549-626 */
PHC_API int phc_motion_state(const PhcLib* lib, const int64_t* motion_ids, const float* motion_times,
                     const float* offset_or_null /* [n,3] */, int64_t n, const PhcMotionOut* out,
                     phc_stream_t stream);

/* compute_humanoid_observations_smpl_max(...)                        envs/common.py:23-103
 * Writes [root_h? | local pos 3(J-1) | rot 6J | vel 3J | ang vel 3J] per row; the optional
 * smpl / limb-weight columns are appended by the caller (they are copies of inputs). */
#define PHC_OBS_LOCAL_ROOT 1u   /* local_root_obs   */
#define PHC_OBS_ROOT_HEIGHT 2u  /* root_height_obs  */
#define PHC_OBS_UPRIGHT 4u      /* upright          */
PHC_API int phc_self_obs_smpl_max(const PhcBodyState* body, int64_t n, uint32_t flags, float* out,
                          int64_t out_stride, phc_stream_t stream);

/* compute_imitation_observations_v6(root_pos, root_rot, body_*, ref_body_*, time_steps,
 * upright)                                                          envs/common.py:106-176
 * ref is [n*T, J, .] (env-major, then t).  mode 6 -> 24*J floats per future step;
 * mode 7 -> the position/velocity column subset [d_pos | d_vel | l_pos], 9*J per step
 * (the reference has no v7; SURVEY.md §8(a) A4). */
PHC_API int phc_imitation_obs(const float* root_pos, int64_t root_pos_stride, const float* root_rot,
                      int64_t root_rot_stride, const PhcBodyState* body, const PhcBodyState* ref,
                      int64_t n, int32_t time_steps, int32_t upright, int32_t mode, float* out,
                      int64_t out_stride, phc_stream_t stream);

/* build_amp_observations_smpl(root_pos, root_rot, root_vel, root_ang_vel, dof_pos, dof_vel,
 * key_body_pos, shape_params, limb_weight_params, dof_subset, local_root_obs, root_height_obs,
 * has_dof_subset, has_shape_obs_disc, has_limb_weight_obs, upright)      envs/common.py:192-267
 * (dof_to_obs_smpl :179-189, exp_map_to_quat torch_utils.py:334-366).  Writes
 * [root_h? | root rot 6 | root vel 3 | root ang vel 3 | dof obs 6*nj | dof vel 3*nj | key pos 3*K]
 * per row; shape / limb-weight columns are appended by the caller (copies of inputs).
 * dof_subset: NULL (all dofs) or num_sel int64 dof indices (a multiple of 3). */
typedef struct PhcAmpArgs {
  const float* root_pos;     int64_t root_pos_stride;      /* [n,3] */
  const float* root_rot;     int64_t root_rot_stride;      /* [n,4] */
  const float* root_vel;     int64_t root_vel_stride;      /* [n,3] */
  const float* root_ang_vel; int64_t root_ang_vel_stride;  /* [n,3] */
  const float* dof_pos;      int64_t dof_pos_stride, dof_pos_elem_stride; /* [n,D] */
  const float* dof_vel;      int64_t dof_vel_stride, dof_vel_elem_stride; /* [n,D] */
  PhcView key_body_pos;      /* [n,K,3] */
  int32_t num_key_bodies;    /* K <= 8 */
  const int64_t* dof_subset; /* NULL or [num_sel] */
  int32_t num_sel;           /* dofs used (D when dof_subset is NULL), multiple of 3, <= 96 */
  uint32_t flags;            /* PHC_OBS_LOCAL_ROOT | PHC_OBS_ROOT_HEIGHT | PHC_OBS_UPRIGHT */
} PhcAmpArgs;
PHC_API int phc_amp_obs(const PhcAmpArgs* args, int64_t n, float* out, int64_t out_stride, phc_stream_t stream);

/* rwd_specs of compute_imitation_reward (config.py:38-46). */
typedef struct PhcRewardSpec {
  float k_pos, k_rot, k_vel, k_ang_vel;
  float w_pos, w_rot, w_vel, w_ang_vel;
} PhcRewardSpec;

/* compute_imitation_reward(root_pos, root_rot, body_*, ref_body_*, rwd_specs)
 *                                                                   envs/common.py:270-322 */
PHC_API int phc_imitation_reward(const PhcBodyState* body, const PhcBodyState* ref, int64_t n,
                         const PhcRewardSpec* spec, float* reward /* [n] */,
                         float* reward_raw /* [n,4] */, int64_t reward_raw_stride,
                         phc_stream_t stream);

/* compute_humanoid_im_reset(reset_buf, progress_buf, contact_buf, contact_body_ids,
 * rigid_body_pos, ref_body_pos, pass_time, enable_early_termination, termination_distance,
 * use_mean)                                                         envs/common.py:325-364
 * contact_buf / contact_body_ids are never read by the reference and are not taken. */
PHC_API int phc_im_reset(const PhcView* rigid_body_pos, const PhcView* ref_body_pos, int32_t num_reset_bodies,
                 const int16_t* progress_buf, const uint8_t* pass_time,
                 const float* termination_distance /* [R] */, int32_t enable_early_termination,
                 int32_t use_mean, int64_t n, uint8_t* reset, uint8_t* terminated,
                 phc_stream_t stream);

/* ------------------------------------------------------------------------------------
 * The fused step: the post-physics half of HumanoidPHC.step   envs/humanoid_phc.py:138-149
 *   progress_buf += 1 (:138); _compute_reward (:1230-1271); _compute_reset (:1313-1335);
 *   _compute_observations (:937-961) = smpl_max self obs (:963-998) + v6 task obs at
 *   t+dt .. t+T*dt (:1050-1123), written as one row of obs_buf.
 * One kernel; no host reads; graph-capturable.
 * ---------------------------------------------------------------------------------- */
#define PHC_STEP_MAPPED_HOST_IO 1u /* sim state / clock / outputs are pinned host memory mapped into the
                                      device address space: no L2 prefetch, no pre-dependency speculation */
#define PHC_STEP_OBS_NORM_BF16 2u  /* obs_norm points to bfloat16 rows (the policy's input dtype under autocast): each
                                      normalised fp32 value is rounded to nearest-even; obs_norm_stride counts bf16 elements */
#define PHC_EPISODE_SUM_COLS 12
struct PhcResetArgs;
typedef struct PhcStepArgs {
  PhcBodyState body;                     /* sim state views, J must be 24               */
  int16_t* progress_buf;                 /* [n] in/out                  humanoid_phc.py:571 */
  const float* motion_start_times;       /* [n]                         humanoid_phc.py:592 */
  const float* motion_start_times_offset;/* [n]                         humanoid_phc.py:593 */
  const float* global_offset;            /* [n,3] or NULL               humanoid_phc.py:591 */
  const int64_t* sampled_motion_ids;     /* [n]                         humanoid_phc.py:597 */
  const float* termination_distances;    /* [24]                        humanoid_phc.py:240 */
  uint32_t reset_body_mask;              /* bit b = body b is in _reset_bodies_id       */
  int32_t use_mean;                      /* flag_im_eval                humanoid_phc.py:1334 */
  int32_t enable_early_termination;      /* config.py:99                                */
  int32_t advance_progress;              /* 1: progress_buf += 1 first, as step() does  */
  int32_t time_steps;                    /* future reference frames T (1 in the env)    */
  float dt;                              /* isaac_base.dt = 2*(1/60)    isaacgym_env.py:41 */
  PhcRewardSpec rwd;
  float* obs_buf;                        /* [n, 358+576*T]              humanoid_phc.py:557 */
  int64_t obs_stride;
  float* rew_buf;                        /* [n]                         humanoid_phc.py:560 */
  float* reward_raw;                     /* [n, >=4]                    humanoid_phc.py:562 */
  int64_t reward_raw_stride;
  uint8_t* reset_buf;                    /* [n] bool                    humanoid_phc.py:573 */
  uint8_t* terminate_buf;                /* [n] bool                    humanoid_phc.py:575 */
  uint32_t flags;                        /* PHC_STEP_* bits, 0 by default                */
  /* power reward (humanoid_phc.py:1297-1305), off when dof_force is NULL:
   *   power = sum_dof |dof_force * dof_vel|; r = -rew_power_coef * power, 0 while progress <= 3;
   *   rew_buf += r; reward_raw[:, power_col] = r                                           */
  const float* dof_force;                /* NULL or [n, 69]             humanoid_phc.py:506  */
  int64_t dof_force_stride;
  const float* dof_vel;                  /* [n, 69] view of the dof state humanoid_phc.py:536 */
  int64_t dof_vel_stride;                /* row stride in elements                           */
  int64_t dof_vel_elem_stride;           /* 2 for the reference's (pos, vel) interleaved state */
  float rew_power_coef;                  /* config.py rew_power_coef                          */
  int32_t power_col;                     /* column of reward_raw that receives r (4)          */
  double* obs_moments;                   /* NULL, or [2*(358+576*T)] fp64: per-column sum
                                            and sum of squares accumulated (+=) for
                                            RunningNorm.update           running_norm.py:23 */
  /* RunningNorm.forward fused into the obs epilogue (policies/running_norm.py:15-20), off when
   * obs_norm is NULL:  obs_norm = clamp((obs - mean) / sqrt(var + epsilon), -clip, clip), written
   * IN ADDITION to obs_buf (the experience buffer keeps the raw rows, RunningNorm.update needs them) */
  float* obs_norm;                       /* NULL or [n, 358+576*T] fp32 (bf16 with PHC_STEP_OBS_NORM_BF16) */
  int64_t obs_norm_stride;
  const float* norm_mean;                /* [358+576*T] running_mean                         */
  const float* norm_var;                 /* [358+576*T] running_var                          */
  float norm_epsilon;                    /* 1e-5 in the reference                            */
  float norm_clip;                       /* 10.0 in the reference                            */
  float* mpjpe;                          /* NULL or [n]: extras["mpjpe"] of eval mode, the mean over all
                                            24 bodies of |rigid_body_pos - ref rg_pos| at the reward
                                            time                              humanoid_phc.py:159-167 */
  int32_t obs_moments_buckets;           /* 0 / 1: obs_moments is one [2*(358+576*T)] accumulator.  B > 1: obs_moments is
                                            [B][2*(358+576*T)] and block b adds into bucket b % B — fp64 atomics on ONE
                                            address serialise (~30 ns each), so 1024 blocks on a single accumulator cost
                                            35 us per 4096-env step; 32 buckets make the epilogue free.  The consumer
                                            sums the buckets (phc_obs_moments_fold).                                  */
  /* PHCPufferEnv.step's per-env episode bookkeeping (clean_pufferl/env.py:121-159; phc_episode_update is the standalone
   * form and documents the semantics) done by the step itself, off when ep_returns is NULL.  The T = 1 kernel does it in
   * its reduction warp; the other kernels are followed by one small launch.  The sums go to ep_buckets accumulators
   * of PHC_EPISODE_SUM_COLS doubles {episodes finished, sum of returns, sum of lengths, truncations, sum over envs of
   * reward_raw[:, c]}, folded by phc_episode_fold when the caller logs.  A block of the T = 1 kernel sums its four
   * envs in fp32 (counts and lengths exact) and adds the row of bucket blockIdx % ep_buckets with one atomic
   * instruction; ceil(n / 4) buckets give every block its own row.                                                */
  uint8_t* ep_terminals;                 /* [n] out */
  uint8_t* ep_truncations;               /* [n] out */
  uint8_t* ep_masks;                     /* [n] out */
  float* ep_returns;                     /* [n] in/out */
  int32_t* ep_lengths;                   /* [n] in/out */
  double* ep_sums;                       /* [ep_buckets][PHC_EPISODE_SUM_COLS], zeroed by the caller once */
  int32_t ep_buckets;                    /* 1 .. 4096; ceil(n / 4) = one row per block    */
  int32_t ep_raw_cols;                   /* columns of reward_raw that are logged, <= 8 */
  /* ---- ABI 3 ------------------------------------------------------------------------------------------------- */
  float* rew_out;                        /* NULL or [n]: a second copy of rew_buf — `rew = self.rewards.clone()` of
                                            PHCPufferEnv.step (clean_pufferl/env.py:121), written with it            */
  uint8_t* reset_out;                    /* NULL or [n]: the step's reset flags, kept when auto_reset clears reset_buf */
  uint8_t* terminate_out;                /* NULL or [n]: extras["terminate"] = _terminate_buf.clone()  humanoid_phc.py:151 */
  /* The reset of the envs this step flags, INSIDE the step (clean_pufferl/env.py:133-135 -> HumanoidPHC.reset(indices),
   * humanoid_phc.py:665-676), off when NULL.  A block that has flagged envs re-poses them from the motion library
   * (exactly phc_reset_envs: sample_time_interval, full get_motion_state, _set_env_state scatter, clock and buffer
   * resets), recomputes their observation rows from the new state before the rows leave shared memory, and clears
   * reset_buf / terminate_buf / progress_buf of those envs; the step's own flags survive in reset_out /
   * terminate_out, and the moments / normaliser epilogues and the episode bookkeeping see what the reference's
   * wrapper would see (final rows, the step's flags).  Every buffer is bit-identical to phc_step_fused followed by
   * phc_reset_envs(env_mask = reset_buf).  The struct's body / progress_buf / reset_buf / terminate_buf / obs_buf /
   * sampled_motion_ids / clock pointers / time_steps / dt must be the step's own (PHC_ERR_SHAPE otherwise); env_mask
   * is ignored.  Kernels without the in-kernel path (T > 1, strided inputs) are followed by phc_reset_envs.         */
  const struct PhcResetArgs* auto_reset;
  /* res_action (humanoid_phc.py:1115-1120, 1218-1228): the reference keeps ref_dof_pos = dof_pos of the motion query
   * at the observation time t + dt for the next _action_to_pd_targets.  NULL, or [n, 69] (needs the library's lrs).  */
  float* ref_dof_pos;
  int64_t ref_dof_pos_stride;
  /* self-observation flags of compute_humanoid_observations_smpl_max (humanoid_phc.py:963-998, config.py:61-69):
   * PHC_OBS_LOCAL_ROOT | PHC_OBS_ROOT_HEIGHT | PHC_OBS_UPRIGHT.  0 means the env's defaults (all three); any other
   * combination changes the self-obs columns (no height column: 357 + 576 T floats per row) and, for !upright, the
   * heading both observations are expressed in.  PHC_STEP_OBS_FLAGS_SET marks the field as given.                   */
  uint32_t obs_flags;
} PhcStepArgs;
#define PHC_STEP_OBS_FLAGS_SET 0x80000000u

/* Kernel selection (all bit-identical): T == 1 on one AoS-13 sim tensor with a dense 16-B aligned obs_buf runs the
 * single-wave TMA kernel, or — from 10240 envs on, when none of the optional epilogues is asked for — the persistent
 * warp-specialised kernel, whose blocks draw env tiles from a device-side counter owned by `lib` (256 counter slots used
 * round robin, each left zero by the launch that used it: launches of one PhcLib may overlap on different streams as
 * long as fewer than 256 of them are in flight or captured in concurrently replayed graphs); T > 1 runs the pipelined
 * multi-query kernel; anything else (strided views, non-default flags with T > 1) the generic kernel. */
PHC_API int phc_step_fused(const PhcLib* lib, const PhcStepArgs* args, int64_t n, phc_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Reference-state-init reset of a subset of envs, on the device, with no host sync:
 *   HumanoidPHC._reset_envs (envs/humanoid_phc.py:665-676) =
 *     _sample_ref_state (:845-875; MotionLibBase.sample_time_interval motion_lib.py:526-535)
 *     -> get_motion_state -> _set_env_state (:901-931) -> clock updates of
 *     _reset_ref_state_init (:724-731) -> buffer zeroing of _reset_env_tensors (:775-778)
 *     -> _compute_observations(env_ids) (:937-961).
 * The PhysX setters (:748-765) are out of scope.  Envs are selected by a byte mask (reset_buf
 * itself, or a copy), so the `nonzero()` of clean_pufferl/env.py:133 is not needed.  Random numbers
 * come from the caller (`phase`, what torch.rand gives in sample_time_interval), indexed by env.
 * ONE launch: a block scatters the new state of its 8 envs and then computes their observation
 * rows from what it has just written; a block without a selected env reads 8 mask bytes and leaves.
 * ---------------------------------------------------------------------------------- */
#define PHC_STATE_INIT_START 0  /* motion time 0                       state_init.py */
#define PHC_STATE_INIT_RANDOM 1 /* sample_time_interval(phase)                       */
/* ABI 4.  StateInit.Default (_reset_default, envs/humanoid_phc.py:688-692): root / dof state of the selected envs from
 * the initial_* buffers; the rigid-body tensors and the motion clock (start times, global offset) stay as they are,
 * progress / reset / terminate -> 0, the observation rows are those of the (unchanged) rigid-body state at the restarted
 * clock.  StateInit.Hybrid (_reset_hybrid_state_init, :733-745): an env whose default_mask byte is set takes the
 * default path, the others reference-state init at a sampled time; the reference draws the mask with
 * torch.bernoulli(hybrid_init_prob) — the caller supplies it, like `phase`.  (AMP buffers: the reference raises
 * NotImplementedError for default-reset envs, :795-797.) */
#define PHC_STATE_INIT_DEFAULT 2
#define PHC_STATE_INIT_HYBRID 3
typedef struct PhcResetArgs {
  PhcBodyState body;                      /* sim state views, written for the selected envs (J = 24) */
  float* humanoid_root_states;            /* NULL or [n,13]: pos3|rot4|vel3|ang vel3  humanoid_phc.py:518 */
  int64_t root_stride;
  float* dof_pos;                         /* NULL or [n,69] view          humanoid_phc.py:535 */
  float* dof_vel;                         /* NULL or [n,69] view          humanoid_phc.py:536 */
  int64_t dof_stride;                     /* row stride in elements (both views)             */
  int64_t dof_elem_stride;                /* 2 for the interleaved (pos, vel) dof state       */
  int16_t* progress_buf;                  /* [n] -> 0                                         */
  uint8_t* reset_buf;                     /* [n] -> 0                                         */
  uint8_t* terminate_buf;                 /* [n] -> 0                                         */
  float* motion_start_times;              /* [n] -> sampled motion time                       */
  float* motion_start_times_offset;       /* [n] -> 0                                         */
  float* global_offset;                   /* [n,3] read (old value offsets the pose), then -> 0 */
  const int64_t* sampled_motion_ids;      /* [n]                                              */
  const uint8_t* env_mask;                /* [n] 1 = reset this env; may be reset_buf itself   */
  const float* phase;                     /* [n] uniform [0,1), used when state_init == RANDOM */
  int32_t state_init;                     /* PHC_STATE_INIT_*                                 */
  int32_t flag_test;                      /* motion_times[:] = 0         humanoid_phc.py:856  */
  int32_t time_steps;                     /* T of the observation                             */
  float dt;
  float* obs_buf;                         /* [n, 358+576*T]: rows of the selected envs rewritten */
  int64_t obs_stride;
  /* ---- ABI 3: keep the step's fused epilogues consistent with the rows a reset rewrites ------------------------- */
  float* obs_norm;                        /* NULL, or the normalised copy of obs_buf (PhcStepArgs.obs_norm): the rows of
                                             the selected envs are rewritten too          policies/running_norm.py:15-20 */
  int64_t obs_norm_stride;
  const float* norm_mean;                 /* [358+576*T] */
  const float* norm_var;                  /* [358+576*T] */
  float norm_epsilon, norm_clip;
  int32_t obs_norm_bf16;                  /* obs_norm holds bfloat16 rows */
  int32_t obs_moments_mode;               /* 0: moments untouched; 1: the new rows are ADDED (an initial reset: the rows
                                             were never counted); 2: the old rows are REPLACED (subtract old, add new:
                                             the step that flagged the envs had counted the rows it wrote)             */
  double* obs_moments;                    /* NULL, or [buckets][2*(358+576*T)] fp64 accumulators as in PhcStepArgs      */
  int32_t obs_moments_buckets;
  uint32_t obs_flags;                     /* as PhcStepArgs.obs_flags (0 = the env's defaults)                          */
  float* ref_dof_pos;                     /* NULL or [n, 69]: _compute_task_obs(env_ids) of the reset keeps the dof_pos of
                                             the query at t + dt for res_action            humanoid_phc.py:1115-1120 */
  int64_t ref_dof_pos_stride;
  /* ---- ABI 4: StateInit.Default / Hybrid ------------------------------------------------------------------------- */
  const float* initial_root_states;       /* [n,13] _initial_humanoid_root_states (:521); needed for DEFAULT / HYBRID
                                             when humanoid_root_states is set */
  int64_t initial_root_stride;
  const float* initial_dof_pos;           /* [n,69] _initial_dof_pos (:543), dense rows of initial_dof_stride floats */
  const float* initial_dof_vel;           /* [n,69] _initial_dof_vel (:544) */
  int64_t initial_dof_stride;
  const uint8_t* default_mask;            /* HYBRID: [n], 1 = this env takes the default path */
} PhcResetArgs;
PHC_API int phc_reset_envs(const PhcLib* lib, const PhcResetArgs* args, int64_t n, phc_stream_t stream);

/* Process-wide tuning / test switches of phc_step_fused (not part of the reference surface).
 * phc_step_fused picks the TMA fast kernel when time_steps == 1, the four body views are one
 * 16-B aligned AoS-13 tensor and obs_buf is dense and 16-B aligned; otherwise, or when
 * PHC_OPT_FORCE_GENERIC_STEP is set, the generic kernel (any T, any strides). */
#define PHC_OPT_FORCE_GENERIC_STEP 1 /* value 0/1 */
#define PHC_OPT_STEP_EPB 2           /* envs per block of the fast kernel: 4 (the only value built) */
#define PHC_OPT_STEP_PDL 3           /* 1 (default): launch the fast kernel with programmatic stream
                                        serialization so its prologue overlaps the previous kernel's tail */
#define PHC_OPT_TEST_SPEC_FAULT 4     /* test hook, bit mask: perturb the clock the fast kernel speculated on
                                        (1 progress-1, 2 start time, 4 progress-2, 8 motion id) so the
                                        validation / redo paths run; results must not change */
#define PHC_OPT_MULTI_GROUPS 5        /* thread groups per block of the T > 1 kernel: 2 (default; also value 0): the queries of an
                                        env are worked on in pairs; 1: the single-group pipeline, kept as the cross-check */
#define PHC_OPT_MOMENTS_BULK 6        /* 1: the T = 1 kernel's moments epilogue (obs_moments) hands each block's 1868 partial sums to the TMA
                                        engine as three bulk fp64 reductions; 0 (default, measured a little faster): one atomic per sum */
#define PHC_OPT_STEP_PERSIST 7        /* the persistent warp-specialised T = 1 kernel for multi-wave grids: 1 (default) from 10240 envs on
                                        (env PHC_STEP_PERSIST_MIN), 0 never, 2 always (tests), 3 always with four
                                        frame slots per env and four blocks per SM instead of three and five (comparison) */
PHC_API int phc_set_option(int key, int value);
/* Profiling aid: when a device buffer of capacity_warps x 8 uint64 is set, every warp of the
 * fast step kernel (EPB 4: 3 warps per block) stamps %globaltimer (ns) at its phase boundaries:
 * 0 entry, 1 TMA issued (warp 0), 2 dependency wait returned (warp 0), 3 data landed, 4 phase 1 done,
 * 5 stage written, 6 past barrier 3, 7 exit.  Consecutive launches use consecutive slices of
 * the buffer until it is full.  NULL switches it off. */
PHC_API int phc_set_trace_buffer(uint64_t* device_buf, int64_t capacity_warps);

/* HumanoidPHC._action_to_pd_targets(action)                      envs/humanoid_phc.py:1218-1228
 *   res_action == 0:  pd = pd_action_offset + pd_action_scale * action
 *   res_action != 0:  pd = clamp(ref_dof_pos + pd_action_scale * action, dof_pos -+ pi/2)
 * offset / scale are [D]; action, ref_dof_pos, out are dense [n, D]; dof_pos is the strided view
 * of the dof state.  The freeze_hand / freeze_toe zeroing of step() (:118-127) is `zero_mask`:
 * bit j set = the 3 dofs of joint j are written as 0.
 * The wrapper's action clip rides in the same launch (clean_pufferl/env.py:110-112: np.clip(actions, -1, 1) into
 * self.actions, which env.step then turns into PD targets): with action_clip > 0 the action is clamped to
 * [-action_clip, action_clip] first; when actions_out is not NULL the (clamped) action is stored there. */
PHC_API int phc_action_to_pd_targets(const float* action, const float* pd_action_offset, const float* pd_action_scale,
                                     int32_t res_action, const float* ref_dof_pos, const float* dof_pos,
                                     int64_t dof_pos_stride, int64_t dof_pos_elem_stride, uint32_t zero_mask,
                                     int64_t n, int32_t num_dof, float action_clip, float* actions_out, float* out,
                                     phc_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Host-buffer pipeline around the fused step (the end-to-end call): chunked
 * H2D(sim state, clock) -> phc_step_fused -> D2H(obs, reward, flags) on internal streams.
 * All pointers in PhcHostStepArgs are HOST pointers (pinned for full speed); a device pointer is refused with
 * PHC_ERR_UNSUPPORTED.  On any error the internal streams are drained before the call returns.
 * ---------------------------------------------------------------------------------- */
typedef struct PhcHostStep PhcHostStep;

typedef struct PhcHostStepArgs {
  const float* state;                    /* host [n, 24, 13] AoS sim state              */
  int16_t* progress_buf;                 /* host [n] in/out                             */
  const float* motion_start_times;       /* host [n]                                    */
  const float* motion_start_times_offset;/* host [n]                                    */
  const float* global_offset;            /* host [n,3]                                  */
  const int64_t* sampled_motion_ids;     /* host [n]                                    */
  float* obs_buf;                        /* host [n, 358+576*T]                         */
  float* rew_buf;                        /* host [n]                                    */
  float* reward_raw;                     /* host [n,4]                                  */
  uint8_t* reset_buf;                    /* host [n]                                    */
  uint8_t* terminate_buf;                /* host [n]                                    */
} PhcHostStepArgs;

PHC_API int phc_host_step_create(const PhcLib* lib, int64_t max_envs, int32_t time_steps, int32_t num_chunks,
                         const float* termination_distances_host /* [24] */, uint32_t reset_body_mask,
                         int32_t use_mean, int32_t enable_early_termination, float dt,
                         const PhcRewardSpec* rwd, PhcHostStep** out);
PHC_API int phc_host_step(PhcHostStep* ctx, const PhcHostStepArgs* args, int64_t n);
/* Destroy waits for every slot in flight (as phc_host_step_wait would) before it frees anything. */
PHC_API void phc_host_step_destroy(PhcHostStep* ctx);

/* Asynchronous form: submit a step on one of PHC_HOST_SLOTS slots, collect it later.  Each slot is a pipeline of its
 * own (device buffers, pinned staging, three streams), so two batches can be in flight at once: the inbound copy of
 * one rides under the outbound traffic of the other, and the caller's thread is free between submit and wait (the
 * send / recv of a double-buffered env loop).
 *
 *   submit   Checks everything phc_host_step checks (NULL pointers, 0 <= n <= max_envs, device pointers ->
 *            PHC_ERR_UNSUPPORTED) and 0 <= slot < PHC_HOST_SLOTS (PHC_ERR_SHAPE), all before anything is enqueued.
 *            Packs the clock into the slot's pinned staging, enqueues the slot's chunks and returns without waiting.
 *            The first submit on slot 1 allocates that slot's buffers and may block on the allocation.
 *   buffers  From submit until wait returns, all 11 buffers of args belong to the library: on the direct path the
 *            kernels write obs, rewards, flags and progress into them asynchronously, and the copy engine reads state.
 *   wait     Blocks until the slot's outputs are in the caller's buffers (on the staged path it also unpacks the
 *            scalar outputs).  Returns PHC_OK, or the step's deferred error (PHC_ERR_CUDA + phc_last_cuda_error()).
 *            Waiting on an idle slot returns PHC_OK at once.  It also collects the two submits with resets below.
 *   busy     A submit to a slot with a step in flight returns PHC_ERR_BUSY, enqueues nothing and leaves the step in
 *            flight untouched.  phc_host_step is submit + wait on slot 0: it returns PHC_ERR_BUSY while slot 0 is in
 *            flight and runs normally while only slot 1 is.
 *   tuning   Only phc_host_step calls made while no slot is in flight count toward the (path, chunks) tuner.  A
 *            submit uses the settled schedule; before tuning has finished it uses the first candidate (direct, three
 *            chunks, unless num_chunks / PHC_HOST_PATH narrow it); pageable callers always take the staged path.
 *   errors   An error inside submit after the first enqueue drains that slot's streams before returning; the other
 *            slot is not touched.  After any error the slot is idle.
 *   threads  One host thread drives a context.  Contexts over one PhcLib may be driven from different threads. */
#define PHC_HOST_SLOTS 2
PHC_API int phc_host_step_submit(PhcHostStep* ctx, int32_t slot, const PhcHostStepArgs* args, int64_t n);
PHC_API int phc_host_step_wait(PhcHostStep* ctx, int32_t slot);
/* The schedule pinned callers are on.  phc_host_step_path: 1 = direct (each chunk's kernel posts obs rows / rewards /
 * flags into the mapped host buffers), 2 = staged (device buffers + copy-engine D2H; always the case for pageable
 * callers; the buffers of the last submit decide), 0 = not decided yet.  phc_host_step_chunks: the chunk count in use (0 = not decided yet).  With
 * num_chunks = 0 at create the context tunes (path, chunk count) over its first phc_host_step_tuning_calls() calls —
 * every candidate timed four times, interleaved, under whatever load the other GPUs of the box put on the host at
 * that moment — and keeps the fastest (three chunks on the direct path unless another schedule is 2 % faster); num_chunks > 0 fixes the chunk count and PHC_HOST_PATH=direct|staged the path. */
PHC_API int phc_host_step_path(const PhcHostStep* ctx);
PHC_API int phc_host_step_chunks(const PhcHostStep* ctx);
PHC_API int phc_host_step_tuning_calls(const PhcHostStep* ctx);
PHC_API int64_t phc_host_step_h2d_bytes(const PhcHostStep* ctx, int64_t n);
PHC_API int64_t phc_host_step_d2h_bytes(const PhcHostStep* ctx, int64_t n);

/* Resets on the host-buffer path (ABI 6): what HumanoidPHC.step() with auto-reset and HumanoidPHC.reset(env_ids, phase)
 * do (phc_step_fused with PhcStepArgs.auto_reset / phc_reset_envs, humanoid_phc.py:665-676), on host buffers.  The
 * reset runs over the slot's device copies of the chunk; then one small kernel per chunk writes the rows of the re-posed
 * envs (and nothing else) into the caller's buffers — straight into them when every output buffer below is pinned, else
 * through the slot's pinned staging, unpacked by phc_host_step_wait.  A re-posed env's new state is about 1.9 KB, so
 * only the reset envs' rows cross the link.  The clock arrays of PhcHostStepArgs are const: the new clock leaves through
 * the *_out pointers, which may alias them (and state_out may alias args->state): the inputs are consumed before any
 * output of the same rows is written.  Everything here is a HOST pointer.
 *
 *   phc_host_step_submit_reset  The step with auto-reset.  When phc_host_step_wait returns: obs_buf holds the final rows
 *            (a re-posed env's row is recomputed from its new state), rew_buf / reward_raw the step's, reset_buf /
 *            terminate_buf the STEP's flags (extras["reset"] / ["terminate"] of the device path: the envs whose
 *            physics the caller must re-pose, and the dones), progress_buf advanced and 0 for re-posed envs; for the
 *            re-posed envs only: the clock outs (new start time, offset 0, global offset 0) and state_out / root_states /
 *            dof_pos / dof_vel (what _set_env_state writes, humanoid_phc.py:901-931).  Other rows of the reset outputs
 *            are not written.  env_mask is ignored.
 *   phc_host_reset_submit  HumanoidPHC.reset(env_ids, phase) for the envs whose env_mask byte is set: reads the clock,
 *            sampled_motion_ids, phase and env_mask (not state, not obs_buf; progress is not advanced).  For the masked
 *            envs only it writes obs rows, state_out / root_states / dof_pos / dof_vel rows, the clock outs,
 *            progress_buf = 0 and reset_buf = terminate_buf = 0; rew_buf / reward_raw are not touched.  This is how a
 *            host loop gets its first observation and resets envs it picks itself.
 *   validation  Everything phc_host_step_submit checks, plus: NULL reset pointers (env_mask for phc_host_reset_submit,
 *            phase for PHC_STATE_INIT_RANDOM) -> PHC_ERR_NULL; PHC_STATE_INIT_DEFAULT / HYBRID (they need per-env
 *            initial_* buffers: phc_host_step_submit_env / phc_host_reset_submit_env below) or any other state_init, a device pointer, or a motion library without local rotations
 *            / dof velocities -> PHC_ERR_UNSUPPORTED; a busy slot -> PHC_ERR_BUSY.  All before anything is enqueued;
 *            after any error the slot is idle.
 *   buffers / tuning / destroy  As for phc_host_step_submit: the reset buffers belong to the library until
 *            phc_host_step_wait returns; these submits are not timed by the tuner and use the settled schedule;
 *            destroy waits for them. */
typedef struct PhcHostResetArgs {
  const float* phase;                   /* host [n]: the uniform [0,1) numbers of sample_time_interval (RANDOM)  */
  const uint8_t* env_mask;              /* host [n]: phc_host_reset_submit only, 1 = reset this env             */
  int32_t state_init;                   /* PHC_STATE_INIT_START | PHC_STATE_INIT_RANDOM                          */
  int32_t flag_test;                    /* motion_times[:] = 0         humanoid_phc.py:856                       */
  float* state_out;                     /* host [n,24,13] rigid-body rows of re-posed envs (may alias args->state) */
  float* root_states;                   /* host [n,13] humanoid_root_states rows    humanoid_phc.py:518          */
  float* dof_pos;                       /* host [n,69] dense                        humanoid_phc.py:535          */
  float* dof_vel;                       /* host [n,69] dense                        humanoid_phc.py:536          */
  float* motion_start_times_out;        /* host [n]   (may alias args->motion_start_times)                       */
  float* motion_start_times_offset_out; /* host [n]   (may alias args->motion_start_times_offset)                */
  float* global_offset_out;             /* host [n,3] (may alias args->global_offset)                            */
} PhcHostResetArgs;
PHC_API int phc_host_step_submit_reset(PhcHostStep* ctx, int32_t slot, const PhcHostStepArgs* args,
                                       const PhcHostResetArgs* reset, int64_t n);
PHC_API int phc_host_reset_submit(PhcHostStep* ctx, int32_t slot, const PhcHostStepArgs* args,
                                  const PhcHostResetArgs* reset, int64_t n);

/* Host in, device out: the two submits above with the observation rows written into caller-owned device tensors
 * instead of host memory.  For a caller whose physics runs on the CPU and whose policy runs on the GPU, the rows are
 * 99 % of what a host step sends back (3736 B per env at T = 1, against 24 B of rewards, flags and progress); here they
 * never cross the link, and the fused normaliser (PhcStepArgs.obs_norm) and the RunningNorm moments epilogue
 * (obs_moments) are available as on the device path.  Sim state and clock still come from host buffers, and rewards,
 * reward_raw, flags, progress and the reset rows still go to host buffers, exactly as in phc_host_step_submit /
 * phc_host_step_submit_reset / phc_host_reset_submit.
 *
 *   phc_host_step_submit_device   The step (reset == NULL) or the step with auto-reset (reset != NULL).  obs holds
 *            the step's rows (with a reset: the final rows, a re-posed env's recomputed from its new state), obs_norm
 *            their normalised copy, and obs_moments += the column sums and sums of squares of the rows written (with a
 *            reset the final rows are the ones counted, as on the device path with auto-reset).
 *   phc_host_reset_submit_device  The host reset of the masked envs: their obs rows and normalised rows are written,
 *            and with obs_moments the new rows are ADDED (HumanoidPHC.reset(): rows no step has counted).  Rows of
 *            other envs are not touched.
 *   rows     args->obs_buf must be NULL (writing the rows to both places is not offered: PHC_ERR_UNSUPPORTED).  Every
 *            other field of PhcHostStepArgs / PhcHostResetArgs keeps its meaning and must be a host pointer.
 *   ordering A submit records an event on dev->stream, and each of the slot's streams waits for it before its first
 *            write into a device output; the host-to-device copies of the sim state do not wait.  So the policy may
 *            still be reading the previous rows of the same tensors, enqueued on dev->stream, when the next submit is
 *            issued.  When phc_host_step_wait returns, the device outputs are complete (wait blocks on the slot's
 *            events); work the caller enqueues afterwards on any stream sees them.  `dev` itself is read during the
 *            submit only; the tensors it names belong to the library until wait returns.
 *   validation  Everything the host submits check, plus, before anything is enqueued: dev or dev->obs NULL, obs_norm
 *            without norm_mean / norm_var -> PHC_ERR_NULL; a device field that is not device memory on the context's
 *            device, or a flag other than PHC_STEP_OBS_NORM_BF16 -> PHC_ERR_UNSUPPORTED; obs or obs_norm not 16-B
 *            aligned -> PHC_ERR_ALIGN; obs_moments_buckets outside 0..4096, or norm_clip <= 0 with obs_norm ->
 *            PHC_ERR_SHAPE; a busy slot -> PHC_ERR_BUSY.  After any error the slot is idle and the device outputs are
 *            untouched.
 *   schedule As the other submits: not timed by the tuner, the settled schedule (pageable callers: staged).  On the
 *            staged path no obs transfer is made; on the direct path the scalars are posted into the pinned buffers. */
typedef struct PhcHostDeviceOut {
  float* obs;                /* device [n, 358+576*T] fp32, dense rows, 16-B aligned                                   */
  float* obs_norm;           /* NULL, or device [n, 358+576*T] fp32 (bf16 with PHC_STEP_OBS_NORM_BF16), 16-B aligned   */
  const float* norm_mean;    /* device [358+576*T] running_mean, required with obs_norm                                */
  const float* norm_var;     /* device [358+576*T] running_var                                                         */
  float norm_epsilon, norm_clip;
  uint32_t flags;            /* 0 or PHC_STEP_OBS_NORM_BF16                                                            */
  double* obs_moments;       /* NULL, or device [buckets][2*(358+576*T)] fp64 accumulators (+=), as PhcStepArgs        */
  int32_t obs_moments_buckets;
  phc_stream_t stream;       /* the caller's stream that reads / writes these tensors (the policy's)                   */
} PhcHostDeviceOut;
PHC_API int phc_host_step_submit_device(PhcHostStep* ctx, int32_t slot, const PhcHostStepArgs* args,
                                        const PhcHostResetArgs* reset /* NULL: no auto-reset */,
                                        const PhcHostDeviceOut* dev, int64_t n);
PHC_API int phc_host_reset_submit_device(PhcHostStep* ctx, int32_t slot, const PhcHostStepArgs* args,
                                         const PhcHostResetArgs* reset, const PhcHostDeviceOut* dev, int64_t n);

/* Env options on the host-buffer path: the power reward, eval-mode mpjpe and StateInit.Default / Hybrid, which the
 * reference's default configuration uses (config.py:50, humanoid_phc.py:159-167, :678-745).  Added without a change to
 * any existing struct or entry point, so PHC_ABI_VERSION stays 6; a caller finds these by their symbols.
 *
 *   phc_host_step_submit_env   phc_host_step_submit (reset == NULL, dev == NULL), _submit_reset (reset != NULL) or
 *            _submit_device (dev != NULL) with the options of env (NULL: none).  Everything those submits do and check
 *            still holds.
 *   phc_host_reset_submit_env  phc_host_reset_submit (dev == NULL) or phc_host_reset_submit_device, likewise.  It
 *            takes only env->default_mask: dof_force, dof_vel and mpjpe are ignored.
 *   power    With dof_force set, args->reward_raw is [n, 5]: column 4 receives r = -rew_power_coef * sum_dof |dof_force *
 *            dof_vel|, 0 while progress <= 3, and rew_buf includes it (reward_raw[:, -1] of the reference,
 *            humanoid_phc.py:1297-1305); exactly PhcStepArgs.dof_force / power_col.  Each chunk's dof_force and dof_vel
 *            rows are copied to the device by the copy engine, straight from these buffers (pin them for speed).
 *   mpjpe    With mpjpe set, mpjpe[i] = mean over the 24 bodies of |rigid_body_pos - ref rg_pos| at the reward time
 *            (PhcStepArgs.mpjpe), written like rew_buf: posted by the kernel on the direct path (mpjpe then joins the
 *            buffers that decide it), unpacked by wait on the staged path.
 *   state init  PHC_STATE_INIT_DEFAULT / HYBRID are accepted once phc_host_step_set_initial_state has given the slot its
 *            initial rows: row i stands for env i of every batch submitted on that slot.  A default-path env keeps its
 *            rigid-body rows and clock; its root / dof rows become the initial ones; its observation is that of the
 *            unchanged state at the restarted progress.  HYBRID takes env->default_mask (1 = default path) and phase
 *            (the envs that take reference-state init).  The re-posed rows leave as with the other reset modes.
 *   validation  Before anything is enqueued, on top of the checks of the matching submit: dof_force without dof_vel
 *            or the reverse, HYBRID without default_mask or phase, DEFAULT / HYBRID on a slot without initial rows ->
 *            PHC_ERR_NULL; n larger than the slot's initial rows (DEFAULT / HYBRID) -> PHC_ERR_SHAPE; a device pointer
 *            in env -> PHC_ERR_UNSUPPORTED.  After any error the slot is idle and nothing is written.
 *   buffers / schedule  As the matching submit: env's buffers belong to the library until phc_host_step_wait returns;
 *            not timed by the tuner; the settled schedule.  phc_host_step_h2d_bytes / _d2h_bytes describe the plain
 *            step: the power reward adds 2 x 276 B per env inbound, mpjpe and the fifth reward column 4 B each outbound.
 *
 * phc_host_step_set_initial_state  Copies n initial rows (_initial_humanoid_root_states [n,13], _initial_dof_pos /
 *            _initial_dof_vel [n,69], dense; humanoid_phc.py:521, 543-544) once, synchronously, into the slot's device
 *            buffers (allocated at the first call, max_envs rows), replacing any earlier rows.  Host memory, pinned or
 *            pageable: the reference sets them once at setup, so they do not travel with every submit.  NULL pointer ->
 *            PHC_ERR_NULL; bad slot or n outside 0..max_envs -> PHC_ERR_SHAPE; a device pointer -> PHC_ERR_UNSUPPORTED;
 *            the slot in flight -> PHC_ERR_BUSY. */
typedef struct PhcHostEnvArgs {
  const float* dof_force;    /* host [n,69] dense, or NULL: no power reward              humanoid_phc.py:506     */
  const float* dof_vel;      /* host [n,69] dense, required with dof_force               humanoid_phc.py:536     */
  float rew_power_coef;      /* config.py:112                                                                    */
  float* mpjpe;              /* host [n] out, or NULL                                    humanoid_phc.py:159-167 */
  const uint8_t* default_mask; /* host [n], PHC_STATE_INIT_HYBRID: 1 = default path      humanoid_phc.py:733-745 */
} PhcHostEnvArgs;
PHC_API int phc_host_step_submit_env(PhcHostStep* ctx, int32_t slot, const PhcHostStepArgs* args,
                                     const PhcHostResetArgs* reset /* NULL: no auto-reset */,
                                     const PhcHostDeviceOut* dev /* NULL: host obs */,
                                     const PhcHostEnvArgs* env /* may be NULL */, int64_t n);
PHC_API int phc_host_reset_submit_env(PhcHostStep* ctx, int32_t slot, const PhcHostStepArgs* args,
                                      const PhcHostResetArgs* reset, const PhcHostDeviceOut* dev /* may be NULL */,
                                      const PhcHostEnvArgs* env /* may be NULL */, int64_t n);
PHC_API int phc_host_step_set_initial_state(PhcHostStep* ctx, int32_t slot, const float* root_states /* [n,13] */,
                                            const float* dof_pos /* [n,69] */, const float* dof_vel /* [n,69] */,
                                            int64_t n);

/* ------------------------------------------------------------------------------------
 * RunningNorm statistics                                   policies/running_norm.py:23-34
 * phc_obs_moments accumulates (+=) per-column fp64 sum and sum of squares of x[rows,cols]
 * into sums[2*cols]; the caller all-reduces sums (and the row count) across GPUs, then
 * phc_running_norm_update applies mean/var(unbiased=False) with the reference's 1/count
 * blend to the fp32 running buffers in place.
 * ---------------------------------------------------------------------------------- */
PHC_API int phc_obs_moments(const float* x, int64_t rows, int64_t cols, int64_t row_stride, double* sums,
                    phc_stream_t stream);
/* sums[cols2] += sum over b of buckets[b][cols2] (fixed order), then buckets are zeroed for the next rollout */
PHC_API int phc_obs_moments_fold(double* buckets, int32_t num_buckets, int64_t cols2, double* sums, phc_stream_t stream);
PHC_API int phc_running_norm_update(float* running_mean, float* running_var, float* count, const double* sums,
                            const double* total_rows /* device scalar */, int64_t cols,
                            phc_stream_t stream);
/* ------------------------------------------------------------------------------------
 * RunningNorm.update across the GPUs of one node in ONE launch per rank: the all-reduce of the
 * [2*cols + 1] fp64 partials over NVLink peer memory fused with the blend (running_norm.py:23-34
 * over the concatenated batch of all ranks).  Replaces ncclAllReduce + phc_running_norm_update.
 *   create            -> allocates this rank's mailbox (device memory, two slots + flags)
 *   handle / connect  -> CUDA IPC: every rank exports PHC_PEER_HANDLE_BYTES, the caller all-gathers
 *                        them (any host channel) and hands connect() the world * 64 bytes in rank order
 *   connect_local     -> same for "ranks" that live in one process (tests, one-process-many-GPUs)
 *   update_peers      -> one kernel: publish sums[2*cols] + rows, wait for every rank's epoch flag,
 *                        add the payloads in rank order (bit-identical statistics on every rank),
 *                        blend into running_mean / running_var, count += 1, zero sums.
 *                        rows: device scalar if rows_dev != NULL, else the value `rows`.
 *                        Never synchronises; CUDA-graph capturable (the epoch lives on the device).
 *   status            -> synchronises; PHC_PEER_TIMEOUT if a launch gave up waiting, and the number of completed
 *                        reductions.  The wait is decided ONCE per launch: a timed-out launch touches neither
 *                        running_mean / running_var nor sums, count or the epoch.
 *   resync            -> after a timeout the ranks are out of step (this rank published an epoch its peers may or
 *                        may not have completed).  Collective recovery: host barrier, every rank calls resync
 *                        (synchronises its device; clears its mailbox, flags, epoch and status), host barrier.
 *                        The caller re-broadcasts running_mean / running_var / count if a peer did complete the
 *                        epoch this rank gave up on, and keeps its own partials (they were not consumed).
 * ---------------------------------------------------------------------------------- */
#define PHC_PEER_MAX_WORLD 16
#define PHC_PEER_HANDLE_BYTES 64 /* sizeof(cudaIpcMemHandle_t) */
typedef struct PhcPeerReduce PhcPeerReduce;
PHC_API int phc_peer_reduce_create(int32_t rank, int32_t world, int64_t cols, int64_t timeout_ms /* <= 0: 5000 */,
                                   PhcPeerReduce** out);
PHC_API int phc_peer_reduce_handle(const PhcPeerReduce* ctx, void* handle_out /* 64 bytes */);
PHC_API int phc_peer_reduce_connect(PhcPeerReduce* ctx, const void* handles /* world * 64 bytes, rank order */);
PHC_API int phc_peer_reduce_connect_local(PhcPeerReduce* ctx, PhcPeerReduce* const* all /* [world] */);
PHC_API int phc_running_norm_update_peers(PhcPeerReduce* ctx, double* sums, const double* rows_dev, double rows,
                                          float* running_mean, float* running_var, float* count,
                                          phc_stream_t stream);
PHC_API int phc_peer_reduce_status(PhcPeerReduce* ctx, int64_t* completed_out /* may be NULL */);
PHC_API int phc_peer_reduce_resync(PhcPeerReduce* ctx);
PHC_API void phc_peer_reduce_destroy(PhcPeerReduce* ctx);

/* RunningNorm.forward                                      policies/running_norm.py:15-20 */
PHC_API int phc_running_norm_forward(const float* x, int64_t rows, int64_t cols, int64_t row_stride,
                             const float* running_mean, const float* running_var, float epsilon,
                             float clip, float* out, int64_t out_stride, phc_stream_t stream);

/* Per-env episode bookkeeping of the pufferlib wrapper, PHCPufferEnv.step   clean_pufferl/env.py:121-159
 *   raw_rewards += mean_env(reward_raw)                                           (:124)
 *   terminals = terminate;  truncations = reset & ~terminate;  masks = ~truncations   (:130-154)
 *   for reset envs: stats += {1, episode_return, episode_length, truncated};  return = length = 0  (:136-140)
 *   then EVERY env: episode_return += reward;  episode_length += 1   (:158-159 — env.reset() has already
 *   cleared reset_buf there, humanoid_phc.py:778, so the mask is all-true)
 * `reset` is reset_buf as the step left it (before the reset), `terminate` is extras["terminate"].
 * `stats` replaces the three Python lists mean_and_log (:191-204) averages, so no host sync is
 * needed per step: {episodes finished, sum of returns, sum of lengths, truncations} in fp64.
 * `workspace` is PHC_EPISODE_WORKSPACE_DOUBLES doubles, zeroed once by the caller; every launch
 * leaves it zero.  Flags are bytes (torch.bool). */
#define PHC_EPISODE_WORKSPACE_DOUBLES 16
typedef struct PhcEpisodeArgs {
  const uint8_t* reset;       /* [n] */
  const uint8_t* terminate;   /* [n] */
  const float* rewards;       /* [n] rew_buf */
  const float* reward_raw;    /* [n, reward_raw_cols] rows `reward_raw_stride` floats apart, or NULL when cols == 0 */
  int64_t reward_raw_stride;
  int32_t reward_raw_cols;    /* <= 8 (the reference logs 5) */
  int32_t _pad0;
  uint8_t* terminals;         /* [n] out */
  uint8_t* truncations;       /* [n] out */
  uint8_t* masks;             /* [n] out */
  float* episode_returns;     /* [n] in/out */
  int32_t* episode_lengths;   /* [n] in/out */
  double* stats;              /* [4] accumulated */
  float* raw_rewards;         /* [reward_raw_cols] accumulated */
  double* workspace;          /* [PHC_EPISODE_WORKSPACE_DOUBLES] */
} PhcEpisodeArgs;
PHC_API int phc_episode_update(const PhcEpisodeArgs* args, int64_t n, phc_stream_t stream);
/* stats[0..3] += sum over buckets; raw_rewards[c] += (sum over buckets of column 4 + c) / n; the buckets are zeroed */
PHC_API int phc_episode_fold(double* ep_sums, int32_t num_buckets, int32_t raw_cols, int64_t n, double* stats,
                             float* raw_rewards, phc_stream_t stream);

/* The env's AMP observation buffers                          envs/humanoid_phc.py:596-611
 *   _amp_obs_buf [n, S, P]: slot 0 = _curr_amp_obs_buf, slots 1.. = _hist_amp_obs_buf; P as phc_amp_obs
 *   writes it.  Dense.  `env_mask` (NULL = all envs) selects envs by a byte mask, as phc_reset_envs does.
 *
 * phc_amp_step: per-step update (:153-156) — with roll_history the history roll of
 *   _update_hist_amp_obs (:1341-1350: slot k+1 <- slot k, i.e. the .clone() branch the reference takes on
 *   its pinned torch), then _compute_amp_observations (:1125-1176) writes slot 0 from the sim state:
 *   root = body 0, key bodies by id, dof_pos / dof_vel the strided dof-state views.  With
 *   roll_history == 0 and a mask it is _compute_amp_observations(env_ids) of a reset (:792).
 * phc_amp_init_ref: _init_amp_obs_ref (:805-819) for the selected envs — slot k >= 1 is the AMP
 *   observation of clip motion_ids[env] at motion_times[env] - k*dt (_get_amp_obs :821-838, no global
 *   offset), then the env's whole row is copied to amp_obs_demo_buf (may be NULL).  motion_ids /
 *   motion_times are indexed by env (after a reset: _sampled_motion_ids / _motion_start_times).
 *   With init_slot0 it is the whole _init_amp_obs(env_ids) (:791-799): slot 0 is written from the sim
 *   state first, as phc_amp_step(roll_history = 0) under the same mask would.  A block of 8 envs
 *   without a selected env reads 8 mask bytes and leaves. */
typedef struct PhcAmpEnvArgs {
  PhcBodyState body;           /* sim state views (phc_amp_step); num_bodies also bounds key_body_ids */
  const float* dof_pos;        /* [n,69] view (phc_amp_step)       humanoid_phc.py:535 */
  const float* dof_vel;        /* [n,69] view                      humanoid_phc.py:536 */
  int64_t dof_stride;          /* row stride in elements (both views) */
  int64_t dof_elem_stride;     /* 2 for the interleaved (pos, vel) dof state */
  int32_t key_body_ids[8];     /* _key_body_ids                    humanoid_phc.py:245 */
  int32_t num_key_bodies;
  int32_t num_sel;             /* dofs used (69 when dof_subset is NULL), a multiple of 3 */
  const int64_t* dof_subset;   /* NULL or [num_sel]                humanoid_phc.py:186-194 */
  uint32_t flags;              /* PHC_OBS_LOCAL_ROOT | PHC_OBS_ROOT_HEIGHT | PHC_OBS_UPRIGHT */
  int32_t num_steps;           /* S = num_amp_obs_steps <= 16      config.py:141 */
  int32_t obs_per_step;        /* P */
  int32_t init_slot0;          /* phc_amp_init_ref only: 1 = also write slot 0 from the sim state (:792), same launch */
  float* amp_obs_buf;          /* [n, S, P] */
  float* amp_obs_demo_buf;     /* [n, S, P] or NULL (phc_amp_init_ref) */
  const uint8_t* env_mask;     /* NULL or [n] */
} PhcAmpEnvArgs;
PHC_API int phc_amp_step(const PhcAmpEnvArgs* args, int64_t n, int32_t roll_history, phc_stream_t stream);
PHC_API int phc_amp_init_ref(const PhcLib* lib, const PhcAmpEnvArgs* args, const int64_t* motion_ids,
                             const float* motion_times, float dt, int64_t n, phc_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Motion-library build: the per-clip work of MotionLibSMPL.load_motions (motion_lib.py:257-428,
 * worker load_motion_with_skeleton :748-824) for all clips at once, on the device.  Inputs are the
 * pkl entries of scripts/phc_convert_amass_data.py:186-194 concatenated on the frame axis (after
 * the caller's max_length crop, :773-778) as fp64, exactly the dtypes the reference computes in:
 *   heading (optional, :789-799)  -> rotates the global rotations, the root translation and
 *                                    pose_aa[:, :3];
 *   SkeletonState.from_rotation_and_root_translation(is_local=False) (:806) -> lrs (fp64 product
 *   rounded to fp32, poselib_skeleton.py:575-594) and, by fp32 forward kinematics (:519-539), gts;
 *   SkeletonMotion.from_skeleton_state (:810, poselib_skeleton.py:1167-1251) -> gvs (np.gradient +
 *   gaussian_filter1d sigma 2 "nearest") and gavs; compute_motion_dof_vels_jit (:120-142) -> dvs.
 * grvs / gravs are gvs[:,0] / gavs[:,0].  fix_trans_height (:696-745) needs the SMPL mesh model and
 * is not implemented: this is the mesh_parsers == None path (:692-694, :801).  Clips need >= 2
 * frames (np.gradient raises below that); shorter clips get zero velocities.
 * ---------------------------------------------------------------------------------- */
#define PHC_BUILD_FILTER_RADIUS 8 /* int(4.0 * sigma + 0.5), sigma = 2: scipy.ndimage.gaussian_filter1d */
typedef struct PhcBuildArgs {
  const double* pose_quat_global;     /* [F,24,4] xyzw, 32-B aligned      motion_lib.py:784 */
  const double* root_trans;           /* [F,3] root_trans_offset          motion_lib.py:781 */
  const double* pose_aa;              /* [F,72] or NULL                   motion_lib.py:783 */
  const float* local_translation;     /* [M,24,3] skeleton_trees[m].local_translation (fp32, poselib_skeleton.py:318) */
  const int64_t* num_frames;          /* [M] */
  const int64_t* length_starts;       /* [M] exclusive prefix sum of num_frames */
  const double* fps;                  /* [M] curr_file.get("fps", 30)     motion_lib.py:810 */
  const double* heading_zw;           /* NULL or [M,2]: (sin, cos) of half the heading angle pi*(2u-1) */
  const int32_t* parent_indices_host; /* HOST [24], -1 for the root, parents precede children */
  const double* filter_weights_host;  /* HOST [17] gaussian taps, scipy's _gaussian_kernel1d(2, 0, 8) */
  int64_t total_frames;               /* F */
  int64_t num_motions;                /* M */
  float* gts;                         /* [F,24,3] out */
  float* grs;                         /* [F,24,4] out, 16-B aligned */
  float* lrs;                         /* [F,24,4] out, 16-B aligned */
  float* gvs;                         /* [F,24,3] out */
  float* gavs;                        /* [F,24,3] out */
  float* dvs;                         /* [F,23,3] out */
  float* motion_aa;                   /* [F,72] out, NULL iff pose_aa is NULL */
  double* scratch;                    /* F*108 doubles of work space: [F,24,3] fp64 unfiltered angular velocity, then
                                         [F,24,3] fp32 unfiltered linear velocity */
} PhcBuildArgs;
PHC_API int phc_motion_build(const PhcBuildArgs* args, phc_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PHC_B200_H_ */
