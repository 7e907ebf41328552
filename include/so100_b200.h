/*
 * so100_b200.h — C ABI of the B200-native batched so100 simulator (libso100_b200.so).
 *
 * This is the drop-in boundary for ONE hot path of PieterBecking/so100-mujoco-rl: the per-step work of
 * Env01 / Env02 / Env05 (`reset()` / `step(a)`), which in the reference is Python task logic wrapped around
 * MuJoCo's `mj_step(model, data, nstep=16)`.  Reference interfaces replaced (paths relative to the reference repo):
 *
 *   so100_create      <- So100BaseEnv.__init__            src/so100_mujoco_rl/envs/env_base_01.py:35-61
 *                        (MjModel.from_xml_path + MujocoEnv.__init__, frame_skip 16) and
 *                        Env03._set_initial_values         src/so100_mujoco_rl/envs/env03_v1.py:35-57
 *   so100_reset       <- MujocoEnv.reset -> reset_model    env01_v1.py:39-63, env02_v1.py:70-81, env03_v1.py:203-215
 *   so100_step        <- Env01.step / Env02.step / Env03.step (used by Env05) + Env05._get_obs
 *                        env01_v1.py:15-37, env02_v1.py:18-50, env03_v1.py:124-201, env05_v1.py:32-75,
 *                        the 16x mujoco.mj_step at env01_v1.py:26 / env02_v1.py:39 / env03_v1.py:142,
 *                        the gymnasium TimeLimit wrapper (src/so100_mujoco_rl/__init__.py:5-45) and the
 *                        auto-reset that SB3's DummyVecEnv performs around a done env
 *   so100_get_state / so100_set_state  <- direct reads/writes of mjData (data.qpos, data.qvel, ...) used for tests
 *   so100_forward_dynamics <- one mj_forward restricted to the arm (debug/parity entry; not on the step path)
 *
 * Conventions
 *   - every entry point returns SO100_OK (0) or a negative error code; the message is available per thread through
 *     so100_last_error().  No C++ exception crosses this boundary.
 *   - all *_dev pointers are DEVICE pointers owned by the caller (e.g. torch tensors); the library never
 *     allocates or frees them.  `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all work
 *     is enqueued on it and the call returns without synchronising.
 *   - the *_host entry points take HOST pointers (pinned memory recommended), do the H2D/D2H copies themselves
 *     on `stream` and synchronise that stream before returning: this is the reference-facing call.
 *   - external observation / action layout is row-major [num_envs, dim] float32 (what SB3 / torch policies
 *     consume).  Internal state is structure-of-arrays.
 *   - one ctx per (device, task); calls on one ctx must be serialised by the caller.
 */
#ifndef SO100_B200_H
#define SO100_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SO100_ABI_VERSION 3
#define SO100_NJ 6            /* arm hinges incl. the jaw */
#define SO100_MAX_START 64    /* rows available for Env01 start poses (reference: 36) */
#define SO100_MAX_GROUPS 16   /* env groups of the asynchronous host path */
#define SO100_MAX_PAD 8       /* primitive box colliders on the arm (reference: 4 + 4 jaw pads) */

/* error codes */
#define SO100_OK 0
#define SO100_ERR_ARG (-1)
#define SO100_ERR_CUDA (-2)
#define SO100_ERR_MODEL (-3)
#define SO100_ERR_STATE (-4)

/* tasks (reference env ids "Env01-v1", "Env02-v1", "Env05-v1") */
#define SO100_TASK_ENV01 1
#define SO100_TASK_ENV02 2
#define SO100_TASK_ENV05 5
#define SO100_TASK_ENV06 6   /* Env02's scene and reset, no relocation, gripper-closing reward (envs/env06_v1.py, env_base_06.py) */

/* quirk flags (task_cfg.flags). Default 0 reproduces the reference bit for bit in behaviour. */
#define SO100_FLAG_FRESH_FK_ON_RESET 1u /* run kinematics in reset (the reference does not: SURVEY Q2) */
#define SO100_FLAG_CLIP_ACTIONS 2u      /* clip actions to [-1,1] on device (the reference env does not) */
#define SO100_FLAG_GENERIC_KERNEL 4u    /* never use the model-specialised kernel (tests: generic vs specialised) */
#define SO100_FLAG_STATIC_BLOCK 8u      /* hold the Env01/02/06 block at its spawn pose: no gravity, no floor contact (round-1 behaviour) */
#define SO100_FLAG_ARM_CONTACT 16u      /* jaw-pad <-> floor contact (the reference's primitive colliders).  Exact against the oracle, but the
                                           Newton solve it needs is a long serial chain per touching env: ~18x the step time at 65 536 envs
                                           (DESIGN.md "Arm-floor contact"), so it is opt-in; without it the arm passes through the floor */

/*
 * Model constants as they stand in the MJCF (so_arm100_camera.xml + env01.xml), nothing derived.
 * Index 0..5 = Rotation, Pitch, Elbow, Wrist_Pitch, Wrist_Roll, Jaw; body i carries joint i and is the child of
 * body i-1 (body -1 = the welded Base).  Quaternions are (w,x,y,z) and need not be normalised.
 */
typedef struct so100_model {
  int32_t struct_size;       /* = sizeof(so100_model), checked by so100_create */
  int32_t nsubstep;          /* frame_skip, 16 (env_base_01.py:45) */
  double timestep;           /* 0.002 */
  double gravity[3];         /* 0 0 -9.81 */
  double base_pos[3];        /* Base body in the world (welded) */
  double base_quat[4];
  double body_pos[SO100_NJ][3];
  double body_quat[SO100_NJ][4];
  double body_ipos[SO100_NJ][3];
  double body_iquat[SO100_NJ][4];
  double body_mass[SO100_NJ];
  double body_inertia[SO100_NJ][3]; /* diaginertia in the inertial frame */
  double jnt_axis[SO100_NJ][3];     /* in the body frame; joint anchor is the body origin */
  double jnt_range[SO100_NJ][2];
  double jnt_armature[SO100_NJ];
  double jnt_frictionloss[SO100_NJ];
  double jnt_solref_limit[SO100_NJ][2];
  double jnt_solimp_limit[SO100_NJ][5];
  double dof_solref_friction[SO100_NJ][2];
  double dof_solimp_friction[SO100_NJ][5];
  double act_kp[SO100_NJ];
  double act_dampratio[SO100_NJ];   /* >0: kv = dampratio*2*sqrt(kp*dof_M0) (MuJoCo mj_setConst) */
  double act_kv[SO100_NJ];          /* used when act_dampratio <= 0 */
  double act_ctrlrange[SO100_NJ][2];
  double act_forcerange[SO100_NJ][2];
  int32_t ee_body;           /* Fixed_Jaw = 4 */
  int32_t wrist_body;        /* Wrist_Pitch_Roll = 3 */
  int32_t cam_body;          /* body carrying so100_end_point_camera = 4 */
  int32_t _pad0;
  double ee_offset[3];       /* (0,-0.1,0) in the Fixed_Jaw frame, env_base_01.py:125 */
  double cam_pos[3];
  double cam_quat[4];
  double cam_fovy_deg;       /* 120 */
  /* block <-> floor contact (env01.xml:29-34, :39): a free box on the z = 0 plane, all contact parameters default.
     The arm cannot reach the block's spawn annulus with a colliding body (env01.xml:42-49 excludes the others), so
     the block only ever moves along z: see DESIGN.md "Block-floor contact". */
  double block_half_z;       /* box half-size along z, 0.01 (env01.xml:32) */
  double block_mass;         /* 0.008 = default density 1000 x 0.02^3 (inertiafromgeom="true", env01.xml:2) */
  double block_friction;     /* sliding friction of the geom pair (max of the two geoms) = 1 */
  double contact_solref[2];  /* 0.02 1 */
  double contact_solimp[5];  /* 0.9 0.95 0.001 0.5 2 */
  int32_t block_ncon;        /* contact points of MuJoCo's plane-box collider for a flat box: 4; 0 = the pair does not collide */
  int32_t _pad1;
  /* arm <-> floor contact: the PRIMITIVE box colliders the reference MJCF puts on the jaws (so_arm100_camera.xml:60-61
     class finger_collision; :108-111 fixed_jaw_pad_1..4; :120-123 moving_jaw_pad_1..4) against the floor plane
     (env01.xml:39; env01.xml:42-49 excludes only block <-> arm pairs).  Boxes are axis-aligned in their body frame.
     Geom parameters as they stand in the MJCF; the library mixes the pair like mj_contactParam (mean solref / solimp,
     max friction) and clamps solimp like getsolparam.  The arm's mesh colliders are not available (DESIGN.md D2). */
  int32_t n_pad;             /* 8; 0 = the arm has no primitive colliders */
  int32_t _pad2;
  int32_t pad_body[SO100_MAX_PAD];   /* 4 = Fixed_Jaw, 5 = Moving_Jaw */
  double pad_pos[SO100_MAX_PAD][3];  /* box centre in the body frame */
  double pad_size[SO100_MAX_PAD][3]; /* half sizes */
  double pad_solref[2];      /* 0.01 1 */
  double pad_solimp[5];      /* 2 1 0.01 0.5 2 (clamped to 0.9999 0.9999 ... at use) */
  double pad_friction;       /* 1 */
  double floor_solref[2];    /* 0.02 1 */
  double floor_solimp[5];    /* 0.9 0.95 0.001 0.5 2 */
  double floor_friction;     /* 1 */
} so100_model;

/* Task constants: the literals of envs/utils.py, env03_v1.py, env05_v1.py, env_base_02.py, __init__.py. */
typedef struct so100_task_cfg {
  int32_t struct_size;       /* = sizeof(so100_task_cfg) */
  int32_t task;              /* SO100_TASK_* */
  int32_t num_envs;          /* envs owned by this ctx */
  int32_t max_episode_steps; /* TimeLimit: 4000 (Env01) / 6000 (Env02, Env05) */
  int64_t env_offset;        /* global id of local env 0 (RNG is keyed by the global id) */
  uint64_t seed;
  uint32_t flags;            /* SO100_FLAG_* */
  int32_t n_start;           /* rows used in start_positions (Env01) */
  double joint_step_scale;   /* 0.075, utils.py:9 */
  double start_positions[SO100_MAX_START][SO100_NJ]; /* VALID_START_POSITIONS, utils.py:13-50 */
  double rest_position[SO100_NJ];                     /* REST_POSITION (Env02), utils.py:11 */
  double start_position05[SO100_NJ];                  /* START_POSITION (Env05), env03_v1.py:10 */
  double block_dist_range[2];   /* Env01 (0.18,0.42) env01_v1.py:45; Env02 (0.22,0.42) env02_v1.py:55 */
  double block_theta_half;      /* pi/4 */
  double reach_threshold;       /* 0.03, env02_v1.py:29 */
  double block_space_start[2][3]; /* env05_v1.py:13-16 */
  double block_space_end[2][3];   /* env05_v1.py:17-20 */
  double block_speed_min, block_speed_max; /* env03_v1.py:21-22 */
  double ramp_seconds;          /* 12.0, env03_v1.py:126 */
  double cam_res_w, cam_res_h;  /* 1080 x 1920, env_base_02.py:22-23 */
  double obs_noise;             /* 0.05, env05_v1.py:44-45 */
  int32_t lost_limit;           /* 30, env03_v1.py:155 */
  int32_t _pad0;
} so100_task_cfg;

/*
 * Flat view of the per-env simulation state for parity tests.  All pointers are DEVICE pointers to arrays the
 * caller owns, laid out structure-of-arrays: field[k][env] at  ptr[k * num_envs + env].  NULL = skip the field.
 */
typedef struct so100_state_view {
  float *qpos;          /* [6][N] */
  float *qvel;          /* [6][N] */
  float *qacc_warm;     /* [6][N]  previous substep's qacc (solver warm start, mjData.qacc_warmstart) */
  float *qpos_comp;     /* [6][N]  compensation term of the fp32 qpos integration: qpos_exact ~ qpos - qpos_comp */
  float *block;         /* [4][N]  block position (qpos[6:9] of the reference) and its z velocity (qvel[8]) */
  float *snap;          /* [12][N] stale kinematics snapshot: Env01/02 end_pos(0..2), wrist_z(3), block_xpos(4..6);
                                    Env05 cam_xpos(0..2), cam_xmat(3..11 row-major) */
  float *aux;           /* [24][N] task scalars: Env02 block_pos(0..2), last_block_pos(3..5); Env05 cmd(0..5),
                                    last_angvel(6..11), target(12..14), target_dt(15), last_centre(16..17) */
  int32_t *counters;    /* [4][N]  elapsed_steps, flags (16 = scheduling hint "pads touched the floor"; 1 ever_stepped, 2 has_last_block, 4 angvel_valid,
                                    8 centre_valid), miss_count, target_t0_step */
  float *ep_return;     /* [N] */
} so100_state_view;

typedef struct so100_ctx so100_ctx;

int so100_abi_version(void);
const char *so100_last_error(void);
/* Hash of the env-step kernel's sources this library was built from (keys the ncu figures in profiles/). */
const char *so100_build_id(void);

int so100_obs_dim(int task);   /* 15 for Env01/Env02/Env06, 8 for Env05; <0 on unknown task */
int so100_act_dim(int task);   /* 6 */

/* Parse-free construction: the caller has read the MJCF (see so100_mujoco_rl_b200/model.py) and hands over constants. */
int so100_create(const so100_model *model, const so100_task_cfg *cfg, int device, so100_ctx **out);
void so100_destroy(so100_ctx *ctx);

/*
 * Reset.  mask_dev == NULL resets every env, else only envs with mask_dev[i] != 0.  Writes the reset observation
 * of the envs that were reset into obs_dev[N, obs_dim] (rows of other envs are left untouched).
 */
int so100_reset(so100_ctx *ctx, const uint8_t *mask_dev, float *obs_dev, void *stream);

/*
 * One env step for all envs: pre-step task logic, 16 physics substeps, observation, reward, termination,
 * TimeLimit truncation, and auto-reset of finished envs (SB3 VecEnv semantics: obs_dev holds the first observation
 * of the next episode for finished envs and terminal_obs_dev their last observation).
 * Optional outputs may be NULL: terminal_obs_dev [N, obs_dim], ep_return_dev [N] / ep_len_dev [N] (return and
 * length of the episode that just finished; only written for finished envs).
 */
int so100_step(so100_ctx *ctx, const float *actions_dev, float *obs_dev, float *reward_dev,
               uint8_t *terminated_dev, uint8_t *truncated_dev, float *terminal_obs_dev,
               float *ep_return_dev, int32_t *ep_len_dev, void *stream);

/*
 * Debug / parity triage (SURVEY.md §8 b): advance the PHYSICS of every env by n_substeps x mj_step under
 * ctrl_dev[N, 6] (absolute position-servo targets, i.e. mjData.ctrl), with no task logic around it: no reward,
 * observation, episode counters, auto-reset or RNG tick.  Read the per-substep state back with so100_get_state
 * (qpos, qvel, qacc_warm, block; `snap` holds the kinematics of the last substep's start state, as after a full step).
 * The reference-side equivalent is `mujoco.mj_step(model, data, nstep=n)` at env01_v1.py:26.
 */
int so100_step_substeps(so100_ctx *ctx, const float *ctrl_dev, int n_substeps, void *stream);

/*
 * Host-buffer variants (the reference-facing call), synchronised on return.  Page-locked (pinned / registered) host
 * buffers are read and written by the kernel directly over the host link: ONE launch per step, every CTA pulling its
 * action rows when it starts and posting its obs / reward / flag rows - and the terminal rows of envs whose episode
 * ended - when it ends.  At 65 536 envs all CTAs are resident at once, so the three phases (actions in, arithmetic,
 * results out) run in series; so100_step_host_async below overlaps them across env groups.  Pageable buffers go through
 * chunked H2D copy -> kernel -> D2H copy on helper streams (terminal rows are then copied only on steps in which some
 * episode ended).
 * Environment knobs (experiments): SO100_HOST_ZEROCOPY=0 forces the copy pipeline, SO100_HOST_CHUNKS=1..16 its chunk count.
 */
int so100_reset_host(so100_ctx *ctx, float *obs_host, void *stream);
int so100_step_host(so100_ctx *ctx, const float *actions_host, float *obs_host, float *reward_host,
                    uint8_t *terminated_host, uint8_t *truncated_host, float *terminal_obs_host,
                    float *ep_return_host, int32_t *ep_len_host, void *stream);

/*
 * Pipelined host path (the caller of the reference, main.py:56-64, is host-side code: a policy that maps a batch of
 * observations to a batch of actions).  The envs of a ctx are split into n_groups contiguous ranges
 * (so100_host_group_range); so100_step_host_async enqueues ONE group's step on that group's own stream and returns at
 * once, so100_step_host_wait blocks until that group's rows are in the host buffers.  With >= 2 groups in rotation
 *     async(g0) async(g1) ... | wait(g0) [policy on g0's rows] async(g0) | wait(g1) [policy on g1's rows] async(g1) | ...
 * one group's results cross the host link while another group's arithmetic runs, and the link is used in both
 * directions at once; the floor is max(kernel, D2H) instead of their sum.
 * All pointers are the FULL [num_envs, dim] host arrays of so100_step_host (page-locked: required here); a group reads
 * and writes only its own rows.  `stream` is the caller's stream: the group's step is ordered after the work this library
 * has enqueued on it (so100_reset, so100_set_state, ...).
 * Every group counts its own steps; the RNG tick of a group's k-th step is k, so stepping all groups once equals one
 * so100_step_host / so100_step call bit for bit.  Full-batch calls (so100_step, so100_step_host) return
 * SO100_ERR_STATE while groups are at different step counts or have a step in flight.
 */
int so100_host_groups(so100_ctx *ctx, int n_groups);   /* 1..SO100_MAX_GROUPS; default 1 = the whole batch */
int so100_host_group_range(so100_ctx *ctx, int group, int *env_lo, int *env_hi);
int so100_step_host_async(so100_ctx *ctx, int group, const float *actions_host, float *obs_host, float *reward_host,
                          uint8_t *terminated_host, uint8_t *truncated_host, float *terminal_obs_host,
                          float *ep_return_host, int32_t *ep_len_host, void *stream);
int so100_step_host_wait(so100_ctx *ctx, int group);
/* Blocks until ANY group with a step in flight has finished and returns its index in *group (-1: nothing in flight).
   Serving groups in completion order keeps them from queueing up behind the slowest one. */
int so100_step_host_wait_any(so100_ctx *ctx, int *group);

int so100_get_state(so100_ctx *ctx, const so100_state_view *view, void *stream);
int so100_set_state(so100_ctx *ctx, const so100_state_view *view, void *stream);

/* Re-key the counter-based RNG (gymnasium `reset(seed=...)` / SB3 `VecEnv.seed`): takes effect from the next reset / step. */
int so100_set_seed(so100_ctx *ctx, uint64_t seed);

/* global step counter t (number of so100_step calls so far); part of the RNG key. */
int so100_get_tick(so100_ctx *ctx, int64_t *tick);
int so100_set_tick(so100_ctx *ctx, int64_t tick);

/*
 * Debug / parity entry: for n arbitrary (qpos,qvel,ctrl) triples (SoA [6][n] each, device) evaluate one forward
 * dynamics pass with a cold start: M (21 lower-triangle entries, row-major i>=j), bias (6), qacc (6),
 * and the kinematics snapshot (end_pos 3, wrist 3, cam_xpos 3, cam_xmat 9 = 18).  Any output may be NULL.
 */
int so100_forward_dynamics(so100_ctx *ctx, int n, const float *qpos_dev, const float *qvel_dev,
                           const float *ctrl_dev, float *M_dev, float *bias_dev, float *qacc_dev,
                           float *kin_dev, void *stream);

/*
 * Host-side fp64 evaluation of the SAME recursion templates the kernels instantiate in fp32 (csrc/so100_dyn.cuh);
 * needs no GPU.  It exists so that the kernel mathematics can be checked against the oracle on a CPU-only machine
 * and is how so100_create derives dof_M0 / kv / invweight0.  Row-major host arrays: qpos/qvel/ctrl [n][6],
 * M [n][21] (packed lower triangle), bias [n][6], qacc [n][6] (cold start, `sweeps` Gauss-Seidel sweeps),
 * kin [n][18] (end_pos 3, wrist 3, cam_xpos 3, cam_xmat 9).  Outputs may be NULL.  variant 0 = generic recursion,
 * 1 = the generated model-specialised code (error if `model` is not the one it was generated from), 2 = the generic
 * recursion instantiated in fp32 (what the kernels compute, incl. the arm-floor contact solve; kin is not written).
 * Samples whose jaw pads touch the floor are solved by the contact path (Newton), the others by `sweeps` Gauss-Seidel sweeps.
 */
int so100_host_forward(const so100_model *model, int n, const double *qpos, const double *qvel, const double *ctrl,
                       double *M, double *bias, double *qacc, double *kin, int sweeps, int variant);

/*
 * Host emulation of the kernels' substep loop (same templates; no GPU): advances n states by n_substeps x mj_step under
 * ctrl, in place.  Row-major host arrays [n][6].  variant 0 = fp64, 2 = fp32 incl. the compensated position sum (what the
 * generic kernel computes).  stats (5 x int64, may be NULL): contact substeps, gradient/Hessian evaluations of the contact
 * solve, its line-search evaluations, the largest evaluation count of one solve, unconverged solves.
 */
int so100_host_substeps(const so100_model *model, int n, double *qpos, double *qvel, double *qacc_warm, const double *ctrl,
                        int n_substeps, int variant, int64_t *stats);

/*
 * The link constants the kernels consume, as the library derives them from the MJCF numbers (fp64, host only):
 * for each link i = 0..5: R[9] p[3] m h[3] I[6] armature (23 doubles), then the base acceleration a0[3] = 141 doubles.
 * Frames are re-based so that every hinge turns about local +z (csrc/so100_dyn.cuh).  tools/gen_so100_dyn.py reads
 * these to emit the model-specialised straight-line dynamics (csrc/so100_dyn_gen.cuh).
 */
#define SO100_N_DYN_CONSTANTS 141
int so100_host_constants(const so100_model *model, double *out /*[141]*/);

/*
 * The fp32 constraint-solver and servo constants the kernels consume (host only): friction-loss rows (D, B, loss),
 * joint ranges, limit rows (B, K, invweight0, solimp and its reciprocals), then kp, kv, ctrlrange, forcerange, timestep.
 * then the block-floor contact constants (13).  16 x 6 + 6 x 6 + 1 + 13 floats.  tools/gen_so100_dyn.py bakes them into csrc/so100_dyn_gen.cuh as literals.
 */
#define SO100_N_SOLVER_CONSTANTS 146
int so100_host_solver_constants(const so100_model *model, float *out, int n_out /* = SO100_N_SOLVER_CONSTANTS */);

/*
 * Per-env dynamics randomisation.  Opt-in: until ranges are set every env runs on the model's constants.  Once set, each
 * env holds its own fp32 servo gain kp, damping kv, forcerange and joint friction loss (30 floats per env; at the first
 * call every env starts from the ctx's constants) and redraws them at every episode reset: the auto-reset in so100_step*
 * (termination, truncation, non-finite state) and so100_reset (masked or not); nothing else redraws them.  Draws are
 * keyed by (seed, env_offset + env, tick): results do not depend on sharding, env groups or the host path.  With scales
 *   s = lo + (hi - lo) u,  u uniform in [0, 1):   kp = kp0 s_kp,  kv = kv0 sqrt(s_kp) s_damping,
 *   forcerange = forcerange0 s_force (both ends),  frictionloss = frictionloss0 s_frictionloss
 * where kp0, ... are the model's fp32 constants; s_damping is the damping ratio relative to the model's.  [1, 1] leaves a
 * parameter at the model's value bit for bit.  Env i then steps bit for bit like env i of a ctx whose model carries its
 * values (act_dampratio = 0, act_kv = kv).  Link masses, inertias and armature are not randomised.
 */
typedef struct so100_param_ranges {   /* scale ranges [lo, hi] per joint; lo == hi == 1 leaves a parameter at the model's value */
  int32_t struct_size, _pad0;         /* = sizeof(so100_param_ranges) */
  double kp[SO100_NJ][2];             /* kp = model kp x U, lo > 0 */
  double damping[SO100_NJ][2];        /* kv = model kv x sqrt(kp scale) x U (damping ratio relative to the model's), lo >= 0 */
  double forcerange[SO100_NJ][2];     /* both ends of the model's forcerange x U, lo > 0 */
  double frictionloss[SO100_NJ][2];   /* model frictionloss x U, lo >= 0 */
} so100_param_ranges;
/* DEVICE pointers to [6][N] fp32 arrays (SoA, [joint][env]); NULL = skip the field */
typedef struct so100_param_view { float *kp, *kv, *force_lo, *force_hi, *frictionloss; } so100_param_view;

/* ranges == NULL: off, back to the model's constants and the default kernels.  A change of ranges applies from each env's
   next reset.  Synchronous. */
int so100_set_param_ranges(so100_ctx *ctx, const so100_param_ranges *ranges);
/* Read / overwrite the per-env values (SO100_ERR_STATE while ranges are off); written values hold until the env's next
   reset.  All three calls return SO100_ERR_STATE while an asynchronous group step is in flight. */
int so100_get_env_params(so100_ctx *ctx, const so100_param_view *view, void *stream);
int so100_set_env_params(so100_ctx *ctx, const so100_param_view *view, void *stream);

/*
 * Actuator latency and joint-angle observation noise, for policies meant for the physical arm.  Opt-in: until a config
 * is set, a new servo target acts from the first substep of the env step and the observed joint angles are exact.
 *
 * Latency.  Each env holds an integer latency d in [lo, hi] substeps (0 <= lo <= hi <= nsubstep).  In an env step,
 * substeps 0 .. d-1 run on the env's PREVIOUS servo target and substeps d .. nsubstep-1 on the target this step's action
 * sets; d = 0 is the behaviour without a config, d = nsubstep runs the whole step on the previous target.  The target is
 * the full control value before clamping: Env01/02/06 keep the pair (ctrl_hi, ctrl_lo) = (qpos, a * joint_step_scale -
 * qpos_comp) per env (ctrl_prev); Env05's previous target is its previous command, aux[0:6] of the state.  Substep 0 and
 * substep d both get the first substep's Gauss-Seidel sweeps, so a latency-d step equals so100_step_substeps(d, previous
 * target) followed by so100_step_substeps(nsubstep - d, new target).  d is drawn at every episode reset and only then,
 * d = lo + umulhi(x, hi - lo + 1) on one Philox block (stream 14 at the auto-reset in so100_step*, including the
 * non-finite forced reset; 22 at so100_reset), and the previous target becomes the reset pose: (qpos_reset, 0) for
 * Env01/02/06, the start pose in aux for Env05.  so100_step_substeps (explicit ctrl), so100_set_state and Env02
 * relocations leave d and ctrl_prev alone.
 *
 * Noise.  Env01/02/06: obs[:, j] (j < 6, the joint angle) becomes fp32(q_j + fp32(sigma_j z_j)) with z standard normals
 * (Box-Muller on two Philox blocks, as the PPO act kernel; z[0..5] of the 8 it gives) on streams 24-25 for the step's
 * observation (also the terminal_obs row), 26-27 for the auto-reset's first observation and 28-29 at so100_reset.  Output
 * only: state, reward, flags, ep_return and ep_len do not depend on it.  sigma_j == 0 leaves the column's bits untouched.
 * Env05 observes its commanded angles, which the robot knows exactly: a non-zero sigma there is SO100_ERR_ARG.
 *
 * A config applies from each env's next reset (latency) and from the next step (noise).  At the first call every env has
 * d = 0 and, Env01/02/06, ctrl_prev = the exact current position (qpos, -qpos_comp).  All draws are keyed by (seed,
 * env_offset + env, tick, stream): shards, env groups and the host path stay bit-exact.
 */
typedef struct so100_sim2real {
  int32_t struct_size;            /* = sizeof(so100_sim2real) */
  int32_t latency[2];             /* substeps [lo, hi], 0 <= lo <= hi <= nsubstep */
  int32_t _pad0;
  double obs_noise[SO100_NJ];     /* std (rad) of the noise on observed joint angle j, finite, >= 0; Env05: all 0 */
} so100_sim2real;
/* DEVICE pointers; NULL = skip.  latency [N]; ctrl_prev_hi / _lo [6][N] (Env01/02/06 only: Env05's is aux[0:6]) */
typedef struct so100_actuator_view { int32_t *latency; float *ctrl_prev_hi, *ctrl_prev_lo; } so100_actuator_view;

/* cfg == NULL: latency and noise off at once, back to the default kernels unless param ranges are set.  Synchronous. */
int so100_set_sim2real(so100_ctx *ctx, const so100_sim2real *cfg);
/* Read / overwrite the per-env actuator state (SO100_ERR_STATE while no config is set; SO100_ERR_ARG for ctrl_prev on
   Env05); written values hold until the env's next reset, and a latency outside [0, nsubstep] acts as the nearer end.
   All three calls return SO100_ERR_STATE while an asynchronous group step is in flight. */
int so100_get_actuator_state(so100_ctx *ctx, const so100_actuator_view *view, void *stream);
int so100_set_actuator_state(so100_ctx *ctx, const so100_actuator_view *view, void *stream);

/* Which step kernel this ctx launches: 0 = generic (constants at run time), 1 = specialised to the baked so100 model. */
int so100_kernel_variant(so100_ctx *ctx);

/* Derived constants as the library computed them (host, fp64): dof_M0[6], kv[6], invweight0[6]. */
int so100_get_derived(so100_ctx *ctx, double *dof_M0, double *kv, double *invweight0);

/* Kernel launches issued by this ctx so far; env steps in which the last Gauss-Seidel sweep of some substep still
   moved qacc by more than 2e-3 (relative; the sweep itself contracts the error ~100x further); envs force-reset because their state went non-finite (device counters, syncs). */
int so100_get_stats(so100_ctx *ctx, int64_t *launches, int64_t *solver_fallbacks, int64_t *nan_resets);

/*
 * Bench utility (not part of the env API): measures this GPU's achievable FP32 FMA rate with a register-resident
 * FFMA loop (8 independent chains per thread, every SM filled) and returns TFLOP/s (FMA = 2 FLOP).  It is the
 * denominator of the FP32 roofline in bench.py, because MEASURED_PEAKS.json carries no CUDA-core figure.
 */
int so100_bench_fp32_peak(int device, int iters, double *tflops_out);

#ifdef __cplusplus
}
#endif
#endif /* SO100_B200_H */
