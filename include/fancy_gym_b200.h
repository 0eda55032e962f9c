/*
 * fancy_gym_b200 — C ABI of the B200-native movement-primitive black-box rollout path.
 *
 * This is the drop-in boundary for ONE path of ALRhub/fancy_gym (reference v0.3.0):
 *   BlackBoxWrapper.step(params)                fancy_gym/black_box/black_box_wrapper.py:150-217
 *     get_trajectory -> mp_pytorch traj_gen     fancy_gym/black_box/black_box_wrapper.py:96-120
 *     tracking controller                       fancy_gym/black_box/controller/{pd,vel,pos}_controller.py
 *     classic_control reacher step              fancy_gym/envs/classic_control/ (all files)
 * The reference is pure Python and has no FFI of its own; the entry points below are what a
 * ctypes binding inside fancy_gym would call instead of the Python loops cited at each function
 * (INTEGRATION.md shows that binding).  Plain pointers and sizes only: no torch / C++ types.
 *
 * Conventions
 *   - every function returns fg_status (0 = OK, < 0 = error); fg_last_error() returns a
 *     thread-local message.  No exceptions cross the ABI.
 *   - the CALLER owns every device buffer (PyTorch allocates them); the library allocates only
 *     inside fg_handle (basis / phase tables) at fg_create.  No hidden synchronisation, no
 *     allocation per call; launches are ordered on the `stream` argument (a cudaStream_t cast
 *     to void*, 0 = default stream).
 *   - a handle is immutable after creation: calls are re-entrant and stream ordered.  One handle
 *     per (config, device).
 *   - all matrices are row-major and dense.
 */
#ifndef FANCY_GYM_B200_H
#define FANCY_GYM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FG_ABI_VERSION 2
#define FG_MAX_DOF 8      /* links / action dimensions handled in registers */
#define FG_MAX_OBS 40     /* 3*FG_MAX_DOF + 5 (+1 time-aware column) */
#define FG_MAX_PLANS 32   /* plans of one episode that one fg_rollout launch can loop over */

typedef enum fg_status {
  FG_OK = 0,
  FG_ERR_INVALID = -1,      /* bad argument (maps to ValueError) */
  FG_ERR_UNSUPPORTED = -2,  /* valid but not implemented combination (NotImplementedError) */
  FG_ERR_CUDA = -3,         /* CUDA runtime error (RuntimeError) */
  FG_ERR_NOMEM = -4
} fg_status;

/* step-based env restated by the fused kernel (fancy_gym/envs/classic_control/ ...) */
typedef enum fg_env_kind {
  FG_ENV_HOLE_REACHER = 0,     /* hole_reacher/hole_reacher.py, velocity controlled */
  FG_ENV_VIAPOINT_REACHER = 1, /* viapoint_reacher/viapoint_reacher.py, velocity controlled */
  FG_ENV_SIMPLE_REACHER = 2,   /* simple_reacher/simple_reacher.py, torque controlled */
  FG_ENV_TOY = 3               /* the reference tests' ToyEnv (test/test_black_box.py:27-45): reward 1, never ends */
} fg_env_kind;

/* trajectory generator (mp_pytorch.mp.{ProMP,DMP,ProDMP}; factory:
 * fancy_gym/black_box/factory/trajectory_generator_factory.py:7-21) */
typedef enum fg_mp_kind {
  FG_MP_PROMP = 0,
  FG_MP_DMP = 1,
  FG_MP_PRODMP = 2,
  FG_MP_TRAJ = 3            /* desired trajectory supplied in HBM ([B,T,dof] pos and vel) */
} fg_mp_kind;

/* tracking controller (fancy_gym/black_box/factory/controller_factory.py:9-21) */
typedef enum fg_ctrl_kind {
  FG_CTRL_VELOCITY = 0,  /* vel_controller.py:8-9 */
  FG_CTRL_POSITION = 1,  /* pos_controller.py:8-9 */
  FG_CTRL_MOTOR = 2      /* pd_controller.py:21-29 */
} fg_ctrl_kind;

/* bits of the per-env `flags` output */
#define FG_FLAG_TERMINATED 1u
#define FG_FLAG_TRUNCATED 2u
#define FG_FLAG_SUCCESS 4u    /* info["is_success"] of the last executed step */
#define FG_FLAG_COLLIDED 8u   /* info["is_collided"] of the last executed step */

typedef struct fg_config {
  uint32_t struct_size;        /* sizeof(fg_config), checked */
  int32_t env_kind;            /* fg_env_kind */
  int32_t mp_kind;             /* fg_mp_kind */
  int32_t ctrl_kind;           /* fg_ctrl_kind */
  int32_t n_dof;               /* links == action dim, 1..FG_MAX_DOF */
  int32_t n_steps;             /* T: points of one planned trajectory (times init_time + dt*(1..T)) */
  int32_t n_basis;             /* K: weighted basis functions per dof */
  int32_t max_episode_steps;   /* gymnasium TimeLimit of the registration (200) */
  double dt;                   /* env.dt (base_reacher.py:21 -> 0.01) */

  /* PD gains (pd_controller.py:15-19), per joint */
  double p_gains[FG_MAX_DOF];
  double d_gains[FG_MAX_DOF];

  /* movement-primitive scalars */
  float tau;                   /* phase tau: DMP / ProDMP velocity un-scaling */
  float dmp_alpha;             /* DMP: alpha (25), beta = alpha/4 */
  float weights_scale;         /* DMP: multiplies the weights in-kernel (ProMP/ProDMP fold it into the tables) */
  float goal_scale;            /* DMP: multiplies the goal in-kernel */
  int32_t relative_goal;       /* ProDMP: goal += init_pos */

  /* env options (constructor kwargs of the reference envs) */
  int32_t allow_self_collision;
  int32_t allow_wall_collision;
  double collision_penalty;
  int32_t rew_fct;             /* hole reacher (hole_reacher.py:48-58): 0 = "simple" (hr_simple_reward.py),
                                  1 = "vel_acc" (hr_dist_vel_acc_reward.py), 2 = "unbounded" (hr_unbounded_reward.py) */
  int32_t wall_mode;           /* 0 = exact transition search over the 100 samples/link: closed-form estimate + fix-up (default),
                                  1 = literal evaluation of all 100 samples/link (hole_reacher.py:148-179), 2 = the same without
                                  skipping links that stay above ground, 3 = transition search by bisection (round 1) */
  int32_t time_aware;          /* append elapsed/max_episode_steps to obs (utils/wrappers.py:49-63) */

  /* observation compaction: obs_out[:, j] = full_step_obs[:, obs_index[j]] (context mask,
   * black_box_wrapper.py:89-94) */
  int32_t n_obs_out;
  int32_t obs_index[FG_MAX_OBS];

  /* Tables, HOST pointers, copied into the handle.  float32, row-major.
   *   ProMP : tab_a = weights_scale * Phi            [T, K]   (learnable columns only)
   *           tab_b = times[t+1] - times[t]          [T-1]
   *   DMP   : tab_a = x(t) * Phi                     [T, K]
   *           tab_b = scaled-time increments         [T-1]
   *   ProDMP: tab_a = [xi1, xi2, H_pos(0..K)]        [T, K+3]
   *           tab_b = [xi3, xi4, H_vel(0..K)]        [T, K+3]
   *   TRAJ  : unused (NULL) */
  const float* tab_a;
  const float* tab_b;
} fg_config;

struct fg_phase_basis;

/* Buffers of one fused-rollout launch.  DEVICE pointers.  B = number of envs. */
typedef struct fg_rollout_io {
  uint32_t struct_size;
  /* inputs */
  const float* params;     /* [B, P]: per dof K weights (+ goal for DMP / ProDMP), dof-major;
                              FG_MP_TRAJ: unused */
  const double* ctx;       /* [B, 4]  hole: x, width, depth, -   viapoint: via_x, via_y, goal_x, goal_y
                                      simple: goal_x, goal_y, -, -   toy: unused */
  const float* traj_pos;   /* FG_MP_TRAJ: [B, T, dof] */
  const float* traj_vel;   /* FG_MP_TRAJ: [B, T, dof] */
  /* persistent per-env state, in/out (reset writes it, every plan segment continues it) */
  double* q;               /* [B, dof] joint angles (base_reacher.py: _joint_angles) */
  double* v;               /* [B, dof] joint velocities (_angle_velocity) */
  int32_t* steps;          /* [B] env steps executed in this episode (_steps == TimeLimit._elapsed_steps) */
  uint8_t* done;           /* [B] episode over (terminated or truncated earlier): env is skipped */
  float* cond_pos;         /* [B, dof] condition_on_desired boundary values (black_box_wrapper.py:199-201) or NULL */
  float* cond_vel;         /* [B, dof] */
  int32_t use_cond;        /* 1: boundary condition = cond_pos/vel, 0: current q / v (black_box_wrapper.py:110-111) */
  int32_t write_cond;      /* 1: store the desired pos/vel of the last executed step of envs that stop early */
  /* outputs */
  double* ret;             /* [B] sum of step rewards of this segment (black_box_wrapper.py:216, np.sum) */
  int32_t* length;         /* [B] executed steps = infos['trajectory_length'] */
  uint8_t* flags;          /* [B] FG_FLAG_* */
  float* obs;              /* [B, n_obs_out] observation after the last executed step */
  double* info;            /* [B, 4] hole/viapoint: end_effector x,y; simple: reward_dist, reward_ctrl;
                              [2..3]: in/out state of rew_fct "unbounded" (end effector latched at step 180), else 0 */
  /* optional per-step outputs of verbose>=2 (black_box_wrapper.py:208-213); NULL to skip.
   * (infos['positions'] / ['velocities'] are the whole planned trajectory: use fg_trajgen.) */
  double* dbg_actions;     /* [B, T, dof] infos['step_actions'] */
  float* dbg_obs;          /* [B, T, n_obs_full] infos['step_observations'] */
  double* dbg_rewards;     /* [B, T] infos['step_rewards'] */
  /* optional unpacked copies of the flag bits, one byte (0 / 1) per env each, or NULL: what step() returns as
   * terminated / truncated and infos['is_success'] / ['is_collided'] without any post-processing kernel */
  uint8_t* flag_bytes;     /* [4, B]: rows terminated, truncated, success, collided */
  const int32_t* seg_steps_env; /* [B] or NULL: per-env bound on the steps of this segment (ragged sub-trajectories); the
                                   scalar seg_steps argument still bounds all of them */
  const float* prev_obs;   /* [B, n_obs_out] or NULL: observation / info rows reported for envs that are skipped because their */
  const double* prev_info; /* [B, 4] or NULL      episode ended in an earlier call (they keep reporting their last values)   */
  int32_t keep_state;      /* 1: q / v / steps / done are read but NOT written back: the batch can be evaluated again from the
                              same start state with other parameters (population-based search on one context) */
  /* Re-planning inside ONE launch (black_box_wrapper.py:197-203 with a schedule that depends on the step counter only — every
   * schedule in the reference has the form t % k == 0): n_plans > 1 makes `params` [B, n_plans, P]; plan j executes
   * plan_seg[j] steps (the schedule's break points, evaluated by the caller) and reads rows plan_row0[j] + t of the handle's
   * tables, which then hold the rows of all plans one after the other (each plan planned from its own start time, plus one
   * look-ahead row); plan_T = points of one plan.  The boundary condition of plan j + 1 is the env's state at the break or,
   * with write_cond != 0 (condition_on_desired), the desired state of the break step.  Every output buffer then holds
   * n_plans blocks ([n_plans, B, ...]: what the j-th step() call of the reference returns); an env whose episode ends in
   * plan j reports 0 steps and its last observation for the plans after it.  0 / 1: one plan (the seg_steps argument). */
  int32_t n_plans;
  int32_t plan_T;
  int32_t plan_seg[FG_MAX_PLANS];
  int32_t plan_row0[FG_MAX_PLANS];
  double* dbg_state;       /* [B, T, 2 * dof] or NULL: joint angles and velocities after every executed step (current_pos /
                              current_vel as black_box_wrapper.py:197 hands them to a state-dependent replanning_schedule) */
  /* Multi-GPU gather fused into the rollout (one process per GPU, env shards): n_peers > 0 makes every env ALSO store its
   * result row (return f64 | length i32 | flags u8 | 4 flag bytes, laid out as one block of B envs exactly like ret / length /
   * flags / flag_bytes of a contiguous result block) into the buffer of every peer, straight over NVLink:
   * peer_bufs[r] + peer_offset is where THIS rank's block lives inside rank r's gather buffer (peer-mapped device memory,
   * e.g. torch symmetric memory; peer_bufs itself is a DEVICE array of n_peers pointers).  No collective kernel runs: the
   * caller only orders a barrier behind the launch before the gathered blocks are read.  One plan per launch. */
  void* const* peer_bufs;
  int32_t n_peers;
  int64_t peer_offset;
  /* Per-env learned tau / delay evaluated INSIDE the rollout (no fg_trajgen_phase launch, no [B, T, dof] trajectory in HBM):
   * phase = HOST pointer to the generator constants (as for fg_trajgen_phase; its n_steps_env / times_table give ragged plans),
   * phase_tau / phase_delay [B] float32 and phase_times [T] float32 DEVICE pointers.  The handle is the ProMP / DMP handle of the
   * generator (its tables are not read).  Instantiated for the registry's shapes — 5 weighted RBFs of 5 or 6 in total (zero
   * padding in front), 5 or 2 links, velocity / motor control, no per-step buffers; FG_ERR_UNSUPPORTED otherwise (use
   * fg_trajgen_phase and a FG_MP_TRAJ handle).  Same arithmetic as fg_trajgen_phase with eval_f64 = 1: bit-identical results. */
  const struct fg_phase_basis* phase;
  const float* phase_tau;
  const float* phase_delay;
  const float* phase_times;
} fg_rollout_io;

/* Episode reset of the classic_control reachers on the device (replaces the host-side samplers
 * hole_reacher.py:60-112, viapoint_reacher.py:45-77, simple_reacher.py:46-96, base_reacher.py:73-93). */
typedef struct fg_reset_cfg {
  uint32_t struct_size;
  int32_t env_kind;            /* FG_ENV_HOLE_REACHER / _VIAPOINT_REACHER / _SIMPLE_REACHER */
  int32_t n_dof;
  int32_t random_start;        /* constructor kwarg random_start (base_reacher.py:77-86) */
  int32_t time_aware;          /* append the (zero) elapsed-time column to the observation */
  int32_t device;              /* CUDA device ordinal the buffers live on */
  /* fixed task context (constructor kwargs hole_x, hole_width, hole_depth | via_target, target | target);
   * has_fixed[i] == 0: entry i is sampled.  Layout as fg_rollout_io.ctx. */
  double fixed[4];
  int32_t has_fixed[4];
  int32_t n_obs_out;           /* observation compaction as in fg_config */
  int32_t obs_index[FG_MAX_OBS];
} fg_reset_cfg;

typedef struct fg_reset_io {
  uint32_t struct_size;
  const int64_t* seeds;        /* [B] per-env seeds (DEVICE) or NULL: env i uses seed0 + i */
  int64_t seed0;
  int32_t reseed;              /* 1: every env starts the numpy stream Generator(PCG64(SeedSequence(seed_i)));
                                  0: continue the streams stored in rng_state (reset(seed=None)) */
  uint64_t* rng_state;         /* [B, 5] in/out: PCG64 state hi, lo, increment hi, lo, buffered uint32 (bit 32 = valid) */
  const uint8_t* mask;         /* [B] or NULL: only envs with mask != 0 are reset (vector-env auto-reset of finished envs) */
  double* q;                   /* outputs: as fg_rollout_io */
  double* v;
  int32_t* steps;
  uint8_t* done;
  double* ctx;                 /* [B, 4] */
  float* obs;                  /* [B, n_obs_out] observation of the reset state, or NULL */
} fg_reset_io;

/* One control step of the step-based reachers (the `fancy/<Name>-v0` ids: env.step(action) as PPO / SAC call it). */
typedef struct fg_env_step_cfg {
  uint32_t struct_size;
  int32_t env_kind;            /* FG_ENV_HOLE_REACHER / _VIAPOINT_REACHER / _SIMPLE_REACHER */
  int32_t n_dof;               /* 2..7 */
  int32_t max_episode_steps;   /* gymnasium TimeLimit: truncated = steps >= max_episode_steps; <= 0: never truncates */
  double dt;                   /* env.dt (0.01) */
  int32_t allow_self_collision;
  int32_t allow_wall_collision;
  double collision_penalty;
  int32_t rew_fct;             /* hole reacher: 0 simple, 1 vel_acc, 2 unbounded (as fg_config) */
  int32_t action_f64;          /* 0: action is float32 [B, dof], 1: float64 (the reference's arithmetic follows the dtype) */
} fg_env_step_cfg;

typedef struct fg_env_step_io {
  uint32_t struct_size;
  const void* action;          /* [B, dof] float32 or float64 (cfg.action_f64); the env applies no clip */
  int32_t v_is_f32;            /* velocity-controlled envs: 1 if every env with steps > 0 holds the previous call's float32
                                  action in v (then acc = (a - v) / dt is float32 arithmetic), 0 otherwise */
  /* state, in/out (as fg_rollout_io; fg_reset writes it) */
  double* q;                   /* [B, dof] */
  double* v;                   /* [B, dof] */
  int32_t* steps;              /* [B] */
  uint8_t* done;               /* [B] out: terminated or truncated on this step */
  const double* ctx;           /* [B, 4] */
  double* latch;               /* [B, 2] hole reacher rew_fct "unbounded": end effector latched at step 180 or on a collision;
                                  written before it is read within an episode (no reset needed); NULL for the other envs */
  /* outputs */
  float* obs;                  /* [B, n_obs_full] full step observation (3*dof + 4 / 5 / 3 columns) */
  double* reward;              /* [B] */
  uint8_t* flag_bytes;         /* [4, B] rows terminated, truncated, is_success, is_collided (0 / 1) */
  double* info;                /* [B, 2] hole / viapoint: end effector x, y; simple: reward_dist, reward_ctrl */
} fg_env_step_io;

typedef struct fg_handle fg_handle;

const char* fg_last_error(void);
int32_t fg_abi_version(void);

/* Builds the immutable per-config handle on `device` (tables are uploaded synchronously here). */
fg_status fg_create(const fg_config* cfg, int32_t device, fg_handle** out);
fg_status fg_destroy(fg_handle* h);

/* Number of params per env the handle expects (P) and width of the full step observation. */
int32_t fg_num_params(const fg_handle* h);
int32_t fg_obs_full_dim(const fg_handle* h);

/*
 * Fused episode (segment) rollout — replaces the T-iteration Python loop of
 * BlackBoxWrapper.step (black_box_wrapper.py:150-217) together with get_trajectory (:96-120),
 * controller.get_action, np.clip (:176-179) and env.step
 * (base_reacher_direct.py:20-38 / base_reacher_torque.py:20-37) for B envs.
 * Executes at most `seg_steps` (<= n_steps) steps per env; an env stops earlier when it
 * terminates or hits max_episode_steps.  One CUDA thread owns one env; nothing per-step is
 * written to HBM unless a dbg_* pointer is given.
 */
fg_status fg_rollout(const fg_handle* h, const fg_rollout_io* io, int64_t B, int32_t seg_steps, void* stream);

/*
 * Stand-alone trajectory generation — replaces traj_gen.get_traj_pos()/get_traj_vel()
 * (black_box_wrapper.py:117-118).  bc_pos/bc_vel [B,dof] are the initial conditions passed to
 * set_initial_conditions (:113-114; ignored by ProMP, may be NULL).  pos_out/vel_out [B,T,dof].
 */
fg_status fg_trajgen(const fg_handle* h, const float* params, const float* bc_pos, const float* bc_vel,
                     float* pos_out, float* vel_out, int64_t B, void* stream);

/* Phase / basis generator constants for trajectory generation with a PER-ENV phase (learned tau / delay,
 * phase_generator_kwargs learn_tau / learn_delay; mp_pytorch phase_gn + basis_gn).  RBFs: exp(-(phase - center)^2 * bandwidth / 2),
 * normalised over all n_basis_total functions; only [first_learnable, first_learnable + n_basis) carry weights (zero padding). */
typedef struct fg_phase_basis fg_phase_basis;
struct fg_phase_basis {
  uint32_t struct_size;
  int32_t phase_kind;          /* 0 = linear, 1 = exponential decay exp(-alpha_phase * z) */
  double alpha_phase;
  int32_t n_basis_total;       /* <= 16 */
  int32_t first_learnable;
  double centers[16];          /* in phase space */
  double bandwidth[16];
  /* ProDMP only: the pre-integrated bases on the scaled-time grid z_j = j * scaled_dt (mp_pytorch ProDMPBasisGenerator
   * pre-compute; they depend on the construction-time tau only) — float64 DEVICE tables, rows = grid points */
  const double* pc_pos;        /* [n_pc, n_basis + 1] position bases (weights..., goal) */
  const double* pc_vel;        /* [n_pc, n_basis + 1] velocity bases */
  const double* pc_y;          /* [n_pc, 4]  y1, y2, dy1, dy2 of the homogeneous solution */
  int32_t n_pc;
  float scaled_dt;             /* float32(dt) / float32(tau at construction): grid step the library rounds indices with */
  float init_time;             /* boundary-condition time of this plan */
  double scale[17];            /* weights_scale (x n_basis), goal_scale (x auto-scale factors) */
  /* ragged plans (learn_sub_trajectories with a different tau per env): env b plans n_steps_env[b] <= n_steps points on
   * the time grid times_table[n_steps_env[b] * times_stride + i] (float32 DEVICE table with one row per possible length,
   * built by the caller with the library's own linspace); NULL / NULL: every env uses `times` and n_steps points */
  const int32_t* n_steps_env;
  const float* times_table;
  int32_t times_stride;
  /* readings of mp_pytorch that are kept switchable (fancy_gym_b200/mp/assumptions.py; the defaults are 1 and 1.0) */
  int32_t exp_right_clip;      /* exponential phase: 1 = x = exp(-alpha * clip(z, 0, 1)), 0 = exp(-alpha * max(z, 0)) */
  double basis_scale;          /* DMP: factor on the forcing basis x * Phi (weights_scale when it is not on the parameters) */
  int32_t eval_f64;            /* RBFs / exponential phase of ProMP and DMP: 1 = float64 rounded once to float32 (the arithmetic of
                                  the host-built shared tables; what the Python facade passes by default), 0 = float32 elementwise
                                  ops like the library's torch tensors (cheaper; velocities carry the library's float32 noise) */
};

/*
 * fg_trajgen with per-env tau / delay: the basis is evaluated in the kernel (ProMP, DMP) or looked up per env in the
 * pre-integrated tables (ProDMP) instead of read from the handle's shared per-time-point tables.  times [T] float32 time grid and tau / delay [B] float32 are DEVICE pointers; params holds the
 * MP parameters only (tau / delay already stripped).  The fused rollout consumes pos_out / vel_out through a FG_MP_TRAJ handle.
 */
fg_status fg_trajgen_phase(const fg_handle* h, const fg_phase_basis* pb, const float* times, const float* tau,
                           const float* delay, const float* params, const float* bc_pos, const float* bc_vel,
                           float* pos_out, float* vel_out, int64_t B, void* stream);

/*
 * Trajectory covariance of the probabilistic MPs — replaces mp_pytorch's ProMP / ProDMP get_traj_pos_cov() /
 * get_traj_pos_std() behind the traj_gen object (no call site inside fancy_gym; SURVEY.md §8 row a20):
 *   Sigma_y = Psi (L L^T) Psi^T + reg * max(diag) * I,   Psi = blockdiag over dof of the handle's basis [T, Kc]
 * with Kc = n_basis (ProMP) or n_basis + 1 (ProDMP: weights and goal).  Rows / columns are dof-major (d * T + t).
 *   params_L  [B, D, D], D = n_dof * Kc: lower-triangular Cholesky factor of the weight covariance (upper part ignored)
 *   cov_out   [B, n_dof*T, n_dof*T] or NULL;  std_out [B, T, n_dof] or NULL (sqrt of the regularised diagonal)
 *   work      [fg_traj_cov_work_floats(h, B)] float scratch
 *   reg_scope 0: max over each env's own diagonal; 1: max over the whole batch (what mp_pytorch does on a batched tensor)
 *   path      0: automatic; 1: CUDA cores; 2: tcgen05 tensor cores (3xTF32 split, TMEM accumulators)
 */
int64_t fg_traj_cov_work_floats(const fg_handle* h, int64_t B);
fg_status fg_traj_cov(const fg_handle* h, const float* params_L, float reg, int32_t reg_scope, float* cov_out,
                      float* std_out, float* work, int32_t path, int64_t B, void* stream);

/*
 * Resets B envs: samples the task context and the start pose with numpy-exact streams (env i == the reference env
 * reset with seed_i), zeroes velocities / step counters / done flags and writes the context observation.
 */
fg_status fg_reset(const fg_reset_cfg* cfg, const fg_reset_io* io, int64_t B, void* stream);

/*
 * Advances B step-based envs by ONE control step — replaces env.step(action) of base_reacher_direct.py:20-38 /
 * base_reacher_torque.py:20-37 with the reward of the configured env, plus gymnasium's TimeLimit truncation.
 * Envs that terminated or were truncated keep being stepped (an env that is not reset keeps integrating).  Launches on
 * the CURRENT device, on `stream`; no allocation, no synchronisation.  FG_ERR_UNSUPPORTED for the toy env and for n_dof
 * outside 2..7.
 */
fg_status fg_env_step(const fg_env_step_cfg* cfg, const fg_env_step_io* io, int64_t B, void* stream);

/*
 * FP32 FFMA-chain microbenchmark used as the roofline denominator of the fused rollout
 * (MEASURED_PEAKS.json has no CUDA-core figure).  Runs `iters` dependent FMA rounds of 8
 * independent chains per thread on `blocks` x 256 threads; *flops = 2 * fmas executed.
 */
fg_status fg_ffma_probe(int32_t blocks, int32_t iters, float* sink_dev, double* flops, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FANCY_GYM_B200_H */
