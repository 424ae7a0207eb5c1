/* drloco_b200.h — C ABI of libdrloco_b200.so, the B200-native batched DeepMimic walker environment.
 *
 * The reference (rgalljamov/DRLoco) has no native layer of its own: its environment step runs in Python
 * (drloco/mujoco/mimic_env.py:60-126) on top of gym's MujocoEnv -> mujoco-py -> the MuJoCo C library, one process per
 * environment behind Stable-Baselines3's SubprocVecEnv (drloco/common/utils.py:97-134).  This header is the boundary a
 * maintainer binds instead of that stack: every entry point below names the reference interface it replaces.
 *
 * Conventions
 *  - plain C types only; every pointer marked "device" is a CUDA device pointer owned by the caller (PyTorch tensors);
 *    the library borrows it for the duration of the enqueued work and never frees it.
 *  - all work is enqueued on the caller's stream (``void* stream`` is a cudaStream_t); no hidden device synchronisation.
 *  - return value 0 = success, negative = DrlStatus error; message through drl_last_error() (thread local).
 *  - simulator blow-ups are not errors: the environment reports done=1 with reward 0 (mimic_env.py:86-91).
 */
#ifndef DRLOCO_B200_H
#define DRLOCO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DRL_ABI_VERSION 4

#define DRL_MAX_DOF 24
#define DRL_MAX_BODY 12
#define DRL_MAX_ACT 16
#define DRL_MAX_SPHERE 16
#define DRL_MAX_BOX 8
#define DRL_MAX_SITE 16
#define DRL_MAX_OBS 64
#define DRL_MAX_PHASE_JOINTS 4
#define DRL_MAX_EE 4

typedef enum {
  DRL_OK = 0,
  DRL_ERR_INVALID = -1,      /* bad argument / configuration */
  DRL_ERR_CUDA = -2,         /* CUDA runtime error (message has the cudaError string) */
  DRL_ERR_STATE = -3,        /* call order violated (e.g. step before model/mocap upload) */
  DRL_ERR_UNSUPPORTED = -4
} DrlStatus;

typedef enum { DRL_INTEGRATOR_RK4 = 0, DRL_INTEGRATOR_EULER = 1 } DrlIntegrator;
typedef enum { DRL_CURSOR_STEPWISE = 0, DRL_CURSOR_WRAP = 1 } DrlCursorMode;
typedef enum { DRL_PHASE_FROM_CURSOR = 0, DRL_PHASE_FROM_JOINTS = 1 } DrlPhaseMode;

/* Compiled walker: what MuJoCo's model compiler would hold for the reference's MJCF files
 * (drloco/mujoco/xml/walker3d_flat_feet.xml, walker_165cm_65kg.xml).  Bodies exclude the world; parent -1 = world.
 * All joints are 1-DoF (nq == nv); joint axes are +-coordinate axes of the body frame. */
typedef struct {
  int32_t nv, nb, nu, n_sphere, n_box, n_site;
  double timestep;               /* <option timestep>, xml:11 */
  double gravity_z;              /* -9.81 */
  double solref[2];              /* MuJoCo default 0.02 1 */
  double solimp[5];              /* MuJoCo default 0.9 0.95 0.001 0.5 2 */
  int32_t body_parent[DRL_MAX_BODY];
  double body_pos[DRL_MAX_BODY][3];
  double body_mass[DRL_MAX_BODY];
  double body_ipos[DRL_MAX_BODY][3];
  double body_inertia[DRL_MAX_BODY][3];
  double body_invweight0[DRL_MAX_BODY][2];
  int32_t dof_body[DRL_MAX_DOF];
  int32_t dof_type[DRL_MAX_DOF];      /* 0 slide, 1 hinge */
  int32_t dof_axis_idx[DRL_MAX_DOF];  /* 0,1,2 */
  double dof_axis_sign[DRL_MAX_DOF];  /* +1 / -1 */
  double dof_ref[DRL_MAX_DOF];        /* qpos0 */
  double dof_damping[DRL_MAX_DOF];
  double dof_armature[DRL_MAX_DOF];
  int32_t dof_limited[DRL_MAX_DOF];
  double dof_range[DRL_MAX_DOF][2];
  double dof_invweight0[DRL_MAX_DOF];
  int32_t act_dof[DRL_MAX_ACT];
  double act_gear[DRL_MAX_ACT];
  double act_ctrlrange[DRL_MAX_ACT][2];
  double act_forcerange[DRL_MAX_ACT][2];
  int32_t sphere_body[DRL_MAX_SPHERE];
  double sphere_pos[DRL_MAX_SPHERE][3];
  double sphere_radius[DRL_MAX_SPHERE];
  double sphere_mu[DRL_MAX_SPHERE];
  int32_t box_body[DRL_MAX_BOX];
  double box_center[DRL_MAX_BOX][3];
  double box_corner[DRL_MAX_BOX][8][3];
  double box_mu[DRL_MAX_BOX];
  int32_t site_body[DRL_MAX_SITE];
  double site_pos[DRL_MAX_SITE][3];
  /* end-effector points of the optional DeepMimic end-effector reward (DrlConfig.ee_weight): the centre of every box
   * geom on a leaf body that does not hang directly from the root (both walkers: the two foot boxes), in the frame of
   * its body.  n_ee may be 0 when the term stays off. */
  int32_t n_ee;
  int32_t ee_body[DRL_MAX_EE];
  double ee_pos[DRL_MAX_EE][3];
} DrlWalkerModel;

/* Environment configuration: the fields of drloco/config/config.py + hypers.py that the step path reads. */
typedef struct {
  int32_t num_envs;              /* environments resident on this device */
  int32_t device;                /* CUDA device ordinal */
  int32_t frame_skip;            /* sim_freq / CTRL_FREQ, mimic_env.py:194-207 */
  int32_t integrator;            /* DrlIntegrator; the reference XML selects RK4 */
  int32_t ep_dur_max;            /* hypers.py:58 */
  int32_t mirror_policy;         /* hypers.MOD_MIRR_POLICY active, hypers.py:20-29 */
  int32_t phase_mode;            /* DrlPhaseMode, mimic_env.py:416-419 */
  int32_t n_phase_joints;
  int32_t phase_joints[DRL_MAX_PHASE_JOINTS];   /* mimic_walker_165cm_65kg.py:40-43 */
  int32_t eval_n_times;          /* config.py:23, deterministic-init cycle length */
  double ctrl_freq;              /* config.py:20-21 */
  double rew_weights[4];         /* pos, vel, com, energy(unused) hypers.py:48 */
  double rew_scale;              /* hypers.py:51 */
  double alive_bonus;            /* hypers.py:55 */
  double fall_z;                 /* 0.5, mimic_env.py:120 */
  uint64_t seed;                 /* RSI stream seed (counter-based generator, see DESIGN.md) */
  int64_t env_id_offset;         /* global index of local env 0 (multi-GPU sharding) */
  /* mirror tables (mimic_env.py:440-489); identity when mirror_policy == 0 */
  int32_t obs_dim, act_dim;
  int32_t mirror_obs_idx[DRL_MAX_OBS];
  float mirror_obs_sign[DRL_MAX_OBS];
  int32_t mirror_act_idx[DRL_MAX_ACT];
  float mirror_act_sign[DRL_MAX_ACT];
  int32_t lanes_per_env;         /* lanes per environment; fixed by the model: 16 for nv <= 16 (walker3d), 32 otherwise.
                                  * 0 = that value; anything else must equal it (drl_upload_model rejects a mismatch) */
  int32_t early_termination;     /* MimicEnv.do_terminate_early (mimic_env.py:652-702).  The reference defines the check
                                  * but never lets it end an episode (mimic_env.py:120-123): 0 = same here, the three
                                  * reasons are only counted (DRL_STAT_ET_*); 1 = a firing check also sets done (the
                                  * terminal reward is then -0.0 like a fall). */
  int32_t monitor_median_torque; /* 1 = keep every env's per-episode history of the mean |actuator torque| (4 * ep_dur_max
                                  * bytes per env) so that Monitor.median_abs_torque_smoothed (monitor_wrapper.py:131) can
                                  * be served (drl_get_median_torque); 0 = skip it */
  /* DeepMimic end-effector term, an extension the reference does not have: with S = sum over the model's end-effector
   * points of |p_sim - p_ref|^2 (positions relative to the root-body origin, world axes; p_ref from the reference qpos
   * at the cursor), ee_rew = exp(-ee_scale * S) and the reward becomes
   * (w_pos*pos + w_vel*vel + w_com*com + ee_weight*ee_rew) * rew_scale + alive_bonus.  ee_weight = 0 switches the term
   * off (the reference's reward, no per-env buffers); ee_weight > 0 needs n_ee > 0 and ee_scale > 0 (DeepMimic: 40). */
  double ee_weight, ee_scale;
} DrlConfig;

typedef struct DrlEnv DrlEnv;    /* opaque: persistent per-env state, mocap tables, RNG counters */

/* library */
int drl_version(void);                       /* == DRL_ABI_VERSION */
const char* drl_last_error(void);

/* lifetime — replaces MimicEnv.__init__ / MujocoEnv.__init__ (mimic_env.py:19-57) for N environments at once */
int drl_create(const DrlConfig* cfg, DrlEnv** out);
int drl_destroy(DrlEnv* env);

/* replaces MuJoCo's load_model_from_path on the walker XML (mimic_env.py:52) */
int drl_upload_model(DrlEnv* env, const DrlWalkerModel* model);

/* replaces BaseReferenceTrajectories._load_ref_trajecs (base_ref_trajecs.py:28, straight_walk_trajecs.py:304-320).
 * ref: host float64 [n_samples][2*nv] (qpos rows then qvel rows in model order); step tables host arrays of n_steps.
 * des_vel_prefix: host float64 [n_samples+1][2] or NULL (loco3d desired velocity, loco3d_trajecs.py:58-68). */
int drl_upload_mocap(DrlEnv* env, int32_t cursor_mode, int32_t increment, const double* ref, int32_t n_samples,
                     const int32_t* step_off, const int32_t* step_len, const uint8_t* left_step,
                     const double* step_vel, const double* step_last_comx, int32_t n_steps, int32_t com_z_col,
                     const double* des_vel_prefix, int32_t des_vel_window);

/* VecEnv.reset (SB3) = MujocoEnv.reset + MimicEnv.reset_model (mimic_env.py:526-572) for every env whose mask byte is
 * non-zero (mask == NULL: all).  inj_istep/inj_pos (device int32[N], nullable) inject the RSI draw instead of the
 * library's generator (parity tests; straight_walk_trajecs.py:460-474).  obs: device float [N][obs_dim]. */
int drl_reset(DrlEnv* env, const uint8_t* mask, const int32_t* inj_istep, const int32_t* inj_pos, float* obs,
              void* stream);

/* VecEnv.step_async + step_wait = MimicEnv.step (mimic_env.py:60-126) + Monitor.step statistics
 * (monitor_wrapper.py:88-166) + the auto-reset of DummyVecEnv/SubprocVecEnv.  All pointers device.
 *   actions  float [N][act_dim]   policy output, clipped to [-1,1] inside (mimic_env.py:170-192)
 *   obs      float [N][obs_dim]   observation after the step; for done envs the post-reset observation
 *   rew      float [N]            reward of the step
 *   done     uint8 [N]
 *   terminal_obs float [N][obs_dim] nullable; rows of done envs receive the pre-reset observation
 * inj_istep/inj_pos as in drl_reset, used for the auto-resets of this step. */
int drl_step(DrlEnv* env, const float* actions, float* obs, float* rew, uint8_t* done, float* terminal_obs,
             const int32_t* inj_istep, const int32_t* inj_pos, void* stream);

/* state access for parity injection — replaces MujocoEnv.set_state / sim.data.qpos, qvel (mimic_env.py:211-212,539) and
 * refs._i_step/_pos.  qpos/qvel device float [N][nv]; cursor device int32 [N][4] = (i_step, pos, count_same_vel, ep_dur).
 * Any pointer may be NULL to skip it. */
int drl_get_state(DrlEnv* env, float* qpos, float* qvel, int32_t* cursor, void* stream);
int drl_set_state(DrlEnv* env, const float* qpos, const float* qvel, const int32_t* cursor, void* stream);

/* per-env extras read through VecEnv.get_attr / env_method in the reference:
 *   extras device float [N][DRL_EXTRA_COUNT] see DrlExtra. */
typedef enum {
  DRL_EXTRA_POS_REW = 0, DRL_EXTRA_VEL_REW = 1, DRL_EXTRA_COM_REW = 2,   /* mimic_env.py:645 */
  DRL_EXTRA_WALKED_DISTANCE = 3,                                         /* mimic_env.py:295 */
  DRL_EXTRA_MEAN_ABS_TORQUE = 4,                                         /* mimic_env.py:251-253 */
  DRL_EXTRA_DES_VEL = 5, DRL_EXTRA_PHASE = 6, DRL_EXTRA_Z_OFFSET = 7,
  /* Monitor attributes, per env (monitor_wrapper.py:104-133), exponentially smoothed at every episode end */
  DRL_EXTRA_EP_LEN_SMOOTHED = 8, DRL_EXTRA_EP_RET_SMOOTHED = 9, DRL_EXTRA_MEAN_REWARD_SMOOTHED = 10,
  DRL_EXTRA_MEAN_EP_POS_REW_SMOOTHED = 11, DRL_EXTRA_MEAN_EP_VEL_REW_SMOOTHED = 12,
  DRL_EXTRA_MEAN_EP_COM_REW_SMOOTHED = 13, DRL_EXTRA_MOVED_DISTANCE = 14, DRL_EXTRA_MEAN_ABS_EP_TORQUE_SMOOTHED = 15,
  DRL_EXTRA_COUNT = 16
} DrlExtra;
int drl_get_extras(DrlEnv* env, float* extras, void* stream);

/* Monitor statistics (monitor_wrapper.py:45-166) reduced over the local envs into one packed host-visible vector:
 * device double [DRL_STATS_COUNT], sums and counts only so that ranks can all-reduce(sum) it (SURVEY.md §8e). */
typedef enum {
  DRL_STAT_EPISODES = 0,         /* episodes finished since the last drl_reset_stats */
  DRL_STAT_EP_LEN_SUM = 1, DRL_STAT_EP_RET_SUM = 2, DRL_STAT_EP_MEAN_REW_SUM = 3,
  DRL_STAT_POS_REW_SUM = 4, DRL_STAT_VEL_REW_SUM = 5, DRL_STAT_COM_REW_SUM = 6, DRL_STAT_REW_STEPS = 7,
  DRL_STAT_MOVED_DISTANCE_SUM = 8, DRL_STAT_ABS_TORQUE_SUM = 9,
  DRL_STAT_ENV_STEPS = 10, DRL_STAT_BLOWUPS = 11, DRL_STAT_FALLS = 12, DRL_STAT_TIMEOUTS = 13,
  DRL_STAT_SOLVER_ITERS = 14, DRL_STAT_DYN_EVALS = 15,
  DRL_STAT_SOLVER_CAPPED = 16,   /* evaluations whose active-set iteration stopped at the cap instead of converging */
  /* env-steps on which do_terminate_early's reasons held: COM-Z < 0.75 / trunk angle out of range / |COM-Y| > 0.2 */
  DRL_STAT_ET_COM_LOW = 17, DRL_STAT_ET_TRUNK = 18, DRL_STAT_ET_DRUNK = 19,
  DRL_STATS_COUNT = 20
} DrlStat;
int drl_get_stats(DrlEnv* env, double* stats, void* stream);
int drl_reset_stats(DrlEnv* env, void* stream);

/* per-episode records for the ep_lens histogram (callback.py:227-230): a device ring of the most recent episodes.
 * ep_len device int32 [capacity], ep_ret device float [capacity]; returns the number of valid entries in *count (host). */
int drl_get_episode_ring(DrlEnv* env, int32_t* ep_len, float* ep_ret, int32_t capacity, int64_t* total_episodes,
                         void* stream);

/* the same ring slots as drl_get_episode_ring for Monitor's per-episode position records (monitor_wrapper.py:91-93,
 * 104-107,123-124): rsi_pos = refs._pos after the first step of the episode (`rsi_positions`), et_pos = refs._pos when
 * the episode ended (`et_positions`; for a simulator blow-up the cursor before the internal reset), difficult = 1 when
 * ep_len < 0.75 * ep_len_smoothed (the episode's rsi_pos then also belongs to `difficult_rsi_phases`).
 * device int32 / int32 / uint8 [capacity], each nullable. */
int drl_get_episode_positions(DrlEnv* env, int32_t* rsi_pos, int32_t* et_pos, uint8_t* difficult, int32_t capacity,
                              void* stream);

/* Monitor.rsi_positions also lists the episodes still running (the entry is appended on an episode's first step,
 * monitor_wrapper.py:91-93): rsi_pos device int32 [N] = refs._pos after the first step of env i's current episode, or
 * -1 while that episode has not stepped yet. */
int drl_get_running_rsi_positions(DrlEnv* env, int32_t* rsi_pos, void* stream);

/* Monitor.median_abs_torque_smoothed (monitor_wrapper.py:131) of every env: the median over the finished episode of
 * the per-step mean |actuator torque|, exponentially smoothed (0.75) at every episode end.  out: device float [N].
 * DRL_ERR_STATE when the env was created with monitor_median_torque == 0. */
int drl_get_median_torque(DrlEnv* env, float* out, void* stream);

/* the end-effector term (DrlConfig.ee_weight > 0) of every env: last = ee_rew of the latest step (not updated on a
 * terminal step, 1 after a reset, as the pose / velocity / COM terms), smoothed = Monitor-style mean of ee_rew over all
 * steps of the env so far, exponentially smoothed (0.9) at every episode end.  last, smoothed: device float [N], each
 * nullable.  DRL_ERR_STATE when the env was created with ee_weight == 0. */
int drl_get_ee_reward(DrlEnv* env, float* last, float* smoothed, void* stream);

/* MimicEnv.activate_evaluation (mimic_env.py:245): deterministic init states (straight_walk_trajecs.py:237-265) */
int drl_set_eval_mode(DrlEnv* env, int32_t on);

/* StraightWalkingTrajectories.n_deterministic_inits (straight_walk_trajecs.py:126,248-253) of every env: the index of
 * the mocap step the NEXT deterministic init starts from.  counts: HOST int32 [num_envs].  A batched evaluation sets
 * counts[i] = i so that env i plays the i-th of the reference's EVAL_N_TIMES consecutive evaluation episodes
 * (callback.py:296-297).  Synchronises the device. */
int drl_set_det_init_counters(DrlEnv* env, const int32_t* counts);

/* VecEnv.seed - the reference seeds every worker env with seed + rank*100 when it builds them (utils.py:113).  Re-keys the
 * counter-based RSI generator: env i draws splitmix64(seed, env_id_offset + i, reset #).  Synchronises the device. */
int drl_set_seed(DrlEnv* env, uint64_t seed);

/* MimicEnv.activate_speed_control (mimic_env.py:298-327): from now on the desired-velocity observation of every env is
 * speeds[ep_dur % n] (mimic_env.py:406-408) and resets use the deterministic init state (mimic_env.py:536-537).
 * `speeds` is a HOST array with one desired speed per control step (the host builds it with the reference's
 * linspace regions); n = 0 switches speed control off.  Synchronises the device (not for the stepping loop). */
int drl_set_speed_profile(DrlEnv* env, const float* speeds, int32_t n);

/* MimicEnv.playback_ref_trajectories (mimic_env.py:265-282): while on, drl_step skips the physics and, after
 * refs.next(), sets qpos / qvel from the mocap (set_joint_kinematics_in_sim, mimic_env.py:284-293) before the
 * observation, reward and termination logic run.  A kinematic check of tables, cursor and ground shift: the imitation
 * reward of every such step is its maximum.  Rendering is not part of this library. */
int drl_set_playback(DrlEnv* env, int32_t on);

/* test / tuning hooks: frame_skip_override >= 0 replaces cfg.frame_skip (0 = environment logic only, used to test the
 * reward / cursor / reset path on injected states); block_threads > 0 sets the CTA size; enable_dump keeps, per env, the
 * intermediate results of the last dynamics evaluation (mass matrix, bias force, qacc) for drl_debug_read (host buffer). */
int drl_debug_set(DrlEnv* env, int32_t frame_skip_override, int32_t block_threads, int32_t enable_dump);
int drl_debug_read(DrlEnv* env, float* host_out, int32_t n_floats);

/* VecNormalize on the device — replaces SB3 VecNormalize.step_wait / reset around the env (utils.py:130-132).
 * drl_vecnorm_moments: the batch moments of obs [n][d] (device), for the statistics update of observations the step
 *   kernel did not produce (the reset observations).  ret = ret*gamma + rew (in place; skipped when rew == NULL) and
 *   packed[2d+3] = { sum_obs[d], sumsq_obs[d], n, sum_ret, sumsq_ret } in float64 (device; zeroed, then filled) — the
 *   all-reduce(sum) payload that drl_vecnorm_step merges into the running statistics. */
int drl_vecnorm_moments(const float* obs, int32_t n, int32_t d, const float* rew, float* ret, float gamma,
                        double* packed, void* stream);

/* Fused VecNormalize path (what B200VecNormalize uses): ONE kernel per step after drl_step.
 *
 * drl_attach_vecnorm: from now on drl_step itself maintains ret = ret*gamma + rew (device float [N], in/out) and leaves
 *   the batch moments of the step in packed (device double [2*obs_dim+3], layout as drl_vecnorm_moments) - computed in
 *   the step kernel's epilogue from the observations it returns, block sums then a fixed-order grid sum, no atomics:
 *   the moments (and the Monitor statistics, drl_get_stats) are bit-reproducible.  Two NULLs detach.
 * DrlComm: the statistics exchange between the ranks of one node (one process per GPU) without a host-issued
 *   collective - replaces the all-reduce of SB3-style data-parallel VecNormalize statistics (SURVEY.md section 8e).
 *   Every rank creates one (current CUDA device), publishes its 64-byte CUDA IPC handle (drl_comm_export), gathers the
 *   handles of all ranks by any means (torch.distributed.all_gather) and maps its peers' mailboxes (drl_comm_connect,
 *   handles = world x 64 bytes in rank order).  world == 1 needs no export / connect.
 * drl_vecnorm_step: exchange (peer stores into the mailboxes over NVLink + flags, summed in rank order: identical bits
 *   on every rank) + Chan merge into the running statistics rms = { mean[d], var[d], count, ret_mean, ret_var,
 *   ret_count } in float64 (RunningMeanStd.update_from_moments; rms_in -> rms_out, must not alias) + normalisation
 *   obs_out = clip((obs_in-mean)/sqrt(var+eps), +-clip_obs), rew_out = clip(rew_in/sqrt(ret_var+eps), +-clip_rew) +
 *   ret[done] = 0.  flags: bit0 update the observation statistics, bit1 norm_obs, bit2 norm_reward, bit3 update the
 *   return statistics.  packed == NULL or no update bit: normalise only.  done_out (nullable): a copy of `done`
 *   next to the normalised outputs, so that one device-to-host copy can fetch a whole step.  sync_every = K >= 1: a "cycle" call - the
 *   moments are accumulated locally and exchanged / merged on every K-th cycle call (K = 1: every call, SB3's
 *   semantics; K > 1 is an opt-in amortisation); sync_every = 0: an "immediate" call - exchange and merge `packed` now,
 *   leaving the cycle alone (VecNormalize.reset).  All ranks must make the same sequence of calls.  Asynchronous on `stream`; CUDA-graph capturable (the step counter lives on
 *   the device). */
typedef struct DrlComm DrlComm;
int drl_attach_vecnorm(DrlEnv* env, float* ret, float gamma, double* packed);
int drl_comm_create(int32_t world, int32_t rank, int32_t obs_dim, DrlComm** out);
int drl_comm_export(DrlComm* comm, void* handle64);
int drl_comm_connect(DrlComm* comm, const void* handles);
int drl_comm_destroy(DrlComm* comm);
int drl_vecnorm_step(const float* obs_in, float* obs_out, const float* rew_in, float* rew_out, int32_t n, int32_t d,
                     const double* packed, const double* rms_in, double* rms_out, float* ret, const uint8_t* done,
                     uint8_t* done_out, float clip_obs, float clip_rew, float eps, int32_t flags, DrlComm* comm,
                     int32_t sync_every, void* stream);

/* rows of tobs_in whose done byte is set, normalised with rms ({mean[d], var[d], ...}): the
 * infos[i]["terminal_observation"] VecNormalize returns (SB3 VecNormalize.step_wait), compacted so that only finished
 * environments cross PCIe: out_words (4 + n*(d+1) 32-bit words) = header { count, -, -, - } + one record
 * { env index (int32), d floats } per finished environment, in arbitrary order.
 * out_words may be device memory or pinned host memory (mapped into the device's address space: the kernel then writes
 * the records across PCIe itself).  The same holds for obs_out / rew_out / done_out of drl_vecnorm_step.
 * counters: device int32 [2], zero before the first call, left zero by every call (slot counter, block ticket).
 * rms may be NULL when norm_obs == 0 (raw terminal observations). */
int drl_vecnorm_terminal_compact(const float* tobs_in, const uint8_t* done, int32_t n, int32_t d, const double* rms,
                                 float clip_obs, float eps, int32_t norm_obs, float* out_words, int32_t* counters,
                                 void* stream);

/* measured sustained FFMA rate of `device` in TFLOP/s (8 independent FMA chains per thread, all SMs): the FP32
 * roofline denominator bench.py reports next to the HBM one (SURVEY.md §8d). Synchronises the device. */
int drl_fp32_peak_probe(int32_t device, double* tflops_out);

/* introspection for benchmarks */
int drl_launch_info(DrlEnv* env, int32_t* lanes_per_env, int32_t* block_threads, int32_t* grid_blocks,
                    int32_t* smem_bytes);

#ifdef __cplusplus
}
#endif
#endif /* DRLOCO_B200_H */
