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
#define DRL_MAX_OBS 64             /* DrlConfig.obs_dim and its mirror tables */
#define DRL_MAX_PHASE_JOINTS 4
#define DRL_MAX_EE 4
#define DRL_MAX_REF_OBS 3          /* reference-pose frames of drl_set_ref_obs */
#define DRL_MAX_OBS_TOTAL 101      /* widest observation row: obs_dim + the frames (walker_165cm_65kg: 47 + 3 * 18) */

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
 * des_vel_prefix: host float64 [n_samples+n_steps][2] or NULL (loco3d desired velocity, loco3d_trajecs.py:58-68): per
 * step, a zero row and the running sums over its samples (one step: [n_samples+1][2]).  A wrap-mode mocap of more than
 * one step is a library of one-step clips and needs drl_set_mocap_clips before it can be stepped.  Every upload makes
 * the mocap one clip spanning the table. */
int drl_upload_mocap(DrlEnv* env, int32_t cursor_mode, int32_t increment, const double* ref, int32_t n_samples,
                     const int32_t* step_off, const int32_t* step_len, const uint8_t* left_step,
                     const double* step_vel, const double* step_last_comx, int32_t n_steps, int32_t com_z_col,
                     const double* des_vel_prefix, int32_t des_vel_window);

/* VecEnv.reset (SB3) = MujocoEnv.reset + MimicEnv.reset_model (mimic_env.py:526-572) for every env whose mask byte is
 * non-zero (mask == NULL: all).  inj_istep/inj_pos (device int32[N], nullable) inject the RSI draw instead of the
 * library's generator (parity tests; straight_walk_trajecs.py:460-474).  obs: device float [N][obs_dim] (with
 * reference-pose frames, drl_set_ref_obs: [N][obs_dim + n * (nv - 1)], as every obs row below). */
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

/* Actuation of the walker's motors.  The reference drives every joint with a motor whose force is the (rescaled)
 * action, held for the whole control step (mimic_env.py:170-192): DRL_ACTUATION_TORQUE, the state after
 * drl_upload_model.  DRL_ACTUATION_PD turns every motor into a MuJoCo position servo, <position kp kv> (the
 * "PD/torque actuation" of the step kernel's scope, BASELINE.json north_star):
 *   - the clipped action a_u in [-1, 1] of actuator u maps to the target ctrl_u = mid_u + a_u * half_u over the range
 *     [lo, hi] of the joint it drives (mid = (lo + hi) / 2, half = (hi - lo) / 2, rounded to float32), then the policy
 *     mirror applies as in torque mode; ctrl is held for the control step and clamped to the joint range;
 *   - at every dynamics evaluation (all four RK4 stages of every substep; the one Euler evaluation, where kv is explicit
 *     and only joint damping is implicit) the actuator force is f_u = clamp(kp_u (ctrl_u - gear_u q) - kv_u gear_u v,
 *     forcerange_u) at that evaluation's q, v, and the generalised force gear_u f_u;
 *   - the Monitor torque (DRL_EXTRA_MEAN_ABS_TORQUE, DRL_STAT_ABS_TORQUE_SUM, the median history) is mean_u |f_u| at
 *     the state the step starts from.
 * kp, kv: HOST float64 [nu] in actuator order, kp finite and > 0, kv finite and >= 0; ignored (may be NULL) for
 * DRL_ACTUATION_TORQUE.  Every actuated joint must be limited.  DRL_ERR_STATE before drl_upload_model,
 * DRL_ERR_INVALID for an unknown mode, bad gains or an unlimited actuated joint.  May be called again to switch modes.
 * Synchronises the device (not for the stepping loop; a captured CUDA graph keeps the instance it captured). */
typedef enum { DRL_ACTUATION_TORQUE = 0, DRL_ACTUATION_PD = 1 } DrlActuation;
int drl_set_actuation(DrlEnv* env, int32_t mode, const double* kp, const double* kv);

/* DeepMimic contact termination (not in the reference): the episode also ends when a body of body_mask (bit b = body b)
 * touches the floor, i.e. when a contact candidate of one of its geoms (a box corner, or a capsule end sphere at
 * centre_z - radius) is at or below z = 0.  Checked once per control step, at the state the step ends in (not at the
 * intermediate RK4 stages), and skipped on a simulator blow-up and in playback.  Such a step is terminal like a fall:
 * reward -0 (+0 when it is also the timeout), counted in DRL_STAT_FALLS (DRL_STAT_TIMEOUTS with the timeout).
 * body_mask = 0 turns it off, the state after drl_upload_model.  DRL_ERR_STATE before drl_upload_model,
 * DRL_ERR_INVALID for a bit >= nb or a body that carries a foot-corner site (the reset puts the lowest of those on the
 * floor).  The first call with a non-zero mask allocates and zeroes the per-env counter of drl_get_contact_terminations.
 * Synchronises the device (not for the stepping loop; a captured CUDA graph keeps the arguments it captured). */
int drl_set_contact_termination(DrlEnv* env, uint32_t body_mask);

/* lifetime count per env of the episodes that ended on a step where the contact check held (blow-ups excluded; also
 * the ones that fell or timed out on the same step).  out: device int32 [N].  DRL_ERR_STATE when contact termination
 * was never enabled on this env. */
int drl_get_contact_terminations(DrlEnv* env, int32_t* out, void* stream);

/* Failure-weighted reference state initialisation (not in the reference, whose RSI draw is uniform: a uniform mocap
 * step, then a uniform sample in it, straight:460-474 / base:79-85).  The mocap is cut into bins of at most bin_samples
 * consecutive samples inside each step (bins never straddle steps), in step order.  Per bin b the env keeps two
 * decayed float64 counts: s_b, episodes that started in b, and f_b, those of them that were "difficult" by Monitor's
 * rule (ep_len < 0.75 * ep_len_smoothed after the smoothing update, monitor_wrapper.py:123-124).  After every
 * drl_step a one-block kernel on the same stream applies x <- rho x + dx (rho = 2^(-1/halflife_steps)) and builds the
 * weighted distribution q_b = u_b rate_b / sum(u rate), rate_b = (f_b + 1) / (s_b + 2), u_b = the probability of b
 * under the uniform draw; an empty table gives q = u.  A random RSI draw tosses its own counter-based coin: with
 * probability lambda it picks a bin from q and a sample uniform in the bin, otherwise it is the uniform draw, bit for
 * bit.  Resets in step k sample the table as it stood after step k - 1; the update is deterministic (integer atomics
 * for the increments, a fixed-order float64 pass for the rest).  Counted: episodes whose start was a random RSI draw
 * (either branch).  Not counted: deterministic inits (evaluation mode, speed profile), injected draws, states set
 * with drl_set_state, playback.  Each env (each rank of a sharded run) keeps its own table; nothing is exchanged.
 * lambda = 0 turns it off (drl_step then enqueues one kernel, as without it); the tables are kept.  DRL_ERR_INVALID
 * for lambda outside [0, 1], halflife_steps <= 0 or bin_samples <= 0; DRL_ERR_STATE before drl_upload_mocap.  The
 * first enable for a mocap upload and bin width allocates a zeroed table and marks every running episode uncounted.
 * While it is on, drl_upload_mocap returns DRL_ERR_STATE (the bins would go stale).  Synchronises the device (not for
 * the stepping loop; a captured CUDA graph keeps the kernels and arguments it captured). */
int drl_set_adaptive_rsi(DrlEnv* env, float lambda, int32_t halflife_steps, int32_t bin_samples);

/* The table: started, difficult, prob (the full mixture (1 - lambda) u_b + lambda q_b): device float64 [n_bins];
 * env_bin: device int32 [N], the start bin of every running episode (-1: not counted).  Each pointer is nullable.
 * n_bins follows from the mocap step lengths and bin_samples as described above.  DRL_ERR_STATE if the option was
 * never enabled on this env. */
int drl_get_adaptive_rsi(DrlEnv* env, double* started, double* difficult, double* prob, int32_t* env_bin,
                         void* stream);

/* Overwrite the counts (HOST float64 [n_bins] each, 0 <= difficult <= started, finite), e.g. to resume a run, and
 * rebuild the sampling tables; pending increments are dropped.  DRL_ERR_STATE if the option was never enabled,
 * DRL_ERR_INVALID for a bad count.  Synchronises the device. */
int drl_set_adaptive_rsi_counts(DrlEnv* env, const double* started, const double* difficult);

/* Mocap library (not in the reference, which imitates one recording): the uploaded table as n_clips clips of
 * consecutive mocap steps, clip k = steps [clip_first_step[k], clip_first_step[k + 1]) (HOST int32 [n_clips + 1],
 * starting at 0 and ending at n_steps).  An episode stays in the clip it started in:
 *   - stepwise mode (walker3d): the last step of clip k wraps to its first step + (left ? 0 : 1) (straight:330-333 per
 *     clip; a clip needs at least 2 steps), and the desired-velocity step i_step - count + 1 is clamped at the clip's
 *     first step;
 *   - wrap mode (loco3d): every clip is one step and i_step is the clip; the desired-velocity window stays in the clip.
 * A random RSI draw picks clip k with probability clip_weight[k] / sum (HOST float64 [n_clips], finite, >= 0, positive
 * sum; a zero weight is never drawn) from its own counter-based hash, then the reference's draw inside the clip.
 * Evaluation mode and the speed profile use clip 0.  An injected inj_istep is the mocap step (stepwise) or the clip
 * (wrap mode with more than one clip).  The failure-weighted RSI base probability of a bin becomes
 * weight_k / steps_k * width / step_len.  With more than one clip the env keeps the per-clip episode counters of
 * drl_get_clip_stats (zeroed here).  n_clips = 1 is the single-clip behaviour.  DRL_ERR_INVALID for clips that do not
 * cover the table in order, a stepwise clip of fewer than 2 steps, a wrap-mode clip of other than 1 step or bad
 * weights; DRL_ERR_STATE before drl_upload_mocap and while failure-weighted RSI is on (its bins would go stale).
 * Synchronises the device (not for the stepping loop; a captured CUDA graph keeps the arguments it captured). */
int drl_set_mocap_clips(DrlEnv* env, int32_t n_clips, const int32_t* clip_first_step, const double* clip_weight);

/* Per-clip episode counters since drl_set_mocap_clips, by the clip of the episode's start step: out device int64
 * [n_clips][5] = episodes, sum of episode lengths, falls (every terminal step that is neither a timeout nor a
 * blow-up, so early and contact terminations too), timeouts, blow-ups.  Exact integer counts, per env (per rank).
 * DRL_ERR_STATE while the mocap has a single clip. */
int drl_get_clip_stats(DrlEnv* env, int64_t* out, void* stream);

/* MimicEnv.playback_ref_trajectories (mimic_env.py:265-282): while on, drl_step skips the physics and, after
 * refs.next(), sets qpos / qvel from the mocap (set_joint_kinematics_in_sim, mimic_env.py:284-293) before the
 * observation, reward and termination logic run.  A kinematic check of tables, cursor and ground shift: the imitation
 * reward of every such step is its maximum.  Rendering is not part of this library. */
int drl_set_playback(DrlEnv* env, int32_t on);

/* Reference-pose observations (not in the reference, whose policy sees the phase, the desired velocity and its own
 * state only): n frames are appended to every observation row, frame f = the reference qpos[1:] (nv - 1 floats, the
 * entries of the observation's own qpos block) offsets[f] control steps ahead.  Exactly: for the cursor c the
 * observation was built at, apply StraightWalkingTrajectories.next / BaseReferenceTrajectories.next (the library's
 * per-clip wrap included) offsets[f] times to a copy of c and read the reference qpos there with the episode's COM-Z
 * shift: the target the pose reward compares against that many steps later if the episode runs on.  A mirrored
 * observation (mirror_policy, a left step) mirrors every frame with its own decision, through the qpos-block part of
 * mirror_obs_idx / mirror_obs_sign, which must map the block onto itself.  Frames are in every row the library writes:
 * obs, terminal_obs (at the pre-reset cursor), the auto-reset and drl_reset observations, in playback, evaluation mode
 * and with a speed profile.  From the call on, drl_reset / drl_step write rows of obs_dim + n * (nv - 1) floats and the
 * fused VecNormalize moments (drl_attach_vecnorm) cover the whole row: packed has 2 * that + 3 doubles.  n = 0 is off,
 * the state after drl_upload_model.  offsets: HOST int32 [n], strictly increasing, each in [1, 256]; n <=
 * DRL_MAX_REF_OBS.  DRL_ERR_STATE before drl_upload_model, after the first drl_reset or drl_step, and while a
 * VecNormalize is attached; DRL_ERR_INVALID for bad offsets or a mirror map that leaves the qpos block.  Synchronises
 * the device; a failed call changes nothing. */
int drl_set_ref_obs(DrlEnv* env, int32_t n, const int32_t* offsets);

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
 *   the batch moments of the step in packed (device double [2*D+3], D the row width, layout as drl_vecnorm_moments) - computed in
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
