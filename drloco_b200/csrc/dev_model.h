// dev_model.h — device-side view of the compiled walker + environment configuration (internal to libdrloco_b200).
//
// Built on the host from DrlWalkerModel / DrlConfig (include/drloco_b200.h) in drl_upload_model(), stored once in
// global memory and staged into shared memory by every thread block of the step kernel.
#pragma once
#include <stddef.h>
#include <stdint.h>

namespace drl {

constexpr int kMaxBody = 8;      // bodies handled in-kernel (walker3d: 7, walker_165cm_65kg: 8)
constexpr int kMaxDof = 32;
constexpr int kMaxAct = 16;
constexpr int kMaxCand = 64;     // contact candidates: 8 corners per box, 1 per capsule end
constexpr int kMaxSite = 16;
constexpr int kMaxObs = 64;
constexpr int kMaxEE = 4;        // end-effector points (DRL_MAX_EE)

// alignas(16): the step kernel stages this struct into shared memory in 16-byte chunks (sizeof must be a multiple of 16)
struct alignas(16) DevModel {
  // sizes
  int nv, nb, nu, ncand, nbox_cand, nsite, nslide, pad_sz_;
  float timestep, gravity_z;
  float Kc, Bc;                      // 1/(dmax^2 tc^2 dr^2), 2/(dmax tc)  (solref)
  float imp_d0, imp_dmax, imp_width, imp_mid, imp_power;
  float imp_inv_width, imp_inv_mid, imp_inv_1mmid;   // reciprocals used by the power-2 impedance curve
  float root_z0;                     // body_pos[root].z
  // bodies
  // (the tree topology itself is compiled into the kernels: Topo<NV> in fd_tree.cuh)
  int body_parent[kMaxBody];
  float body_pos[kMaxBody][3], body_ipos[kMaxBody][3], body_inertia[kMaxBody][3];
  float body_mass[kMaxBody], body_invw_tran[kMaxBody];
  // dofs
  int dof_body[kMaxDof], dof_type[kMaxDof], dof_limited[kMaxDof];
  int dof_code[kMaxDof];             // axis index | (axis sign < 0) << 2
  float dof_sign[kMaxDof], dof_ref[kMaxDof], dof_damping[kMaxDof], dof_armature[kMaxDof];
  float dof_lo[kMaxDof], dof_hi[kMaxDof], dof_invw[kMaxDof], dof_slide_z[kMaxDof];
  // actuators
  int act_dof[kMaxAct];
  float act_gear[kMaxAct], act_clo[kMaxAct], act_chi[kMaxAct], act_flo[kMaxAct], act_fhi[kMaxAct];
  // contact candidates: box corners first (8 consecutive slots per box), then capsule end spheres
  int cand_body[kMaxCand];
  float cand_pos[kMaxCand][3];       // box: corner relative to box centre (body frame); sphere: centre (body frame)
  float cand_aux[kMaxCand][3];       // box: box centre (body frame); sphere: radius, -, -
  float cand_mu[kMaxCand];
  // sites
  int site_body[kMaxSite];
  float site_pos[kMaxSite][3];
  // ---- environment configuration (DrlConfig) ----
  int frame_skip, integrator, ep_dur_max, mirror_policy, phase_mode, n_phase_joints, eval_n_times;
  int phase_joints[4];
  int obs_dim, act_dim, n_phase_obs, n_des_vel;
  float ctrl_freq_inv, w_pos, w_vel, w_com, rew_scale, alive_bonus, fall_z;
  int mirror_obs_idx[kMaxObs], mirror_act_idx[kMaxAct];
  float mirror_obs_sign[kMaxObs], mirror_act_sign[kMaxAct];
  unsigned box_body_mask;            // bodies that carry a box geom (their contact accumulators are segment-written)
  unsigned com_mask;                 // dofs excluded from the pose / velocity reward (COM indices 0,1,2)
  int com_z_dof;
  int early_termination, trunk_dof0;   // do_terminate_early: off/on, first of the three trunk rotation dofs
  unsigned et_contact_mask;          // DeepMimic contact termination (drl_set_contact_termination): bodies that end
                                     // the episode when they touch the floor; 0 = off
  int obs_row;                       // floats per obs / terminal_obs row: obs_dim, plus the reference-pose frames of
                                     // drl_set_ref_obs
  // ---- mocap ----
  int cursor_mode, increment, n_steps, n_samples, com_z_col, des_vel_window;
  unsigned long long seed;
  long long env_id_offset;
  // ---- optional end-effector reward term (DrlConfig.ee_weight; w_ee == 0: off) ----
  int n_ee, ee_body[kMaxEE];
  float ee_pos[kMaxEE][3];           // point in the body frame
  float w_ee, ee_scale;
  // ---- PD position servos (drl_set_actuation; read by the PD instances of the step kernel only, which alone stage
  // this tail of the block into shared memory: kModelBytesTorque) ----
  // per dof, zero on dofs without an actuator: f = clamp(kp (ctrl - gear q) - kv gear v, flo, fhi), tau = gear f
  alignas(16) float pd_kp[kMaxDof];
  float pd_kv[kMaxDof], pd_gear[kMaxDof], pd_flo[kMaxDof], pd_fhi[kMaxDof];
  // per actuator: action a in [-1, 1] -> target ctrl = mid + a * half over the range of the joint it drives
  float pd_mid[kMaxAct], pd_half[kMaxAct];
};

static_assert(sizeof(DevModel) % 16 == 0, "DevModel is copied in int4 chunks");
// bytes of DevModel a torque-actuated step kernel stages and reserves (everything before the PD tables)
constexpr size_t kModelBytesTorque = offsetof(DevModel, pd_kp);
static_assert(kModelBytesTorque % 16 == 0, "the PD tables start on an int4 boundary");

// per-env persistent state rows (see DESIGN.md "data layout in HBM")
constexpr int kMiscDist = 0, kMiscZoff = 1, kMiscWalked = 2, kMiscEpRet = 3, kMiscEpTor = 4, kMiscPrevPos = 5,
              kMiscPrevVel = 6, kMiscPrevCom = 7, kMiscEpLenSm = 8, kMiscEpRetSm = 9, kMiscMeanRewSm = 10,
              kMiscPosSm = 11, kMiscVelSm = 12, kMiscComSm = 13, kMiscMoved = 14, kMiscTorSm = 15;
constexpr int kMiscCount = 16;
constexpr int kCurIstep = 0, kCurPos = 1, kCurCount = 2, kCurEpDur = 3, kCurRsiStep = 4, kCurNDet = 5,
              kCurResets = 6, kCurFlags = 7;
constexpr int kCurCount8 = 8;
constexpr int kStatGroup = 16;        // blocks per group in the step kernel's two-level statistics sum

// A mocap library in global memory (drl_set_mocap_clips): clips are runs of consecutive mocap steps; an episode never
// leaves the clip it started in.
struct ClipLibrary {
  int n_clips;
  const int* clip_first;             // [n_clips + 1] first mocap step of each clip, then n_steps
  const int* step_clip;              // [n_steps] clip of each mocap step
  const double* clip_cdf;            // [n_clips] cumulative distribution of the RSI clip draw
  unsigned long long* clip_stats;    // [n_clips][kClipStatCount] episode counts by start clip
};

struct StepArgs {
  const DevModel* model;
  int num_envs;
  int frame_skip;                    // runtime override (0 = logic only, used by parity tests)
  // persistent state
  float* state_f;                    // [N][4*G]  q | v | qacc_warm | misc
  int* state_i;                      // [N][8]
  int* state_as;                     // [N][G] packed active set of each lane's contact candidates / limit row
  double* state_d;                   // [N][4] lifetime sums of pos/vel/com reward + count (monitor_wrapper.py:97-99)
  // mocap tables
  const float* ref;                  // [n_samples][2*G]
  const int* step_off;
  const int* step_len;
  const unsigned char* left_step;
  const float* step_vel;
  const float* step_last_comx;
  const double* des_vel_prefix;      // [n_samples+n_steps][2] or null (float64 prefix sums, restarting at every step)
  // io
  const float* actions;              // [N][act_dim]
  float* obs;                        // [N][obs_row]
  float* rew;                        // [N]
  unsigned char* done;               // [N]
  float* terminal_obs;               // [N][obs_row] nullable
  const unsigned char* reset_mask;   // reset kernel only, nullable
  const int* inj_istep;              // nullable
  const int* inj_pos;                // nullable
  float* extras;                     // [N][16] last-step extras, nullable
  double* stats;                     // [DRL_STATS_COUNT]
  int* ring_len;                     // episode ring
  float* ring_ret;
  int* ring_rsi_pos;                 // Monitor.rsi_positions / et_positions / difficult flag of the same episode slots
  int* ring_et_pos;
  unsigned char* ring_difficult;
  unsigned long long* ring_head;
  int ring_cap;
  int eval_mode;
  const float* speed_profile;        // desired speed per control step (activate_speed_control), null when off
  int speed_profile_len;
  int playback;                      // kinematic playback: the state is set from the mocap instead of simulated
  float* debug;                      // nullable: per-env dump of one forward evaluation (tests)
  // Monitor.median_abs_torque_smoothed (monitor_wrapper.py:131): per-episode history of the mean |torque| of every step
  float* tor_hist;                   // [N][ep_dur_max], nullable (DrlConfig.monitor_median_torque)
  float* med_tor_sm;                 // [N] smoothed median, written at episode ends
  // per-step statistics without atomics: every thread block writes one row of sums, the last block of every group of
  // kStatGroup blocks adds the group's rows, the last group to finish adds the group rows
  double* cta_rows;                  // [grid + groups][2*obs_row + 2 + DRL_STATS_COUNT]
  unsigned* cta_ticket;              // [1 + groups]
  // fused VecNormalize (drl_attach_vecnorm; null = not attached)
  float* vn_ret;                     // [N] discounted-return accumulator, in/out
  float vn_gamma;
  double* packed;                    // [2*obs_row + 3] batch moments of the step, out
  // end-effector term, allocated only when it is on (DevModel::w_ee != 0), null otherwise
  float* ee_f;                       // [N][2] ee_rew of the last step (1 after a reset), Monitor-smoothed mean
  double* ee_d;                      // [N] lifetime sum of ee_rew (Monitor never clears its per-step lists)
  // contact termination (DevModel::et_contact_mask != 0), null while it is off
  int* contact_et;                   // [N] lifetime count of episodes that ended on a step with a listed body on the floor
  // failure-weighted reference state initialisation (drl_set_adaptive_rsi), null / 0 while it is off.  A random RSI
  // draw takes the weighted branch when the low 32 bits of its coin are below ars_coin (= lambda * 2^32).
  unsigned long long ars_coin;
  int ars_n_bins, ars_bin_samples;
  const double* ars_cdf;             // [n_bins] cumulative distribution of the weighted part, built by the update kernel
  const int* ars_bins;               // [n_bins][3] mocap step, first sample, width; then [n_steps] first bin of each step
  unsigned* ars_inc;                 // [2][n_bins] episodes started / difficult in each bin since the last update
  int* ars_env_bin;                  // [N] start bin of the running episode, -1 = not counted
  // mocap library (drl_set_mocap_clips), null with one clip.  Behind one pointer so that the parameter block, which
  // the kernel copies to its stack, grows by 8 bytes only.
  const ClipLibrary* clips;
  // reference-pose observations (drl_set_ref_obs), 0 while off: byte 0 = the number of frames, byte f + 1 = frame f's
  // offset in control steps, minus 1.  Each frame appends the reference qpos[1:] (nv - 1 floats) to the row.
  unsigned ref_obs;
};

// per-clip episode counters (drl_get_clip_stats)
constexpr int kClipEpisodes = 0, kClipLenSum = 1, kClipFalls = 2, kClipTimeouts = 3, kClipBlowups = 4;
constexpr int kClipStatCount = 5;

// one-block kernel that folds a step's increments into the decayed counts and rebuilds the sampling tables
struct AdaptiveRsiArgs {
  int n_bins;
  double rho;                        // decay per update (2^(-1/halflife); 1 = fold in without decay)
  double lambda;                     // mixture weight of the weighted part (for prob)
  const double* u;                   // [n_bins] probability of each bin under the reference's uniform draw
  double* counts;                    // [2][n_bins] started, difficult
  unsigned* inc;                     // [2][n_bins]
  double* cdf;                       // [n_bins]
  double* prob;                      // [n_bins] full mixture (1 - lambda) u + lambda q
};

}  // namespace drl
