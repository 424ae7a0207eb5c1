// dev_model.h — device-side view of the compiled walker + environment configuration (internal to libdrloco_b200).
//
// Built on the host from DrlWalkerModel / DrlConfig (include/drloco_b200.h) in drl_upload_model(), stored once in
// global memory and staged into shared memory by every thread block of the step kernel.
#pragma once
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
  int early_termination, trunk_dof0, pad_et[2];   // do_terminate_early: off/on, first of the three trunk rotation dofs
  // ---- mocap ----
  int cursor_mode, increment, n_steps, n_samples, com_z_col, des_vel_window;
  unsigned long long seed;
  long long env_id_offset;
  // ---- optional end-effector reward term (DrlConfig.ee_weight; w_ee == 0: off) ----
  int n_ee, ee_body[kMaxEE];
  float ee_pos[kMaxEE][3];           // point in the body frame
  float w_ee, ee_scale;
};

static_assert(sizeof(DevModel) % 16 == 0, "DevModel is copied in int4 chunks");

// per-env persistent state rows (see DESIGN.md "data layout in HBM")
constexpr int kMiscDist = 0, kMiscZoff = 1, kMiscWalked = 2, kMiscEpRet = 3, kMiscEpTor = 4, kMiscPrevPos = 5,
              kMiscPrevVel = 6, kMiscPrevCom = 7, kMiscEpLenSm = 8, kMiscEpRetSm = 9, kMiscMeanRewSm = 10,
              kMiscPosSm = 11, kMiscVelSm = 12, kMiscComSm = 13, kMiscMoved = 14, kMiscTorSm = 15;
constexpr int kMiscCount = 16;
constexpr int kCurIstep = 0, kCurPos = 1, kCurCount = 2, kCurEpDur = 3, kCurRsiStep = 4, kCurNDet = 5,
              kCurResets = 6, kCurFlags = 7;
constexpr int kCurCount8 = 8;
constexpr int kStatGroup = 16;        // blocks per group in the step kernel's two-level statistics sum

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
  const double* des_vel_prefix;      // [n_samples+1][2] or null (float64 prefix sums)
  // io
  const float* actions;              // [N][act_dim]
  float* obs;                        // [N][obs_dim]
  float* rew;                        // [N]
  unsigned char* done;               // [N]
  float* terminal_obs;               // [N][obs_dim] nullable
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
  double* cta_rows;                  // [grid + groups][2*obs_dim + 2 + DRL_STATS_COUNT]
  unsigned* cta_ticket;              // [1 + groups]
  // fused VecNormalize (drl_attach_vecnorm; null = not attached)
  float* vn_ret;                     // [N] discounted-return accumulator, in/out
  float vn_gamma;
  double* packed;                    // [2*obs_dim + 3] batch moments of the step, out
  // end-effector term, allocated only when it is on (DevModel::w_ee != 0), null otherwise
  float* ee_f;                       // [N][2] ee_rew of the last step (1 after a reset), Monitor-smoothed mean
  double* ee_d;                      // [N] lifetime sum of ee_rew (Monitor never clears its per-step lists)
};

}  // namespace drl
