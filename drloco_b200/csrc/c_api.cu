// c_api.cu — extern "C" boundary of libdrloco_b200.so (declarations and the reference interfaces they replace are in
// include/drloco_b200.h).  Host-side only: validates the model, builds the device tables, owns the opaque DrlEnv and
// enqueues the kernels of mimic_step.cu on the caller's stream.  No CPU fallback: every entry point needs a CUDA device.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "../../include/drloco_b200.h"
#include "dev_buf.h"
#include "dev_model.h"

namespace drl {
size_t step_smem_bytes(int G, int envs_per_block, bool pd);
cudaError_t launch_step(const StepArgs& a, int nv, int G, int rk4, int reset_only, int block, bool debug, bool pd,
                        cudaStream_t st);
cudaError_t launch_running_rsi(const int* state_i, int* out, int n, cudaStream_t st);
bool topology_matches(int nv, int nb, const int* body_parent, const int* dof_body, const int* dof_type);
cudaError_t launch_extras(const float* state_f, const float* last, float* out, int n, int G, cudaStream_t st);
cudaError_t launch_adaptive_rsi_update(const AdaptiveRsiArgs& a, cudaStream_t st);
cudaError_t launch_state_copy(float* state_f, int* state_i, int* state_as, float* qpos, float* qvel, int* cursor, int n,
                              int nv, int G, int to_state, cudaStream_t st);
}  // namespace drl

using namespace drl;

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
  return code;
}

#define CUDA_TRY(expr)                                                                        \
  do {                                                                                        \
    cudaError_t e__ = (expr);                                                                 \
    if (e__ != cudaSuccess) return fail(DRL_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e__)); \
  } while (0)

// Every entry point runs on the env's device and leaves the caller's current device as it found it (several envs on
// different GPUs may live in one process; PyTorch's current device must not change under the caller).
struct DeviceGuard {
  int prev = -1, dev;
  explicit DeviceGuard(int d) : dev(d) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    if (prev >= 0 && prev != dev) cudaSetDevice(prev);
  }
};

// The device buffers of an env, grouped by lifetime.  A call that replaces a group builds the new one complete in a
// local, synchronises when enqueued steps may still read the old one, and only then moves it into the env together
// with its host copies: a call that fails leaves the env as it was.
struct StateBufs {                        // alloc_state: per-env state and statistics
  DevBuf<float> state_f, extras_last;
  DevBuf<int> state_i, state_as;
  DevBuf<double> state_d, stats;
  DevBuf<float> tor_hist, med_tor_sm;     // cfg.monitor_median_torque
  DevBuf<float> ee_f;                     // cfg.ee_weight > 0: [N][2] last / smoothed ee_rew
  DevBuf<double> ee_d;                    // cfg.ee_weight > 0: [N] lifetime sum of ee_rew
  // per-step statistics rows (one per thread block of the step kernel) + the ticket that elects the summing block
  DevBuf<double> cta_rows;
  DevBuf<unsigned> cta_ticket;
};

struct RingBufs {                         // alloc_state: the episode ring
  DevBuf<int> len, rsi_pos, et_pos;
  DevBuf<float> ret;
  DevBuf<unsigned char> difficult;
  DevBuf<unsigned long long> head;
};

struct MocapBufs {                        // drl_upload_mocap
  DevBuf<float> ref, step_vel, step_last_comx;
  DevBuf<double> des_vel_prefix;          // float64: differences of long prefix sums lose ~1e-5 in float32
  DevBuf<int> step_off, step_len;
  DevBuf<unsigned char> left_step;
  std::vector<int> step_len_h;            // host copy (the failure-weighted RSI bin layout is built from it)
};

// mocap library (drl_set_mocap_clips); one clip spanning the table after every drl_upload_mocap.  Device tables only
// while there is more than one clip.
struct ClipBufs {
  std::vector<int> first_h;               // [n_clips + 1]
  std::vector<double> weight_h;           // [n_clips] normalised
  DevBuf<int> first;                      // [n_clips + 1]
  DevBuf<int> step_clip;                  // [n_steps]
  DevBuf<double> cdf;                     // [n_clips]
  DevBuf<unsigned long long> stats;       // [n_clips][kClipStatCount]
  DevBuf<ClipLibrary> lib;                // the device struct StepArgs::clips points at
};

// failure-weighted RSI (drl_set_adaptive_rsi): the table of one mocap and bin width, built when first enabled for them
struct ArsBufs {
  int gen = -1, bin_samples = 0;          // the mocap_gen and bin width it was built for
  DevBuf<double> counts;                  // [2][n_bins] started, difficult
  DevBuf<double> u, cdf, prob;            // [n_bins]
  DevBuf<int> bins;                       // [n_bins][3] step, first, width; [n_steps] first bin of each step
  DevBuf<unsigned> inc;                   // [2][n_bins]
  DevBuf<int> env_bin;                    // [N]
  int n_bins() const { return (int)u.size(); }
};

struct DrlEnv {
  DrlConfig cfg;
  DevModel hm;                 // host copy
  bool have_model = false, have_mocap = false;
  int G = 16, block = 128, nv = 0;
  int actuation = DRL_ACTUATION_TORQUE;   // drl_set_actuation
  double dof_range[kMaxDof][2];           // joint ranges in float64: the PD target map is computed from them
  DevBuf<DevModel> d_model;               // the model block hm is published to (publish_model)
  StateBufs st;
  RingBufs ring;
  int ring_cap = 1 << 16;
  MocapBufs mocap;
  int mocap_gen = 0;                      // bumped by every drl_upload_mocap and drl_set_mocap_clips
  ClipBufs clips;
  ArsBufs ars;
  int ars_halflife = 0;
  float ars_lambda = 0.f;                 // 0 = off
  int eval_mode = 0;
  DevBuf<float> speed_profile;            // drl_set_speed_profile; empty when off
  int playback = 0;
  int frame_skip_override = -1;
  unsigned ref_obs = 0;                   // drl_set_ref_obs, packed as StepArgs::ref_obs; 0 = off
  bool stepped = false;                   // a drl_reset or drl_step has been enqueued
  DevBuf<float> debug;                    // drl_debug_set
  // contact termination (drl_set_contact_termination): per-env episode count, allocated when first enabled
  DevBuf<int> contact_et;
  // fused VecNormalize moments (drl_attach_vecnorm): borrowed device pointers
  float* vn_ret = nullptr;
  float vn_gamma = 0.f;
  double* vn_packed = nullptr;
};

extern "C" int drl_version(void) { return DRL_ABI_VERSION; }
extern "C" const char* drl_last_error(void) { return g_err; }

extern "C" int drl_create(const DrlConfig* cfg, DrlEnv** out) {
  if (!cfg || !out) return fail(DRL_ERR_INVALID, "drl_create: null argument");
  if (cfg->num_envs <= 0) return fail(DRL_ERR_INVALID, "drl_create: num_envs must be positive");
  if (cfg->obs_dim <= 0 || cfg->obs_dim > kMaxObs || cfg->act_dim <= 0 || cfg->act_dim > kMaxAct)
    return fail(DRL_ERR_INVALID, "drl_create: obs_dim/act_dim out of range");
  if (cfg->frame_skip < 0) return fail(DRL_ERR_INVALID, "drl_create: frame_skip must be >= 0");
  if (cfg->integrator != DRL_INTEGRATOR_RK4 && cfg->integrator != DRL_INTEGRATOR_EULER)
    return fail(DRL_ERR_INVALID, "drl_create: unknown integrator");
  if (!isfinite(cfg->ee_weight) || cfg->ee_weight < 0.0)
    return fail(DRL_ERR_INVALID, "drl_create: ee_weight must be finite and >= 0");
  if (cfg->ee_weight > 0.0 && !(cfg->ee_scale > 0.0 && isfinite(cfg->ee_scale)))
    return fail(DRL_ERR_INVALID, "drl_create: ee_scale must be positive and finite when ee_weight > 0");
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(DRL_ERR_INVALID, "drl_create: no CUDA device %d", cfg->device);
  DrlEnv* e = new DrlEnv();
  e->cfg = *cfg;
  *out = e;
  return DRL_OK;
}

extern "C" int drl_destroy(DrlEnv* e) {
  if (!e) return DRL_OK;
  DeviceGuard guard__(e->cfg.device);
  delete e;
  return DRL_OK;
}

// the smallest CTA the library launches carries 32 / G environments
static size_t max_cta_blocks(const DrlEnv* e, size_t N) { return (N + (32 / e->G) - 1) / (32 / e->G); }

// per-step statistics rows for observation rows of obs_row floats: one per block, then one per group of kStatGroup
// blocks (two-level fixed-order sum in the step kernel)
static cudaError_t alloc_cta_rows(const DrlEnv* e, size_t N, int obs_row, DevBuf<double>& rows) {
  const size_t max_blocks = max_cta_blocks(e, N), max_groups = (max_blocks + kStatGroup - 1) / kStatGroup;
  return rows.alloc((max_blocks + max_groups) * (2 * (size_t)obs_row + 2 + DRL_STATS_COUNT));
}

// persistent per-env state, statistics and episode ring, moved into the env once all of it is allocated
static int alloc_state(DrlEnv* e, size_t N) {
  DevBuf<DevModel> model;
  StateBufs s;
  RingBufs r;
  CUDA_TRY(model.alloc(1));
  CUDA_TRY(s.state_f.zeros(N * 4 * e->G));
  CUDA_TRY(s.state_i.alloc(N * kCurCount8));
  CUDA_TRY(s.state_as.zeros(N * e->G));
  CUDA_TRY(s.state_d.zeros(N * 4));
  CUDA_TRY(s.extras_last.zeros(N * 16));
  CUDA_TRY(s.stats.zeros(DRL_STATS_COUNT));
  CUDA_TRY(r.len.alloc(e->ring_cap));
  CUDA_TRY(r.ret.alloc(e->ring_cap));
  CUDA_TRY(r.rsi_pos.alloc(e->ring_cap));
  CUDA_TRY(r.et_pos.alloc(e->ring_cap));
  CUDA_TRY(r.difficult.alloc(e->ring_cap));
  CUDA_TRY(r.head.zeros(1));
  if (e->cfg.monitor_median_torque) {
    const size_t cap = (size_t)(e->cfg.ep_dur_max > 0 ? e->cfg.ep_dur_max : 1);
    CUDA_TRY(s.tor_hist.zeros(N * cap));
    CUDA_TRY(s.med_tor_sm.zeros(N));
  }
  if (e->cfg.ee_weight > 0.0) {
    CUDA_TRY(s.ee_f.zeros(N * 2));
    CUDA_TRY(s.ee_d.zeros(N));
  }
  {
    const size_t max_groups = (max_cta_blocks(e, N) + kStatGroup - 1) / kStatGroup;
    CUDA_TRY(alloc_cta_rows(e, N, e->cfg.obs_dim, s.cta_rows));
    // tickets: [0] counts finished groups, [1 + g] the finished blocks of group g
    CUDA_TRY(s.cta_ticket.zeros(1 + max_groups));
  }
  // count_steps_same_vel starts at 1 (straight_walk_trajecs.py:124)
  std::vector<int> init(N * kCurCount8, 0);
  for (size_t i = 0; i < N; i++) init[i * kCurCount8 + kCurCount] = 1;
  CUDA_TRY(cudaMemcpy(s.state_i.get(), init.data(), init.size() * sizeof(int), cudaMemcpyHostToDevice));
  e->d_model = std::move(model);
  e->st = std::move(s);
  e->ring = std::move(r);
  return DRL_OK;
}

// m becomes the model block on the device, then the env's host copy; the caller holds the env's DeviceGuard
static int publish_model(DrlEnv* e, const DevModel& m) {
  CUDA_TRY(cudaDeviceSynchronize());          // enqueued steps may still read the model block
  CUDA_TRY(cudaMemcpy(e->d_model.get(), &m, sizeof(DevModel), cudaMemcpyHostToDevice));
  e->hm = m;
  return DRL_OK;
}

extern "C" int drl_upload_model(DrlEnv* e, const DrlWalkerModel* m) {
  if (!e || !m) return fail(DRL_ERR_INVALID, "drl_upload_model: null argument");
  const DrlConfig& c = e->cfg;
  if (m->nv <= 0 || m->nv > kMaxDof || m->nv > DRL_MAX_DOF) return fail(DRL_ERR_INVALID, "model: nv out of range");
  if (m->nb <= 0 || m->nb > kMaxBody) return fail(DRL_ERR_INVALID, "model: at most %d bodies are supported", kMaxBody);
  if (m->nu <= 0 || m->nu > kMaxAct || m->nu != c.act_dim) return fail(DRL_ERR_INVALID, "model: nu != act_dim");
  if (m->nv != 14 && m->nv != 19)
    return fail(DRL_ERR_UNSUPPORTED, "model: kernels are instantiated for nv = 14 and nv = 19 (got %d)", m->nv);
  if (e->have_model) return fail(DRL_ERR_STATE, "drl_upload_model: a model is already attached to this env");
  DevModel& d = e->hm;
  memset(&d, 0, sizeof d);
  d.nv = m->nv; d.nb = m->nb; d.nu = m->nu; d.nsite = m->n_site;
  d.timestep = (float)m->timestep; d.gravity_z = (float)m->gravity_z;
  // solref -> (K, B) as MuJoCo's mj_makeImpedance; timeconst is clamped to 2*timestep (refsafe)
  const double tc = fmax(m->solref[0], 2 * m->timestep), dr = m->solref[1];
  const double dmax = fmin(0.9999, fmax(0.0001, m->solimp[1])), d0 = fmin(0.9999, fmax(0.0001, m->solimp[0]));
  d.Kc = (float)(1.0 / (dmax * dmax * tc * tc * dr * dr));
  d.Bc = (float)(2.0 / (dmax * tc));
  d.imp_d0 = (float)d0; d.imp_dmax = (float)dmax; d.imp_width = (float)fmax(1e-15, m->solimp[2]);
  d.imp_mid = (float)fmin(0.9999, fmax(0.0001, m->solimp[3])); d.imp_power = (float)fmax(1.0, m->solimp[4]);
  d.imp_inv_width = 1.f / d.imp_width; d.imp_inv_mid = 1.f / d.imp_mid; d.imp_inv_1mmid = 1.f / (1.f - d.imp_mid);
  if (m->body_parent[0] != -1) return fail(DRL_ERR_INVALID, "model: body 0 must be the root");
  d.root_z0 = (float)m->body_pos[0][2];
  for (int b = 0; b < m->nb; b++) {
    const int p = m->body_parent[b];
    if (p >= b) return fail(DRL_ERR_INVALID, "model: bodies must be topologically ordered");
    if (b > 0 && p < 0) return fail(DRL_ERR_INVALID, "model: exactly one root body is supported");
    d.body_parent[b] = p;
    d.body_mass[b] = (float)m->body_mass[b];
    d.body_invw_tran[b] = (float)m->body_invweight0[b][0];
    for (int i = 0; i < 3; i++) {
      d.body_pos[b][i] = (float)m->body_pos[b][i];
      d.body_ipos[b][i] = (float)m->body_ipos[b][i];
      d.body_inertia[b][i] = (float)m->body_inertia[b][i];
    }
  }
  int G = m->nv <= 16 ? 16 : 32;
  if (c.lanes_per_env != 0 && c.lanes_per_env != G)
    return fail(DRL_ERR_INVALID, "config: lanes_per_env must be 0 or %d for this model", G);
  bool seen_hinge_root = false;
  int body_ndof[kMaxBody] = {0};
  for (int j = 0; j < m->nv; j++) {
    const int b = m->dof_body[j];
    if (b < 0 || b >= m->nb) return fail(DRL_ERR_INVALID, "model: dof %d has a bad body", j);
    if (j > 0 && b < m->dof_body[j - 1]) return fail(DRL_ERR_INVALID, "model: dofs must be ordered by body");
    body_ndof[b]++;
    d.dof_body[j] = b; d.dof_type[j] = m->dof_type[j];
    d.dof_limited[j] = m->dof_limited[j];
    d.dof_code[j] = m->dof_axis_idx[j] | (m->dof_axis_sign[j] < 0 ? 4 : 0);
    d.dof_sign[j] = (float)m->dof_axis_sign[j]; d.dof_ref[j] = (float)m->dof_ref[j];
    d.dof_damping[j] = (float)m->dof_damping[j]; d.dof_armature[j] = (float)m->dof_armature[j];
    d.dof_lo[j] = (float)m->dof_range[j][0]; d.dof_hi[j] = (float)m->dof_range[j][1];
    e->dof_range[j][0] = m->dof_range[j][0]; e->dof_range[j][1] = m->dof_range[j][1];
    d.dof_invw[j] = (float)m->dof_invweight0[j];
    if (m->dof_type[j] == 0) {
      if (b != 0 || seen_hinge_root) return fail(DRL_ERR_UNSUPPORTED, "model: slides are supported on the root body, before its hinges");
      if (j != d.nslide) return fail(DRL_ERR_UNSUPPORTED, "model: root slides must come first");
      d.nslide++;
      d.dof_slide_z[j] = m->dof_axis_idx[j] == 2 ? (float)m->dof_axis_sign[j] : 0.f;
    } else if (b == 0) {
      seen_hinge_root = true;
    }
  }
  // the tree itself (which body hangs where, which dofs move it) is compiled into the kernels as chain tables
  if (!topology_matches(m->nv, m->nb, d.body_parent, d.dof_body, d.dof_type))
    return fail(DRL_ERR_UNSUPPORTED, "model: the kernels are compiled for the chain layout of walker3d_flat_feet.xml "
                                     "(nv 14) and walker_165cm_65kg.xml (nv 19); this model's tree differs");
  for (int b = 0; b < m->nb; b++)
    if (body_ndof[b] == 0) return fail(DRL_ERR_UNSUPPORTED, "model: every body needs at least one joint");
  for (int u = 0; u < m->nu; u++) {
    d.act_dof[u] = m->act_dof[u]; d.act_gear[u] = (float)m->act_gear[u];
    d.act_clo[u] = (float)m->act_ctrlrange[u][0]; d.act_chi[u] = (float)m->act_ctrlrange[u][1];
    d.act_flo[u] = (float)m->act_forcerange[u][0]; d.act_fhi[u] = (float)m->act_forcerange[u][1];
    for (int u2 = 0; u2 < u; u2++)
      if (m->act_dof[u2] == m->act_dof[u]) return fail(DRL_ERR_UNSUPPORTED, "model: one motor per joint");
  }
  // contact candidates: box corners first (8 per box), then spheres
  int nc = 0;
  for (int x = 0; x < m->n_box; x++)
    for (int i = 0; i < 8; i++, nc++) {
      if (nc >= kMaxCand) return fail(DRL_ERR_INVALID, "model: too many contact candidates");
      d.cand_body[nc] = m->box_body[x];
      d.cand_mu[nc] = (float)m->box_mu[x];
      for (int k = 0; k < 3; k++) {
        d.cand_pos[nc][k] = (float)m->box_corner[x][i][k];
        d.cand_aux[nc][k] = (float)m->box_center[x][k];
      }
    }
  d.nbox_cand = nc;
  for (int x = 0; x < m->n_box; x++) {
    if (d.box_body_mask & (1u << m->box_body[x])) return fail(DRL_ERR_UNSUPPORTED, "model: at most one box geom per body");
    d.box_body_mask |= 1u << m->box_body[x];
  }
  for (int s = 0; s < m->n_sphere; s++, nc++) {
    if (nc >= kMaxCand) return fail(DRL_ERR_INVALID, "model: too many contact candidates");
    d.cand_body[nc] = m->sphere_body[s];
    d.cand_mu[nc] = (float)m->sphere_mu[s];
    for (int k = 0; k < 3; k++) d.cand_pos[nc][k] = (float)m->sphere_pos[s][k];
    d.cand_aux[nc][0] = (float)m->sphere_radius[s];
  }
  d.ncand = nc;
  if (d.nbox_cand > G) return fail(DRL_ERR_UNSUPPORTED, "model: box corners must fit one lane pass");
  if (d.ncand > 2 * G) return fail(DRL_ERR_UNSUPPORTED, "model: more than %d contact candidates", 2 * G);
  // spheres must not share a pass with box corners (the first-four rule uses 8-lane segments of pass 0)
  if (d.nbox_cand % G != 0 && d.ncand > d.nbox_cand) {
    // shift the spheres to the start of the next pass
    const int nsph = d.ncand - d.nbox_cand, dst0 = G;
    if (dst0 + nsph > kMaxCand || dst0 + nsph > 2 * G) return fail(DRL_ERR_UNSUPPORTED, "model: candidate layout");
    for (int s = nsph - 1; s >= 0; s--) {
      d.cand_body[dst0 + s] = d.cand_body[d.nbox_cand + s];
      d.cand_mu[dst0 + s] = d.cand_mu[d.nbox_cand + s];
      for (int k = 0; k < 3; k++) {
        d.cand_pos[dst0 + s][k] = d.cand_pos[d.nbox_cand + s][k];
        d.cand_aux[dst0 + s][k] = d.cand_aux[d.nbox_cand + s][k];
      }
    }
    for (int s = d.nbox_cand; s < dst0; s++) {   // dead slots: a sphere far above the ground
      d.cand_body[s] = 0; d.cand_mu[s] = 1.f;
      d.cand_pos[s][0] = d.cand_pos[s][1] = 0.f; d.cand_pos[s][2] = 1e6f;
      d.cand_aux[s][0] = 0.f;
    }
    d.ncand = dst0 + nsph;
  }
  for (int s = 0; s < m->n_site; s++) {
    if (s >= kMaxSite) return fail(DRL_ERR_INVALID, "model: too many sites");
    d.site_body[s] = m->site_body[s];
    for (int k = 0; k < 3; k++) d.site_pos[s][k] = (float)m->site_pos[s][k];
  }
  if (m->n_site == 0) return fail(DRL_ERR_INVALID, "model: foot-corner sites are required (mimic_env.py:546-559)");
  if (m->n_ee < 0 || m->n_ee > DRL_MAX_EE || m->n_ee > kMaxEE)
    return fail(DRL_ERR_INVALID, "model: n_ee must be in 0..%d", DRL_MAX_EE);
  d.n_ee = m->n_ee;
  for (int x = 0; x < m->n_ee; x++) {
    if (m->ee_body[x] < 0 || m->ee_body[x] >= m->nb) return fail(DRL_ERR_INVALID, "model: ee_body[%d] out of range", x);
    d.ee_body[x] = m->ee_body[x];
    for (int k = 0; k < 3; k++) d.ee_pos[x][k] = (float)m->ee_pos[x][k];
  }
  if (c.ee_weight > 0.0 && m->n_ee == 0)
    return fail(DRL_ERR_INVALID, "config: ee_weight > 0 needs end-effector points in the model (n_ee == 0)");
  // ---- configuration ----
  d.frame_skip = c.frame_skip; d.integrator = c.integrator; d.ep_dur_max = c.ep_dur_max;
  d.mirror_policy = c.mirror_policy; d.phase_mode = c.phase_mode; d.n_phase_joints = c.n_phase_joints;
  d.eval_n_times = c.eval_n_times > 0 ? c.eval_n_times : 1;
  for (int i = 0; i < 4; i++) d.phase_joints[i] = c.phase_joints[i];
  d.obs_dim = c.obs_dim; d.act_dim = c.act_dim;
  d.obs_row = c.obs_dim;   // drl_set_ref_obs widens it
  d.n_phase_obs = c.phase_mode == DRL_PHASE_FROM_CURSOR ? 1 : 2 * c.n_phase_joints;
  d.n_des_vel = c.obs_dim - d.n_phase_obs - (m->nv - 1) - m->nv;
  if (d.n_des_vel < 1 || d.n_des_vel > 2) return fail(DRL_ERR_INVALID, "config: obs_dim inconsistent with the model");
  d.ctrl_freq_inv = (float)(1.0 / c.ctrl_freq);
  d.w_pos = (float)c.rew_weights[0]; d.w_vel = (float)c.rew_weights[1]; d.w_com = (float)c.rew_weights[2];
  d.rew_scale = (float)c.rew_scale; d.alive_bonus = (float)c.alive_bonus; d.fall_z = (float)c.fall_z;
  d.w_ee = (float)c.ee_weight; d.ee_scale = (float)c.ee_scale;
  for (int i = 0; i < c.obs_dim; i++) {
    d.mirror_obs_idx[i] = c.mirror_obs_idx[i]; d.mirror_obs_sign[i] = c.mirror_obs_sign[i];
    if (c.mirror_obs_idx[i] < 0 || c.mirror_obs_idx[i] >= c.obs_dim) return fail(DRL_ERR_INVALID, "config: mirror_obs_idx");
  }
  for (int i = 0; i < c.act_dim; i++) {
    d.mirror_act_idx[i] = c.mirror_act_idx[i]; d.mirror_act_sign[i] = c.mirror_act_sign[i];
    if (c.mirror_act_idx[i] < 0 || c.mirror_act_idx[i] >= c.act_dim) return fail(DRL_ERR_INVALID, "config: mirror_act_idx");
  }
  d.com_mask = 0x7u;     // _get_COM_indices() == [0,1,2] for both walkers
  d.com_z_dof = 2;
  d.early_termination = c.early_termination ? 1 : 0;
  d.trunk_dof0 = 3;      // _get_trunk_rot_joint_indices() == [3,4,5] for both walkers (frontal, sagittal, axial)
  d.seed = c.seed; d.env_id_offset = c.env_id_offset;
  e->nv = m->nv;
  e->G = G;
  e->block = 128;
  DeviceGuard guard__(c.device);
  const int rc = alloc_state(e, (size_t)c.num_envs);
  if (rc != DRL_OK) {            // e.g. out of memory for a very large batch: leave the env without a model
    (void)cudaGetLastError();     // a failed cudaMalloc also parks its code as the "last error": clear it
    return rc;
  }
  e->have_model = true;
  return e->have_mocap ? publish_model(e, e->hm) : DRL_OK;
}

extern "C" int drl_upload_mocap(DrlEnv* e, int32_t cursor_mode, int32_t increment, const double* ref, int32_t n_samples,
                                const int32_t* step_off, const int32_t* step_len, const uint8_t* left_step,
                                const double* step_vel, const double* step_last_comx, int32_t n_steps,
                                int32_t com_z_col, const double* des_vel_prefix, int32_t des_vel_window) {
  if (!e || !ref || !step_off || !step_len || !left_step || !step_vel || !step_last_comx)
    return fail(DRL_ERR_INVALID, "drl_upload_mocap: null argument");
  if (!e->have_model) return fail(DRL_ERR_STATE, "drl_upload_mocap: upload the model first");
  if (n_samples <= 0 || n_steps <= 0 || increment <= 0) return fail(DRL_ERR_INVALID, "drl_upload_mocap: empty mocap");
  if (e->ars_lambda > 0.f)
    return fail(DRL_ERR_STATE, "drl_upload_mocap: failure-weighted RSI is on (its bins would go stale); set lambda 0 first");
  if (cursor_mode != DRL_CURSOR_STEPWISE && cursor_mode != DRL_CURSOR_WRAP)
    return fail(DRL_ERR_INVALID, "drl_upload_mocap: unknown cursor mode");
  if (cursor_mode == DRL_CURSOR_WRAP && !des_vel_prefix)
    return fail(DRL_ERR_INVALID, "drl_upload_mocap: wrap mode needs the desired-velocity prefix sums");
  for (int i = 0; i < n_steps; i++) {
    if (step_off[i] < 0 || step_len[i] <= 2 * increment || step_off[i] + step_len[i] > n_samples)
      return fail(DRL_ERR_INVALID, "drl_upload_mocap: step %d out of range or shorter than two increments", i);
  }
  DeviceGuard guard__(e->cfg.device);
  const int G = e->G, nv = e->nv;
  std::vector<float> padded((size_t)n_samples * 2 * G, 0.f);
  for (int t = 0; t < n_samples; t++)
    for (int j = 0; j < nv; j++) {
      padded[(size_t)t * 2 * G + j] = (float)ref[(size_t)t * 2 * nv + j];
      padded[(size_t)t * 2 * G + G + j] = (float)ref[(size_t)t * 2 * nv + nv + j];
    }
  MocapBufs t;
  // des_vel_prefix: one leading zero row per step (the prefix sums restart at every clip of a wrap-mode library)
  if (t.ref.from_host(padded.data(), padded.size()) || t.step_off.from_host(step_off, n_steps) ||
      t.step_len.from_host(step_len, n_steps) || t.left_step.from_host(left_step, n_steps) ||
      t.step_vel.from_host(step_vel, n_steps) || t.step_last_comx.from_host(step_last_comx, n_steps) ||
      (des_vel_prefix && t.des_vel_prefix.from_host(des_vel_prefix, (size_t)(n_samples + n_steps) * 2)))
    return fail(DRL_ERR_CUDA, "drl_upload_mocap: device copy failed");
  t.step_len_h.assign(step_len, step_len + n_steps);
  DevModel d = e->hm;
  d.cursor_mode = cursor_mode; d.increment = increment; d.n_steps = n_steps; d.n_samples = n_samples;
  d.com_z_col = com_z_col; d.des_vel_window = des_vel_window;
  if (const int rc = publish_model(e, d)) return rc;   // synchronises: enqueued steps may still read the old tables
  e->mocap = std::move(t);
  e->clips = ClipBufs{{0, n_steps}, {1.0}};    // one clip spanning the table
  e->mocap_gen++;
  e->have_mocap = true;
  return DRL_OK;
}

static int ready(DrlEnv* e, const char* who) {
  if (!e) return fail(DRL_ERR_INVALID, "%s: null env", who);
  if (!e->have_model || !e->have_mocap) return fail(DRL_ERR_STATE, "%s: model and mocap must be uploaded first", who);
  if (e->hm.cursor_mode == DRL_CURSOR_WRAP && (int)e->clips.first_h.size() != e->hm.n_steps + 1)
    return fail(DRL_ERR_STATE, "%s: a wrap-mode mocap of %d steps needs drl_set_mocap_clips with one clip per step", who,
                e->hm.n_steps);
  return DRL_OK;
}

extern "C" int drl_set_mocap_clips(DrlEnv* e, int32_t n_clips, const int32_t* clip_first_step, const double* clip_weight) {
  if (!e || !clip_first_step || !clip_weight) return fail(DRL_ERR_INVALID, "drl_set_mocap_clips: null argument");
  if (!e->have_model || !e->have_mocap) return fail(DRL_ERR_STATE, "drl_set_mocap_clips: upload the mocap first");
  if (e->ars_lambda > 0.f)
    return fail(DRL_ERR_STATE, "drl_set_mocap_clips: failure-weighted RSI is on (its bins would go stale); set lambda 0 first");
  const int n_steps = e->hm.n_steps;
  const bool wrap = e->hm.cursor_mode == DRL_CURSOR_WRAP;
  if (n_clips < 1 || n_clips > n_steps) return fail(DRL_ERR_INVALID, "drl_set_mocap_clips: n_clips = %d outside [1, %d]",
                                                    n_clips, n_steps);
  if (clip_first_step[0] != 0 || clip_first_step[n_clips] != n_steps)
    return fail(DRL_ERR_INVALID, "drl_set_mocap_clips: the clips must start at step 0 and end at step %d", n_steps);
  double total = 0.0;
  for (int k = 0; k < n_clips; k++) {
    const int len = clip_first_step[k + 1] - clip_first_step[k];
    // the reference's wrap (straight:330-333) goes to the clip's step 0 or 1
    if (wrap ? len != 1 : len < 2)
      return fail(DRL_ERR_INVALID, "drl_set_mocap_clips: clip %d has %d steps (%s)", k, len,
                  wrap ? "a wrap-mode clip is one step" : "a stepwise clip needs at least 2");
    if (!(isfinite(clip_weight[k]) && clip_weight[k] >= 0.0))
      return fail(DRL_ERR_INVALID, "drl_set_mocap_clips: clip_weight[%d] = %g must be finite and >= 0", k, clip_weight[k]);
    total += clip_weight[k];
  }
  if (!(total > 0.0 && isfinite(total)))
    return fail(DRL_ERR_INVALID, "drl_set_mocap_clips: the clip weights must have a positive finite sum");
  DeviceGuard guard__(e->cfg.device);
  ClipBufs c;
  c.first_h.assign(clip_first_step, clip_first_step + n_clips + 1);
  c.weight_h.resize(n_clips);
  for (int k = 0; k < n_clips; k++) c.weight_h[k] = clip_weight[k] / total;
  if (n_clips > 1) {
    std::vector<int> step_clip(n_steps);
    for (int k = 0; k < n_clips; k++)
      for (int s = clip_first_step[k]; s < clip_first_step[k + 1]; s++) step_clip[s] = k;
    // CDF of the clip draw; 1 from the last clip with a positive weight on, so that no rounding selects a trailing
    // zero-weight clip
    int last_pos = 0;
    for (int k = 0; k < n_clips; k++)
      if (clip_weight[k] > 0.0) last_pos = k;
    std::vector<double> cdf(n_clips);
    double acc = 0.0;
    for (int k = 0; k < n_clips; k++) {
      acc += clip_weight[k];
      cdf[k] = k >= last_pos ? 1.0 : acc / total;
    }
    if (c.first.from_host(clip_first_step, (size_t)n_clips + 1) || c.step_clip.from_host(step_clip.data(), n_steps) ||
        c.cdf.from_host(cdf.data(), n_clips))
      return fail(DRL_ERR_CUDA, "drl_set_mocap_clips: device copy failed");
    CUDA_TRY(c.stats.zeros((size_t)n_clips * kClipStatCount));
    const ClipLibrary h{n_clips, c.first.get(), c.step_clip.get(), c.cdf.get(), c.stats.get()};
    CUDA_TRY(c.lib.from_host(&h, 1));
  }
  CUDA_TRY(cudaDeviceSynchronize());          // enqueued steps may still read the tables
  e->clips = std::move(c);
  e->mocap_gen++;                             // the failure-weighted RSI bins weigh the clips: rebuild them
  return DRL_OK;
}

extern "C" int drl_get_clip_stats(DrlEnv* e, int64_t* out, void* stream) {
  if (!e || !out) return fail(DRL_ERR_INVALID, "drl_get_clip_stats: null argument");
  if (!e->clips.stats.get()) return fail(DRL_ERR_STATE, "drl_get_clip_stats: the mocap has a single clip");
  DeviceGuard guard__(e->cfg.device);
  CUDA_TRY(cudaMemcpyAsync(out, e->clips.stats.get(), e->clips.stats.size() * sizeof(int64_t), cudaMemcpyDeviceToDevice,
                           (cudaStream_t)stream));
  return DRL_OK;
}

static AdaptiveRsiArgs ars_args(DrlEnv* e, double rho) {
  AdaptiveRsiArgs a;
  a.n_bins = e->ars.n_bins(); a.rho = rho; a.lambda = (double)e->ars_lambda;
  a.u = e->ars.u.get(); a.counts = e->ars.counts.get(); a.inc = e->ars.inc.get(); a.cdf = e->ars.cdf.get();
  a.prob = e->ars.prob.get();
  return a;
}

static StepArgs make_args(DrlEnv* e) {
  StepArgs a;
  memset(&a, 0, sizeof a);
  const StateBufs& s = e->st;
  const MocapBufs& m = e->mocap;
  const RingBufs& r = e->ring;
  a.model = e->d_model.get(); a.num_envs = e->cfg.num_envs;
  a.frame_skip = e->frame_skip_override >= 0 ? e->frame_skip_override : e->cfg.frame_skip;
  a.state_f = s.state_f.get(); a.state_i = s.state_i.get(); a.state_as = s.state_as.get(); a.state_d = s.state_d.get();
  a.ref = m.ref.get(); a.step_off = m.step_off.get(); a.step_len = m.step_len.get(); a.left_step = m.left_step.get();
  a.step_vel = m.step_vel.get(); a.step_last_comx = m.step_last_comx.get(); a.des_vel_prefix = m.des_vel_prefix.get();
  a.extras = s.extras_last.get(); a.stats = s.stats.get();
  a.ring_len = r.len.get(); a.ring_ret = r.ret.get(); a.ring_head = r.head.get(); a.ring_cap = e->ring_cap;
  a.ring_rsi_pos = r.rsi_pos.get(); a.ring_et_pos = r.et_pos.get(); a.ring_difficult = r.difficult.get();
  a.eval_mode = e->eval_mode;
  a.speed_profile = e->speed_profile.get(); a.speed_profile_len = (int)e->speed_profile.size();   // null / 0 when off
  a.playback = e->playback;
  a.cta_rows = s.cta_rows.get(); a.cta_ticket = s.cta_ticket.get();
  a.tor_hist = s.tor_hist.get(); a.med_tor_sm = s.med_tor_sm.get();
  a.ee_f = s.ee_f.get(); a.ee_d = s.ee_d.get();
  a.contact_et = e->hm.et_contact_mask ? e->contact_et.get() : nullptr;
  if (e->ars_lambda > 0.f) {
    a.ars_coin = (unsigned long long)llround((double)e->ars_lambda * 4294967296.0);
    a.ars_n_bins = e->ars.n_bins(); a.ars_bin_samples = e->ars.bin_samples;
    a.ars_cdf = e->ars.cdf.get(); a.ars_bins = e->ars.bins.get(); a.ars_inc = e->ars.inc.get();
    a.ars_env_bin = e->ars.env_bin.get();
  }
  a.clips = e->clips.lib.get();
  a.ref_obs = e->ref_obs;
  a.vn_ret = e->vn_ret; a.vn_gamma = e->vn_gamma; a.packed = e->vn_packed;
  if (e->playback) a.frame_skip = 0;
  a.debug = e->debug.get();
  return a;
}

extern "C" int drl_reset(DrlEnv* e, const uint8_t* mask, const int32_t* inj_istep, const int32_t* inj_pos, float* obs,
                         void* stream) {
  int rc = ready(e, "drl_reset");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  if (!obs) return fail(DRL_ERR_INVALID, "drl_reset: obs is null");
  StepArgs a = make_args(e);
  a.reset_mask = mask; a.inj_istep = inj_istep; a.inj_pos = inj_pos; a.obs = obs;
  a.debug = nullptr;
  CUDA_TRY(launch_step(a, e->nv, e->G, e->cfg.integrator == DRL_INTEGRATOR_RK4, 1, e->block, false, false,
                       (cudaStream_t)stream));
  e->stepped = true;
  return DRL_OK;
}

extern "C" int drl_step(DrlEnv* e, const float* actions, float* obs, float* rew, uint8_t* done, float* terminal_obs,
                        const int32_t* inj_istep, const int32_t* inj_pos, void* stream) {
  int rc = ready(e, "drl_step");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  if (!actions || !obs || !rew || !done) return fail(DRL_ERR_INVALID, "drl_step: null tensor");
  StepArgs a = make_args(e);
  a.actions = actions; a.obs = obs; a.rew = rew; a.done = done; a.terminal_obs = terminal_obs;
  a.inj_istep = inj_istep; a.inj_pos = inj_pos;
  const bool rk4 = e->cfg.integrator == DRL_INTEGRATOR_RK4, pd = e->actuation == DRL_ACTUATION_PD;
  if (a.debug && rk4) return fail(DRL_ERR_UNSUPPORTED, "drl_step: the dump variant exists for the Euler integrator only");
  if (a.debug && pd) return fail(DRL_ERR_UNSUPPORTED, "drl_step: the dump variant exists for torque actuation only");
  CUDA_TRY(launch_step(a, e->nv, e->G, rk4, 0, e->block, a.debug != nullptr, pd, (cudaStream_t)stream));
  e->stepped = true;
  if (e->ars_lambda > 0.f) CUDA_TRY(launch_adaptive_rsi_update(ars_args(e, pow(2.0, -1.0 / e->ars_halflife)),
                                                               (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_attach_vecnorm(DrlEnv* e, float* ret, float gamma, double* packed) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_attach_vecnorm: null env");
  if ((ret == nullptr) != (packed == nullptr))
    return fail(DRL_ERR_INVALID, "drl_attach_vecnorm: pass both tensors, or two nulls to detach");
  e->vn_ret = ret; e->vn_gamma = gamma; e->vn_packed = packed;
  return DRL_OK;
}

extern "C" int drl_get_state(DrlEnv* e, float* qpos, float* qvel, int32_t* cursor, void* stream) {
  int rc = ready(e, "drl_get_state");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  CUDA_TRY(launch_state_copy(e->st.state_f.get(), e->st.state_i.get(), e->st.state_as.get(), qpos, qvel, cursor,
                             e->cfg.num_envs, e->nv, e->G, 0, (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_set_state(DrlEnv* e, const float* qpos, const float* qvel, const int32_t* cursor, void* stream) {
  int rc = ready(e, "drl_set_state");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  CUDA_TRY(launch_state_copy(e->st.state_f.get(), e->st.state_i.get(), e->st.state_as.get(), const_cast<float*>(qpos),
                             const_cast<float*>(qvel), const_cast<int32_t*>(cursor), e->cfg.num_envs, e->nv, e->G, 1,
                             (cudaStream_t)stream));
  // an episode that continues from a state set here is no longer one that started with a random RSI draw
  if (e->ars.env_bin.get())
    CUDA_TRY(cudaMemsetAsync(e->ars.env_bin.get(), 0xFF, (size_t)e->cfg.num_envs * sizeof(int), (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_get_extras(DrlEnv* e, float* extras, void* stream) {
  int rc = ready(e, "drl_get_extras");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  if (!extras) return fail(DRL_ERR_INVALID, "drl_get_extras: null tensor");
  CUDA_TRY(launch_extras(e->st.state_f.get(), e->st.extras_last.get(), extras, e->cfg.num_envs, e->G,
                         (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_get_stats(DrlEnv* e, double* stats, void* stream) {
  int rc = ready(e, "drl_get_stats");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  if (!stats) return fail(DRL_ERR_INVALID, "drl_get_stats: null tensor");
  CUDA_TRY(cudaMemcpyAsync(stats, e->st.stats.get(), DRL_STATS_COUNT * sizeof(double), cudaMemcpyDeviceToDevice,
                           (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_reset_stats(DrlEnv* e, void* stream) {
  int rc = ready(e, "drl_reset_stats");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  CUDA_TRY(cudaMemsetAsync(e->st.stats.get(), 0, DRL_STATS_COUNT * sizeof(double), (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_get_episode_ring(DrlEnv* e, int32_t* ep_len, float* ep_ret, int32_t capacity,
                                    int64_t* total_episodes, void* stream) {
  int rc = ready(e, "drl_get_episode_ring");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  if (!total_episodes) return fail(DRL_ERR_INVALID, "drl_get_episode_ring: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const RingBufs& r = e->ring;
  unsigned long long head = 0;
  CUDA_TRY(cudaMemcpyAsync(&head, r.head.get(), sizeof head, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));     // the count is returned to the host by value
  *total_episodes = (int64_t)head;
  const int n = capacity < e->ring_cap ? capacity : e->ring_cap;
  if (ep_len && n > 0) CUDA_TRY(cudaMemcpyAsync(ep_len, r.len.get(), n * sizeof(int), cudaMemcpyDeviceToDevice, st));
  if (ep_ret && n > 0) CUDA_TRY(cudaMemcpyAsync(ep_ret, r.ret.get(), n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return DRL_OK;
}

extern "C" int drl_get_episode_positions(DrlEnv* e, int32_t* rsi_pos, int32_t* et_pos, uint8_t* difficult,
                                         int32_t capacity, void* stream) {
  int rc = ready(e, "drl_get_episode_positions");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  const int n = capacity < e->ring_cap ? capacity : e->ring_cap;
  if (n <= 0) return DRL_OK;
  if (rsi_pos) CUDA_TRY(cudaMemcpyAsync(rsi_pos, e->ring.rsi_pos.get(), n * sizeof(int), cudaMemcpyDeviceToDevice, st));
  if (et_pos) CUDA_TRY(cudaMemcpyAsync(et_pos, e->ring.et_pos.get(), n * sizeof(int), cudaMemcpyDeviceToDevice, st));
  if (difficult) CUDA_TRY(cudaMemcpyAsync(difficult, e->ring.difficult.get(), n, cudaMemcpyDeviceToDevice, st));
  return DRL_OK;
}

extern "C" int drl_get_running_rsi_positions(DrlEnv* e, int32_t* rsi_pos, void* stream) {
  int rc = ready(e, "drl_get_running_rsi_positions");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  if (!rsi_pos) return fail(DRL_ERR_INVALID, "drl_get_running_rsi_positions: null tensor");
  CUDA_TRY(launch_running_rsi(e->st.state_i.get(), rsi_pos, e->cfg.num_envs, (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_get_median_torque(DrlEnv* e, float* out, void* stream) {
  int rc = ready(e, "drl_get_median_torque");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  if (!out) return fail(DRL_ERR_INVALID, "drl_get_median_torque: null tensor");
  if (!e->st.med_tor_sm.get()) return fail(DRL_ERR_STATE, "drl_get_median_torque: the env was created with monitor_median_torque = 0");
  CUDA_TRY(cudaMemcpyAsync(out, e->st.med_tor_sm.get(), (size_t)e->cfg.num_envs * sizeof(float), cudaMemcpyDeviceToDevice,
                           (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_get_ee_reward(DrlEnv* e, float* last, float* smoothed, void* stream) {
  int rc = ready(e, "drl_get_ee_reward");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  const float* ee_f = e->st.ee_f.get();
  if (!ee_f) return fail(DRL_ERR_STATE, "drl_get_ee_reward: the env was created with ee_weight = 0");
  const size_t n = (size_t)e->cfg.num_envs;
  cudaStream_t st = (cudaStream_t)stream;
  // columns of the [N][2] rows
  if (last)
    CUDA_TRY(cudaMemcpy2DAsync(last, sizeof(float), ee_f, 2 * sizeof(float), sizeof(float), n,
                               cudaMemcpyDeviceToDevice, st));
  if (smoothed)
    CUDA_TRY(cudaMemcpy2DAsync(smoothed, sizeof(float), ee_f + 1, 2 * sizeof(float), sizeof(float), n,
                               cudaMemcpyDeviceToDevice, st));
  return DRL_OK;
}

extern "C" int drl_set_eval_mode(DrlEnv* e, int32_t on) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_set_eval_mode: null env");
  e->eval_mode = on ? 1 : 0;
  return DRL_OK;
}

extern "C" int drl_set_det_init_counters(DrlEnv* e, const int32_t* counts) {
  if (!e || !counts) return fail(DRL_ERR_INVALID, "drl_set_det_init_counters: null argument");
  if (!e->have_model) return fail(DRL_ERR_STATE, "drl_set_det_init_counters: upload the model first");
  const int n = e->cfg.num_envs;
  for (int i = 0; i < n; i++)
    if (counts[i] < 0 || counts[i] >= (e->cfg.eval_n_times > 0 ? e->cfg.eval_n_times : 1))
      return fail(DRL_ERR_INVALID, "drl_set_det_init_counters: counts[%d] = %d outside [0, eval_n_times)", i, counts[i]);
  DeviceGuard guard__(e->cfg.device);
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpy2D(e->st.state_i.get() + kCurNDet, kCurCount8 * sizeof(int), counts, sizeof(int), sizeof(int), (size_t)n,
                        cudaMemcpyHostToDevice));
  return DRL_OK;
}

extern "C" int drl_set_seed(DrlEnv* e, uint64_t seed) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_set_seed: null env");
  if (!e->have_model) return fail(DRL_ERR_STATE, "drl_set_seed: upload the model first");
  DeviceGuard guard__(e->cfg.device);
  DevModel d = e->hm;
  d.seed = seed;
  const int rc = publish_model(e, d);
  if (rc == DRL_OK) e->cfg.seed = seed;
  return rc;
}

extern "C" int drl_set_actuation(DrlEnv* e, int32_t mode, const double* kp, const double* kv) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_set_actuation: null env");
  if (mode != DRL_ACTUATION_TORQUE && mode != DRL_ACTUATION_PD)
    return fail(DRL_ERR_INVALID, "drl_set_actuation: unknown mode %d", mode);
  if (!e->have_model) return fail(DRL_ERR_STATE, "drl_set_actuation: upload the model first");
  DevModel d = e->hm;
  if (mode == DRL_ACTUATION_PD) {
    if (!kp || !kv) return fail(DRL_ERR_INVALID, "drl_set_actuation: PD needs kp and kv");
    for (int u = 0; u < d.nu; u++) {
      if (!(isfinite(kp[u]) && kp[u] > 0.0))
        return fail(DRL_ERR_INVALID, "drl_set_actuation: kp[%d] = %g must be finite and > 0", u, kp[u]);
      if (!(isfinite(kv[u]) && kv[u] >= 0.0))
        return fail(DRL_ERR_INVALID, "drl_set_actuation: kv[%d] = %g must be finite and >= 0", u, kv[u]);
      const int j = d.act_dof[u];
      if (!d.dof_limited[j] || !(e->dof_range[j][1] > e->dof_range[j][0]))
        return fail(DRL_ERR_INVALID, "drl_set_actuation: actuator %d drives dof %d, which has no joint range", u, j);
    }
  }
  // the gains and the target map are rewritten in full: switching back to torque leaves the block as after the upload
  memset(d.pd_kp, 0, sizeof d.pd_kp); memset(d.pd_kv, 0, sizeof d.pd_kv); memset(d.pd_gear, 0, sizeof d.pd_gear);
  memset(d.pd_flo, 0, sizeof d.pd_flo); memset(d.pd_fhi, 0, sizeof d.pd_fhi);
  memset(d.pd_mid, 0, sizeof d.pd_mid); memset(d.pd_half, 0, sizeof d.pd_half);
  if (mode == DRL_ACTUATION_PD) {
    for (int u = 0; u < d.nu; u++) {
      const int j = d.act_dof[u];
      d.pd_kp[j] = (float)kp[u]; d.pd_kv[j] = (float)kv[u]; d.pd_gear[j] = d.act_gear[u];
      d.pd_flo[j] = d.act_flo[u]; d.pd_fhi[j] = d.act_fhi[u];
      const double lo = e->dof_range[j][0], hi = e->dof_range[j][1];
      d.pd_mid[u] = (float)(0.5 * (lo + hi));
      d.pd_half[u] = (float)(0.5 * (hi - lo));
    }
  }
  DeviceGuard guard__(e->cfg.device);
  const int rc = publish_model(e, d);
  if (rc == DRL_OK) e->actuation = mode;
  return rc;
}

extern "C" int drl_set_contact_termination(DrlEnv* e, uint32_t body_mask) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_set_contact_termination: null env");
  if (!e->have_model) return fail(DRL_ERR_STATE, "drl_set_contact_termination: upload the model first");
  DevModel d = e->hm;
  if (body_mask >> d.nb) return fail(DRL_ERR_INVALID, "drl_set_contact_termination: mask 0x%x names a body >= nb = %d",
                                     body_mask, d.nb);
  // the reset puts the lowest foot-corner site on the floor: a body that carries one would end every episode at once
  for (int s = 0; s < d.nsite; s++)
    if ((body_mask >> d.site_body[s]) & 1u)
      return fail(DRL_ERR_INVALID, "drl_set_contact_termination: body %d carries a foot-corner site", d.site_body[s]);
  DeviceGuard guard__(e->cfg.device);
  DevBuf<int> counts;
  if (body_mask && !e->contact_et.get()) CUDA_TRY(counts.zeros((size_t)e->cfg.num_envs));
  d.et_contact_mask = body_mask;
  const int rc = publish_model(e, d);
  if (rc == DRL_OK && counts.get()) e->contact_et = std::move(counts);
  return rc;
}

extern "C" int drl_get_contact_terminations(DrlEnv* e, int32_t* out, void* stream) {
  if (!e || !out) return fail(DRL_ERR_INVALID, "drl_get_contact_terminations: null argument");
  if (!e->contact_et.get())
    return fail(DRL_ERR_STATE, "drl_get_contact_terminations: contact termination was never enabled on this env");
  DeviceGuard guard__(e->cfg.device);
  CUDA_TRY(cudaMemcpyAsync(out, e->contact_et.get(), (size_t)e->cfg.num_envs * sizeof(int32_t), cudaMemcpyDeviceToDevice,
                           (cudaStream_t)stream));
  return DRL_OK;
}

// the bin layout of the failure-weighted RSI table for the current mocap: bins of at most bin_samples consecutive samples
// inside each mocap step, in step order.  Fills bins ([n_bins][3] step, first, width, then [n_steps] first bin of each
// step) and u (the probability of each bin under the reference's uniform draw).
static void ars_layout(const std::vector<int>& step_len, const std::vector<int>& clip_first,
                       const std::vector<double>& clip_weight, int bin_samples, std::vector<int>& bins,
                       std::vector<double>& u) {
  bins.clear(); u.clear();
  std::vector<int> first_bin;
  size_t k = 0;                               // clip of step s: a step of clip k is drawn with weight_k / steps_k
  double inv_steps = 0.0;
  for (size_t s = 0; s < step_len.size(); s++) {
    if (s == 0 || (int)s == clip_first[k + 1]) {
      if (s != 0) k++;
      inv_steps = clip_weight[k] / (double)(clip_first[k + 1] - clip_first[k]);
    }
    first_bin.push_back((int)u.size());
    for (int p = 0; p < step_len[s]; p += bin_samples) {
      const int w = step_len[s] - p < bin_samples ? step_len[s] - p : bin_samples;
      bins.push_back((int)s); bins.push_back(p); bins.push_back(w);
      u.push_back(inv_steps * (double)w / (double)step_len[s]);
    }
  }
  bins.insert(bins.end(), first_bin.begin(), first_bin.end());
}

extern "C" int drl_set_adaptive_rsi(DrlEnv* e, float lambda, int32_t halflife_steps, int32_t bin_samples) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_set_adaptive_rsi: null env");
  if (!(lambda >= 0.f && lambda <= 1.f))
    return fail(DRL_ERR_INVALID, "drl_set_adaptive_rsi: lambda = %g outside [0, 1]", (double)lambda);
  if (halflife_steps <= 0) return fail(DRL_ERR_INVALID, "drl_set_adaptive_rsi: halflife_steps must be > 0");
  if (bin_samples <= 0) return fail(DRL_ERR_INVALID, "drl_set_adaptive_rsi: bin_samples must be > 0");
  if (!e->have_model || !e->have_mocap)
    return fail(DRL_ERR_STATE, "drl_set_adaptive_rsi: model and mocap must be uploaded first");
  DeviceGuard guard__(e->cfg.device);
  CUDA_TRY(cudaDeviceSynchronize());          // enqueued steps may still read the tables
  if (lambda > 0.f && (e->ars.gen != e->mocap_gen || e->ars.bin_samples != bin_samples)) {
    // first enable for this mocap and bin width: a new, empty table; every running episode is uncounted
    std::vector<int> bins;
    std::vector<double> u;
    ars_layout(e->mocap.step_len_h, e->clips.first_h, e->clips.weight_h, bin_samples, bins, u);
    const size_t nb = u.size(), N = (size_t)e->cfg.num_envs;
    ArsBufs t;
    t.gen = e->mocap_gen; t.bin_samples = bin_samples;
    CUDA_TRY(t.counts.zeros(2 * nb));
    CUDA_TRY(t.u.from_host(u.data(), nb));
    CUDA_TRY(t.cdf.alloc(nb));
    CUDA_TRY(t.prob.alloc(nb));
    CUDA_TRY(t.bins.from_host(bins.data(), bins.size()));
    CUDA_TRY(t.inc.zeros(2 * nb));
    CUDA_TRY(t.env_bin.alloc(N));
    CUDA_TRY(cudaMemset(t.env_bin.get(), 0xFF, N * sizeof(int)));
    e->ars = std::move(t);
  }
  e->ars_lambda = lambda;
  e->ars_halflife = halflife_steps;
  if (e->ars.counts.get()) {                  // rebuild the sampling tables (and prob, which depends on lambda)
    CUDA_TRY(launch_adaptive_rsi_update(ars_args(e, 1.0), nullptr));
    CUDA_TRY(cudaDeviceSynchronize());
  }
  return DRL_OK;
}

extern "C" int drl_get_adaptive_rsi(DrlEnv* e, double* started, double* difficult, double* prob, int32_t* env_bin,
                                    void* stream) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_get_adaptive_rsi: null env");
  const double* counts = e->ars.counts.get();
  if (!counts) return fail(DRL_ERR_STATE, "drl_get_adaptive_rsi: failure-weighted RSI was never enabled");
  DeviceGuard guard__(e->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  const size_t nb = (size_t)e->ars.n_bins();
  if (started) CUDA_TRY(cudaMemcpyAsync(started, counts, nb * sizeof(double), cudaMemcpyDeviceToDevice, st));
  if (difficult) CUDA_TRY(cudaMemcpyAsync(difficult, counts + nb, nb * sizeof(double), cudaMemcpyDeviceToDevice, st));
  if (prob) CUDA_TRY(cudaMemcpyAsync(prob, e->ars.prob.get(), nb * sizeof(double), cudaMemcpyDeviceToDevice, st));
  if (env_bin)
    CUDA_TRY(cudaMemcpyAsync(env_bin, e->ars.env_bin.get(), (size_t)e->cfg.num_envs * sizeof(int),
                             cudaMemcpyDeviceToDevice, st));
  return DRL_OK;
}

extern "C" int drl_set_adaptive_rsi_counts(DrlEnv* e, const double* started, const double* difficult) {
  if (!e || !started || !difficult) return fail(DRL_ERR_INVALID, "drl_set_adaptive_rsi_counts: null argument");
  double* counts = e->ars.counts.get();
  if (!counts) return fail(DRL_ERR_STATE, "drl_set_adaptive_rsi_counts: failure-weighted RSI was never enabled");
  const int nb = e->ars.n_bins();
  for (int b = 0; b < nb; b++)
    if (!(isfinite(started[b]) && difficult[b] >= 0.0 && difficult[b] <= started[b]))
      return fail(DRL_ERR_INVALID, "drl_set_adaptive_rsi_counts: bin %d: need 0 <= difficult <= started < inf", b);
  DeviceGuard guard__(e->cfg.device);
  CUDA_TRY(cudaDeviceSynchronize());          // enqueued steps may still read the tables
  CUDA_TRY(cudaMemcpy(counts, started, nb * sizeof(double), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(counts + nb, difficult, nb * sizeof(double), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemset(e->ars.inc.get(), 0, 2 * (size_t)nb * sizeof(unsigned)));
  CUDA_TRY(launch_adaptive_rsi_update(ars_args(e, 1.0), nullptr));
  CUDA_TRY(cudaDeviceSynchronize());
  return DRL_OK;
}

extern "C" int drl_set_playback(DrlEnv* e, int32_t on) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_set_playback: null env");
  e->playback = on ? 1 : 0;
  return DRL_OK;
}

extern "C" int drl_set_ref_obs(DrlEnv* e, int32_t n, const int32_t* offsets) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_set_ref_obs: null env");
  if (!e->have_model) return fail(DRL_ERR_STATE, "drl_set_ref_obs: upload the model first");
  if (e->stepped) return fail(DRL_ERR_STATE, "drl_set_ref_obs: the env has been reset or stepped (the row width is fixed)");
  if (e->vn_packed) return fail(DRL_ERR_STATE, "drl_set_ref_obs: a VecNormalize is attached (its moments have the old width)");
  if (n < 0 || n > DRL_MAX_REF_OBS) return fail(DRL_ERR_INVALID, "drl_set_ref_obs: n = %d outside [0, %d]", n, DRL_MAX_REF_OBS);
  if (n > 0 && !offsets) return fail(DRL_ERR_INVALID, "drl_set_ref_obs: null offsets");
  unsigned packed = (unsigned)n;
  for (int f = 0; f < n; f++) {
    if (offsets[f] < 1 || offsets[f] > 256)
      return fail(DRL_ERR_INVALID, "drl_set_ref_obs: offsets[%d] = %d outside [1, 256]", f, offsets[f]);
    if (f > 0 && offsets[f] <= offsets[f - 1])
      return fail(DRL_ERR_INVALID, "drl_set_ref_obs: the offsets must be strictly increasing");
    packed |= (unsigned)(offsets[f] - 1) << (8 * f + 8);
  }
  DevModel d = e->hm;
  const int nq = d.nv - 1, B = d.n_phase_obs + d.n_des_vel;
  if (d.mirror_policy)      // a frame is mirrored through the qpos-block part of the table: it must stay in the block
    for (int k = B; k < B + nq; k++)
      if (d.mirror_obs_idx[k] < B || d.mirror_obs_idx[k] >= B + nq)
        return fail(DRL_ERR_INVALID, "drl_set_ref_obs: mirror_obs_idx[%d] = %d leaves the qpos block [%d, %d)", k,
                    d.mirror_obs_idx[k], B, B + nq);
  const int row = d.obs_dim + n * nq;
  if (row > DRL_MAX_OBS_TOTAL) return fail(DRL_ERR_INVALID, "drl_set_ref_obs: row of %d floats > %d", row, DRL_MAX_OBS_TOTAL);
  DeviceGuard guard__(e->cfg.device);
  DevBuf<double> rows;
  CUDA_TRY(alloc_cta_rows(e, (size_t)e->cfg.num_envs, row, rows));
  d.obs_row = row;
  if (const int rc = publish_model(e, d)) return rc;   // synchronises: no step reads the old rows any more
  e->st.cta_rows = std::move(rows);
  e->ref_obs = n > 0 ? packed : 0u;
  return DRL_OK;
}

extern "C" int drl_set_speed_profile(DrlEnv* e, const float* speeds, int32_t n) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_set_speed_profile: null env");
  if (n < 0 || (n > 0 && !speeds)) return fail(DRL_ERR_INVALID, "drl_set_speed_profile: n=%d with %s table", n,
                                               speeds ? "a" : "a null");
  DeviceGuard guard__(e->cfg.device);
  DevBuf<float> table;
  if (n > 0) CUDA_TRY(table.from_host(speeds, (size_t)n));
  CUDA_TRY(cudaDeviceSynchronize());   // the previous table may still be read by enqueued steps
  e->speed_profile = std::move(table);
  return DRL_OK;
}

extern "C" int drl_launch_info(DrlEnv* e, int32_t* lanes_per_env, int32_t* block_threads, int32_t* grid_blocks,
                               int32_t* smem_bytes) {
  if (!e || !e->have_model) return fail(DRL_ERR_STATE, "drl_launch_info: upload the model first");
  const int epb = e->block / e->G;
  if (lanes_per_env) *lanes_per_env = e->G;
  if (block_threads) *block_threads = e->block;
  if (grid_blocks) *grid_blocks = (e->cfg.num_envs + epb - 1) / epb;
  if (smem_bytes) *smem_bytes = (int)step_smem_bytes(e->G, epb, e->actuation == DRL_ACTUATION_PD);
  return DRL_OK;
}

// ---- test / tuning hooks (declared in include/drloco_b200.h under "debug") ----
extern "C" int drl_debug_set(DrlEnv* e, int32_t frame_skip_override, int32_t block_threads, int32_t enable_dump) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_debug_set: null env");
  if (block_threads > 0 && (block_threads % 32 != 0 || block_threads > 128))
    return fail(DRL_ERR_INVALID, "drl_debug_set: block size must be 32, 64, 96 or 128");
  DeviceGuard guard__(e->cfg.device);
  if (enable_dump && !e->debug.get()) {
    DevBuf<float> dump;
    CUDA_TRY(dump.zeros((size_t)e->cfg.num_envs * 32 * 40));
    e->debug = std::move(dump);
  } else if (!enable_dump) {
    e->debug = DevBuf<float>();
  }
  e->frame_skip_override = frame_skip_override;
  if (block_threads > 0) e->block = block_threads;
  return DRL_OK;
}

extern "C" int drl_debug_read(DrlEnv* e, float* host_out, int32_t n_floats) {
  if (!e || !e->debug.get()) return fail(DRL_ERR_STATE, "drl_debug_read: dump not enabled");
  CUDA_TRY(cudaMemcpy(host_out, e->debug.get(), (size_t)n_floats * sizeof(float), cudaMemcpyDeviceToHost));
  return DRL_OK;
}
