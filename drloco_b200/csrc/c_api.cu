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
#include "dev_model.h"

namespace drl {
size_t step_smem_bytes(int G, int envs_per_block);
cudaError_t launch_step(const StepArgs& a, int nv, int G, int rk4, int reset_only, int block, bool debug,
                        cudaStream_t st);
cudaError_t launch_running_rsi(const int* state_i, int* out, int n, cudaStream_t st);
bool topology_matches(int nv, int nb, const int* body_parent, const int* dof_body, const int* dof_type);
cudaError_t launch_extras(const float* state_f, const float* last, float* out, int n, int G, cudaStream_t st);
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

struct DrlEnv {
  DrlConfig cfg;
  DevModel hm;                 // host copy
  bool have_model = false, have_mocap = false;
  int G = 16, block = 128, nv = 0;
  DevModel* d_model = nullptr;
  float* state_f = nullptr;
  int* state_i = nullptr;
  int* state_as = nullptr;
  double* state_d = nullptr;
  float* extras_last = nullptr;
  double* stats = nullptr;
  float *ref = nullptr, *step_vel = nullptr, *step_last_comx = nullptr;
  double* des_vel_prefix = nullptr;   // float64: differences of long prefix sums lose ~1e-5 in float32
  int *step_off = nullptr, *step_len = nullptr;
  unsigned char* left_step = nullptr;
  int* ring_len = nullptr;
  float* ring_ret = nullptr;
  int *ring_rsi_pos = nullptr, *ring_et_pos = nullptr;
  unsigned char* ring_difficult = nullptr;
  unsigned long long* ring_head = nullptr;
  int ring_cap = 1 << 16;
  int eval_mode = 0;
  float* speed_profile = nullptr;
  int speed_profile_len = 0;
  int playback = 0;
  int frame_skip_override = -1;
  float* debug = nullptr;
  float* tor_hist = nullptr;
  float* med_tor_sm = nullptr;
  // end-effector term (cfg.ee_weight > 0): last / smoothed ee_rew, lifetime sum
  float* ee_f = nullptr;
  double* ee_d = nullptr;
  // per-step statistics rows (one per thread block of the step kernel) + the ticket that elects the summing block
  double* cta_rows = nullptr;
  unsigned* cta_ticket = nullptr;
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

// the buffers of alloc_state; drl_destroy frees the rest
static void free_state(DrlEnv* e) {
  void** ptrs[] = {(void**)&e->d_model, (void**)&e->state_f, (void**)&e->state_i, (void**)&e->state_as,
                   (void**)&e->state_d, (void**)&e->extras_last, (void**)&e->stats, (void**)&e->ring_len,
                   (void**)&e->ring_ret, (void**)&e->ring_head, (void**)&e->ring_rsi_pos, (void**)&e->ring_et_pos,
                   (void**)&e->ring_difficult, (void**)&e->cta_rows, (void**)&e->cta_ticket,
                   (void**)&e->tor_hist, (void**)&e->med_tor_sm, (void**)&e->ee_f, (void**)&e->ee_d};
  for (void** p : ptrs) {
    if (*p) cudaFree(*p);
    *p = nullptr;
  }
}

extern "C" int drl_destroy(DrlEnv* e) {
  if (!e) return DRL_OK;
  DeviceGuard guard__(e->cfg.device);
  free_state(e);
  // mocap tables, speed profile, debug dump
  void* ptrs[] = {e->ref, e->step_off, e->step_len, e->left_step, e->step_vel, e->step_last_comx, e->des_vel_prefix,
                  e->speed_profile, e->debug};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  delete e;
  return DRL_OK;
}

// persistent per-env state; on failure the caller releases whatever was allocated (free_state)
static int alloc_state(DrlEnv* e, size_t N) {
  CUDA_TRY(cudaMalloc(&e->d_model, sizeof(DevModel)));
  CUDA_TRY(cudaMalloc(&e->state_f, N * 4 * e->G * sizeof(float)));
  CUDA_TRY(cudaMalloc(&e->state_i, N * kCurCount8 * sizeof(int)));
  CUDA_TRY(cudaMalloc(&e->state_as, N * e->G * sizeof(int)));
  CUDA_TRY(cudaMemset(e->state_as, 0, N * e->G * sizeof(int)));
  CUDA_TRY(cudaMalloc(&e->state_d, N * 4 * sizeof(double)));
  CUDA_TRY(cudaMalloc(&e->extras_last, N * 16 * sizeof(float)));
  CUDA_TRY(cudaMalloc(&e->stats, DRL_STATS_COUNT * sizeof(double)));
  CUDA_TRY(cudaMalloc(&e->ring_len, e->ring_cap * sizeof(int)));
  CUDA_TRY(cudaMalloc(&e->ring_ret, e->ring_cap * sizeof(float)));
  CUDA_TRY(cudaMalloc(&e->ring_rsi_pos, e->ring_cap * sizeof(int)));
  CUDA_TRY(cudaMalloc(&e->ring_et_pos, e->ring_cap * sizeof(int)));
  CUDA_TRY(cudaMalloc(&e->ring_difficult, e->ring_cap));
  CUDA_TRY(cudaMalloc(&e->ring_head, sizeof(unsigned long long)));
  if (e->cfg.monitor_median_torque) {
    const size_t cap = (size_t)(e->cfg.ep_dur_max > 0 ? e->cfg.ep_dur_max : 1);
    CUDA_TRY(cudaMalloc(&e->tor_hist, N * cap * sizeof(float)));
    CUDA_TRY(cudaMemset(e->tor_hist, 0, N * cap * sizeof(float)));
    CUDA_TRY(cudaMalloc(&e->med_tor_sm, N * sizeof(float)));
    CUDA_TRY(cudaMemset(e->med_tor_sm, 0, N * sizeof(float)));
  }
  if (e->cfg.ee_weight > 0.0) {
    CUDA_TRY(cudaMalloc(&e->ee_f, N * 2 * sizeof(float)));
    CUDA_TRY(cudaMemset(e->ee_f, 0, N * 2 * sizeof(float)));
    CUDA_TRY(cudaMalloc(&e->ee_d, N * sizeof(double)));
    CUDA_TRY(cudaMemset(e->ee_d, 0, N * sizeof(double)));
  }
  {
    // the smallest CTA the library launches carries 32 / G environments
    const size_t max_blocks = (N + (32 / e->G) - 1) / (32 / e->G);
    const size_t row = 2 * (size_t)e->cfg.obs_dim + 2 + DRL_STATS_COUNT;
    // rows of the blocks, then one row per group of kStatGroup blocks (two-level fixed-order sum in the step kernel);
    // tickets: [0] counts finished groups, [1 + g] the finished blocks of group g
    const size_t max_groups = (max_blocks + kStatGroup - 1) / kStatGroup;
    CUDA_TRY(cudaMalloc(&e->cta_rows, (max_blocks + max_groups) * row * sizeof(double)));
    CUDA_TRY(cudaMalloc(&e->cta_ticket, (1 + max_groups) * sizeof(unsigned)));
    CUDA_TRY(cudaMemset(e->cta_ticket, 0, (1 + max_groups) * sizeof(unsigned)));
  }
  CUDA_TRY(cudaMemset(e->state_f, 0, N * 4 * e->G * sizeof(float)));
  CUDA_TRY(cudaMemset(e->state_i, 0, N * kCurCount8 * sizeof(int)));
  CUDA_TRY(cudaMemset(e->state_d, 0, N * 4 * sizeof(double)));
  CUDA_TRY(cudaMemset(e->extras_last, 0, N * 16 * sizeof(float)));
  CUDA_TRY(cudaMemset(e->stats, 0, DRL_STATS_COUNT * sizeof(double)));
  CUDA_TRY(cudaMemset(e->ring_head, 0, sizeof(unsigned long long)));
  // count_steps_same_vel starts at 1 (straight_walk_trajecs.py:124)
  std::vector<int> init(N * kCurCount8, 0);
  for (size_t i = 0; i < N; i++) init[i * kCurCount8 + kCurCount] = 1;
  CUDA_TRY(cudaMemcpy(e->state_i, init.data(), init.size() * sizeof(int), cudaMemcpyHostToDevice));
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
    free_state(e);
    (void)cudaGetLastError();     // a failed cudaMalloc also parks its code as the "last error": clear it
    return rc;
  }
  e->have_model = true;
  if (e->have_mocap) CUDA_TRY(cudaMemcpy(e->d_model, &e->hm, sizeof(DevModel), cudaMemcpyHostToDevice));
  return DRL_OK;
}

template <typename T, typename S>
static int upload(T** dst, const S* src, size_t n) {
  std::vector<T> tmp(n);
  for (size_t i = 0; i < n; i++) tmp[i] = (T)src[i];
  if (*dst) cudaFree(*dst);
  if (cudaMalloc(dst, n * sizeof(T)) != cudaSuccess) return -1;
  if (cudaMemcpy(*dst, tmp.data(), n * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) return -1;
  return 0;
}

extern "C" int drl_upload_mocap(DrlEnv* e, int32_t cursor_mode, int32_t increment, const double* ref, int32_t n_samples,
                                const int32_t* step_off, const int32_t* step_len, const uint8_t* left_step,
                                const double* step_vel, const double* step_last_comx, int32_t n_steps,
                                int32_t com_z_col, const double* des_vel_prefix, int32_t des_vel_window) {
  if (!e || !ref || !step_off || !step_len || !left_step || !step_vel || !step_last_comx)
    return fail(DRL_ERR_INVALID, "drl_upload_mocap: null argument");
  if (!e->have_model) return fail(DRL_ERR_STATE, "drl_upload_mocap: upload the model first");
  if (n_samples <= 0 || n_steps <= 0 || increment <= 0) return fail(DRL_ERR_INVALID, "drl_upload_mocap: empty mocap");
  if (cursor_mode != DRL_CURSOR_STEPWISE && cursor_mode != DRL_CURSOR_WRAP)
    return fail(DRL_ERR_INVALID, "drl_upload_mocap: unknown cursor mode");
  if (cursor_mode == DRL_CURSOR_WRAP && (n_steps != 1 || !des_vel_prefix))
    return fail(DRL_ERR_INVALID, "drl_upload_mocap: wrap mode needs one step and the desired-velocity prefix sums");
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
  if (upload(&e->ref, padded.data(), padded.size())) return fail(DRL_ERR_CUDA, "drl_upload_mocap: device copy failed");
  if (upload(&e->step_off, step_off, n_steps) || upload(&e->step_len, step_len, n_steps) ||
      upload(&e->left_step, left_step, n_steps) || upload(&e->step_vel, step_vel, n_steps) ||
      upload(&e->step_last_comx, step_last_comx, n_steps))
    return fail(DRL_ERR_CUDA, "drl_upload_mocap: device copy failed");
  if (des_vel_prefix) {
    if (upload(&e->des_vel_prefix, des_vel_prefix, (size_t)(n_samples + 1) * 2))
      return fail(DRL_ERR_CUDA, "drl_upload_mocap: device copy failed");
  }
  DevModel& d = e->hm;
  d.cursor_mode = cursor_mode; d.increment = increment; d.n_steps = n_steps; d.n_samples = n_samples;
  d.com_z_col = com_z_col; d.des_vel_window = des_vel_window;
  CUDA_TRY(cudaMemcpy(e->d_model, &e->hm, sizeof(DevModel), cudaMemcpyHostToDevice));
  e->have_mocap = true;
  return DRL_OK;
}

static int ready(DrlEnv* e, const char* who) {
  if (!e) return fail(DRL_ERR_INVALID, "%s: null env", who);
  if (!e->have_model || !e->have_mocap) return fail(DRL_ERR_STATE, "%s: model and mocap must be uploaded first", who);
  return DRL_OK;
}

static StepArgs make_args(DrlEnv* e) {
  StepArgs a;
  memset(&a, 0, sizeof a);
  a.model = e->d_model; a.num_envs = e->cfg.num_envs;
  a.frame_skip = e->frame_skip_override >= 0 ? e->frame_skip_override : e->cfg.frame_skip;
  a.state_f = e->state_f; a.state_i = e->state_i; a.state_as = e->state_as; a.state_d = e->state_d;
  a.ref = e->ref; a.step_off = e->step_off; a.step_len = e->step_len; a.left_step = e->left_step;
  a.step_vel = e->step_vel; a.step_last_comx = e->step_last_comx; a.des_vel_prefix = e->des_vel_prefix;
  a.extras = e->extras_last; a.stats = e->stats;
  a.ring_len = e->ring_len; a.ring_ret = e->ring_ret; a.ring_head = e->ring_head; a.ring_cap = e->ring_cap;
  a.ring_rsi_pos = e->ring_rsi_pos; a.ring_et_pos = e->ring_et_pos; a.ring_difficult = e->ring_difficult;
  a.eval_mode = e->eval_mode;
  a.speed_profile = e->speed_profile_len > 0 ? e->speed_profile : nullptr;
  a.speed_profile_len = e->speed_profile_len;
  a.playback = e->playback;
  a.cta_rows = e->cta_rows; a.cta_ticket = e->cta_ticket;
  a.tor_hist = e->tor_hist; a.med_tor_sm = e->med_tor_sm;
  a.ee_f = e->ee_f; a.ee_d = e->ee_d;
  a.vn_ret = e->vn_ret; a.vn_gamma = e->vn_gamma; a.packed = e->vn_packed;
  if (e->playback) a.frame_skip = 0;
  a.debug = e->debug;
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
  CUDA_TRY(launch_step(a, e->nv, e->G, e->cfg.integrator == DRL_INTEGRATOR_RK4, 1, e->block, false, (cudaStream_t)stream));
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
    const bool rk4 = e->cfg.integrator == DRL_INTEGRATOR_RK4;
  if (e->debug && rk4) return fail(DRL_ERR_UNSUPPORTED, "drl_step: the dump variant exists for the Euler integrator only");
  CUDA_TRY(launch_step(a, e->nv, e->G, rk4, 0, e->block, e->debug != nullptr, (cudaStream_t)stream));
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
  CUDA_TRY(launch_state_copy(e->state_f, e->state_i, e->state_as, qpos, qvel, cursor, e->cfg.num_envs, e->nv, e->G, 0,
                             (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_set_state(DrlEnv* e, const float* qpos, const float* qvel, const int32_t* cursor, void* stream) {
  int rc = ready(e, "drl_set_state");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  CUDA_TRY(launch_state_copy(e->state_f, e->state_i, e->state_as, const_cast<float*>(qpos), const_cast<float*>(qvel),
                             const_cast<int32_t*>(cursor), e->cfg.num_envs, e->nv, e->G, 1, (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_get_extras(DrlEnv* e, float* extras, void* stream) {
  int rc = ready(e, "drl_get_extras");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  if (!extras) return fail(DRL_ERR_INVALID, "drl_get_extras: null tensor");
  CUDA_TRY(launch_extras(e->state_f, e->extras_last, extras, e->cfg.num_envs, e->G, (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_get_stats(DrlEnv* e, double* stats, void* stream) {
  int rc = ready(e, "drl_get_stats");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  if (!stats) return fail(DRL_ERR_INVALID, "drl_get_stats: null tensor");
  CUDA_TRY(cudaMemcpyAsync(stats, e->stats, DRL_STATS_COUNT * sizeof(double), cudaMemcpyDeviceToDevice,
                           (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_reset_stats(DrlEnv* e, void* stream) {
  int rc = ready(e, "drl_reset_stats");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  CUDA_TRY(cudaMemsetAsync(e->stats, 0, DRL_STATS_COUNT * sizeof(double), (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_get_episode_ring(DrlEnv* e, int32_t* ep_len, float* ep_ret, int32_t capacity,
                                    int64_t* total_episodes, void* stream) {
  int rc = ready(e, "drl_get_episode_ring");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  if (!total_episodes) return fail(DRL_ERR_INVALID, "drl_get_episode_ring: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long head = 0;
  CUDA_TRY(cudaMemcpyAsync(&head, e->ring_head, sizeof head, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));     // the count is returned to the host by value
  *total_episodes = (int64_t)head;
  const int n = capacity < e->ring_cap ? capacity : e->ring_cap;
  if (ep_len && n > 0) CUDA_TRY(cudaMemcpyAsync(ep_len, e->ring_len, n * sizeof(int), cudaMemcpyDeviceToDevice, st));
  if (ep_ret && n > 0) CUDA_TRY(cudaMemcpyAsync(ep_ret, e->ring_ret, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
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
  if (rsi_pos) CUDA_TRY(cudaMemcpyAsync(rsi_pos, e->ring_rsi_pos, n * sizeof(int), cudaMemcpyDeviceToDevice, st));
  if (et_pos) CUDA_TRY(cudaMemcpyAsync(et_pos, e->ring_et_pos, n * sizeof(int), cudaMemcpyDeviceToDevice, st));
  if (difficult) CUDA_TRY(cudaMemcpyAsync(difficult, e->ring_difficult, n, cudaMemcpyDeviceToDevice, st));
  return DRL_OK;
}

extern "C" int drl_get_running_rsi_positions(DrlEnv* e, int32_t* rsi_pos, void* stream) {
  int rc = ready(e, "drl_get_running_rsi_positions");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  if (!rsi_pos) return fail(DRL_ERR_INVALID, "drl_get_running_rsi_positions: null tensor");
  CUDA_TRY(launch_running_rsi(e->state_i, rsi_pos, e->cfg.num_envs, (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_get_median_torque(DrlEnv* e, float* out, void* stream) {
  int rc = ready(e, "drl_get_median_torque");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  if (!out) return fail(DRL_ERR_INVALID, "drl_get_median_torque: null tensor");
  if (!e->med_tor_sm) return fail(DRL_ERR_STATE, "drl_get_median_torque: the env was created with monitor_median_torque = 0");
  CUDA_TRY(cudaMemcpyAsync(out, e->med_tor_sm, (size_t)e->cfg.num_envs * sizeof(float), cudaMemcpyDeviceToDevice,
                           (cudaStream_t)stream));
  return DRL_OK;
}

extern "C" int drl_get_ee_reward(DrlEnv* e, float* last, float* smoothed, void* stream) {
  int rc = ready(e, "drl_get_ee_reward");
  if (rc) return rc;
  DeviceGuard guard__(e->cfg.device);
  if (!e->ee_f) return fail(DRL_ERR_STATE, "drl_get_ee_reward: the env was created with ee_weight = 0");
  const size_t n = (size_t)e->cfg.num_envs;
  cudaStream_t st = (cudaStream_t)stream;
  // columns of the [N][2] rows
  if (last)
    CUDA_TRY(cudaMemcpy2DAsync(last, sizeof(float), e->ee_f, 2 * sizeof(float), sizeof(float), n,
                               cudaMemcpyDeviceToDevice, st));
  if (smoothed)
    CUDA_TRY(cudaMemcpy2DAsync(smoothed, sizeof(float), e->ee_f + 1, 2 * sizeof(float), sizeof(float), n,
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
  CUDA_TRY(cudaMemcpy2D(e->state_i + kCurNDet, kCurCount8 * sizeof(int), counts, sizeof(int), sizeof(int), (size_t)n,
                        cudaMemcpyHostToDevice));
  return DRL_OK;
}

extern "C" int drl_set_seed(DrlEnv* e, uint64_t seed) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_set_seed: null env");
  if (!e->have_model) return fail(DRL_ERR_STATE, "drl_set_seed: upload the model first");
  e->cfg.seed = seed;
  e->hm.seed = seed;
  DeviceGuard guard__(e->cfg.device);
  CUDA_TRY(cudaDeviceSynchronize());          // enqueued steps may still read the model block
  CUDA_TRY(cudaMemcpy(e->d_model, &e->hm, sizeof(DevModel), cudaMemcpyHostToDevice));
  return DRL_OK;
}

extern "C" int drl_set_playback(DrlEnv* e, int32_t on) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_set_playback: null env");
  e->playback = on ? 1 : 0;
  return DRL_OK;
}

extern "C" int drl_set_speed_profile(DrlEnv* e, const float* speeds, int32_t n) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_set_speed_profile: null env");
  if (n < 0 || (n > 0 && !speeds)) return fail(DRL_ERR_INVALID, "drl_set_speed_profile: n=%d with %s table", n,
                                               speeds ? "a" : "a null");
  DeviceGuard guard__(e->cfg.device);
  CUDA_TRY(cudaDeviceSynchronize());   // the previous table may still be read by enqueued steps
  if (e->speed_profile) CUDA_TRY(cudaFree(e->speed_profile));
  e->speed_profile = nullptr;
  e->speed_profile_len = 0;
  if (n > 0) {
    CUDA_TRY(cudaMalloc(&e->speed_profile, (size_t)n * sizeof(float)));
    CUDA_TRY(cudaMemcpy(e->speed_profile, speeds, (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
    e->speed_profile_len = n;
  }
  return DRL_OK;
}

extern "C" int drl_launch_info(DrlEnv* e, int32_t* lanes_per_env, int32_t* block_threads, int32_t* grid_blocks,
                               int32_t* smem_bytes) {
  if (!e || !e->have_model) return fail(DRL_ERR_STATE, "drl_launch_info: upload the model first");
  const int epb = e->block / e->G;
  if (lanes_per_env) *lanes_per_env = e->G;
  if (block_threads) *block_threads = e->block;
  if (grid_blocks) *grid_blocks = (e->cfg.num_envs + epb - 1) / epb;
  if (smem_bytes) *smem_bytes = (int)step_smem_bytes(e->G, epb);
  return DRL_OK;
}

// ---- test / tuning hooks (declared in include/drloco_b200.h under "debug") ----
extern "C" int drl_debug_set(DrlEnv* e, int32_t frame_skip_override, int32_t block_threads, int32_t enable_dump) {
  if (!e) return fail(DRL_ERR_INVALID, "drl_debug_set: null env");
  e->frame_skip_override = frame_skip_override;
  if (block_threads > 0) {
    if (block_threads % 32 != 0 || block_threads > 128) return fail(DRL_ERR_INVALID, "drl_debug_set: block size must be 32, 64, 96 or 128");
    e->block = block_threads;
  }
  DeviceGuard guard__(e->cfg.device);
  if (enable_dump && !e->debug) {
    const size_t n = (size_t)e->cfg.num_envs * 32 * 40;
    CUDA_TRY(cudaMalloc(&e->debug, n * sizeof(float)));
    CUDA_TRY(cudaMemset(e->debug, 0, n * sizeof(float)));
  } else if (!enable_dump && e->debug) {
    cudaFree(e->debug);
    e->debug = nullptr;
  }
  return DRL_OK;
}

extern "C" int drl_debug_read(DrlEnv* e, float* host_out, int32_t n_floats) {
  if (!e || !e->debug) return fail(DRL_ERR_STATE, "drl_debug_read: dump not enabled");
  CUDA_TRY(cudaMemcpy(host_out, e->debug, (size_t)n_floats * sizeof(float), cudaMemcpyDeviceToHost));
  return DRL_OK;
}
