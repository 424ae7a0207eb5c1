// mimic_step.cu — the hot path of drloco_b200: one fused sm_100a kernel per VecEnv.step().
//
// Replaces, for N environments at once, the reference's per-process Python + MuJoCo stack:
//   MimicEnv.step                drloco/mujoco/mimic_env.py:60-126
//   MujocoEnv.do_simulation      frame_skip x mj_step with RK4 (xml:11), restated in oracle/walker_physics.c
//   StraightWalkingTrajectories.next / BaseReferenceTrajectories.next   straight_walk_trajecs.py:141-159, base:95-103
//   get_imitation_reward / _get_ET_reward / _get_obs / mirror_*          mimic_env.py:142-168,403-489,592-649
//   reset_model (RSI + ground-contact shift)                             mimic_env.py:526-572
//   Monitor.step statistics                                              monitor_wrapper.py:88-166
//   DummyVecEnv/SubprocVecEnv auto-reset with terminal_observation       (SB3 1.0)
//
// Mapping: one environment per group of G lanes (G = 16 for nv <= 16: two environments per warp; G = 32 otherwise),
// lane j owns dof j: its q/v/RK4 accumulators, its motion vector S_j and column j of the constraint Hessian live in
// registers for the whole launch; per-env tree quantities (body frames, spatial inertias, velocities, contact
// Hessians) live in shared memory and are produced by chain-ordered scans (fd_tree.cuh); all frame_skip x 4 dynamics
// evaluations run inside the launch, HBM is touched once on entry and once on exit.  Control flow is kept warp-uniform (the two environments of a warp run in lockstep, with
// predicated effects), so every shuffle / ballot / barrier uses the full-warp mask and compiles to a bare instruction.
// Spatial quantities are expressed in world orientation about O = the root body origin (keeps fp32 cancellation
// independent of how far the walker has travelled).
//
// Constraint solve per evaluation (same minimiser as MuJoCo's Newton solver, see oracle/walker_physics.c):
//   H = M + sum_b S_b^T W_b S_b + diag(limits),   H qacc = tau - c + sum_b S_b^T u_b + limits
// with W_b the 6x6 wrench-space Hessian of the active pyramid rows of all contacts on body b; primal active-set
// iteration with full Newton steps, warm-started from the previous evaluation; LDL^T in registers via shuffles.
#include "fd_common.cuh"
#include "fd_tree.cuh"

namespace drl {

// splitmix64 finaliser: counter-based generator for the RSI draws (stateless in (seed, env, reset#))
__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

struct Cursor {
  int i_step, pos, count, ep_dur, rsi_step, n_det, resets, flags;
};

// Deterministic initialisation (evaluation, straight:237-265) leaves the reference reading the table and the length
// of mocap step 0 (`reset()` aliases `_qpos_full = data[0]`, :161-167, and nothing re-points it) while `_i_step` and
// `_step` already name step n; the first step transition repairs it.  flags bit 2: still reading step 0's table;
// bit 3: the episode began with a deterministic init, so the in-place COM-Z shift went to step 0's table.
constexpr int kFlagReadStep0 = 4, kFlagDetEpisode = 8;
__device__ __forceinline__ int data_step(const Cursor& c) { return (c.flags & kFlagReadStep0) ? 0 : c.i_step; }
__device__ __forceinline__ int shift_step(const Cursor& c) { return (c.flags & kFlagDetEpisode) ? 0 : c.rsi_step; }

// mocap library (A.clips != null): first and last mocap step of the clip that holds step s
__device__ __forceinline__ int clip_bounds(const ClipLibrary* L, int s, int& last) {
  const int* first = L->clip_first;
  const int k = __ldg(L->step_clip + s);
  last = __ldg(first + k + 1) - 1;
  return __ldg(first + k);
}

// StraightWalkingTrajectories.next (straight:141-159, :322-348) / BaseReferenceTrajectories.next (base:95-103).
// Library: the reference's wrap rule applies per clip, so an episode stays in the clip it started in.
__device__ __forceinline__ void cursor_next(const DevModel& M, const StepArgs& A, Cursor& c, float& dist) {
  const int len = A.step_len[data_step(c)];
  c.pos += M.increment;
  if (M.cursor_mode == DRL_CURSOR_STEPWISE) {
    const int dif = c.pos - len + 1;
    if (dif > 0) {
      int first = 0, last = M.n_steps - 1;
      if (A.clips) first = clip_bounds(A.clips, c.i_step, last);
      if (c.i_step >= last) {
        c.i_step = first + (A.left_step[c.i_step] ? 0 : 1);
      } else {
        c.i_step += 1;
        c.count += 1;
      }
      dist = A.step_last_comx[c.rsi_step];   // Q2: `_step` stays the RSI step
      c.pos = dif;
      c.flags &= ~kFlagReadStep0;
    }
  } else {
    if (c.pos >= len - 1) c.pos = 0;
  }
}

// reference sample for this lane's dof at the cursor, with the per-episode COM-X / COM-Z adjustments
__device__ __forceinline__ void ref_lookup(const DevModel& M, const StepArgs& A, const Cursor& c, float dist,
                                           float zoff, int l, int G, bool isdof, float& rq, float& rv) {
  rq = 0.f; rv = 0.f;
  if (!isdof) return;
  const int ds = data_step(c);
  const size_t row = (size_t)(A.step_off[ds] + c.pos) * (size_t)(2 * G);
  rq = A.ref[row + l];
  rv = A.ref[row + G + l];
  if (M.cursor_mode == DRL_CURSOR_STEPWISE) {
    if (l == 0) rq += dist;
    if (l == M.com_z_col && ds == shift_step(c)) rq -= zoff;
  } else {
    if (l == M.com_z_col) rq -= zoff;
  }
}

// sums / minima over the G lanes of an environment (xor offsets below G never leave the group)
template <int G>
__device__ __forceinline__ float group_sum(float x) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) x += __shfl_xor_sync(kFull, x, o);
  return x;
}
template <int G>
__device__ __forceinline__ float group_min(float x) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) x = fminf(x, __shfl_xor_sync(kFull, x, o));
  return x;
}

template <int G>
__device__ __forceinline__ int group_sum_int(int x) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) x += __shfl_xor_sync(kFull, x, o);
  return x;
}

// np.median of the first n entries of hist (non-negative floats) for Monitor.median_abs_torque_smoothed
// (monitor_wrapper.py:102,131), computed by the G lanes of an environment: the values are staged in the environment's
// (by then dead) shared-memory scratch and the middle order statistic is found by a radix select, 8 bits per pass with
// a 256-bin histogram.  Called by every lane of the warp at the end of a step in which an episode ended; n may differ
// between the two environments of a warp, n == 0 returns 0.  scratch: cap floats + 256 ints of this environment.
template <int G>
__device__ __noinline__ float group_median(const float* __restrict__ hist, float* scratch, int cap, int n, int l) {
  unsigned* keys = reinterpret_cast<unsigned*>(scratch);
  int* bins = reinterpret_cast<int*>(scratch + cap);
  const int ns = n < cap ? n : cap;                     // staged part; a longer episode reads the rest from global
  for (int i = l; i < ns; i += G) keys[i] = __float_as_uint(hist[i]);
  __syncwarp();
  auto key_at = [&](int i) -> unsigned { return i < ns ? keys[i] : __float_as_uint(hist[i]); };
  const int nmax = __reduce_max_sync(kFull, n);
  int k = (n - 1) / 2;                                  // lower middle
  unsigned prefix = 0u;
#pragma unroll 1
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int i = l; i < 256; i += G) bins[i] = 0;
    __syncwarp();
    for (int i = l; i < nmax; i += G) {
      if (i < n) {
        const unsigned key = key_at(i);
        if (shift == 24 || (key >> (shift + 8)) == prefix) atomicAdd(&bins[(key >> shift) & 255u], 1);
      }
    }
    __syncwarp();
    // bucket holding rank k: every lane sums 256 / G consecutive bins, a scan over the lanes finds the lane, which
    // then walks its own bins
    constexpr int kPer = 256 / G;
    int mine = 0;
#pragma unroll
    for (int j = 0; j < kPer; j++) mine += bins[l * kPer + j];
    int incl = mine;
#pragma unroll
    for (int o = 1; o < G; o <<= 1) {
      const int t = __shfl_up_sync(kFull, incl, o, G);
      if (l >= o) incl += t;
    }
    const int before = incl - mine;
    const bool owner = n > 0 && k >= before && k < incl;
    int bucket = 0, kk = 0;
    if (owner) {
      int acc = before;
      for (int j = 0; j < kPer; j++) {
        const int c = bins[l * kPer + j];
        if (k < acc + c) { bucket = l * kPer + j; kk = k - acc; break; }
        acc += c;
      }
    }
    // broadcast from the owning lane of this environment (exactly one when n > 0)
    const unsigned own_mask = __ballot_sync(kFull, owner);
    const unsigned grp = (G == 32) ? kFull : (0xFFFFu << (16 * ((threadIdx.x & 31) / 16)));
    const int src = (own_mask & grp) ? __ffs(own_mask & grp) - 1 : 0;
    bucket = __shfl_sync(kFull, bucket, src);
    kk = __shfl_sync(kFull, kk, src);
    prefix = (prefix << 8) | (unsigned)bucket;
    k = kk;
    __syncwarp();
  }
  const unsigned lo = prefix;
  // upper middle (even n): the same value when it is repeated, else the smallest value above it
  unsigned hi = lo;
  if ((nmax > 0) && true) {
    int cnt_le = 0;
    unsigned min_gt = 0xFFFFFFFFu;
    for (int i = l; i < nmax; i += G) {
      if (i < n) {
        const unsigned key = key_at(i);
        if (key <= lo) cnt_le++;
        else min_gt = key < min_gt ? key : min_gt;
      }
    }
    cnt_le = group_sum_int<G>(cnt_le);
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) {
      const unsigned t = __shfl_xor_sync(kFull, min_gt, o);
      min_gt = t < min_gt ? t : min_gt;
    }
    if ((n & 1) == 0 && cnt_le < n / 2 + 1) hi = min_gt;
  }
  return n > 0 ? 0.5f * (__uint_as_float(lo) + __uint_as_float(hi)) : 0.f;
}

// desired walking velocity vector (straight:417-422,479-480 / loco3d:51-97)
__device__ __forceinline__ void desired_velocity(const DevModel& M, const StepArgs& A, const Cursor& c, float& d0,
                                                 float& d1) {
  d1 = 0.f;
  if (A.speed_profile != nullptr) {            // mimic_env.py:406-408 (scalar profile; second component stays 0)
    d0 = A.speed_profile[c.ep_dur % A.speed_profile_len];
  } else if (M.cursor_mode == DRL_CURSOR_STEPWISE) {
    int idx = c.i_step - c.count + 1;
    int lo = 0;                                // library: clamped at the first step of the episode's clip
    if (A.clips) { int last; lo = clip_bounds(A.clips, c.i_step, last); }
    d0 = A.step_vel[idx < lo ? lo : idx];
  } else {
    // library: i_step is the clip; its prefix sums start at row step_off + clip (one leading zero row per clip)
    int len = A.step_len[0];
    const double* pre = A.des_vel_prefix;
    if (A.clips) { len = A.step_len[c.i_step]; pre += 2 * (A.step_off[c.i_step] + c.i_step); }
    int end = c.pos + M.des_vel_window;
    if (end > len - 1) end = len - 1;
    const int n = end - c.pos;
    if (n <= 0) {
      d0 = d1 = nanf("");   // mean of an empty slice (Q23)
    } else {
      d0 = (float)((pre[2 * end] - pre[2 * c.pos]) / (double)n);
      d1 = (float)((pre[2 * end + 1] - pre[2 * c.pos + 1]) / (double)n);
    }
  }
}

// _get_obs (mimic_env.py:403-437) into E.obsbuf (unmirrored); returns phase / des_vel for the extras
template <int G, class ES>
__device__ __forceinline__ void build_obs(const DevModel& M, const StepArgs& A, ES& E, const LaneConst& L,
                                          const Cursor& c, float q, float v, float& phase0, float& des0) {
  const int l = L.l;
  float d0, d1;
  desired_velocity(M, A, c, d0, d1);
  des0 = d0;
  const int np = M.n_phase_obs, nd = M.n_des_vel;
  phase0 = 0.f;
  if (M.phase_mode == DRL_PHASE_FROM_CURSOR) {
    phase0 = (float)c.pos / (float)A.step_len[data_step(c)];
    if (l == 0) E.obsbuf[0] = phase0;
  } else if (L.isdof) {
    for (int k = 0; k < M.n_phase_joints; k++)
      if (M.phase_joints[k] == l) {
        E.obsbuf[2 * k] = atan2f(v, -q) * 0.31830988618379067154f;
        E.obsbuf[2 * k + 1] = sqrtf(q * q + v * v) / 5.f;
      }
  }
  if (l == 0) {
    E.obsbuf[np] = d0;
    if (nd > 1) E.obsbuf[np + 1] = d1;
  }
  if (L.isdof) {
    if (l >= 1) E.obsbuf[np + nd + l - 1] = q;
    E.obsbuf[np + nd + M.nv - 1 + l] = v;
  }
  __syncwarp();
}

// obs (optionally mirrored, mimic_env.py:440-480) from E.obsbuf to global memory; `enable` predicates the stores.
// ov (nullable): this lane's two entries (columns l and l + G) of the observation the step returns, kept for the fused
// VecNormalize moments.
template <int G, class ES>
__device__ __forceinline__ void write_obs(const DevModel& M, ES& E, int l, bool mirror, bool enable,
                                          float* __restrict__ dst, float* ov = nullptr) {
  if (enable) {
#pragma unroll
    for (int t = 0; t < 2; t++) {
      const int k = l + t * G;
      if (k < M.obs_dim) {
        const float x = mirror ? M.mirror_obs_sign[k] * E.obsbuf[M.mirror_obs_idx[k]] : E.obsbuf[k];
        dst[k] = x;
        if (ov) ov[t] = x;
      }
    }
  }
  __syncwarp();
}

// Reference-pose observations (drl_set_ref_obs, A.ref_obs != 0): frame f of the row is the reference qpos[1:] at the
// cursor that cursor_next would reach after offset_f more control steps from the cursor (i_step, pos, flags, rsi_step)
// the observation was built at: the target the pose reward compares against offset_f steps from now.  The cursor copy
// advances once per step transition (pos accumulates, so this equals offset_f calls of cursor_next).  Every frame is
// mirrored with the observation's own decision, through the qpos-block part of the mirror table (closed: the host
// checks it).  dst / dst2 (nullable): row starts; `enable` predicates the stores, `moments` also stores x, x^2 into the
// statistics row srow.  Called by every lane of the warp; no shared memory.
template <int G>
__device__ __noinline__ void ref_obs_frames(const DevModel& M, const StepArgs& A, int i_step, int pos, int flags,
                                            int rsi_step, float zoff, int l, bool mirror, bool enable,
                                            float* __restrict__ dst, float* __restrict__ dst2, double* srow,
                                            bool moments) {
  Cursor c;
  c.i_step = i_step; c.pos = pos; c.flags = flags; c.rsi_step = rsi_step;
  const int nq = M.nv - 1, B = M.n_phase_obs + M.n_des_vel, inc = M.increment;
  const bool own = l >= 1 && l < M.nv;            // lane l carries qpos[l], column l - 1 of a frame
  int src = l;
  float sgn = 1.f;
  if (mirror && own) { src = M.mirror_obs_idx[B + l - 1] - B + 1; sgn = M.mirror_obs_sign[B + l - 1]; }
  const int n = (int)(A.ref_obs & 0xFFu);
  int ahead = 0;
  for (int f = 0; f < n; f++) {
    const int k = (int)((A.ref_obs >> (8 * f + 8)) & 0xFFu) + 1;
    int r = k - ahead;                            // control steps from the previous frame's cursor (offsets increase)
    ahead = k;
    while (r > 0) {
      const int len = A.step_len[data_step(c)];
      const int room = len - 1 - c.pos;
      if (M.cursor_mode == DRL_CURSOR_STEPWISE) {
        // cursor_next steps to the next mocap step on the first call that takes pos past len - 1
        const int j = room < 0 ? 1 : room / inc + 1;
        if (j > r) { c.pos += r * inc; break; }
        int first = 0, last = M.n_steps - 1;
        if (A.clips) first = clip_bounds(A.clips, c.i_step, last);
        c.i_step = c.i_step >= last ? first + (A.left_step[c.i_step] ? 0 : 1) : c.i_step + 1;
        c.pos += j * inc - len + 1;
        c.flags &= ~kFlagReadStep0;
        r -= j;
      } else {
        // ... and wraps to pos 0 on the first call that takes pos to len - 1 or beyond
        const int j = room <= 0 ? 1 : (room + inc - 1) / inc;
        if (j > r) { c.pos += r * inc; break; }
        c.pos = 0;
        r -= j;
      }
    }
    float rq, rv;
    ref_lookup(M, A, c, 0.f, zoff, l, G, own, rq, rv);   // (dist only moves lane 0, the dropped root x)
    const float o = __shfl_sync(kFull, rq, src, G);
    const float x = (mirror && own) ? sgn * o : rq;
    if (enable && own) {
      const int col = M.obs_dim + f * nq + l - 1;
      dst[col] = x;
      if (dst2) dst2[col] = x;
      if (moments) {
        srow[col] = (double)x;
        srow[M.obs_row + col] = (double)x * (double)x;
      }
    }
  }
}

// cos / sin of every hinge angle (slides: displacement) of the joint configuration q into E.cssn, the input of
// tree_kinematics
template <class ES>
__device__ __forceinline__ void publish_joint_trig(const DevModel& M, ES& E, const LaneConst& L, float q) {
  const int l = L.l;
  const float ref = M.dof_ref[L.isdof ? l : 0];
  float s = q - ref, cc = 1.f;
  if (L.isdof && L.type == 1) sincos_joint(M.dof_sign[l] * (q - ref), s, cc);
  if (L.isdof) *reinterpret_cast<float2*>(&E.cssn[l][0]) = make_float2(cc, s);
  __syncwarp();
}

// Sum over the end-effector points of |p(q) - p(rq)|^2, p = the point relative to the root-body origin in world axes
// (the frame of E.bodyR, so the root slides drop out).  Lane e < n_ee owns point e.  Overwrites E.cssn and the body
// frames / joint axes of the first EnvSmem union; E.obsbuf and E.Mt are untouched.  Called by every lane of the warp.
template <int NV, int G, class ES>
__device__ __noinline__ float ee_sq_error(const DevModel& M, ES& E, const LaneConst& L, const ChainLane& CL, float q,
                                          float rq) {
  const int l = L.l;
  const bool own = l < M.n_ee;
  const int e = own ? l : 0;
  const int b = M.ee_body[e];
  const float p0 = M.ee_pos[e][0], p1 = M.ee_pos[e][1], p2 = M.ee_pos[e][2];
  float d[3] = {0.f, 0.f, 0.f};
#pragma unroll 1
  for (int pass = 0; pass < 2; pass++) {
    publish_joint_trig(M, E, L, pass == 0 ? q : rq);
    tree_kinematics<NV, G>(M, E, CL, l);
#pragma unroll
    for (int r = 0; r < 3; r++) {
      const float4 row = *reinterpret_cast<const float4*>(&E.bodyR[b][4 * r]);
      const float x = row.w + row.x * p0 + row.y * p1 + row.z * p2;
      d[r] = pass == 0 ? x : d[r] - x;
    }
  }
  return group_sum<G>(own ? d[0] * d[0] + d[1] * d[1] + d[2] * d[2] : 0.f);
}

// DeepMimic contact termination: does a body of M.et_contact_mask touch the floor at the joint configuration q?  A
// contact candidate touches when its signed distance to the floor is <= 0, the test with which forward_dynamics
// activates it, taken before the plane-box cap of four corners (which does not change whether a body touches).  The
// root height and the distances restate forward_dynamics (fd_tree.cuh, steps 1 and 7) so that its hot loop stays as it
// is.  Overwrites E.cssn and the body frames / joint axes of the first EnvSmem union; E.obsbuf and E.Mt are untouched.
// Called by every lane of the warp; every lane of an environment gets its environment's answer.
template <int NV, int G, class ES>
__device__ __noinline__ bool floor_contact(const DevModel& M, ES& E, const LaneConst& L, const ChainLane& CL,
                                           float q) {
  using T = Topo<NV>;
  const int l = L.l;
  const unsigned mask = M.et_contact_mask;
  publish_joint_trig(M, E, L, q);
  float zO = M.root_z0;
#pragma unroll
  for (int j = 0; j < T::NSLIDE; j++) zO = fmaf(M.dof_slide_z[j], E.cssn[j][1], zO);
  tree_kinematics<NV, G>(M, E, CL, l);
  bool touch = false;
  if (l < M.nbox_cand) {                       // box corner s = l
    const int b = M.cand_body[l];
    const float4 r2 = *reinterpret_cast<const float4*>(&E.bodyR[b][8]);
    const float rz = r2.x * M.cand_pos[l][0] + r2.y * M.cand_pos[l][1] + r2.z * M.cand_pos[l][2];
    const float cz = zO + r2.w + r2.x * M.cand_aux[l][0] + r2.y * M.cand_aux[l][1] + r2.z * M.cand_aux[l][2];
    touch = ((mask >> b) & 1u) && !(cz + rz > 0.f);
  }
  const int s1 = G + l;                        // capsule end sphere s = G + l
  if (s1 < M.ncand) {
    const int b1 = M.cand_body[s1];
    const float4 r2 = *reinterpret_cast<const float4*>(&E.bodyR[b1][8]);
    const float rz = r2.x * M.cand_pos[s1][0] + r2.y * M.cand_pos[s1][1] + r2.z * M.cand_pos[s1][2];
    const float dist1 = zO + r2.w + rz - M.cand_aux[s1][0];
    touch = touch || (((mask >> b1) & 1u) && !(dist1 > 0.f));
  }
  return env_any(touch, L.emask);
}

// Failure-weighted RSI, weighted branch: a bin by inverse CDF over the weighted part of the mixture (binary search in
// global memory; the table is a few KB and stays in L2), then a sample uniform within the bin.  h: the draw's coin
// hash; its high 32 bits pick the bin, mix64(h) the sample.  Returns the bin.
__device__ __noinline__ int ars_weighted_draw(const StepArgs& A, unsigned long long h, int& i_step, int& pos) {
  const double x = (double)(h >> 32) * 0x1p-32;
  int lo = 0, hi = A.ars_n_bins - 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(A.ars_cdf + mid) > x) hi = mid;
    else lo = mid + 1;
  }
  const int* bin = A.ars_bins + 3 * lo;
  i_step = __ldg(bin);
  pos = __ldg(bin + 1) + (int)(((mix64(h) & 0xFFFFFFFFull) * (unsigned long long)__ldg(bin + 2)) >> 32);
  return lo;
}

// Failure-weighted RSI, episode end: lane 0 of an episode whose start was a random RSI draw counts it in its start bin
__device__ __noinline__ void ars_count_episode(const StepArgs& A, int env, bool difficult) {
  const int b = A.ars_env_bin[env];
  if (b < 0) return;
  atomicAdd(A.ars_inc + b, 1u);
  if (difficult) atomicAdd(A.ars_inc + A.ars_n_bins + b, 1u);
}

// Mocap library, random RSI draw: a clip with probability clip_weight / sum (inverse CDF, binary search in global
// memory) from an independent hash of the draw r.  Returns the clip's first step, n_steps: its number of steps.
__device__ __noinline__ int clip_draw(const ClipLibrary* L, unsigned long long r, int& n_steps) {
  const double x = (double)(mix64(r ^ 0x3C6EF372FE94F82Bull) >> 32) * 0x1p-32;
  const double* cdf = L->clip_cdf;
  int lo = 0, hi = L->n_clips - 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(cdf + mid) > x) hi = mid;
    else lo = mid + 1;
  }
  const int first = __ldg(L->clip_first + lo);
  n_steps = __ldg(L->clip_first + lo + 1) - first;
  return first;
}

// Mocap library, episode end: lane 0 counts the episode in the clip of its start step
__device__ __noinline__ void clip_count_episode(const ClipLibrary* L, int rsi_step, int ep_len, int kind) {
  unsigned long long* s = L->clip_stats + (size_t)__ldg(L->step_clip + rsi_step) * kClipStatCount;
  atomicAdd(s + kClipEpisodes, 1ull);
  atomicAdd(s + kClipLenSum, (unsigned long long)ep_len);
  atomicAdd(s + kind, 1ull);
}

// Returns the start bin of the failure-weighted RSI table for a random RSI draw while the option is on, else -1 (the
// episode is not counted): deterministic inits, injected draws, playback.
template <int NV, int G, class ES>
__device__ __noinline__ int reset_env(const DevModel& M, const StepArgs& A, ES& E, const LaneConst& L,
                                      const ChainLane& CL, int env, Cursor& c, float& q, float& v, float& dist,
                                      float& zoff) {
  const int l = L.l;
  int start_bin = -1;
  c.ep_dur = 0;
  if (A.eval_mode || A.speed_profile != nullptr) {   // mimic_env.py:536-537; straight:237-265 / base:69-77
    if (M.cursor_mode == DRL_CURSOR_STEPWISE) {
      c.i_step = c.n_det;
      c.pos = (3 * A.step_len[c.i_step]) / 4;
      c.n_det += 1;
      if (c.n_det >= M.eval_n_times) c.n_det = 0;
      c.flags |= kFlagReadStep0 | kFlagDetEpisode;
    } else {
      c.i_step = 0; c.pos = 0;
    }
  } else if (A.inj_istep != nullptr && A.inj_pos != nullptr && A.inj_pos[env] >= 0) {
    c.flags &= ~(kFlagReadStep0 | kFlagDetEpisode);
    // (wrap mode: the injected step is the clip of a library, and ignored with one clip)
    c.i_step = (M.cursor_mode == DRL_CURSOR_STEPWISE || A.clips) ? A.inj_istep[env] : 0;
    c.pos = A.inj_pos[env];
  } else {                                     // straight:460-474 / base:79-85
    c.flags &= ~(kFlagReadStep0 | kFlagDetEpisode);
    const unsigned long long gid = (unsigned long long)(M.env_id_offset + env);
    const unsigned long long r = mix64(mix64(M.seed ^ (gid * 0xD1342543DE82EF95ull)) + (unsigned long long)c.resets);
    // failure-weighted RSI: with probability lambda (its own counter-based coin) the weighted draw replaces the
    // uniform one, which otherwise stays the draw of r, bit for bit
    const unsigned long long h = A.ars_coin ? mix64(r ^ 0x6A09E667F3BCC909ull) : 0ull;
    if ((h & 0xFFFFFFFFull) < A.ars_coin) {
      start_bin = ars_weighted_draw(A, h, c.i_step, c.pos);
    } else {
      // library: a weighted clip first, then the reference's draw inside it
      int first = 0, n = M.n_steps;
      if (A.clips) first = clip_draw(A.clips, r, n);
      c.i_step = first + (int)(((r & 0xFFFFFFFFull) * (unsigned long long)n) >> 32);
      c.pos = (int)(((r >> 32) * (unsigned long long)A.step_len[c.i_step]) >> 32);
      if (A.ars_env_bin) start_bin = A.ars_bins[3 * A.ars_n_bins + c.i_step] + c.pos / A.ars_bin_samples;
    }
    if (A.playback) start_bin = -1;
  }
  c.resets += 1;
  c.rsi_step = c.i_step;
  dist = 0.f;
  zoff = 0.f;
  float rq, rv;
  ref_lookup(M, A, c, dist, zoff, l, G, L.isdof, rq, rv);
  q = rq; v = rv;
  // set_state + sim.forward: lowest foot-corner site (mimic_env.py:546-559)
  publish_joint_trig(M, E, L, q);
  float zO = M.root_z0;
  for (int j = 0; j < M.nslide; j++) zO = fmaf(M.dof_slide_z[j], E.cssn[j][1], zO);
  tree_kinematics<NV, G>(M, E, CL, l);
  float sz = 3.0e38f;
  for (int s = l; s < M.nsite; s += G) sz = fminf(sz, zO + body_point_z<G>(E, M.site_body[s], M.site_pos[s]));
  const float lowest = group_min<G>(sz);
  if (l == M.com_z_dof) q -= lowest;
  zoff = lowest;                               // refs.adjust_COM_Z_pos(lowest)
  cursor_next(M, A, c, dist);                  // mimic_env.py:568
  __syncwarp();
  return start_bin;
}

// PD position servo of dof lane jd (MuJoCo <position kp kv>, actuator length gear*q, velocity gear*v): the actuator
// force f for the target ctrl at the state (q, v).  Zero on dofs without an actuator (their gains, gear and force
// range are zero in DevModel).
__device__ __forceinline__ float pd_force(const DevModel& M, int jd, float ctrl, float q, float v) {
  const float g = M.pd_gear[jd];
  return fminf(fmaxf(M.pd_kp[jd] * (ctrl - g * q) - M.pd_kv[jd] * (g * v), M.pd_flo[jd]), M.pd_fhi[jd]);
}

// PD: the instance drives every motor as a position servo whose force is recomputed from the state of every dynamics
// evaluation (drl_set_actuation); false: the force is the clipped action, held for the whole control step.
template <int NV, int G, bool RK4, bool DBG, bool PD>
__global__ void __launch_bounds__(128, 4) mimic_step_kernel(const StepArgs A, const int do_reset_only) {
  using ES = EnvSmem<G>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  DevModel& M = *reinterpret_cast<DevModel*>(smem_raw);
  constexpr int kModelBytes = PD ? sizeof(DevModel) : kModelBytesTorque;   // torque: the PD tables stay in HBM
  ES* envs = reinterpret_cast<ES*>(smem_raw + kModelBytes);
  {
    const int4* src = reinterpret_cast<const int4*>(A.model);
    int4* dst = reinterpret_cast<int4*>(smem_raw);
    for (int i = threadIdx.x; i < kModelBytes / 16; i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  const int epb = blockDim.x / G;
  const int eib = threadIdx.x / G;
  const int env_raw = blockIdx.x * epb + eib;
  // a warp whose second environment is past the end recomputes the last valid one with all stores disabled
  const bool live = env_raw < A.num_envs;
  const int env = live ? env_raw : A.num_envs - 1;
  // (warps entirely past the end keep running on the clamped environment: the CTA-wide barriers in the substep loop
  //  need every warp, and only the last CTA has such warps)
  ES& E = envs[eib];
  LaneConst L;
  L.l = threadIdx.x % G;
  const int l = L.l;
  ChainLane CL;
  CL.c3 = l / 3; CL.row = l - 3 * CL.c3;
  CL.c6 = l / 6; CL.comp = l - 6 * CL.c6;
  L.emask = (G == 32) ? kFull : (0xFFFFu << (16 * ((threadIdx.x & 31) / 16)));
  L.isdof = l < M.nv;
  L.isbody = l < M.nb;
  const int jd = L.isdof ? l : 0;
  L.body = M.dof_body[jd]; L.type = M.dof_type[jd];

  float* sf = A.state_f + (size_t)env * (4 * G);
  int* si = A.state_i + (size_t)env * kCurCount8;
  float q = sf[l], v = sf[G + l], a = sf[2 * G + l];
  Cursor c;
  c.i_step = si[kCurIstep]; c.pos = si[kCurPos]; c.count = si[kCurCount]; c.ep_dur = si[kCurEpDur];
  c.rsi_step = si[kCurRsiStep]; c.n_det = si[kCurNDet]; c.resets = si[kCurResets]; c.flags = si[kCurFlags];
  float dist = sf[3 * G + kMiscDist], zoff = sf[3 * G + kMiscZoff];
  if (l == 0) { E.cnt[0] = 0; E.cnt[1] = 0; }
  // active set of the last evaluation of the previous step (bits 0-3 / 4-7: pyramid rows of the two candidates,
  // 8-9: candidates in contact, 10: limit row active, 11: limit violated)
  int* sa = A.state_as + (size_t)env * G;
  ActiveSet AS;
  {
    const unsigned pk = (unsigned)sa[l];
    AS.bits[0] = pk & 0xFu; AS.bits[1] = (pk >> 4) & 0xFu; AS.prev_act = (pk >> 8) & 3u;
    AS.lbit = (pk >> 10) & 1u; AS.prev_lim = (pk >> 11) & 1u;
  }
  float* obs_out = A.obs + (size_t)env * M.obs_row;

  if (do_reset_only) {
    // VecEnv.reset(): (masked) reset of the episode state
    const bool want = live && (A.reset_mask == nullptr || A.reset_mask[env]);
    if (!__any_sync(kFull, want)) return;
    const int start_bin = reset_env<NV, G>(M, A, E, L, CL, env, c, q, v, dist, zoff);
    float ph, dv;
    build_obs<G>(M, A, E, L, c, q, v, ph, dv);
    const bool left = M.mirror_policy && A.left_step[c.i_step];
    write_obs<G>(M, E, l, left, want, obs_out);
    if (A.ref_obs)
      ref_obs_frames<G>(M, A, c.i_step, c.pos, c.flags, c.rsi_step, zoff, l, left, want, obs_out, nullptr, nullptr,
                        false);
    if (want) {
      sf[l] = q; sf[G + l] = v; sf[2 * G + l] = 0.f;
      if (l == 0) {
        sf[3 * G + kMiscDist] = dist; sf[3 * G + kMiscZoff] = zoff;
        sf[3 * G + kMiscWalked] = 0.f; sf[3 * G + kMiscEpRet] = 0.f; sf[3 * G + kMiscEpTor] = 0.f;
        sf[3 * G + kMiscPrevPos] = 1.f; sf[3 * G + kMiscPrevVel] = 1.f; sf[3 * G + kMiscPrevCom] = 1.f;
        if (A.ee_f) A.ee_f[2 * (size_t)env] = 1.f;
        si[kCurIstep] = c.i_step; si[kCurPos] = c.pos; si[kCurCount] = c.count; si[kCurEpDur] = 0;
        si[kCurRsiStep] = c.rsi_step; si[kCurNDet] = c.n_det; si[kCurResets] = c.resets; si[kCurFlags] = c.flags;
        if (A.ars_env_bin) A.ars_env_bin[env] = start_bin;
      }
    }
    return;
  }

  // ---- actions -> joint torques (mimic_env.py:170-192, :483-489; MuJoCo ctrl/force clamps) ---------------------
  // PD: actions -> servo targets over the joint ranges, then the same mirror; the target is clamped to the range of
  // the joint (the servo's ctrlrange)
  const bool left0 = M.mirror_policy && A.left_step[c.i_step];
  float force = 0.f;
  {
    float sc = 0.f;
    if (l < M.nu) {
      float act = A.actions[(size_t)env * M.act_dim + l];
      act = fminf(fmaxf(act, -1.f), 1.f);
      if (PD) sc = __fadd_rn(M.pd_mid[l], __fmul_rn(act, M.pd_half[l]));
      else sc = act > 0.f ? __fmul_rn(act, M.act_chi[l]) : __fmul_rn(fabsf(act), M.act_clo[l]);
    }
    {
      const int src = l < M.nu ? M.mirror_act_idx[l] : 0;
      const float o = __shfl_sync(kFull, sc, src, G);
      if (left0) sc = l < M.nu ? M.mirror_act_sign[l] * o : 0.f;
    }
    E.tau[l] = 0.f;
    __syncwarp();
    if (l < M.nu) {
      const int j = M.act_dof[l];
      if (PD) {
        E.tau[j] = fminf(fmaxf(sc, M.dof_lo[j]), M.dof_hi[j]);
      } else {
        const float cc = fminf(fmaxf(sc, M.act_clo[l]), M.act_chi[l]);
        force = fminf(fmaxf(M.act_gear[l] * cc, M.act_flo[l]), M.act_fhi[l]);
        E.tau[j] = M.act_gear[l] * force;
      }
    }
    __syncwarp();
  }
  // torque: the generalised actuator force of this dof for the whole step; PD: the servo target of this dof
  const float tau_in = E.tau[l];
  if (PD) {
    // Monitor torque: the servo forces at the state the step starts from, gathered to the actuator lanes
    const float f0 = L.isdof ? pd_force(M, jd, tau_in, q, v) : 0.f;
    const float fu = __shfl_sync(kFull, f0, l < M.nu ? M.act_dof[l] : 0, G);
    if (l < M.nu) force = fu;
  }
  const float mean_abs_torque = group_sum<G>(l < M.nu ? fabsf(force) : 0.f) / (float)M.nu;

  // ---- physics: frame_skip x (RK4 | semi-implicit Euler) ---------------------------------------------------------
  const float h = M.timestep;
  bool bad = false;      // MuJoCo's mj_checkPos / mj_checkVel: non-finite or huge state -> MujocoException
  float* dbgp = (DBG && A.debug) ? A.debug + (size_t)env * 32 * 40 : nullptr;
  for (int sub = 0; sub < A.frame_skip; sub++) {
    {
      // (collectives must be reached by every lane: no short-circuit around env_any)
      const bool blown = env_any(L.isdof && (!(fabsf(q) <= 1e10f) || !(fabsf(v) <= 1e10f)), L.emask);
      bad = bad || blown;
    }
    if (bad) { q = M.dof_ref[jd]; v = 0.f; a = 0.f; }   // park the environment on a harmless state; it resets below
    if (RK4) {
      const float q0 = q, v0 = v;
      float accq = 0.f, accv = 0.f;
#pragma unroll 1
      for (int st = 0; st < 4; st++) {
        // keep the warps of a CTA within one evaluation of each other: they then share instruction-cache lines
        // (the dynamics evaluation is ~80 KB of straight-line code); measured +3 %
        // (one barrier per substep instead of per stage loses the gain; a second barrier inside the evaluation adds none;
        // no barrier or one before the solver is slower at 64, 96 and 128 threads per CTA: profiles/r02_kernel_ab.md)
        __syncthreads();
        Vec6 Sj;
        const float tau = PD ? (L.isdof ? M.pd_gear[jd] * pd_force(M, jd, tau_in, q, v) : 0.f) : tau_in;
        forward_dynamics<NV, G, DBG>(M, E, L, CL, q, v, tau, a, AS, Sj, dbgp);
        const float bw = (st == 0 || st == 3) ? (1.f / 6.f) : (1.f / 3.f);
        accq = fmaf(bw, v, accq);
        accv = fmaf(bw, a, accv);
        if (st < 3) {
          const float aw = st == 2 ? 1.f : 0.5f;
          const float vn = fmaf(h * aw, a, v0);
          q = fmaf(h * aw, v, q0);
          v = vn;
        }
      }
      q = fmaf(h, accq, q0);
      v = fmaf(h, accv, v0);
    } else {
      // mj_Euler with implicit joint damping: (M + h B) a' = M a   [M a = tau_total + J'f]
      float Hc[NV + 1];
      float Ma = 0.f;
      Vec6 Sj;
      // (PD: kv acts explicitly, as in MuJoCo's Euler; only joint damping is implicit)
      const float tau = PD ? (L.isdof ? M.pd_gear[jd] * pd_force(M, jd, tau_in, q, v) : 0.f) : tau_in;
      forward_dynamics<NV, G, DBG>(M, E, L, CL, q, v, tau, a, AS, Sj, dbgp);
      pure_mass_column<NV, G>(M, E, L, Sj, Hc);     // E.acc holds the constrained qacc of every dof
#pragma unroll
      for (int r = 0; r < NV; r++) {
        if (DBG && dbgp) dbgp[(2 + r) * 32 + l] = Hc[r];
        Ma = fmaf(Hc[r], E.acc[r], Ma);
        if (r == l) Hc[r] += h * M.dof_damping[jd];
      }
      Hc[NV] = Ma;
      float an = ldl_solve_tree<NV, G>(Hc, l);
      if (!L.isdof) an = 0.f;
      v = fmaf(h, an, v);
      q = fmaf(h, v, q);
    }
  }
  {
    const bool blown = env_any(L.isdof && (!(fabsf(q) <= 1e10f) || !(fabsf(v) <= 1e10f)), L.emask);
    bad = bad || blown;
  }
  if (bad) { q = M.dof_ref[jd]; v = 0.f; a = 0.f; }

  // ---- environment logic (computed for every lane; the blow-up path overrides the outcome) ------------------------
  float walked = sf[3 * G + kMiscWalked];
  float ep_ret = sf[3 * G + kMiscEpRet], ep_tor = sf[3 * G + kMiscEpTor];
  float pos_rew = sf[3 * G + kMiscPrevPos], vel_rew = sf[3 * G + kMiscPrevVel], com_rew = sf[3 * G + kMiscPrevCom];
  float reward, phase0 = 0.f, des0 = 0.f;
  float ov[2] = {0.f, 0.f};       // this lane's entries of the returned observation (fused VecNormalize moments)
  bool done;
  const int ep_dur_before = c.ep_dur;
  cursor_next(M, A, c, dist);                                   // mimic_env.py:96
  // Monitor: refs._pos after the first step of an episode (monitor_wrapper.py:91-93), kept in the upper half of flags
  if (ep_dur_before == 0) c.flags = (c.flags & 0xFFFF) | (c.pos << 16);
  if (A.playback) {                                             // set_joint_kinematics_in_sim (mimic_env.py:273-293)
    float rq, rv;
    ref_lookup(M, A, c, dist, zoff, l, G, L.isdof, rq, rv);
    if (L.isdof) { q = rq; v = rv; }
  }
  build_obs<G>(M, A, E, L, c, q, v, phase0, des0);               // mimic_env.py:99
  c.ep_dur += 1;                                                // mimic_env.py:106
  {                                                             // mimic_env.py:131-139
    const float vx = __shfl_sync(kFull, v, 0, G), vy = __shfl_sync(kFull, v, 1, G);
    const float cx = fminf(fmaxf(vx, -5.5f), 5.5f), cy = fminf(fmaxf(vy, -5.5f), 5.5f);
    walked += sqrtf(cx * cx + cy * cy) * M.ctrl_freq_inv;
  }
  const float comz = __shfl_sync(kFull, q, M.com_z_dof, G);
  const bool timeout = c.ep_dur >= M.ep_dur_max;
  float rq, rv;
  ref_lookup(M, A, c, dist, zoff, l, G, L.isdof, rq, rv);
  // do_terminate_early (mimic_env.py:652-702, 3D branch): the reference computes nothing from it in step(); here the
  // reasons are counted and, when configured, end the episode
  bool et_low, et_trunk, et_drunk;
  {
    const int t0 = M.trunk_dof0;
    const float front_dev = fabsf(__shfl_sync(kFull, q - rq, t0, G));
    const float sag = __shfl_sync(kFull, q, t0 + 1, G), comy = __shfl_sync(kFull, q, 1, G);
    et_low = comz < 0.75f;
    et_trunk = (sag > 0.3f || sag < -0.05f) || front_dev > 0.2f;
    et_drunk = fabsf(comy) > 0.2f;
    if (A.playback) et_low = et_trunk = et_drunk = false;
  }
  const bool et_done = M.early_termination && (et_low || et_trunk || et_drunk);
  // optional DeepMimic contact termination (et_contact_mask lives in the CTA's shared model block, playback is a launch
  // argument: warp-uniform), at the state the step ends in.  A blow-up wins, and playback skips it like the reasons
  // above.  Runs before ee_sq_error: both overwrite the body frames.  A step on which it holds is always terminal, so
  // the episode counter is incremented here (A.contact_et is non-null whenever the mask is).
  bool et_contact = false;
  if (M.et_contact_mask != 0u && !A.playback) {
    et_contact = floor_contact<NV, G>(M, E, L, CL, q) && !bad;
    if (et_contact && l == 0 && live) A.contact_et[env] += 1;
  }
  done = (comz < M.fall_z) || timeout || et_done || et_contact;   // mimic_env.py:113-120
  {
    const float dq = L.isdof ? q - rq : 0.f, dv = L.isdof ? v - rv : 0.f;
    const bool iscom = (M.com_mask >> l) & 1u;
    const float sp = group_sum<G>(iscom ? 0.f : dq * dq);
    const float sv = group_sum<G>(iscom ? 0.f : dv * dv);
    const float sc = group_sum<G>(iscom ? dq * dq : 0.f);
    if (!done && !bad) {
      pos_rew = expf(-3.f * sp);                                // mimic_env.py:592-622
      vel_rew = expf(-0.05f * sv);
      com_rew = expf(-16.f * sc);
    }
  }
  // optional DeepMimic end-effector term (w_ee lives in the CTA's shared model block: warp-uniform).  Same rules as the
  // three terms above: kept from the previous step on a terminal step or a blow-up, 1 after a reset.
  float ee_rew = 1.f;
  if (M.w_ee != 0.f) {
    ee_rew = A.ee_f[2 * (size_t)env];
    const float se = ee_sq_error<NV, G>(M, E, L, CL, q, rq);
    if (!done && !bad) ee_rew = expf(-M.ee_scale * se);
  }
  if (bad) {
    // MujocoException path (mimic_env.py:86-91): reset, reward 0, done; the VecEnv then resets again (Q19) — here a
    // single reset serves both, and the terminal observation is the post-reset observation as in the reference
    done = true;
    reward = 0.f;
  } else if (done) {
    reward = timeout ? 0.f : -0.f;                              // _get_ET_reward always evaluates to +-0 (Q1)
  } else {
    float imit = M.w_pos * pos_rew + M.w_vel * vel_rew + M.w_com * com_rew;
    if (M.w_ee != 0.f) imit = fmaf(M.w_ee, ee_rew, imit);
    reward = imit * M.rew_scale + M.alive_bonus;
  }
  const bool left1 = M.mirror_policy && A.left_step[c.i_step];
  float* const dst1 = (done && A.terminal_obs) ? A.terminal_obs + (size_t)env * M.obs_row : obs_out;
  write_obs<G>(M, E, l, left1, live && !bad, dst1, done ? nullptr : ov);
  // ---- per-environment row of sums for the step's statistics: [ sum obs[D] | sum obs^2[D] | ret, ret^2 | stats[20] ].
  // It lives in this environment's (now dead) solver scratch; the rows of a thread block are added up in a fixed order
  // at the end of the kernel, the blocks' rows by the last block to finish: no atomics, bit-reproducible sums.
  // (D = obs_row: with reference-pose frames the row reaches the end of E.Mt, over the union's W and U, which nothing
  //  after this point writes: reset_env and build_obs touch the body frames, E.cssn and E.obsbuf, group_median the
  //  scratch before E.Mt)
  const int kRowStats = 2 * M.obs_row + 2, kRowLen = kRowStats + DRL_STATS_COUNT;
  double* srow = reinterpret_cast<double*>(E.Mt);
  for (int i = l; i < kRowLen; i += G) srow[i] = 0.0;
  __syncwarp();
  // the frames of the terminal or returned observation, at the cursor it was built at; the returned one's moments
  if (A.ref_obs)
    ref_obs_frames<G>(M, A, c.i_step, c.pos, c.flags, c.rsi_step, zoff, l, left1, live && !bad, dst1, nullptr, srow,
                      !done);
  // ---- Monitor.step (monitor_wrapper.py:88-166) --------------------------------------------------------------------
  ep_ret += reward;
  ep_tor += mean_abs_torque;
  const int ep_len_now = bad ? ep_dur_before + 1 : c.ep_dur;
  // per-episode history of the mean |torque| for Monitor's median statistic (monitor_wrapper.py:102,131)
  float med_tor = 0.f;
  if (A.tor_hist) {
    float* hist = A.tor_hist + (size_t)env * M.ep_dur_max;
    if (l == 0 && live && ep_dur_before < M.ep_dur_max) hist[ep_dur_before] = mean_abs_torque;
    __syncwarp();
    if (__any_sync(kFull, done)) {
      const int nh = ep_len_now < M.ep_dur_max ? ep_len_now : M.ep_dur_max;
      // scratch: this environment's solver arrays up to (not including) the statistics row in E.Mt
      float* scratch = &E.S[0][0];
      const int cap = (int)((reinterpret_cast<float*>(E.Mt) - scratch)) - 256;
      med_tor = group_median<G>(hist, scratch, cap, (done && live) ? nh : 0, l);
    }
  }
  double* sd = A.state_d + (size_t)env * 4;
  if (l == 0 && live) {
    sd[0] += (double)pos_rew; sd[1] += (double)vel_rew; sd[2] += (double)com_rew; sd[3] += 1.0;
    if (A.ee_d) A.ee_d[env] += (double)ee_rew;
    srow[kRowStats + DRL_STAT_ENV_STEPS] = 1.0;
    srow[kRowStats + DRL_STAT_POS_REW_SUM] = (double)pos_rew;
    srow[kRowStats + DRL_STAT_VEL_REW_SUM] = (double)vel_rew;
    srow[kRowStats + DRL_STAT_COM_REW_SUM] = (double)com_rew;
    srow[kRowStats + DRL_STAT_REW_STEPS] = 1.0;
    srow[kRowStats + DRL_STAT_ABS_TORQUE_SUM] = (double)mean_abs_torque;
    srow[kRowStats + DRL_STAT_SOLVER_ITERS] = (double)E.cnt[0];
    srow[kRowStats + DRL_STAT_DYN_EVALS] = (double)(A.frame_skip * (RK4 ? 4 : 1));
    srow[kRowStats + DRL_STAT_SOLVER_CAPPED] = (double)E.cnt[1];
    if (!bad) {
      srow[kRowStats + DRL_STAT_ET_COM_LOW] = et_low ? 1.0 : 0.0;
      srow[kRowStats + DRL_STAT_ET_TRUNK] = et_trunk ? 1.0 : 0.0;
      srow[kRowStats + DRL_STAT_ET_DRUNK] = et_drunk ? 1.0 : 0.0;
    }
    // VecNormalize: ret = ret * gamma + reward (SB3 VecNormalize.step_wait), its batch moments
    // (ret[done] = 0 afterwards; the normalised reward itself is computed by drl_vecnorm_step from `rew`)
    if (A.vn_ret) {
      const float r = A.vn_ret[env] * A.vn_gamma + reward;
      A.vn_ret[env] = done ? 0.f : r;
      srow[2 * M.obs_row] = (double)r;
      srow[2 * M.obs_row + 1] = (double)r * (double)r;
    }
    if (A.extras) {
      float* ex = A.extras + (size_t)env * 16;
      ex[0] = pos_rew; ex[1] = vel_rew; ex[2] = com_rew; ex[3] = walked; ex[4] = mean_abs_torque;
      ex[5] = des0; ex[6] = phase0; ex[7] = zoff;
    }
  }
  if (done && l == 0 && live) {
    const int ep_len = ep_len_now;
    float* ms = sf + 3 * G;
    const int fl = c.flags;
    auto smooth = [&](int slot, int bit, float nv, float f) {
      ms[slot] = (fl >> bit) & 1 ? f * nv + (1.f - f) * ms[slot] : nv;   // utils.py:312-329
    };
    if (ep_len > 1) { smooth(kMiscMeanRewSm, 0, ep_ret / (float)(ep_len - 1), 0.9f); c.flags |= 1; }
    smooth(kMiscPosSm, 1, (float)(sd[0] / sd[3]), 0.9f);
    smooth(kMiscVelSm, 1, (float)(sd[1] / sd[3]), 0.9f);
    smooth(kMiscComSm, 1, (float)(sd[2] / sd[3]), 0.9f);
    smooth(kMiscEpRetSm, 1, ep_ret, 0.25f);
    smooth(kMiscEpLenSm, 1, (float)ep_len, 0.75f);
    smooth(kMiscTorSm, 1, ep_tor / (float)ep_len, 0.75f);
    if (A.tor_hist) A.med_tor_sm[env] = (fl >> 1) & 1 ? 0.75f * med_tor + 0.25f * A.med_tor_sm[env] : med_tor;
    if (A.ee_f) {
      const float nv = (float)(A.ee_d[env] / sd[3]);
      float& sm = A.ee_f[2 * (size_t)env + 1];
      sm = (fl >> 1) & 1 ? 0.9f * nv + (1.f - 0.9f) * sm : nv;
    }
    c.flags |= 2;
    ms[kMiscMoved] = walked;
    srow[kRowStats + DRL_STAT_EPISODES] = 1.0;
    srow[kRowStats + DRL_STAT_EP_LEN_SUM] = (double)ep_len;
    srow[kRowStats + DRL_STAT_EP_RET_SUM] = (double)ep_ret;
    if (ep_len > 1) srow[kRowStats + DRL_STAT_EP_MEAN_REW_SUM] = (double)(ep_ret / (float)(ep_len - 1));
    srow[kRowStats + DRL_STAT_MOVED_DISTANCE_SUM] = (double)walked;
    srow[kRowStats + (bad ? DRL_STAT_BLOWUPS : (timeout ? DRL_STAT_TIMEOUTS : DRL_STAT_FALLS))] = 1.0;
    if (A.ring_cap > 0) {
      const unsigned long long slot = atomicAdd(A.ring_head, 1ull) % (unsigned long long)A.ring_cap;
      A.ring_len[slot] = ep_len;
      A.ring_ret[slot] = ep_ret;
      A.ring_rsi_pos[slot] = (int)((unsigned)c.flags >> 16);           // monitor_wrapper.py:91-93
      A.ring_et_pos[slot] = c.pos;                                      // :104-107
      A.ring_difficult[slot] = (float)ep_len < ms[kMiscEpLenSm] * 0.75f ? 1 : 0;   // :123-124 (after the smoothing)
    }
    // failure-weighted RSI: Monitor's difficult bit of the episode, counted in its start bin (not in playback)
    if (A.ars_env_bin && !A.playback) ars_count_episode(A, env, (float)ep_len < ms[kMiscEpLenSm] * 0.75f);
    // mocap library: the episode in the counters of the clip it started in, classified as the statistics above
    if (A.clips)
      clip_count_episode(A.clips, c.rsi_step, ep_len, bad ? kClipBlowups : (timeout ? kClipTimeouts : kClipFalls));
  }
  c.flags = __shfl_sync(kFull, c.flags, 0, G);
  // ---- auto-reset (DummyVecEnv.step_wait), warp-uniform: both environments compute it, only `done` ones commit -----
  if (__any_sync(kFull, done)) {
    Cursor c2 = c;
    float q2 = q, v2 = v, dist2 = dist, zoff2 = zoff;
    const int start_bin = reset_env<NV, G>(M, A, E, L, CL, env, c2, q2, v2, dist2, zoff2);
    float ph, dv;
    build_obs<G>(M, A, E, L, c2, q2, v2, ph, dv);
    const bool left2 = M.mirror_policy && A.left_step[c2.i_step];
    write_obs<G>(M, E, l, left2, live && done, obs_out, ov);
    float* const tdst = A.terminal_obs ? A.terminal_obs + (size_t)env * M.obs_row : obs_out;
    write_obs<G>(M, E, l, left2, live && bad && A.terminal_obs != nullptr, tdst);
    if (A.ref_obs)       // the returned observation's frames and moments (a blow-up's terminal observation is the same)
      ref_obs_frames<G>(M, A, c2.i_step, c2.pos, c2.flags, c2.rsi_step, zoff2, l, left2, live && done, obs_out,
                        (bad && A.terminal_obs) ? tdst : nullptr, srow, true);
    if (done) {
      c = c2; q = q2; v = v2; dist = dist2; zoff = zoff2;
      a = 0.f;
      AS.bits[0] = AS.bits[1] = 0u; AS.prev_act = 0u; AS.lbit = AS.prev_lim = false;
      walked = 0.f; ep_ret = 0.f; ep_tor = 0.f;
      pos_rew = vel_rew = com_rew = 1.f;      // get_imitation_reward() inside reset_model (mimic_env.py:562)
      ee_rew = 1.f;
      if (l == 0 && live && A.ars_env_bin) A.ars_env_bin[env] = start_bin;
    }
  }
  // ---- store -------------------------------------------------------------------------------------------------------
  if (live) {
    sf[l] = q; sf[G + l] = v; sf[2 * G + l] = a;
    sa[l] = (int)(AS.bits[0] | (AS.bits[1] << 4) | (AS.prev_act << 8) | ((AS.lbit ? 1u : 0u) << 10) |
                  ((AS.prev_lim ? 1u : 0u) << 11));
    if (l == 0) {
      A.rew[env] = reward;
      A.done[env] = done ? 1 : 0;
      float* ms = sf + 3 * G;
      ms[kMiscDist] = dist; ms[kMiscZoff] = zoff; ms[kMiscWalked] = walked; ms[kMiscEpRet] = ep_ret;
      ms[kMiscEpTor] = ep_tor; ms[kMiscPrevPos] = pos_rew; ms[kMiscPrevVel] = vel_rew; ms[kMiscPrevCom] = com_rew;
      if (A.ee_f) A.ee_f[2 * (size_t)env] = ee_rew;
      si[kCurIstep] = c.i_step; si[kCurPos] = c.pos; si[kCurCount] = c.count; si[kCurEpDur] = c.ep_dur;
      si[kCurRsiStep] = c.rsi_step; si[kCurNDet] = c.n_det; si[kCurResets] = c.resets; si[kCurFlags] = c.flags;
    }
  }
  // ---- statistics of the step: obs moments of the returned observation, then block sum, then grid sum ---------------
  if (live) {
#pragma unroll
    for (int t = 0; t < 2; t++) {
      const int k = l + t * G;
      if (k < M.obs_dim) {
        const double x = (double)ov[t];
        srow[k] = x;
        srow[M.obs_row + k] = x * x;
      }
    }
  }
  __syncthreads();
  {
    // rows of this block's environments, added in environment order
    double* rows0 = reinterpret_cast<double*>(envs[0].Mt);
    const size_t estride = sizeof(ES) / sizeof(double);
    for (int col = threadIdx.x; col < kRowLen; col += blockDim.x) {
      double sum = 0.0;
      for (int e = 0; e < epb; e++) sum += rows0[(size_t)e * estride + col];
      A.cta_rows[(size_t)blockIdx.x * kRowLen + col] = sum;
    }
  }
  __threadfence();
  __syncthreads();
  // two-level sum in a fixed order, whichever blocks end up doing it: the last block of a group of kStatGroup blocks
  // adds the group's rows (one round of independent loads), the last group to finish adds the group rows and
  // publishes: batch moments -> A.packed, statistics -> added to A.stats.  The serial tail behind the slowest block is
  // two short rounds instead of one pass over every block's row.
  __shared__ unsigned s_ticket;
  const unsigned grp = blockIdx.x / kStatGroup, ngroups = (gridDim.x + kStatGroup - 1) / kStatGroup;
  const int gcount = min((int)kStatGroup, (int)gridDim.x - (int)grp * kStatGroup);
  if (threadIdx.x == 0) s_ticket = atomicAdd(A.cta_ticket + 1 + grp, 1u);
  __syncthreads();
  if (s_ticket != (unsigned)gcount - 1u) return;
  __threadfence();
  double* grows = A.cta_rows + (size_t)gridDim.x * kRowLen;
  for (int col = threadIdx.x; col < kRowLen; col += blockDim.x) {
    const double* src = A.cta_rows + (size_t)grp * kStatGroup * kRowLen + col;
    double p[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int r = 0; r < kStatGroup; r++)
      if (r < gcount) p[r & 3] += __ldcg(src + (size_t)r * kRowLen);
    grows[(size_t)grp * kRowLen + col] = (p[0] + p[1]) + (p[2] + p[3]);
  }
  if (threadIdx.x == 0) A.cta_ticket[1 + grp] = 0u;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_ticket = atomicAdd(A.cta_ticket, 1u);
  __syncthreads();
  if (s_ticket != ngroups - 1u) return;
  __threadfence();
  for (int col = threadIdx.x; col < kRowLen; col += blockDim.x) {
    double p[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    const double* src = grows + col;
    unsigned r = 0;
    for (; r + 7 < ngroups; r += 8) {
#pragma unroll
      for (int u = 0; u < 8; u++) p[u] += __ldcg(src + (size_t)(r + u) * kRowLen);
    }
    for (; r < ngroups; r++) p[0] += __ldcg(src + (size_t)r * kRowLen);
    const double tot = ((p[0] + p[1]) + (p[2] + p[3])) + ((p[4] + p[5]) + (p[6] + p[7]));
    if (col < kRowStats) {
      if (A.packed) {
        // packed layout of the VecNormalize kernels: [ sum obs[D], sumsq obs[D], n, sum ret, sumsq ret ]
        const int D = M.obs_row;
        A.packed[col < 2 * D ? col : col + 1] = tot;
      }
    } else {
      A.stats[col - kRowStats] += tot;
    }
  }
  if (threadIdx.x == 0) {
    if (A.packed) A.packed[2 * M.obs_row] = (double)A.num_envs;
    *A.cta_ticket = 0u;
  }
}

// gather of the per-env extras (Monitor attributes served through VecEnv.get_attr)
__global__ void extras_kernel(const float* __restrict__ state_f, const float* __restrict__ last, float* out, int n,
                              int G) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 16) return;
  const int env = i / 16, k = i % 16;
  float val;
  if (k < 8) val = last ? last[env * 16 + k] : 0.f;
  else val = state_f[(size_t)env * 4 * G + 3 * G + k];     // misc slots 8..15 line up with extras 8..15
  if (k == 3) val = state_f[(size_t)env * 4 * G + 3 * G + kMiscWalked];
  if (k == 7) val = state_f[(size_t)env * 4 * G + 3 * G + kMiscZoff];
  out[i] = val;
}

// Monitor.rsi_positions of the RUNNING episodes (monitor_wrapper.py:91-93): refs._pos after the first step of the episode,
// kept in the upper half of the cursor flags; -1 while the episode has not made its first step
__global__ void running_rsi_kernel(const int* __restrict__ state_i, int* __restrict__ out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int* si = state_i + (size_t)i * kCurCount8;
  out[i] = si[kCurEpDur] > 0 ? (int)((unsigned)si[kCurFlags] >> 16) : -1;
}

// Failure-weighted RSI table update, one block after every step kernel: decay the counts and add the step's integer
// increments (x <- rho x + dx, rounded in that order), zero the increments, then build the distribution of the
// weighted part, w_b = u_b (f_b + 1) / (s_b + 2), as a float64 CDF in a fixed order: every thread sums a contiguous
// run of bins, thread 0 scans the runs' totals.  The result does not depend on how the step kernel's atomics landed.
constexpr int kArsThreads = 256;
__global__ void __launch_bounds__(kArsThreads) adaptive_rsi_update_kernel(const AdaptiveRsiArgs a) {
  __shared__ double run_off[kArsThreads + 1];
  const int n = a.n_bins, per = (n + kArsThreads - 1) / kArsThreads;
  const int b0 = min(n, (int)threadIdx.x * per), b1 = min(n, b0 + per);
  double* s = a.counts;
  double* f = a.counts + n;
  auto weight = [&](int b) { return a.u[b] * ((f[b] + 1.0) / (s[b] + 2.0)); };
  double run = 0.0;
  for (int b = b0; b < b1; b++) {
    s[b] = __dadd_rn(__dmul_rn(a.rho, s[b]), (double)a.inc[b]);
    f[b] = __dadd_rn(__dmul_rn(a.rho, f[b]), (double)a.inc[n + b]);
    a.inc[b] = 0u;
    a.inc[n + b] = 0u;
    run += weight(b);
  }
  run_off[threadIdx.x] = run;
  __syncthreads();
  if (threadIdx.x == 0) {
    double acc = 0.0;
    for (int t = 0; t < kArsThreads; t++) {
      const double x = run_off[t];
      run_off[t] = acc;
      acc += x;
    }
    run_off[kArsThreads] = acc;
  }
  __syncthreads();
  const double total = run_off[kArsThreads];
  double acc = run_off[threadIdx.x];
  for (int b = b0; b < b1; b++) {
    const double w = weight(b);
    acc += w;
    a.cdf[b] = b == n - 1 ? 1.0 : acc / total;
    a.prob[b] = (1.0 - a.lambda) * a.u[b] + a.lambda * (w / total);
  }
}

// strided copies between the padded state rows and dense [N][nv] user tensors
__global__ void state_copy_kernel(float* state_f, int* state_i, int* state_as, float* qpos, float* qvel, int* cursor,
                                  int n, int nv, int G, int to_state) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * G) return;
  const int env = i / G, l = i % G;
  float* sf = state_f + (size_t)env * 4 * G;
  if (l < nv) {
    if (to_state) {
      if (qpos) sf[l] = qpos[env * nv + l];
      if (qvel) sf[G + l] = qvel[env * nv + l];
      sf[2 * G + l] = 0.f;
      if (qpos || qvel) state_as[(size_t)env * G + l] = 0;
    } else {
      if (qpos) qpos[env * nv + l] = sf[l];
      if (qvel) qvel[env * nv + l] = sf[G + l];
    }
  }
  if (cursor && l < 4) {
    const int slot = l == 0 ? kCurIstep : (l == 1 ? kCurPos : (l == 2 ? kCurCount : kCurEpDur));
    if (to_state) state_i[env * kCurCount8 + slot] = cursor[env * 4 + l];
    else cursor[env * 4 + l] = state_i[env * kCurCount8 + slot];
  }
}

// ------------------------------------------------------------------------------------------------------------------
// launch helpers used by c_api.cu
// ------------------------------------------------------------------------------------------------------------------
// BASELINE.json configs[1] (4096 walker3d envs = 27.7 envs per SM) is one wave only if four 128-thread blocks fit an SM:
// 4 x (model + 8 environments + 1 KB reserved) <= 228 KB
static_assert(4 * (sizeof(DevModel) + 8 * sizeof(EnvSmem<16>) + 1024) <= 228 * 1024,
              "walker3d: four blocks per SM must fit in shared memory");
// the statistics row of an environment, 2 * obs_row + 2 + DRL_STATS_COUNT doubles, lives in E.Mt: it fits the widest
// row, walker_165cm_65kg (47 base columns, nv 19) with DRL_MAX_REF_OBS reference-pose frames
static_assert(47 + DRL_MAX_REF_OBS * (19 - 1) <= DRL_MAX_OBS_TOTAL, "DRL_MAX_OBS_TOTAL holds the widest row");
static_assert(2 * DRL_MAX_OBS_TOTAL + 2 + DRL_STATS_COUNT <= (int)(sizeof(EnvSmem<32>::Mt) / sizeof(double)),
              "the statistics row of the widest observation fits E.Mt");

size_t step_smem_bytes(int G, int envs_per_block, bool pd) {
  const size_t model = pd ? sizeof(DevModel) : kModelBytesTorque;
  return model + (size_t)envs_per_block * (G == 16 ? sizeof(EnvSmem<16>) : sizeof(EnvSmem<32>));
}

template <int NV, int G, bool RK4, bool DBG, bool PD>
static cudaError_t launch_one(const StepArgs& a, int reset_only, int block, cudaStream_t st) {
  const int epb = block / G;
  const size_t smem = step_smem_bytes(G, epb, PD);
  auto kern = mimic_step_kernel<NV, G, RK4, DBG, PD>;
  // function attributes are per device: set them once for every device this process launches on
  static unsigned long long attr_done = 0ull;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (!((attr_done >> (dev & 63)) & 1ull)) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    // all of the unified L1/shared array as shared memory: residency is bounded by the per-env scratch, not by L1 hits
    e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    attr_done |= 1ull << (dev & 63);
  }
  const int grid = (a.num_envs + epb - 1) / epb;
  kern<<<grid, block, smem, st>>>(a, reset_only);
  return cudaGetLastError();
}

template <int NV, int G>
static cudaError_t launch_model(const StepArgs& a, int rk4, int reset_only, int block, bool debug, bool pd,
                                cudaStream_t st) {
  if (pd) return rk4 ? launch_one<NV, G, true, false, true>(a, reset_only, block, st)
                     : launch_one<NV, G, false, false, true>(a, reset_only, block, st);
  if (rk4) return launch_one<NV, G, true, false, false>(a, reset_only, block, st);
  return debug ? launch_one<NV, G, false, true, false>(a, reset_only, block, st)
               : launch_one<NV, G, false, false, false>(a, reset_only, block, st);
}

// instantiated: walker3d (nv 14, 16 lanes) and walker_165cm_65kg (nv 19, 32 lanes), RK4 and Euler, torque and PD
// actuation; the dump variant exists for the torque Euler kernels only (tests evaluate single forward passes with it).
// A reset-only launch never reads the actions: callers use the torque instance for it.
cudaError_t launch_step(const StepArgs& a, int nv, int G, int rk4, int reset_only, int block, bool debug, bool pd,
                        cudaStream_t st) {
  if (debug && (rk4 || pd)) return cudaErrorInvalidValue;
  if (nv == 14 && G == 16) return launch_model<14, 16>(a, rk4, reset_only, block, debug, pd, st);
  if (nv == 19 && G == 32) return launch_model<19, 32>(a, rk4, reset_only, block, debug, pd, st);
  return cudaErrorInvalidValue;
}

// does the uploaded model have the chain shape the kernels are compiled for?  (host-side check, c_api.cu)
template <int NV>
static bool topo_ok(int nb, const int* body_parent, const int* dof_body, const int* dof_type) {
  using T = Topo<NV>;
  if (nb != T::NB) return false;
  int parent[kMaxBody], dofb[kMaxDof];
  for (int b = 0; b < kMaxBody; b++) parent[b] = -2;
  for (int j = 0; j < kMaxDof; j++) dofb[j] = -1;
  parent[0] = -1;
  for (int j = 0; j < T::NROOT; j++) dofb[j] = 0;
  for (int c = 0; c < T::NCHAIN; c++)
    for (int k = 1; k < T::chain_len(c); k++) {
      const int b = T::chain_body1(c) + k - 1;
      if (b >= nb) return false;
      parent[b] = k == 1 ? 0 : b - 1;
      for (int s = 0; s < T::nd(k); s++) dofb[T::chain_dof0(c) + T::dof_off(k) + s] = b;
    }
  for (int b = 0; b < nb; b++)
    if (parent[b] != body_parent[b]) return false;
  for (int j = 0; j < NV; j++) {
    if (dofb[j] != dof_body[j]) return false;
    if ((dof_type[j] == 0) != (j < T::NSLIDE)) return false;
  }
  return true;
}
bool topology_matches(int nv, int nb, const int* body_parent, const int* dof_body, const int* dof_type) {
  if (nv == 14) return topo_ok<14>(nb, body_parent, dof_body, dof_type);
  if (nv == 19) return topo_ok<19>(nb, body_parent, dof_body, dof_type);
  return false;
}

cudaError_t launch_running_rsi(const int* state_i, int* out, int n, cudaStream_t st) {
  running_rsi_kernel<<<(n + 255) / 256, 256, 0, st>>>(state_i, out, n);
  return cudaGetLastError();
}

cudaError_t launch_adaptive_rsi_update(const AdaptiveRsiArgs& a, cudaStream_t st) {
  adaptive_rsi_update_kernel<<<1, kArsThreads, 0, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_extras(const float* state_f, const float* last, float* out, int n, int G, cudaStream_t st) {
  const int total = n * 16;
  extras_kernel<<<(total + 255) / 256, 256, 0, st>>>(state_f, last, out, n, G);
  return cudaGetLastError();
}

cudaError_t launch_state_copy(float* state_f, int* state_i, int* state_as, float* qpos, float* qvel, int* cursor, int n,
                              int nv, int G, int to_state, cudaStream_t st) {
  const int total = n * G;
  state_copy_kernel<<<(total + 255) / 256, 256, 0, st>>>(state_f, state_i, state_as, qpos, qvel, cursor, n, nv, G,
                                                         to_state);
  return cudaGetLastError();
}

}  // namespace drl
