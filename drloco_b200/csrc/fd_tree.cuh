// fd_tree.cuh — the dynamics evaluation of the step kernel (one mj_forward per call; restated in
// oracle/walker_physics.c).  Lane j of an environment owns dof j and one or two contact candidates; every tree
// recursion is laid out along the walker's kinematic CHAINS (root -> leg / root -> trunk), whose shape is a
// compile-time property of the two reference models (drloco/mujoco/xml/walker3d_flat_feet.xml, walker_165cm_65kg.xml):
//
//   * body frames: three "row lanes" per chain carry one row of the rotation matrix down the whole chain in registers
//     (v1: one shared-memory round trip and a warp barrier per tree level);
//   * velocities, bias accelerations, constraint-space twists: six "component lanes" per chain run a prefix sum along
//     the chain's dofs (v1: every dof lane looped over its ancestors, every body lane over its supporting dofs);
//   * composite inertias, subtree forces, subtree contact Hessians: suffix sums along the chains, one component per lane;
//   * the contact Hessians W_b are folded into the composite inertias before the joint-space matrix is formed:
//     H = M + sum_b S_b^T W_b S_b is the CRBA matrix of the tree with inertias I_b + W_b, so the per-body
//     "S^T (W S)" assembly of v1 (one 14-row pass per contact body and solver iteration) disappears;
//   * contact detection evaluates only the signed distance first; everything else runs for touching candidates only.
#pragma once
#include "fd_common.cuh"

namespace drl {

// ---- chain shape of the two walkers ----------------------------------------------------------------------------------
// Bodies of chain c: root (0), then chain_body1(c) + k - 1 for depth k = 1 .. chain_len(c) - 1.  Dofs of chain c: the
// NROOT root dofs, then chain_dof0(c) + dof_off(k) + s for s < nd(k).  drl_upload_model() checks the uploaded model
// against these tables (topology_matches).
template <int NV>
struct Topo;

template <>
struct Topo<14> {   // walker3d_flat_feet.xml: torso -> {right, left} x (thigh[2] -> shank[1] -> foot[1])
  static constexpr int NB = 7, NCHAIN = 2, KMAX = 4, NROOT = 6, NSLIDE = 3;
  __host__ __device__ static constexpr int nd(int k) { return k == 0 ? 6 : (k == 1 ? 2 : 1); }
  __host__ __device__ static constexpr int dof_off(int k) { return k <= 1 ? 0 : (k == 2 ? 2 : (k == 3 ? 3 : 4)); }
  __host__ __device__ static constexpr int chain_dof0(int c) { return c == 0 ? 6 : 10; }
  __host__ __device__ static constexpr int chain_body1(int c) { return c == 0 ? 1 : 4; }
  __host__ __device__ static constexpr int chain_len(int) { return 4; }
  // axis index of the s-th hinge at depth k when it is the same on every chain, else -1 (read from the model)
  __host__ __device__ static constexpr int axis(int k, int s) { return k == 0 ? s : (k == 1 ? (s == 0 ? 1 : 0) : 1); }
  __host__ __device__ static constexpr int chain_of(int j) { return (j - 6) / 4; }     // for j >= NROOT
  static constexpr int NBOX = 2;
  __host__ __device__ static constexpr int box_body(int bx) { return bx == 0 ? 3 : 6; }   // the feet
};

template <>
struct Topo<19> {   // walker_165cm_65kg.xml: pelvis -> {right, left} x (thigh[3] -> shank[1] -> foot[1]), pelvis -> torso[3]
  static constexpr int NB = 8, NCHAIN = 3, KMAX = 4, NROOT = 6, NSLIDE = 3;
  __host__ __device__ static constexpr int nd(int k) { return k == 0 ? 6 : (k == 1 ? 3 : 1); }
  __host__ __device__ static constexpr int dof_off(int k) { return k <= 1 ? 0 : (k == 2 ? 3 : (k == 3 ? 4 : 5)); }
  __host__ __device__ static constexpr int chain_dof0(int c) { return c == 0 ? 9 : (c == 1 ? 14 : 6); }
  __host__ __device__ static constexpr int chain_body1(int c) { return c == 0 ? 2 : (c == 1 ? 5 : 1); }
  __host__ __device__ static constexpr int chain_len(int c) { return c == 2 ? 2 : 4; }
  __host__ __device__ static constexpr int axis(int k, int s) { return k == 0 ? s : (k == 1 ? (s == 2 ? 2 : -1) : 1); }
  __host__ __device__ static constexpr int chain_of(int j) { return j < 9 ? 2 : (j < 14 ? 0 : 1); }   // for j >= NROOT
  static constexpr int NBOX = 4;
  __host__ __device__ static constexpr int box_body(int bx) { return bx == 0 ? 0 : (bx == 1 ? 1 : (bx == 2 ? 4 : 7)); }
};

// bodies of the subtree rooted at body b (bit mask), from the chain tables
template <int NV>
__host__ __device__ constexpr unsigned body_subtree_mask(int b) {
  using T = Topo<NV>;
  if (b == 0) return (1u << T::NB) - 1u;
  unsigned m = 0;
  for (int c = 0; c < T::NCHAIN; c++)
    for (int k = 1; k < T::chain_len(c); k++) {
      const int x = T::chain_body1(c) + k - 1;
      if (x == b)
        for (int k2 = k; k2 < T::chain_len(c); k2++) m |= 1u << (T::chain_body1(c) + k2 - 1);
    }
  return m;
}

// is dof r a strict ancestor of dof k (r moves the body k is attached to)?  The chains are serial, so: an earlier dof
// of the root or of k's own chain.
template <int NV>
__host__ __device__ constexpr bool dof_is_anc(int r, int k) {
  return r < k && (r < Topo<NV>::NROOT || Topo<NV>::chain_of(r) == Topo<NV>::chain_of(k));
}
// lanes (dofs) that are strict ancestors of dof k, as a bit mask
template <int NV>
__host__ __device__ constexpr unsigned dof_anc_mask(int k) {
  unsigned m = 0;
  for (int r = 0; r < k; r++)
    if (dof_is_anc<NV>(r, k)) m |= 1u << r;
  return m;
}

// lanes (dofs) that descend from dof k
template <int NV>
__host__ __device__ constexpr unsigned dof_desc_mask(int k) {
  unsigned m = 0;
  for (int c = k + 1; c < NV; c++)
    if (dof_is_anc<NV>(k, c)) m |= 1u << c;
  return m;
}

// LDL^T solve of the tree-structured system H x = z with H spread one column per lane (H[0..NV-1] = rows of this
// lane's column, both triangles; H[NV] = this lane's rhs entry).  Elimination runs from the leaves to the root, which
// creates no fill-in: pivot k touches only rows / columns of k's ancestors (Featherstone's sparse factorisation).
// Column k is left unscaled (H[r][k] = l_rk d_k) so that each update is one shuffle + one FMA.  Returns x for this
// lane's row.
template <int NV, int G>
__device__ __forceinline__ float ldl_solve_tree(float (&H)[NV + 1], int l) {
  float invd = 0.f;
  const unsigned me = 1u << l;
#pragma unroll
  for (int k = NV - 1; k >= 0; k--) {
    const float dk = __shfl_sync(kFull, H[k], k, G);
    const float inv = fast_rcp(fmaxf(dk, 1e-30f));
    const float lck = H[k] * inv;                      // lane c in anc(k): l_kc = H[k][c] / d_k (H is symmetric)
    const bool upd = (dof_anc_mask<NV>(k) & me) != 0u;
    if (l == k) invd = inv;
#pragma unroll
    for (int r = 0; r <= NV; r++) {
      if (r == NV || dof_is_anc<NV>(r, k)) {
        const float vr = __shfl_sync(kFull, H[r], k, G);   // H[r][k];  r == NV: rhs entry z_k
        if (upd) H[r] = fmaf(-vr, lck, H[r]);
      }
    }
  }
  // x_k = (z_k - sum_{r in anc(k)} H[r][k] x_r) / d_k, root first
  float sacc = H[NV], x = 0.f;
#pragma unroll
  for (int k = 0; k < NV; k++) {
    const float xk = __shfl_sync(kFull, sacc * invd, k, G);
    if (dof_desc_mask<NV>(k) & me) sacc = fmaf(-H[k], xk, sacc);
    if (l == k) x = xk;
  }
  return x;
}

// Staging layout of the per-corner contact Hessians: corner c of box bx, entry i lives at
//   (c >> 2) * kWredHalf + (bx * kWredBox + i) * 4 + (c & 3)
// so that the summing lane reads two conflict-free float4 (corners 0-3, 4-7) and the strides keep the eight lanes of a
// box, the boxes and the two environments of a warp (8 banks apart) on different banks: box stride = 20 and half = 16
// (mod 32 floats).
constexpr int kWredBox = 29;                         // entries reserved per box (27 used)

template <int G>
struct EnvSmem {
  static constexpr int kWredHalf = (G == 16 ? 2 * kWredBox * 4 + 8 : 4 * kWredBox * 4);
  static_assert(kWredHalf % 32 == 16, "bank layout of the staging buffer");
  float v[G];               // qvel at the current stage
  float acc[G];             // qacc iterate
  float tau[G];             // actuator force per dof
  float cssn[G][2];         // cos, sin of hinge angles (slides: -, displacement)
  float S[G][12];           // motion vectors (omega, v_O); row stride 12 floats keeps 8-lane vector loads conflict-free
  union {
    struct {
      float Fd[G][12];          // chain-prefix velocity before dof j -> (V x S_j) v_j -> (Ic + Wsub) S_j
      float bodyR[kMaxBody][16];  // row r of the rotation + r-th coordinate of the origin relative to O: [4r .. 4r+3]
      float Ib[kMaxBody][12];   // spatial inertia about O: m, h[3], Ixx Ixy Ixz Iyy Iyz Izz
      float axw[G][4];          // joint axes in world orientation
    };
    // Solver-time tenants of the same storage (the body frames, body inertias and joint axes are dead by then):
    // Wred = staging of the per-corner contact Hessians for the per-box sums, [box][entry 0..26][corner 0..7], written
    // and consumed at the start of a solver pass (Fd is rewritten right after); sph = the touching capsule-end contacts
    // of each lane (rare), which persist over the solver passes and therefore sit behind Wred, clear of Fd.
    struct {
      float Wred[2 * kWredHalf];
      float sph[G][12];
    };
  };
  float Ic[kMaxBody][12];   // composite
  union {
    struct {
      float V[kMaxBody][8];     // spatial velocity
      float Ab[kMaxBody][8];    // bias acceleration -> body force -> subtree force
      float T[kMaxBody][8];     // S_b * qacc
      float W[kMaxBody][24];    // contact Hessian (21 unique entries) -> subtree sums
      float U[kMaxBody][8];     // contact rhs wrench -> subtree sums
    };
    // lower triangle of the joint-space matrix with an odd row stride (transposed without bank conflicts); lives
    // between the last read of W / U and the first write of T of a solver pass
    float Mt[kMaxBody * 56];
  };
  float obsbuf[kMaxObs];
  int cnt[4];               // solver passes, capped evaluations of this control step (statistics)
  // pad the per-environment stride to 8 (mod 32) floats: the two environments of a warp then use disjoint banks in the
  // chain scans (six components per chain, chains 16 banks apart)
  float pad_[(G == 16) ? 20 : 4];
};
static_assert((sizeof(EnvSmem<16>) / 4) % 32 == 8, "environment stride must be 8 mod 32 floats (bank layout)");
static_assert(sizeof(EnvSmem<16>) % 16 == 0 && sizeof(EnvSmem<32>) % 16 == 0, "vector loads need 16-byte rows");

// lane roles that depend on the chain layout (constant over the launch)
struct ChainLane {
  int c3, row;          // row lanes of the kinematics: chain, rotation-matrix row (l < 3 * NCHAIN)
  int c6, comp;         // component lanes of the chain scans: chain, spatial component (l < 6 * NCHAIN)
};

// row (R0, R1, R2) of a rotation matrix times the rotation about coordinate axis `ax` by the angle whose (cos, sin) is
// (c, s).  `ax` is a compile-time constant wherever the chain tables fix it (the branches then fold away).
__device__ __forceinline__ void rot_row(int ax, float& R0, float& R1, float& R2, float c, float s) {
  if (ax == 0) { const float u = R1, w = R2; R1 = c * u + s * w; R2 = c * w - s * u; }
  else if (ax == 1) { const float u = R2, w = R0; R2 = c * u + s * w; R0 = c * w - s * u; }
  else { const float u = R0, w = R1; R0 = c * u + s * w; R1 = c * w - s * u; }
}

// Body frames relative to O and world joint axes for the joint configuration published in E.cssn (mj_kinematics for
// hinges anchored at the body origin; the root slides move O itself).  Lane (chain, row) walks its chain once.
template <int NV, int G>
__device__ __forceinline__ void tree_kinematics(const DevModel& M, EnvSmem<G>& E, const ChainLane& C, int l) {
  using T = Topo<NV>;
  if (l < 3 * T::NCHAIN) {
    const int c = C.c3, r = C.row;
    const int cd0 = T::chain_dof0(c), cb1 = T::chain_body1(c), clen = T::chain_len(c);
    float R0 = r == 0 ? 1.f : 0.f, R1 = r == 1 ? 1.f : 0.f, R2 = r == 2 ? 1.f : 0.f, pr = 0.f;
#pragma unroll
    for (int k = 0; k < T::KMAX; k++) {
      if (k < clen) {
        const int b = k == 0 ? 0 : cb1 + k - 1;
        const bool own = k > 0 || c == 0;             // the root is recomputed by every chain, published by chain 0
        if (k > 0) pr = pr + R0 * M.body_pos[b][0] + R1 * M.body_pos[b][1] + R2 * M.body_pos[b][2];
        const int j0 = k == 0 ? T::NSLIDE : cd0 + T::dof_off(k);
#pragma unroll
        for (int s = 0; s < 3; s++) {
          if (s < (k == 0 ? T::NROOT - T::NSLIDE : T::nd(k))) {
            const int j = j0 + s;
            const int code = M.dof_code[j];             // axis index | negative-axis flag << 2
            const float2 cs = *reinterpret_cast<const float2*>(&E.cssn[j][0]);
            const int a = T::axis(k, s) >= 0 ? T::axis(k, s) : (code & 3);
            const float ax = a == 0 ? R0 : (a == 1 ? R1 : R2);
            if (own) E.axw[j][r] = (code & 4) ? -ax : ax;
            rot_row(a, R0, R1, R2, cs.x, cs.y);
          }
        }
        if (own) *reinterpret_cast<float4*>(&E.bodyR[b][4 * r]) = make_float4(R0, R1, R2, pr);
      }
    }
  }
  __syncwarp();
}

// z of a point given in the frame of body b, relative to O
template <int G>
__device__ __forceinline__ float body_point_z(const EnvSmem<G>& E, int b, const float* p) {
  const float4 r2 = *reinterpret_cast<const float4*>(&E.bodyR[b][8]);
  return r2.w + r2.x * p[0] + r2.y * p[1] + r2.z * p[2];
}

// Prefix sum of coef[j] * S_j along chain c for spatial component `comp`.  PRE: store the value before each dof into
// E.Fd[j]; body-end values go to dst[b][comp] (dst rows are 8 floats).
template <int NV, int G, bool PRE>
__device__ __forceinline__ void chain_prefix(EnvSmem<G>& E, const float* coef, float (*dst)[8], int c, int comp,
                                             float init) {
  using T = Topo<NV>;
  const int cd0 = T::chain_dof0(c), cb1 = T::chain_body1(c), clen = T::chain_len(c);
  float acc = init;
#pragma unroll
  for (int k = 0; k < T::KMAX; k++) {
    if (k < clen) {
      const int b = k == 0 ? 0 : cb1 + k - 1;
      const int j0 = k == 0 ? 0 : cd0 + T::dof_off(k);
      const bool own = k > 0 || c == 0;
#pragma unroll
      for (int s = 0; s < 6; s++) {
        if (s < T::nd(k)) {
          const int j = j0 + s;
          if (PRE && own) E.Fd[j][comp] = acc;
          acc = fmaf(coef[j], E.S[j][comp], acc);
        }
      }
      if (own) dst[b][comp] = acc;
    }
  }
}

// Sum of src rows [b][comp] (stride floats apart) into running totals along every chain without a product: used for
// the bias accelerations, whose terms are already per dof (E.Fd rows).
template <int NV, int G>
__device__ __forceinline__ void chain_prefix_rows(EnvSmem<G>& E, float (*dst)[8], int c, int comp, float init) {
  using T = Topo<NV>;
  const int cd0 = T::chain_dof0(c), cb1 = T::chain_body1(c), clen = T::chain_len(c);
  float acc = init;
#pragma unroll
  for (int k = 0; k < T::KMAX; k++) {
    if (k < clen) {
      const int b = k == 0 ? 0 : cb1 + k - 1;
      const int j0 = k == 0 ? 0 : cd0 + T::dof_off(k);
#pragma unroll
      for (int s = 0; s < 6; s++)
        if (s < T::nd(k)) acc += E.Fd[j0 + s][comp];
      if (k > 0 || c == 0) dst[b][comp] = acc;
    }
  }
}

// Subtree sums along the chains for one component: dst[b] = sum of src over the subtree of b.  `present`: bodies whose
// src entry is valid (others count as zero).  src may equal dst.
template <int NV>
__device__ __forceinline__ void subtree_scan(const float* src, float* dst, int stride, unsigned present) {
  using T = Topo<NV>;
  float root = (present & 1u) ? src[0] : 0.f;
#pragma unroll
  for (int c = 0; c < T::NCHAIN; c++) {
    float s = 0.f;
#pragma unroll
    for (int k = T::KMAX - 1; k >= 1; k--) {
      if (k < T::chain_len(c)) {
        const int b = T::chain_body1(c) + k - 1;
        if ((present >> b) & 1u) s += src[b * stride];
        dst[b * stride] = s;
      }
    }
    root += s;
  }
  dst[0] = root;
}

// one touching contact candidate: point (relative to O, at mid-penetration), D = 1 / R of its pyramid rows, friction,
// reference acceleration of the four rows
struct Contact {
  float Px, Py, Pz, D, mu, ar[4];
};
__device__ __forceinline__ void st_contact(float* p, const Contact& c) {
  *reinterpret_cast<float4*>(p) = make_float4(c.Px, c.Py, c.Pz, c.D);
  *reinterpret_cast<float4*>(p + 4) = make_float4(c.mu, c.ar[0], c.ar[1], c.ar[2]);
  p[8] = c.ar[3];
}
__device__ __forceinline__ Contact ld_contact(const float* p) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  return Contact{a.x, a.y, a.z, a.w, b.x, {b.y, b.z, b.w, p[8]}};
}

// contact point, regulariser and reference accelerations of candidate s on body b at signed distance dist
template <int G, bool BOX>
__device__ __forceinline__ void contact_setup(const DevModel& M, const EnvSmem<G>& E, int s, int b, float dist,
                                              Contact& c) {
  const float4 r0 = *reinterpret_cast<const float4*>(&E.bodyR[b][0]);
  const float4 r1 = *reinterpret_cast<const float4*>(&E.bodyR[b][4]);
  const float4 r2 = *reinterpret_cast<const float4*>(&E.bodyR[b][8]);
  const float x = M.cand_pos[s][0], y = M.cand_pos[s][1], z = M.cand_pos[s][2];
  if (BOX) {
    const float ux = M.cand_aux[s][0], uy = M.cand_aux[s][1], uz = M.cand_aux[s][2];
    c.Px = (r0.w + r0.x * ux + r0.y * uy + r0.z * uz) + (r0.x * x + r0.y * y + r0.z * z);
    c.Py = (r1.w + r1.x * ux + r1.y * uy + r1.z * uz) + (r1.x * x + r1.y * y + r1.z * z);
    c.Pz = (r2.w + r2.x * ux + r2.y * uy + r2.z * uz) + (r2.x * x + r2.y * y + r2.z * z) - 0.5f * dist;
  } else {
    const float rad = M.cand_aux[s][0];
    c.Px = r0.w + (r0.x * x + r0.y * y + r0.z * z);
    c.Py = r1.w + (r1.x * x + r1.y * y + r1.z * z);
    c.Pz = r2.w + (r2.x * x + r2.y * y + r2.z * z) - rad - 0.5f * dist;
  }
  const float mu = M.cand_mu[s];
  const float imp = impedance(M, dist);
  // D = 1 / (2 mu^2 R_n),  R_n = (1-imp)/imp * invweight * (1 + mu^2)
  const float Rn = fmaxf(kMinVal, (1.f - imp) * M.body_invw_tran[b] * (1.f + mu * mu));
  c.D = imp * fast_rcp(2.f * mu * mu * Rn);
  c.mu = mu;
  // reference acceleration of the four pyramid rows: aref = -B (J v) - K imp dist   (E.V is complete since step 4)
  const Vec6 Vb = ld6(E.V[b]);
  float ux, uy, uz;
  cross3(ux, uy, uz, Vb.w0, Vb.w1, Vb.w2, c.Px, c.Py, c.Pz);
  ux += Vb.v0; uy += Vb.v1; uz += Vb.v2;
  const float base = -M.Kc * imp * dist;
  c.ar[0] = -M.Bc * (uz + mu * ux) + base;
  c.ar[1] = -M.Bc * (uz - mu * ux) + base;
  c.ar[2] = -M.Bc * (uz + mu * uy) + base;
  c.ar[3] = -M.Bc * (uz - mu * uy) + base;
}

// wrench-space Hessian of the active pyramid rows `bt` of a contact: w = (P x d, d), W = sum D w w^T (wv[0..20], packed
// upper triangle) and rhs wrench U = sum D aref w (wv[21..26]); zeros when no row is active
__device__ __forceinline__ void contact_hessian(const Contact& c, unsigned bt, float (&wv)[28]) {
#pragma unroll
  for (int i = 0; i < 28; i++) wv[i] = 0.f;
  if (bt) {
    const float D = c.D, mu = c.mu;
    const float s0 = (bt & 1u) ? 1.f : 0.f, s1 = (bt & 2u) ? 1.f : 0.f;
    const float s2 = (bt & 4u) ? 1.f : 0.f, s3 = (bt & 8u) ? 1.f : 0.f;
    const float Qxx = D * mu * mu * (s0 + s1), Qyy = D * mu * mu * (s2 + s3), Qzz = D * (s0 + s1 + s2 + s3);
    const float Qxz = D * mu * (s0 - s1), Qyz = D * mu * (s2 - s3);
    const float Px = c.Px, Py = c.Py, Pz = c.Pz;
    // X = [P]x Q with Q rows (Qxx,0,Qxz) (0,Qyy,Qyz) (Qxz,Qyz,Qzz);  Nn row i = P x X_i
    const float X00 = Py * Qxz, X01 = -Pz * Qyy + Py * Qyz, X02 = -Pz * Qyz + Py * Qzz;
    const float X10 = Pz * Qxx - Px * Qxz, X11 = -Px * Qyz, X12 = Pz * Qxz - Px * Qzz;
    const float X20 = -Py * Qxx, X21 = Px * Qyy, X22 = -Py * Qxz + Px * Qyz;
    float t0, t1, t2;
    cross3(wv[sym6(0, 0)], wv[sym6(0, 1)], wv[sym6(0, 2)], Px, Py, Pz, X00, X01, X02);
    cross3(t0, wv[sym6(1, 1)], wv[sym6(1, 2)], Px, Py, Pz, X10, X11, X12);
    cross3(t1, t2, wv[sym6(2, 2)], Px, Py, Pz, X20, X21, X22);
    (void)t0; (void)t1; (void)t2;
    wv[sym6(0, 3)] = X00; wv[sym6(0, 4)] = X01; wv[sym6(0, 5)] = X02;
    wv[sym6(1, 3)] = X10; wv[sym6(1, 4)] = X11; wv[sym6(1, 5)] = X12;
    wv[sym6(2, 3)] = X20; wv[sym6(2, 4)] = X21; wv[sym6(2, 5)] = X22;
    wv[sym6(3, 3)] = Qxx; wv[sym6(3, 5)] = Qxz; wv[sym6(4, 4)] = Qyy; wv[sym6(4, 5)] = Qyz;
    wv[sym6(5, 5)] = Qzz;
    const float a0 = s0 * c.ar[0], a1 = s1 * c.ar[1], a2 = s2 * c.ar[2], a3 = s3 * c.ar[3];
    const float gx = D * mu * (a0 - a1), gy = D * mu * (a2 - a3), gz = D * (a0 + a1 + a2 + a3);
    cross3(wv[21], wv[22], wv[23], Px, Py, Pz, gx, gy, gz);
    wv[24] = gx; wv[25] = gy; wv[26] = gz;
  }
}

// which pyramid rows of a contact pull (J_i a - aref_i < 0) at the body twist Tb = S_b qacc
__device__ __forceinline__ unsigned contact_rows(const Contact& c, const Vec6& Tb) {
  float ux, uy, uz;
  cross3(ux, uy, uz, Tb.w0, Tb.w1, Tb.w2, c.Px, c.Py, c.Pz);
  ux += Tb.v0; uy += Tb.v1; uz += Tb.v2;
  const float mu = c.mu;
  return ((uz + mu * ux - c.ar[0] < 0.f) ? 1u : 0u) | ((uz - mu * ux - c.ar[1] < 0.f) ? 2u : 0u) |
         ((uz + mu * uy - c.ar[2] < 0.f) ? 4u : 0u) | ((uz - mu * uy - c.ar[3] < 0.f) ? 8u : 0u);
}

// Column l of the joint-space matrix H[r][c] = S_c . (Ic*_{body(r)} S_r) for r = c or a descendant of c (CRBA on the
// contact-augmented composite inertias; E.Fd holds Ic* S).  Each lane computes its column at and below the diagonal; the
// part above comes from the transposed entries through shared memory.  E.Mt aliases V/Ab/T/W/U: callers guarantee
// those are dead.  Output in registers H[0..NV-1] (armature on the diagonal).
template <int NV, int G>
__device__ __forceinline__ void mass_column(const DevModel& M, EnvSmem<G>& E, const LaneConst& L, const Vec6& S,
                                             float (&H)[NV + 1]) {
  constexpr int kMs = (NV % 2 == 0) ? NV + 1 : NV + 2;
  static_assert(NV * kMs <= (int)(sizeof(E.Mt) / sizeof(float)), "Mt too small");
  const int l = L.l;
  const unsigned me = L.isdof ? (1u << l) : 0u;
#pragma unroll
  for (int r = 0; r < NV; r++) {
    const float d = dot6(S, ld6(E.Fd[r]));
    // rows at and below the diagonal: r == l or r a descendant of l
    H[r] = (((dof_anc_mask<NV>(r) | (1u << r)) & me) != 0u) ? d : 0.f;
    if (L.isdof) E.Mt[r * kMs + l] = H[r];
  }
  __syncwarp();
  const float arm = L.isdof ? M.dof_armature[l] : 0.f;
#pragma unroll
  for (int r = 0; r < NV; r++) {
    if (L.isdof && r < l) H[r] = E.Mt[l * kMs + r];
    if (r == l) H[r] += arm;
  }
}

// One forward-dynamics evaluation (mj_forward).  q, v: this lane's coordinates; a: qacc out.  AS: active set carried
// between evaluations.  Must be called by all 32 lanes of the warp (warp-uniform control flow).  On return E.S holds the
// motion vectors, E.Ic the composite inertias and E.acc the accelerations (used by the Euler damping solve).
template <int NV, int G, bool DBG>
__device__ __forceinline__ void forward_dynamics(const DevModel& M, EnvSmem<G>& E, const LaneConst& L,
                                                  const ChainLane& C, float q, float v, float tau, float& a,
                                                  ActiveSet& AS, Vec6& S, float* dbg) {
  using T = Topo<NV>;
  using ES = EnvSmem<G>;
  const int l = L.l;
  const bool iscomp = l < 6 * T::NCHAIN;
  // ---- 1. joint trig + velocity ------------------------------------------------------------------------------------
  {
    const float ref = M.dof_ref[L.isdof ? l : 0];
    float s = q - ref, c = 1.f;
    if (L.isdof && L.type == 1) sincos_joint(M.dof_sign[l] * (q - ref), s, c);
    if (L.isdof) { *reinterpret_cast<float2*>(&E.cssn[l][0]) = make_float2(c, s); E.v[l] = v; }
  }
  __syncwarp();
  float zO = M.root_z0;
#pragma unroll
  for (int j = 0; j < T::NSLIDE; j++) zO = fmaf(M.dof_slide_z[j], E.cssn[j][1], zO);
  // ---- 2. body frames ----------------------------------------------------------------------------------------------
  tree_kinematics<NV, G>(M, E, C, l);
  // ---- 3. motion vectors, body inertias about O ----------------------------------------------------------------------
  S = Vec6{0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (L.isdof) {
    if (L.type == 1) {
      const float4 ax = *reinterpret_cast<const float4*>(&E.axw[l][0]);
      const float* Rb = E.bodyR[L.body];
      const float px = Rb[3], py = Rb[7], pz = Rb[11];
      S.w0 = ax.x; S.w1 = ax.y; S.w2 = ax.z;
      cross3(S.v0, S.v1, S.v2, px, py, pz, ax.x, ax.y, ax.z);     // v_O = anchor x axis
    } else {                                                       // root slide: constant world axis +-e_k
      const int k = M.dof_code[l] & 3;
      const float sg = (M.dof_code[l] & 4) ? -1.f : 1.f;
      S.v0 = k == 0 ? sg : 0.f; S.v1 = k == 1 ? sg : 0.f; S.v2 = k == 2 ? sg : 0.f;
    }
    st6(E.S[l], S);
  }
  if (L.isbody) {
    const float4 r0 = *reinterpret_cast<const float4*>(&E.bodyR[l][0]);
    const float4 r1 = *reinterpret_cast<const float4*>(&E.bodyR[l][4]);
    const float4 r2 = *reinterpret_cast<const float4*>(&E.bodyR[l][8]);
    const float ix = M.body_ipos[l][0], iy = M.body_ipos[l][1], iz = M.body_ipos[l][2];
    const float m = M.body_mass[l];
    const float cx = r0.w + r0.x * ix + r0.y * iy + r0.z * iz;
    const float cy = r1.w + r1.x * ix + r1.y * iy + r1.z * iz;
    const float cz = r2.w + r2.x * ix + r2.y * iy + r2.z * iz;
    const float I0 = M.body_inertia[l][0], I1 = M.body_inertia[l][1], I2 = M.body_inertia[l][2];
    float Ixx = r0.x * r0.x * I0 + r0.y * r0.y * I1 + r0.z * r0.z * I2;
    float Ixy = r0.x * r1.x * I0 + r0.y * r1.y * I1 + r0.z * r1.z * I2;
    float Ixz = r0.x * r2.x * I0 + r0.y * r2.y * I1 + r0.z * r2.z * I2;
    float Iyy = r1.x * r1.x * I0 + r1.y * r1.y * I1 + r1.z * r1.z * I2;
    float Iyz = r1.x * r2.x * I0 + r1.y * r2.y * I1 + r1.z * r2.z * I2;
    float Izz = r2.x * r2.x * I0 + r2.y * r2.y * I1 + r2.z * r2.z * I2;
    Ixx += m * (cy * cy + cz * cz); Iyy += m * (cx * cx + cz * cz); Izz += m * (cx * cx + cy * cy);
    Ixy -= m * cx * cy; Ixz -= m * cx * cz; Iyz -= m * cy * cz;
    float* I = E.Ib[l];
    *reinterpret_cast<float4*>(I) = make_float4(m, m * cx, m * cy, m * cz);
    *reinterpret_cast<float4*>(I + 4) = make_float4(Ixx, Ixy, Ixz, Iyy);
    *reinterpret_cast<float2*>(I + 8) = make_float2(Iyz, Izz);
  }
  __syncwarp();
  // ---- 4. chain velocities (prefix before every dof, body velocities); composite inertias ------------------------------
  if (iscomp) chain_prefix<NV, G, true>(E, E.v, E.V, C.c6, C.comp, 0.f);
  if (l < 10) subtree_scan<NV>(&E.Ib[0][l], &E.Ic[0][l], 12, 0xFFu);
  __syncwarp();
  // ---- 5. bias-acceleration term of every dof: cdof_dot * v = (V_prefix x_m S) v ------------------------------------------
  if (L.isdof) {
    const Vec6 Vp = ld6(E.Fd[l]);
    Vec6 cd;
    float tx, ty, tz;
    cross3(cd.w0, cd.w1, cd.w2, Vp.w0, Vp.w1, Vp.w2, S.w0, S.w1, S.w2);
    cross3(cd.v0, cd.v1, cd.v2, Vp.w0, Vp.w1, Vp.w2, S.v0, S.v1, S.v2);
    cross3(tx, ty, tz, Vp.v0, Vp.v1, Vp.v2, S.w0, S.w1, S.w2);
    cd.v0 += tx; cd.v1 += ty; cd.v2 += tz;
    cd.w0 *= v; cd.w1 *= v; cd.w2 *= v; cd.v0 *= v; cd.v1 *= v; cd.v2 *= v;
    st6(E.Fd[l], cd);
  }
  __syncwarp();
  // ---- 6. bias acceleration of every body (gravity as a fictitious base acceleration) ----------------------------------------
  if (iscomp) chain_prefix_rows<NV, G>(E, E.Ab, C.c6, C.comp, C.comp == 5 ? -M.gravity_z : 0.f);
  __syncwarp();
  // ---- 7. body forces; contact candidates ---------------------------------------------------------------------------------
  if (L.isbody) {
    const Vec6 Ab = ld6(E.Ab[l]);
    const Vec6 Vb = ld6(E.V[l]);
    Vec6 f = inertia_mul(E.Ib[l], Ab);
    const Vec6 mom = inertia_mul(E.Ib[l], Vb);
    float tx, ty, tz;
    cross3(tx, ty, tz, Vb.w0, Vb.w1, Vb.w2, mom.w0, mom.w1, mom.w2);
    f.w0 += tx; f.w1 += ty; f.w2 += tz;
    cross3(tx, ty, tz, Vb.v0, Vb.v1, Vb.v2, mom.v0, mom.v1, mom.v2);
    f.w0 += tx; f.w1 += ty; f.w2 += tz;
    cross3(tx, ty, tz, Vb.w0, Vb.w1, Vb.w2, mom.v0, mom.v1, mom.v2);
    f.v0 += tx; f.v1 += ty; f.v2 += tz;
    st6(E.Ab[l], f);
  }
  // contacts: candidate s = pass * G + l.  Pass 0 holds the box corners (feet: the common case, kept in registers),
  // pass 1 the capsule end spheres (a fallen walker: rare; their data lives in shared memory and every step that
  // touches it sits in a cold branch).  Signed distance first; the rest only for touching candidates.
  const int wl = threadIdx.x & 31;
  bool act0 = false, act1 = false;
  float dist0 = 0.f, dist1 = 0.f;
  const int body0 = M.cand_body[l < M.ncand ? l : 0];
  {
    if (l < M.nbox_cand) {
      const float4 r2 = *reinterpret_cast<const float4*>(&E.bodyR[body0][8]);
      const float rz = r2.x * M.cand_pos[l][0] + r2.y * M.cand_pos[l][1] + r2.z * M.cand_pos[l][2];
      const float cz = zO + r2.w + r2.x * M.cand_aux[l][0] + r2.y * M.cand_aux[l][1] + r2.z * M.cand_aux[l][2];
      dist0 = cz + rz;
      act0 = !(dist0 > 0.f || rz > 0.f);
    }
    // plane-box keeps at most the first four penetrating corners (MuJoCo mjc_PlaneBox)
    const unsigned bal = __ballot_sync(kFull, act0);
    const unsigned seg = 0xFFu << (wl & ~7);
    const int rank = __popc(bal & seg & ((1u << wl) - 1u));
    if (rank >= 4) act0 = false;
    const int s1 = G + l;
    if (s1 < M.ncand) {
      const int b1 = M.cand_body[s1];
      const float4 r2 = *reinterpret_cast<const float4*>(&E.bodyR[b1][8]);
      const float rz = r2.x * M.cand_pos[s1][0] + r2.y * M.cand_pos[s1][1] + r2.z * M.cand_pos[s1][2];
      dist1 = zO + r2.w + rz - M.cand_aux[s1][0];
      act1 = !(dist1 > 0.f);
    }
  }
  __syncwarp();   // E.Ab (body forces) complete
  const bool any0 = __any_sync(kFull, act0);
  const bool sph_any = __builtin_expect(__any_sync(kFull, act1), 0);
  unsigned conmask = 0;
  Contact c0 = {0.f, 0.f, 0.f, 0.f, 0.f, {0.f, 0.f, 0.f, 0.f}};
  if (any0 && act0) {
    contact_setup<G, true>(M, E, l, body0, dist0, c0);
    conmask |= 1u << body0;
  }
  if (sph_any) {
    Contact c1 = {0.f, 0.f, 0.f, 0.f, 0.f, {0.f, 0.f, 0.f, 0.f}};
    const int b1 = M.cand_body[G + l < M.ncand ? G + l : 0];
    if (act1) {
      contact_setup<G, false>(M, E, G + l, b1, dist1, c1);
      conmask |= 1u << b1;
    }
    __syncwarp();          // E.sph shares storage with the body frames read above
    if (act1) st_contact(E.sph[l], c1);
  }
  // bodies with a contact in either environment of the warp (W/U are kept valid for the union in both)
  conmask = __reduce_or_sync(kFull, conmask);
  // ---- 7b. subtree forces, bias force, smooth rhs ----------------------------------------------------------------------------
  if (l < 6) subtree_scan<NV>(&E.Ab[0][l], &E.Ab[0][l], 8, 0xFFu);
  __syncwarp();
  float rhs0 = 0.f;
  if (L.isdof) {
    const float cb = dot6(S, ld6(E.Ab[L.body]));
    rhs0 = tau - M.dof_damping[l] * v - cb;
    if (DBG) { dbg[0 * 32 + l] = cb; dbg[1 * 32 + l] = rhs0; }
  }
  // ---- joint limits ----------------------------------------------------------------------------------------------------------
  float lsg = 0.f, lD = 0.f, laref = 0.f;
  if (L.isdof && M.dof_limited[l]) {
    float dist = 0.f;
    const float lo = M.dof_lo[l], hi = M.dof_hi[l];
    if (q < lo) { lsg = 1.f; dist = q - lo; }
    else if (q > hi) { lsg = -1.f; dist = hi - q; }
    if (lsg != 0.f) {
      const float imp = impedance(M, dist);
      lD = imp * fast_rcp(fmaxf(kMinVal, (1.f - imp) * M.dof_invw[l]));
      laref = -M.Bc * lsg * v - M.Kc * imp * dist;
    }
  }
  // ---- 8. active-set iteration -----------------------------------------------------------------------------------------------
  // The active set of the previous evaluation (same lane <-> same contact candidate) is the starting guess; a contact
  // or limit that was not present before starts with all of its rows active.  Without any constraint in the warp the
  // loop body runs once and is the plain solve M qacc = rhs0.
  if (!act0) AS.bits[0] = 0u;
  else if (!(AS.prev_act & 1u)) AS.bits[0] = 0xFu;
  if (!act1) AS.bits[1] = 0u;
  else if (!(AS.prev_act & 2u)) AS.bits[1] = 0xFu;
  if (lsg == 0.f) AS.lbit = false;
  else if (!AS.prev_lim) AS.lbit = true;
  const bool any_limit = __any_sync(kFull, lsg != 0.f);
  const bool constrained = (conmask != 0u) || any_limit;
  // bodies whose subtree carries a contact (their composite inertia is augmented)
  unsigned subcon = 0u;
#pragma unroll
  for (int b = 0; b < T::NB; b++)
    if (body_subtree_mask<NV>(b) & conmask) subcon |= 1u << b;
  int n_iter = 0;
  bool capped = false;
  float H[NV + 1];
  for (int it = 0; it < kMaxSolverIter; it++) {
    if (constrained) n_iter++;
    if (conmask != 0u) {
      // Per-body accumulators W (21) / U (6), then their sums over subtrees.  Box corners: the 8 lanes of a segment
      // belong to one box = one body.  Every corner lane stages the 27 numbers of its contact (wrench-space Hessian of
      // the active pyramid rows + rhs wrench), then the lanes share out the 27 x (number of boxes) sums over the 8
      // corners in a fixed order.  No atomics anywhere: the result does not depend on scheduling.
      float wv[28];
      contact_hessian(c0, act0 ? AS.bits[0] : 0u, wv);
      if (l < M.nbox_cand) {
        float* dst = &E.Wred[((l >> 2) & 1) * ES::kWredHalf + (l >> 3) * kWredBox * 4 + (l & 3)];
#pragma unroll
        for (int i = 0; i < 27; i++) dst[i * 4] = wv[i];
      }
      __syncwarp();
      if (!sph_any) {
        // common case (boxes only): the lane that sums entry i of every box also forms the subtree sums - body b
        // receives the boxes of its subtree (compile-time subsets) - so no scan over the tree is needed
#pragma unroll
        for (int i0 = 0; i0 < 27; i0 += G) {
          const int i = i0 + l;
          if (i < 27) {
            float sb[T::NBOX];
#pragma unroll
            for (int bx = 0; bx < T::NBOX; bx++) {
              const float4 x0 = *reinterpret_cast<const float4*>(&E.Wred[(bx * kWredBox + i) * 4]);
              const float4 x1 = *reinterpret_cast<const float4*>(&E.Wred[ES::kWredHalf + (bx * kWredBox + i) * 4]);
              sb[bx] = ((x0.x + x0.y) + (x0.z + x0.w)) + ((x1.x + x1.y) + (x1.z + x1.w));
            }
#pragma unroll
            for (int b = 0; b < T::NB; b++) {
              float tot = 0.f;
              bool any = false;
#pragma unroll
              for (int bx = 0; bx < T::NBOX; bx++)
                if ((body_subtree_mask<NV>(b) >> T::box_body(bx)) & 1u) { tot = any ? tot + sb[bx] : sb[bx]; any = true; }
              if (any) {
                if (i < 21) E.W[b][i] = tot; else E.U[b][i - 21] = tot;
              }
            }
          }
        }
        __syncwarp();
      } else {
        // a capsule touches the ground (fallen walker): per-body accumulators first, then the generic subtree scan
        for (unsigned mk = conmask & ~M.box_body_mask; mk; mk &= mk - 1) {
          const int b = __ffs(mk) - 1;
          for (int i = l; i < 24; i += G) E.W[b][i] = 0.f;
          if (l < 8) E.U[b][l] = 0.f;
        }
#pragma unroll
        for (int bx = 0; bx < T::NBOX; bx++) {
#pragma unroll
          for (int i0 = 0; i0 < 27; i0 += G) {
            const int i = i0 + l;
            if (i < 27) {
              const float4 x0 = *reinterpret_cast<const float4*>(&E.Wred[(bx * kWredBox + i) * 4]);
              const float4 x1 = *reinterpret_cast<const float4*>(&E.Wred[ES::kWredHalf + (bx * kWredBox + i) * 4]);
              const float sum = ((x0.x + x0.y) + (x0.z + x0.w)) + ((x1.x + x1.y) + (x1.z + x1.w));
              const int b = T::box_body(bx);
              if (i < 21) E.W[b][i] = sum; else E.U[b][i - 21] = sum;
            }
          }
        }
        {
          // capsule end spheres: added one contact at a time in lane order (deterministic)
          float wv1[28];
          Contact c1 = {0.f, 0.f, 0.f, 0.f, 0.f, {0.f, 0.f, 0.f, 0.f}};
          const unsigned bt = act1 ? AS.bits[1] : 0u;
          if (bt) c1 = ld_contact(E.sph[l]);
          contact_hessian(c1, bt, wv1);
          const int b1 = M.cand_body[G + l < M.ncand ? G + l : 0];
          __syncwarp();
          for (unsigned sm = __ballot_sync(kFull, bt != 0u); sm; sm &= sm - 1) {
            if (wl == __ffs(sm) - 1) {
              float* Wb = E.W[b1];
              float* Ub = E.U[b1];
#pragma unroll
              for (int i = 0; i < 21; i++) Wb[i] += wv1[i];
#pragma unroll
              for (int i = 0; i < 6; i++) Ub[i] += wv1[21 + i];
            }
            __syncwarp();
          }
        }
        __syncwarp();
        // subtree sums of W (21 entries) and U (6): what the composite inertia / subtree force of every body gains
        const unsigned present = conmask | M.box_body_mask;   // box bodies are always written (zeros without contact)
        for (int i = l; i < 27; i += G) {
          if (i < 21) subtree_scan<NV>(&E.W[0][i], &E.W[0][i], 24, present);
          else subtree_scan<NV>(&E.U[0][i - 21], &E.U[0][i - 21], 8, present);
        }
        __syncwarp();
      }
    }
    // (Ic + Wsub) S and the rhs of this lane's dof
    H[NV] = rhs0;
    if (L.isdof) {
      Vec6 F = inertia_mul(E.Ic[L.body], S);
      if ((subcon >> L.body) & 1u) {
        float Wl[24];
#pragma unroll
        for (int i = 0; i < 24; i += 4) {
          const float4 t = *reinterpret_cast<const float4*>(&E.W[L.body][i]);
          Wl[i] = t.x; Wl[i + 1] = t.y; Wl[i + 2] = t.z; Wl[i + 3] = t.w;
        }
        const float Sv[6] = {S.w0, S.w1, S.w2, S.v0, S.v1, S.v2};
        float y[6];
#pragma unroll
        for (int i = 0; i < 6; i++) {
          float t = 0.f;
#pragma unroll
          for (int j = 0; j < 6; j++) t = fmaf(Wl[sym6(i, j)], Sv[j], t);
          y[i] = t;
        }
        F.w0 += y[0]; F.w1 += y[1]; F.w2 += y[2]; F.v0 += y[3]; F.v1 += y[4]; F.v2 += y[5];
        H[NV] += dot6(S, ld6(E.U[L.body]));
      }
      st6(E.Fd[l], F);
    }
    __syncwarp();      // also: every lane is done with W / U before Mt (same storage) is written
    mass_column<NV, G>(M, E, L, S, H);
    if (AS.lbit) {
#pragma unroll
      for (int r = 0; r < NV; r++)
        if (r == l) H[r] += lD;
      H[NV] += lD * lsg * laref;
    }
    a = ldl_solve_tree<NV, G>(H, l);
    if (!L.isdof) a = 0.f;
    if (L.isdof) E.acc[l] = a;
    if (!constrained) break;
    __syncwarp();
    // ---- re-evaluate the rows at the new qacc: J_i a = w_i . (S_b a) ----
    if (conmask != 0u) {
      if (iscomp) chain_prefix<NV, G, false>(E, E.acc, E.T, C.c6, C.comp, 0.f);
      __syncwarp();
    }
    bool changed = false;
    if (act0) {
      const unsigned nb = contact_rows(c0, ld6(E.T[body0]));
      changed = nb != AS.bits[0];
      AS.bits[0] = nb;
    }
    if (sph_any) {
      if (act1) {
        const Contact c1 = ld_contact(E.sph[l]);
        const unsigned nb = contact_rows(c1, ld6(E.T[M.cand_body[G + l]]));
        changed = changed || (nb != AS.bits[1]);
        AS.bits[1] = nb;
      }
    }
    {
      const bool nl = (lsg != 0.f) && (lsg * a - laref < 0.f);
      changed = changed || (nl != AS.lbit);
      AS.lbit = nl;
    }
    if (!__any_sync(kFull, changed)) break;
    if (it == kMaxSolverIter - 1 && env_any(changed, L.emask)) capped = true;
    __syncwarp();      // T (same storage as W / U / Mt) is read before the next pass rewrites W
  }
  AS.prev_act = (act0 ? 1u : 0u) | (act1 ? 2u : 0u);
  AS.prev_lim = lsg != 0.f;
  // solver statistics (DRL_STAT_SOLVER_ITERS / _CAPPED) are kept per environment in shared memory, off the registers
  if (l == 0) { E.cnt[0] += n_iter; E.cnt[1] += capped ? 1 : 0; }
  if (DBG) {
    dbg[(2 + NV) * 32 + l] = a;
    if (l == 0) {
      dbg[(3 + NV) * 32 + 0] = zO;
      dbg[(3 + NV) * 32 + 1] = (float)__popc(conmask);
    }
    dbg[(4 + NV) * 32 + l] = (float)((act0 ? 1 : 0) + (act1 ? 1 : 0));
  }
}

// Column l of the plain joint-space inertia matrix (no contact terms) from the motion vectors and composite inertias
// left behind by forward_dynamics: the implicit-damping solve of the Euler integrator and the test dump use it.
template <int NV, int G>
__device__ __forceinline__ void pure_mass_column(const DevModel& M, EnvSmem<G>& E, const LaneConst& L,
                                                  const Vec6& S, float (&H)[NV + 1]) {
  __syncwarp();
  if (L.isdof) st6(E.Fd[L.l], inertia_mul(E.Ic[L.body], S));
  __syncwarp();
  mass_column<NV, G>(M, E, L, S, H);
  __syncwarp();
}

}  // namespace drl
