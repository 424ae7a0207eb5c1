// vecnorm.cu — VecNormalize on the device (SB3 1.0 VecNormalize as built at reference drloco/common/utils.py:130-132).
//
//   moments : ret = ret*gamma + rew;  packed = [ sum_obs[D], sumsq_obs[D], n, sum_ret, sumsq_ret ]   (float64 sums)
//             (the step kernel computes the same moments itself when drl_attach_vecnorm is on)
//   step    : exchange of the packed moments between ranks, Chan merge into the running statistics,
//             obs <- clip((obs-mean)/sqrt(var+eps)), rew <- clip(rew/sqrt(ret_var+eps)), ret[done] = 0
//   terminal: the observations of finished environments, normalised and compacted
// Running statistics layout (float64): rms = [ mean[D], var[D], count, ret_mean, ret_var, ret_count ].
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "../../include/drloco_b200.h"

namespace drl {

constexpr int kVnThreads = 256;

// grid-stride over envs; each thread owns one obs column (t % D) of a strip of rows so that loads stay coalesced.
__global__ void vecnorm_moments_kernel(const float* __restrict__ obs, int n, int d, const float* __restrict__ rew,
                                       float* __restrict__ ret, float gamma, double* __restrict__ packed) {
  extern __shared__ double sh[];      // [2*d + 2]
  for (int i = threadIdx.x; i < 2 * d + 2; i += blockDim.x) sh[i] = 0.0;
  __syncthreads();
  const long long total = (long long)n * d;
  const long long stride = (long long)gridDim.x * blockDim.x;
  // obs: element index e -> column e % d.  Use a stride that is a multiple of d so each thread keeps one column.
  const long long tpb = (long long)blockDim.x * gridDim.x;
  const long long step = (tpb / d) * d;
  if (step > 0) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < step) {
      double s = 0.0, ss = 0.0;
      for (long long e = t; e < total; e += step) {
        const double x = (double)obs[e];
        s += x; ss += x * x;
      }
      const int col = (int)(t % d);
      atomicAdd(&sh[col], s);
      atomicAdd(&sh[d + col], ss);
    }
  }
  if (rew != nullptr) {
    double s = 0.0, ss = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
      const float r = ret[i] * gamma + rew[i];
      ret[i] = r;
      s += (double)r; ss += (double)r * (double)r;
    }
    // warp reduce before the shared atomics
    for (int o = 16; o > 0; o >>= 1) {
      s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
      ss += __shfl_xor_sync(0xFFFFFFFFu, ss, o);
    }
    if ((threadIdx.x & 31) == 0) { atomicAdd(&sh[2 * d], s); atomicAdd(&sh[2 * d + 1], ss); }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * d; i += blockDim.x) atomicAdd(&packed[i], sh[i]);
  if (threadIdx.x == 0) {
    if (blockIdx.x == 0) atomicAdd(&packed[2 * d], (double)n);
    atomicAdd(&packed[2 * d + 1], sh[2 * d]);
    atomicAdd(&packed[2 * d + 2], sh[2 * d + 1]);
  }
}

__device__ __forceinline__ void chan_merge(double mean, double var, double count, double bsum, double bsumsq,
                                           double bn, double& nmean, double& nvar, double& ncount) {
  // RunningMeanStd.update_from_moments (SB3 common/running_mean_std.py)
  const double bmean = bsum / bn;
  double bvar = bsumsq / bn - bmean * bmean;
  if (bvar < 0.0) bvar = 0.0;
  const double delta = bmean - mean, tot = count + bn;
  nmean = mean + delta * bn / tot;
  const double m2 = var * count + bvar * bn + delta * delta * count * bn / tot;
  nvar = m2 / tot;
  ncount = tot;
}

}  // namespace drl

// obs [n][d] device, rew [n] device (nullable: reset-time update of the observation statistics only), ret [n] device
// in/out, packed device float64 [2d+3] (zeroed here, then filled).
extern "C" int drl_vecnorm_moments(const float* obs, int32_t n, int32_t d, const float* rew, float* ret, float gamma,
                                   double* packed, void* stream) {
  if (!obs || !packed || n <= 0 || d <= 0 || (rew && !ret)) return DRL_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(packed, 0, (2 * d + 3) * sizeof(double), st) != cudaSuccess) return DRL_ERR_CUDA;
  long long work = (long long)n * d;
  int blocks = (int)((work + drl::kVnThreads * 8 - 1) / (drl::kVnThreads * 8));
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 4) blocks = 148 * 4;
  drl::vecnorm_moments_kernel<<<blocks, drl::kVnThreads, (2 * d + 2) * sizeof(double), st>>>(obs, n, d, rew, ret, gamma,
                                                                                             packed);
  return cudaGetLastError() == cudaSuccess ? DRL_OK : DRL_ERR_CUDA;
}

// ---------------------------------------------------------------------------------------------------------------------
// Statistics exchange + merge + normalisation: ONE kernel per step.
//
// The batch moments of the step arrive in `packed` (written by the step kernel's own epilogue, drl_attach_vecnorm).
// With more than one rank (one process per GPU of a node) every rank owns a small mailbox in its HBM that its peers map
// through CUDA IPC (NVLink peer access): block 0 stores the rank's 2d+3 doubles into slot [rank] of every peer's
// mailbox, fences, and raises a flag; every block of every rank waits for the `world` flags in its LOCAL mailbox, adds
// the slots in rank order (identical bits on every rank), merges them into the running statistics (Chan) and
// normalises its share of the batch.  Nothing returns to the host and there is no second kernel or library call on
// the critical path.  Two mailbox parities alternate: a rank can be at most one exchange ahead of its slowest peer,
// because its next exchange needs that peer's next flag.
//
// sync_every = K > 1 (opt-in, not SB3 semantics): the moments of "cycle" calls (the env steps) are accumulated locally
// and exchanged / merged on every K-th such call only; the steps in between are normalised with the statistics of the
// last merge.  "Immediate" calls (VecNormalize.reset) exchange their own moments at once and leave the cycle alone.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kMaxPeers = 8;
constexpr int kMaxPayload = 2 * DRL_MAX_OBS + 3;

struct DrlComm {
  int world = 1, rank = 0, payload = 0, device = 0;
  void* base = nullptr;                  // local mailbox allocation (exported): mail [2][world][payload] f64, flags [2][world] u64
  double* mail = nullptr;
  unsigned long long* flags = nullptr;
  unsigned long long* step = nullptr;    // [2] device-side counters (the chain is CUDA-graph capturable): exchanges done so
                                         // far (mailbox parity / flag value), cycle calls since the last merge
  unsigned* ticket = nullptr;
  double* pending = nullptr;             // [payload] moments accumulated since the last exchange
  void* peer_base[kMaxPeers] = {};
  bool connected = false;
};

namespace drl {
struct CommView {
  int world, rank, payload, sync_every;
  const double* mail;                    // local
  const unsigned long long* flags;       // local
  double* peer_mail[kMaxPeers];
  unsigned long long* peer_flags[kMaxPeers];
  unsigned long long* step;
  unsigned* ticket;
  double* pending;
};

__device__ __forceinline__ unsigned long long ld_flag(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_flag(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__global__ void __launch_bounds__(256) vecnorm_step_kernel(
    const float* __restrict__ obs_in, float* __restrict__ obs_out, const float* __restrict__ rew_in,
    float* __restrict__ rew_out, int n, int d, const double* __restrict__ packed, const double* __restrict__ rms_in,
    double* __restrict__ rms_out, float* __restrict__ ret, const unsigned char* __restrict__ done,
    unsigned char* __restrict__ done_out, float clip_obs, float clip_rew, float eps, int upd_obs, int upd_ret,
    int norm_obs, int norm_rew, const CommView cv) {
  __shared__ double s_tot[kMaxPayload];
  __shared__ float s_mean[DRL_MAX_OBS], s_inv[DRL_MAX_OBS + 1];
  __shared__ unsigned long long s_ctr[2];
  const int P = cv.payload;        // 2d + 3
  if (threadIdx.x < 2) s_ctr[threadIdx.x] = reinterpret_cast<volatile unsigned long long*>(cv.step)[threadIdx.x];
  __syncthreads();
  const unsigned long long x = s_ctr[0];       // exchanges done so far
  const unsigned long long cyc = s_ctr[1];     // cycle calls accumulated since the last merge
  const int K = cv.sync_every;                 // K >= 1: cycle call; K == 0: immediate call
  const bool update = (upd_obs || upd_ret) && packed != nullptr;
  const bool immediate = K == 0;
  const bool sync = update && (immediate || cyc + 1 >= (unsigned long long)K);
  const bool fresh = immediate || cyc == 0;    // nothing pending from earlier cycle calls (or not to be used)
  bool merged = false;
  if (update) {
    if (!sync) {
      if (blockIdx.x == 0)
        for (int t = threadIdx.x; t < P; t += blockDim.x) cv.pending[t] = (fresh ? 0.0 : cv.pending[t]) + packed[t];
    } else {
      if (cv.world > 1) {
        const int par = (int)(x & 1ull);
        if (blockIdx.x == 0) {
          for (int t = threadIdx.x; t < P; t += blockDim.x) {
            const double v = (fresh ? 0.0 : cv.pending[t]) + packed[t];
            for (int r = 0; r < cv.world; r++) cv.peer_mail[r][((size_t)par * cv.world + cv.rank) * P + t] = v;
          }
          __threadfence_system();
          __syncthreads();
          if (threadIdx.x < cv.world) st_flag(&cv.peer_flags[threadIdx.x][par * cv.world + cv.rank], x + 1ull);
        }
        if (threadIdx.x < cv.world) {
          while (ld_flag(&cv.flags[par * cv.world + threadIdx.x]) < x + 1ull) {
          }
        }
        __syncthreads();
        for (int t = threadIdx.x; t < P; t += blockDim.x) {
          double sum = 0.0;
          for (int r = 0; r < cv.world; r++) sum += __ldcg(&cv.mail[((size_t)par * cv.world + r) * P + t]);   // rank order
          s_tot[t] = sum;
        }
      } else {
        for (int t = threadIdx.x; t < P; t += blockDim.x) s_tot[t] = (fresh ? 0.0 : cv.pending[t]) + packed[t];
      }
      merged = true;
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k <= d; k += blockDim.x) {
    double mean, var, count;
    if (k < d) { mean = rms_in[k]; var = rms_in[d + k]; count = rms_in[2 * d]; }
    else { mean = rms_in[2 * d + 1]; var = rms_in[2 * d + 2]; count = rms_in[2 * d + 3]; }
    const double bn = merged ? s_tot[2 * d] : 0.0;
    if (bn > 0.0 && (k < d ? upd_obs : upd_ret)) {
      const double bs = k < d ? s_tot[k] : s_tot[2 * d + 1];
      const double bss = k < d ? s_tot[d + k] : s_tot[2 * d + 2];
      chan_merge(mean, var, count, bs, bss, bn, mean, var, count);
    }
    if (blockIdx.x == 0) {
      if (k < d) { rms_out[k] = mean; rms_out[d + k] = var; if (k == 0) rms_out[2 * d] = count; }
      else { rms_out[2 * d + 1] = mean; rms_out[2 * d + 2] = var; rms_out[2 * d + 3] = count; }
    }
    if (k < d) { s_mean[k] = (float)mean; s_inv[k] = (float)(1.0 / sqrt(var + (double)eps)); }
    else s_inv[d] = (float)(1.0 / sqrt(var + (double)eps));
  }
  __syncthreads();
  const long long total = (long long)n * d;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
    const int col = (int)(e % d);
    float x = obs_in[e];
    if (norm_obs) x = fminf(fmaxf((x - s_mean[col]) * s_inv[col], -clip_obs), clip_obs);
    obs_out[e] = x;
  }
  if (rew_in != nullptr) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
      float r = rew_in[i];
      if (norm_rew) r = fminf(fmaxf(r * s_inv[d], -clip_rew), clip_rew);
      rew_out[i] = r;
      if (done != nullptr && done[i]) ret[i] = 0.f;
    }
  }
  if (done != nullptr && done_out != nullptr)       // the flags travel with the normalised outputs (one host copy)
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) done_out[i] = done[i];
  // the last block to finish advances the step counter (every block has read it by then)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(cv.ticket, 1u) == gridDim.x - 1) {
      if (update) {
        if (sync) cv.step[0] = x + 1ull;
        if (!immediate) cv.step[1] = sync ? 0ull : cyc + 1ull;
      }
      *cv.ticket = 0u;
      __threadfence();
    }
  }
}
}  // namespace drl

#define VN_TRY(expr)                                   \
  do {                                                 \
    if ((expr) != cudaSuccess) {                       \
      (void)cudaGetLastError();                        \
      return DRL_ERR_CUDA;                             \
    }                                                  \
  } while (0)

extern "C" int drl_comm_create(int32_t world, int32_t rank, int32_t obs_dim, DrlComm** out) {
  if (!out || world < 1 || world > kMaxPeers || rank < 0 || rank >= world || obs_dim <= 0 || obs_dim > DRL_MAX_OBS)
    return DRL_ERR_INVALID;
  DrlComm* c = new DrlComm();
  c->world = world; c->rank = rank; c->payload = 2 * obs_dim + 3;
  VN_TRY(cudaGetDevice(&c->device));
  const size_t mail_bytes = (size_t)2 * world * c->payload * sizeof(double);
  const size_t flag_bytes = (size_t)2 * world * sizeof(unsigned long long);
  VN_TRY(cudaMalloc(&c->base, mail_bytes + flag_bytes));
  VN_TRY(cudaMemset(c->base, 0, mail_bytes + flag_bytes));
  c->mail = (double*)c->base;
  c->flags = (unsigned long long*)((char*)c->base + mail_bytes);
  VN_TRY(cudaMalloc(&c->step, 2 * sizeof(unsigned long long)));
  VN_TRY(cudaMemset(c->step, 0, 2 * sizeof(unsigned long long)));
  VN_TRY(cudaMalloc(&c->ticket, sizeof(unsigned)));
  VN_TRY(cudaMemset(c->ticket, 0, sizeof(unsigned)));
  VN_TRY(cudaMalloc(&c->pending, c->payload * sizeof(double)));
  VN_TRY(cudaMemset(c->pending, 0, c->payload * sizeof(double)));
  VN_TRY(cudaDeviceSynchronize());
  c->peer_base[rank] = c->base;
  c->connected = world == 1;
  *out = c;
  return DRL_OK;
}

extern "C" int drl_comm_export(DrlComm* c, void* handle64) {
  if (!c || !handle64) return DRL_ERR_INVALID;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaIpcMemHandle_t h;
  VN_TRY(cudaIpcGetMemHandle(&h, c->base));
  memcpy(handle64, &h, 64);
  return DRL_OK;
}

extern "C" int drl_comm_connect(DrlComm* c, const void* handles) {
  if (!c || !handles) return DRL_ERR_INVALID;
  VN_TRY(cudaSetDevice(c->device));
  for (int r = 0; r < c->world; r++) {
    if (r == c->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, (const char*)handles + 64 * r, 64);
    VN_TRY(cudaIpcOpenMemHandle(&c->peer_base[r], h, cudaIpcMemLazyEnablePeerAccess));
  }
  c->connected = true;
  return DRL_OK;
}

extern "C" int drl_comm_destroy(DrlComm* c) {
  if (!c) return DRL_OK;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (int r = 0; r < c->world; r++)
    if (r != c->rank && c->peer_base[r]) cudaIpcCloseMemHandle(c->peer_base[r]);
  if (c->base) cudaFree(c->base);
  if (c->step) cudaFree(c->step);
  if (c->ticket) cudaFree(c->ticket);
  if (c->pending) cudaFree(c->pending);
  delete c;
  return DRL_OK;
}

// flags: bit0 update the observation statistics, bit1 norm_obs, bit2 norm_reward, bit3 update the return statistics
extern "C" int drl_vecnorm_step(const float* obs_in, float* obs_out, const float* rew_in, float* rew_out, int32_t n,
                                int32_t d, const double* packed, const double* rms_in, double* rms_out, float* ret,
                                const uint8_t* done, uint8_t* done_out, float clip_obs, float clip_rew, float eps,
                                int32_t flags, DrlComm* c, int32_t sync_every, void* stream) {
  if (!obs_in || !obs_out || !rms_in || !rms_out || n <= 0 || d <= 0 || d > DRL_MAX_OBS || rms_in == rms_out || !c)
    return DRL_ERR_INVALID;
  if (c->payload != 2 * d + 3 || !c->connected || sync_every < 0) return DRL_ERR_STATE;
  drl::CommView cv;
  cv.world = c->world; cv.rank = c->rank; cv.payload = c->payload; cv.sync_every = sync_every;
  cv.mail = c->mail; cv.flags = c->flags; cv.step = c->step; cv.ticket = c->ticket; cv.pending = c->pending;
  const size_t mail_bytes = (size_t)2 * c->world * c->payload * sizeof(double);
  for (int r = 0; r < kMaxPeers; r++) {
    cv.peer_mail[r] = r < c->world ? (double*)c->peer_base[r] : nullptr;
    cv.peer_flags[r] = r < c->world ? (unsigned long long*)((char*)c->peer_base[r] + mail_bytes) : nullptr;
  }
  long long work = (long long)n * d;
  int blocks = (int)((work + drl::kVnThreads * 4 - 1) / (drl::kVnThreads * 4));
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 4) blocks = 148 * 4;      // every block waits for the peers' flags: keep the grid resident
  drl::vecnorm_step_kernel<<<blocks, drl::kVnThreads, 0, (cudaStream_t)stream>>>(
      obs_in, obs_out, rew_in, rew_out, n, d, packed, rms_in, rms_out, ret, done, done_out, clip_obs, clip_rew, eps,
      flags & 1, (flags >> 3) & 1, (flags >> 1) & 1, (flags >> 2) & 1, cv);
  return cudaGetLastError() == cudaSuccess ? DRL_OK : DRL_ERR_CUDA;
}

// Terminal observations of the environments that finished this step, normalised with the current statistics (what
// VecNormalize hands to SB3 in infos[i]["terminal_observation"]), compacted: only the rows of finished environments
// leave the device.  out = 4 header words (out[0] = number of finished environments) followed by one record per
// finished environment, record = { env index (int32 bits), d floats }.  Record order is arbitrary (one atomic slot per
// finished row); the host maps rows back through the index.  `out` may be device memory or pinned host memory mapped
// into the device's address space (the records are then written across PCIe by the kernel itself: no copy node).
// counters: device int32 [2] = { slot counter, block ticket }, zero before the first launch; the last block to finish
// publishes the count in the header and zeroes both again.
namespace drl {
__global__ void vecnorm_terminal_compact_kernel(const float* __restrict__ tin, const unsigned char* __restrict__ done,
                                                int n, int d, const double* __restrict__ rms, float clip_obs, float eps,
                                                int norm_obs, float* __restrict__ out, int* __restrict__ counters) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarp = (gridDim.x * blockDim.x) >> 5;
  for (int row = warp; row < n; row += nwarp) {
    if (!done[row]) continue;
    int slot = 0;
    if (lane == 0) slot = atomicAdd(&counters[0], 1);
    slot = __shfl_sync(0xFFFFFFFFu, slot, 0);
    float* rec = out + 4 + (size_t)slot * (d + 1);
    if (lane == 0) reinterpret_cast<int*>(rec)[0] = row;
    for (int col = lane; col < d; col += 32) {
      float x = tin[(size_t)row * d + col];
      if (norm_obs)
        x = fminf(fmaxf((x - (float)rms[col]) * (float)(1.0 / sqrt(rms[d + col] + (double)eps)), -clip_obs), clip_obs);
      rec[1 + col] = x;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(&counters[1], 1) == (int)gridDim.x - 1) {
      __threadfence();
      reinterpret_cast<int*>(out)[0] = *reinterpret_cast<volatile int*>(&counters[0]);
      counters[0] = 0;
      counters[1] = 0;
      __threadfence_system();
    }
  }
}
}  // namespace drl

extern "C" int drl_vecnorm_terminal_compact(const float* tobs_in, const uint8_t* done, int32_t n, int32_t d,
                                            const double* rms, float clip_obs, float eps, int32_t norm_obs,
                                            float* out_words, int32_t* counters, void* stream) {
  if (!tobs_in || !done || !out_words || !counters || n <= 0 || d <= 0 || (norm_obs && !rms)) return DRL_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  int blocks = (n * 32 + drl::kVnThreads - 1) / drl::kVnThreads;
  if (blocks > 148 * 4) blocks = 148 * 4;
  drl::vecnorm_terminal_compact_kernel<<<blocks, drl::kVnThreads, 0, st>>>(tobs_in, done, n, d, rms, clip_obs, eps,
                                                                         norm_obs, out_words, counters);
  return cudaGetLastError() == cudaSuccess ? DRL_OK : DRL_ERR_CUDA;
}

// ---- FP32 roofline denominator: sustained FFMA rate of the device, measured (bench.py "fp32.peak") ----
namespace drl {
__global__ void __launch_bounds__(256) ffma_probe_kernel(float* out, int iters, float a, float b) {
  float x0 = threadIdx.x * 1e-3f, x1 = x0 + 1.f, x2 = x0 + 2.f, x3 = x0 + 3.f;
  float x4 = x0 + 4.f, x5 = x0 + 5.f, x6 = x0 + 6.f, x7 = x0 + 7.f;
#pragma unroll 4
  for (int i = 0; i < iters; i++) {     // 8 independent chains per thread: issue-bound, not latency-bound
    x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
    x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}
}  // namespace drl

extern "C" int drl_fp32_peak_probe(int32_t device, double* tflops_out) {
  if (!tflops_out) return DRL_ERR_INVALID;
  if (cudaSetDevice(device) != cudaSuccess) return DRL_ERR_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return DRL_ERR_CUDA;
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 16;
  float* buf = nullptr;
  if (cudaMalloc(&buf, (size_t)blocks * threads * sizeof(float)) != cudaSuccess) return DRL_ERR_CUDA;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  double best = 0.0;
  for (int rep = 0; rep < 4; rep++) {
    cudaEventRecord(e0);
    drl::ffma_probe_kernel<<<blocks, threads>>>(buf, iters, 0.999f, 1e-3f);
    cudaEventRecord(e1);
    if (cudaEventSynchronize(e1) != cudaSuccess) { cudaFree(buf); return DRL_ERR_CUDA; }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    const double flops = 2.0 * 8.0 * (double)iters * blocks * threads;
    if (rep > 0 && ms > 0.f) best = fmax(best, flops / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(buf);
  *tflops_out = best;
  return DRL_OK;
}
