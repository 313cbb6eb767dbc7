// Device-resident replay buffer with HER "future" relabelling (the HerReplayBuffer + SAC data path of train_agent.py:61-88).
// SB3 keeps that buffer in host RAM and relabels with one python compute_reward call per row; at batch scale every vectorised
// step would copy N x 2 x 20 KB of observations to the host.  Here the transitions never leave HBM:
//
//   k_replay_begin  : writes the observations the next actions are taken on into the pending slot and closes every open
//                     episode at its newest stored transition (an explicit reset ends episodes without a `done`).
//   k_replay_add    : one launch per vectorised step, one block per environment.  Completes the pending slot (next_obs =
//                     terminal_obs on done, else obs; action, reward, done, info row), advances and writes the current obs
//                     into the next slot.  Images move as 16-byte vectors.  On done it writes the episode's last index into
//                     the episode's stored slots (<= capacity int64 writes), so sampling finds the episode's end in O(1).
//   k_replay_sample : one block per sample.  Environment and transition drawn uniformly among the complete ones; with
//                     probability her_ratio the desired goal becomes the achieved goal of a transition drawn uniformly from
//                     the same episode at or after the sampled one, and the goal term of the reward is recomputed.  Random
//                     numbers come from a counter-based hash of (seed, draw, sample, k): a batch is a pure function of the
//                     buffer contents and these arguments, with no generator state on the device.
//
// Layout: `capacity + 1` slots per environment, slot-major [S][N] like the PPO rollout storage; transition t (counted from 0
// in lock-step over the environments) lives in slot t % S.  The extra slot holds the pending observation, so `capacity`
// complete transitions stay sampleable once the ring has wrapped.
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <cstring>
#include <string>

#include "../../include/b200_gripper_sim.h"

int grl_set_error(const std::string& m);  // train_kernels.cu: grl_last_error()'s message

struct grl_replay {
  int K, S, N, C, H, W, A, her_reward, device;
  unsigned seed;
  long long img;     // bytes of one observation, a multiple of 16
  long long added;   // complete transitions per environment ever added
  bool begun;
  uint8_t *obs, *next_obs, *done;
  float *actions, *reward, *info;
  long long *ep_end;    // [S][N] transition index of the episode's last transition, -1 while the episode is open
  long long *ep_start;  // [N]    first transition of each environment's open episode
};

namespace {

constexpr int THREADS = 256;

struct Ring {
  uint8_t *obs, *next_obs, *done;
  float *actions, *reward, *info;
  long long *ep_end, *ep_start;
  long long img, S;
  int N, A;
};

Ring ring_of(const grl_replay* r) {
  return Ring{r->obs, r->next_obs, r->done, r->actions, r->reward, r->info, r->ep_end, r->ep_start, r->img, r->S, r->N, r->A};
}

__host__ __device__ inline unsigned fmix(unsigned h) {
  h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
  return h;
}
// counter-based hash of (seed, draw, sample): the k-th 32-bit random number of one sample is fmix(base ^ (k + 1) * 0x27D4EB2F)
__host__ __device__ inline unsigned sample_base(unsigned seed, unsigned long long draw, unsigned b) {
  unsigned h = fmix(seed ^ 0x9E3779B9u);
  h = fmix(h ^ (unsigned)draw);
  h = fmix(h ^ (unsigned)(draw >> 32));
  return fmix(h ^ b);
}
__device__ inline unsigned sample_u32(unsigned base, unsigned k) { return fmix(base ^ (k + 1u) * 0x27D4EB2Fu); }
// uniform integer in [0, n) from 32 random bits
__device__ inline long long below(unsigned u, long long n) { return (long long)(((unsigned long long)u * (unsigned long long)n) >> 32); }

// the goal term of the step reward, written exactly as env_finalize computes it (env_kernels.cuh, robot_env.py:268-271)
__device__ inline float goal_term(const float* a, const float* d) {
  const float gx = d[0] - a[0], gy = d[1] - a[1];
  return 1.0f / expf(sqrtf(gx * gx + gy * gy));
}

// marks transitions [max(start, t_end - K + 1), t_end] of environment n as ending at t_end (the older ones are overwritten)
__device__ inline void close_episode(const Ring& r, int n, long long start, long long t_end, long long K) {
  const long long lo = start > t_end - K + 1 ? start : t_end - K + 1;
  for (long long u = lo + threadIdx.x; u <= t_end; u += blockDim.x) r.ep_end[(u % r.S) * r.N + n] = t_end;
}

__global__ void __launch_bounds__(THREADS) k_replay_begin(Ring r, const uint8_t* __restrict__ obs, long long added, long long K) {
  const int n = blockIdx.x;
  const int4* src = reinterpret_cast<const int4*>(obs + (size_t)n * r.img);
  int4* dst = reinterpret_cast<int4*>(r.obs + ((size_t)(added % r.S) * r.N + n) * r.img);
  for (long long i = threadIdx.x; i < r.img / 16; i += blockDim.x) dst[i] = __ldg(src + i);
  const long long start = r.ep_start[n];
  __syncthreads();  // every thread has read ep_start before thread 0 moves it
  if (added > start) close_episode(r, n, start, added - 1, K);
  if (threadIdx.x == 0) r.ep_start[n] = added;
}

__global__ void __launch_bounds__(THREADS) k_replay_add(Ring r, const float* __restrict__ actions, const float* __restrict__ reward,
                                                       const uint8_t* __restrict__ done, const float* __restrict__ info,
                                                       const uint8_t* __restrict__ obs, const uint8_t* __restrict__ terminal_obs,
                                                       long long t, long long K) {
  const int n = blockIdx.x;
  const size_t row = (size_t)(t % r.S) * r.N + n, nrow = (size_t)((t + 1) % r.S) * r.N + n;
  const int d = done[n] != 0;
  const int4* cur = reinterpret_cast<const int4*>(obs + (size_t)n * r.img);
  const int4* nxt = d ? reinterpret_cast<const int4*>(terminal_obs + (size_t)n * r.img) : cur;
  int4* dn = reinterpret_cast<int4*>(r.next_obs + row * r.img);
  int4* dobs = reinterpret_cast<int4*>(r.obs + nrow * r.img);
  for (long long i = threadIdx.x; i < r.img / 16; i += blockDim.x) {
    const int4 v = __ldg(nxt + i);
    __stcs(dn + i, v);  // the ring is read back by sampling much later: do not keep it in L2
    __stcs(dobs + i, d ? __ldg(cur + i) : v);
  }
  if (threadIdx.x < r.A) r.actions[row * r.A + threadIdx.x] = actions[(size_t)n * r.A + threadIdx.x];
  if (threadIdx.x < GRS_INFO_STRIDE) r.info[row * GRS_INFO_STRIDE + threadIdx.x] = info[(size_t)n * GRS_INFO_STRIDE + threadIdx.x];
  const long long start = r.ep_start[n];
  __syncthreads();  // every thread has read ep_start before thread 0 moves it
  if (d) close_episode(r, n, start, t, K);
  if (threadIdx.x == 0) {
    r.reward[row] = reward[n];
    r.done[row] = (uint8_t)d;
    if (!d) r.ep_end[row] = -1;
    else r.ep_start[n] = t + 1;
  }
}

struct SampleOut {
  uint8_t *obs, *next_obs, *done;
  float *actions, *reward, *desired, *achieved, *info;
  long long *index, *goal_index;
};

__global__ void __launch_bounds__(THREADS) k_replay_sample(Ring r, SampleOut o, long long added, long long size, unsigned seed,
                                                          unsigned long long draw, float her_ratio, int her_reward) {
  __shared__ long long s_row, s_grow;
  const int b = blockIdx.x;
  if (threadIdx.x == 0) {
    const unsigned base = sample_base(seed, draw, (unsigned)b);
    const long long env = below(sample_u32(base, 0), r.N);
    const long long t = added - size + below(sample_u32(base, 1), size);
    const long long row = (t % r.S) * r.N + env;
    long long grow = -1;
    if ((float)(sample_u32(base, 2) >> 8) * (1.0f / 16777216.0f) < her_ratio) {
      const long long e = r.ep_end[row];
      long long end = e >= 0 ? e : added - 1;
      // a step whose state went non-finite (FLAGS bit 1, always the done step of its episode) records a non-finite achieved
      // goal: it is never a goal source, and a sample that is such a step itself is not relabelled
      if (e >= 0 && ((int)r.info[((e % r.S) * r.N + env) * GRS_INFO_STRIDE + GRS_INFO_FLAGS] & 2)) end = e - 1;
      if (end >= t) grow = ((t + below(sample_u32(base, 3), end - t + 1)) % r.S) * r.N + env;
    }
    s_row = row; s_grow = grow;
  }
  __syncthreads();
  const long long row = s_row, grow = s_grow;
  const long long nv = r.img / 16;
  const int4* so = reinterpret_cast<const int4*>(r.obs + row * r.img);
  const int4* sn = reinterpret_cast<const int4*>(r.next_obs + row * r.img);
  int4* dobs = reinterpret_cast<int4*>(o.obs + (size_t)b * r.img);
  int4* dn = reinterpret_cast<int4*>(o.next_obs + (size_t)b * r.img);
  for (long long i = threadIdx.x; i < nv; i += blockDim.x) {
    dobs[i] = __ldcs(so + i);
    dn[i] = __ldcs(sn + i);
  }
  const float* inf = r.info + row * GRS_INFO_STRIDE;
  if (threadIdx.x < r.A) o.actions[(size_t)b * r.A + threadIdx.x] = r.actions[row * r.A + threadIdx.x];
  if (o.info && threadIdx.x < GRS_INFO_STRIDE) o.info[(size_t)b * GRS_INFO_STRIDE + threadIdx.x] = inf[threadIdx.x];
  if (threadIdx.x == 0) {
    const float* ag = inf + GRS_INFO_ACHIEVED;
    const float* dg_old = inf + GRS_INFO_DESIRED;
    const float* dg = grow >= 0 ? r.info + grow * GRS_INFO_STRIDE + GRS_INFO_ACHIEVED : dg_old;
    float rew = r.reward[row];
    if (grow >= 0 && her_reward) rew = ((int)inf[GRS_INFO_FLAGS] & 2) ? 0.0f : rew - goal_term(ag, dg_old) + goal_term(ag, dg);
    o.reward[b] = rew;
    o.done[b] = r.done[row];
    o.achieved[2 * b] = ag[0]; o.achieved[2 * b + 1] = ag[1];
    o.desired[2 * b] = dg[0]; o.desired[2 * b + 1] = dg[1];
    if (o.index) o.index[b] = row;
    if (o.goal_index) o.goal_index[b] = grow;
  }
}

// runs f with `device` current, then restores the caller's device
template <class F>
int on_device(int device, F f) {
  int prev = 0;
  cudaGetDevice(&prev);
  if (prev != device && cudaSetDevice(device) != cudaSuccess) return grl_set_error("cudaSetDevice failed");
  const int rc = f();
  if (prev != device) cudaSetDevice(prev);
  return rc;
}

int launched(const char* who) {
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : grl_set_error(std::string(who) + ": " + cudaGetErrorString(e));
}

bool misaligned(const void* p) { return ((uintptr_t)p & 15) != 0; }

void release(grl_replay* r) {
  int prev = 0;
  cudaGetDevice(&prev);
  cudaSetDevice(r->device);
  for (void* p : {(void*)r->obs, (void*)r->next_obs, (void*)r->done, (void*)r->actions, (void*)r->reward, (void*)r->info, (void*)r->ep_end,
                  (void*)r->ep_start})
    if (p) cudaFree(p);
  cudaSetDevice(prev);
  delete r;
}

}  // namespace

extern "C" grl_replay* grl_replay_create(int32_t capacity, int32_t num_envs, int32_t channels, int32_t height, int32_t width, int32_t action_dim,
                                         int32_t her_reward, uint32_t seed, int32_t device) {
  if (capacity <= 0 || num_envs <= 0) { grl_set_error("grl_replay_create: capacity and num_envs must be positive"); return nullptr; }
  if (channels <= 0 || height <= 0 || width <= 0 || ((long long)channels * height * width) % 16 != 0) {
    grl_set_error("grl_replay_create: observation C*H*W must be a positive multiple of 16 bytes (images move as 16-byte vectors)");
    return nullptr;
  }
  if (action_dim <= 0 || action_dim > THREADS) { grl_set_error("grl_replay_create: action_dim must be within 1..256"); return nullptr; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    grl_set_error("grl_replay_create: no CUDA device available: the replay buffer has no CPU fallback");
    return nullptr;
  }
  if (device < 0 || device >= ndev) { grl_set_error("grl_replay_create: invalid CUDA device index"); return nullptr; }
  grl_replay* r = new grl_replay();
  r->K = capacity; r->S = capacity + 1; r->N = num_envs; r->C = channels; r->H = height; r->W = width; r->A = action_dim;
  r->her_reward = her_reward != 0; r->seed = seed; r->device = device;
  r->img = (long long)channels * height * width;
  const size_t rows = (size_t)r->S * r->N;
  const int rc = on_device(device, [&]() -> int {
    const bool ok = cudaMalloc(&r->obs, rows * r->img) == cudaSuccess && cudaMalloc(&r->next_obs, rows * r->img) == cudaSuccess &&
                    cudaMalloc(&r->done, rows) == cudaSuccess && cudaMalloc(&r->actions, rows * r->A * sizeof(float)) == cudaSuccess &&
                    cudaMalloc(&r->reward, rows * sizeof(float)) == cudaSuccess &&
                    cudaMalloc(&r->info, rows * GRS_INFO_STRIDE * sizeof(float)) == cudaSuccess &&
                    cudaMalloc(&r->ep_end, rows * sizeof(long long)) == cudaSuccess && cudaMalloc(&r->ep_start, r->N * sizeof(long long)) == cudaSuccess;
    if (!ok) {
      cudaGetLastError();
      return grl_set_error("grl_replay_create: cudaMalloc of " + std::to_string(rows) + " slots failed");
    }
    if (cudaMemset(r->ep_end, 0xff, rows * sizeof(long long)) != cudaSuccess || cudaMemset(r->ep_start, 0, r->N * sizeof(long long)) != cudaSuccess)
      return grl_set_error("grl_replay_create: cudaMemset failed");
    return 0;
  });
  if (rc != 0) { release(r); return nullptr; }
  return r;
}

extern "C" void grl_replay_destroy(grl_replay* rb) {
  if (rb) release(rb);
}

extern "C" int32_t grl_replay_begin(grl_replay* rb, const uint8_t* obs_dev, void* stream) {
  if (!rb || !obs_dev) return grl_set_error("grl_replay_begin: null pointer");
  if (misaligned(obs_dev)) return grl_set_error("grl_replay_begin: obs must be 16-byte aligned");
  return on_device(rb->device, [&]() -> int {
    k_replay_begin<<<rb->N, THREADS, 0, (cudaStream_t)stream>>>(ring_of(rb), obs_dev, rb->added, rb->K);
    const int rc = launched("grl_replay_begin");
    if (rc == 0) rb->begun = true;
    return rc;
  });
}

extern "C" int32_t grl_replay_add(grl_replay* rb, const float* actions_dev, const float* reward_dev, const uint8_t* done_dev, const float* info_dev,
                                  const uint8_t* obs_dev, const uint8_t* terminal_obs_dev, void* stream) {
  if (!rb || !actions_dev || !reward_dev || !done_dev || !info_dev || !obs_dev || !terminal_obs_dev) return grl_set_error("grl_replay_add: null pointer");
  if (!rb->begun) return grl_set_error("grl_replay_add: call grl_replay_begin with the observations the actions were taken on first");
  if (misaligned(obs_dev) || misaligned(terminal_obs_dev)) return grl_set_error("grl_replay_add: obs and terminal_obs must be 16-byte aligned");
  return on_device(rb->device, [&]() -> int {
    k_replay_add<<<rb->N, THREADS, 0, (cudaStream_t)stream>>>(ring_of(rb), actions_dev, reward_dev, done_dev, info_dev, obs_dev, terminal_obs_dev,
                                                             rb->added, rb->K);
    const int rc = launched("grl_replay_add");
    if (rc == 0) rb->added++;
    return rc;
  });
}

extern "C" int64_t grl_replay_size(const grl_replay* rb) {
  if (!rb) return -1;
  return rb->added < rb->K ? rb->added : rb->K;
}

extern "C" int32_t grl_replay_sample(grl_replay* rb, int32_t batch, float her_ratio, uint64_t draw, uint8_t* obs_dev, uint8_t* next_obs_dev,
                                     float* actions_dev, float* reward_dev, uint8_t* done_dev, float* desired_goal_dev, float* achieved_goal_dev,
                                     float* info_dev, int64_t* index_dev, int64_t* goal_index_dev, void* stream) {
  if (!rb || !obs_dev || !next_obs_dev || !actions_dev || !reward_dev || !done_dev || !desired_goal_dev || !achieved_goal_dev)
    return grl_set_error("grl_replay_sample: null pointer");
  const long long size = grl_replay_size(rb);
  if (size <= 0) return grl_set_error("grl_replay_sample: the buffer holds no complete transition");
  if (batch <= 0) return grl_set_error("grl_replay_sample: batch size must be positive");
  if (!(her_ratio >= 0.0f && her_ratio <= 1.0f)) return grl_set_error("grl_replay_sample: her_ratio must lie in [0, 1]");
  if (misaligned(obs_dev) || misaligned(next_obs_dev)) return grl_set_error("grl_replay_sample: obs and next_obs must be 16-byte aligned");
  const SampleOut o{obs_dev, next_obs_dev, done_dev, actions_dev, reward_dev, desired_goal_dev, achieved_goal_dev, info_dev,
                    reinterpret_cast<long long*>(index_dev), reinterpret_cast<long long*>(goal_index_dev)};
  return on_device(rb->device, [&]() -> int {
    k_replay_sample<<<batch, THREADS, 0, (cudaStream_t)stream>>>(ring_of(rb), o, rb->added, size, rb->seed, (unsigned long long)draw, her_ratio,
                                                                rb->her_reward);
    return launched("grl_replay_sample");
  });
}

extern "C" int32_t grl_replay_buffer(grl_replay* rb, const char* name, void** ptr, uint64_t* bytes) {
  if (!rb || !name || !ptr || !bytes) return grl_set_error("grl_replay_buffer: null pointer");
  const uint64_t rows = (uint64_t)rb->S * rb->N;
  struct { const char* n; void* p; uint64_t b; } views[] = {
      {"obs", rb->obs, rows * rb->img}, {"next_obs", rb->next_obs, rows * rb->img}, {"actions", rb->actions, rows * rb->A * sizeof(float)},
      {"reward", rb->reward, rows * sizeof(float)}, {"done", rb->done, rows}, {"info", rb->info, rows * GRS_INFO_STRIDE * sizeof(float)}};
  for (auto& v : views)
    if (std::strcmp(v.n, name) == 0) { *ptr = v.p; *bytes = v.b; return 0; }
  return grl_set_error(std::string("grl_replay_buffer: unknown buffer '") + name + "'");
}
