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
// Layout: `capacity + 1` slots per environment, slot-major [S][N] like the PPO rollout storage; transition t of environment n
// lives in slot t % S.  The extra slot holds the pending observation, so `capacity` complete transitions stay sampleable once
// the ring has wrapped.
//
// Write modes, fixed by a buffer's first begin call:
//   lock-step (k_replay_begin / k_replay_add): every environment adds in every call; t is one host-side counter.
//   indexed (k_replay_begin_indexed / k_replay_add_indexed): the environments of an asynchronous pool advance at their own
//     rates, so each has its own device-side cursor added[n].  An add call lists the environments it writes; the first listing
//     after begin_indexed only records the observation (arms the environment), every later one completes a transition.
//     Sampling first scans min(added[n], capacity) into csum (k_replay_scan) and then draws a transition uniformly over all
//     complete ones: g < total, env = upper bound of g in csum.  With equal counts that is below(u0, N), the lock-step draw.
//     Bad ids and an empty buffer set bits of a sticky device error word (ERR_*), read and cleared by grl_replay_status.
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/b200_gripper_sim.h"

int grl_set_error(const std::string& m);  // train_kernels.cu: grl_last_error()'s message

enum { MODE_NONE = 0, MODE_LOCKSTEP, MODE_INDEXED };
enum { ERR_RANGE = 1, ERR_DUPLICATE = 2, ERR_EMPTY = 4 };  // bits of the sticky device error word

struct grl_replay {
  int K, S, N, C, H, W, A, her_reward, device;
  unsigned seed;
  long long img;     // bytes of one observation, a multiple of 16
  long long added;   // lock-step mode: complete transitions per environment ever added
  int mode;          // MODE_*: fixed by the first begin call
  unsigned long long calls;  // indexed mode: add calls so far (the stamp of the next one is calls + 1)
  uint8_t *obs, *next_obs, *done;
  float *actions, *reward, *info;
  long long *ep_end;    // [S][N] transition index of the episode's last transition, -1 while the episode is open
  long long *ep_start;  // [N]    first transition of each environment's open episode
  // indexed mode
  long long* env_added;     // [N] complete transitions of each environment ever added
  int* armed;               // [N] the environment's pending observation is recorded
  unsigned long long* stamp;  // [N] the last add call that wrote the environment (duplicate ids in one call)
  long long* csum;          // [N] inclusive prefix sum of min(env_added, K), written before every indexed sample
  int* err;                 // sticky ERR_* bits
};

namespace {

constexpr int THREADS = 256;

struct Ring {
  uint8_t *obs, *next_obs, *done;
  float *actions, *reward, *info;
  long long *ep_end, *ep_start;
  long long img, S;
  int N, A;
  long long *env_added, *csum;
  int *armed, *err;
  unsigned long long* stamp;
};

Ring ring_of(const grl_replay* r) {
  return Ring{r->obs, r->next_obs, r->done, r->actions, r->reward, r->info, r->ep_end, r->ep_start, r->img, r->S, r->N, r->A,
              r->env_added, r->csum, r->armed, r->err, r->stamp};
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

// copies environment n's observation obs[n] into slot `slot` (the pending observation)
__device__ inline void put_pending(const Ring& r, int n, long long slot, const uint8_t* __restrict__ obs) {
  const int4* src = reinterpret_cast<const int4*>(obs + (size_t)n * r.img);
  int4* dst = reinterpret_cast<int4*>(r.obs + ((size_t)slot * r.N + n) * r.img);
  for (long long i = threadIdx.x; i < r.img / 16; i += blockDim.x) dst[i] = __ldg(src + i);
}

// an explicit reset: closes environment n's open episode at its newest stored transition (added - 1), the next one starts at added
__device__ inline void restart_episode(const Ring& r, int n, long long added, long long K) {
  const long long start = r.ep_start[n];
  __syncthreads();  // every thread has read ep_start before thread 0 moves it
  if (added > start) close_episode(r, n, start, added - 1, K);
  if (threadIdx.x == 0) r.ep_start[n] = added;
}

__global__ void __launch_bounds__(THREADS) k_replay_begin(Ring r, const uint8_t* __restrict__ obs, long long added, long long K) {
  const int n = blockIdx.x;
  put_pending(r, n, added % r.S, obs);
  restart_episode(r, n, added, K);
}

__global__ void __launch_bounds__(THREADS) k_replay_begin_indexed(Ring r, long long K) {
  const int n = blockIdx.x;
  restart_episode(r, n, r.env_added[n], K);
  if (threadIdx.x == 0) r.armed[n] = 0;  // the environment's next listing in an add call records its observation
}

// Completes transition t of environment n from row n of the simulator's buffers (the whole block calls it): next_obs =
// terminal_obs on done, else obs; action, reward, done and info row; the episode's bookkeeping; then obs (the reset observation
// where done) becomes the pending observation of slot (t + 1) % S.
__device__ inline void add_transition(const Ring& r, int n, long long t, long long K, const float* __restrict__ actions,
                                      const float* __restrict__ reward, const uint8_t* __restrict__ done, const float* __restrict__ info,
                                      const uint8_t* __restrict__ obs, const uint8_t* __restrict__ terminal_obs) {
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

__global__ void __launch_bounds__(THREADS) k_replay_add(Ring r, const float* __restrict__ actions, const float* __restrict__ reward,
                                                       const uint8_t* __restrict__ done, const float* __restrict__ info,
                                                       const uint8_t* __restrict__ obs, const uint8_t* __restrict__ terminal_obs,
                                                       long long t, long long K) {
  add_transition(r, blockIdx.x, t, K, actions, reward, done, info, obs, terminal_obs);
}

// one block per listed id; reads row id of the simulator's per-environment buffers
__global__ void __launch_bounds__(THREADS) k_replay_add_indexed(Ring r, const int32_t* __restrict__ env_ids, const float* __restrict__ actions,
                                                               const float* __restrict__ reward, const uint8_t* __restrict__ done,
                                                               const float* __restrict__ info, const uint8_t* __restrict__ obs,
                                                               const uint8_t* __restrict__ terminal_obs, unsigned long long call, long long K) {
  __shared__ int s_go, s_armed;
  __shared__ long long s_t;
  const int id = env_ids[blockIdx.x];
  if (id < 0) return;  // a short recv's missing entries
  if (threadIdx.x == 0) {
    s_go = 0;
    if (id >= r.N) atomicOr(r.err, ERR_RANGE);
    else if (atomicExch(r.stamp + id, call) == call) atomicOr(r.err, ERR_DUPLICATE);  // an earlier block of this call has it
    else { s_go = 1; s_armed = r.armed[id]; s_t = r.env_added[id]; }
  }
  __syncthreads();
  if (!s_go) return;
  const long long t = s_t;
  if (!s_armed) {
    put_pending(r, id, t % r.S, obs);
    if (threadIdx.x == 0) r.armed[id] = 1;
    return;
  }
  add_transition(r, id, t, K, actions, reward, done, info, obs, terminal_obs);
  if (threadIdx.x == 0) r.env_added[id] = t + 1;
}

// csum[n] = sum of min(env_added[m], K) over m <= n: one block, each thread scans a contiguous run of environments
__global__ void __launch_bounds__(1024) k_replay_scan(Ring r, long long K) {
  __shared__ long long part[1024];
  const int per = (r.N + blockDim.x - 1) / blockDim.x, lo = threadIdx.x * per, hi = min(lo + per, r.N);
  long long s = 0;
  for (int n = lo; n < hi; n++) s += min(r.env_added[n], K);
  part[threadIdx.x] = s;
  __syncthreads();
  for (int d = 1; d < blockDim.x; d <<= 1) {  // Hillis-Steele inclusive scan of the per-thread sums
    const long long v = threadIdx.x >= d ? part[threadIdx.x - d] : 0;
    __syncthreads();
    part[threadIdx.x] += v;
    __syncthreads();
  }
  s = threadIdx.x ? part[threadIdx.x - 1] : 0;
  for (int n = lo; n < hi; n++) r.csum[n] = s += min(r.env_added[n], K);
}

struct SampleOut {
  uint8_t *obs, *next_obs, *done;
  float *actions, *reward, *desired, *achieved, *info;
  long long *index, *goal_index;
};

// INDEXED: `added` and `size` are ignored; the environment is drawn in proportion to its complete transitions (csum, written by
// k_replay_scan on the same stream), then the transition uniformly among them.  An empty buffer gives index = goal_index = -1.
template <bool INDEXED>
__global__ void __launch_bounds__(THREADS) k_replay_sample(Ring r, SampleOut o, long long added, long long size, unsigned seed,
                                                          unsigned long long draw, float her_ratio, int her_reward) {
  __shared__ long long s_row, s_grow;
  const int b = blockIdx.x;
  if (threadIdx.x == 0) {
    const unsigned base = sample_base(seed, draw, (unsigned)b);
    long long env = 0;
    if constexpr (INDEXED) {
      const long long total = r.csum[r.N - 1];
      if (total > 0) {
        const long long g = below(sample_u32(base, 0), total);
        int lo = 0, hi = r.N - 1;  // the first environment whose csum exceeds g
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (r.csum[mid] > g) hi = mid;
          else lo = mid + 1;
        }
        env = lo;
        added = r.env_added[env];
        size = r.csum[env] - (env ? r.csum[env - 1] : 0);
      } else {
        env = -1;
      }
    } else {
      env = below(sample_u32(base, 0), r.N);
    }
    if (INDEXED && env < 0) {  // nothing to sample
      atomicOr(r.err, ERR_EMPTY);
      s_row = -1;
    } else {
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
  }
  __syncthreads();
  const long long row = s_row, grow = s_grow;
  if (INDEXED && row < 0) {
    if (threadIdx.x == 0 && o.index) o.index[b] = -1;
    if (threadIdx.x == 0 && o.goal_index) o.goal_index[b] = -1;
    return;
  }
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
                  (void*)r->ep_start, (void*)r->env_added, (void*)r->armed, (void*)r->stamp, (void*)r->csum, (void*)r->err})
    if (p) cudaFree(p);
  cudaSetDevice(prev);
  delete r;
}

// refuses a call of the other write mode; otherwise fixes the buffer's mode to `mode`
int claim_mode(grl_replay* rb, int mode, const char* who) {
  if (rb->mode != MODE_NONE && rb->mode != mode)
    return grl_set_error(std::string(who) + ": the buffer is in " + (rb->mode == MODE_INDEXED ? "indexed" : "lock-step") +
                         " write mode; the two modes cannot be mixed on one buffer");
  rb->mode = mode;
  return 0;
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
                    cudaMalloc(&r->ep_end, rows * sizeof(long long)) == cudaSuccess && cudaMalloc(&r->ep_start, r->N * sizeof(long long)) == cudaSuccess &&
                    cudaMalloc(&r->env_added, r->N * sizeof(long long)) == cudaSuccess && cudaMalloc(&r->armed, r->N * sizeof(int)) == cudaSuccess &&
                    cudaMalloc(&r->stamp, r->N * sizeof(unsigned long long)) == cudaSuccess &&
                    cudaMalloc(&r->csum, r->N * sizeof(long long)) == cudaSuccess && cudaMalloc(&r->err, sizeof(int)) == cudaSuccess;
    if (!ok) {
      cudaGetLastError();
      return grl_set_error("grl_replay_create: cudaMalloc of " + std::to_string(rows) + " slots failed");
    }
    if (cudaMemset(r->ep_end, 0xff, rows * sizeof(long long)) != cudaSuccess || cudaMemset(r->ep_start, 0, r->N * sizeof(long long)) != cudaSuccess ||
        cudaMemset(r->env_added, 0, r->N * sizeof(long long)) != cudaSuccess || cudaMemset(r->armed, 0, r->N * sizeof(int)) != cudaSuccess ||
        cudaMemset(r->stamp, 0, r->N * sizeof(unsigned long long)) != cudaSuccess || cudaMemset(r->err, 0, sizeof(int)) != cudaSuccess)
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
  if (const int rc = claim_mode(rb, MODE_LOCKSTEP, "grl_replay_begin")) return rc;
  return on_device(rb->device, [&]() -> int {
    k_replay_begin<<<rb->N, THREADS, 0, (cudaStream_t)stream>>>(ring_of(rb), obs_dev, rb->added, rb->K);
    return launched("grl_replay_begin");
  });
}

extern "C" int32_t grl_replay_begin_indexed(grl_replay* rb, void* stream) {
  if (!rb) return grl_set_error("grl_replay_begin_indexed: null pointer");
  if (const int rc = claim_mode(rb, MODE_INDEXED, "grl_replay_begin_indexed")) return rc;
  return on_device(rb->device, [&]() -> int {
    k_replay_begin_indexed<<<rb->N, THREADS, 0, (cudaStream_t)stream>>>(ring_of(rb), rb->K);
    return launched("grl_replay_begin_indexed");
  });
}

extern "C" int32_t grl_replay_add(grl_replay* rb, const float* actions_dev, const float* reward_dev, const uint8_t* done_dev, const float* info_dev,
                                  const uint8_t* obs_dev, const uint8_t* terminal_obs_dev, void* stream) {
  if (!rb || !actions_dev || !reward_dev || !done_dev || !info_dev || !obs_dev || !terminal_obs_dev) return grl_set_error("grl_replay_add: null pointer");
  if (rb->mode == MODE_INDEXED) return grl_set_error("grl_replay_add: the buffer is in indexed write mode (grl_replay_add_indexed)");
  if (rb->mode != MODE_LOCKSTEP) return grl_set_error("grl_replay_add: call grl_replay_begin with the observations the actions were taken on first");
  if (misaligned(obs_dev) || misaligned(terminal_obs_dev)) return grl_set_error("grl_replay_add: obs and terminal_obs must be 16-byte aligned");
  return on_device(rb->device, [&]() -> int {
    k_replay_add<<<rb->N, THREADS, 0, (cudaStream_t)stream>>>(ring_of(rb), actions_dev, reward_dev, done_dev, info_dev, obs_dev, terminal_obs_dev,
                                                             rb->added, rb->K);
    const int rc = launched("grl_replay_add");
    if (rc == 0) rb->added++;
    return rc;
  });
}

extern "C" int32_t grl_replay_add_indexed(grl_replay* rb, const int32_t* env_ids_dev, int32_t count, const float* actions_dev, const float* reward_dev,
                                          const uint8_t* done_dev, const float* info_dev, const uint8_t* obs_dev, const uint8_t* terminal_obs_dev,
                                          void* stream) {
  if (!rb || !env_ids_dev || !actions_dev || !reward_dev || !done_dev || !info_dev || !obs_dev || !terminal_obs_dev)
    return grl_set_error("grl_replay_add_indexed: null pointer");
  if (rb->mode == MODE_LOCKSTEP) return grl_set_error("grl_replay_add_indexed: the buffer is in lock-step write mode (grl_replay_add)");
  if (rb->mode != MODE_INDEXED) return grl_set_error("grl_replay_add_indexed: call grl_replay_begin_indexed first");
  if (count < 0) return grl_set_error("grl_replay_add_indexed: count must not be negative");
  if (misaligned(obs_dev) || misaligned(terminal_obs_dev)) return grl_set_error("grl_replay_add_indexed: obs and terminal_obs must be 16-byte aligned");
  if (count == 0) return 0;
  return on_device(rb->device, [&]() -> int {
    k_replay_add_indexed<<<count, THREADS, 0, (cudaStream_t)stream>>>(ring_of(rb), env_ids_dev, actions_dev, reward_dev, done_dev, info_dev, obs_dev,
                                                                     terminal_obs_dev, rb->calls + 1, rb->K);
    const int rc = launched("grl_replay_add_indexed");
    if (rc == 0) rb->calls++;
    return rc;
  });
}

extern "C" int64_t grl_replay_size(const grl_replay* rb) {
  if (!rb) return -1;
  if (rb->mode == MODE_INDEXED) {
    grl_set_error("grl_replay_size: the environments of an indexed-mode buffer hold different counts; grl_replay_status gives the total");
    return -1;
  }
  return rb->added < rb->K ? rb->added : rb->K;
}

extern "C" int32_t grl_replay_status(grl_replay* rb, int64_t* transitions) {
  if (!rb || !transitions) return grl_set_error("grl_replay_status: null pointer");
  if (rb->mode != MODE_INDEXED) {
    *transitions = (rb->added < rb->K ? rb->added : rb->K) * (int64_t)rb->N;
    return 0;
  }
  return on_device(rb->device, [&]() -> int {
    std::vector<long long> added(rb->N);
    int err = 0;
    if (cudaDeviceSynchronize() != cudaSuccess || cudaMemcpy(added.data(), rb->env_added, rb->N * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess ||
        cudaMemcpy(&err, rb->err, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess || (err && cudaMemset(rb->err, 0, sizeof(int)) != cudaSuccess)) {
      const cudaError_t e = cudaGetLastError();
      return grl_set_error(std::string("grl_replay_status: ") + cudaGetErrorString(e));
    }
    long long total = 0;
    for (long long a : added) total += a < rb->K ? a : rb->K;
    *transitions = total;
    if (!err) return 0;
    std::string m = "grl_replay_status:";
    if (err & ERR_RANGE) m += " an add_indexed call listed an environment id >= num_envs (skipped);";
    if (err & ERR_DUPLICATE) m += " an add_indexed call listed an environment id twice (written once);";
    if (err & ERR_EMPTY) m += " a sample found no complete transition (its rows have index -1);";
    m.pop_back();
    return grl_set_error(m);
  });
}

extern "C" int32_t grl_replay_sample(grl_replay* rb, int32_t batch, float her_ratio, uint64_t draw, uint8_t* obs_dev, uint8_t* next_obs_dev,
                                     float* actions_dev, float* reward_dev, uint8_t* done_dev, float* desired_goal_dev, float* achieved_goal_dev,
                                     float* info_dev, int64_t* index_dev, int64_t* goal_index_dev, void* stream) {
  if (!rb || !obs_dev || !next_obs_dev || !actions_dev || !reward_dev || !done_dev || !desired_goal_dev || !achieved_goal_dev)
    return grl_set_error("grl_replay_sample: null pointer");
  const bool indexed = rb->mode == MODE_INDEXED;
  const long long size = indexed ? 0 : grl_replay_size(rb);
  if (!indexed && size <= 0) return grl_set_error("grl_replay_sample: the buffer holds no complete transition");
  if (batch <= 0) return grl_set_error("grl_replay_sample: batch size must be positive");
  if (!(her_ratio >= 0.0f && her_ratio <= 1.0f)) return grl_set_error("grl_replay_sample: her_ratio must lie in [0, 1]");
  if (misaligned(obs_dev) || misaligned(next_obs_dev)) return grl_set_error("grl_replay_sample: obs and next_obs must be 16-byte aligned");
  const SampleOut o{obs_dev, next_obs_dev, done_dev, actions_dev, reward_dev, desired_goal_dev, achieved_goal_dev, info_dev,
                    reinterpret_cast<long long*>(index_dev), reinterpret_cast<long long*>(goal_index_dev)};
  return on_device(rb->device, [&]() -> int {
    const cudaStream_t st = (cudaStream_t)stream;
    if (indexed) {
      k_replay_scan<<<1, 1024, 0, st>>>(ring_of(rb), rb->K);
      if (const int rc = launched("grl_replay_sample")) return rc;
      k_replay_sample<true><<<batch, THREADS, 0, st>>>(ring_of(rb), o, 0, 0, rb->seed, (unsigned long long)draw, her_ratio, rb->her_reward);
    } else {
      k_replay_sample<false><<<batch, THREADS, 0, st>>>(ring_of(rb), o, rb->added, size, rb->seed, (unsigned long long)draw, her_ratio, rb->her_reward);
    }
    return launched("grl_replay_sample");
  });
}

extern "C" int32_t grl_replay_buffer(grl_replay* rb, const char* name, void** ptr, uint64_t* bytes) {
  if (!rb || !name || !ptr || !bytes) return grl_set_error("grl_replay_buffer: null pointer");
  const uint64_t rows = (uint64_t)rb->S * rb->N;
  struct { const char* n; void* p; uint64_t b; } views[] = {
      {"obs", rb->obs, rows * rb->img}, {"next_obs", rb->next_obs, rows * rb->img}, {"actions", rb->actions, rows * rb->A * sizeof(float)},
      {"reward", rb->reward, rows * sizeof(float)}, {"done", rb->done, rows}, {"info", rb->info, rows * GRS_INFO_STRIDE * sizeof(float)},
      {"added", rb->env_added, (uint64_t)rb->N * sizeof(long long)}};
  for (auto& v : views)
    if (std::strcmp(v.n, name) == 0) { *ptr = v.p; *bytes = v.b; return 0; }
  return grl_set_error(std::string("grl_replay_buffer: unknown buffer '") + name + "'");
}
