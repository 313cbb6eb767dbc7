// Rollout post-processing and optimiser step of the on-device learners (SURVEY.md §8f N1, BASELINE.json configs[3]).
// The reference trains with SB3's SAC, whose Adam step runs on the host side of a single environment (train_agent.py:82-88);
// its replay buffer has a device-resident counterpart in replay_kernels.cu.  The two kernels here serve the PPO rollout
// storage (k_gae) and every flat-bucket optimiser, PPO's and SAC's (k_adam):
//
//   k_gae   : generalised advantage estimation + returns over the [T][N] rollout storage, one thread per environment walking
//             its T transitions backwards (coalesced across N), plus the sum / sum of squares of the advantages (double
//             atomics) for the batch normalisation that follows.  Reads the simulator's reward / done records as stored.
//   k_adam  : Adam over ONE flat fp32 bucket that is at the same time the NCCL all-reduce buffer of the gradients
//             (parameters, gradients and moments are views into flat arrays: no concatenate / scatter-back), with the
//             1/world averaging of the all-reduced sum folded in; float4 vectorised, grid sized to the SM count.
//
// Both are HBM-bound elementwise passes (GAE: 13 B read + 8 B written per transition; Adam: 16 B read + 12 B written per
// parameter); ~1 M parameters and <= 1 M transitions per update keep them in the microsecond range.
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <string>

#include "../../include/b200_gripper_sim.h"

namespace {

thread_local std::string t_err;
int tfail(const std::string& m) { t_err = m; return 1; }

__global__ void k_gae(const float* __restrict__ rewards, const unsigned char* __restrict__ dones, const float* __restrict__ values,
                      float* __restrict__ adv, float* __restrict__ ret, double* __restrict__ moments, int T, int N, float gamma, float lam) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  double s1 = 0, s2 = 0;
  if (n < N) {
    float last = 0.0f, vnext = values[(size_t)T * N + n];
    for (int k = T - 1; k >= 0; k--) {
      const size_t i = (size_t)k * N + n;
      const float nd = dones[i] ? 0.0f : 1.0f, v = values[i];
      const float delta = rewards[i] + gamma * vnext * nd - v;
      last = delta + gamma * lam * nd * last;
      adv[i] = last;
      ret[i] = last + v;
      s1 += last; s2 += (double)last * last;
      vnext = v;
    }
  }
  if (moments) {
    for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
    if ((threadIdx.x & 31) == 0) { atomicAdd(moments, s1); atomicAdd(moments + 1, s2); }
  }
}

__global__ void k_adam(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long count,
                       float lr, float b1, float b2, float eps, float bc1, float bc2, float gscale, float weight_decay) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long n4 = count >> 2;
  float4* p4 = reinterpret_cast<float4*>(p);
  const float4* g4 = reinterpret_cast<const float4*>(g);
  float4* m4 = reinterpret_cast<float4*>(m);
  float4* v4 = reinterpret_cast<float4*>(v);
  auto upd = [&](float& pp, float gg, float& mm, float& vv) {
    gg = gg * gscale + weight_decay * pp;
    mm = b1 * mm + (1.0f - b1) * gg;
    vv = b2 * vv + (1.0f - b2) * gg * gg;
    pp -= lr * (mm / bc1) / (sqrtf(vv / bc2) + eps);  // torch.optim.Adam: denom = sqrt(v_hat) + eps
  };
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 pp = p4[i], gg = g4[i], mm = m4[i], vv = v4[i];
    upd(pp.x, gg.x, mm.x, vv.x); upd(pp.y, gg.y, mm.y, vv.y); upd(pp.z, gg.z, mm.z, vv.z); upd(pp.w, gg.w, mm.w, vv.w);
    p4[i] = pp; m4[i] = mm; v4[i] = vv;
  }
  for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) upd(p[i], g[i], m[i], v[i]);
}

}  // namespace

extern "C" const char* grl_last_error(void) { return t_err.c_str(); }
int grl_set_error(const std::string& m) { return tfail(m); }  // shared with replay_kernels.cu

extern "C" int32_t grl_gae(const float* rewards_dev, const uint8_t* dones_dev, const float* values_dev, float* adv_dev, float* ret_dev, double* moments_dev,
                           int32_t T, int32_t N, float gamma, float lam, void* stream) {
  if (!rewards_dev || !dones_dev || !values_dev || !adv_dev || !ret_dev) return tfail("grl_gae: null pointer");
  if (T <= 0 || N <= 0) return tfail("grl_gae: T and N must be positive");
  cudaStream_t st = (cudaStream_t)stream;
  if (moments_dev && cudaMemsetAsync(moments_dev, 0, 2 * sizeof(double), st) != cudaSuccess) return tfail("grl_gae: cudaMemsetAsync failed");
  k_gae<<<(N + 127) / 128, 128, 0, st>>>(rewards_dev, dones_dev, values_dev, adv_dev, ret_dev, moments_dev, T, N, gamma, lam);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : tfail(std::string("grl_gae: ") + cudaGetErrorString(e));
}

extern "C" int32_t grl_adam_step(float* params_dev, const float* grads_dev, float* exp_avg_dev, float* exp_avg_sq_dev, int64_t count, int32_t step,
                                 float lr, float beta1, float beta2, float eps, float grad_scale, float weight_decay, void* stream) {
  if (!params_dev || !grads_dev || !exp_avg_dev || !exp_avg_sq_dev) return tfail("grl_adam_step: null pointer");
  if (count <= 0 || step <= 0) return tfail("grl_adam_step: count and step must be positive");
  if ((((uintptr_t)params_dev | (uintptr_t)grads_dev | (uintptr_t)exp_avg_dev | (uintptr_t)exp_avg_sq_dev) & 15) != 0)
    return tfail("grl_adam_step: buffers must be 16-byte aligned");
  int dev = 0, nsm = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
  const double bc1 = 1.0 - std::pow((double)beta1, (double)step), bc2 = 1.0 - std::pow((double)beta2, (double)step);
  long long blocks = ((count >> 2) + 255) / 256;
  if (blocks > 8LL * nsm) blocks = 8LL * nsm;
  if (blocks < 1) blocks = 1;
  k_adam<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(params_dev, grads_dev, exp_avg_dev, exp_avg_sq_dev, count, lr, beta1, beta2, eps, (float)bc1, (float)bc2,
                                                       grad_scale, weight_decay);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : tfail(std::string("grl_adam_step: ") + cudaGetErrorString(e));
}
