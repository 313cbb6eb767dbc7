// Rollout-time policy inference on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a only.
//
// Network (reference models/feature_extractor.py:19-49 `AugmentedNatureCNN` + the stable-baselines3 SAC actor built by
// train_agent.py:18-20 with net_arch=[256,256]):
//   obs u8 [N,C,H,W] --/255--> conv 8x8 s4 (C-1 -> 32) ReLU -> conv 4x4 s2 (32 -> 64) ReLU -> conv 3x3 s1 (64 -> 64) ReLU
//   -> flatten -> linear (-> 512) ReLU -> concat obs[:, C-1, 0, 0:2]/255 (514) -> 256 ReLU -> 256 ReLU -> mu | log_std -> tanh
//
// One forward is five kernels.  Which conv kernels run depends only on the observation shape, fixed at grp_create:
//   64 x 64 observations with 4 image planes (the reference's full observation), the descriptor-addressed chain:
//     k_conv1_ws          conv1 WITHOUT im2col: the tensor core reads the fp16 image through a no-swizzle shared-memory descriptor,
//                         16 MMAs (M 128, N 96 = W | Wa | Wb) per image; warp-specialised (TMA producer, converters, issuer, epilogue)
//     k_conv_direct<2|3>  conv2 / conv3 WITHOUT im2col: the previous layer's padded, pre-swizzled activations arrive by one bulk copy
//                         per image pair and every k-block is a start address inside that copy
//   any other shape (e.g. full_observation=False: 3 image planes), the generic chain:
//     k_layer<CONV1 | CONV2 | CONV3>  the implicit-GEMM layer described below, gathering its A operand from dense NHWC activations
//   every shape:
//     k_layer<DENSE>      the linear layer (+ the two direct features)
//     k_mlp_fused         latent_pi.0, latent_pi.2 and the mu | log_std head; hidden activations TMEM -> registers -> shared memory
// k_layer<MODE, BN, EPI> is round 1's generic layer: an implicit GEMM  D[128 x BN] += A[128 x 64] * W[BN x 64]^T per k-block, with
//   * A gathered by the CTA's threads straight from the previous layer's activations (im2col on the fly, NHWC bf16; the
//     first layer reads the uint8 observation planes and converts) into the canonical K-major SWIZZLE_128B shared-memory
//     layout that tcgen05.mma reads through a shared-memory descriptor,
//   * W (bf16, K-major, pre-permuted to the gather order on the host) staged the same way,
//   * one elected thread issuing tcgen05.mma.cta_group::1.kind::f16 (M=128, N=BN, K=16) into a TMEM accumulator and
//     tcgen05.commit-ing each stage to an mbarrier, so the gather of k-block i+1.. overlaps the MMAs of k-block i
//     (3-stage ring),
//   * the epilogue reading the accumulator back with tcgen05.ld (32 lanes x 16 columns per warp at a time), applying
//     scale/bias/ReLU and writing bf16 NHWC rows for the next layer.
// No cuBLAS / cuDNN / CUTLASS calls; descriptor bit layouts follow the PTX ISA (matrix-descriptor and instruction-descriptor
// tables for tcgen05.mma).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/b200_gripper_sim.h"

namespace grp {

enum Mode { DENSE = 0, CONV1 = 1, CONV2 = 2, CONV3 = 3 };
enum Epi { EPI_RELU = 0, EPI_FEATURES = 1 };

constexpr int BM = 128;      // rows of A per CTA = TMEM lanes = UMMA M
constexpr int BK = 64;       // bf16 elements per k-block = one 128-byte swizzle row
constexpr int LAYER_STAGES = 3;  // k_layer's ring of staged k-blocks
constexpr int THREADS = 128;
constexpr int FEAT_LD = 576;  // 512 CNN features + 2 direct features, zero padded to a multiple of BK
constexpr int HEAD_N = 16;    // mu rows 0..A-1, log_std rows 8..8+A-1

struct LayerArgs {
  const void* A;             // activations of the previous layer (u8 observation for CONV1, bf16 otherwise)
  const __nv_bfloat16* W;    // [N_total][K] bf16, K-major
  const float* bias;         // [N_total]
  __nv_bfloat16* out;        // [M][ldo] bf16 (EPI_RELU / EPI_FEATURES)
  int M, K, lda, ldo;
  float scale;               // accumulator scale before the bias (1/255 folds the observation normalisation into conv1)
  int C, H, W_;              // observation planes (CONV1, EPI_FEATURES)
  int ih, iw, oh, ow;        // input / output feature-map size of a convolution
  const unsigned char* obs;  // EPI_FEATURES: the two direct features come from obs[:, C-1, 0, 0:2]
};

// ------------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  const uint32_t a = smem_u32(bar);
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(a), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory"); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]^T, bf16 x bf16 -> fp32
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// the same with the descriptors as 32-bit halves (only the low word — the 14-bit start address — changes between the MMAs of a
// tile: one 32-bit add per operand instead of a 64-bit one) and the accumulate flag as a compile-time constant
template <int ACC>
__device__ __forceinline__ void umma_bf16_lo(uint32_t tmem_d, uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(tmem_d), "r"(alo), "r"(ahi), "r"(blo), "r"(bhi), "r"(idesc), "n"(ACC)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 16 consecutive fp32 columns of the accumulator -> 16 registers per thread (thread t = lane 32*(warp%4)+t)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
        "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
}
// the same for 32 consecutive columns
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
        "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; i++) v[i] = __uint_as_float(r[i]);
}

// shared-memory matrix descriptor: K-major operand, SWIZZLE_128B (rows of 128 bytes, 8-row groups 1024 bytes apart)
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);  // start address, 16-byte units            bits [0,14)
  d |= (uint64_t)1 << 16;                    // leading byte offset (unused for swizzled K-major)   [16,30)
  d |= (uint64_t)(1024 >> 4) << 32;          // stride byte offset between 8-row groups             [32,46)
  d |= (uint64_t)1 << 46;                    // descriptor version (Blackwell)                      [46,48)
  d |= (uint64_t)2 << 61;                    // layout type SWIZZLE_128B                            [61,64)
  return d;
}
// instruction descriptor for kind::f16: D = fp32, A = B = bf16 (format 1) or fp16 (format 0), both K-major, M x N
__host__ __device__ constexpr uint32_t instr_desc_f16(int m, int n, bool bf16) {
  return (1u << 4) | ((bf16 ? 1u : 0u) << 7) | ((bf16 ? 1u : 0u) << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// 16-byte asynchronous global -> shared copy (LDGSTS); `valid == false` zero-fills the destination (rows >= M)
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool valid) {
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Implicit-GEMM addressing, split into a per-row part (computed once per CTA: the integer divisions) and a per-k-block part.
// Element offset (in units of the input type) of row `r`, chunk `ch` at k-block 0; rows >= M return -1.
//   DENSE  row-major [M][lda]: chunk = 8 consecutive bf16
//   CONV1  uint8 planes [n][C][ih][iw], 8x8 stride 4, K order (c, ky, kx) = torch's [Cin][8][8]: k-block = input channel,
//          chunk = kernel row ky, the 8 pixels of one image row
//   CONV2  NHWC bf16, 32 channels, 4x4 stride 2, K order (ky, kx, c): k-block = (ky, kx pair) = 2 adjacent pixels = 128 bytes
//   CONV3  NHWC bf16, 64 channels, 3x3 stride 1: k-block = one kernel tap = one pixel = 128 bytes
template <int MODE>
__device__ __forceinline__ int a_row_base(const LayerArgs& a, int r, int ch) {
  if (r >= a.M) return -1;
  if (MODE == DENSE) return r * a.lda + ch * 8;
  const int per = a.oh * a.ow, n = r / per, p = r - n * per, oy = p / a.ow, ox = p - oy * a.ow;
  if (MODE == CONV1) return ((n * a.C) * a.ih + (4 * oy + ch)) * a.iw + 4 * ox;
  if (MODE == CONV2) return ((n * a.ih + 2 * oy) * a.iw + 2 * ox) * 32 + ch * 8;
  return ((n * a.ih + oy) * a.iw + ox) * 64 + ch * 8;
}
template <int MODE>
__device__ __forceinline__ int a_kb_offset(const LayerArgs& a, int kb) {
  if (MODE == DENSE) return kb * BK;
  if (MODE == CONV1) return kb * a.ih * a.iw;
  if (MODE == CONV2) return ((kb >> 1) * a.iw + (kb & 1) * 2) * 32;
  return ((kb / 3) * a.iw + (kb % 3)) * 64;
}
// eight uint8 -> eight fp16, exact: the byte lands in the mantissa of 1024.0 (0x6400 | b = 1024 + b), then 1024 is subtracted
__device__ __forceinline__ uint32_t u8x2_to_f16x2(uint32_t p, uint32_t sel) {
  uint32_t v;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(v) : "r"(p), "r"(0x64646464u), "r"(sel));
  __half2 h = __hsub2(*reinterpret_cast<__half2*>(&v), __half2half2(__ushort_as_half((unsigned short)0x6400)));
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint4 u8x8_to_f16x8(uint2 raw) {
  // prmt selectors: result bytes {b0, 0x64, b1, 0x64} -> halves (0x6400 | b0), (0x6400 | b1); source bytes 4..7 are the constant
  return make_uint4(u8x2_to_f16x2(raw.x, 0x4140u), u8x2_to_f16x2(raw.x, 0x4342u), u8x2_to_f16x2(raw.y, 0x4140u), u8x2_to_f16x2(raw.y, 0x4342u));
}

template <int BN>
__host__ __device__ constexpr int tmem_cols() { return BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256; }
template <int BN>
__host__ __device__ constexpr size_t layer_smem_bytes() { return (size_t)LAYER_STAGES * (BM * 128 + BN * 128) + 1024; }

template <int MODE, int BN, int EPI>
__global__ void __launch_bounds__(THREADS) k_layer(const LayerArgs a) {
  constexpr int STAGES = LAYER_STAGES;
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bar_stage[STAGES];
  __shared__ uint64_t bar_done;
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;                         // STAGES x [128 rows x 128 B]
  uint8_t* sB = smem + STAGES * BM * 128;     // STAGES x [BN rows x 128 B]
  __shared__ __align__(16) float sbias[BN];  // this CTA's slice of the bias (a parameter, not an activation: safe to read before griddepcontrol.wait)
  for (int i = tid; i < BN; i += THREADS) sbias[i] = __ldg(a.bias + blockIdx.y * BN + i);
  if (tid == 0) {
    for (int s = 0; s < STAGES; s++) mbar_init(&bar_stage[s], 1);
    mbar_init(&bar_done, 1);
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(&tmem_base_s, tmem_cols<BN>());
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // Programmatic dependent launch: this grid may have started while the previous layer was still running (its barrier
  // initialisation and TMEM allocation above overlap that layer's tail).  Let the next layer do the same, then wait for the
  // previous grid to complete and flush before the first read of its activations.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const uint32_t tmem = tmem_base_s;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int nkb = a.K / BK;
  constexpr uint32_t idesc = instr_desc_f16(BM, BN, MODE != CONV1);

  // elected thread: the four K=16 MMAs of one staged k-block, committed to the stage's barrier
  auto issue_mma = [&](int kb) {
    const int s = kb % STAGES;
    tc_fence_after();
    const uint32_t aaddr = smem_u32(sA + s * BM * 128), baddr = smem_u32(sB + s * BN * 128);
#pragma unroll
    for (int k = 0; k < BK / 16; k++) {
      const uint64_t ad = smem_desc_sw128(aaddr + k * 32), bd = smem_desc_sw128(baddr + k * 32);
      umma_bf16(tmem, ad, bd, idesc, (kb | k) != 0);
    }
    umma_commit(&bar_stage[s]);
    if (kb == nkb - 1) umma_commit(&bar_done);
  };
  // W tile of k-block kb -> stage (asynchronous copies, swizzled destination)
  auto copy_w = [&](int kb) {
    const uint32_t dB = smem_u32(sB + (kb % STAGES) * BN * 128);
#pragma unroll
    for (int i = 0; i < (BN * 8 + THREADS - 1) / THREADS; i++) {
      const int c = i * THREADS + tid, row = c >> 3, ch = c & 7;
      if (c < BN * 8) cp_async16(dB + row * 128 + ((ch ^ (row & 7)) << 4), a.W + (size_t)(n0 + row) * a.K + kb * BK + ch * 8, true);
    }
  };

  // this thread's 8 (row, chunk) pairs: input offset at k-block 0 and swizzled offset inside a stage (constant over k-blocks)
  int rbase[BM * 8 / THREADS], soff[BM * 8 / THREADS];
#pragma unroll
  for (int i = 0; i < BM * 8 / THREADS; i++) {
    // bf16 layers: 8 consecutive threads copy the 8 chunks (128 contiguous bytes) of one row.  conv1: one thread per row and
    // chunk i = kernel row i, so a warp's 4-byte loads walk along an image row (2-3 cache lines per request instead of 8).
    const int c = i * THREADS + tid, row = MODE == CONV1 ? tid : c >> 3, ch = MODE == CONV1 ? i : c & 7;
    rbase[i] = a_row_base<MODE>(a, m0 + row, ch);
    soff[i] = row * 128 + ((ch ^ (row & 7)) << 4);
  }

  if (MODE == CONV1) {
    // The observation is uint8 and has to pass through registers (u8 -> fp16 is exact; this layer's weights are fp16 too).  All the raw loads of up to four
    // k-blocks (= input channels) are issued before the first use, so a CTA pays the global-memory latency once, not
    // once per k-block.
    constexpr int PRE = 4;
    const unsigned char* obs = reinterpret_cast<const unsigned char*>(a.A);
    const int plane = a_kb_offset<CONV1>(a, 1);
#pragma unroll 1
    for (int kb0 = 0; kb0 < nkb; kb0 += PRE) {
      uint2 raw[PRE][BM * 8 / THREADS];
#pragma unroll
      for (int i = 0; i < BM * 8 / THREADS; i++) {
        const int base = rbase[i];
#pragma unroll
        for (int j = 0; j < PRE; j++) {
          raw[j][i] = make_uint2(0, 0);
          if (base >= 0 && kb0 + j < nkb) {
            const unsigned char* src = obs + base + (kb0 + j) * plane;
            raw[j][i] = make_uint2(__ldg(reinterpret_cast<const uint32_t*>(src)), __ldg(reinterpret_cast<const uint32_t*>(src + 4)));
          }
        }
      }
#pragma unroll
      for (int j = 0; j < PRE; j++) {
        const int kb = kb0 + j;
        if (kb < nkb) {
          const int s = kb % STAGES;
          if (kb >= STAGES) {  // the MMAs that read this stage (k-block kb - STAGES) must have retired
            mbar_wait(&bar_stage[s], ((kb / STAGES) - 1) & 1);
            tc_fence_after();
          }
          copy_w(kb);
          cp_async_commit();
          uint8_t* dA = sA + s * BM * 128;
#pragma unroll
          for (int i = 0; i < BM * 8 / THREADS; i++) *reinterpret_cast<uint4*>(dA + soff[i]) = u8x8_to_f16x8(raw[j][i]);
          cp_async_wait<0>();
          fence_async_smem();  // generic-proxy writes -> visible to the tensor core's async proxy
          __syncthreads();
          if (tid == 0) issue_mma(kb);
        }
      }
    }
  } else {
    // bf16 activations: A and W tiles are straight 16-byte copies, so they go global -> shared asynchronously (LDGSTS),
    // STAGES - 1 k-blocks ahead of the MMAs; no registers, no per-k-block latency exposure.
    const __nv_bfloat16* act = reinterpret_cast<const __nv_bfloat16*>(a.A);
    auto copy_stage = [&](int kb) {
      const uint32_t dA = smem_u32(sA + (kb % STAGES) * BM * 128);
      const int koff = a_kb_offset<MODE>(a, kb);
#pragma unroll
      for (int i = 0; i < BM * 8 / THREADS; i++) {
        const bool valid = rbase[i] >= 0;
        cp_async16(dA + soff[i], valid ? act + rbase[i] + koff : act, valid);
      }
      copy_w(kb);
    };
#pragma unroll
    for (int kb = 0; kb < STAGES - 1; kb++) {
      if (kb < nkb) copy_stage(kb);
      cp_async_commit();
    }
#pragma unroll 1
    for (int kb = 0; kb < nkb; kb++) {
      const int kn = kb + STAGES - 1;  // refill the stage that k-block kb - 1 used, once its MMAs have retired
      if (kn < nkb) {
        if (kb >= 1) {
          mbar_wait(&bar_stage[(kb - 1) % STAGES], ((kb - 1) / STAGES) & 1);
          tc_fence_after();
        }
        copy_stage(kn);
      }
      cp_async_commit();
      cp_async_wait<STAGES - 1>();  // k-block kb has landed (this thread's copies; the barrier below covers the others)
      fence_async_smem();
      __syncthreads();
      if (tid == 0) issue_mma(kb);
    }
  }
  mbar_wait(&bar_done, 0);
  tc_fence_after();
  __syncwarp();

  // ---- epilogue: thread t of warp w owns accumulator row 32*w + t
  const int row = m0 + warp * 32 + lane;
  const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
  for (int c0 = 0; c0 < BN; c0 += 16) {
    float v[16];
    tmem_ld16(trow + c0, v);
    if (row < a.M) {
      uint32_t o[8];
      float bv[16];  // four 16-byte broadcast loads instead of sixteen scalar ones
#pragma unroll
      for (int k = 0; k < 4; k++) *reinterpret_cast<float4*>(bv + 4 * k) = *reinterpret_cast<const float4*>(sbias + c0 + 4 * k);
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const float x = fmaxf(fmaf(v[2 * k], a.scale, bv[2 * k]), 0.0f);
        const float y = fmaxf(fmaf(v[2 * k + 1], a.scale, bv[2 * k + 1]), 0.0f);
        o[k] = pack_bf16(x, y);
      }
      uint4* dst = reinterpret_cast<uint4*>(a.out + (size_t)row * a.ldo + n0 + c0);
      dst[0] = make_uint4(o[0], o[1], o[2], o[3]);
      dst[1] = make_uint4(o[4], o[5], o[6], o[7]);
    }
  }
  if (EPI == EPI_FEATURES && blockIdx.y == 0 && row < a.M) {
    // feature_extractor.py:42,48 — the two direct features ride behind the 512 CNN features (then zero padding)
    const unsigned char* p = a.obs + ((size_t)row * a.C + (a.C - 1)) * a.H * a.W_;
    uint4* dst = reinterpret_cast<uint4*>(a.out + (size_t)row * a.ldo + 512);
    dst[0] = make_uint4(pack_bf16((float)p[0] * (1.0f / 255.0f), (float)p[1] * (1.0f / 255.0f)), 0, 0, 0);
#pragma unroll
    for (int k = 1; k < (FEAT_LD - 512) / 8; k++) dst[k] = make_uint4(0, 0, 0, 0);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, tmem_cols<BN>());
}


// ------------------------------------------------------------------------------------------------ conv1 without im2col
// The 8x8 stride-4 convolution read straight off the image by the tensor core's shared-memory descriptor — no im2col copy.
// With K ordered (c, ky, kx), the K row of output pixel (oy, ox) for one (c, ky) is 8 consecutive pixels of image row
// 4*oy + ky starting at pixel 4*ox: 16 bytes of fp16.  The canonical K-major layout WITHOUT swizzle is made of 8-row x 16-byte
// core matrices whose rows are 16 bytes apart: the eight EVEN output pixels of a row (ox = 2r -> pixels 8r .. 8r + 7, chunk r)
// are exactly one fp16 image row, i.e. one core matrix already sits in the image as it is.  The next core matrix along K
// (ky + 1) is the next image row (leading byte offset = 128), the next 8-row group along M (oy + 1) is four image rows on
// (stride byte offset = 512).  One MMA (M = 128, K = 16) therefore covers 16 x 8 chunk rows for two kernel rows of one
// channel, 16 MMAs the whole K = 256.
// The ODD output pixels (ox = 2r + 1) need the 8 pixels from 8r + 4 on: the upper half of chunk r and the lower half of chunk
// r + 1 — not addressable as one row (descriptors have 16-byte granularity).  They are computed from whole chunks with
// zero-padded weights: odd(r) = chunk r x Wa + chunk r + 1 x Wb with Wa = [0 0 0 0 w0 w1 w2 w3], Wb = [w4 w5 w6 w7 0 0 0 0].
// All three products of a chunk row share the A operand, so they are ONE MMA with N = 96: B = [W ; Wa ; Wb], accumulator
// columns 0-31 = even(r), 32-63 = chunk r x Wa, 64-95 = chunk r x Wb, and the epilogue adds column block 2 of accumulator row
// m + 1 (a register shuffle from the next lane: rows are lanes) to column block 1 of row m.  16 MMAs per image; the image is read
// from shared memory once per 96 output columns (one N = 32 MMA per product was bound by the tensor core's operand reads,
// 240 KB per image); ONE fp16 copy of the image, one 16-byte store per 8-pixel chunk instead of 7 200 im2col chunks per image.
constexpr int CD_STAGE = 4 * 64 * 64 * 2 + 1024;  // the fp16 copy of the four planes + slack (group 15 of the last plane reads 512 B past it)
constexpr int CD_W = 4 * 96 * 128;                // 4 k-blocks (= input channels) x [96 rows = W | Wa | Wb] x 128 B, SWIZZLE_128B

// shared-memory matrix descriptor: K-major operand, no swizzle (8 x 16-byte core matrices; LBO = K step, SBO = 8-row group step)
__device__ __forceinline__ uint64_t smem_desc_nosw(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(lbo_bytes >> 4) << 16;
  d |= (uint64_t)(sbo_bytes >> 4) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}

// Warp-specialised: converting the next image, multiplying the current one and writing out the previous one are three different
// sets of warps that meet only at mbarriers.  With one set of warps doing the three jobs one after the other between block
// barriers, 46 % of the stall samples sat at __syncthreads and the tensor pipe was active 34 % of the time.
//   warp  17     producer: the image's four uint8 planes (16 KB, contiguous) by cp.async.bulk into a 4-deep raw ring — 64 KB per SM in
//                flight from HBM: with register prefetch two images ahead the kernel was bound by memory latency (1.7 TB/s)
//   warps 0-7    converters: raw ring -> fp16 copy of image k in stage k % 3, fence.proxy.async, one arrive per warp on full[stage]
//   warp  16     MMA issuer: waits full[stage] and tempty[acc], 16 x tcgen05.mma (N = 96), tcgen05.commit -> empty[stage], tfull[acc]
//   warps 8-15   epilogue: tcgen05.ld of accumulator k % 2 (even | Wa | Wb column blocks), arrive tempty[acc], lane shuffle for the
//                odd columns, bias + ReLU, bf16, stores in the layout conv2 reads
constexpr int CW_THREADS = 18 * 32;
constexpr int CW_STAGES = 3;       // fp16 image copies
constexpr int CW_ACC = 2;          // TMEM accumulators (128 columns each; 4 measured no faster: the kernel is bound by the issue rate of its 16 worker warps)
constexpr int CW_RAW = 4;          // uint8 images in flight from HBM (16 KB each): 64 KB per SM outstanding
constexpr size_t CW_SMEM = CD_W + CW_STAGES * CD_STAGE + CW_RAW * 16384 + 1024;

__global__ void __launch_bounds__(CW_THREADS, 1) k_conv1_ws(const LayerArgs a, int nimg) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bar_full[CW_STAGES], bar_empty[CW_STAGES], bar_tfull[CW_ACC], bar_tempty[CW_ACC], bar_rfull[CW_RAW], bar_rempty[CW_RAW];
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sB = smem;                                   // [4 k-blocks][96 rows: W | Wa | Wb][128 B]
  uint8_t* st0 = smem + CD_W;                           // stage s: the fp16 image at st0 + s * CD_STAGE
  uint8_t* raw0 = st0 + CW_STAGES * CD_STAGE;           // raw ring: the four uint8 planes of an image, 16 KB each
  if (tid == 0) {
    for (int i = 0; i < CW_STAGES; i++) { mbar_init(&bar_full[i], 8); mbar_init(&bar_empty[i], 1); }
    for (int i = 0; i < CW_ACC; i++) { mbar_init(&bar_tfull[i], 1); mbar_init(&bar_tempty[i], 8); }
    for (int i = 0; i < CW_RAW; i++) { mbar_init(&bar_rfull[i], 1); mbar_init(&bar_rempty[i], 8); }
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(&tmem_base_s, 128 * CW_ACC);  // accumulator t: columns 128 t .. 128 t + 95
  for (int i = tid; i < 4 * 96 * 8; i += CW_THREADS) {  // weights: parameters, staged before the dependency wait
    const int kb = i / 768, c = i - kb * 768, row = c >> 3, ch = c & 7;
    cp_async16(smem_u32(sB + kb * 96 * 128 + row * 128 + ((ch ^ (row & 7)) << 4)), a.W + (size_t)row * a.K + kb * BK + ch * 8, true);
  }
  cp_async_commit();
  for (int i = tid; i < CW_STAGES * 1024 / 16; i += CW_THREADS) *reinterpret_cast<uint4*>(st0 + (i >> 6) * CD_STAGE + (CD_STAGE - 1024) + (i & 63) * 16) = make_uint4(0, 0, 0, 0);
  cp_async_wait<0>();
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const uint32_t tmem = tmem_base_s;
  const int stride = gridDim.x;
  if (warp == 17) {
    // ---- producer: the image planes (one contiguous 16 KB block of the [n][C][64][64] uint8 tensor) by bulk copy, CW_RAW images ahead
    if (lane == 0) {
      const unsigned char* obs = reinterpret_cast<const unsigned char*>(a.A);
      const size_t img_bytes = (size_t)a.C * 4096;
      int k = 0;
#pragma unroll 1
      for (int n = blockIdx.x; n < nimg; n += stride, k++) {
        const int rs = k % CW_RAW;
        mbar_wait(&bar_rempty[rs], ((k / CW_RAW) & 1) ^ 1);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&bar_rfull[rs])), "r"(16384) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(raw0 + rs * 16384)), "l"(obs + (size_t)n * img_bytes), "r"(16384), "r"(smem_u32(&bar_rfull[rs])) : "memory");
      }
    }
  } else if (warp < 8) {
    // ---- converters: uint8 -> fp16, chunk q = 8 pixels at byte 8 q of the raw image, byte 16 q of the copy
    int k = 0;
#pragma unroll 1
    for (int n = blockIdx.x; n < nimg; n += stride, k++) {
      const int s = k % CW_STAGES, rs = k % CW_RAW;
      mbar_wait(&bar_rfull[rs], (k / CW_RAW) & 1);
      uint2 raw[8];
#pragma unroll
      for (int j = 0; j < 8; j++) raw[j] = *reinterpret_cast<const uint2*>(raw0 + rs * 16384 + (tid + 256 * j) * 8);
      mbar_wait(&bar_empty[s], ((k / CW_STAGES) & 1) ^ 1);
      uint8_t* E = st0 + s * CD_STAGE;
#pragma unroll
      for (int j = 0; j < 8; j++) *reinterpret_cast<uint4*>(E + (tid + 256 * j) * 16) = u8x8_to_f16x8(raw[j]);
      fence_async_smem();
      __syncwarp();
      if (lane == 0) { mbar_arrive(&bar_full[s]); mbar_arrive(&bar_rempty[rs]); }
    }
  } else if (warp == 16) {
    // ---- MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = instr_desc_f16(BM, 96, false);
      const uint64_t b0 = smem_desc_sw128(smem_u32(sB));
      const uint32_t blo = (uint32_t)b0, bhi = (uint32_t)(b0 >> 32);
      int k = 0;
#pragma unroll 1
      for (int n = blockIdx.x; n < nimg; n += stride, k++) {
        const int s = k % CW_STAGES, t = k % CW_ACC;
        mbar_wait(&bar_tempty[t], ((k / CW_ACC) & 1) ^ 1);
        mbar_wait(&bar_full[s], (k / CW_STAGES) & 1);
        tc_fence_after();
        const uint64_t a0 = smem_desc_nosw(smem_u32(st0 + s * CD_STAGE), 128, 512);
        const uint32_t alo = (uint32_t)a0, ahi = (uint32_t)(a0 >> 32), td = tmem + t * 128;
#pragma unroll
        for (int c = 0; c < 4; c++)
#pragma unroll
          for (int kyp = 0; kyp < 4; kyp++) {
            if ((c | kyp) == 0) umma_bf16_lo<0>(td, alo + ((c * 8192 + kyp * 256) >> 4), ahi, blo + ((c * 96 * 128 + kyp * 32) >> 4), bhi, idesc);
            else umma_bf16_lo<1>(td, alo + ((c * 8192 + kyp * 256) >> 4), ahi, blo + ((c * 96 * 128 + kyp * 32) >> 4), bhi, idesc);
          }
        umma_commit(&bar_empty[s]);
        umma_commit(&bar_tfull[t]);
      }
    }
  } else {
    // ---- epilogue: accumulator row m = 32 (warp % 4) + lane = 8 oy + r, output channels 16 half .. + 15 of pixels ox = 2r and 2r + 1
    const int ew = warp - 8, half = ew >> 2, em = 32 * (ew & 3) + lane, eoy = em >> 3, er = em & 7;
    const bool evalid = eoy < 15;
    float eb[16];
#pragma unroll
    for (int i = 0; i < 16; i++) eb[i] = __ldg(a.bias + half * 16 + i);
    const float escale = a.scale;
    int k = 0;
#pragma unroll 1
    for (int n = blockIdx.x; n < nimg; n += stride, k++) {
      const int t = k % CW_ACC;
      mbar_wait(&bar_tfull[t], (k / CW_ACC) & 1);
      tc_fence_after();
      float ve[16], va[16], vb[16];
      const uint32_t tb = tmem + t * 128 + half * 16 + ((uint32_t)(32 * (ew & 3)) << 16);
      tmem_ld16(tb, ve);
      tmem_ld16(tb + 32, va);
      tmem_ld16(tb + 64, vb);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_tempty[t]);
#pragma unroll
      for (int i = 0; i < 16; i++) va[i] += __shfl_down_sync(0xffffffffu, vb[i], 1);  // odd(r) = chunk r x Wa + chunk r + 1 x Wb
      if (evalid) {
        uint32_t oe[8], oo[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
          oe[i] = pack_bf16(fmaxf(fmaf(ve[2 * i], escale, eb[2 * i]), 0.0f), fmaxf(fmaf(ve[2 * i + 1], escale, eb[2 * i + 1]), 0.0f));
          oo[i] = pack_bf16(fmaxf(fmaf(va[2 * i], escale, eb[2 * i]), 0.0f), fmaxf(fmaf(va[2 * i + 1], escale, eb[2 * i + 1]), 0.0f));
        }
        if (a.ldo == 32) {  // dense [225][32] rows (the gather-based conv2)
          __nv_bfloat16* row = a.out + ((size_t)n * 225 + eoy * 15 + 2 * er) * 32 + half * 16;
          reinterpret_cast<uint4*>(row)[0] = make_uint4(oe[0], oe[1], oe[2], oe[3]);
          reinterpret_cast<uint4*>(row)[1] = make_uint4(oe[4], oe[5], oe[6], oe[7]);
          if (er < 7) {
            reinterpret_cast<uint4*>(row + 32)[0] = make_uint4(oo[0], oo[1], oo[2], oo[3]);
            reinterpret_cast<uint4*>(row + 32)[1] = make_uint4(oo[4], oo[5], oo[6], oo[7]);
          }
        } else {
          // [15][16 px][32 ch]: 128-byte lines of two pixels (2r, 2r + 1), chunk j of line l stored at position j ^ (l & 7)
          const int l = eoy * 8 + er;
          uint8_t* line = reinterpret_cast<uint8_t*>(a.out) + (size_t)n * 16384 + l * 128;
#pragma unroll
          for (int g = 0; g < 2; g++) {
            *reinterpret_cast<uint4*>(line + (((half * 2 + g) ^ (l & 7)) << 4)) = make_uint4(oe[4 * g], oe[4 * g + 1], oe[4 * g + 2], oe[4 * g + 3]);
            if (er < 7) *reinterpret_cast<uint4*>(line + (((4 + half * 2 + g) ^ (l & 7)) << 4)) = make_uint4(oo[4 * g], oo[4 * g + 1], oo[4 * g + 2], oo[4 * g + 3]);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 128 * CW_ACC);
}

// ------------------------------------------------------------------------------------------------ conv2 / conv3 without im2col
// Same idea with the 128-byte swizzle.  The previous layer leaves its activations in HBM in exactly the byte order the tensor
// core wants to find them in shared memory (padded NHWC lines of 128 bytes, 16-byte chunks XOR-swizzled by the line index), so
//   * a pair of images is ONE contiguous bulk copy (cp.async.bulk, the TMA engine's 1-D path, completing on an mbarrier),
//   * every k-block of the convolution is a start address inside that copy: the A rows of output pixels ox = 0..7 of one
//     output row are 8 consecutive 128-byte lines (conv2: 4x4 stride 2 on [15][16 px][32 ch], a line = two pixels, k-block
//     (ky, kx pair) starts ky rows + kx-pair lines in; conv3: 3x3 stride 1 on [8][8 px][64 ch], a line = one pixel, k-block
//     (ky, kx) starts ky rows + kx lines in), the next output row is the next 8-row group (stride byte offset = two image
//     rows / one image row), and the second image of the pair follows at 8 groups' distance, so M = 128 is two images.
// The weights stay resident in shared memory for the whole (persistent) CTA.  Warp-specialised: one producer thread (bulk
// copies, STAGES deep), one MMA-issuer thread (32 / 36 tcgen05.mma per image pair into one of two TMEM accumulators, stage and
// accumulator hand-over by tcgen05.commit on mbarriers), eight epilogue warps (tcgen05.ld, bias + ReLU, bf16, store in the
// layout the next layer reads) that overlap the MMAs of the next pair.
template <int LAYER> struct DirectConv;
template <> struct DirectConv<2> {  // 32 -> 64 channels, 4x4 stride 2, [15][16][32] (16 KB per image) -> [8][8][64] (8 KB per image)
  static constexpr int IMG_IN = 16384, NKB = 8, SBO = 2048, OUT = 6, STAGES = 3, WROWS = 64;
  __device__ static constexpr int kb_offset(int kb) { return (kb >> 1) * 1024 + (kb & 1) * 128; }
};
template <> struct DirectConv<3> {  // 64 -> 64 channels, 3x3 stride 1, [8][8][64] -> dense [16][64] (the linear layer's flatten order)
  static constexpr int IMG_IN = 8192, NKB = 9, SBO = 1024, OUT = 4, STAGES = 4, WROWS = 64;
  __device__ static constexpr int kb_offset(int kb) { return ((kb / 3) * 8 + (kb % 3)) * 128; }
};
constexpr int DC_THREADS = 320;  // warps 0-7 epilogue, warp 8 producer, warp 9 MMA issuer
template <int LAYER>
constexpr size_t dc_smem() { return (size_t)DirectConv<LAYER>::NKB * 64 * 128 + (size_t)DirectConv<LAYER>::STAGES * 2 * DirectConv<LAYER>::IMG_IN + 8192 + 1024; }


template <int LAYER>
__global__ void __launch_bounds__(DC_THREADS, 1) k_conv_direct(const LayerArgs a, int nimg) {
  using L = DirectConv<LAYER>;
  constexpr int STAGES = L::STAGES, PAIR = 2 * L::IMG_IN;
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bar_full[STAGES], bar_empty[STAGES], bar_tfull[2], bar_tempty[2];
  __shared__ uint32_t tmem_base_s;
  __shared__ __align__(16) float sbias[64];
  if (threadIdx.x < 64) sbias[threadIdx.x] = __ldg(a.bias + threadIdx.x);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sW = smem;                                  // NKB k-blocks x [64 rows x 128 B], SWIZZLE_128B
  uint8_t* sA = smem + L::NKB * 64 * 128;              // STAGES x image pair (+ 8 KB behind: the junk groups of the last pair read past it)
  if (tid == 0) {
    for (int i = 0; i < STAGES; i++) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
    for (int i = 0; i < 2; i++) { mbar_init(&bar_tfull[i], 1); mbar_init(&bar_tempty[i], 8); }
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(&tmem_base_s, 128);  // two accumulators of 64 columns
  // weights: a parameter, not an activation — staged before the dependency wait
  for (int i = tid; i < L::NKB * 64 * 8; i += DC_THREADS) {
    const int kb = i >> 9, row = (i >> 3) & 63, ch = i & 7;
    cp_async16(smem_u32(sW + kb * 64 * 128 + row * 128 + ((ch ^ (row & 7)) << 4)), a.W + (size_t)row * a.K + kb * BK + ch * 8, true);
  }
  cp_async_commit();
  for (int i = tid; i < 8192 / 16; i += DC_THREADS) *reinterpret_cast<uint4*>(sA + STAGES * PAIR + i * 16) = make_uint4(0, 0, 0, 0);
  cp_async_wait<0>();
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const uint32_t tmem = tmem_base_s;
  const int npair = (nimg + 1) >> 1;
  if (warp == 8) {
    // ---- producer: one bulk copy per image pair
    if (lane == 0) {
      const uint8_t* src = reinterpret_cast<const uint8_t*>(a.A);
      int k = 0;
      for (int pr = blockIdx.x; pr < npair; pr += gridDim.x, k++) {
        const int s = k % STAGES;
        mbar_wait(&bar_empty[s], ((k / STAGES) & 1) ^ 1);
        const uint32_t bytes = (2 * pr + 1 < nimg) ? PAIR : L::IMG_IN;  // the last pair of an odd batch is one image (the other half keeps stale, unused rows)
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&bar_full[s])), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(sA + s * PAIR)), "l"(src + (size_t)pr * PAIR), "r"(bytes), "r"(smem_u32(&bar_full[s])) : "memory");
      }
    }
  } else if (warp == 9) {
    // ---- MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = instr_desc_f16(BM, 64, true);
      const uint64_t w0 = smem_desc_sw128(smem_u32(sW));
      int k = 0;
      for (int pr = blockIdx.x; pr < npair; pr += gridDim.x, k++) {
        const int s = k % STAGES, t = k & 1;
        mbar_wait(&bar_tempty[t], ((k >> 1) & 1) ^ 1);
        mbar_wait(&bar_full[s], (k / STAGES) & 1);
        tc_fence_after();
        // A descriptor: 8-row groups SBO apart (the 1024 of smem_desc_sw128 replaced)
        uint64_t a0 = smem_desc_sw128(smem_u32(sA + s * PAIR));
        a0 = (a0 & ~((uint64_t)0x3FFF << 32)) | ((uint64_t)(L::SBO >> 4) << 32);
#pragma unroll
        for (int kb = 0; kb < L::NKB; kb++)
#pragma unroll
          for (int k16 = 0; k16 < 4; k16++)
            umma_bf16(tmem + t * 64, a0 + (uint64_t)((L::kb_offset(kb) + k16 * 32) >> 4), w0 + (uint64_t)((kb * 64 * 128 + k16 * 32) >> 4), idesc, (kb | k16) != 0);
        umma_commit(&bar_empty[s]);
        umma_commit(&bar_tfull[t]);
      }
    }
  } else {
    // ---- epilogue: accumulator row m = 32 (warp % 4) + lane = 64 * image-in-pair + 8 * oy + ox, columns 32 (warp / 4) .. + 31
    const int half = warp >> 2, m = 32 * (warp & 3) + lane, img = m >> 6, oy = (m >> 3) & 7, ox = m & 7;
    const bool valid = oy < L::OUT && ox < L::OUT;
    int k = 0;
    for (int pr = blockIdx.x; pr < npair; pr += gridDim.x, k++) {
      const int t = k & 1, n = 2 * pr + img;
      mbar_wait(&bar_tfull[t], (k >> 1) & 1);
      tc_fence_after();
      float v[32];
      tmem_ld32(tmem + t * 64 + half * 32 + ((uint32_t)(32 * (warp & 3)) << 16), v);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_tempty[t]);  // the accumulator is in registers: the next pair's MMAs may overwrite it
      if (valid && n < nimg) {
        uint32_t o[16];
        float eb[32];  // broadcast 16-byte loads from shared memory (the compiler re-issued global loads every pair when they were __ldg'ed up front)
#pragma unroll
        for (int i = 0; i < 8; i++) *reinterpret_cast<float4*>(eb + 4 * i) = *reinterpret_cast<const float4*>(sbias + half * 32 + 4 * i);
#pragma unroll
        for (int i = 0; i < 16; i++) o[i] = pack_bf16(fmaxf(v[2 * i] + eb[2 * i], 0.0f), fmaxf(v[2 * i + 1] + eb[2 * i + 1], 0.0f));
        if (LAYER == 2) {
          // -> [8][8 px][64 ch] lines of 128 bytes, chunk j of line l stored at position j ^ (l & 7) (what conv3's descriptor expects)
          const int l = oy * 8 + ox;
          uint8_t* line = reinterpret_cast<uint8_t*>(a.out) + (size_t)n * 8192 + l * 128;
#pragma unroll
          for (int j = 0; j < 4; j++) *reinterpret_cast<uint4*>(line + (((half * 4 + j) ^ (l & 7)) << 4)) = make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
        } else {
          uint4* dst = reinterpret_cast<uint4*>(a.out + ((size_t)n * 16 + oy * 4 + ox) * 64 + half * 32);
#pragma unroll
          for (int j = 0; j < 4; j++) dst[j] = make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 128);
}

// ------------------------------------------------------------------------------------------------ actor MLP in one kernel
// latent_pi.0 (576 -> 256, ReLU), latent_pi.2 (256 -> 256, ReLU) and the mu | log_std head (256 -> 16) for a tile of 128
// observations, without the two trips of the hidden activations through HBM and without two of the three launches (the three
// layers together are 3 % of the forward's flops but were a quarter of its time: each launch is latency, not work).
// The hidden activations go TMEM -> registers (bias, ReLU, bf16) -> shared memory in the K-major SWIZZLE_128B layout, where
// the next layer's MMAs read them as their A operand; the weights stream through a three-stage ring (cp.async, committed to
// mbarriers by tcgen05.commit as in k_layer); one TMEM accumulator of 256 columns is reused by both hidden layers.
struct MlpArgs {
  const __nv_bfloat16 *feat, *W0, *W1, *Wh;   // [M][576], [256][576], [256][256], [16][256]
  const float *b0, *b1, *bh;
  int M, adim;
  float *mu, *log_std, *action;
  const float* noise;
};
constexpr int MF_STAGES = 3;
constexpr int MF_A = BM * 128, MF_W = 256 * 128;                 // one k-block of A (128 rows) and of a 256-row weight matrix
constexpr size_t MF_SMEM = MF_STAGES * (MF_A + MF_W) + 4 * MF_A + 1024;

__global__ void __launch_bounds__(THREADS, 1) k_mlp_fused(const MlpArgs a) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bar_stage[MF_STAGES];
  __shared__ uint64_t bar_done;
  __shared__ uint32_t tmem_base_s;
  __shared__ __align__(16) float sb0[256], sb1[256], sbh[HEAD_N];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;                                   // MF_STAGES x [128 rows x 128 B]
  uint8_t* sW = smem + MF_STAGES * MF_A;                // MF_STAGES x [256 rows x 128 B]
  uint8_t* sH = smem + MF_STAGES * (MF_A + MF_W);       // hidden activations: 4 k-blocks x [128 rows x 128 B]
  for (int i = tid; i < 256; i += THREADS) { sb0[i] = __ldg(a.b0 + i); sb1[i] = __ldg(a.b1 + i); }
  if (tid < HEAD_N) sbh[tid] = __ldg(a.bh + tid);
  if (tid == 0) {
    for (int s = 0; s < MF_STAGES; s++) mbar_init(&bar_stage[s], 1);
    mbar_init(&bar_done, 1);
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(&tmem_base_s, 512);  // columns 0-255: hidden-layer accumulator, 256-271: head
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const uint32_t tmem = tmem_base_s;
  const int m0 = blockIdx.x * BM;
  const int row = m0 + warp * 32 + lane;      // this thread's accumulator row (epilogues)
  const int r = warp * 32 + lane;
  const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
  constexpr uint32_t idesc256 = instr_desc_f16(BM, 256, true), idesc16 = instr_desc_f16(BM, HEAD_N, true);

  int g = 0;  // k-blocks staged so far over all three layers: stage = g % MF_STAGES, barrier phase = (g / MF_STAGES) & 1
  // `wrows` rows of weight k-block kb (row stride K) -> stage, swizzled; optionally the A k-block from the feature matrix
  auto copy_stage = [&](int gi, const __nv_bfloat16* W, int K, int kb, int wrows, bool with_a) {
    const int s = gi % MF_STAGES;
    const uint32_t dW = smem_u32(sW + s * MF_W);
    for (int c = tid; c < wrows * 8; c += THREADS) {
      const int wr = c >> 3, ch = c & 7;
      cp_async16(dW + wr * 128 + ((ch ^ (wr & 7)) << 4), W + (size_t)wr * K + kb * BK + ch * 8, true);
    }
    if (with_a) {
      const uint32_t dA = smem_u32(sA + s * MF_A);
#pragma unroll
      for (int i = 0; i < BM * 8 / THREADS; i++) {
        const int c = i * THREADS + tid, ar = c >> 3, ch = c & 7;
        const bool valid = m0 + ar < a.M;
        cp_async16(dA + ar * 128 + ((ch ^ (ar & 7)) << 4), valid ? a.feat + (size_t)(m0 + ar) * FEAT_LD + kb * BK + ch * 8 : a.feat, valid);
      }
    }
  };
  // one layer: nkb k-blocks, A from the feature matrix (from_feat) or from sH, accumulator columns dcol .., N = wrows
  auto run_layer = [&](const __nv_bfloat16* W, int K, int nkb, int wrows, bool from_feat, uint32_t dcol, uint32_t idesc, uint32_t done_parity) {
    const int g0 = g;
#pragma unroll 1
    for (int kb = 0; kb < MF_STAGES - 1; kb++) {
      if (kb < nkb) {
        const int gi = g0 + kb;
        if (gi >= MF_STAGES) { mbar_wait(&bar_stage[gi % MF_STAGES], ((gi / MF_STAGES) - 1) & 1); tc_fence_after(); }
        copy_stage(gi, W, K, kb, wrows, from_feat);
      }
      cp_async_commit();
    }
#pragma unroll 1
    for (int kb = 0; kb < nkb; kb++) {
      const int kn = kb + MF_STAGES - 1;
      if (kn < nkb) {
        const int gi = g0 + kn;
        if (gi >= MF_STAGES) { mbar_wait(&bar_stage[gi % MF_STAGES], ((gi / MF_STAGES) - 1) & 1); tc_fence_after(); }
        copy_stage(gi, W, K, kn, wrows, from_feat);
      }
      cp_async_commit();
      cp_async_wait<MF_STAGES - 1>();
      fence_async_smem();
      __syncthreads();
      if (tid == 0) {
        const int s = (g0 + kb) % MF_STAGES;
        tc_fence_after();
        const uint32_t aaddr = from_feat ? smem_u32(sA + s * MF_A) : smem_u32(sH + kb * MF_A), baddr = smem_u32(sW + s * MF_W);
#pragma unroll
        for (int k = 0; k < BK / 16; k++) umma_bf16(tmem + dcol, smem_desc_sw128(aaddr + k * 32), smem_desc_sw128(baddr + k * 32), idesc, (kb | k) != 0);
        umma_commit(&bar_stage[s]);
        if (kb == nkb - 1) umma_commit(&bar_done);
      }
    }
    g = g0 + nkb;
    mbar_wait(&bar_done, done_parity);
    tc_fence_after();
    __syncwarp();
  };
  // accumulator columns 0-255 -> bias, ReLU, bf16 -> sH (row r, k-block c0 / 64, 16-byte chunk (c0 % 64) / 8, swizzled)
  auto hidden_epilogue = [&](const float* sb) {
#pragma unroll 1
    for (int c0 = 0; c0 < 256; c0 += 16) {
      float v[16], bv[16];
      tmem_ld16(trow + c0, v);
#pragma unroll
      for (int k = 0; k < 4; k++) *reinterpret_cast<float4*>(bv + 4 * k) = *reinterpret_cast<const float4*>(sb + c0 + 4 * k);
      uint32_t o[8];
#pragma unroll
      for (int k = 0; k < 8; k++) o[k] = pack_bf16(fmaxf(v[2 * k] + bv[2 * k], 0.0f), fmaxf(v[2 * k + 1] + bv[2 * k + 1], 0.0f));
      uint8_t* dst = sH + (c0 >> 6) * MF_A + r * 128;
      const int j = (c0 & 63) >> 3;
      *reinterpret_cast<uint4*>(dst + ((j ^ (r & 7)) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
      *reinterpret_cast<uint4*>(dst + (((j + 1) ^ (r & 7)) << 4)) = make_uint4(o[4], o[5], o[6], o[7]);
    }
    fence_async_smem();   // generic-proxy writes of sH -> visible to the tensor core
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  };
  run_layer(a.W0, FEAT_LD, FEAT_LD / BK, 256, true, 0, idesc256, 0);
  hidden_epilogue(sb0);
  run_layer(a.W1, 256, 256 / BK, 256, false, 0, idesc256, 1);
  hidden_epilogue(sb1);
  run_layer(a.Wh, 256, 256 / BK, HEAD_N, false, 256, idesc16, 0);
  {
    float v[16];
    tmem_ld16(trow + 256, v);
    if (row < a.M) {
      for (int k = 0; k < a.adim; k++) {
        const float mu = v[k] + sbh[k];
        float ls = v[8 + k] + sbh[8 + k];
        ls = fminf(fmaxf(ls, -20.0f), 2.0f);  // stable-baselines3 sac/policies.py LOG_STD_MIN / LOG_STD_MAX
        float pre = mu;
        if (a.noise) pre += __expf(ls) * a.noise[(size_t)row * a.adim + k];
        a.mu[(size_t)row * a.adim + k] = mu;
        a.log_std[(size_t)row * a.adim + k] = ls;
        a.action[(size_t)row * a.adim + k] = tanhf(pre);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

// padded / swizzled activations -> dense NHWC (tests and debugging only: grp_buffer("act1" / "act2"))
__global__ void k_unpack_act(const uint8_t* __restrict__ src, __nv_bfloat16* __restrict__ dst, int nimg, int layer) {
  // layer 1: [15][16 px][32 ch] lines of two pixels -> [225][32]; layer 2: [8][8 px][64 ch] lines of one pixel -> [36][64]
  const int hw = layer == 1 ? 15 : 6, C = layer == 1 ? 32 : 64, img_bytes = layer == 1 ? 16384 : 8192;
  const long total = (long)nimg * hw * hw * (C / 8);
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c8 = (int)(i % (C / 8));
    const long px = i / (C / 8);
    const int x = (int)(px % hw), y = (int)((px / hw) % hw);
    const long n = px / (hw * hw);
    const int l = layer == 1 ? y * 8 + (x >> 1) : y * 8 + x, j = layer == 1 ? (x & 1) * 4 + c8 : c8;
    const uint4 v = *reinterpret_cast<const uint4*>(src + n * img_bytes + l * 128 + ((j ^ (l & 7)) << 4));
    *reinterpret_cast<uint4*>(dst + (px * C + c8 * 8)) = v;
  }
}

// ------------------------------------------------------------------------------------------------ host side
static thread_local std::string g_err;
#define CU(call)                                                                                       \
  do {                                                                                                 \
    cudaError_t e_ = (call);                                                                           \
    if (e_ != cudaSuccess) throw std::runtime_error(std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

static uint16_t f2bf(float f) {  // round to nearest even
  uint32_t u;
  std::memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

static uint16_t f2h(float f) {  // fp32 -> fp16, round to nearest even (conv1 weights; magnitudes far inside the normal range)
  uint32_t u;
  std::memcpy(&u, &f, 4);
  const uint32_t sign = (u >> 16) & 0x8000u;
  const int32_t e = (int32_t)((u >> 23) & 0xff) - 127 + 15;
  uint32_t m = u & 0x7fffffu;
  if (((u >> 23) & 0xff) == 0xff) return (uint16_t)(sign | 0x7c00u | (m ? 0x200u : 0));
  if (e >= 31) return (uint16_t)(sign | 0x7c00u);
  if (e <= 0) {  // subnormal or zero
    if (e < -10) return (uint16_t)sign;
    m |= 0x800000u;
    const int shift = 14 - e;
    uint32_t h = m >> shift;
    const uint32_t rem = m & ((1u << shift) - 1), half = 1u << (shift - 1);
    if (rem > half || (rem == half && (h & 1))) h++;
    return (uint16_t)(sign | h);
  }
  uint32_t h = ((uint32_t)e << 10) | (m >> 13);
  const uint32_t rem = m & 0x1fffu;
  if (rem > 0x1000u || (rem == 0x1000u && (h & 1))) h++;
  return (uint16_t)(sign | h);
}

struct Shape {
  int C, H, W, cin, o1h, o1w, o2h, o2w, o3h, o3w, nflat, adim;
};

}  // namespace grp

using namespace grp;

struct grp_policy {
  Shape sh{};
  int max_envs = 0, device = 0, num_sms = 148;
  std::vector<float> params;  // fp32 master copy, torch state_dict order (see grp_num_params)
  // device copies: bf16 K-major weights in gather order, fp32 biases
  __nv_bfloat16 *w1 = nullptr, *w2 = nullptr, *w3 = nullptr, *wfc = nullptr, *wp0 = nullptr, *wp1 = nullptr, *wh = nullptr;
  float *b1 = nullptr, *b2 = nullptr, *b3 = nullptr, *bfc = nullptr, *bp0 = nullptr, *bp1 = nullptr, *bh = nullptr;
  // true: 64 x 64 observations with 4 image planes run k_conv1_ws -> k_conv_direct<2|3>, and act1 / act2 are padded + swizzled;
  // false: k_layer<CONV1|CONV2|CONV3>, and act1 / act2 are dense NHWC
  bool direct = false;
  // activations (bf16) and outputs
  __nv_bfloat16 *act1 = nullptr, *act2 = nullptr, *act3 = nullptr, *feat = nullptr;
  __nv_bfloat16 *act1_dense = nullptr, *act2_dense = nullptr;  // grp_buffer("act1" / "act2") of the descriptor-addressed chain
  int last_n = 0;
  float *mu = nullptr, *log_std = nullptr;
  std::vector<void*> owned;
  cudaStream_t stream = nullptr;
  uint64_t launches = 0;
  bool have_params = false;
};

template <class T>
static T* palloc(grp_policy* p, size_t count) {
  void* d = nullptr;
  CU(cudaMalloc(&d, count * sizeof(T)));
  CU(cudaMemset(d, 0, count * sizeof(T)));
  p->owned.push_back(d);
  return (T*)d;
}

struct ParamLayout {
  int64_t c1w, c1b, c2w, c2b, c3w, c3b, fcw, fcb, p0w, p0b, p1w, p1b, muw, mub, lsw, lsb, total;
};
static ParamLayout layout_of(const Shape& s) {
  ParamLayout L{};
  int64_t o = 0;
  L.c1w = o; o += 32LL * s.cin * 64;
  L.c1b = o; o += 32;
  L.c2w = o; o += 64LL * 32 * 16;
  L.c2b = o; o += 64;
  L.c3w = o; o += 64LL * 64 * 9;
  L.c3b = o; o += 64;
  L.fcw = o; o += 512LL * s.nflat;
  L.fcb = o; o += 512;
  L.p0w = o; o += 256LL * 514;
  L.p0b = o; o += 256;
  L.p1w = o; o += 256LL * 256;
  L.p1b = o; o += 256;
  L.muw = o; o += (int64_t)s.adim * 256;
  L.mub = o; o += s.adim;
  L.lsw = o; o += (int64_t)s.adim * 256;
  L.lsb = o; o += s.adim;
  L.total = o;
  return L;
}

extern "C" const char* grp_last_error(void) { return g_err.c_str(); }

extern "C" grp_policy* grp_create(int32_t max_envs, int32_t channels, int32_t height, int32_t width, int32_t action_dim, int32_t device) {
  try {
    if (max_envs <= 0) throw std::runtime_error("max_envs must be positive");
    if (channels < 2 || channels > 8) throw std::runtime_error("observation channels must be within 2..8 (image channels + the padding channel)");
    if (action_dim < 1 || action_dim > 8) throw std::runtime_error("action_dim must be within 1..8");
    if (width % 4 != 0) throw std::runtime_error("observation width must be a multiple of 4 (uint8 rows are read as 32-bit words)");
    Shape s{};
    s.C = channels; s.H = height; s.W = width; s.cin = channels - 1; s.adim = action_dim;
    s.o1h = (height - 8) / 4 + 1; s.o1w = (width - 8) / 4 + 1;
    s.o2h = (s.o1h - 4) / 2 + 1; s.o2w = (s.o1w - 4) / 2 + 1;
    s.o3h = s.o2h - 2; s.o3w = s.o2w - 2;
    if (height < 8 || width < 8 || s.o2h < 1 || s.o2w < 1 || s.o3h < 1 || s.o3w < 1) throw std::runtime_error("observation too small for the NatureCNN stack");
    s.nflat = 64 * s.o3h * s.o3w;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) throw std::runtime_error("no CUDA device available: the policy has no CPU fallback");
    if (device < 0 || device >= ndev) throw std::runtime_error("invalid CUDA device index");
    int major = 0;
    CU(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major != 10) throw std::runtime_error("the policy kernels use tcgen05 / TMEM and need an sm_100-class GPU");
    auto p = std::make_unique<grp_policy>();
    p->sh = s; p->max_envs = max_envs; p->device = device;
    p->direct = s.H == 64 && s.W == 64 && s.cin == 4;
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    const size_t N = max_envs;
    p->params.assign(layout_of(s).total, 0.0f);
    p->w1 = palloc<__nv_bfloat16>(p.get(), 3 * 32 * (size_t)s.cin * 64); /* W | Wa | Wb (k_conv1_ws) */ p->b1 = palloc<float>(p.get(), 32);
    p->w2 = palloc<__nv_bfloat16>(p.get(), 64 * 512); p->b2 = palloc<float>(p.get(), 64);
    p->w3 = palloc<__nv_bfloat16>(p.get(), 64 * 576); p->b3 = palloc<float>(p.get(), 64);
    p->wfc = palloc<__nv_bfloat16>(p.get(), 512 * (size_t)s.nflat); p->bfc = palloc<float>(p.get(), 512);
    p->wp0 = palloc<__nv_bfloat16>(p.get(), 256 * (size_t)FEAT_LD); p->bp0 = palloc<float>(p.get(), 256);
    p->wp1 = palloc<__nv_bfloat16>(p.get(), 256 * 256); p->bp1 = palloc<float>(p.get(), 256);
    p->wh = palloc<__nv_bfloat16>(p.get(), HEAD_N * 256); p->bh = palloc<float>(p.get(), HEAD_N);
    // direct: padded [15][16][32] and [8][8][64] per image (+ two images of slack); otherwise dense [o1h][o1w][32] and [o2h][o2w][64]
    p->act1 = palloc<__nv_bfloat16>(p.get(), p->direct ? (N + 2) * 8192 : N * s.o1h * s.o1w * 32);
    p->act2 = palloc<__nv_bfloat16>(p.get(), p->direct ? (N + 2) * 4096 : N * s.o2h * s.o2w * 64);
    p->act3 = palloc<__nv_bfloat16>(p.get(), N * s.nflat);
    p->feat = palloc<__nv_bfloat16>(p.get(), N * FEAT_LD);
    p->mu = palloc<float>(p.get(), N * s.adim);
    p->log_std = palloc<float>(p.get(), N * s.adim);
#define SET_SMEM(M_, BN_, E_) CU(cudaFuncSetAttribute(k_layer<M_, BN_, E_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)layer_smem_bytes<BN_>()))
    SET_SMEM(CONV1, 32, EPI_RELU);
    CU(cudaFuncSetAttribute(k_mlp_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MF_SMEM));
    CU(cudaFuncSetAttribute(k_conv_direct<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dc_smem<2>()));
    CU(cudaFuncSetAttribute(k_conv_direct<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dc_smem<3>()));
    CU(cudaFuncSetAttribute(k_conv1_ws, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CW_SMEM));
    CU(cudaDeviceGetAttribute(&p->num_sms, cudaDevAttrMultiProcessorCount, device));
    SET_SMEM(CONV2, 64, EPI_RELU);
    SET_SMEM(CONV3, 64, EPI_RELU);
    SET_SMEM(DENSE, 128, EPI_FEATURES);
#undef SET_SMEM
    return p.release();
  } catch (const std::exception& e) {
    g_err = e.what();
    return nullptr;
  }
}

extern "C" void grp_destroy(grp_policy* p) {
  if (!p) return;
  cudaSetDevice(p->device);
  if (p->stream) cudaStreamSynchronize(p->stream);
  for (void* d : p->owned) cudaFree(d);
  if (p->stream) cudaStreamDestroy(p->stream);
  delete p;
}

extern "C" int64_t grp_num_params(const grp_policy* p) { return p ? layout_of(p->sh).total : 0; }

static void upload_bf16(__nv_bfloat16* dst, const std::vector<uint16_t>& h) { CU(cudaMemcpy(dst, h.data(), h.size() * 2, cudaMemcpyHostToDevice)); }
static void upload_f32(float* dst, const float* h, size_t n) { CU(cudaMemcpy(dst, h, n * 4, cudaMemcpyHostToDevice)); }

extern "C" int32_t grp_set_params(grp_policy* p, const float* host, int64_t count) {
  if (!p || !host) { g_err = "null argument"; return 1; }
  try {
    const Shape& s = p->sh;
    const ParamLayout L = layout_of(s);
    if (count != L.total) throw std::runtime_error("parameter count mismatch: expected " + std::to_string(L.total) + ", got " + std::to_string(count));
    CU(cudaSetDevice(p->device));
    CU(cudaStreamSynchronize(p->stream));
    std::memcpy(p->params.data(), host, (size_t)count * 4);
    const float* P = p->params.data();
    std::vector<uint16_t> h;
    // conv1 [32][cin][8][8]: K order (c, ky, kx) is torch's own
    {
      const size_t n1 = 32 * (size_t)s.cin * 64;
      h.assign(3 * n1, 0);
      for (size_t i = 0; i < n1; i++) {  // fp16: the uint8 pixels convert to fp16 exactly and cheaply
        const uint16_t v = f2h(P[L.c1w + i]);
        const size_t kx = i & 7;
        h[i] = v;
        if (kx < 4) h[n1 + i + 4] = v;          // Wa = [0 0 0 0 w0 w1 w2 w3] per kernel row
        else h[2 * n1 + i - 4] = v;             // Wb = [w4 w5 w6 w7 0 0 0 0]
      }
      upload_bf16(p->w1, h);
    }
    // conv2 [64][32][4][4] -> [64][(ky, kx, c)]
    h.assign(64 * 512, 0);
    for (int o = 0; o < 64; o++)
      for (int c = 0; c < 32; c++)
        for (int ky = 0; ky < 4; ky++)
          for (int kx = 0; kx < 4; kx++) h[(size_t)o * 512 + (ky * 4 + kx) * 32 + c] = f2bf(P[L.c2w + (((size_t)o * 32 + c) * 4 + ky) * 4 + kx]);
    upload_bf16(p->w2, h);
    // conv3 [64][64][3][3] -> [64][(ky, kx, c)]
    h.assign(64 * 576, 0);
    for (int o = 0; o < 64; o++)
      for (int c = 0; c < 64; c++)
        for (int ky = 0; ky < 3; ky++)
          for (int kx = 0; kx < 3; kx++) h[(size_t)o * 576 + (ky * 3 + kx) * 64 + c] = f2bf(P[L.c3w + (((size_t)o * 64 + c) * 3 + ky) * 3 + kx]);
    upload_bf16(p->w3, h);
    // linear [512][nflat], torch flatten order (c, y, x) -> activation order (y, x, c)
    const int hw = s.o3h * s.o3w;
    h.assign(512 * (size_t)s.nflat, 0);
    for (int o = 0; o < 512; o++)
      for (int c = 0; c < 64; c++)
        for (int q = 0; q < hw; q++) h[(size_t)o * s.nflat + (size_t)q * 64 + c] = f2bf(P[L.fcw + (size_t)o * s.nflat + (size_t)c * hw + q]);
    upload_bf16(p->wfc, h);
    // latent_pi.0 [256][514] -> [256][576] zero padded
    h.assign(256 * (size_t)FEAT_LD, 0);
    for (int o = 0; o < 256; o++)
      for (int k = 0; k < 514; k++) h[(size_t)o * FEAT_LD + k] = f2bf(P[L.p0w + (size_t)o * 514 + k]);
    upload_bf16(p->wp0, h);
    h.resize(256 * 256);
    for (size_t i = 0; i < h.size(); i++) h[i] = f2bf(P[L.p1w + i]);
    upload_bf16(p->wp1, h);
    // head: rows 0.. = mu, rows 8.. = log_std
    h.assign(HEAD_N * 256, 0);
    std::vector<float> bh(HEAD_N, 0.0f);
    for (int o = 0; o < s.adim; o++) {
      for (int k = 0; k < 256; k++) {
        h[(size_t)o * 256 + k] = f2bf(P[L.muw + (size_t)o * 256 + k]);
        h[(size_t)(8 + o) * 256 + k] = f2bf(P[L.lsw + (size_t)o * 256 + k]);
      }
      bh[o] = P[L.mub + o];
      bh[8 + o] = P[L.lsb + o];
    }
    upload_bf16(p->wh, h);
    upload_f32(p->b1, P + L.c1b, 32);
    upload_f32(p->b2, P + L.c2b, 64);
    upload_f32(p->b3, P + L.c3b, 64);
    upload_f32(p->bfc, P + L.fcb, 512);
    upload_f32(p->bp0, P + L.p0b, 256);
    upload_f32(p->bp1, P + L.p1b, 256);
    upload_f32(p->bh, bh.data(), HEAD_N);
    p->have_params = true;
    return 0;
  } catch (const std::exception& e) {
    g_err = e.what();
    return 1;
  }
}

extern "C" int32_t grp_get_params(const grp_policy* p, float* host, int64_t count) {
  if (!p || !host) { g_err = "null argument"; return 1; }
  if (count != (int64_t)p->params.size()) { g_err = "parameter count mismatch"; return 1; }
  std::memcpy(host, p->params.data(), (size_t)count * 4);
  return 0;
}

// Every kernel of the forward is launched with programmatic dependent launch: it may begin while the previous one on the stream
// is still running, and waits for it at griddepcontrol.wait before it reads that kernel's output (see k_layer).
template <class... Params, class... Args>
static void launch_pdl(grp_policy* p, void (*kernel)(Params...), dim3 grid, int threads, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  CU(cudaLaunchKernelEx(&cfg, kernel, args...));
  p->launches++;
}

template <int MODE, int BN, int EPI>
static void launch_layer(grp_policy* p, const LayerArgs& a, int n_total, cudaStream_t st) {
  launch_pdl(p, k_layer<MODE, BN, EPI>, dim3((a.M + BM - 1) / BM, n_total / BN), THREADS, layer_smem_bytes<BN>(), st, a);
}

extern "C" int32_t grp_forward(grp_policy* p, const uint8_t* obs_dev, float* actions_dev, const float* noise_dev, int32_t n, void* stream) {
  if (!p) { g_err = "null policy handle"; return 1; }
  if (!obs_dev || !actions_dev) { g_err = "null device pointer"; return 1; }
  if (n <= 0 || n > p->max_envs) { g_err = "n must be within 1..max_envs"; return 1; }
  if (!p->have_params) { g_err = "grp_set_params has not been called"; return 1; }
  try {
    CU(cudaSetDevice(p->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : p->stream;
    const Shape& s = p->sh;
    p->last_n = n;
    const dim3 pairs(std::min((n + 1) / 2, p->num_sms));  // k_conv_direct: persistent CTAs over image pairs
    LayerArgs a{};
    // conv1: uint8 planes -> act1
    a.A = obs_dev; a.W = p->w1; a.bias = p->b1; a.out = p->act1;
    a.M = n * s.o1h * s.o1w; a.K = s.cin * 64; a.ldo = 32; a.scale = 1.0f / 255.0f;
    a.C = s.C; a.H = s.H; a.W_ = s.W; a.ih = s.H; a.iw = s.W; a.oh = s.o1h; a.ow = s.o1w;
    if (p->direct) {
      a.ldo = 0;  // act1 in the padded, swizzled layout k_conv_direct<2>'s descriptor reads
      launch_pdl(p, k_conv1_ws, dim3(std::min(n, p->num_sms)), CW_THREADS, CW_SMEM, st, a, (int)n);
    } else {
      launch_layer<CONV1, 32, EPI_RELU>(p, a, 32, st);
    }
    // conv2
    a = LayerArgs{};
    a.A = p->act1; a.W = p->w2; a.bias = p->b2; a.out = p->act2;
    a.M = n * s.o2h * s.o2w; a.K = 512; a.ldo = 64; a.scale = 1.0f;
    a.ih = s.o1h; a.iw = s.o1w; a.oh = s.o2h; a.ow = s.o2w;
    if (p->direct) launch_pdl(p, k_conv_direct<2>, pairs, DC_THREADS, dc_smem<2>(), st, a, (int)n);
    else launch_layer<CONV2, 64, EPI_RELU>(p, a, 64, st);
    // conv3
    a = LayerArgs{};
    a.A = p->act2; a.W = p->w3; a.bias = p->b3; a.out = p->act3;
    a.M = n * s.o3h * s.o3w; a.K = 576; a.ldo = 64; a.scale = 1.0f;
    a.ih = s.o2h; a.iw = s.o2w; a.oh = s.o3h; a.ow = s.o3w;
    if (p->direct) launch_pdl(p, k_conv_direct<3>, pairs, DC_THREADS, dc_smem<3>(), st, a, (int)n);
    else launch_layer<CONV3, 64, EPI_RELU>(p, a, 64, st);
    // linear -> 512 features + the two direct features
    a = LayerArgs{};
    a.A = p->act3; a.W = p->wfc; a.bias = p->bfc; a.out = p->feat;
    a.M = n; a.K = s.nflat; a.lda = s.nflat; a.ldo = FEAT_LD; a.scale = 1.0f;
    a.C = s.C; a.H = s.H; a.W_ = s.W; a.obs = obs_dev;
    launch_layer<DENSE, 128, EPI_FEATURES>(p, a, 512, st);
    // latent_pi and the mu | log_std head -> squashed Gaussian action
    MlpArgs ma{};
    ma.feat = p->feat; ma.W0 = p->wp0; ma.W1 = p->wp1; ma.Wh = p->wh; ma.b0 = p->bp0; ma.b1 = p->bp1; ma.bh = p->bh;
    ma.M = n; ma.adim = s.adim; ma.mu = p->mu; ma.log_std = p->log_std; ma.action = actions_dev; ma.noise = noise_dev;
    launch_pdl(p, k_mlp_fused, dim3((n + BM - 1) / BM), THREADS, MF_SMEM, st, ma);
    return 0;
  } catch (const std::exception& e) {
    g_err = e.what();
    return 1;
  }
}

extern "C" int32_t grp_buffer(grp_policy* p, const char* name, void** ptr, uint64_t* bytes) {
  if (!p || !name || !ptr) { g_err = "null argument"; return 1; }
  const Shape& s = p->sh;
  const size_t N = p->max_envs;
  std::string k = name;
  void* d = nullptr;
  uint64_t sz = 0;
  if (k == "mu") { d = p->mu; sz = N * s.adim * 4; }
  else if (k == "log_std") { d = p->log_std; sz = N * s.adim * 4; }
  else if (k == "features") { d = p->feat; sz = N * FEAT_LD * 2; }
  else if (k == "act1" || k == "act2") {
    const int layer = k == "act1" ? 1 : 2;
    sz = layer == 1 ? N * s.o1h * s.o1w * 32 * 2 : N * s.o2h * s.o2w * 64 * 2;
    d = layer == 1 ? (void*)p->act1 : (void*)p->act2;
    if (p->direct) {  // the buffer is padded + swizzled: hand out a dense copy
      __nv_bfloat16*& dense = layer == 1 ? p->act1_dense : p->act2_dense;
      try {
        CU(cudaSetDevice(p->device));
        if (!dense) dense = palloc<__nv_bfloat16>(p, sz / 2);
        CU(cudaDeviceSynchronize());  // the forward may have run on the caller's stream
        k_unpack_act<<<1024, 256, 0, p->stream>>>(reinterpret_cast<const uint8_t*>(d), dense, p->last_n, layer);
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(p->stream));
      } catch (const std::exception& e) { g_err = e.what(); return 1; }
      d = dense;
    }
  }
  else if (k == "act3") { d = p->act3; sz = N * (size_t)s.nflat * 2; }
  else { g_err = "unknown buffer name '" + k + "'"; return 1; }
  *ptr = d;
  if (bytes) *bytes = sz;
  return 0;
}

extern "C" int32_t grp_shape(const grp_policy* p, int32_t* out10) {
  if (!p || !out10) { g_err = "null argument"; return 1; }
  const Shape& s = p->sh;
  const int v[10] = {s.C, s.H, s.W, s.o1h, s.o1w, s.o2h, s.o2w, s.o3h, s.o3w, s.adim};
  for (int i = 0; i < 10; i++) out10[i] = v[i];
  return 0;
}

extern "C" uint64_t grp_launch_count(const grp_policy* p) { return p ? p->launches : 0; }
extern "C" void* grp_stream(const grp_policy* p) { return p ? (void*)p->stream : nullptr; }
