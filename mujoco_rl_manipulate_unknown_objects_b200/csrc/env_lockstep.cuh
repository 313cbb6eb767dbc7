// The fused agent-step kernel, in lock-step rounds.
//
// One warp integrates one environment's substeps.  Warps that each run their own environment's controller freely are
// INSTRUCTION-FETCH bound: ~120 KB of hot code per substep, 20 warps per SM at unrelated program counters, 58 % hit rate
// in the 32 KB SM instruction cache and half of all issue slots lost to "no instruction" stalls (DESIGN.md §3.1).  Here
// all warps of a block walk the substep pipeline TOGETHER — smooth forces | constraint rows | Newton solve | integrate +
// kinematics | CRB | collision — with block barriers between the stages, so the SM's instruction cache holds one stage's
// code at a time.  The per-environment controller state machine (reference robot_env.py:77-241) is an explicit `tick`
// that runs between rounds and decides, per warp, whether this round carries a physics substep; environments come from
// an atomic queue, so ragged trip counts only cost idle warps inside a round, never idle rounds.
//
// Around that core: k_order_count / k_order_envs queue the environments longest chain first and group them by contact count;
// a block whose physics work is exhausted becomes an observation builder (render_phase) for the environments that have
// already finished; the physics phase is timed on the device (%globaltimer).
#pragma once
#include "env_kernels.cuh"
#include "render_kernels.cuh"

namespace grs {

enum Stage { S_IDLE = 0, S_LOADED, S_BEGIN, S_A_PRE, S_A_POST, S_AFTER_A, S_B_PRE, S_B_POST, S_AFTER_B, S_OPEN_PRE, S_OPEN_POST, S_CLOSE_PRE, S_CLOSE_POST, S_FINISH };

struct EnvCtl {
  int stage, i, step_limit, env;
  float open_close, deltas, init_obj[3];
  StepCounters k;
  EnvFlags f;
};

__device__ __forceinline__ void ctl_stats(EnvCtl& t, const WS& w, int iters) {
  t.k.iters += iters;
  t.k.nconmax = max(t.k.nconmax, w.ncon);
  t.k.flags |= w.overflow;
}

// Advances the controller state machine of one environment up to the next physics substep.
// Returns true when a substep has to be integrated this round (controls are set), false when the agent step is complete
// (w.out holds the info record, t.f the updated flags).  `solver_iters` = Newton iterations of the substep just taken.
static __device__ __noinline__ bool env_tick(const DevModel& m, const EnvCfg& c, WS& w, EnvCtl& t, const float* __restrict__ act, int solver_iters, int lane) {
  const float scale = lane < 3 ? 1.0f / c.max_trans : 1.0f / c.max_rot;
#pragma unroll 1
  for (;;) {
    switch (t.stage) {
      case S_BEGIN: {  // robot_env.py:87-95
        float a6[6];
        if (c.include_roll) { for (int k = 0; k < 6; k++) a6[k] = act[k]; }
        else { a6[0] = act[0]; a6[1] = act[1]; a6[2] = act[2]; a6[3] = 0; a6[4] = act[3]; a6[5] = act[4]; }
        t.open_close = a6[5];
        for (int k = 0; k < 3; k++) t.init_obj[k] = w.xpos[m.body_object][k];
        if (lane < 5) w.init_q[lane] = w.qpos[lane];
        if (lane == 0) get_target_pose(m, c, w, a6);
        __syncwarp();
        t.k.tq_rec = lane < 5 ? w.tgt[lane] : 0.0f;
        t.k.nsa = t.k.nsb = t.k.nsc = t.k.iters = t.k.fail = t.k.object_grasped = 0;
        t.k.nconmax = w.ncon;
        t.k.flags = w.overflow;  // the contact set the step starts from counts (its position stage ran at load time)
        t.k.reached_target = t.k.reached_initial = false;
        t.step_limit = c.max_steps;
        t.i = 0;
        t.stage = S_A_PRE;
        break;
      }
      case S_A_PRE:  // robot_env.py:97-100
      case S_B_PRE:  // robot_env.py:116-119
        if (t.i >= c.max_steps) { t.stage = t.stage == S_A_PRE ? S_AFTER_A : S_AFTER_B; break; }
        if (lane < 5) w.ctrl[lane] = (w.tgt[lane] - w.qpos[lane]) * scale;
        __syncwarp();
        t.i++;
        t.stage = t.stage == S_A_PRE ? S_A_POST : S_B_POST;
        return true;
      case S_A_POST:
      case S_B_POST: {  // robot_env.py:104-110, 121-128
        const bool isA = t.stage == S_A_POST;
        if (isA) { t.k.nsa++; t.step_limit--; } else t.k.nsb++;
        ctl_stats(t, w, solver_iters);
        float d = lane < 5 ? fabsf(w.qpos[lane] - w.tgt[lane]) : 0.0f;
        d = warp_max(d);
        if (d < c.pos_tol) {
          if (isA) t.k.reached_target = true; else t.k.reached_initial = true;
          if (lane < 5) w.ctrl[lane] = 0;
          __syncwarp();
          t.stage = isA ? S_AFTER_A : S_AFTER_B;
        } else if (!(d == d)) {
          t.stage = isA ? S_AFTER_A : S_AFTER_B;  // non-finite state: bail out, env_finalize turns it into a FAIL
        } else {
          t.stage = isA ? S_A_PRE : S_B_PRE;
        }
        break;
      }
      case S_AFTER_A:  // robot_env.py:112-114
        if (t.step_limit == 0) {
          if (lane < 5) w.tgt[lane] = w.init_q[lane];
          __syncwarp();
          t.i = 0;
          t.stage = S_B_PRE;
        } else {
          t.stage = S_AFTER_B;
        }
        break;
      case S_AFTER_B:  // robot_env.py:130-136
        if (!t.k.reached_target && !t.k.reached_initial) { t.k.fail = 1; t.f.status = 1; }
        t.i = 0;
        if (t.k.reached_target && t.open_close > 0.f && !t.f.gripper_open) {
          if (lane == 0) { w.ctrl[5] = 0.5f; w.ctrl[6] = 0.5f; }
          __syncwarp();
          t.stage = S_OPEN_PRE;
        } else if (t.k.reached_target && t.open_close < 0.f && t.f.gripper_open) {
          if (lane == 0) { w.ctrl[5] = -1.0f; w.ctrl[6] = -1.0f; }
          __syncwarp();
          t.stage = S_CLOSE_PRE;
        } else {
          t.stage = S_FINISH;
        }
        break;
      case S_OPEN_PRE:   // robot_env.py:139-142
      case S_CLOSE_PRE:  // robot_env.py:152-157
        if (t.i >= c.max_steps) {
          __syncwarp();
          if (lane == 0) { w.ctrl[5] = 0; w.ctrl[6] = 0; }
          __syncwarp();
          t.stage = S_FINISH;
          break;
        }
        if (t.stage == S_OPEN_PRE) {
          t.deltas = fmaxf(fabsf(0.4f - w.qpos[5]), fabsf(0.4f - w.qpos[6]));
          t.stage = S_OPEN_POST;
        } else {
          t.deltas = fmaxf(fabsf(-0.4f - w.qpos[5]), fabsf(-0.4f - w.qpos[6]));
          t.k.object_grasped = check_grasp(m, w);
          t.stage = S_CLOSE_POST;
        }
        t.i++;
        return true;
      case S_OPEN_POST:
      case S_CLOSE_POST: {  // robot_env.py:145-149, 160-168
        t.k.nsc++;
        ctl_stats(t, w, solver_iters);
        bool stop;
        if (t.stage == S_OPEN_POST) {
          stop = t.deltas < c.grasp_tol || (w.qpos[5] > 0.4f && w.qpos[6] > 0.4f);
          if (stop) t.f.gripper_open = 1;
        } else {
          stop = t.deltas < c.grasp_tol || t.k.object_grasped == 3;
          if (stop) t.f.gripper_open = 0;
        }
        if (stop || !(t.deltas == t.deltas)) {
          __syncwarp();
          if (lane == 0) { w.ctrl[5] = 0; w.ctrl[6] = 0; }
          __syncwarp();
          t.stage = S_FINISH;
        } else {
          t.stage = t.stage == S_OPEN_POST ? S_OPEN_PRE : S_CLOSE_PRE;
        }
        break;
      }
      case S_FINISH:
        env_finalize(m, c, w, t.f, t.init_obj, t.k, lane);
        t.stage = S_IDLE;
        return false;
      default:
        return false;
    }
  }
}

// results of a finished agent step -> HBM (+ SB3 auto-reset, which starts the variant next_object names)
static __device__ __noinline__ void env_writeback(const DevModel& m, const EnvCfg& c, const SimBuffers& s, WS& w, EnvCtl& t, int lane) {
  const int env = t.env;
  float* st = s.state + (size_t)env * ST_STRIDE;
  int vo = 0;
  if (lane == 0) vo = s.object[env];  // lane 0 alone reads and (below) writes object[env]
  const float v_step = (float)__shfl_sync(FULL, vo, 0);  // IN_OBJECT: the variant of the episode this step belongs to
  for (int k = lane; k < IN_STRIDE; k += 32) s.info[(size_t)env * IN_STRIDE + k] = k == IN_OBJECT ? v_step : w.out[k];
  write_render_state(m, w, c.obs_cam, s.render_state + (size_t)env * RS_STRIDE, lane);
  const int done = (int)w.out[IN_DONE];
  if (lane == 0) {
    s.reward[env] = w.out[IN_REWARD];
    s.done[env] = (unsigned char)done;
    s.achieved[2 * env] = w.out[IN_ACHIEVED]; s.achieved[2 * env + 1] = w.out[IN_ACHIEVED + 1];
    s.desired[2 * env] = w.out[IN_DESIRED]; s.desired[2 * env + 1] = w.out[IN_DESIRED + 1];
  }
  if (done && c.auto_reset) {
    int v = 0;
    if (lane == 0) v = take_next_object(s, env);
    v = __shfl_sync(FULL, v, 0);
    const float* rec = s.reset_record + (size_t)v * REC_STRIDE;
    for (int k = lane; k < ST_STRIDE; k += 32) st[k] = rec[k];
    __syncwarp();
    if (lane == 0) {
      s.achieved[2 * env] = rec[ST_STRIDE + IN_ACHIEVED]; s.achieved[2 * env + 1] = rec[ST_STRIDE + IN_ACHIEVED + 1];
      s.desired[2 * env] = rec[ST_STRIDE + IN_DESIRED]; s.desired[2 * env + 1] = rec[ST_STRIDE + IN_DESIRED + 1];
      if (c.reset_noise_xy != 0.f || c.reset_noise_yaw != 0.f) apply_reset_noise(s, smem_model(v), c, env, st);
    }
  } else {
    store_state(w, t.f, st, lane);
  }
  // publish: this environment's results are complete (release: every lane fences its own stores, then lane 0 appends the
  // environment to the finished list that the observation phase consumes in order)
  __threadfence();
  __syncwarp();
  if (lane == 0) atomicExch(s.done_list + atomicAdd(s.queue + 3, 1), env);
}

// Longest-first queue order.  An agent step is a chain of dependent substeps whose length is ragged (SURVEY.md F5) and
// largely known in advance: the gripper phase (robot_env.py:136-168, ~100-400 extra substeps) runs only when the open/close
// action disagrees with the gripper's state.  The kernel's duration is the longest chain, so those environments must
// start in the first wave; short ones fill the slots that free up.  Order within a bucket is irrelevant to the results.
// A second key groups environments of similar cost per substep: a lock-step round lasts as long as its slowest warp in each
// stage, and the expensive stage (narrowphase: full MPR runs) is expensive exactly for environments whose gripper touches
// something.  The contact count of the previous agent step is the predictor.  Classes are queued chain-length class first
// (close the gripper | arm only | open it), most contacts first inside each; k_order_count sizes them, k_order_envs places.
constexpr int ORDER_BUCKETS = 8;  // contact-count buckets per chain-length class; 3 x 8 classes; counters live in SimBuffers::queue[16..39] (sizes) and [40..63] (cursors)
__device__ __forceinline__ int order_class(const SimBuffers& s, const float* __restrict__ actions, int adim, int env) {
  const float oc = actions[(size_t)env * adim + adim - 1];
  const bool open = s.state[(size_t)env * ST_STRIDE + ST_GRIPPER_OPEN] != 0.0f;
  // chain-length class: closing the gripper (~175 extra substeps) first, then the rest shortest first (arm only, then opening
  // it, ~75): every environment has then STARTED by round ~150 instead of ~300, which bounds the damage of the chains nobody
  // can predict (0.1 % of the environments run into the 400-substep arm time-out, tools/chain_predict.py: a 500-800-substep
  // chain that starts late ends late)
  const bool arm_only = !((oc < 0.f && open) || (oc > 0.f && !open));
  const int len = (oc < 0.f && open) ? 0 : (arm_only ? 1 : 2);
  const int ncon = (int)s.info[(size_t)env * IN_STRIDE + IN_NCON_MAX];
  return len * ORDER_BUCKETS + (ORDER_BUCKETS - 1 - min(max(ncon, 0), ORDER_BUCKETS - 1));  // most contacts first
}
static __global__ void k_order_count(SimBuffers s, const float* __restrict__ actions, int adim) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= s.n) return;
  atomicAdd(s.queue + 16 + order_class(s, actions, adim, env), 1);
}
static __global__ void k_order_envs(SimBuffers s, const float* __restrict__ actions, int adim) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= s.n) return;
  const int c = order_class(s, actions, adim, env);
  int base = 0;
  for (int k = 0; k < c; k++) base += s.queue[16 + k];
  s.order[base + atomicAdd(s.queue + 40 + c, 1)] = env;
  s.done_list[env] = -1;
}

// Launch bounds (320 threads, 2 blocks per SM) are a register cap, not a block width: they hold the kernel at 96 registers,
// while every launch uses LS_WARPS * 32 = 256 threads (bounds of 256 x 2 would allow 128 registers).  Measured in the steady
// state of the bench workload (profiles/r2e_warps_regs_ab.log, r2f_regs.log): 113-120 registers (bounds 512, 1) 18.2 M
// substeps/s, 96 registers 19.1 M, 80 registers 18.4 M, 72 registers 17.4 M, 64 registers 17.2 M; the stack frame grows by
// only 40 bytes at 96.
constexpr int LS_MAX_THREADS = 320, LS_MIN_BLOCKS = 2;
// Warps (= environments in flight) per block: the optimum between barrier max-ing (more warps) and instruction-cache diversity
// (more blocks per SM), profiles/r2m_sweep.log.  The observation phase runs on the same blocks: it needs RTHREADS threads and
// reuses the workspaces' shared memory for its tile.
constexpr int LS_WARPS = 8;
static_assert(LS_WARPS * 32 == RTHREADS, "the observation phase needs blocks of RTHREADS threads");
static_assert(LS_WARPS * sizeof(WS) >= render_phase_smem_bytes(), "the observation tile must fit in the step kernel's shared memory");

__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ---- asynchronous step (EnvPool send / recv; DESIGN.md §3.1 "Asynchronous step").  Every environment of a pool is in one
// of four states.  A launch of the ASYNC instantiation integrates the pending and parked environments until `need` more of
// them have finished; an environment still mid-step at that point is parked at a substep boundary: its state row (which
// already holds qpos, qvel, ctrl, warm start and the env flags) plus a park record with the controller and the workspace
// values an agent step carries across substeps.  Resuming it in a later launch reproduces the synchronous step bit for bit.
enum AsyncState { A_RETURNED = 0, A_PENDING = 1, A_PARKED = 2, A_READY = 3 };
// park record [N][PK_STRIDE] floats (every integer in it is < 2^24, so a float holds it exactly)
enum { PK_STAGE = 0, PK_I, PK_STEP_LIMIT, PK_OPEN_CLOSE, PK_DELTAS, PK_INIT_OBJ /*3*/, PK_NSA = 8, PK_NSB, PK_NSC, PK_ITERS, PK_NCONMAX,
       PK_FLAGS, PK_FAIL, PK_GRASPED, PK_REACHED_TARGET, PK_REACHED_INITIAL, PK_TQ_REC = 18 /*5*/, PK_TGT = 24 /*5*/, PK_INIT_Q = 32 /*5*/,
       PK_QPOS = 40 /*NQ: qpos as it entered the last position stage, before kinematics renormalised the free joint's quaternion*/,
       PK_STRIDE = 56 };
// control words [AC_WORDS] ints: the ready ring (slot of its oldest entry, number of entries), sticky error bits, this launch's
// goal, the queue of this launch and its class sizes / cursors (class 0 = parked, 1 + order_class = pending)
enum { AC_HEAD = 0, AC_READY, AC_ERR, AC_NEED, AC_NQUEUE, AC_SIZES = 32, AC_CURSORS = 64, AC_WORDS = 96 };
enum { AERR_SEND = 1, AERR_SEND_RANGE = 2, AERR_RECV_SHORT = 4 };
constexpr int ASYNC_CLASSES = 2 + 3 * ORDER_BUCKETS;
constexpr int S_RESUME = S_FINISH + 1;  // a parked environment whose state was loaded this round (its position stage runs now)
struct AsyncArgs {
  int* astate;  // [N] AsyncState
  int* ctl;     // [AC_WORDS]
  float* park;  // [N][PK_STRIDE]
  int* waited;  // [N] 1: pending and already queued by an earlier launch that stopped before fetching it
};

// park: the controls of the next substep are set; store the state and the controller instead of integrating it
__device__ __forceinline__ void park_env(const SimBuffers& s, const AsyncArgs& aa, const WS& w, const EnvCtl& t, int lane) {
  const int env = t.env;
  store_state(w, t.f, s.state + (size_t)env * ST_STRIDE, lane);
  float* pk = aa.park + (size_t)env * PK_STRIDE;
  if (lane < 5) { pk[PK_TQ_REC + lane] = t.k.tq_rec; pk[PK_TGT + lane] = w.tgt[lane]; pk[PK_INIT_Q + lane] = w.init_q[lane]; }
  if (lane == 0) {
    pk[PK_STAGE] = (float)t.stage; pk[PK_I] = (float)t.i; pk[PK_STEP_LIMIT] = (float)t.step_limit;
    pk[PK_OPEN_CLOSE] = t.open_close; pk[PK_DELTAS] = t.deltas;
    for (int k = 0; k < 3; k++) pk[PK_INIT_OBJ + k] = t.init_obj[k];
    pk[PK_NSA] = (float)t.k.nsa; pk[PK_NSB] = (float)t.k.nsb; pk[PK_NSC] = (float)t.k.nsc; pk[PK_ITERS] = (float)t.k.iters;
    pk[PK_NCONMAX] = (float)t.k.nconmax; pk[PK_FLAGS] = (float)t.k.flags; pk[PK_FAIL] = (float)t.k.fail; pk[PK_GRASPED] = (float)t.k.object_grasped;
    pk[PK_REACHED_TARGET] = t.k.reached_target ? 1.0f : 0.0f; pk[PK_REACHED_INITIAL] = t.k.reached_initial ? 1.0f : 0.0f;
    aa.astate[env] = A_PARKED;
  }
  __syncwarp();
}
// resume: restore the controller of a parked environment whose state row is loaded, so that it runs the substep it was
// parked before without ticking again
__device__ __forceinline__ void resume_env(const AsyncArgs& aa, WS& w, EnvCtl& t, int lane) {
  const float* pk = aa.park + (size_t)t.env * PK_STRIDE;
  t.stage = (int)pk[PK_STAGE]; t.i = (int)pk[PK_I]; t.step_limit = (int)pk[PK_STEP_LIMIT];
  t.open_close = pk[PK_OPEN_CLOSE]; t.deltas = pk[PK_DELTAS];
  for (int k = 0; k < 3; k++) t.init_obj[k] = pk[PK_INIT_OBJ + k];
  t.k.nsa = (int)pk[PK_NSA]; t.k.nsb = (int)pk[PK_NSB]; t.k.nsc = (int)pk[PK_NSC]; t.k.iters = (int)pk[PK_ITERS];
  t.k.nconmax = (int)pk[PK_NCONMAX]; t.k.flags = (int)pk[PK_FLAGS]; t.k.fail = (int)pk[PK_FAIL]; t.k.object_grasped = (int)pk[PK_GRASPED];
  t.k.reached_target = pk[PK_REACHED_TARGET] != 0.0f; t.k.reached_initial = pk[PK_REACHED_INITIAL] != 0.0f;
  t.k.tq_rec = lane < 5 ? pk[PK_TQ_REC + lane] : 0.0f;
  if (lane < 5) { w.tgt[lane] = pk[PK_TGT + lane]; w.init_q[lane] = pk[PK_INIT_Q + lane]; }
  __syncwarp();
}

// Launched with LS_WARPS warps per block.  ASYNC = false, the synchronous step: a block whose physics work is exhausted goes on
// to build observations (render_phase) instead of exiting, so the rasteriser fills the SMs that idle while the longest substep
// chains finish, and the physics phase is timed on the device.  ASYNC = true: the asynchronous step above, without either (the
// observation phase would wait for environments that get parked; k_render_obs_indexed renders its finished environments).
// MULTI = true: a mixed simulator (SimBuffers::nobj > 1); each warp runs the model of its environment's variant.  The
// single-scene instantiation keeps the model at a constant shared-memory address; the MULTI ones are compiled in
// multi_kernels.cu only (see SimKernels below).
template <bool ASYNC, bool MULTI>
__global__ void __launch_bounds__(LS_MAX_THREADS, LS_MIN_BLOCKS) k_env_step_ls(SimBuffers s, EnvCfg c, const float* __restrict__ actions, int adim, RenderScene sc, ObsArgs oa,
                                                                                  AsyncArgs aa) {
  unsigned smid = 0;
  if (!ASYNC && threadIdx.x == 0) {
    atomicMin(s.tstamp, global_ns());
    atomicAdd(s.queue + 6, 1);  // blocks of this launch that are resident (render_phase)
    asm("mov.u32 %0, %%smid;" : "=r"(smid));
    atomicAdd(s.sm_phys + (smid & 255), 1);
  }
  // Block staging by the TMA engine: the compiled models of every variant (3.8 KB each) and, when they fit beside two blocks'
  // workspaces, the convex-hull vertices of every geom (<= 18.7 KB for one scene; the support scans of the collision stage then
  // cost shared-memory latency instead of L1/L2 round trips, which were half of that stage's stall samples) arrive as two bulk
  // asynchronous copies (cp.async.bulk, 1-D) that complete on one mbarrier; no thread touches the bytes on their way in.
  __shared__ unsigned long long stage_bar;
  const float4* hull = s.hull;
  {
    const unsigned bar = (unsigned)__cvta_generic_to_shared(&stage_bar);
    const unsigned model_bytes = (MULTI ? (unsigned)s.nobj : 1u) * MODEL_BYTES;
    const unsigned hull_off = model_bytes + (unsigned)(blockDim.x >> 5) * (unsigned)sizeof(WS), hull_bytes = s.hull_smem ? (unsigned)s.hull_count * 16u : 0u;
    if (threadIdx.x == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(model_bytes + hull_bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"((unsigned)__cvta_generic_to_shared(grs_smem)), "l"(s.model), "r"(model_bytes), "r"(bar) : "memory");
      if (hull_bytes)
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"((unsigned)__cvta_generic_to_shared(grs_smem + hull_off)), "l"(s.hull), "r"(hull_bytes), "r"(bar) : "memory");
    }
    __syncthreads();  // the barrier is initialised before anyone polls it
    unsigned done = 0;
    while (!done)
      asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(bar) : "memory");
    if (s.hull_smem) hull = reinterpret_cast<const float4*>(grs_smem + hull_off);
  }
  const DevModel* mp = &smem_model(0);  // the model of the warp's current environment (its variant, set when it is loaded)
  WS& w = my_ws(MULTI ? s.nobj : 1);
  const int lane = threadIdx.x & 31;
  EnvCtl t;
  t.stage = S_IDLE; t.env = -1;
  bool exhausted = false, first = true;
  int iters = 0;
#pragma unroll 1
  for (;;) {
    // ---- controller round: finish / fetch / decide (per warp, no block-wide dependency)
    bool dyn = false, pos = false, stop = false;
    if constexpr (ASYNC) {
      // stop rule: once `need` environments have finished in this launch (s.queue[3] counts them), nothing new is fetched and
      // every environment still mid-step is parked at its next substep boundary
      stop = *reinterpret_cast<volatile int*>(s.queue + 3) >= __ldg(aa.ctl + AC_NEED);
      if (t.stage == S_RESUME) {
        if (stop) {
          t.stage = S_IDLE;  // dropped before it moved: its state row and park record still describe it, it stays parked
        } else {
          resume_env(aa, w, t, lane);
          dyn = true;
        }
      } else if (t.stage == S_LOADED && stop) {
        t.stage = S_IDLE;  // loaded but not begun: it stays pending
      }
    }
    if (t.stage == S_LOADED) t.stage = S_BEGIN;
    if (t.stage != S_IDLE && !dyn) {
      dyn = env_tick(*mp, c, w, t, actions + (size_t)t.env * adim, iters, lane);
      if (!dyn) {
        env_writeback(*mp, c, s, w, t, lane);
      } else if (stop) {
        park_env(s, aa, w, t, lane);
        t.stage = S_IDLE;
        dyn = false;
      }
    }
    if (t.stage == S_IDLE && !exhausted && !stop) {
      // first environment of a warp: static slot, so that a block starts with consecutive queue entries (environments of the
      // same class, see k_order_envs); later ones come from the shared counter, which starts behind the static slots
      const int nstatic = gridDim.x * (blockDim.x >> 5);
      const int slot = first ? blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5) : nstatic + next_env(s.queue, lane);
      first = false;
      if (slot < (ASYNC ? __ldg(aa.ctl + AC_NQUEUE) : s.n)) {
        const int env = __ldg(s.order + slot);
        t.env = env;
        if constexpr (MULTI) mp = &smem_model(s.object[env]);
        load_state(w, t.f, s.state + (size_t)env * ST_STRIDE, lane);
        t.stage = S_LOADED;
        if constexpr (ASYNC) {
          if (__ldg(aa.astate + env) == A_PARKED) {
            // the position stage below has to see the qpos the synchronous step's position stage saw (kinematics
            // renormalises the free joint's quaternion in place, and renormalising twice can move its last bit)
            if (lane < NQ) w.qpos[lane] = aa.park[(size_t)env * PK_STRIDE + PK_QPOS + lane];
            __syncwarp();
            t.stage = S_RESUME;
          }
        }
        pos = true;  // position stage of the loaded state (no dynamics this round)
      } else {
        exhausted = true;
      }
    }
    pos = pos || dyn;
    if (!__syncthreads_or(pos)) break;
    const DevModel& m = *mp;
    // ---- the substep pipeline, stage by stage, whole block in step (dm_control legacy step: mj_step2 then mj_step1)
    if (dyn) smooth_forces(m, w, lane, true, t.f.xfrc_z);
    // block barriers after the constraint rows, the Newton solve and CRB only (profiles/r2m_sweep.log: none 5 % slower)
    if (dyn) make_constraint(m, w, lane);
    __syncthreads();
    iters = 0;
    if (dyn) iters = solve_newton(m, w, lane, m.iterations);
    __syncthreads();
    if (dyn) euler_integrate(m, w, lane);
    if constexpr (ASYNC) {
      if (pos) {  // PK_QPOS: what this position stage starts from, for a resume after a park in the next round
        __syncwarp();
        if (lane < NQ) aa.park[(size_t)t.env * PK_STRIDE + PK_QPOS + lane] = w.qpos[lane];
        __syncwarp();
      }
    }
    if (pos) kinematics(m, w, lane);
    if (pos) com_pos_crb(m, w, lane);
    __syncthreads();
    if (pos) collision(m, w, hull, s.adj, lane);
  }
  if constexpr (!ASYNC) {
    if (threadIdx.x == 0) {  // end of this block's physics phase
      atomicMax(s.tstamp + 1, global_ns());
      atomicSub(s.sm_phys + (smid & 255), 1);
    }
    render_phase(sc, oa, s, grs_smem, s.sm_phys + (smid & 255));
    if (threadIdx.x == 0) {
      __threadfence();
      if (atomicAdd(s.queue + 5, 1) == (int)gridDim.x - 1) {  // last block out: account the physics phase of this launch
        const unsigned long long t0 = atomicAdd(s.tstamp, 0ull), t1 = atomicAdd(s.tstamp + 1, 0ull);
        s.tstamp[2] += t1 - t0; s.tstamp[3] += 1;
        s.tstamp[0] = ~0ull; s.tstamp[1] = 0;
      }
    }
  }
}

// ---- the small kernels around the asynchronous step (grs_async_* in gripper_sim.cu)

// every environment ready with its current outputs, in id order
static __global__ void k_async_begin(AsyncArgs aa, int* __restrict__ ring, int n) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env < n) { aa.astate[env] = A_READY; aa.waited[env] = 0; ring[env] = env; }
  if (env < AC_WORDS) aa.ctl[env] = env == AC_READY ? n : 0;
}

// send: each listed environment must be returned; its action row is written and it becomes pending
static __global__ void k_async_send(AsyncArgs aa, float* __restrict__ actions, int adim, const float* __restrict__ src, const int* __restrict__ ids, int cnt, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cnt) return;
  const int env = ids[i];
  if (env < 0 || env >= n) { atomicOr(aa.ctl + AC_ERR, AERR_SEND_RANGE); return; }
  if (atomicCAS(aa.astate + env, A_RETURNED, A_PENDING) != A_RETURNED) { atomicOr(aa.ctl + AC_ERR, AERR_SEND); return; }
  aa.waited[env] = 0;
  for (int k = 0; k < adim; k++) actions[(size_t)env * adim + k] = src[(size_t)i * adim + k];
}

// queue of one launch: parked environments first (they carry the long chains), then the pending ones that an earlier launch
// queued but stopped before fetching, then the other pending ones by order_class; nothing when `batch` environments are ready
// already.  The second class keeps a pending environment from starving: when the pool holds more environments than the grid
// has warps, a launch fetches only the head of the queue, and fresh sends of an earlier order_class would otherwise overtake
// the same tail of the queue launch after launch.  Two passes as k_order_count / k_order_envs; AC_SIZES.. / AC_CURSORS.. are zero.
__device__ __forceinline__ int async_class(const SimBuffers& s, const AsyncArgs& aa, const float* __restrict__ actions, int adim, int env, int batch) {
  const int st = aa.astate[env];
  if (aa.ctl[AC_READY] >= batch || (st != A_PARKED && st != A_PENDING)) return -1;
  return st == A_PARKED ? 0 : aa.waited[env] ? 1 : 2 + order_class(s, actions, adim, env);
}
static __global__ void k_async_order_count(SimBuffers s, AsyncArgs aa, const float* __restrict__ actions, int adim, int batch) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= s.n) return;
  const int c = async_class(s, aa, actions, adim, env, batch);
  if (c >= 0) atomicAdd(aa.ctl + AC_SIZES + c, 1);
}
static __global__ void k_async_order_envs(SimBuffers s, AsyncArgs aa, const float* __restrict__ actions, int adim, int batch) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env == 0) {
    int q = 0;
    for (int k = 0; k < ASYNC_CLASSES; k++) q += aa.ctl[AC_SIZES + k];
    aa.ctl[AC_NQUEUE] = q;
    aa.ctl[AC_NEED] = batch - aa.ctl[AC_READY];
  }
  if (env >= s.n) return;
  const int c = async_class(s, aa, actions, adim, env, batch);
  if (c < 0) return;
  int base = 0;
  for (int k = 0; k < c; k++) base += aa.ctl[AC_SIZES + k];
  s.order[base + atomicAdd(aa.ctl + AC_CURSORS + c, 1)] = env;
  if (c > 0) aa.waited[env] = 1;  // read again only by the next launch's queue (a fetched one is parked or ready by then)
}

// after the step kernel and the observations: the environments this launch finished (s.done_list[0 .. s.queue[3]), in the
// order they finished) join the ready ring; the first `batch` of the ring are returned.  One block.
static __global__ void k_async_recv(SimBuffers s, AsyncArgs aa, int* __restrict__ ring, int* __restrict__ out_ids, int batch) {
  const int n = s.n, fin = s.queue[3], head = aa.ctl[AC_HEAD], ready = aa.ctl[AC_READY];  // head < n, ready + fin <= n
  for (int i = threadIdx.x; i < fin; i += blockDim.x) {
    const int env = s.done_list[i];
    ring[(head + ready + i) % n] = env;
    aa.astate[env] = A_READY;
  }
  __syncthreads();
  const int take = min(batch, ready + fin);
  for (int j = threadIdx.x; j < batch; j += blockDim.x) {
    int env = -1;
    if (j < take) { env = ring[(head + j) % n]; aa.astate[env] = A_RETURNED; }
    out_ids[j] = env;
  }
  if (threadIdx.x == 0) {
    aa.ctl[AC_HEAD] = (head + take) % n;
    aa.ctl[AC_READY] = ready + fin - take;
    if (take < batch) aa.ctl[AC_ERR] |= AERR_RECV_SHORT;
  }
}

// ---- host: the kernels one simulator launches.  The mixed-simulator instantiations (MULTI = true) are compiled in their own
// translation unit (multi_kernels.cu): there the stage functions (collision, kinematics, the solver, ...) receive a model address
// that varies per warp.  In this one every caller passes the block's single model at its constant shared-memory address, so the
// compiler specialises the noinline stage functions to it; a second, per-warp caller in the same module undoes that and the
// single-scene step kernel's narrowphase callees spill (DESIGN.md §3.6).
using StepKernel = void (*)(SimBuffers, EnvCfg, const float*, int, RenderScene, ObsArgs, AsyncArgs);
struct SimKernels {
  StepKernel step, step_async;
  void (*make_reset_record)(SimBuffers, EnvCfg);
  void (*substep)(SimBuffers, int);
  void (*contacts)(SimBuffers);
  void (*debug_step)(SimBuffers);
  void (*camera_state)(SimBuffers, int);
};
template <bool MULTI>
inline SimKernels sim_kernels() {
  return SimKernels{k_env_step_ls<false, MULTI>, k_env_step_ls<true, MULTI>, k_make_reset_record<MULTI>, k_substep<MULTI>, k_contacts<MULTI>,
                    k_debug_step<MULTI>, k_camera_state<MULTI>};
}
SimKernels multi_sim_kernels();  // sim_kernels<true>(), multi_kernels.cu

}  // namespace grs
