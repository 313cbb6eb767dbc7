// libgripper_sim_b200.so — the C-ABI of include/b200_gripper_sim.h on top of the sm_100a kernels.
//
// Host side only owns buffers, the CUDA stream and launch bookkeeping; every per-environment computation is in
// env_kernels.cuh / sim_kernels.cuh / render_kernels.cuh.  There is no CPU fallback: without a CUDA device
// grs_create fails (grs_compile_only, the model compiler, is the one entry point that works without a GPU).
#include <cuda_runtime.h>

#include <cmath>
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/b200_gripper_sim.h"
#include "env_kernels.cuh"
#include "env_lockstep.cuh"
#include "render_kernels.cuh"

using namespace grs;

static_assert(GRS_INFO_STRIDE == IN_STRIDE && GRS_STATE_STRIDE == ST_STRIDE && GRS_DEBUG_STRIDE == DEBUG_STRIDE && GRS_RENDER_STATE_STRIDE == RS_STRIDE,
              "header / kernel record layouts diverged");
static_assert(GRS_ST_XFRC_Z == ST_XFRC_Z && GRS_INFO_TARGET_QPOS == IN_TARGET_QPOS && GRS_INFO_EPISODE_RETURN == IN_EPISODE_RETURN && GRS_INFO_OBJECT == IN_OBJECT,
              "record layouts diverged");

static thread_local std::string g_err;
static int fail(const std::string& msg) { g_err = msg; return 1; }
#define CU(call)                                                                                     \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess) throw std::runtime_error(std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)


// cudaFuncAttributeMaxDynamicSharedMemorySize belongs to the (kernel, device) pair, not to a simulator: several simulators of one
// process (different scenes -> different hull sizes) share it, so it is only ever raised — lowering it would make the launches of
// an older, larger simulator fail with "invalid argument".
static void raise_dyn_smem(const void* func, size_t bytes, int device) {
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> cur;
  std::lock_guard<std::mutex> g(mu);
  size_t& c = cur[std::make_pair(func, device)];
  if (bytes > c) {
    CU(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    c = bytes;
  }
}

struct grs_sim {
  HostModel hm;  // variant 0: what grs_model_get* answer for
  std::vector<std::string> scenes;  // scene file of each variant
  bool compile_only = false;
  int n = 0, device = 0, C = 5, H = 64, W = 64, adim = 6;
  grs_config cfg{};
  EnvCfg ecfg{};
  cudaStream_t stream = nullptr;
  cudaStream_t last_dev_stream = nullptr;  // caller's stream of the last device-path call that has not been joined yet
  SimBuffers b{};
  RenderScene scene{};
  DevModel* d_model = nullptr;
  float4* d_hull = nullptr;
  int* d_adj = nullptr;
  unsigned char *d_obs = nullptr, *d_terminal_obs = nullptr, *d_reset_obs = nullptr;
  float* d_actions = nullptr;
  float* d_hist = nullptr;  // [N][2][256] histograms of the previous observation (intrinsic reward)
  std::vector<void*> owned;
  uint64_t launches = 0;
  // timing of the fused step kernel
  static constexpr int NEV = 64;
  cudaEvent_t ev0[NEV]{}, ev1[NEV]{};
  int ev_n = 0;
  double ms_sum = 0;
  long ms_cnt = 0;
  int grid = 0;
  size_t smem = 0;
  // step kernel geometry (LS_WARPS warps per block)
  int ls_grid = 0;
  size_t ls_smem = 0;
  SimKernels kern{};  // single-scene or mixed-simulator instantiations (env_lockstep.cuh)
  ObsArgs obs_args{};
  // asynchronous step (grs_async_*): per-environment states, control words, park records, ready ring
  bool async_on = false;
  int async_batch = 0;
  AsyncArgs aa{};
  int* d_ring = nullptr;
};

template <class T>
static T* dalloc(grs_sim* s, size_t count) {
  void* p = nullptr;
  CU(cudaMalloc(&p, count * sizeof(T)));
  CU(cudaMemset(p, 0, count * sizeof(T)));
  s->owned.push_back(p);
  return (T*)p;
}

extern "C" const char* grs_last_error(void) { return g_err.c_str(); }

extern "C" void grs_default_config(grs_config* c) {
  if (!c) return;
  c->max_steps = 400; c->time_horizon = 400; c->include_roll = 1; c->full_observation = 1; c->im_reward = 0; c->her_buffer = 0;
  c->direction = 0; c->width = 64; c->height = 64; c->auto_reset = 1;
  c->pos_tolerance = 0.002f; c->grasp_tolerance = 0.03f; c->max_translation = 0.05f; c->max_rotation = 0.15f;
  c->reset_noise_xy = 0.0f; c->reset_noise_yaw = 0.0f; c->seed = 0;
}

extern "C" grs_sim* grs_compile_only(const char* xml_path) {
  try {
    auto s = std::make_unique<grs_sim>();
    s->hm = compile_mjcf(xml_path ? xml_path : "");
    s->compile_only = true;
    return s.release();
  } catch (const std::exception& e) { g_err = e.what(); return nullptr; }
}

static void harvest_events(grs_sim* s) {
  for (int i = 0; i < s->ev_n; i++) {
    float ms = 0;
    if (cudaEventSynchronize(s->ev1[i]) == cudaSuccess && cudaEventElapsedTime(&ms, s->ev0[i], s->ev1[i]) == cudaSuccess) { s->ms_sum += ms; s->ms_cnt++; }
  }
  s->ev_n = 0;
}

static void launch_queue_kernel_prep(grs_sim* s, cudaStream_t st) { CU(cudaMemsetAsync(s->b.queue, 0, 64 * sizeof(int), st)); }


extern "C" grs_sim* grs_create(const char* xml_path, int32_t num_envs, const grs_config* cfg_in, int32_t device) {
  return grs_create_scenes(&xml_path, 1, num_envs, cfg_in, device);
}

extern "C" grs_sim* grs_create_scenes(const char* const* xml_paths, int32_t count, int32_t num_envs, const grs_config* cfg_in, int32_t device) {
  grs_sim* raw = nullptr;
  try {
    if (count < 1 || count > MAXOBJ) throw std::runtime_error("a simulator holds 1.." + std::to_string(MAXOBJ) + " scenes (got " + std::to_string(count) + ")");
    if (!xml_paths) throw std::runtime_error("xml_paths is null");
    if (num_envs <= 0) throw std::runtime_error("num_envs must be positive");
    grs_config cfg;
    if (cfg_in) cfg = *cfg_in; else grs_default_config(&cfg);
    if (cfg.direction < -360 || cfg.direction > 360) throw std::runtime_error("direction must be an angle in degrees within [-360, 360] (robot_env.py:30-33: 0 and 45 are the reference's cases)");
    // the observation is one rasteriser tile
    if (cfg.width <= 0 || cfg.height <= 0 || cfg.width > TILE || cfg.height > TILE) throw std::runtime_error("observation size must be within 1.." + std::to_string(TILE));
    if (cfg.max_steps <= 0 || cfg.time_horizon <= 0) throw std::runtime_error("max_steps and time_horizon must be positive");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0) throw std::runtime_error("no CUDA device available: this library has no CPU fallback");
    if (device < 0 || device >= ndev) throw std::runtime_error("invalid CUDA device index");
    auto s = std::make_unique<grs_sim>();
    raw = s.get();
    // every variant is compiled on its own; they must agree on everything the simulator stores once (scene_mismatch)
    std::vector<HostModel> hms;
    for (int v = 0; v < count; v++) {
      s->scenes.push_back(xml_paths[v] ? xml_paths[v] : "");
      hms.push_back(compile_mjcf(s->scenes[v]));
      const std::string f = v ? scene_mismatch(hms[0], hms[v]) : "";
      if (!f.empty()) throw std::runtime_error("scene " + s->scenes[v] + " cannot share a simulator with " + s->scenes[0] + ": " + f + " differs");
    }
    s->hm = hms[0];
    const int K = count;
    s->n = num_envs; s->device = device; s->cfg = cfg;
    s->C = cfg.full_observation ? 5 : 4; s->H = cfg.height; s->W = cfg.width; s->adim = cfg.include_roll ? 6 : 5;
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
    // one DevModel per variant, MODEL_BYTES apart (the step kernel bulk-copies them in 16-byte units); variant 0's hulls first, then
    // the object hull of every other variant
    std::vector<float> hv;
    std::vector<int> adj;
    std::vector<unsigned char> models((size_t)K * MODEL_BYTES, 0);
    for (int v = 0; v < K; v++) {
      DevModel dm;
      std::vector<float> hv_v;
      std::vector<int> adj_v;
      build_dev_model(hms[v], dm, v ? hv_v : hv, v ? adj_v : adj);
      if (v) rebase_hull(*reinterpret_cast<const DevModel*>(models.data()), dm, hv_v, adj_v, hv, adj);
      std::memcpy(models.data() + (size_t)v * MODEL_BYTES, &dm, sizeof dm);
    }
    s->d_model = (DevModel*)dalloc<unsigned char>(s.get(), models.size());
    CU(cudaMemcpy(s->d_model, models.data(), models.size(), cudaMemcpyHostToDevice));
    s->d_hull = dalloc<float4>(s.get(), hv.size() / 4 + 1);
    CU(cudaMemcpy(s->d_hull, hv.data(), hv.size() * sizeof(float), cudaMemcpyHostToDevice));
    s->d_adj = dalloc<int>(s.get(), adj.size() + 1);
    CU(cudaMemcpy(s->d_adj, adj.data(), adj.size() * sizeof(int), cudaMemcpyHostToDevice));
    const size_t N = num_envs;
    SimBuffers& b = s->b;
    b.n = num_envs; b.model = s->d_model; b.hull = s->d_hull; b.adj = s->d_adj; b.nobj = K;
    b.hull_count = (int)(hv.size() / 4); b.hull_smem = 0;
    b.state = dalloc<float>(s.get(), N * ST_STRIDE);
    b.info = dalloc<float>(s.get(), N * IN_STRIDE);
    b.reward = dalloc<float>(s.get(), N);
    b.done = dalloc<unsigned char>(s.get(), N);
    b.achieved = dalloc<float>(s.get(), N * 2);
    b.desired = dalloc<float>(s.get(), N * 2);
    b.render_state = dalloc<float>(s.get(), N * RS_STRIDE);
    b.reset_record = dalloc<float>(s.get(), (size_t)K * REC_STRIDE);
    {
      // both start as n % K; the first grs_reset below copies next_object into object
      std::vector<int> first(N);
      for (size_t e = 0; e < N; e++) first[e] = (int)(e % K);
      int* next = dalloc<int>(s.get(), N);
      CU(cudaMemcpy(next, first.data(), N * sizeof(int), cudaMemcpyHostToDevice));
      b.next_object = next;
      b.object = dalloc<int>(s.get(), N);
      CU(cudaMemcpy(b.object, first.data(), N * sizeof(int), cudaMemcpyHostToDevice));
    }
    b.debug = dalloc<float>(s.get(), N * DEBUG_STRIDE);
    b.queue = dalloc<int>(s.get(), 64);
    b.done_list = dalloc<int>(s.get(), N);
    b.sm_phys = dalloc<int>(s.get(), 256);
    b.episode_count = dalloc<int>(s.get(), N);
    b.reset_obj = dalloc<float>(s.get(), N * 12);
    b.tstamp = dalloc<unsigned long long>(s.get(), 4);
    { const unsigned long long init[4] = {~0ull, 0, 0, 0}; CU(cudaMemcpy(b.tstamp, init, sizeof init, cudaMemcpyHostToDevice)); }
    b.order = dalloc<int>(s.get(), N);
    const size_t obs_bytes = (size_t)s->C * s->H * s->W;
    s->d_obs = dalloc<unsigned char>(s.get(), N * obs_bytes);
    s->d_terminal_obs = dalloc<unsigned char>(s.get(), N * obs_bytes);
    s->d_reset_obs = dalloc<unsigned char>(s.get(), K * obs_bytes);
    s->d_actions = dalloc<float>(s.get(), N * 6);
    s->d_hist = dalloc<float>(s.get(), (N + K) * 512);
    s->aa.astate = dalloc<int>(s.get(), N);
    s->aa.ctl = dalloc<int>(s.get(), AC_WORDS);
    s->aa.park = dalloc<float>(s.get(), N * PK_STRIDE);
    s->aa.waited = dalloc<int>(s.get(), N);
    s->d_ring = dalloc<int>(s.get(), N);
    EnvCfg& e = s->ecfg;
    e.max_steps = cfg.max_steps; e.time_horizon = cfg.time_horizon; e.include_roll = cfg.include_roll; e.her_buffer = cfg.her_buffer;
    e.im_reward = cfg.im_reward; e.auto_reset = cfg.auto_reset; e.full_observation = cfg.full_observation;
    e.obs_cam = 0;
    for (int c = 0; c < s->hm.ncam; c++) if (s->hm.cam_names[c] == "gripper_camera") e.obs_cam = c;  // robot_env.py:281
    e.dir[0] = 1.0f; e.dir[1] = cfg.direction == 45 ? 1.0f : 0.0f;  // robot_env.py:30-33: (1, 0) and the un-normalised (1, 1)
    if (cfg.direction != 0 && cfg.direction != 45) {
      // robot_env.py:46-54 `_get_direction` (disabled upstream at :29): unit vector at an arbitrary angle, theta rounded to 2 decimals
      const double theta = std::round(cfg.direction * (3.14159265358979323846 / 180.0) * 100.0) / 100.0;
      e.dir[0] = (float)std::cos(theta); e.dir[1] = (float)std::sin(theta);
    }
    if (!(cfg.reset_noise_xy >= 0.f) || !(cfg.reset_noise_yaw >= 0.f)) throw std::runtime_error("reset_noise_xy / reset_noise_yaw must be >= 0");
    e.reset_noise_xy = cfg.reset_noise_xy; e.reset_noise_yaw = cfg.reset_noise_yaw; e.seed = cfg.seed;
    e.pos_tol = cfg.pos_tolerance; e.grasp_tol = cfg.grasp_tolerance; e.max_trans = cfg.max_translation; e.max_rot = cfg.max_rotation;
    // launch geometry of the per-environment kernels (k_substep, k_contacts, k_debug_step, k_camera_state): persistent blocks,
    // as many as fit (one WS per warp in shared memory)
    s->kern = K > 1 ? multi_sim_kernels() : sim_kernels<false>();
    const SimKernels& kn = s->kern;
    s->smem = smem_bytes(K);
    raise_dyn_smem((const void*)kn.substep, s->smem, device);
    raise_dyn_smem((const void*)kn.contacts, s->smem, device);
    raise_dyn_smem((const void*)kn.debug_step, s->smem, device);
    raise_dyn_smem((const void*)kn.make_reset_record, s->smem, device);
    raise_dyn_smem((const void*)kn.camera_state, s->smem, device);  // above the 48 KB default with several models
    int per_sm = 0, nsm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kn.substep, WARPS_PER_BLOCK * 32, s->smem));
    CU(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device));
    if (per_sm < 1) throw std::runtime_error("substep kernel does not fit on this device");
    int want = (num_envs + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
    s->grid = std::min(want, per_sm * nsm);
    // step kernel geometry
    s->ls_smem = (size_t)K * MODEL_BYTES + (size_t)LS_WARPS * sizeof(WS);
    {
      int optin = 0;
      CU(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
      if (s->ls_smem > (size_t)optin)
        throw std::runtime_error(std::to_string(K) + " models and " + std::to_string(LS_WARPS) + " workspaces need " + std::to_string(s->ls_smem) +
                                 " bytes of shared memory per block, more than the device's " + std::to_string(optin));
    }
    {
      // hull vertices in shared memory when two blocks per SM still fit (227 KB per block, 228 KB per SM, 1 KB reserved each)
      const size_t with_hull = s->ls_smem + (size_t)s->b.hull_count * sizeof(float4);
      if (2 * (with_hull + 1024) <= 228 * 1024) { s->ls_smem = with_hull; s->b.hull_smem = 1; }
    }
    raise_dyn_smem((const void*)kn.step, s->ls_smem, device);
    raise_dyn_smem((const void*)kn.step_async, s->ls_smem, device);
    int ls_per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ls_per_sm, kn.step, LS_WARPS * 32, s->ls_smem));
    if (ls_per_sm < 1) throw std::runtime_error("step kernel does not fit on this device");
    s->ls_grid = std::min((num_envs + LS_WARPS - 1) / LS_WARPS, ls_per_sm * nsm);
    for (int i = 0; i < grs_sim::NEV; i++) { CU(cudaEventCreate(&s->ev0[i])); CU(cudaEventCreate(&s->ev1[i])); }
    render_scene_upload(hms, s->scene, s->owned);
    // the reset record and the observation of a freshly reset environment of each variant (identical for every env and every episode)
    kn.make_reset_record<<<K, 32, s->smem, s->stream>>>(s->b, s->ecfg);
    CU(cudaGetLastError());
    s->launches++;
    ObsArgs& oa = s->obs_args;
    oa.obs = s->d_obs; oa.terminal_obs = s->d_terminal_obs; oa.reset_obs = s->d_reset_obs; oa.hist_prev = s->d_hist; oa.hist_reset = s->d_hist + N * 512;
    oa.object = s->b.object;
    oa.C = s->C; oa.H = s->H; oa.W = s->W; oa.fovy = (float)s->hm.cam_fovy[e.obs_cam]; oa.auto_reset = e.auto_reset; oa.im_reward = e.im_reward;
    oa.obs_host = nullptr; oa.terminal_obs_host = nullptr;
    oa.info = s->b.info; oa.state = s->b.state; oa.info_stride = IN_STRIDE; oa.state_stride = ST_STRIDE;
    oa.in_reward = IN_REWARD; oa.in_ep_return = IN_EPISODE_RETURN; oa.st_ep_return = ST_EP_RETURN;
    for (int v = 0; v < K; v++) {
      ObsArgs r = oa;  // the reset image: one environment, no previous histograms (they go to hist_reset), no reward
      r.obs = s->d_reset_obs + v * obs_bytes; r.terminal_obs = nullptr; r.reset_obs = nullptr; r.hist_prev = nullptr; r.hist_reset = oa.hist_reset + v * 512;
      r.auto_reset = 0; r.im_reward = 0; r.info = nullptr; r.state = nullptr;
      const float* rec = s->b.reset_record + (size_t)v * REC_STRIDE;
      launch_render_obs(s->scene, r, rec + ST_STRIDE + IN_STRIDE, rec + ST_STRIDE, nullptr, nullptr, 1, s->stream);
      s->launches++;
    }
    CU(cudaStreamSynchronize(s->stream));
    {
      // reset randomisation: the new episode's observation is rendered per environment (object geom at its own pose)
      std::vector<float> rec((size_t)K * REC_STRIDE);
      CU(cudaMemcpy(rec.data(), s->b.reset_record, rec.size() * sizeof(float), cudaMemcpyDeviceToHost));
      oa.reset_noise = (e.reset_noise_xy != 0.f || e.reset_noise_yaw != 0.f) ? 1 : 0;
      oa.obj_geom = s->scene.obj_geom;
      oa.reset_rs = s->b.reset_record + ST_STRIDE + IN_STRIDE;
      oa.reset_obj = s->b.reset_obj;
      for (int v = 0; v < K; v++) {
        oa.reset_pad0[v] = (unsigned char)rec[(size_t)v * REC_STRIDE + ST_STRIDE + IN_GRASP];
        oa.reset_pad1[v] = (unsigned char)rec[(size_t)v * REC_STRIDE + ST_STRIDE + IN_PHEROMONE];
      }
    }
    if (grs_reset(s.get(), nullptr, nullptr) != 0) throw std::runtime_error(g_err);
    CU(cudaStreamSynchronize(s->stream));
    return s.release();
  } catch (const std::exception& e) {
    g_err = e.what();
    (void)raw;
    return nullptr;
  }
}

extern "C" void grs_destroy(grs_sim* s) {
  if (!s) return;
  if (!s->compile_only) {
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    for (void* p : s->owned) cudaFree(p);
    for (int i = 0; i < grs_sim::NEV; i++) { if (s->ev0[i]) cudaEventDestroy(s->ev0[i]); if (s->ev1[i]) cudaEventDestroy(s->ev1[i]); }
    if (s->stream) cudaStreamDestroy(s->stream);
  }
  delete s;
}

extern "C" int32_t grs_num_envs(const grs_sim* s) { return s ? s->n : 0; }
extern "C" int32_t grs_num_scenes(const grs_sim* s) { return s ? (s->compile_only ? 1 : (int32_t)s->scenes.size()) : 0; }
extern "C" int32_t grs_action_dim(const grs_sim* s) { return s ? s->adim : 0; }
extern "C" int32_t grs_obs_shape(const grs_sim* s, int32_t* chw) {
  if (!s || !chw) return fail("null argument");
  chw[0] = s->C; chw[1] = s->H; chw[2] = s->W;
  return 0;
}
extern "C" void* grs_stream(const grs_sim* s) { return s ? (void*)s->stream : nullptr; }

#define GUARD(s)                                                          \
  if (!(s)) return fail("null simulator handle");                         \
  if ((s)->compile_only) return fail("handle was created by grs_compile_only: no device state");
// calls that step, reset or overwrite the state rows would corrupt parked environments: refused in asynchronous mode
#define GUARD_SYNC(s)                                                                                                        \
  GUARD(s);                                                                                                                 \
  if ((s)->async_on) return fail("asynchronous mode is on: drain the pool and call grs_async_end before stepping, resetting or setting state");

extern "C" int32_t grs_reset(grs_sim* s, const uint8_t* mask_dev, void* stream) {
  GUARD_SYNC(s);
  try {
    CU(cudaSetDevice(s->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if (st != s->stream) s->last_dev_stream = st;  // a later host-path call (own stream) must order itself behind this one
    const int wpb = 8;
    k_reset<<<(s->n + wpb - 1) / wpb, wpb * 32, 0, st>>>(s->b, s->ecfg, mask_dev);
    CU(cudaGetLastError());
    if (s->obs_args.reset_noise) launch_render_reset(s->scene, s->obs_args, mask_dev, s->n, st);
    else launch_copy_reset_obs(s->d_obs, s->d_reset_obs, s->d_hist, s->d_hist + (size_t)s->n * 512, s->b.object, mask_dev, s->n, s->C * s->H * s->W, st);
    s->launches += 2;
    return 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}


// The *_host entry points run on the simulator's own (non-blocking) stream and end synchronised; the device-path entry points run
// on the caller's stream.  Mixing them on one simulator is legal: a host-path call first joins the caller's stream.
static void join_device_path(grs_sim* s) {
  if (s->last_dev_stream) {
    CU(cudaStreamSynchronize(s->last_dev_stream));
    s->last_dev_stream = nullptr;
  }
}

extern "C" int32_t grs_step(grs_sim* s, const float* actions_dev, void* stream) {
  GUARD_SYNC(s);
  if (!actions_dev) return fail("actions pointer is null");
  try {
    CU(cudaSetDevice(s->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if (st != s->stream) s->last_dev_stream = st;  // a later host-path call (own stream) must order itself behind this one
    launch_queue_kernel_prep(s, st);
    if (s->ev_n == grs_sim::NEV) harvest_events(s);
    CU(cudaEventRecord(s->ev0[s->ev_n], st));
    k_order_count<<<(s->n + 255) / 256, 256, 0, st>>>(s->b, actions_dev, s->adim);
    k_order_envs<<<(s->n + 255) / 256, 256, 0, st>>>(s->b, actions_dev, s->adim);
    s->launches += 2;
    s->kern.step<<<s->ls_grid, LS_WARPS * 32, s->ls_smem, st>>>(s->b, s->ecfg, actions_dev, s->adim, s->scene, s->obs_args, AsyncArgs{});
    CU(cudaGetLastError());
    CU(cudaEventRecord(s->ev1[s->ev_n], st));
    s->ev_n++;
    s->launches += 1;
    return 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}

// Device-visible address of a caller's host buffer if it is page-locked (cudaHostAlloc / cudaHostRegister, e.g. torch's
// pin_memory()): the observation phase then stores finished observations straight into it.  NULL for pageable memory.
static unsigned char* mapped_host_ptr(void* host) {
  if (!host) return nullptr;
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  if (a.type != cudaMemoryTypeHost || !a.devicePointer) return nullptr;
  return (unsigned char*)a.devicePointer;
}

extern "C" int32_t grs_step_host(grs_sim* s, const float* actions_host, uint8_t* obs_host, float* achieved_host, float* desired_host,
                                 float* reward_host, uint8_t* done_host, float* info_host, uint8_t* terminal_obs_host) {
  GUARD_SYNC(s);
  if (!actions_host) return fail("actions pointer is null");
  try {
    CU(cudaSetDevice(s->device));
    join_device_path(s);
    const size_t N = s->n, ob = (size_t)s->C * s->H * s->W;
    CU(cudaMemcpyAsync(s->d_actions, actions_host, N * s->adim * sizeof(float), cudaMemcpyHostToDevice, s->stream));
    // pinned destination buffers are written by the observation phase itself, environment by environment as their agent
    // steps finish (render_kernels.cuh : mirror_to_host): no bulk copy of the images after the kernel
    unsigned char* obs_m = mapped_host_ptr(obs_host);
    unsigned char* tobs_m = mapped_host_ptr(terminal_obs_host);
    s->obs_args.obs_host = obs_m; s->obs_args.terminal_obs_host = tobs_m;
    const int rc = grs_step(s, s->d_actions, nullptr);
    s->obs_args.obs_host = nullptr; s->obs_args.terminal_obs_host = nullptr;
    if (rc != 0) return 1;
    std::vector<uint8_t> done_tmp;
    uint8_t* dn = done_host;
    if (terminal_obs_host && !tobs_m && !dn) { done_tmp.resize(N); dn = done_tmp.data(); }
    if (dn) CU(cudaMemcpyAsync(dn, s->b.done, N, cudaMemcpyDeviceToHost, s->stream));
    if (obs_host && !obs_m) CU(cudaMemcpyAsync(obs_host, s->d_obs, N * ob, cudaMemcpyDeviceToHost, s->stream));
    if (achieved_host) CU(cudaMemcpyAsync(achieved_host, s->b.achieved, N * 2 * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
    if (desired_host) CU(cudaMemcpyAsync(desired_host, s->b.desired, N * 2 * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
    if (reward_host) CU(cudaMemcpyAsync(reward_host, s->b.reward, N * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
    if (info_host) CU(cudaMemcpyAsync(info_host, s->b.info, N * IN_STRIDE * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    if (terminal_obs_host && !tobs_m) {
      // terminal observations exist only for environments whose episode ended in this step: copy those rows alone
      // (rows of the other environments are left untouched)
      size_t nd = 0;
      for (size_t e = 0; e < N; e++) nd += dn[e] != 0;
      if (nd * 8 > N) {
        CU(cudaMemcpyAsync(terminal_obs_host, s->d_terminal_obs, N * ob, cudaMemcpyDeviceToHost, s->stream));
      } else {
        for (size_t e = 0; e < N; e++)
          if (dn[e]) CU(cudaMemcpyAsync(terminal_obs_host + e * ob, s->d_terminal_obs + e * ob, ob, cudaMemcpyDeviceToHost, s->stream));
      }
      if (nd) CU(cudaStreamSynchronize(s->stream));
    }
    return 0;
  } catch (const std::exception& e) { s->obs_args.obs_host = nullptr; s->obs_args.terminal_obs_host = nullptr; return fail(e.what()); }
}

extern "C" int32_t grs_reset_host(grs_sim* s, uint8_t* obs_host, float* achieved_host, float* desired_host) {
  GUARD_SYNC(s);
  try {
    CU(cudaSetDevice(s->device));
    join_device_path(s);
    if (grs_reset(s, nullptr, nullptr) != 0) return 1;
    const size_t N = s->n, ob = (size_t)s->C * s->H * s->W;
    if (obs_host) CU(cudaMemcpyAsync(obs_host, s->d_obs, N * ob, cudaMemcpyDeviceToHost, s->stream));
    if (achieved_host) CU(cudaMemcpyAsync(achieved_host, s->b.achieved, N * 2 * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
    if (desired_host) CU(cudaMemcpyAsync(desired_host, s->b.desired, N * 2 * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    return 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}

extern "C" int32_t grs_substep(grs_sim* s, int32_t n, void* stream) {
  GUARD_SYNC(s);
  if (n < 0) return fail("negative substep count");
  try {
    CU(cudaSetDevice(s->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if (st != s->stream) s->last_dev_stream = st;  // a later host-path call (own stream) must order itself behind this one
    launch_queue_kernel_prep(s, st);
    s->kern.substep<<<s->grid, WARPS_PER_BLOCK * 32, s->smem, st>>>(s->b, n);
    CU(cudaGetLastError());
    s->launches++;
    return 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}

extern "C" int32_t grs_buffer(grs_sim* s, const char* name, void** ptr, uint64_t* bytes) {
  GUARD(s);
  if (!name || !ptr) return fail("null argument");
  const size_t N = s->n, ob = (size_t)s->C * s->H * s->W;
  std::string k = name;
  void* p = nullptr;
  uint64_t sz = 0;
  if (k == "state") { p = s->b.state; sz = N * ST_STRIDE * 4; }
  else if (k == "info") { p = s->b.info; sz = N * IN_STRIDE * 4; }
  else if (k == "obs") { p = s->d_obs; sz = N * ob; }
  else if (k == "terminal_obs") { p = s->d_terminal_obs; sz = N * ob; }
  else if (k == "reset_obs") { p = s->d_reset_obs; sz = s->scenes.size() * ob; }
  else if (k == "object") { p = s->b.object; sz = N * 4; }
  else if (k == "next_object") { p = const_cast<int*>(s->b.next_object); sz = N * 4; }
  else if (k == "reward") { p = s->b.reward; sz = N * 4; }
  else if (k == "done") { p = s->b.done; sz = N; }
  else if (k == "achieved") { p = s->b.achieved; sz = N * 8; }
  else if (k == "desired") { p = s->b.desired; sz = N * 8; }
  else if (k == "render_state") { p = s->b.render_state; sz = N * RS_STRIDE * 4; }
  else if (k == "debug") { p = s->b.debug; sz = N * DEBUG_STRIDE * 4; }
  else if (k == "actions") { p = s->d_actions; sz = N * 6 * 4; }
  else if (k == "async_state") { p = s->aa.astate; sz = N * 4; }
  else return fail("unknown buffer name '" + k + "'");
  *ptr = p;
  if (bytes) *bytes = sz;
  return 0;
}

extern "C" int32_t grs_get_state(grs_sim* s, float* qpos, float* qvel, float* ctrl, float* warm, int32_t* flags, float* xfrc_z) {
  GUARD(s);
  try {
    CU(cudaSetDevice(s->device));
    std::vector<float> h((size_t)s->n * ST_STRIDE);
    CU(cudaStreamSynchronize(s->stream));
    CU(cudaMemcpy(h.data(), s->b.state, h.size() * 4, cudaMemcpyDeviceToHost));
    for (int e = 0; e < s->n; e++) {
      const float* r = &h[(size_t)e * ST_STRIDE];
      if (qpos) std::memcpy(qpos + (size_t)e * NQ, r + ST_QPOS, NQ * 4);
      if (qvel) std::memcpy(qvel + (size_t)e * NV, r + ST_QVEL, NV * 4);
      if (ctrl) std::memcpy(ctrl + (size_t)e * NU, r + ST_CTRL, NU * 4);
      if (warm) std::memcpy(warm + (size_t)e * NV, r + ST_WARM, NV * 4);
      if (flags) { flags[3 * e] = (int)r[ST_GRIPPER_OPEN]; flags[3 * e + 1] = (int)r[ST_EPISODE_STEP]; flags[3 * e + 2] = (int)r[ST_STATUS]; }
      if (xfrc_z) xfrc_z[e] = r[ST_XFRC_Z];
    }
    return 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}

extern "C" int32_t grs_set_state(grs_sim* s, const float* qpos, const float* qvel, const float* ctrl, const float* warm, const int32_t* flags,
                                 const float* xfrc_z) {
  GUARD_SYNC(s);
  try {
    CU(cudaSetDevice(s->device));
    std::vector<float> h((size_t)s->n * ST_STRIDE);
    CU(cudaStreamSynchronize(s->stream));
    CU(cudaMemcpy(h.data(), s->b.state, h.size() * 4, cudaMemcpyDeviceToHost));
    for (int e = 0; e < s->n; e++) {
      float* r = &h[(size_t)e * ST_STRIDE];
      if (qpos) std::memcpy(r + ST_QPOS, qpos + (size_t)e * NQ, NQ * 4);
      if (qvel) std::memcpy(r + ST_QVEL, qvel + (size_t)e * NV, NV * 4);
      if (ctrl) std::memcpy(r + ST_CTRL, ctrl + (size_t)e * NU, NU * 4);
      if (warm) std::memcpy(r + ST_WARM, warm + (size_t)e * NV, NV * 4);
      if (flags) { r[ST_GRIPPER_OPEN] = (float)flags[3 * e]; r[ST_EPISODE_STEP] = (float)flags[3 * e + 1]; r[ST_STATUS] = (float)flags[3 * e + 2]; }
      if (xfrc_z) r[ST_XFRC_Z] = xfrc_z[e];
    }
    CU(cudaMemcpy(s->b.state, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
    return 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}

extern "C" int32_t grs_max_contacts(void) { return MAXCON; }

extern "C" int32_t grs_get_contacts(grs_sim* s, int32_t* ncon, int32_t* geom, float* dist, float* pos, float* frame) {
  GUARD(s);
  try {
    CU(cudaSetDevice(s->device));
    launch_queue_kernel_prep(s, s->stream);
    s->kern.contacts<<<s->grid, WARPS_PER_BLOCK * 32, s->smem, s->stream>>>(s->b);
    CU(cudaGetLastError());
    s->launches++;
    CU(cudaStreamSynchronize(s->stream));
    std::vector<float> h((size_t)s->n * DEBUG_STRIDE);
    CU(cudaMemcpy(h.data(), s->b.debug, h.size() * 4, cudaMemcpyDeviceToHost));
    const int K = MAXCON;
    for (int e = 0; e < s->n; e++) {
      const float* d = &h[(size_t)e * DEBUG_STRIDE];
      int nc = (int)d[0];
      if (ncon) ncon[e] = nc;
      for (int c = 0; c < K; c++) {
        const float* o = d + 2 + c * 15;
        bool live = c < nc;
        if (geom) { geom[((size_t)e * K + c) * 2] = live ? (int)o[0] : -1; geom[((size_t)e * K + c) * 2 + 1] = live ? (int)o[1] : -1; }
        if (dist) dist[(size_t)e * K + c] = live ? o[2] : 0;
        if (pos) for (int k = 0; k < 3; k++) pos[((size_t)e * K + c) * 3 + k] = live ? o[3 + k] : 0;
        if (frame) for (int k = 0; k < 9; k++) frame[((size_t)e * K + c) * 9 + k] = live ? o[6 + k] : 0;
      }
    }
    return 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}

extern "C" int32_t grs_debug_step(grs_sim* s) {
  GUARD_SYNC(s);
  try {
    CU(cudaSetDevice(s->device));
    launch_queue_kernel_prep(s, s->stream);
    s->kern.debug_step<<<s->grid, WARPS_PER_BLOCK * 32, s->smem, s->stream>>>(s->b);
    CU(cudaGetLastError());
    s->launches++;
    CU(cudaStreamSynchronize(s->stream));
    return 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}

// ------------------------------------------------------------------------------------------ model constants
static const std::vector<double>* model_field(const HostModel& m, const std::string& k) {
#define F(nm) if (k == #nm) return &m.nm;
  F(body_mass) F(body_pos) F(body_quat) F(body_ipos) F(body_iquat) F(body_inertia) F(body_invweight0) F(dof_invweight0) F(dof_armature)
  F(dof_damping) F(geom_pos) F(geom_quat) F(geom_rbound) F(geom_friction) F(geom_margin) F(geom_gap) F(geom_solref) F(geom_solimp) F(geom_rgba) F(geom_size)
  F(geom_mass) F(geom_matprop) F(light_diffuse) F(light_ambient) F(light_specular) F(qpos0) F(jnt_pos) F(jnt_axis) F(jnt_range) F(act_gear) F(act_ctrlrange) F(cam_pos) F(cam_quat) F(cam_fovy) F(light_pos) F(light_dir)
#undef F
  return nullptr;
}
static const std::vector<int>* model_field_int(const HostModel& m, const std::string& k) {
#define F(nm) if (k == #nm) return &m.nm;
  F(body_parentid) F(body_weldid) F(body_jntadr) F(body_jntnum) F(body_dofadr) F(body_dofnum) F(body_rootid) F(jnt_type) F(jnt_bodyid) F(jnt_qposadr)
  F(jnt_dofadr) F(jnt_limited) F(dof_bodyid) F(dof_jntid) F(dof_parentid) F(geom_type) F(geom_bodyid) F(geom_meshid) F(geom_condim) F(act_dofid)
  F(pair_geom1) F(pair_geom2) F(cam_bodyid) F(cam_mode) F(cam_target) F(light_bodyid) F(light_directional)
#undef F
  return nullptr;
}

extern "C" int64_t grs_model_get(const grs_sim* s, const char* name, double* out, int64_t cap) {
  if (!s || !name) return -1;
  const HostModel& m = s->hm;
  std::string k = name;
  std::vector<double> tmp;
  const std::vector<double>* v = model_field(m, k);
  if (!v) {
    if (k == "meaninertia") tmp = {m.meaninertia};
    else if (k == "extent") tmp = {m.extent};
    else if (k == "center") tmp = {m.center[0], m.center[1], m.center[2]};
    else if (k == "timestep") tmp = {m.timestep};
    else if (k == "impratio") tmp = {m.impratio};
    else if (k == "tolerance") tmp = {m.tolerance};
    else if (k == "gravity") tmp = {m.gravity[0], m.gravity[1], m.gravity[2]};
    else if (k == "znear") tmp = {m.znear};
    else if (k == "zfar") tmp = {m.zfar};
    else if (k == "tex_rgb1") tmp = {m.tex_rgb1[0], m.tex_rgb1[1], m.tex_rgb1[2]};
    else if (k == "tex_rgb2") tmp = {m.tex_rgb2[0], m.tex_rgb2[1], m.tex_rgb2[2]};
    else if (k == "texrepeat") tmp = {m.texrepeat[0], m.texrepeat[1]};
    else if (k == "sky_rgb1") tmp = {m.sky_rgb1[0], m.sky_rgb1[1], m.sky_rgb1[2]};
    else if (k == "sky_rgb2") tmp = {m.sky_rgb2[0], m.sky_rgb2[1], m.sky_rgb2[2]};
    else if (k == "jnt_solref") tmp = {m.jnt_solref[0], m.jnt_solref[1]};
    else if (k == "jnt_solimp") tmp = {m.jnt_solimp[0], m.jnt_solimp[1], m.jnt_solimp[2], m.jnt_solimp[3], m.jnt_solimp[4]};
    else if (k.rfind("mesh_tri:", 0) == 0) {
      std::string mn = k.substr(9);
      const HostMesh* hm = nullptr;
      for (auto& x : m.meshes) if (x.name == mn) hm = &x;
      if (!hm) return -1;
      tmp.assign(hm->tri.begin(), hm->tri.end());
    }
    else if (k.rfind("hull_verts:", 0) == 0 || k.rfind("mesh_pos:", 0) == 0 || k.rfind("mesh_quat:", 0) == 0 || k.rfind("mesh_volume:", 0) == 0 ||
             k.rfind("mesh_inertia:", 0) == 0) {
      std::string mn = k.substr(k.find(':') + 1);
      const HostMesh* hm = nullptr;
      for (auto& x : m.meshes) if (x.name == mn) hm = &x;
      if (!hm) return -1;
      if (k[0] == 'h') tmp = hm->hull_verts;
      else if (k.rfind("mesh_pos:", 0) == 0) tmp = {hm->pos[0], hm->pos[1], hm->pos[2]};
      else if (k.rfind("mesh_quat:", 0) == 0) tmp = {hm->quat[0], hm->quat[1], hm->quat[2], hm->quat[3]};
      else if (k.rfind("mesh_volume:", 0) == 0) tmp = {hm->volume};
      else tmp = {hm->inertia_unit[0], hm->inertia_unit[1], hm->inertia_unit[2]};
    } else return -1;
    v = &tmp;
  }
  if (!out) return (int64_t)v->size();
  int64_t nw = std::min<int64_t>(cap, (int64_t)v->size());
  for (int64_t i = 0; i < nw; i++) out[i] = (*v)[i];
  return nw;
}

extern "C" int64_t grs_model_get_int(const grs_sim* s, const char* name, int32_t* out, int64_t cap) {
  if (!s || !name) return -1;
  const HostModel& m = s->hm;
  std::string k = name;
  std::vector<int> tmp;
  const std::vector<int>* v = model_field_int(m, k);
  if (!v) {
    if (k == "sizes") tmp = {m.nbody, m.njnt, m.nq, m.nv, m.nu, m.ngeom, m.nmesh, m.npair, m.ncam, m.nlight};
    else if (k == "iterations") tmp = {m.iterations};
    else if (k == "cone_elliptic") tmp = {m.cone_elliptic};
    else if (k == "named_bodies") tmp = {m.body_ee, m.body_object, m.finger1[0], m.finger1[1], m.finger2[0], m.finger2[1]};
    else if (k == "step_smem" && !s->compile_only) tmp = {(int)s->ls_smem, s->b.hull_smem, s->b.hull_count, LS_WARPS};
    else if (k.rfind("hull_adjadr:", 0) == 0 || k.rfind("hull_adj:", 0) == 0 || k.rfind("hull_faces:", 0) == 0) {
      std::string mn = k.substr(k.find(':') + 1);
      const HostMesh* hm = nullptr;
      for (auto& x : m.meshes) if (x.name == mn) hm = &x;
      if (!hm) return -1;
      tmp = k.rfind("hull_adjadr:", 0) == 0 ? hm->adjadr : k.rfind("hull_adj:", 0) == 0 ? hm->adj : hm->hull_faces;
    } else return -1;
    v = &tmp;
  }
  if (!out) return (int64_t)v->size();
  int64_t nw = std::min<int64_t>(cap, (int64_t)v->size());
  for (int64_t i = 0; i < nw; i++) out[i] = (*v)[i];
  return nw;
}

/* names of bodies / geoms / meshes / cameras, '\n'-separated; returns the length needed */
extern "C" int64_t grs_model_names(const grs_sim* s, const char* kind, char* out, int64_t cap) {
  if (!s || !kind) return -1;
  std::string k = kind, r;
  const std::vector<std::string>* v = nullptr;
  std::vector<std::string> tmp;
  if (k == "body") v = &s->hm.body_names;
  else if (k == "geom") v = &s->hm.geom_names;
  else if (k == "joint") v = &s->hm.jnt_names;
  else if (k == "camera") v = &s->hm.cam_names;
  else if (k == "mesh") { for (auto& m : s->hm.meshes) tmp.push_back(m.name); v = &tmp; }
  else return -1;
  for (size_t i = 0; i < v->size(); i++) { if (i) r += "\n"; r += (*v)[i]; }
  if (out && cap > 0) { size_t nw = std::min<size_t>((size_t)cap - 1, r.size()); std::memcpy(out, r.data(), nw); out[nw] = 0; }
  return (int64_t)r.size() + 1;
}

extern "C" int32_t grs_render(grs_sim* s, int32_t camera_id, int32_t width, int32_t height, uint8_t* rgb_dev, float* depth_dev, void* stream) {
  GUARD(s);
  if (camera_id < 0 || camera_id >= s->hm.ncam) return fail("camera_id out of range");
  if (width <= 0 || height <= 0 || width * height > 640 * 480) return fail("render size out of range");
  try {
    CU(cudaSetDevice(s->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if (st != s->stream) s->last_dev_stream = st;  // a later host-path call (own stream) must order itself behind this one
    launch_queue_kernel_prep(s, st);
    s->kern.camera_state<<<s->grid, WARPS_PER_BLOCK * 32, s->smem, st>>>(s->b, camera_id);
    CU(cudaGetLastError());
    launch_render_raw(s->scene, s->b.debug, DEBUG_STRIDE, s->b.object, rgb_dev, depth_dev, s->n, height, width, s->hm.cam_fovy[camera_id], st);
    s->launches += 2;
    return 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}

extern "C" uint64_t grs_launch_count(const grs_sim* s) { return s ? s->launches : 0; }

extern "C" float grs_step_kernel_ms(grs_sim* s, int32_t reset_counters) {
  if (!s || s->compile_only) return 0.0f;
  cudaSetDevice(s->device);
  harvest_events(s);
  float avg = s->ms_cnt ? (float)(s->ms_sum / s->ms_cnt) : 0.0f;
  // the synchronous step kernel times its physics phase on the device (globaltimer: first block start -> last block leaving the
  // substep loop, accumulated by the last block of every launch); the events above cover physics + observation phases and are
  // the answer when only asynchronous launches ran since the last reset
  unsigned long long t[4] = {0, 0, 0, 0};
  if (cudaStreamSynchronize(s->stream) == cudaSuccess && cudaMemcpy(t, s->b.tstamp, sizeof t, cudaMemcpyDeviceToHost) == cudaSuccess && t[3])
    avg = (float)((double)t[2] / (double)t[3] * 1e-6);
  if (reset_counters) {
    cudaMemset(s->b.tstamp + 2, 0, 2 * sizeof(unsigned long long));
    s->ms_sum = 0; s->ms_cnt = 0;
  }
  return avg;
}

// ------------------------------------------------------------------------------------------ asynchronous step
static const char* async_err_text(int bits) {
  if (bits & AERR_SEND_RANGE) return "grs_async_send: an environment id was out of range";
  if (bits & AERR_SEND) return "grs_async_send: an environment id was not in the returned state (sent twice, duplicated, or not received yet)";
  return "grs_async_recv: fewer than `batch` environments were in flight or ready (send actions for the returned ones first)";
}

extern "C" int32_t grs_async_begin(grs_sim* s, int32_t batch, void* stream) {
  GUARD(s);
  if (s->async_on) return fail("grs_async_begin: asynchronous mode is already on (grs_async_end first)");
  if (batch <= 0 || batch > s->n) return fail("grs_async_begin: batch must be within 1..num_envs");
  if (!s->cfg.auto_reset) return fail("grs_async_begin: the asynchronous step needs auto_reset=1");
  try {
    CU(cudaSetDevice(s->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if (st != s->stream) s->last_dev_stream = st;
    k_async_begin<<<(std::max(s->n, (int)AC_WORDS) + 255) / 256, 256, 0, st>>>(s->aa, s->d_ring, s->n);
    CU(cudaGetLastError());
    s->launches++;
    s->async_on = true;
    s->async_batch = batch;
    return 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}

extern "C" int32_t grs_async_send(grs_sim* s, const float* actions_dev, const int32_t* env_ids_dev, int32_t n, void* stream) {
  GUARD(s);
  if (!s->async_on) return fail("grs_async_send: asynchronous mode is off (grs_async_begin first)");
  if (n < 0 || n > s->n) return fail("grs_async_send: n must be within 0..num_envs");
  if (n == 0) return 0;
  if (!actions_dev || !env_ids_dev) return fail("grs_async_send: null pointer");
  try {
    CU(cudaSetDevice(s->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if (st != s->stream) s->last_dev_stream = st;
    k_async_send<<<(n + 255) / 256, 256, 0, st>>>(s->aa, s->d_actions, s->adim, actions_dev, env_ids_dev, n, s->n);
    CU(cudaGetLastError());
    s->launches++;
    return 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}

extern "C" int32_t grs_async_recv(grs_sim* s, int32_t* out_ids_dev, void* stream) {
  GUARD(s);
  if (!s->async_on) return fail("grs_async_recv: asynchronous mode is off (grs_async_begin first)");
  if (!out_ids_dev) return fail("grs_async_recv: null pointer");
  try {
    CU(cudaSetDevice(s->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if (st != s->stream) s->last_dev_stream = st;
    const int B = s->async_batch, g = (s->n + 255) / 256;
    launch_queue_kernel_prep(s, st);
    CU(cudaMemsetAsync(s->aa.ctl + AC_SIZES, 0, (AC_WORDS - AC_SIZES) * sizeof(int), st));
    k_async_order_count<<<g, 256, 0, st>>>(s->b, s->aa, s->d_actions, s->adim, B);
    k_async_order_envs<<<g, 256, 0, st>>>(s->b, s->aa, s->d_actions, s->adim, B);
    if (s->ev_n == grs_sim::NEV) harvest_events(s);
    CU(cudaEventRecord(s->ev0[s->ev_n], st));
    s->kern.step_async<<<s->ls_grid, LS_WARPS * 32, s->ls_smem, st>>>(s->b, s->ecfg, s->d_actions, s->adim, s->scene, s->obs_args, s->aa);
    CU(cudaGetLastError());
    CU(cudaEventRecord(s->ev1[s->ev_n], st));
    s->ev_n++;
    k_render_obs_indexed<<<s->n, RTHREADS, render_phase_smem_bytes(), st>>>(s->scene, s->obs_args, s->b.render_state, s->b.info, IN_STRIDE, s->b.done, s->b.reward,
                                                                            s->b.done_list, s->b.queue + 3);
    CU(cudaGetLastError());
    k_async_recv<<<1, 1024, 0, st>>>(s->b, s->aa, s->d_ring, out_ids_dev, B);
    CU(cudaGetLastError());
    s->launches += 5;
    return 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}

// counts[0..3]: environments returned / pending / parked / ready; counts[4]: the sticky error bits (reported and cleared here)
static int async_counts(grs_sim* s, int64_t counts[5]) {
  join_device_path(s);
  CU(cudaStreamSynchronize(s->stream));
  std::vector<int> st(s->n);
  int ctl[AC_WORDS];
  CU(cudaMemcpy(st.data(), s->aa.astate, st.size() * sizeof(int), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(ctl, s->aa.ctl, sizeof ctl, cudaMemcpyDeviceToHost));
  for (int k = 0; k < 5; k++) counts[k] = 0;
  for (int v : st) counts[std::min(std::max(v, 0), 3)]++;
  counts[4] = ctl[AC_ERR];
  if (ctl[AC_ERR]) CU(cudaMemset(s->aa.ctl + AC_ERR, 0, sizeof(int)));
  return ctl[AC_ERR];
}

extern "C" int32_t grs_async_status(grs_sim* s, int64_t counts[5]) {
  GUARD(s);
  if (!counts) return fail("grs_async_status: null pointer");
  try {
    CU(cudaSetDevice(s->device));
    if (!s->async_on) { for (int k = 0; k < 5; k++) counts[k] = 0; counts[0] = s->n; return 0; }
    const int err = async_counts(s, counts);
    return err ? fail(async_err_text(err)) : 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}

extern "C" int32_t grs_async_end(grs_sim* s) {
  GUARD(s);
  if (!s->async_on) return 0;
  try {
    CU(cudaSetDevice(s->device));
    int64_t c[5];
    const int err = async_counts(s, c);
    if (err) return fail(async_err_text(err));
    if (c[1] || c[2] || c[3])
      return fail("grs_async_end: " + std::to_string(c[1]) + " environments pending, " + std::to_string(c[2]) + " parked, " + std::to_string(c[3]) +
                  " ready but not received: receive them all first");
    s->async_on = false;
    return 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}
