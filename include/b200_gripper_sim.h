/* C-ABI of the B200 batched gripper simulator (libgripper_sim_b200.so).
 *
 * The reference has no FFI of its own for this path: RobotEnv (python) talks to dm_control's `Physics`
 * (python) which wraps libmujoco.  This header is therefore the boundary a maintainer binds INSTEAD of
 * `dm_control.mujoco.Physics` + the per-environment python loop; each entry point cites the reference
 * interface it replaces.  Plain pointers and sizes only; no torch / C++ types.
 *
 * Conventions
 *   - one handle per GPU; a handle is not thread-safe; every call runs on the handle's own CUDA stream
 *     unless a `stream` argument (a cudaStream_t passed as void*) is given (NULL = the handle's stream)
 *   - functions return 0 on success, non-zero on error; grs_last_error() returns the message
 *   - *_dev pointers are device pointers, *_host pointers are host pointers (pinned memory is faster)
 *   - arrays are env-major: actions[N][A], obs[N][C][H][W], goals[N][2]
 */
#ifndef B200_GRIPPER_SIM_H
#define B200_GRIPPER_SIM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define GRS_API __attribute__((visibility("default")))
#else
#define GRS_API
#endif

typedef struct grs_sim grs_sim;

/* Environment constructor contract = the fields RobotEnv reads from its config Namespace
 * (reference config/base_config.py:13-43; defaults in grs_default_config). */
typedef struct grs_config {
  int32_t max_steps;        /* base_config.py:36  substeps allowed per phase of an agent step (400) */
  int32_t time_horizon;     /* base_config.py:43  agent steps per episode (400) */
  int32_t include_roll;     /* base_config.py:33  action dim 6 (1) or 5 (0) */
  int32_t full_observation; /* base_config.py:22  RGB-D+pad (5 channels) or RGB+pad (4) */
  int32_t im_reward;        /* base_config.py:38  add the intrinsic (KL) reward, reward.py:57-77 */
  int32_t her_buffer;       /* base_config.py:39  add exp(-|dg-ag|), robot_env.py:268-271 */
  int32_t direction;        /* base_config.py:42  0 -> (1,0), 45 -> (1,1), robot_env.py:30-33; any other angle (degrees) -> the unit
                               vector of the reference's disabled `_get_direction`, robot_env.py:46-54 */
  int32_t width, height;    /* base_config.py:18-19 observation size (64 x 64) */
  int32_t auto_reset;       /* SB3 VecEnv semantics: reset an environment in the step that ends its episode */
  float pos_tolerance;      /* base_config.py:32 (0.002) */
  float grasp_tolerance;    /* base_config.py:31 (0.03) */
  float max_translation;    /* base_config.py:30 (0.05) */
  float max_rotation;       /* base_config.py:29 (0.15) */
  /* Reset randomisation (SURVEY.md §8f N4; the reference has none: RobotEnv.reset always starts from qpos0, robot_env.py:56-75).
   * 0 / 0 (default) reproduces the reference.  Otherwise every reset moves the object by U(-xy, xy)^2 metres and turns it by
   * U(-yaw, yaw) radians about the vertical, from a counter-based hash of (seed, environment, episode) — see INTEGRATION.md. */
  float reset_noise_xy;
  float reset_noise_yaw;
  uint32_t seed;
} grs_config;

/* per-environment step record written by grs_step (robot_env.py:226-241 `info` + the return tuple) */
enum {
  GRS_INFO_REWARD = 0, GRS_INFO_DONE, GRS_INFO_STATUS, GRS_INFO_GRASP, GRS_INFO_PHEROMONE, GRS_INFO_OBJECT_GRASPED,
  GRS_INFO_GRIPPER_OPEN, GRS_INFO_REACHED_TARGET, GRS_INFO_REACHED_INITIAL, GRS_INFO_FAIL, GRS_INFO_NSUB_A,
  GRS_INFO_NSUB_B, GRS_INFO_NSUB_C, GRS_INFO_TOTAL_DISTANCE, GRS_INFO_LINE_DISTANCE, GRS_INFO_INIT_OBJ_POS /*3*/,
  GRS_INFO_FINAL_OBJ_POS = 18 /*3*/, GRS_INFO_GRIPPER_POS = 21 /*3*/, GRS_INFO_ACHIEVED = 24 /*2*/, GRS_INFO_DESIRED = 26 /*2*/,
  GRS_INFO_SOLVER_ITERS = 28 /* Newton iterations summed over the substeps */, GRS_INFO_NCON_MAX,
  GRS_INFO_FLAGS /* bit 0: contact buffer overflowed, bit 1: non-finite state was reset */, GRS_INFO_EPISODE_STEP,
  GRS_INFO_EPISODE_RETURN = 32 /* Monitor `r` */, GRS_INFO_EPISODE_SUBSTEPS, GRS_INFO_TARGET_QPOS = 34 /*5*/, GRS_INFO_STRIDE = 40
};
/* packed per-environment state record ("state" buffer), floats */
enum {
  GRS_ST_QPOS = 0 /*14*/, GRS_ST_QVEL = 14 /*13*/, GRS_ST_CTRL = 27 /*7*/, GRS_ST_WARMSTART = 34 /*13*/, GRS_ST_GRIPPER_OPEN = 47,
  GRS_ST_EPISODE_STEP = 48, GRS_ST_STATUS = 49, GRS_ST_XFRC_Z = 50 /* xfrc_applied["ee",2], robot_env.py:65 */,
  GRS_ST_EPISODE_RETURN = 51, GRS_ST_EPISODE_SUBSTEPS = 52, GRS_STATE_STRIDE = 64
};
enum { GRS_RENDER_STATE_STRIDE = 96 }; /* 7 geoms x (pos 3 + mat 9) then the gripper camera (pos 3 + mat 9) */
enum { GRS_STATUS_RUNNING = 0, GRS_STATUS_FAIL = 1, GRS_STATUS_TIME_LIMIT = 2 }; /* robot_env.py:19-22 */

GRS_API const char* grs_last_error(void);
GRS_API void grs_default_config(grs_config* cfg);

/* replaces mujoco.Physics.from_xml_path(...) + RobotEnv.__init__ (robot_env.py:24-44) for num_envs instances */
GRS_API grs_sim* grs_create(const char* xml_path, int32_t num_envs, const grs_config* cfg, int32_t device);
GRS_API void grs_destroy(grs_sim* sim);

GRS_API int32_t grs_num_envs(const grs_sim* sim);
GRS_API int32_t grs_action_dim(const grs_sim* sim);               /* actuator.py:236-243 */
GRS_API int32_t grs_obs_shape(const grs_sim* sim, int32_t* chw);  /* sensor.py:12-54 */
GRS_API void* grs_stream(const grs_sim* sim);                     /* cudaStream_t of the handle */

/* replaces RobotEnv.reset (robot_env.py:56-75) for the environments whose mask byte is non-zero (NULL = all) */
GRS_API int32_t grs_reset(grs_sim* sim, const uint8_t* mask_dev, void* stream);

/* replaces RobotEnv.step (robot_env.py:77-241) for all environments: one fused agent step.
 * Results land in the handle's device buffers (grs_buffer). */
GRS_API int32_t grs_step(grs_sim* sim, const float* actions_dev, void* stream);

/* the same through HOST buffers (the call a VecEnv makes): H2D of actions, the step, D2H of results.
 * Any output pointer may be NULL.  info_host receives N x GRS_INFO_STRIDE floats. */
GRS_API int32_t grs_step_host(grs_sim* sim, const float* actions_host, uint8_t* obs_host, float* achieved_host,
                      float* desired_host, float* reward_host, uint8_t* done_host, float* info_host,
                      uint8_t* terminal_obs_host);
GRS_API int32_t grs_reset_host(grs_sim* sim, uint8_t* obs_host, float* achieved_host, float* desired_host);

/* replaces n x physics.step() with the controls currently in the state (robot_env.py:100) — parity tests */
GRS_API int32_t grs_substep(grs_sim* sim, int32_t n, void* stream);

/* named device buffers: "state" f32[N][64], "info" f32[N][40], "obs" u8[N][C][H][W], "terminal_obs" (same),
 * "reward" f32[N], "done" u8[N], "achieved" f32[N][2], "desired" f32[N][2], "render_state" f32[N][96],
 * "debug" f32[N][GRS_DEBUG_STRIDE].  Returns 0 and fills ptr/bytes, or non-zero for an unknown name. */
GRS_API int32_t grs_buffer(grs_sim* sim, const char* name, void** ptr, uint64_t* bytes);

/* physics.data.qpos/qvel/ctrl/qacc_warmstart + the env flags, as host arrays [N][14],[N][13],[N][7],[N][13],[N][3]
 * (gripper_open, episode_step, status), xfrc_z[N].  Any pointer may be NULL. */
GRS_API int32_t grs_get_state(grs_sim* sim, float* qpos, float* qvel, float* ctrl, float* warmstart, int32_t* flags, float* xfrc_z);
GRS_API int32_t grs_set_state(grs_sim* sim, const float* qpos, const float* qvel, const float* ctrl, const float* warmstart, const int32_t* flags,
                      const float* xfrc_z);

/* physics.data.ncon / contact[i].geom1/geom2/dist/pos/frame at the current state (actuator.py:157-176).
 * Host arrays ncon[N], geom[N][K][2], dist[N][K], pos[N][K][3], frame[N][K][9] with K = grs_max_contacts(). */
GRS_API int32_t grs_max_contacts(void);
GRS_API int32_t grs_get_contacts(grs_sim* sim, int32_t* ncon, int32_t* geom, float* dist, float* pos, float* frame);

/* one physics.step() on every environment with a dump of the intermediate quantities of environment
 * state (M, qfrc_bias, qfrc_smooth, qacc_smooth, efc rows, qacc, ...) into the "debug" buffer */
enum { GRS_DEBUG_STRIDE = 2048 };
GRS_API int32_t grs_debug_step(grs_sim* sim);

/* compiled-model constants for compiler parity (mjModel fields). Returns the number of doubles written,
 * or the required count when out == NULL, or -1 for an unknown name.  Names: body_mass, body_ipos, body_iquat,
 * body_inertia, body_invweight0, dof_invweight0, dof_armature, dof_damping, geom_pos, geom_quat, geom_rbound,
 * geom_friction, qpos0, meaninertia, extent, hull_verts:<mesh>, body_pos, body_quat, jnt_axis, jnt_range ... */
GRS_API int64_t grs_model_get(const grs_sim* sim, const char* name, double* out, int64_t cap);
GRS_API int64_t grs_model_get_int(const grs_sim* sim, const char* name, int32_t* out, int64_t cap);
/* names of the model's bodies / geoms / joints / cameras / meshes (kind = "body" ...), '\n'-separated, NUL-terminated;
 * returns the buffer size needed */
GRS_API int64_t grs_model_names(const grs_sim* sim, const char* kind, char* out, int64_t cap);
/* compile only (no GPU needed): returns a model handle usable with grs_model_get*, free with grs_destroy */
GRS_API grs_sim* grs_compile_only(const char* xml_path);

/* replaces RobotEnv.render / physics.render(camera_id,w,h[,depth]) (sensor.py:64-73) for every environment:
 * rgb u8[N][h][w][3] and depth f32[N][h][w] (metres) device buffers; either may be NULL */
GRS_API int32_t grs_render(grs_sim* sim, int32_t camera_id, int32_t width, int32_t height, uint8_t* rgb_dev, float* depth_dev, void* stream);

/* number of kernels launched by this handle since creation (bench.py reports it as gpu_launches) */
GRS_API uint64_t grs_launch_count(const grs_sim* sim);
/* average device time (ms) of the step kernel's PHYSICS phase over the launches since the last call.  Fused kernel (default):
 * timed on the device (%globaltimer, first block start -> last block leaving the substep loop); otherwise CUDA events on the
 * stream around the step kernel.  bench.py's roofline uses it. */
GRS_API float grs_step_kernel_ms(grs_sim* sim, int32_t reset_counters);

/* ---------------------------------------------------------------------------------------------------------------
 * Asynchronous step in the style of EnvPool (DESIGN.md §3.1 "Asynchronous step").  Each environment is RETURNED (its
 * outputs were handed out, it waits for an action), PENDING (action sent, step not started), PARKED (step partly done,
 * its state in HBM) or READY (step done, outputs not handed out yet).  Outputs stay in the grs_buffer arrays, row = id.
 * Needs auto_reset=1.  While asynchronous mode is on, grs_step, grs_step_host, grs_reset, grs_reset_host, grs_substep,
 * grs_set_state and grs_debug_step fail.  send and recv do not synchronise with the host: invalid ids set a sticky error
 * that the next grs_async_status or grs_async_end reports (and clears). */
/* EnvPool async_reset: every environment becomes READY with its current outputs, in id order; the first
 * num_envs / batch recv calls return them without stepping.  1 <= batch <= num_envs. */
GRS_API int32_t grs_async_begin(grs_sim* sim, int32_t batch, void* stream);
/* EnvPool send(action, env_id): actions_dev f32[n][action_dim], env_ids_dev int32[n]; each id must be RETURNED and
 * appear once; it becomes PENDING. */
GRS_API int32_t grs_async_send(grs_sim* sim, const float* actions_dev, const int32_t* env_ids_dev, int32_t n, void* stream);
/* EnvPool recv(): writes `batch` environment ids to out_ids_dev (int32) in completion order (FIFO across calls) and marks
 * them RETURNED.  With fewer than `batch` READY it first steps every PENDING and PARKED environment until `batch` are
 * READY; environments still mid-step then are PARKED at a substep boundary.  Missing ids (too few in flight) read -1. */
GRS_API int32_t grs_async_recv(grs_sim* sim, int32_t* out_ids_dev, void* stream);
/* leaves asynchronous mode; fails while any environment is PENDING, PARKED or READY */
GRS_API int32_t grs_async_end(grs_sim* sim);
/* synchronises; counts[0..3] = environments RETURNED / PENDING / PARKED / READY, counts[4] = sticky error bits
 * (1: a sent id was not RETURNED or was duplicated, 2: a sent id was out of range, 4: a recv found fewer than batch);
 * non-zero error bits make the call fail with their description */
GRS_API int32_t grs_async_status(grs_sim* sim, int64_t counts[5]);

/* ---------------------------------------------------------------------------------------------------------------
 * Policy inference during rollouts (tensor cores: tcgen05 + TMEM).  Replaces, for a whole batch of observations,
 * `model.predict(obs, deterministic=...)` (reference eval_agent.py:57, SB3 SACPolicy._predict) = preprocess_obs (/255)
 * -> AugmentedNatureCNN.forward (reference models/feature_extractor.py:39-49) -> actor latent_pi [256,256]
 * (train_agent.py:18-20) -> mu / log_std -> tanh.
 *
 * Parameters travel as ONE flat fp32 array in torch state_dict order:
 *   cnn.0.weight [32][C-1][8][8], cnn.0.bias [32], cnn.2.weight [64][32][4][4], cnn.2.bias [64],
 *   cnn.4.weight [64][64][3][3], cnn.4.bias [64], linear.0.weight [512][n_flatten], linear.0.bias [512],
 *   latent_pi.0.weight [256][514], latent_pi.0.bias [256], latent_pi.2.weight [256][256], latent_pi.2.bias [256],
 *   mu.weight [A][256], mu.bias [A], log_std.weight [A][256], log_std.bias [A]
 * (n_flatten = 64 * o3h * o3w; 1024 for 64x64 observations).  Arithmetic: bf16 operands, fp32 accumulation. */
typedef struct grp_policy grp_policy;
GRS_API const char* grp_last_error(void);
GRS_API grp_policy* grp_create(int32_t max_envs, int32_t channels, int32_t height, int32_t width, int32_t action_dim, int32_t device);
GRS_API void grp_destroy(grp_policy* p);
GRS_API int64_t grp_num_params(const grp_policy* p);
GRS_API int32_t grp_set_params(grp_policy* p, const float* params_host, int64_t count);
GRS_API int32_t grp_get_params(const grp_policy* p, float* params_host, int64_t count);
/* obs u8[n][C][H][W] (device) -> actions f32[n][A] (device).  noise_dev: f32[n][A] standard-normal samples for the
 * stochastic action tanh(mu + exp(log_std) * noise), or NULL for the deterministic action tanh(mu).
 * stream: cudaStream_t as void* (NULL = the handle's own stream). */
GRS_API int32_t grp_forward(grp_policy* p, const uint8_t* obs_dev, float* actions_dev, const float* noise_dev, int32_t n, void* stream);
/* named device buffers: "mu", "log_std" f32[max_envs][A]; "features" bf16[max_envs][576] (512 CNN + 2 direct + padding);
 * "act1" "act2" "act3" bf16 intermediate activations of the last forward (NHWC) */
GRS_API int32_t grp_buffer(grp_policy* p, const char* name, void** ptr, uint64_t* bytes);
/* {C, H, W, o1h, o1w, o2h, o2w, o3h, o3w, A} */
GRS_API int32_t grp_shape(const grp_policy* p, int32_t* out10);
GRS_API uint64_t grp_launch_count(const grp_policy* p);
GRS_API void* grp_stream(const grp_policy* p);

/* ---------------------------------------------------------------------------------------------------------------
 * On-device PPO loop (SURVEY.md §8f N1): what replaces the host-side replay buffer + optimiser round trip of
 * train_agent.py:82-88 for rollouts whose storage stays in HBM.  Device pointers only; stream = cudaStream_t as void*
 * (NULL = the legacy default stream).
 *
 * grl_gae: generalised advantage estimation over the rollout storage.  rewards f32[T][N], dones u8[T][N] (1 = the episode
 * ended with this transition), values f32[T+1][N] (the last row bootstraps) -> adv f32[T][N], ret = adv + values[:T];
 * moments_dev (may be NULL): double[2] receiving sum(adv) and sum(adv^2) for the advantage normalisation.
 *
 * grl_adam_step: Adam (torch.optim.Adam semantics, eps outside the square root) over ONE flat parameter bucket; grads are
 * multiplied by grad_scale first (1/world after a SUM all-reduce of the same buffer).  step counts from 1.  Buffers must be
 * 16-byte aligned. */
GRS_API const char* grl_last_error(void);
GRS_API int32_t grl_gae(const float* rewards_dev, const uint8_t* dones_dev, const float* values_dev, float* adv_dev, float* ret_dev, double* moments_dev,
                        int32_t T, int32_t N, float gamma, float lam, void* stream);
GRS_API int32_t grl_adam_step(float* params_dev, const float* grads_dev, float* exp_avg_dev, float* exp_avg_sq_dev, int64_t count, int32_t step,
                              float lr, float beta1, float beta2, float eps, float grad_scale, float weight_decay, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Device-resident replay buffer with HER "future" relabelling: replaces SB3's HerReplayBuffer (host RAM, one python
 * compute_reward call per relabelled row) under SAC.train (train_agent.py:61-88).  Errors are reported through grl_last_error().
 *
 * One ring of capacity + 1 slots per environment, slot-major [S][N]; a slot holds obs u8[C][H][W], next_obs u8[C][H][W],
 * action f32[A], reward f32, done u8 and the step's info row f32[GRS_INFO_STRIDE].  Transition t of environment n lives in slot t % S.
 *
 * A buffer has one of two write modes, fixed by its first begin call; the calls of the other mode then fail.
 *   lock-step (grl_replay_begin / grl_replay_add): all environments add in every call and share one host-side count.
 *   indexed (grl_replay_begin_indexed / grl_replay_add_indexed): for an asynchronous pool (grs_async_*), where environments
 *     advance at different rates.  Each environment has its own count on the device ("added"); the calls never synchronise.
 *     Bad ids and an empty sample set a sticky device error that grl_replay_status reports and clears.
 *
 * grl_replay_create: C*H*W must be a multiple of 16.  her_reward: the simulator's her_buffer (the reward carries
 *   exp(-|dg - ag|), recomputed for relabelled goals).  seed feeds the sampling hash.  NULL on bad sizes or no CUDA device.
 * grl_replay_begin: records obs_dev u8[N][C][H][W], the observations the next actions are taken on (after grs_reset, and once
 *   before the first add); closes every open episode at its newest stored transition without marking it done.
 * grl_replay_add: one vectorised step, read from the simulator's buffers after grs_step: next_obs = terminal_obs where done,
 *   else obs; then obs (the reset observation where done) becomes the pending observation of the next slot.
 * grl_replay_begin_indexed: closes every environment's open episode at its newest stored transition without marking it done, and
 *   disarms every environment.  Writes no observation: an environment's next listing in grl_replay_add_indexed records it.
 * grl_replay_add_indexed: env_ids_dev int32[count] (a grs_async_recv batch); the other arrays are the simulator's full
 *   per-environment buffers ([N][...], read at row id; actions_dev = grs_buffer "actions", which grs_async_send fills).  A
 *   disarmed environment gets obs[id] as its pending observation and is armed; an armed one completes its pending transition
 *   as grl_replay_add does, then obs[id] becomes the next pending observation.  Ids < 0 are skipped; ids >= N are skipped and
 *   reported; an id listed twice in one call is written once and reported.
 * grl_replay_size: lock-step mode: complete transitions per environment, min(added, capacity).  Fails in indexed mode.
 * grl_replay_status: synchronises the device; *transitions = the complete transitions stored over all environments (sum of
 *   min(added[n], capacity)).  Reports the sticky error bits of indexed mode as a failure with their description, and clears them.
 * grl_replay_sample: `batch` transitions, a pure function of the buffer, seed, `draw`, batch and her_ratio.  Environment and
 *   transition uniform among the complete ones (in indexed mode each environment is drawn in proportion to its complete
 *   transitions, which with equal counts is the lock-step draw, bit for bit); with probability her_ratio the desired goal is replaced by the achieved goal
 *   (info[GRS_INFO_ACHIEVED]) of a transition drawn uniformly from the same episode at or after the sampled one (the episode ends
 *   at its done transition, or at the newest stored one while it runs), and with her_reward the reward becomes
 *   reward - h(ag, dg_old) + h(ag, dg_new), h(a, d) = 1 / exp(|d - a|) (0 for transitions with FLAGS bit 1).  A step
 *   with FLAGS bit 1 (non-finite state, recorded with non-finite positions) is never a goal source and is not relabelled itself.  Outputs are
 *   device arrays obs, next_obs u8[B][C][H][W] (16-byte aligned), actions f32[B][A], reward f32[B], done u8[B], desired_goal,
 *   achieved_goal f32[B][2]; info f32[B][GRS_INFO_STRIDE], index i64[B] (flat slot * N + env) and goal_index i64[B] (flat index
 *   of the goal's transition, -1 when not relabelled) may be NULL.  Fails on an empty buffer, batch <= 0 or her_ratio outside
 *   [0, 1]; in indexed mode an empty buffer is found on the device instead: every row gets index = goal_index = -1 (the other
 *   outputs are not written) and grl_replay_status reports it.  Indexed sampling uses one scratch array of the buffer: do not
 *   sample one buffer on two streams at once.
 * grl_replay_buffer: named storage views "obs", "next_obs", "actions", "reward", "done", "info" ([S][N][...], S = capacity + 1)
 *   and "added" (int64[N], indexed mode's per-environment counts of complete transitions). */
typedef struct grl_replay grl_replay;
GRS_API grl_replay* grl_replay_create(int32_t capacity, int32_t num_envs, int32_t channels, int32_t height, int32_t width, int32_t action_dim,
                                      int32_t her_reward, uint32_t seed, int32_t device);
GRS_API void grl_replay_destroy(grl_replay* rb);
GRS_API int32_t grl_replay_begin(grl_replay* rb, const uint8_t* obs_dev, void* stream);
GRS_API int32_t grl_replay_add(grl_replay* rb, const float* actions_dev, const float* reward_dev, const uint8_t* done_dev, const float* info_dev,
                               const uint8_t* obs_dev, const uint8_t* terminal_obs_dev, void* stream);
GRS_API int32_t grl_replay_begin_indexed(grl_replay* rb, void* stream);
GRS_API int32_t grl_replay_add_indexed(grl_replay* rb, const int32_t* env_ids_dev, int32_t count, const float* actions_dev, const float* reward_dev,
                                       const uint8_t* done_dev, const float* info_dev, const uint8_t* obs_dev, const uint8_t* terminal_obs_dev,
                                       void* stream);
GRS_API int64_t grl_replay_size(const grl_replay* rb);
GRS_API int32_t grl_replay_status(grl_replay* rb, int64_t* transitions);
GRS_API int32_t grl_replay_sample(grl_replay* rb, int32_t batch, float her_ratio, uint64_t draw, uint8_t* obs_dev, uint8_t* next_obs_dev,
                                  float* actions_dev, float* reward_dev, uint8_t* done_dev, float* desired_goal_dev, float* achieved_goal_dev,
                                  float* info_dev, int64_t* index_dev, int64_t* goal_index_dev, void* stream);
GRS_API int32_t grl_replay_buffer(grl_replay* rb, const char* name, void** ptr, uint64_t* bytes);

#ifdef __cplusplus
}
#endif
#endif
