// Environment layer on the device: RobotEnv.step / reset (reference simulation/environment/robot_env.py:56-241),
// Actuator (simulation/controller/actuator.py) and Reward (simulation/environment/reward.py:18-41) around the physics
// substep of sim_kernels.cuh.  One warp owns one environment: its state is loaded from HBM into the warp's
// shared-memory workspace, and one record per environment goes back to HBM.  This file holds the state and info
// records, the IK target, the end-of-step bookkeeping (env_finalize), reset, and the per-environment kernels of the
// parity tests and the renderer (k_substep, k_contacts, k_debug_step), whose warps pull environments from an atomic
// queue.  The agent-step kernel, which runs the controller between lock-step substep rounds, is in env_lockstep.cuh.
#pragma once
#include "sim_kernels.cuh"

namespace grs {

struct EnvCfg {
  int max_steps, time_horizon, include_roll, her_buffer, im_reward, auto_reset, full_observation, obs_cam;
  float dir[2], pos_tol, grasp_tol, max_trans, max_rot;
  float reset_noise_xy, reset_noise_yaw;  // reset randomisation (0 = the reference's deterministic reset)
  unsigned seed;
};

// indices of the packed records; mirrored by include/b200_gripper_sim.h (GRS_ST_*, GRS_INFO_*)
enum { ST_QPOS = 0, ST_QVEL = 14, ST_CTRL = 27, ST_WARM = 34, ST_GRIPPER_OPEN = 47, ST_EPISODE_STEP = 48, ST_STATUS = 49, ST_XFRC_Z = 50,
       ST_EP_RETURN = 51, ST_EP_SUBSTEPS = 52, ST_STRIDE = 64 };
enum { IN_REWARD = 0, IN_DONE, IN_STATUS, IN_GRASP, IN_PHEROMONE, IN_OBJECT_GRASPED, IN_GRIPPER_OPEN, IN_REACHED_TARGET, IN_REACHED_INITIAL,
       IN_FAIL, IN_NSUB_A, IN_NSUB_B, IN_NSUB_C, IN_TOTAL_DISTANCE, IN_LINE_DISTANCE, IN_INIT_OBJ_POS, IN_FINAL_OBJ_POS = 18,
       IN_GRIPPER_POS = 21, IN_ACHIEVED = 24, IN_DESIRED = 26, IN_SOLVER_ITERS = 28, IN_NCON_MAX, IN_FLAGS, IN_EPISODE_STEP,
       IN_EPISODE_RETURN = 32, IN_EPISODE_SUBSTEPS, IN_TARGET_QPOS = 34, IN_STRIDE = 40 };
constexpr int RS_STRIDE = 96;

struct EnvFlags { int gripper_open, episode_step, status; float xfrc_z, ep_return, ep_substeps; };

__device__ __forceinline__ void load_state(WS& w, EnvFlags& f, const float* __restrict__ st, int lane) {
  if (lane < NQ) w.qpos[lane] = st[ST_QPOS + lane];
  if (lane < NV) { w.qvel[lane] = st[ST_QVEL + lane]; w.warm[lane] = st[ST_WARM + lane]; }
  if (lane < NU) w.ctrl[lane] = st[ST_CTRL + lane];
  f.gripper_open = (int)st[ST_GRIPPER_OPEN]; f.episode_step = (int)st[ST_EPISODE_STEP]; f.status = (int)st[ST_STATUS];
  f.xfrc_z = st[ST_XFRC_Z]; f.ep_return = st[ST_EP_RETURN]; f.ep_substeps = st[ST_EP_SUBSTEPS];
  for (int k = lane; k < MAXPAIR * 3; k += 32) (&w.sep[0][0])[k] = 0.0f;  // no separating-axis cache for a freshly loaded state
  __syncwarp();
}
__device__ __forceinline__ void store_state(const WS& w, const EnvFlags& f, float* __restrict__ st, int lane) {
  __syncwarp();
  if (lane < NQ) st[ST_QPOS + lane] = w.qpos[lane];
  if (lane < NV) { st[ST_QVEL + lane] = w.qvel[lane]; st[ST_WARM + lane] = w.warm[lane]; }
  if (lane < NU) st[ST_CTRL + lane] = w.ctrl[lane];
  if (lane == 0) {
    st[ST_GRIPPER_OPEN] = (float)f.gripper_open; st[ST_EPISODE_STEP] = (float)f.episode_step; st[ST_STATUS] = (float)f.status;
    st[ST_XFRC_Z] = f.xfrc_z; st[ST_EP_RETURN] = f.ep_return; st[ST_EP_SUBSTEPS] = f.ep_substeps;
  }
}

// actuator.py:134-184 — which finger bodies touch the object body (0 none, 1 finger 1, 2 finger 2, 3 both)
__device__ __forceinline__ int check_grasp(const DevModel& m, const WS& w) {
  int t1 = 0, t2 = 0;
  for (int c = 0; c < w.ncon; c++) {
    int b1 = m.geom_body[w.c_g1[c]], b2 = m.geom_body[w.c_g2[c]], other = -1;
    if (b1 == m.body_object) other = b2; else if (b2 == m.body_object) other = b1;
    if (other < 0) continue;
    if (other == m.finger1[0] || other == m.finger1[1]) t1 = 1;
    if (other == m.finger2[0] || other == m.finger2[1]) t2 = 1;
  }
  return t1 + 2 * t2;
}
// utils.py:30-31 — coefficient on the UN-normalised direction
__device__ __forceinline__ float project_dir(const float* p, const float* dir) { return (p[0] * dir[0] + p[1] * dir[1]) / (dir[0] * dir[0] + dir[1] * dir[1]); }
// actuator.py:198-215
__device__ __forceinline__ int pheromone_level(const DevModel& m, const WS& w, const float* dir) {
  const float* ee = w.xpos[m.body_ee];
  float pr = project_dir(ee, dir), dx = pr * dir[0] - ee[0], dy = pr * dir[1] - ee[1];
  float c = 1.0f / expf(sqrtf(dx * dx + dy * dy));
  return c > 0.82f ? 3 : c > 0.6f ? 2 : c > 0.37f ? 1 : 0;
}
// reward.py:18-41
__device__ __forceinline__ float agent_reward(const float* init_obj, const float* final_obj, const float* dir, int gripper_open, float c5, float c6, int grasped) {
  float reward = 0, ip = project_dir(init_obj, dir), fp = project_dir(final_obj, dir);
  float dx = fp * dir[0] - final_obj[0], dy = fp * dir[1] - final_obj[1];
  float lat = sqrtf(dx * dx + dy * dy), trav = fp - ip;
  if (trav > 0.f && trav < 0.1f && lat < 0.1f) {
    reward = trav;
    if (!gripper_open && (c5 != 0.f && c6 != 0.f) && grasped == 3) {  // `np.all(controls) != 0`
      reward *= 2;
      if (final_obj[2] > 0) reward *= 1.5f;
    }
  }
  return reward * 30;
}

// transformations.py:1035 euler_from_matrix(axes='sxyz'), returned as [roll(x), pitch(y), yaw(z)]
__device__ __forceinline__ void euler_sxyz_from_mat(const float* M, float* e) {
  float cy = sqrtf(M[0] * M[0] + M[3] * M[3]);
  if (cy > 8.8817842e-16f) { e[0] = atan2f(M[7], M[8]); e[1] = atan2f(-M[6], cy); e[2] = atan2f(M[3], M[0]); }
  else { e[0] = atan2f(-M[5], M[4]); e[1] = atan2f(-M[6], cy); e[2] = 0; }
}
// transformations.py:972 euler_matrix(ai, aj, ak, 'sxyz'), 3x3 part
__device__ __forceinline__ void euler_matrix_sxyz(float ai, float aj, float ak, float* M) {
  float si, ci, sj, cj, sk, ck;
  sincosf(ai, &si, &ci); sincosf(aj, &sj, &cj); sincosf(ak, &sk, &ck);
  float cc = ci * ck, cs = ci * sk, sc = si * ck, ss = si * sk;
  M[0] = cj * ck; M[1] = sj * sc - cs; M[2] = sj * cc + ss;
  M[3] = cj * sk; M[4] = sj * ss + cc; M[5] = sj * cs - sc;
  M[6] = -sj; M[7] = cj * si; M[8] = cj * ci;
}

// actuator.py:21-44 (_normalise_action), :58-102 (get_target_pose), :249-293 (clip / constraints).
// Executed by lane 0; the five target joint positions land in w.tgt.
__device__ __noinline__ void get_target_pose(const DevModel& m, const EnvCfg& c, WS& w, const float* a6) {
  float t[3] = {a6[0] * c.max_trans, a6[1] * c.max_trans, a6[2] * c.max_trans};
  float rot[2] = {a6[3] * c.max_rot, a6[4] * c.max_rot};
  float len = sqrtf(dot3(t, t));
  if (len > c.max_trans) { float s = c.max_trans / len; t[0] *= s; t[1] *= s; t[2] *= s; }
  for (int k = 0; k < 2; k++) rot[k] = fminf(fmaxf(rot[k], -c.max_rot), c.max_rot);
  const float* cur_pos = w.xpos[m.body_ee];
  const float* q = w.xquat[m.body_ee];
  float qn[4] = {q[0], q[1], q[2], q[3]}, Rq[9], cur_ori[3];
  quat_normalize(qn);
  quat2mat(Rq, qn);
  euler_sxyz_from_mat(Rq, cur_ori);
  float Rold[9], Rrel[9], Rnew[9], pos[3], ori[3];
  euler_matrix_sxyz(cur_ori[0], cur_ori[1], cur_ori[2], Rold);
  euler_matrix_sxyz(rot[0], 0.0f, rot[1], Rrel);
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) Rnew[3 * i + j] = Rold[3 * i] * Rrel[j] + Rold[3 * i + 1] * Rrel[3 + j] + Rold[3 * i + 2] * Rrel[6 + j];
  mulmat3vec(pos, Rold, t);
  for (int k = 0; k < 3; k++) pos[k] += cur_pos[k];
  euler_sxyz_from_mat(Rnew, ori);
  const float QPI = 0.78539816339744831f;
  if (!c.include_roll) ori[0] = 0; else ori[0] = fminf(fmaxf(ori[0], -QPI), QPI);
  ori[1] = 0;
  pos[2] = fminf(fmaxf(pos[2], 0.1f), 0.5f);
  float err[6];
  for (int k = 0; k < 3; k++) { err[k] = pos[k] - cur_pos[k]; err[3 + k] = ori[k] - cur_ori[k]; }
  // mj_jacBody(ee) restricted to the first five dofs, then pinv through the normal equations
  float J[6][5];
  for (int i = 0; i < 5; i++) {
    if ((m.body_dofmask[m.body_ee] >> i) & 1u) {
      float off[3], tt[3];
      for (int k = 0; k < 3; k++) off[k] = cur_pos[k] - w.com[m.body_ee][k];
      cross3(tt, w.cdof[i], off);
      for (int k = 0; k < 3; k++) { J[k][i] = w.cdof[i][3 + k] + tt[k]; J[3 + k][i] = w.cdof[i][k]; }
    } else {
      for (int k = 0; k < 6; k++) J[k][i] = 0;
    }
  }
  float A[5][5], b[5];
  for (int i = 0; i < 5; i++) {
    b[i] = 0;
    for (int r = 0; r < 6; r++) b[i] += J[r][i] * err[r];
    for (int k = 0; k < 5; k++) {
      float v = 0;
      for (int r = 0; r < 6; r++) v += J[r][i] * J[r][k];
      A[i][k] = v;
    }
  }
  for (int j = 0; j < 5; j++) {  // Cholesky
    float s = A[j][j];
    for (int k = 0; k < j; k++) s -= A[j][k] * A[j][k];
    s = sqrtf(fmaxf(s, 1e-30f));
    A[j][j] = s;
    for (int i = j + 1; i < 5; i++) {
      float v = A[i][j];
      for (int k = 0; k < j; k++) v -= A[i][k] * A[j][k];
      A[i][j] = v / s;
    }
  }
  for (int i = 0; i < 5; i++) { float s = b[i]; for (int k = 0; k < i; k++) s -= A[i][k] * b[k]; b[i] = s / A[i][i]; }
  for (int i = 4; i >= 0; i--) { float s = b[i]; for (int k = i + 1; k < 5; k++) s -= A[k][i] * b[k]; b[i] = s / A[i][i]; }
  for (int k = 0; k < 5; k++) w.tgt[k] = w.qpos[k] + b[k];
}

// engine_core_smooth.c : mj_camlight for one camera -> pos[3], mat[9] (camera looks along -z, x right, y up)
__device__ __forceinline__ void camera_pose(const DevModel& m, const WS& w, int cam, float* out12) {
  int b = m.cam_body[cam];
  float t[3], pos[3], mat[9];
  mulmat3vec(t, w.xmat[b], m.cam_pos[cam]);
  for (int k = 0; k < 3; k++) pos[k] = w.xpos[b][k] + t[k];
  if (m.cam_mode[cam] == 1 && m.cam_target[cam] >= 0) {
    float z[3], x[3], y[3], up[3] = {0, 0, 1};
    for (int k = 0; k < 3; k++) z[k] = pos[k] - w.com[m.cam_target[cam]][k];
    normalize3(z);
    cross3(x, up, z); normalize3(x);
    cross3(y, z, x); normalize3(y);
    for (int k = 0; k < 3; k++) { mat[3 * k] = x[k]; mat[3 * k + 1] = y[k]; mat[3 * k + 2] = z[k]; }
  } else {
    float q[4];
    quat_mul(q, w.xquat[b], m.cam_quat[cam]);
    quat_normalize(q);
    quat2mat(mat, q);
  }
  for (int k = 0; k < 3; k++) out12[k] = pos[k];
  for (int k = 0; k < 9; k++) out12[3 + k] = mat[k];
}
// geom poses + camera pose for the renderer
__device__ __forceinline__ void write_render_state(const DevModel& m, const WS& w, int cam, float* __restrict__ rs, int lane) {
  if (lane < m.ngeom && lane < 7) {
    for (int k = 0; k < 3; k++) rs[lane * 12 + k] = w.gpos[lane][k];
    for (int k = 0; k < 9; k++) rs[lane * 12 + 3 + k] = w.gmat[lane][k];
  }
  if (lane == 31) camera_pose(m, w, cam, rs + 84);
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(FULL, v, o));
  return v;
}

// robot_env.py:170-241 — everything after the substep loops: failure checks, goals, observation scalars, reward, done,
// info record (into w.out).  Called by the step kernel's controller (env_lockstep.cuh : env_tick) when an agent step ends.
struct StepCounters { int nsa, nsb, nsc, iters, nconmax, flags, fail, object_grasped; bool reached_target, reached_initial; float tq_rec; };

__device__ __noinline__ void env_finalize(const DevModel& m, const EnvCfg& c, WS& w, EnvFlags& f, const float* init_obj, StepCounters& k, int lane) {
  int nsa = k.nsa, nsb = k.nsb, nsc = k.nsc, iters = k.iters, nconmax = k.nconmax, flags = k.flags, fail = k.fail, object_grasped = k.object_grasped;
  const bool reached_target = k.reached_target, reached_initial = k.reached_initial;
  const float tq_rec = k.tq_rec;
  // NaN / Inf guard (MuJoCo's mj_checkAcc resets the data; here the episode ends as a FAIL and the env is reset)
  float chk = 0;
  if (lane < NQ) chk = w.qpos[lane];
  if (lane >= 16 && lane - 16 < NV) chk = w.qvel[lane - 16];
  bool bad = __any_sync(FULL, !isfinite(chk));
  if (bad) { flags |= 2; f.status = 1; fail = 1; }
  const float* fo = w.xpos[m.body_object];
  const float* fg = w.xpos[m.body_ee];
  float ddx = fo[0] - fg[0], ddy = fo[1] - fg[1];
  if (sqrtf(ddx * ddx + ddy * ddy) > 1.0f) f.status = 1;
  float pr = project_dir(fo, c.dir);
  float desired[2] = {pr * c.dir[0], pr * c.dir[1]}, achieved[2] = {fo[0], fo[1]};
  int grasp = check_grasp(m, w), pher = pheromone_level(m, w, c.dir);
  float reward = agent_reward(init_obj, fo, c.dir, f.gripper_open, w.ctrl[5], w.ctrl[6], object_grasped);
  if (c.her_buffer) {
    float gx = desired[0] - achieved[0], gy = desired[1] - achieved[1];
    reward += 1.0f / expf(sqrtf(gx * gx + gy * gy));
  }
  if (bad) reward = 0;
  int done;
  if (f.status != 0) done = 1;
  else if (f.episode_step == c.time_horizon - 1) { done = 1; f.status = 2; }
  else done = 0;
  float tdx = fo[0] - init_obj[0], tdy = fo[1] - init_obj[1];
  float ip = project_dir(init_obj, c.dir), ldx = pr * c.dir[0] - fo[0], ldy = pr * c.dir[1] - fo[1];
  float lat = sqrtf(ldx * ldx + ldy * ldy), trav = pr - ip;
  f.episode_step++;
  f.ep_return += reward;
  f.ep_substeps += (float)(nsa + nsb + nsc);
  __syncwarp();
  if (lane == 0) {
    float* o = w.out;
    o[IN_REWARD] = reward; o[IN_DONE] = (float)done; o[IN_STATUS] = (float)f.status; o[IN_GRASP] = (float)grasp; o[IN_PHEROMONE] = (float)pher;
    o[IN_OBJECT_GRASPED] = (float)object_grasped; o[IN_GRIPPER_OPEN] = (float)f.gripper_open; o[IN_REACHED_TARGET] = reached_target;
    o[IN_REACHED_INITIAL] = reached_initial; o[IN_FAIL] = (float)fail; o[IN_NSUB_A] = (float)nsa; o[IN_NSUB_B] = (float)nsb; o[IN_NSUB_C] = (float)nsc;
    o[IN_TOTAL_DISTANCE] = sqrtf(tdx * tdx + tdy * tdy);
    o[IN_LINE_DISTANCE] = (trav > 0.f && trav < 0.1f && lat < 0.1f) ? trav : 0.f;
    for (int k = 0; k < 3; k++) { o[IN_INIT_OBJ_POS + k] = init_obj[k]; o[IN_FINAL_OBJ_POS + k] = fo[k]; o[IN_GRIPPER_POS + k] = fg[k]; }
    o[IN_ACHIEVED] = achieved[0]; o[IN_ACHIEVED + 1] = achieved[1]; o[IN_DESIRED] = desired[0]; o[IN_DESIRED + 1] = desired[1];
    o[IN_SOLVER_ITERS] = (float)iters; o[IN_NCON_MAX] = (float)nconmax; o[IN_FLAGS] = (float)flags; o[IN_EPISODE_STEP] = (float)f.episode_step;
    o[IN_EPISODE_RETURN] = f.ep_return; o[IN_EPISODE_SUBSTEPS] = f.ep_substeps;
  }
  if (lane < 5) w.out[IN_TARGET_QPOS + lane] = tq_rec;
  if (lane >= 5 && lane < 6) w.out[IN_TARGET_QPOS + 5] = 0;
  __syncwarp();
}

// ----------------------------------------------------------------------------------------------- kernels
struct SimBuffers {
  float* state;         // [N][ST_STRIDE]
  float* info;          // [N][IN_STRIDE]
  float* reward;        // [N]
  unsigned char* done;  // [N]
  float* achieved;      // [N][2]
  float* desired;       // [N][2]
  float* render_state;  // [N][RS_STRIDE]
  float* reset_record;  // [ST_STRIDE] state + [IN_STRIDE] info + [RS_STRIDE] render state of a freshly reset environment
  float* debug;         // [N][DEBUG_STRIDE]
  int* queue;           // [0] work-queue counter, [1..2] bucket counters of the longest-first order, [3] finished environments,
                        // [4] observation tickets handed out, [5] blocks that left the fused kernel, [6] blocks that started,
                        // [16..63] class sizes / cursors of the queue order
  int* done_list;       // [N] environment ids in the order their agent steps finished (-1 = not yet); fused observation phase
  int* episode_count;   // [N] resets taken so far (reset randomisation: the hash counter)
  float* reset_obj;     // [N][12] pose (pos 3, mat 9) of the object geom at the start of the current episode (reset randomisation)
  int* sm_phys;         // [256] per SM: blocks of the fused kernel still in their physics phase (the observation phase yields to them)
  unsigned long long* tstamp;  // [0] first block start, [1] last physics-phase end (globaltimer ns), [2] sum of ([1]-[0]), [3] launches
  int* order;           // [N] environment ids, expected-long agent steps first (k_order_envs); identity for the other kernels
  const float4* hull;
  int hull_count;       // float4 entries behind `hull`; the lock-step kernel copies them to shared memory when hull_smem is set
  int hull_smem;
  const int* adj;
  const DevModel* model;
  int n;
};
constexpr int DEBUG_STRIDE = 2048;
constexpr int WARPS_PER_BLOCK = 4;


// ---- reset randomisation (not in the reference, SURVEY.md §8f N4).  u in [-1, 1) from a counter-based hash, so a reset is
// a pure function of (seed, environment, episode index, k): any kernel, any order, reproducible; mirrored in tests/.
__host__ __device__ inline float reset_uniform(unsigned seed, unsigned env, unsigned episode, unsigned k) {
  unsigned h = seed * 0x9E3779B1u ^ env * 0x85EBCA77u ^ episode * 0xC2B2AE3Du ^ k * 0x27D4EB2Fu;
  h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12; h *= 0x297A2D39u; h ^= h >> 15;
  return (float)(h >> 8) * (2.0f / 16777216.0f) - 1.0f;
}
// `st` already holds the reset record.  Moves / turns the free object, records the pose of its geom for the observation of the
// new episode and the achieved goal (object xy, robot_env.py:71).  One lane suffices (called by lane 0).
__device__ inline void apply_reset_noise(const SimBuffers& s, const DevModel& m, const EnvCfg& c, int env, float* st) {
  const unsigned ep = (unsigned)(s.episode_count[env] += 1);
  const int qa = m.jnt_qposadr[m.body_jntadr[m.body_object]];  // free joint of the object: pos 3, quat 4
  const float dx = c.reset_noise_xy * reset_uniform(c.seed, env, ep, 0), dy = c.reset_noise_xy * reset_uniform(c.seed, env, ep, 1);
  const float yaw = c.reset_noise_yaw * reset_uniform(c.seed, env, ep, 2);
  float p[3] = {st[ST_QPOS + qa] + dx, st[ST_QPOS + qa + 1] + dy, st[ST_QPOS + qa + 2]};
  float q0[4] = {st[ST_QPOS + qa + 3], st[ST_QPOS + qa + 4], st[ST_QPOS + qa + 5], st[ST_QPOS + qa + 6]}, qz[4], q[4];
  sincosf(0.5f * yaw, &qz[3], &qz[0]);
  qz[1] = 0; qz[2] = 0;
  quat_mul(q, qz, q0);  // world-frame yaw applied on the left
  quat_normalize(q);
  for (int k = 0; k < 3; k++) st[ST_QPOS + qa + k] = p[k];
  for (int k = 0; k < 4; k++) st[ST_QPOS + qa + 3 + k] = q[k];
  int g = 0;
  for (int i = 0; i < m.ngeom; i++) if (m.geom_body[i] == m.body_object) { g = i; break; }
  float R[9], Rg[9], t[3];
  quat2mat(R, q);
  quat2mat(Rg, m.geom_quat[g]);
  mulmat3vec(t, R, m.geom_pos[g]);
  float* o = s.reset_obj + (size_t)env * 12;
  for (int k = 0; k < 3; k++) o[k] = p[k] + t[k];
  for (int r = 0; r < 3; r++)
    for (int cc = 0; cc < 3; cc++) o[3 + 3 * r + cc] = R[3 * r] * Rg[cc] + R[3 * r + 1] * Rg[3 + cc] + R[3 * r + 2] * Rg[6 + cc];
  s.achieved[2 * env] = p[0]; s.achieved[2 * env + 1] = p[1];
}

extern __shared__ __align__(16) unsigned char grs_smem[];

__device__ __forceinline__ const DevModel& stage_model(const DevModel* gm) {
  DevModel* sm = reinterpret_cast<DevModel*>(grs_smem);
  const int nw = sizeof(DevModel) / 4;
  const unsigned* src = reinterpret_cast<const unsigned*>(gm);
  unsigned* dst = reinterpret_cast<unsigned*>(sm);
  for (int i = threadIdx.x; i < nw; i += blockDim.x) dst[i] = src[i];
  __syncthreads();
  return *sm;
}
__device__ __forceinline__ WS& my_ws() {
  constexpr int off = (sizeof(DevModel) + 15) / 16 * 16;
  return reinterpret_cast<WS*>(grs_smem + off)[threadIdx.x >> 5];
}
inline size_t smem_bytes() { return (sizeof(DevModel) + 15) / 16 * 16 + WARPS_PER_BLOCK * sizeof(WS); }

__device__ __forceinline__ int next_env(int* queue, int lane) {
  int e = 0;
  if (lane == 0) e = atomicAdd(queue, 1);
  return __shfl_sync(FULL, e, 0);
}

// RobotEnv.reset executed once (every environment starts from qpos0 — the reference has no reset randomisation):
// mj_resetData + mj_forward with actuation disabled (dm_control Physics.reset), then the env bookkeeping of robot_env.py:62-73
__global__ void __launch_bounds__(32) k_make_reset_record(SimBuffers s, EnvCfg c) {
  const DevModel& m = stage_model(s.model);
  WS& w = my_ws();
  const int lane = threadIdx.x & 31;
  if (lane < NQ) w.qpos[lane] = m.qpos0[lane];
  for (int k = lane; k < MAXPAIR * 3; k += 32) (&w.sep[0][0])[k] = 0.0f;
  if (lane < NV) { w.qvel[lane] = 0; w.warm[lane] = 0; }
  if (lane < NU) w.ctrl[lane] = 0;
  __syncwarp();
  forward_position(m, w, s.hull, s.adj, lane);
  smooth_forces(m, w, lane, false, 0.0f);
  make_constraint(m, w, lane);
  solve_newton(m, w, lane, m.iterations);
  if (lane < NV) w.warm[lane] = w.qacc[lane];
  __syncwarp();
  EnvFlags f;
  f.gripper_open = 1; f.episode_step = 0; f.status = 0; f.xfrc_z = m.xfrc_ee_z; f.ep_return = 0; f.ep_substeps = 0;
  for (int k = lane; k < ST_STRIDE; k += 32) s.reset_record[k] = 0;
  __syncwarp();
  store_state(w, f, s.reset_record, lane);
  float* o = s.reset_record + ST_STRIDE;
  for (int k = lane; k < IN_STRIDE; k += 32) o[k] = 0;
  __syncwarp();
  if (lane == 0) {
    o[IN_GRASP] = (float)check_grasp(m, w);
    o[IN_PHEROMONE] = (float)pheromone_level(m, w, c.dir);
    o[IN_GRIPPER_OPEN] = 1;
    o[IN_ACHIEVED] = w.xpos[m.body_object][0]; o[IN_ACHIEVED + 1] = w.xpos[m.body_object][1];
    o[IN_DESIRED] = c.dir[0]; o[IN_DESIRED + 1] = c.dir[1];  // robot_env.py:72 — the direction itself, not a projection
    for (int k = 0; k < 3; k++) { o[IN_FINAL_OBJ_POS + k] = w.xpos[m.body_object][k]; o[IN_GRIPPER_POS + k] = w.xpos[m.body_ee][k]; }
    o[IN_NCON_MAX] = (float)w.ncon;
  }
  write_render_state(m, w, c.obs_cam, s.reset_record + ST_STRIDE + IN_STRIDE, lane);
}

// RobotEnv.reset for the masked environments: copy the reset record
__global__ void k_reset(SimBuffers s, EnvCfg c, const unsigned char* __restrict__ mask) {
  const int env = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (env >= s.n) return;
  if (mask && !mask[env]) return;
  for (int k = lane; k < ST_STRIDE; k += 32) s.state[(size_t)env * ST_STRIDE + k] = s.reset_record[k];
  for (int k = lane; k < IN_STRIDE; k += 32) s.info[(size_t)env * IN_STRIDE + k] = s.reset_record[ST_STRIDE + k];
  for (int k = lane; k < RS_STRIDE; k += 32) s.render_state[(size_t)env * RS_STRIDE + k] = s.reset_record[ST_STRIDE + IN_STRIDE + k];
  if (lane == 0) {
    s.reward[env] = 0; s.done[env] = 0;
    s.achieved[2 * env] = s.reset_record[ST_STRIDE + IN_ACHIEVED]; s.achieved[2 * env + 1] = s.reset_record[ST_STRIDE + IN_ACHIEVED + 1];
    s.desired[2 * env] = s.reset_record[ST_STRIDE + IN_DESIRED]; s.desired[2 * env + 1] = s.reset_record[ST_STRIDE + IN_DESIRED + 1];
  }
  __syncwarp();
  if (lane == 0 && (c.reset_noise_xy != 0.f || c.reset_noise_yaw != 0.f)) apply_reset_noise(s, *s.model, c, env, s.state + (size_t)env * ST_STRIDE);
}

// n x physics.step() with the controls held in the state (parity tests; robot_env.py:100)
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, 5) k_substep(SimBuffers s, int nsteps) {
  const DevModel& m = stage_model(s.model);
  WS& w = my_ws();
  const int lane = threadIdx.x & 31;
  for (int env = next_env(s.queue, lane); env < s.n; env = next_env(s.queue, lane)) {
    EnvFlags f;
    float* st = s.state + (size_t)env * ST_STRIDE;
    load_state(w, f, st, lane);
    forward_position(m, w, s.hull, s.adj, lane);
    for (int i = 0; i < nsteps; i++) physics_step(m, w, s.hull, s.adj, lane, f.xfrc_z, true);
    store_state(w, f, st, lane);
    __syncwarp();
  }
}

// contacts of the current state -> debug buffer: [0] ncon, then per contact K: g1, g2, dist, pos[3], frame[9]  (stride 15)
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32) k_contacts(SimBuffers s) {
  const DevModel& m = stage_model(s.model);
  WS& w = my_ws();
  const int lane = threadIdx.x & 31;
  for (int env = next_env(s.queue, lane); env < s.n; env = next_env(s.queue, lane)) {
    EnvFlags f;
    load_state(w, f, s.state + (size_t)env * ST_STRIDE, lane);
    forward_position(m, w, s.hull, s.adj, lane);
    float* d = s.debug + (size_t)env * DEBUG_STRIDE;
    if (lane == 0) { d[0] = (float)w.ncon; d[1] = (float)w.overflow; }
    if (lane < w.ncon) {
      float* o = d + 2 + lane * 15;
      o[0] = (float)w.c_g1[lane]; o[1] = (float)w.c_g2[lane]; o[2] = w.c_dist[lane];
      for (int k = 0; k < 3; k++) o[3 + k] = w.c_pos[lane][k];
      for (int k = 0; k < 9; k++) o[6 + k] = w.c_frame[lane][k];
    }
    // body poses for kinematics parity: xpos [200..236), xquat [236..284)
    for (int k = lane; k < MAXB * 3; k += 32) d[200 + k] = (&w.xpos[0][0])[k];
    for (int k = lane; k < MAXB * 4; k += 32) d[236 + k] = (&w.xquat[0][0])[k];
    __syncwarp();
  }
}

// one physics.step() with a dump of the intermediate quantities (layout documented in python/_debug_layout)
enum { DBG_M = 0, DBG_BIAS = 169, DBG_FSMOOTH = 182, DBG_ASMOOTH = 195, DBG_NCON = 208, DBG_NEFC = 209, DBG_NLIM = 210, DBG_ITERS = 211,
       DBG_QACC = 212, DBG_FCON = 225, DBG_D = 238, DBG_AREF = 293, DBG_FORCE = 348, DBG_J = 403, DBG_CONTACT = 1118 /* 12 x 15 */, DBG_MU = 1298, DBG_END = 1310 };
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32) k_debug_step(SimBuffers s) {
  const DevModel& m = stage_model(s.model);
  WS& w = my_ws();
  const int lane = threadIdx.x & 31;
  for (int env = next_env(s.queue, lane); env < s.n; env = next_env(s.queue, lane)) {
    EnvFlags f;
    float* st = s.state + (size_t)env * ST_STRIDE;
    load_state(w, f, st, lane);
    forward_position(m, w, s.hull, s.adj, lane);
    float* d = s.debug + (size_t)env * DEBUG_STRIDE;
    for (int k = lane; k < DEBUG_STRIDE; k += 32) d[k] = 0;
    __syncwarp();
    if (lane < w.ncon) {
      float* o = d + DBG_CONTACT + lane * 15;
      o[0] = (float)w.c_g1[lane]; o[1] = (float)w.c_g2[lane]; o[2] = w.c_dist[lane];
      for (int k = 0; k < 3; k++) o[3 + k] = w.c_pos[lane][k];
      for (int k = 0; k < 9; k++) o[6 + k] = w.c_frame[lane][k];
    }
    smooth_forces(m, w, lane, true, f.xfrc_z);
    for (int k = lane; k < NV * NV; k += 32) d[DBG_M + k] = w.M[k];
    if (lane < NV) { d[DBG_BIAS + lane] = w.bias[lane]; d[DBG_FSMOOTH + lane] = w.fsmooth[lane]; d[DBG_ASMOOTH + lane] = w.asmooth[lane]; }
    make_constraint(m, w, lane);
    int it = solve_newton(m, w, lane, m.iterations);
    if (lane == 0) { d[DBG_NCON] = (float)w.ncon; d[DBG_NEFC] = (float)w.nefc; d[DBG_NLIM] = (float)w.nlim; d[DBG_ITERS] = (float)it; }
    if (lane < NV) { d[DBG_QACC + lane] = w.qacc[lane]; d[DBG_FCON + lane] = w.fcon[lane]; }
    for (int r = lane; r < w.nefc; r += 32) { d[DBG_D + r] = w.e_D[r]; d[DBG_AREF + r] = w.e_aref[r]; d[DBG_FORCE + r] = w.e_force[r]; }
    for (int k = lane; k < w.nefc * NV; k += 32) d[DBG_J + k] = (&w.u.con.J[0][0])[k];
    if (lane < w.ncon) d[DBG_MU + lane] = w.c_mu[lane];
    __syncwarp();
    euler_integrate(m, w, lane);
    forward_position(m, w, s.hull, s.adj, lane);
    store_state(w, f, st, lane);
    __syncwarp();
  }
}

}  // namespace grs
