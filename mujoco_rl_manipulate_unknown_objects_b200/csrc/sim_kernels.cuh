// Device-side physics of the batched gripper simulator: ONE WARP PER ENVIRONMENT.
//
// Every stage of `physics.step()` (reference robot_env.py:100,119,142,157 -> dm_control -> MuJoCo mj_step2 +
// mj_step1) is executed cooperatively by the 32 lanes of a warp on a per-warp shared-memory workspace (WS):
//   kinematics -> comPos -> crb -> (factor) -> comVel -> rne -> collision (plane-hull, MPR hull-hull)
//   -> constraint rows (limits + elliptic condim-4 contacts) -> Newton solve -> implicit-damped Euler.
// Lanes map to bodies / dofs / hull vertices / constraint rows / Hessian entries depending on the stage;
// scalars that are uniform over the warp (MPR portal, line-search state, controller state) live in registers.
// fp32 throughout.  The fp64 restatement in oracle/engine.c is the parity reference (tests/ only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "model.h"

namespace grs {

constexpr int MAXCON = 12;              // contacts kept per environment (typical 3-8, SURVEY.md §8 a-M)
constexpr int MAXEFC = MAXCON * 4 + 7;  // + one row per limited joint
constexpr unsigned FULL = 0xffffffffu;
constexpr float MINVAL = 1e-15f;

// -------------------------------------------------------------------------------- per-warp workspace
struct __align__(16) WS {
  // state
  float qpos[16], qvel[16], ctrl[8], warm[16];
  // position stage
  float xpos[MAXB][3], xquat[MAXB][4], xmat[MAXB][9];
  float xanchor[MAXJ][3], xaxis[MAXJ][3];
  float gpos[MAXG][3], gmat[MAXG][9];
  float com[MAXB][3];  // subtree CoM of the tree root of each body
  float cdof[16][6];
  float M[NV * NV];
  // contacts
  int ncon, nefc, nlim, overflow, coupled, padi[3];
  float c_dist[MAXCON], c_pos[MAXCON][3], c_frame[MAXCON][9], c_mu[MAXCON], c_fric[MAXCON][3];
  int c_g1[MAXCON], c_g2[MAXCON], c_pair[MAXCON];
  // dof-space vectors
  float fsmooth[16], asmooth[16], qacc[16], Ma[16], grad[16], search[16], Mv[16], fcon[16], bias[16];
  // rows
  float e_D[MAXEFC], e_aref[MAXEFC], e_jar[MAXEFC], e_Jv[MAXEFC], e_force[MAXEFC], e_act[MAXEFC];
  float hc[MAXCON][16];
  int istate[32];
  // environment layer (env_kernels.cuh): controller targets and the staged per-step record
  float tgt[8], init_q[8], out[40];
  float sup[5][9];  // MPR portal (collision)
  float cho[16];    // Cholesky right-hand side / solution exchange
  float sep[MAXPAIR][3];  // last separating direction found for each convex pair (zero = none); temporal coherence only
  float gapb[MAXPAIR];    // separation left along sep[p] after subtracting how far the two geoms can have moved since it was measured
  float disp[MAXG];       // bound on the motion of any point of geom g during the last substep (kinematics)
  union {
    struct {  // smooth-dynamics scratch (dead once qfrc_bias is known)
      float xipos[MAXB][3], ximat[MAXB][9], cinert[MAXB][10], crb[MAXB][10], cdofdot[16][6], cvel[MAXB][6], cfrc[MAXB][6];
      float L[NV * NV];
    } dyn;
    struct {  // constraint scratch
      float J[MAXEFC][NV];
      float H[NV * NV];
    } con;
  } u;
};

struct StepStats { int iters_total, max_iters, ncon_max; };

// -------------------------------------------------------------------------------- small helpers
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}
__device__ __forceinline__ float dot3(const float* a, const float* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
__device__ __forceinline__ void cross3(float* r, const float* a, const float* b) {
  float x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  r[0] = x; r[1] = y; r[2] = z;
}
__device__ __forceinline__ float normalize3(float* a) {
  float n = sqrtf(dot3(a, a));
  if (n < MINVAL) { a[0] = 1; a[1] = 0; a[2] = 0; return n; }
  float inv = 1.0f / n;
  a[0] *= inv; a[1] *= inv; a[2] *= inv;
  return n;
}
__device__ __forceinline__ void quat_mul(float* r, const float* a, const float* b) {
  float t0 = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3];
  float t1 = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2];
  float t2 = a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1];
  float t3 = a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0];
  r[0] = t0; r[1] = t1; r[2] = t2; r[3] = t3;
}
__device__ __forceinline__ void quat_normalize(float* q) {
  float n = sqrtf(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  if (n < MINVAL) { q[0] = 1; q[1] = q[2] = q[3] = 0; return; }
  float inv = 1.0f / n;
  q[0] *= inv; q[1] *= inv; q[2] *= inv; q[3] *= inv;
}
__device__ __forceinline__ void quat2mat(float* R, const float* q) {
  float w = q[0], x = q[1], y = q[2], z = q[3];
  R[0] = w * w + x * x - y * y - z * z; R[1] = 2 * (x * y - w * z); R[2] = 2 * (x * z + w * y);
  R[3] = 2 * (x * y + w * z); R[4] = w * w - x * x + y * y - z * z; R[5] = 2 * (y * z - w * x);
  R[6] = 2 * (x * z - w * y); R[7] = 2 * (y * z + w * x); R[8] = w * w - x * x - y * y + z * z;
}
__device__ __forceinline__ void mulmat3vec(float* r, const float* R, const float* v) {
  float x = R[0] * v[0] + R[1] * v[1] + R[2] * v[2], y = R[3] * v[0] + R[4] * v[1] + R[5] * v[2], z = R[6] * v[0] + R[7] * v[1] + R[8] * v[2];
  r[0] = x; r[1] = y; r[2] = z;
}
__device__ __forceinline__ void mulmat3Tvec(float* r, const float* R, const float* v) {
  float x = R[0] * v[0] + R[3] * v[1] + R[6] * v[2], y = R[1] * v[0] + R[4] * v[1] + R[7] * v[2], z = R[2] * v[0] + R[5] * v[1] + R[8] * v[2];
  r[0] = x; r[1] = y; r[2] = z;
}
__device__ __forceinline__ void rot_vec_quat(float* r, const float* v, const float* q) {
  float R[9];
  quat2mat(R, q);
  mulmat3vec(r, R, v);
}
// spatial inertia (Ixx Iyy Izz Ixy Ixz Iyz, m*d, m) times motion vector [ang;lin]
__device__ __forceinline__ void mul_inert_vec(float* r, const float* c, const float* v) {
  float t[3];
  r[0] = c[0] * v[0] + c[3] * v[1] + c[4] * v[2];
  r[1] = c[3] * v[0] + c[1] * v[1] + c[5] * v[2];
  r[2] = c[4] * v[0] + c[5] * v[1] + c[2] * v[2];
  cross3(t, c + 6, v + 3);
  r[0] += t[0]; r[1] += t[1]; r[2] += t[2];
  cross3(t, c + 6, v);
  r[3] = c[9] * v[3] - t[0]; r[4] = c[9] * v[4] - t[1]; r[5] = c[9] * v[5] - t[2];
}
__device__ __forceinline__ float dot6(const float* a, const float* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3] + a[4] * b[4] + a[5] * b[5]; }
__device__ __forceinline__ void cross_motion(float* r, const float* v, const float* mv) {
  float t[3];
  cross3(r, v, mv);
  cross3(r + 3, v, mv + 3);
  cross3(t, v + 3, mv);
  r[3] += t[0]; r[4] += t[1]; r[5] += t[2];
}
__device__ __forceinline__ void cross_force(float* r, const float* v, const float* f) {
  float t[3];
  cross3(r, v, f);
  cross3(t, v + 3, f + 3);
  r[0] += t[0]; r[1] += t[1]; r[2] += t[2];
  cross3(r + 3, v, f + 3);
}

// Fused 13x13 Cholesky factorisation + solve:  x = (L L^T)^-1 b,  A (shared memory, row stride NV, lower triangle read)
// is overwritten by L.  Lane i keeps row i in registers; column j is exchanged through A's own column in shared memory
// (one __syncwarp per column, no shuffles).  The right-hand side rides along as an extra matrix row held by an otherwise
// idle lane, so the forward substitution costs nothing: after the factorisation that lane holds y = L^-1 b.
// Two shapes:
//   BLOCKS = false  dense 13x13 (Newton Hessian when a gripper/object contact couples the two kinematic trees)
//   BLOCKS = true   block diagonal 7x7 (gripper tree, lanes 0-6, rhs lane 13) + 6x6 (free object, lanes 7-12, rhs lane 14),
//                   both factorised at once: M, M + h*damping, and the Hessian whenever no contact couples the trees.
template <bool BLOCKS>
__device__ __noinline__ float chol_factor_solve(float* A, float* tmp, float b, int lane) {
  constexpr int NB = BLOCKS ? 7 : NV;
  const bool is_row = lane < NV;
  const bool is_rhs = BLOCKS ? (lane == 13 || lane == 14) : (lane == NV);
  const int base = BLOCKS ? (((lane >= 7 && lane < NV) || lane == 14) ? 7 : 0) : 0;
  const int nb = BLOCKS ? (base ? 6 : 7) : NV;  // rows of this lane's block
  const int lr = is_rhs ? NB : lane - base;      // local row (the rhs row sits below the block)
  if (is_row) tmp[lane] = b;
  __syncwarp();
  float a[NB];
#pragma unroll
  for (int k = 0; k < NB; k++) {
    a[k] = 0.0f;
    if (k < nb) {
      if (is_row && k <= lr) a[k] = A[lane * NV + base + k];
      else if (is_rhs) a[k] = tmp[base + k];
    }
  }
#pragma unroll
  for (int j = 0; j < NB; j++) {
    if (is_row && lr >= j) A[lane * NV + base + j] = a[j];  // publish the (unscaled) column j
    __syncwarp();
    const int cj = base + (j < nb ? j : 0);
    const float djj = A[cj * NV + cj];
    float rs = rsqrtf(fmaxf(djj, 1e-30f));
    rs = rs * (1.5f - 0.5f * djj * rs * rs);  // one Newton step: full fp32 accuracy
    const float t = a[j] * rs * rs;
    a[j] *= rs;
#pragma unroll
    for (int k = j + 1; k < NB; k++) {
      const int rk = base + (k < nb ? k : 0);
      a[k] -= t * A[rk * NV + cj];
    }
  }
  __syncwarp();
  if (is_row) {
#pragma unroll
    for (int k = 0; k < NB; k++)
      if (k <= lr) A[lane * NV + base + k] = a[k];
  }
  if (is_rhs) {
#pragma unroll
    for (int k = 0; k < NB; k++)
      if (k < nb) tmp[base + k] = a[k];
  }
  __syncwarp();
  float y = is_row ? tmp[lane] : 0.0f;
  // backward substitution L^T x = y, one column per step, x_j broadcast through tmp
#pragma unroll
  for (int j = NB - 1; j >= 0; j--) {
    const bool valid = j < nb;
    const int gj = base + (valid ? j : 0);
    const float ljj = A[gj * NV + gj];
    if (is_row && valid && lr == j) tmp[gj] = __fdividef(y, ljj);
    __syncwarp();
    const float xj = tmp[gj];
    if (is_row && valid) {
      if (lr == j) y = xj;
      else if (lr < j) y -= A[gj * NV + lane] * xj;
    }
  }
  __syncwarp();
  return y;
}

// -------------------------------------------------------------------------------- position stage
// engine_core_smooth.c : mj_kinematics — lanes = bodies of one depth level
static __device__ __noinline__ void kinematics(const DevModel& m, WS& w, int lane) {
  if (lane == 0) {
    // mj_normalizeQuat on the free joint
    for (int j = 0; j < m.njnt; j++)
      if (m.jnt_type[j] == JNT_FREE) quat_normalize(w.qpos + m.jnt_qposadr[j] + 3);
    w.xpos[0][0] = w.xpos[0][1] = w.xpos[0][2] = 0;
    w.xquat[0][0] = 1; w.xquat[0][1] = w.xquat[0][2] = w.xquat[0][3] = 0;
    quat2mat(w.xmat[0], w.xquat[0]);
  }
  __syncwarp();
  for (int lv = 1; lv < m.nlevel; lv++) {
    int idx = m.level_start[lv] + lane;
    if (idx < m.level_start[lv + 1]) {
      int b = m.level_body[idx], pid = m.body_parent[b];
      int jadr = m.body_jntadr[b], jnum = m.body_jntnum[b];
      float pos[3], quat[4];
      if (jnum == 1 && m.jnt_type[jadr] == JNT_FREE) {
        int qa = m.jnt_qposadr[jadr];
        for (int k = 0; k < 3; k++) pos[k] = w.qpos[qa + k];
        for (int k = 0; k < 4; k++) quat[k] = w.qpos[qa + 3 + k];
        for (int k = 0; k < 3; k++) { w.xanchor[jadr][k] = pos[k]; w.xaxis[jadr][k] = 0; }
      } else {
        float t[3];
        mulmat3vec(t, w.xmat[pid], m.body_pos[b]);
        for (int k = 0; k < 3; k++) pos[k] = w.xpos[pid][k] + t[k];
        quat_mul(quat, w.xquat[pid], m.body_quat[b]);
        for (int kj = 0; kj < jnum; kj++) {
          int j = jadr + kj;
          float anchor[3], axis[3];
          rot_vec_quat(t, m.jnt_pos[j], quat);
          for (int k = 0; k < 3; k++) anchor[k] = pos[k] + t[k];
          rot_vec_quat(axis, m.jnt_axis[j], quat);
          float q = w.qpos[m.jnt_qposadr[j]] - m.jnt_qpos0[j];
          if (m.jnt_type[j] == JNT_SLIDE) {
            for (int k = 0; k < 3; k++) pos[k] += axis[k] * q;
          } else {
            float s, c, ql[4];
            sincosf(0.5f * q, &s, &c);
            ql[0] = c; ql[1] = m.jnt_axis[j][0] * s; ql[2] = m.jnt_axis[j][1] * s; ql[3] = m.jnt_axis[j][2] * s;
            quat_mul(quat, quat, ql);
            rot_vec_quat(t, m.jnt_pos[j], quat);
            for (int k = 0; k < 3; k++) pos[k] = anchor[k] - t[k];
          }
          for (int k = 0; k < 3; k++) { w.xanchor[j][k] = anchor[k]; w.xaxis[j][k] = axis[k]; }
        }
      }
      quat_normalize(quat);
      for (int k = 0; k < 3; k++) w.xpos[b][k] = pos[k];
      for (int k = 0; k < 4; k++) w.xquat[b][k] = quat[k];
      quat2mat(w.xmat[b], quat);
    }
    __syncwarp();
  }
  if (lane < m.ngeom) {
    int g = lane, b = m.geom_body[g];
    float t[3], q[4], R[9];
    mulmat3vec(t, w.xmat[b], m.geom_pos[g]);
    quat_mul(q, w.xquat[b], m.geom_quat[g]);
    quat_normalize(q);
    quat2mat(R, q);
    // how far any point of the geom can have moved since the previous pose: |dp| + rbound * |dR|_F  (collision: gapb)
    float d2 = 0, r2 = 0;
    for (int k = 0; k < 3; k++) { const float np_ = w.xpos[b][k] + t[k], d = np_ - w.gpos[g][k]; d2 += d * d; w.gpos[g][k] = np_; }
    for (int k = 0; k < 9; k++) { const float d = R[k] - w.gmat[g][k]; r2 += d * d; w.gmat[g][k] = R[k]; }
    w.disp[g] = sqrtf(d2) + m.geom_rbound[g] * sqrtf(r2);
  }
  __syncwarp();
}

// engine_core_smooth.c : mj_comPos + mj_crb.  Leaves cdof, com, M (with armature) and the dyn scratch (cinert) filled.
static __device__ __noinline__ void com_pos_crb(const DevModel& m, WS& w, int lane) {
  const int nb = m.nbody;
  if (lane < nb) {
    int b = lane;
    float t[3], qi[4];
    mulmat3vec(t, w.xmat[b], m.body_ipos[b]);
    for (int k = 0; k < 3; k++) w.u.dyn.xipos[b][k] = w.xpos[b][k] + t[k];
    quat_mul(qi, w.xquat[b], m.body_iquat[b]);
    quat2mat(w.u.dyn.ximat[b], qi);
  }
  __syncwarp();
  if (lane < nb) {  // subtree CoM of this body's tree root
    int r = m.body_root[lane];
    unsigned mask = m.body_subtree_mask[r];
    float s[3] = {0, 0, 0}, ms = 0;
    for (int b = 1; b < nb; b++)
      if ((mask >> b) & 1u) {
        float mb = m.body_mass[b];
        ms += mb;
        for (int k = 0; k < 3; k++) s[k] += mb * w.u.dyn.xipos[b][k];
      }
    if (ms < MINVAL) { for (int k = 0; k < 3; k++) w.com[lane][k] = w.u.dyn.xipos[r][k]; }
    else { float inv = 1.0f / ms; for (int k = 0; k < 3; k++) w.com[lane][k] = s[k] * inv; }
  }
  __syncwarp();
  if (lane < nb) {  // cinert
    int b = lane;
    float* c = w.u.dyn.cinert[b];
    if (b == 0) { for (int k = 0; k < 10; k++) c[k] = 0; }
    else {
      const float* R = w.u.dyn.ximat[b];
      const float* I = m.body_inertia[b];
      float mb = m.body_mass[b], off[3];
      for (int k = 0; k < 3; k++) off[k] = w.u.dyn.xipos[b][k] - w.com[b][k];
      float dd = dot3(off, off);
      float M00 = R[0] * I[0] * R[0] + R[1] * I[1] * R[1] + R[2] * I[2] * R[2];
      float M11 = R[3] * I[0] * R[3] + R[4] * I[1] * R[4] + R[5] * I[2] * R[5];
      float M22 = R[6] * I[0] * R[6] + R[7] * I[1] * R[7] + R[8] * I[2] * R[8];
      float M01 = R[0] * I[0] * R[3] + R[1] * I[1] * R[4] + R[2] * I[2] * R[5];
      float M02 = R[0] * I[0] * R[6] + R[1] * I[1] * R[7] + R[2] * I[2] * R[8];
      float M12 = R[3] * I[0] * R[6] + R[4] * I[1] * R[7] + R[5] * I[2] * R[8];
      c[0] = M00 + mb * (dd - off[0] * off[0]);
      c[1] = M11 + mb * (dd - off[1] * off[1]);
      c[2] = M22 + mb * (dd - off[2] * off[2]);
      c[3] = M01 - mb * off[0] * off[1];
      c[4] = M02 - mb * off[0] * off[2];
      c[5] = M12 - mb * off[1] * off[2];
      c[6] = mb * off[0]; c[7] = mb * off[1]; c[8] = mb * off[2];
      c[9] = mb;
    }
  }
  if (lane < NV) {  // cdof
    int i = lane, j = m.dof_jnt[i], b = m.dof_body[i], da = m.jnt_dofadr[j];
    float* c = w.cdof[i];
    int type = m.jnt_type[j];
    if (type == JNT_FREE) {
      int k = i - da;
      if (k < 3) { c[0] = c[1] = c[2] = 0; c[3] = k == 0; c[4] = k == 1; c[5] = k == 2; }
      else {
        k -= 3;
        float ax[3] = {w.xmat[b][k], w.xmat[b][3 + k], w.xmat[b][6 + k]}, off[3];
        for (int q = 0; q < 3; q++) off[q] = w.com[b][q] - w.xpos[b][q];
        c[0] = ax[0]; c[1] = ax[1]; c[2] = ax[2];
        cross3(c + 3, ax, off);
      }
    } else if (type == JNT_SLIDE) {
      c[0] = c[1] = c[2] = 0;
      for (int q = 0; q < 3; q++) c[3 + q] = w.xaxis[j][q];
    } else {
      float off[3], ax[3];
      for (int q = 0; q < 3; q++) { off[q] = w.com[b][q] - w.xanchor[j][q]; ax[q] = w.xaxis[j][q]; c[q] = ax[q]; }
      cross3(c + 3, ax, off);
    }
  }
  __syncwarp();
  if (lane < nb) {  // composite inertia of the subtree
    int b = lane;
    unsigned mask = m.body_subtree_mask[b];
    float acc[10];
    for (int k = 0; k < 10; k++) acc[k] = 0;
    if (b > 0)
      for (int bb = b; bb < nb; bb++)
        if ((mask >> bb) & 1u)
          for (int k = 0; k < 10; k++) acc[k] += w.u.dyn.cinert[bb][k];
    for (int k = 0; k < 10; k++) w.u.dyn.crb[b][k] = acc[k];
  }
  __syncwarp();
  float buf[6];
  if (lane < NV) mul_inert_vec(buf, w.u.dyn.crb[m.dof_body[lane]], w.cdof[lane]);
  // reuse cfrc area of the scratch as the 13x6 buffer
  float(*fb)[6] = w.u.dyn.cdofdot;
  if (lane < NV) for (int k = 0; k < 6; k++) fb[lane][k] = buf[k];
  __syncwarp();
  for (int e = lane; e < NV * NV; e += 32) {
    int i = e / NV, j = e - i * NV;
    int hi = i > j ? i : j, lo = i > j ? j : i;
    float v = 0;
    if ((m.dof_ancmask[hi] >> lo) & 1u) v = dot6(w.cdof[lo], fb[hi]);
    if (i == j) v += m.dof_armature[i];
    w.M[e] = v;
  }
  __syncwarp();
}

// -------------------------------------------------------------------------------- collision
// MPR portal, per warp in shared memory: slots 0..3 = portal points p0..p3, slot 4 = the new support point.
// Each slot holds v (Minkowski difference point), v1 (on geom 1), v2 (on geom 2).  Every lane runs the same scalar
// control flow on broadcast reads; only the hull scans inside support_geom use the lanes as lanes.
#define SUPV(k) (w.sup[k])
#define SUPV1(k) (w.sup[k] + 3)
#define SUPV2(k) (w.sup[k] + 6)

// order-preserving image of a float for integer warp reductions (see support_geom)
__device__ __forceinline__ unsigned sortable_key(float x) {
  const unsigned k = __float_as_uint(x + 0.0f);
  return (k & 0x80000000u) ? ~k : (k | 0x80000000u);
}
// engine_collision_convex.c : mjccd_support for a hull — every lane scans a strided slice, arg-max by shuffles
static __device__ __noinline__ int support_geom(const DevModel& m, const WS& w, const float4* __restrict__ hv, int g, const float* dir, float* out, int lane) {
  const float* R = w.gmat[g];
  float l[3];
  mulmat3Tvec(l, R, dir);
  const float4* v = hv + m.geom_hvadr[g];
  const int n = m.geom_hvnum[g];
  float best = -3.0e38f;
  int bi = 0;
#pragma unroll 2
  for (int i = lane; i < n; i += 32) {
    float4 p = v[i];  // generic load: the lock-step kernel stages the hulls in shared memory
    float s = fmaf(p.z, l[2], fmaf(p.y, l[1], p.x * l[0]));  // explicit contraction: the same rounding in every copy of the scan
    if (s > best) { best = s; bi = i; }
  }
  // warp arg-max, ties to the lowest vertex id: two integer warp reductions (redux.sync) on an order-preserving image of
  // the float instead of five rounds of paired shuffles (the reduction, not the scan, dominates for hulls of <= 128 vertices)
  const unsigned key = sortable_key(best);  // (+ 0 inside: -0 and +0 compare equal, as in the float comparison)
  const unsigned kmax = __reduce_max_sync(FULL, key);
  bi = (int)__reduce_min_sync(FULL, key == kmax ? (unsigned)bi : 0xffffffffu);
  float4 p = v[bi];
  float pv[3] = {p.x, p.y, p.z}, t[3];
  mulmat3vec(t, R, pv);
  out[0] = w.gpos[g][0] + t[0]; out[1] = w.gpos[g][1] + t[1]; out[2] = w.gpos[g][2] + t[2];
  return bi;
}
// libccd support.c : __ccdSupport on obj1 - obj2, each inflated by margin/2; result into portal slot `slot`.
// Both hull scans run in ONE loop (two independent compare chains per lane, two pairs of warp reductions back to back), so
// a lone warp overlaps their latencies; vertex order, comparisons and tie rules are those of support_geom.
static __device__ __noinline__ void support_md(const DevModel& m, WS& w, const float4* hv, int g1, int g2, float margin, const float* dir, int slot, int lane) {
  float n[3] = {dir[0], dir[1], dir[2]}, nd[3];
  normalize3(n);
  nd[0] = -n[0]; nd[1] = -n[1]; nd[2] = -n[2];
  const float *R1 = w.gmat[g1], *R2 = w.gmat[g2];
  float l1[3], l2[3];
  mulmat3Tvec(l1, R1, n);
  mulmat3Tvec(l2, R2, nd);
  const float4 *va = hv + m.geom_hvadr[g1], *vb = hv + m.geom_hvadr[g2];
  const int na = m.geom_hvnum[g1], nb = m.geom_hvnum[g2], nmax = max(na, nb);
  float besta = -3.0e38f, bestb = -3.0e38f;
  int ia = 0, ib = 0;
#pragma unroll 2
  for (int i = lane; i < nmax; i += 32) {
    if (i < na) {
      const float4 p = va[i];
      const float s = fmaf(p.z, l1[2], fmaf(p.y, l1[1], p.x * l1[0]));
      if (s > besta) { besta = s; ia = i; }
    }
    if (i < nb) {
      const float4 p = vb[i];
      const float s = fmaf(p.z, l2[2], fmaf(p.y, l2[1], p.x * l2[0]));
      if (s > bestb) { bestb = s; ib = i; }
    }
  }
  const unsigned ka = sortable_key(besta), kb = sortable_key(bestb);
  const unsigned kamax = __reduce_max_sync(FULL, ka), kbmax = __reduce_max_sync(FULL, kb);
  ia = (int)__reduce_min_sync(FULL, ka == kamax ? (unsigned)ia : 0xffffffffu);
  ib = (int)__reduce_min_sync(FULL, kb == kbmax ? (unsigned)ib : 0xffffffffu);
  const float4 pa = va[ia], pb = vb[ib];
  float pva[3] = {pa.x, pa.y, pa.z}, pvb[3] = {pb.x, pb.y, pb.z}, ta[3], tb[3], v1[3], v2[3];
  mulmat3vec(ta, R1, pva);
  mulmat3vec(tb, R2, pvb);
  for (int k = 0; k < 3; k++) { v1[k] = w.gpos[g1][k] + ta[k]; v2[k] = w.gpos[g2][k] + tb[k]; }
  const float hm = 0.5f * margin;
  __syncwarp();
  if (lane < 3) {
    float a = v1[lane] + hm * n[lane], b = v2[lane] + hm * nd[lane];
    w.sup[slot][lane] = a - b; w.sup[slot][3 + lane] = a; w.sup[slot][6 + lane] = b;
  }
  __syncwarp();
}
__device__ __forceinline__ void sup_copy(WS& w, int dst, int src, int lane) {
  __syncwarp();
  float x = lane < 9 ? w.sup[src][lane] : 0.0f;
  if (lane < 9) w.sup[dst][lane] = x;
  __syncwarp();
}
__device__ __forceinline__ void portal_dir(const WS& w, float* dir) {
  float a[3], b[3];
  for (int k = 0; k < 3; k++) { a[k] = SUPV(2)[k] - SUPV(1)[k]; b[k] = SUPV(3)[k] - SUPV(1)[k]; }
  cross3(dir, a, b);
  normalize3(dir);
}
__device__ __forceinline__ bool portal_reach_tol(const WS& w, const float* dir, float tol) {
  float dv4 = dot3(SUPV(4), dir);
  float d1 = dv4 - dot3(SUPV(1), dir), d2 = dv4 - dot3(SUPV(2), dir), d3 = dv4 - dot3(SUPV(3), dir);
  return fminf(d1, fminf(d2, d3)) <= tol;
}
// libccd mpr.c : expandPortal — the new point (slot 4) replaces one of p1..p3
__device__ __forceinline__ void expand_portal(WS& w, int lane) {
  float c[3];
  cross3(c, SUPV(4), SUPV(0));
  int dst;
  if (dot3(SUPV(1), c) > 0) dst = dot3(SUPV(2), c) > 0 ? 1 : 3;
  else dst = dot3(SUPV(3), c) > 0 ? 2 : 1;
  sup_copy(w, dst, 4, lane);
}
// closest point of triangle (a,b,c) to the origin (Ericson, Real-Time Collision Detection 5.1.5)
__device__ __forceinline__ float origin_tri_closest(const float* a, const float* b, const float* c, float* w) {
  float ab[3], ac[3];
  for (int k = 0; k < 3; k++) { ab[k] = b[k] - a[k]; ac[k] = c[k] - a[k]; }
  float d1 = -dot3(ab, a), d2 = -dot3(ac, a);
  if (d1 <= 0 && d2 <= 0) { for (int k = 0; k < 3; k++) w[k] = a[k]; return sqrtf(dot3(w, w)); }
  float d3 = -dot3(ab, b), d4 = -dot3(ac, b);
  if (d3 >= 0 && d4 <= d3) { for (int k = 0; k < 3; k++) w[k] = b[k]; return sqrtf(dot3(w, w)); }
  float vc = d1 * d4 - d3 * d2;
  if (vc <= 0 && d1 >= 0 && d3 <= 0) { float v = d1 / (d1 - d3); for (int k = 0; k < 3; k++) w[k] = a[k] + v * ab[k]; return sqrtf(dot3(w, w)); }
  float d5 = -dot3(ab, c), d6 = -dot3(ac, c);
  if (d6 >= 0 && d5 <= d6) { for (int k = 0; k < 3; k++) w[k] = c[k]; return sqrtf(dot3(w, w)); }
  float vb = d5 * d2 - d1 * d6;
  if (vb <= 0 && d2 >= 0 && d6 <= 0) { float v = d2 / (d2 - d6); for (int k = 0; k < 3; k++) w[k] = a[k] + v * ac[k]; return sqrtf(dot3(w, w)); }
  float va = d3 * d6 - d5 * d4;
  if (va <= 0 && (d4 - d3) >= 0 && (d5 - d6) >= 0) {
    float v = (d4 - d3) / ((d4 - d3) + (d5 - d6));
    for (int k = 0; k < 3; k++) w[k] = b[k] + v * (c[k] - b[k]);
    return sqrtf(dot3(w, w));
  }
  float den = 1.0f / (va + vb + vc), v = vb * den, u = vc * den;
  for (int k = 0; k < 3; k++) w[k] = a[k] + v * ab[k] + u * ac[k];
  return sqrtf(dot3(w, w));
}
// libccd mpr.c : findPos — contact position from the portal's barycentric coordinates of the origin
__device__ __forceinline__ void find_pos(const WS& w, float* pos) {
  float dir[3], b[4], t[3], sum;
  portal_dir(w, dir);
  cross3(t, SUPV(1), SUPV(2)); b[0] = dot3(t, SUPV(3));
  cross3(t, SUPV(3), SUPV(2)); b[1] = dot3(t, SUPV(0));
  cross3(t, SUPV(0), SUPV(1)); b[2] = dot3(t, SUPV(3));
  cross3(t, SUPV(2), SUPV(1)); b[3] = dot3(t, SUPV(0));
  sum = b[0] + b[1] + b[2] + b[3];
  if (sum <= 0) {
    b[0] = 0;
    cross3(t, SUPV(2), SUPV(3)); b[1] = dot3(t, dir);
    cross3(t, SUPV(3), SUPV(1)); b[2] = dot3(t, dir);
    cross3(t, SUPV(1), SUPV(2)); b[3] = dot3(t, dir);
    sum = b[1] + b[2] + b[3];
  }
  float inv = 0.5f / sum;
  for (int k = 0; k < 3; k++)
    pos[k] = inv * (b[0] * (SUPV1(0)[k] + SUPV2(0)[k]) + b[1] * (SUPV1(1)[k] + SUPV2(1)[k]) + b[2] * (SUPV1(2)[k] + SUPV2(2)[k]) + b[3] * (SUPV1(3)[k] + SUPV2(3)[k]));
}
// libccd mpr.c : ccdMPRPenetration (discoverPortal, refinePortal, findPenetr). All lanes carry the same portal.
static __device__ __noinline__ bool mpr_penetration(const DevModel& m, WS& w, const float4* hv, int g1, int g2, float margin,
                                             float* depth, float* dir_out, float* pos, int lane) {
  float dir[3], va[3], vb[3];
  __syncwarp();
  if (lane < 3) {
    float a = w.gpos[g1][lane], b = w.gpos[g2][lane];
    w.sup[0][lane] = a - b; w.sup[0][3 + lane] = a; w.sup[0][6 + lane] = b;
  }
  __syncwarp();
  if (dot3(SUPV(0), SUPV(0)) < 1e-12f) { __syncwarp(); if (lane == 0) w.sup[0][0] += 1e-5f; __syncwarp(); }
  for (int k = 0; k < 3; k++) dir[k] = -SUPV(0)[k];
  normalize3(dir);
  dir_out[0] = dir_out[1] = dir_out[2] = 0;  // on a `false` return: a direction that separates the two shapes, or zero
  support_md(m, w, hv, g1, g2, margin, dir, 1, lane);
  if (dot3(SUPV(1), dir) < 0) { for (int k = 0; k < 3; k++) dir_out[k] = dir[k]; return false; }
  cross3(dir, SUPV(0), SUPV(1));
  if (dot3(dir, dir) < 1e-14f) {
    // origin lies on the segment v0-v1 (findPenetrSegment) or coincides with v1 (findPenetrTouch)
    for (int k = 0; k < 3; k++) { pos[k] = 0.5f * (SUPV1(1)[k] + SUPV2(1)[k]); dir_out[k] = SUPV(1)[k]; }
    *depth = normalize3(dir_out);
    if (*depth < 1e-7f) return false;
    return true;
  }
  normalize3(dir);
  support_md(m, w, hv, g1, g2, margin, dir, 2, lane);
  if (dot3(SUPV(2), dir) < 0) { for (int k = 0; k < 3; k++) dir_out[k] = dir[k]; return false; }
  for (int k = 0; k < 3; k++) { va[k] = SUPV(1)[k] - SUPV(0)[k]; vb[k] = SUPV(2)[k] - SUPV(0)[k]; }
  cross3(dir, va, vb);
  normalize3(dir);
  if (dot3(dir, SUPV(0)) > 0) {  // swap p1 <-> p2 (through slot 4)
    sup_copy(w, 4, 1, lane); sup_copy(w, 1, 2, lane); sup_copy(w, 2, 4, lane);
    dir[0] = -dir[0]; dir[1] = -dir[1]; dir[2] = -dir[2];
  }
#pragma unroll 1
  for (int it = 0; it < 100; it++) {
    support_md(m, w, hv, g1, g2, margin, dir, 3, lane);
    if (dot3(SUPV(3), dir) < 0) { for (int k = 0; k < 3; k++) dir_out[k] = dir[k]; return false; }
    bool cont = false;
    cross3(va, SUPV(1), SUPV(3));
    if (dot3(va, SUPV(0)) < -1e-10f) { sup_copy(w, 2, 3, lane); cont = true; }
    if (!cont) {
      cross3(va, SUPV(3), SUPV(2));
      if (dot3(va, SUPV(0)) < -1e-10f) { sup_copy(w, 1, 3, lane); cont = true; }
    }
    if (!cont) break;
    for (int k = 0; k < 3; k++) { va[k] = SUPV(1)[k] - SUPV(0)[k]; vb[k] = SUPV(2)[k] - SUPV(0)[k]; }
    cross3(dir, va, vb);
    normalize3(dir);
  }
  const float tol = 1e-6f;
#pragma unroll 1
  for (int it = 0; it < 100; it++) {  // refinePortal
    portal_dir(w, dir);
    if (dot3(dir, SUPV(1)) >= 0) break;
    support_md(m, w, hv, g1, g2, margin, dir, 4, lane);
    if (dot3(SUPV(4), dir) < 0) { for (int k = 0; k < 3; k++) dir_out[k] = dir[k]; return false; }
    if (portal_reach_tol(w, dir, tol)) return false;
    expand_portal(w, lane);
  }
#pragma unroll 1
  for (int it = 0;; it++) {  // findPenetr
    portal_dir(w, dir);
    support_md(m, w, hv, g1, g2, margin, dir, 4, lane);
    if (portal_reach_tol(w, dir, tol) || it > 50) {
      float wv[3];
      *depth = origin_tri_closest(SUPV(1), SUPV(2), SUPV(3), wv);
      if (*depth < 1e-9f) { for (int k = 0; k < 3; k++) dir_out[k] = dir[k]; }
      else { for (int k = 0; k < 3; k++) dir_out[k] = wv[k]; normalize3(dir_out); }
      find_pos(w, pos);
      return true;
    }
    expand_portal(w, lane);
  }
}

// mju_makeFrame + contact bookkeeping (lane 0 writes)
static __device__ __noinline__ void add_contact(const DevModel& m, WS& w, int pair, float dist, const float* pos, const float* normal, int lane) {
  int c = w.ncon;
  if (c >= MAXCON) { if (lane == 0) w.overflow = 1; return; }
  if (lane == 0) {
    float f[9];
    f[0] = normal[0]; f[1] = normal[1]; f[2] = normal[2];
    normalize3(f);
    f[3] = 0; f[4] = 0; f[5] = 0;
    if (f[1] < 0.5f && f[1] > -0.5f) f[4] = 1; else f[5] = 1;
    float t = dot3(f, f + 3);
    f[3] -= t * f[0]; f[4] -= t * f[1]; f[5] -= t * f[2];
    normalize3(f + 3);
    cross3(f + 6, f, f + 3);
    for (int k = 0; k < 9; k++) w.c_frame[c][k] = f[k];
    for (int k = 0; k < 3; k++) w.c_pos[c][k] = pos[k];
    w.c_dist[c] = dist;
    w.c_pair[c] = pair;
    w.c_g1[c] = m.pair_g1[pair];
    w.c_g2[c] = m.pair_g2[pair];
    w.c_fric[c][0] = m.pair_fric[pair][0]; w.c_fric[c][1] = m.pair_fric[pair][0]; w.c_fric[c][2] = m.pair_fric[pair][1];
    w.ncon = c + 1;
  }
  __syncwarp();
}

// engine_collision_driver.c : mj_collision over the candidate pair list (+ the bounding-sphere test of mj_collideGeoms)
static __device__ __noinline__ void collision(const DevModel& m, WS& w, const float4* hv, const int* __restrict__ adj, int lane) {
  if (lane == 0) { w.ncon = 0; w.overflow = 0; }
  // broadphase for every candidate pair at once (lane = pair): plane / bounding-sphere rejection of mj_collideGeoms
  bool cand = false;
  if (lane < m.npair) {
    const int g1 = m.pair_g1[lane], g2 = m.pair_g2[lane];
    const float margin = m.pair_margin[lane];
    float dif[3];
    for (int k = 0; k < 3; k++) dif[k] = w.gpos[g2][k] - w.gpos[g1][k];
    if (m.geom_type[g1] == GEOM_PLANE) {
      const float* R1 = w.gmat[g1];
      cand = !(dif[0] * R1[2] + dif[1] * R1[5] + dif[2] * R1[8] > margin + m.geom_rbound[g2]);
    } else {
      const float bound = m.geom_rbound[g1] + m.geom_rbound[g2] + margin;
      cand = !(dot3(dif, dif) > bound * bound);
      // Separation budget.  sep[p] separated the pair by gapb[p] when it was last evaluated; since then no point of either geom
      // moved further than the disp[] bounds accumulated here, so while the budget stays positive sep[p] still separates
      // them: the support evaluation below would say so and skip the pair — skip it without evaluating.  (NaN budgets,
      // e.g. from the garbage pose of a freshly loaded workspace, compare false and fall through to the evaluation.)
      if (m.gap_skip) {
        const float left = w.gapb[lane] - (1.001f * (w.disp[g1] + w.disp[g2]) + 2e-7f);
        w.gapb[lane] = left;
        const bool has_axis = w.sep[lane][0] != 0.0f || w.sep[lane][1] != 0.0f || w.sep[lane][2] != 0.0f;
        if (cand && has_axis && left > 0.0f) cand = false;
      }
    }
  }
  unsigned todo = __ballot_sync(FULL, cand);
  __syncwarp();
  while (todo) {
    const int p = __ffs(todo) - 1;
    todo &= todo - 1;
    int g1 = m.pair_g1[p], g2 = m.pair_g2[p];
    float margin = m.pair_margin[p];
    if (m.geom_type[g1] == GEOM_PLANE) {
      const float* R1 = w.gmat[g1];
      float n[3] = {R1[2], R1[5], R1[8]}, dif[3];
      if (m.geom_type[g2] == GEOM_BOX) {
        // mjc_PlaneBox (engine_collision_primitive.c): corners in index order, lane = corner; the first 4 that lie within
        // the margin and do not point away from the plane become contacts (gripper_two_fingers.xml:133)
        for (int k = 0; k < 3; k++) dif[k] = w.gpos[g2][k] - w.gpos[g1][k];
        const float dist = dot3(dif, n);
        const int i = lane & 7;
        float vec[3] = {(i & 1) ? m.geom_size[g2][0] : -m.geom_size[g2][0], (i & 2) ? m.geom_size[g2][1] : -m.geom_size[g2][1],
                        (i & 4) ? m.geom_size[g2][2] : -m.geom_size[g2][2]}, corner[3];
        mulmat3vec(corner, w.gmat[g2], vec);
        const float ldist = dot3(n, corner);
        unsigned ok = __ballot_sync(FULL, lane < 8 && !(dist + ldist > margin || ldist > 0));
        for (int cnt = 0; ok && cnt < 4; cnt++) {
          const int src = __ffs(ok) - 1;
          ok &= ok - 1;
          float cd = __shfl_sync(FULL, dist + ldist, src), pos[3];
          for (int k = 0; k < 3; k++) pos[k] = __shfl_sync(FULL, corner[k], src) - 0.5f * cd * n[k] + w.gpos[g2][k];
          add_contact(m, w, p, cd, pos, n, lane);
        }
        continue;
      }
      // mjc_PlaneConvex: support vertex, then its hull-graph neighbours that are also within the margin (<= 3 contacts)
      float nn[3] = {-n[0], -n[1], -n[2]}, v[3], pos[3];
      int vi = support_geom(m, w, hv, g2, nn, v, lane);
      for (int k = 0; k < 3; k++) dif[k] = v[k] - w.gpos[g1][k];
      float dist = dot3(dif, n);
      if (dist > margin) continue;
      for (int k = 0; k < 3; k++) pos[k] = v[k] - 0.5f * dist * n[k];
      add_contact(m, w, p, dist, pos, n, lane);
      const int* ga = adj + m.geom_adjadr[g2];  // [nvert+1 offsets][neighbours]
      int nvert = m.geom_hvnum[g2];
      int e0 = __ldg(ga + vi), e1 = __ldg(ga + vi + 1), cnt = 1;
      const float4* hvg = hv + m.geom_hvadr[g2];
      for (int e = e0; e < e1 && cnt < 3; e++) {
        int nb = __ldg(ga + nvert + 1 + e);
        float4 q = hvg[nb];
        float qv[3] = {q.x, q.y, q.z}, t[3];
        mulmat3vec(t, w.gmat[g2], qv);
        for (int k = 0; k < 3; k++) { v[k] = w.gpos[g2][k] + t[k]; dif[k] = v[k] - w.gpos[g1][k]; }
        dist = dot3(dif, n);
        if (dist > margin) continue;
        for (int k = 0; k < 3; k++) pos[k] = v[k] - 0.5f * dist * n[k];
        add_contact(m, w, p, dist, pos, n, lane);
        cnt++;
      }
    } else {
      float depth, dir[3], pos[3];
      // temporal coherence: a direction that separated the pair in the previous substep usually still does (one support
      // evaluation instead of a full MPR run).  It proves the origin lies outside the Minkowski difference, which is
      // exactly when MPR reports no penetration, so the contact set is unchanged.
      float ca[3] = {w.sep[p][0], w.sep[p][1], w.sep[p][2]};
      if (ca[0] != 0.0f || ca[1] != 0.0f || ca[2] != 0.0f) {
        support_md(m, w, hv, g1, g2, margin, ca, 4, lane);
        const float sd = dot3(SUPV(4), ca);
        if (sd < 0) {
          // ca is a unit vector (mpr_penetration normalises what it returns): -sd is the separation along it, in metres
          __syncwarp();
          if (lane == 0) w.gapb[p] = -sd - 2e-6f;
          __syncwarp();
          continue;
        }
      }
      bool hit = mpr_penetration(m, w, hv, g1, g2, margin, &depth, dir, pos, lane);
      __syncwarp();
      if (lane < 3) w.sep[p][lane] = hit ? 0.0f : dir[lane];
      if (lane == 3) w.gapb[p] = 0.0f;  // a new axis (or none): its separation is measured by the next substep's support evaluation
      __syncwarp();
      if (!hit) continue;
      add_contact(m, w, p, margin - depth, pos, dir, lane);
    }
  }
  __syncwarp();
}

__device__ __forceinline__ void forward_position(const DevModel& m, WS& w, const float4* hv, const int* adj, int lane) {
  kinematics(m, w, lane);
  com_pos_crb(m, w, lane);
  collision(m, w, hv, adj, lane);
}

// -------------------------------------------------------------------------------- smooth dynamics
// mj_comVel + mj_rne(flg_acc=0) + passive + actuation + xfrc -> fsmooth, asmooth.  Needs the dyn scratch from com_pos_crb.
static __device__ __noinline__ void smooth_forces(const DevModel& m, WS& w, int lane, bool actuation, float xfrc_z) {
  const int nb = m.nbody;
  // forward pass by levels: cvel, cdof_dot, and cacc (kept in registers, written into cfrc as body force)
  if (lane == 0) for (int k = 0; k < 6; k++) { w.u.dyn.cvel[0][k] = 0; w.u.dyn.cfrc[0][k] = 0; }
  // cacc of each body is needed by its children: stage it in crb[b][0..5] (crb is dead after M was built)
  if (lane == 0) { float* a = w.u.dyn.crb[0]; a[0] = a[1] = a[2] = 0; a[3] = -m.gravity[0]; a[4] = -m.gravity[1]; a[5] = -m.gravity[2]; }
  __syncwarp();
  for (int lv = 1; lv < m.nlevel; lv++) {
    int idx = m.level_start[lv] + lane;
    if (idx < m.level_start[lv + 1]) {
      int b = m.level_body[idx], pid = m.body_parent[b];
      float cvel[6], cacc[6];
      for (int k = 0; k < 6; k++) { cvel[k] = w.u.dyn.cvel[pid][k]; cacc[k] = w.u.dyn.crb[pid][k]; }
      for (int kj = 0; kj < m.body_jntnum[b]; kj++) {
        int j = m.body_jntadr[b] + kj, a = m.jnt_dofadr[j];
        if (m.jnt_type[j] == JNT_FREE) {
          for (int i = 0; i < 3; i++) {
            for (int k = 0; k < 6; k++) w.u.dyn.cdofdot[a + i][k] = 0;
            float qv = w.qvel[a + i];
            for (int k = 0; k < 6; k++) cvel[k] += w.cdof[a + i][k] * qv;
          }
          float dd[3][6];
          for (int i = 0; i < 3; i++) cross_motion(dd[i], cvel, w.cdof[a + 3 + i]);
          for (int i = 0; i < 3; i++) {
            float qv = w.qvel[a + 3 + i];
            for (int k = 0; k < 6; k++) { w.u.dyn.cdofdot[a + 3 + i][k] = dd[i][k]; cvel[k] += w.cdof[a + 3 + i][k] * qv; cacc[k] += dd[i][k] * qv; }
          }
        } else {
          float dd[6], qv = w.qvel[a];
          cross_motion(dd, cvel, w.cdof[a]);
          for (int k = 0; k < 6; k++) { w.u.dyn.cdofdot[a][k] = dd[k]; cvel[k] += w.cdof[a][k] * qv; cacc[k] += dd[k] * qv; }
        }
      }
      float t1[6], t2[6], f[6];
      mul_inert_vec(t1, w.u.dyn.cinert[b], cacc);
      mul_inert_vec(t2, w.u.dyn.cinert[b], cvel);
      cross_force(f, cvel, t2);
      for (int k = 0; k < 6; k++) { w.u.dyn.cvel[b][k] = cvel[k]; w.u.dyn.crb[b][k] = cacc[k]; w.u.dyn.cfrc[b][k] = f[k] + t1[k]; }
    }
    __syncwarp();
  }
  // qfrc_bias_i = cdof_i . sum_{b' in subtree(body_i)} cfrc[b']
  float bias = 0;
  if (lane < NV) {
    int b = m.dof_body[lane];
    unsigned mask = m.body_subtree_mask[b];
    float acc[6] = {0, 0, 0, 0, 0, 0};
    for (int bb = b; bb < nb; bb++)
      if ((mask >> bb) & 1u)
        for (int k = 0; k < 6; k++) acc[k] += w.u.dyn.cfrc[bb][k];
    bias = dot6(w.cdof[lane], acc);
  }
  float f = 0;
  if (lane < NV) {
    f = -m.dof_damping[lane] * w.qvel[lane] - bias;
    if (actuation)
      for (int u = 0; u < NU; u++)
        if (m.act_dof[u] == lane) f += m.act_gear[u] * fminf(fmaxf(w.ctrl[u], m.act_lo[u]), m.act_hi[u]);
    // mj_xfrcAccumulate for the constant +z force on `ee` applied at xipos(ee) (robot_env.py:64-65)
    if (xfrc_z != 0.0f && ((m.body_dofmask[m.body_ee] >> lane) & 1u)) {
      float off[3], t[3];
      for (int k = 0; k < 3; k++) off[k] = w.u.dyn.xipos[m.body_ee][k] - w.com[m.body_ee][k];
      cross3(t, w.cdof[lane], off);
      f += (w.cdof[lane][5] + t[2]) * xfrc_z;
    }
    w.bias[lane] = bias;
    w.fsmooth[lane] = f;
  }
  __syncwarp();
  // factor M into the scratch and solve for qacc_smooth
  for (int e = lane; e < NV * NV; e += 32) w.u.dyn.L[e] = w.M[e];
  __syncwarp();
  float a = chol_factor_solve<true>(w.u.dyn.L, w.cho, f, lane);  // M never couples the gripper tree and the free object
  if (lane < NV) w.asmooth[lane] = a;
  __syncwarp();
}

// -------------------------------------------------------------------------------- constraints
static __device__ __noinline__ float get_impedance(const float* solimp, float pos, float margin) {
  if (solimp[0] == solimp[1] || solimp[2] <= MINVAL) return 0.5f * (solimp[0] + solimp[1]);
  float x = fabsf((pos - margin) / solimp[2]);
  if (x >= 1) return solimp[1];
  if (x <= 0) return solimp[0];
  float y, p = solimp[4], mid = solimp[3];
  if (p == 1.0f) y = x;
  else if (p == 2.0f) y = x <= mid ? x * x / mid : 1 - (1 - x) * (1 - x) / (1 - mid);
  else y = x <= mid ? powf(x, p) / powf(mid, p - 1) : 1 - powf(1 - x, p) / powf(1 - mid, p - 1);
  return solimp[0] + y * (solimp[1] - solimp[0]);
}

// engine_core_constraint.c : mj_makeConstraint (limits + elliptic contacts), mj_makeImpedance, mj_referenceConstraint
static __device__ __noinline__ void make_constraint(const DevModel& m, WS& w, int lane) {
  // ---- joint limits: lane = joint
  bool active = false;
  float dist = 0, sign = 0;
  if (lane < m.njnt && m.jnt_limited[lane] && m.jnt_type[lane] != JNT_FREE) {
    float value = w.qpos[m.jnt_qposadr[lane]];
    float dl = value - m.jnt_range[lane][0], du = m.jnt_range[lane][1] - value;
    if (dl < 0) { active = true; dist = dl; sign = 1; }
    else if (du < 0) { active = true; dist = du; sign = -1; }
  }
  unsigned bal = __ballot_sync(FULL, active);
  int nlim = __popc(bal);
  int ncon = w.ncon;
  int nefc = nlim + 4 * ncon;
  for (int e = lane; e < nefc * NV; e += 32) (&w.u.con.J[0][0])[e] = 0;
  __syncwarp();
  const float h2 = 2 * m.timestep;
  if (active) {
    int r = __popc(bal & ((1u << lane) - 1));
    int dof = m.jnt_dofadr[lane];
    w.u.con.J[r][dof] = sign;
    float tc = fmaxf(m.jnt_solref[0], h2), dr = m.jnt_solref[1], dmax = m.jnt_solimp[1];
    float imp = get_impedance(m.jnt_solimp, dist, 0.0f);
    float R = fmaxf((1 - imp) * m.dof_invweight0[dof] / imp, MINVAL);
    float K = 1.0f / (dmax * dmax * tc * tc * dr * dr), B = 2.0f / (dmax * tc);
    w.e_D[r] = 1.0f / R;
    w.e_aref[r] = -B * sign * w.qvel[dof] - K * imp * dist;
  }
  // ---- contacts: Jacobian rows, lane = dof
  if (lane < NV) {
    const int i = lane;
    for (int c = 0; c < ncon; c++) {
      int b1 = m.geom_body[w.c_g1[c]], b2 = m.geom_body[w.c_g2[c]];
      float jp[3] = {0, 0, 0}, jr[3] = {0, 0, 0};
      if ((m.body_dofmask[b2] >> i) & 1u) {
        float off[3], t[3];
        for (int k = 0; k < 3; k++) off[k] = w.c_pos[c][k] - w.com[b2][k];
        cross3(t, w.cdof[i], off);
        for (int k = 0; k < 3; k++) { jp[k] += w.cdof[i][3 + k] + t[k]; jr[k] += w.cdof[i][k]; }
      }
      if ((m.body_dofmask[b1] >> i) & 1u) {
        float off[3], t[3];
        for (int k = 0; k < 3; k++) off[k] = w.c_pos[c][k] - w.com[b1][k];
        cross3(t, w.cdof[i], off);
        for (int k = 0; k < 3; k++) { jp[k] -= w.cdof[i][3 + k] + t[k]; jr[k] -= w.cdof[i][k]; }
      }
      const float* f = w.c_frame[c];
      int r = nlim + 4 * c;
      w.u.con.J[r][i] = dot3(f, jp);
      w.u.con.J[r + 1][i] = dot3(f + 3, jp);
      w.u.con.J[r + 2][i] = dot3(f + 6, jp);
      w.u.con.J[r + 3][i] = dot3(f, jr);
    }
  }
  __syncwarp();
  // ---- contact impedance / reference: lane = contact
  if (lane < ncon) {
    int c = lane, p = w.c_pair[c], r = nlim + 4 * c;
    int b1 = m.geom_body[w.c_g1[c]], b2 = m.geom_body[w.c_g2[c]];
    float tran = m.body_invweight0[b1][0] + m.body_invweight0[b2][0];
    float tc = fmaxf(m.pair_solref[p][0], h2), dr = m.pair_solref[p][1], dmax = m.pair_solimp[p][1];
    float margin = m.pair_margin[p];
    float imp = get_impedance(m.pair_solimp[p], w.c_dist[c], margin);
    float R0 = fmaxf((1 - imp) * tran / imp, MINVAL);
    float R1 = R0 / fmaxf(MINVAL, m.impratio);
    float f0 = w.c_fric[c][0];
    float R2 = R1 * f0 * f0 / (w.c_fric[c][1] * w.c_fric[c][1]);
    float R3 = R1 * f0 * f0 / (w.c_fric[c][2] * w.c_fric[c][2]);
    w.c_mu[c] = f0 * sqrtf(R1 / R0);
    float K = 1.0f / (dmax * dmax * tc * tc * dr * dr), B = 2.0f / (dmax * tc);
    float vel[4];
    for (int j = 0; j < 4; j++) {
      float v = 0;
      for (int k = 0; k < NV; k++) v += w.u.con.J[r + j][k] * w.qvel[k];
      vel[j] = v;
    }
    w.e_D[r] = 1.0f / R0; w.e_D[r + 1] = 1.0f / R1; w.e_D[r + 2] = 1.0f / R2; w.e_D[r + 3] = 1.0f / R3;
    w.e_aref[r] = -B * vel[0] - K * imp * (w.c_dist[c] - margin);
    w.e_aref[r + 1] = -B * vel[1];
    w.e_aref[r + 2] = -B * vel[2];
    w.e_aref[r + 3] = -B * vel[3];
  }
  // does any contact couple the two kinematic trees (gripper <-> object)?  If not, the Hessian stays block diagonal.
  bool cpl = false;
  if (lane < ncon) {
    int r1 = m.body_root[m.geom_body[w.c_g1[lane]]], r2 = m.body_root[m.geom_body[w.c_g2[lane]]];
    cpl = r1 != 0 && r2 != 0 && r1 != r2;
  }
  cpl = __any_sync(FULL, cpl);
  if (lane == 0) { w.nefc = nefc; w.nlim = nlim; w.coupled = cpl; }
  __syncwarp();
}

// -------------------------------------------------------------------------------- Newton solver
// The small helpers of the solver loop (constraint update, line-search evaluation, the 13-wide products, the Hessian) are inlined
// into solve_newton: as separate functions their call overhead and the register shuffling around every call were 4 % of the step
// (profiles/r2zf_inline.log); the stage functions themselves stay out of line (inlining them into the kernel body costs 6 %).
// engine_solver.c : mj_constraintUpdate — lane = item (limit row or contact). Returns the constraint cost (warp-uniform).
__device__ __forceinline__ float constraint_update(WS& w, int lane, bool want_cone_hessian) {
  const int nlim = w.nlim, nitem = nlim + w.ncon;
  float cost = 0;
  int state = 0;
  if (lane < nlim) {
    float x = w.e_jar[lane];
    if (x < 0) { w.e_force[lane] = -w.e_D[lane] * x; cost = 0.5f * w.e_D[lane] * x * x; state = 1; w.e_act[lane] = w.e_D[lane]; }
    else { w.e_force[lane] = 0; w.e_act[lane] = 0; }
  } else if (lane < nitem) {
    int c = lane - nlim, r = nlim + 4 * c;
    float mu = w.c_mu[c], sc[4] = {mu, w.c_fric[c][0], w.c_fric[c][1], w.c_fric[c][2]};
    float U[4], T = 0;
    for (int j = 0; j < 4; j++) U[j] = w.e_jar[r + j] * sc[j];
    float N = U[0];
    T = sqrtf(U[1] * U[1] + U[2] * U[2] + U[3] * U[3]);
    if (N >= mu * T || (T <= 0 && N >= 0)) {
      for (int j = 0; j < 4; j++) { w.e_force[r + j] = 0; w.e_act[r + j] = 0; }
    } else if (mu * N + T <= 0 || (T <= 0 && N < 0)) {
      for (int j = 0; j < 4; j++) {
        float x = w.e_jar[r + j], D = w.e_D[r + j];
        w.e_force[r + j] = -D * x;
        cost += 0.5f * D * x * x;
        w.e_act[r + j] = D;
      }
      state = 1;
    } else {
      float Dm = w.e_D[r] / (mu * mu * (1 + mu * mu)), NmT = N - mu * T;
      cost = 0.5f * Dm * NmT * NmT;
      float f0 = -Dm * NmT * mu;
      w.e_force[r] = f0;
      for (int j = 1; j < 4; j++) w.e_force[r + j] = -f0 / T * U[j] * sc[j];
      for (int j = 0; j < 4; j++) w.e_act[r + j] = 0;
      state = 2;
      if (want_cone_hessian) {  // engine_solver.c : HessianCone
        float* hc = w.hc[c];
        float invT = 1.0f / T;
        hc[0] = 1;
        for (int j = 1; j < 4; j++) { hc[j] = -mu * invT * U[j]; hc[4 * j] = hc[j]; }
        float scl = mu * N * invT * invT * invT;
        for (int j = 1; j < 4; j++)
          for (int k = 1; k < 4; k++) hc[4 * j + k] = scl * U[j] * U[k];
        float dg = mu * mu - mu * N * invT;
        for (int j = 1; j < 4; j++) hc[4 * j + j] += dg;
        for (int j = 0; j < 4; j++)
          for (int k = 0; k < 4; k++) hc[4 * j + k] *= Dm * sc[j] * sc[k];
      }
    }
  }
  w.istate[lane] = state;
  cost = warp_sum(cost);
  __syncwarp();
  return cost;
}

// derivative and curvature of the cost along qacc + alpha*search (engine_solver.c : PrimalEval)
__device__ __forceinline__ void line_eval(const WS& w, int lane, float alpha, float q1, float q2, float& d1, float& d2) {
  const int nlim = w.nlim, nitem = nlim + w.ncon;
  float D1 = 0, D2 = 0;
  if (lane < nlim) {
    float x = w.e_jar[lane] + alpha * w.e_Jv[lane];
    if (x < 0) { float D = w.e_D[lane], jv = w.e_Jv[lane]; D1 = D * x * jv; D2 = D * jv * jv; }
  } else if (lane < nitem) {
    int c = lane - nlim, r = nlim + 4 * c;
    float mu = w.c_mu[c], sc[4] = {mu, w.c_fric[c][0], w.c_fric[c][1], w.c_fric[c][2]};
    float x[4], jv[4], U[4], V[4];
    for (int j = 0; j < 4; j++) { jv[j] = w.e_Jv[r + j]; x[j] = w.e_jar[r + j] + alpha * jv[j]; U[j] = x[j] * sc[j]; V[j] = jv[j] * sc[j]; }
    float TT = U[1] * U[1] + U[2] * U[2] + U[3] * U[3], T = sqrtf(TT), N = U[0];
    if (N >= mu * T || (T <= 0 && N >= 0)) {
    } else if (mu * N + T <= 0 || (T <= 0 && N < 0)) {
      for (int j = 0; j < 4; j++) { float D = w.e_D[r + j]; D1 += D * x[j] * jv[j]; D2 += D * jv[j] * jv[j]; }
    } else {
      float Dm = w.e_D[r] / (mu * mu * (1 + mu * mu)), NmT = N - mu * T;
      float UV = U[1] * V[1] + U[2] * V[2] + U[3] * V[3], VV = V[1] * V[1] + V[2] * V[2] + V[3] * V[3];
      float T1 = UV / T, T2 = (VV - T1 * T1) / T, a = V[0] - mu * T1;
      D1 = Dm * NmT * a;
      D2 = Dm * (a * a - NmT * mu * T2);
    }
  }
  D1 = warp_sum(D1);
  D2 = warp_sum(D2);
  d1 = q1 + alpha * q2 + D1;
  d2 = q2 + D2;
}

// y_i = sum_k M[i][k] x[k] for lane i < NV (x in shared memory)
__device__ __forceinline__ float mat13_vec(const float* M, const float* x, int lane) {
  float v = 0;
  if (lane < NV) {
    const float* row = M + lane * NV;
#pragma unroll
    for (int k = 0; k < NV; k++) v += row[k] * x[k];
  }
  return v;
}
// out[r] = J[r] . x - sub[r]  for every constraint row (sub may be NULL)
__device__ __forceinline__ void rows_dot(const WS& w, const float* x, const float* sub, float* out, int lane) {
#pragma unroll 1
  for (int r = lane; r < w.nefc; r += 32) {
    const float* row = w.u.con.J[r];
    float v = 0;
#pragma unroll
    for (int k = 0; k < NV; k++) v += row[k] * x[k];
    out[r] = sub ? v - sub[r] : v;
  }
}
// f_i = sum_r J[r][i] force[r]  (lane i < NV)
__device__ __forceinline__ float jt_force(const WS& w, int lane) {
  float fc = 0;
  if (lane < NV) {
#pragma unroll 4
    for (int r = 0; r < w.nefc; r++) fc += w.u.con.J[r][lane] * w.e_force[r];
  }
  return fc;
}
// Lower-triangle entry lists of the 13x13 Hessian: all 91 entries (a contact couples gripper and object), or only the 49
// entries of the two diagonal blocks (7 gripper dofs, 6 object dofs) when it does not.  Packed as (row << 4) | column.
__constant__ unsigned char HESS_TRI[91] = {
    0x00, 0x10, 0x11, 0x20, 0x21, 0x22, 0x30, 0x31, 0x32, 0x33, 0x40, 0x41, 0x42, 0x43, 0x44, 0x50, 0x51, 0x52, 0x53, 0x54, 0x55, 0x60, 0x61, 0x62, 0x63, 0x64,
    0x65, 0x66, 0x77, 0x87, 0x88, 0x97, 0x98, 0x99, 0xa7, 0xa8, 0xa9, 0xaa, 0xb7, 0xb8, 0xb9, 0xba, 0xbb, 0xc7, 0xc8, 0xc9, 0xca, 0xcb, 0xcc,
    // the 42 coupling entries (object rows x gripper columns)
    0x70, 0x71, 0x72, 0x73, 0x74, 0x75, 0x76, 0x80, 0x81, 0x82, 0x83, 0x84, 0x85, 0x86, 0x90, 0x91, 0x92, 0x93, 0x94, 0x95, 0x96, 0xa0, 0xa1, 0xa2, 0xa3, 0xa4,
    0xa5, 0xa6, 0xb0, 0xb1, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xc0, 0xc1, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6};

// Hessian H = M + J^T diag(act*D) J + cone blocks (lower triangle only), engine_solver.c : MakeHessian / HessianCone.
// w.e_act holds act*D per row.  One lane per lower-triangle entry: 2 passes when the trees are uncoupled, 3 otherwise.
__device__ __forceinline__ void make_hessian(WS& w, int lane) {
  const int nefc = w.nefc, nlim = w.nlim, ncon = w.ncon;
  const int nent = w.coupled ? 91 : 49;
#pragma unroll 1
  for (int i = lane; i < nent; i += 32) {
    const int ab = HESS_TRI[i], a = ab >> 4, b = ab & 15;
    float h = w.M[a * NV + b];
#pragma unroll 4
    for (int r = 0; r < nefc; r++) h += w.e_act[r] * w.u.con.J[r][a] * w.u.con.J[r][b];
#pragma unroll 1
    for (int c = 0; c < ncon; c++) {
      if (w.istate[nlim + c] != 2) continue;
      int r = nlim + 4 * c;
      const float* hc = w.hc[c];
      float jb0 = w.u.con.J[r][b], jb1 = w.u.con.J[r + 1][b], jb2 = w.u.con.J[r + 2][b], jb3 = w.u.con.J[r + 3][b];
#pragma unroll
      for (int j = 0; j < 4; j++) h += w.u.con.J[r + j][a] * (hc[4 * j] * jb0 + hc[4 * j + 1] * jb1 + hc[4 * j + 2] * jb2 + hc[4 * j + 3] * jb3);
    }
    w.u.con.H[a * NV + b] = h;
  }
  __syncwarp();
}

// engine_solver.c : mj_solNewton (primal, elliptic cones, exact line search), fp32.
// Returns the number of iterations. On exit w.qacc and w.fcon (= J^T f) are final.
static __device__ __noinline__ int solve_newton(const DevModel& m, WS& w, int lane, int max_iter) {
  const int nefc = w.nefc;
  float qa = 0;
  if (nefc == 0) {
    if (lane < NV) { w.qacc[lane] = w.asmooth[lane]; w.fcon[lane] = 0; }
    __syncwarp();
    return 0;
  }
  // warm start: evaluate the cost at qacc_warmstart and at qacc_smooth, keep the better
  float best_cost = 0, gauss = 0;
#pragma unroll 1
  for (int trial = 0; trial < 2; trial++) {
    float q = lane < NV ? (trial == 0 ? w.warm[lane] : w.asmooth[lane]) : 0.0f;
    if (lane < NV) w.search[lane] = q;  // temp
    __syncwarp();
    float ma = mat13_vec(w.M, w.search, lane);
    rows_dot(w, w.search, w.e_aref, w.e_Jv, lane);  // temp: jar of the trial point
    float g = lane < NV ? 0.5f * (ma - w.fsmooth[lane]) * (q - w.asmooth[lane]) : 0.0f;
    g = warp_sum(g);
    __syncwarp();
    // swap the trial jar in
    float keep0 = 0, keep1 = 0;
    if (lane < nefc) { keep0 = w.e_jar[lane]; w.e_jar[lane] = w.e_Jv[lane]; }
    if (lane + 32 < nefc) { keep1 = w.e_jar[lane + 32]; w.e_jar[lane + 32] = w.e_Jv[lane + 32]; }
    __syncwarp();
    float c = g + constraint_update(w, lane, false);
    if (trial == 0 || c < best_cost) {
      best_cost = c; gauss = g;
      if (lane < NV) { w.qacc[lane] = q; w.Ma[lane] = ma; }
      qa = q;
    } else {
      if (lane < nefc) w.e_jar[lane] = keep0;
      if (lane + 32 < nefc) w.e_jar[lane + 32] = keep1;
    }
    __syncwarp();
  }
  float cost = gauss + constraint_update(w, lane, true);
  const float scale = m.solver_scale;
  const float tol = 1e-8f;  // fp32 working tolerance (reference option tolerance=1e-10 is below fp32 resolution)
  int iter = 0;
  float improvement = 0;
#pragma unroll 1
  for (; iter < max_iter; iter++) {
    // gradient
    float fc = jt_force(w, lane), g = 0;
    if (lane < NV) {
      g = w.Ma[lane] - w.fsmooth[lane] - fc;
      w.fcon[lane] = fc;
      w.grad[lane] = g;
    }
    float gn = scale * sqrtf(warp_sum(g * g));
    if (gn < tol) break;
    if (iter > 0 && improvement < tol) break;
    if (iter > 0 && m.newton_noise > 0.0f) {
      // fp32 resolution of the gradient: g = Ma - fsmooth - J^T f is a difference of terms of magnitude |Ma| + |fsmooth| + |J^T f|,
      // each carrying a few ulps of rounding noise.  Once a Newton step has brought the gradient down to that noise floor a
      // further iteration cannot improve the solution (the fp64 oracle, whose floor is 1e-9 of this, stops here with
      // gradient < tolerance; tools/iter_compare.py: 1.1 vs 2.15 iterations per substep before this test).
      const float mag = lane < NV ? fabsf(w.Ma[lane]) + fabsf(w.fsmooth[lane]) + fabsf(fc) : 0.0f;
      if (gn < m.newton_noise * scale * sqrtf(warp_sum(mag * mag))) break;
    }
    __syncwarp();
    make_hessian(w, lane);
    float s = w.coupled ? chol_factor_solve<false>(w.u.con.H, w.cho, -g, lane) : chol_factor_solve<true>(w.u.con.H, w.cho, -g, lane);
    if (lane < NV) w.search[lane] = s;
    __syncwarp();
    float mv = mat13_vec(w.M, w.search, lane);
    if (lane < NV) w.Mv[lane] = mv;
    rows_dot(w, w.search, nullptr, w.e_Jv, lane);
    float q1 = lane < NV ? s * (w.Ma[lane] - w.fsmooth[lane]) : 0.0f;
    float q2 = lane < NV ? s * mv : 0.0f;
    float sn = lane < NV ? s * s : 0.0f;
    q1 = warp_sum(q1); q2 = warp_sum(q2); sn = sqrtf(warp_sum(sn));
    __syncwarp();
    if (sn < MINVAL) break;
    // exact line search: safeguarded Newton on f'(alpha)
    float d1, d2, alpha = 0, lo = 0, hi = -1;
    line_eval(w, lane, 0.0f, q1, q2, d1, d2);
    if (d1 >= 0 || d2 <= 0) break;
    const float gtol = 1e-6f * fabsf(d1);
    alpha = -d1 / d2;
#pragma unroll 1
    for (int it = 0; it < 20; it++) {
      line_eval(w, lane, alpha, q1, q2, d1, d2);
      if (fabsf(d1) < gtol) break;
      if (d1 < 0) lo = alpha; else hi = alpha;
      float an = alpha - d1 / d2;
      if (hi < 0) { if (an <= lo) an = 2 * lo + 1e-9f; }
      else if (!(an > lo && an < hi)) an = 0.5f * (lo + hi);
      if (hi > 0 && (hi - lo) < 1e-6f * hi) { alpha = 0.5f * (lo + hi); break; }
      alpha = an;
    }
    if (alpha <= 0) break;
    if (lane < NV) { qa += alpha * s; w.qacc[lane] = qa; w.Ma[lane] += alpha * mv; }
#pragma unroll 1
    for (int r = lane; r < nefc; r += 32) w.e_jar[r] += alpha * w.e_Jv[r];
    __syncwarp();
    float gs = lane < NV ? 0.5f * (w.Ma[lane] - w.fsmooth[lane]) * (qa - w.asmooth[lane]) : 0.0f;
    gs = warp_sum(gs);
    float old = cost;
    cost = gs + constraint_update(w, lane, true);
    improvement = scale * (old - cost);
  }
  // final constraint force in joint space: w.fcon is current on every exit through a break (it was computed at the top of that
  // iteration and nothing moved since); only running into the iteration cap leaves it one update behind
  if (iter == max_iter) {
    float fc = jt_force(w, lane);
    if (lane < NV) w.fcon[lane] = fc;
  }
  __syncwarp();
  return iter;
}

// engine_forward.c : mj_Euler with implicit joint damping + mj_integratePos
static __device__ __noinline__ void euler_integrate(const DevModel& m, WS& w, int lane) {
  const float h = m.timestep;
#pragma unroll 1
  for (int e = lane; e < NV * NV; e += 32) {
    int a = e / NV, b = e - a * NV;
    w.u.con.H[e] = w.M[e] + (a == b ? h * m.dof_damping[a] : 0.0f);
  }
  __syncwarp();
  float f = lane < NV ? w.fsmooth[lane] + w.fcon[lane] : 0.0f;
  float qacc = chol_factor_solve<true>(w.u.con.H, w.cho, f, lane);
  if (lane < NV) {
    w.warm[lane] = w.qacc[lane];
    w.qvel[lane] += h * qacc;
  }
  __syncwarp();
  if (lane < m.njnt) {
    int j = lane, qa = m.jnt_qposadr[j], da = m.jnt_dofadr[j];
    if (m.jnt_type[j] == JNT_FREE) {
      for (int k = 0; k < 3; k++) w.qpos[qa + k] += h * w.qvel[da + k];
      float wv[3] = {w.qvel[da + 3], w.qvel[da + 4], w.qvel[da + 5]};
      float ang = sqrtf(dot3(wv, wv));
      if (ang > MINVAL) {
        float inv = 1.0f / ang, s, c, dq[4];
        sincosf(0.5f * ang * h, &s, &c);
        dq[0] = c; dq[1] = wv[0] * inv * s; dq[2] = wv[1] * inv * s; dq[3] = wv[2] * inv * s;
        float q[4] = {w.qpos[qa + 3], w.qpos[qa + 4], w.qpos[qa + 5], w.qpos[qa + 6]};
        quat_mul(q, q, dq);
        quat_normalize(q);
        for (int k = 0; k < 4; k++) w.qpos[qa + 3 + k] = q[k];
      }
    } else {
      w.qpos[qa] += h * w.qvel[da];
    }
  }
  __syncwarp();
}

// dm_control Physics.step() in legacy mode: mj_step2 on the already-computed position stage, then mj_step1.
static __device__ __noinline__ int physics_step(const DevModel& m, WS& w, const float4* hv, const int* adj, int lane, float xfrc_z, bool actuation) {
  smooth_forces(m, w, lane, actuation, xfrc_z);
  make_constraint(m, w, lane);
  int it = solve_newton(m, w, lane, m.iterations);
  euler_integrate(m, w, lane);
  forward_position(m, w, hv, adj, lane);
  return it;
}

}  // namespace grs
