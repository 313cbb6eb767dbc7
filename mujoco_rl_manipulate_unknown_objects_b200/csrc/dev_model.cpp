// HostModel (fp64, mjModel-like) -> DevModel (fp32 POD that the kernels keep in shared memory).
//
// Besides the plain copies this precomputes what the warp-per-environment kernels index by lane:
// depth levels of the kinematic tree, subtree / ancestor bit masks, and the per-pair contact parameters
// that MuJoCo's mj_contactParam (engine_collision_driver.c) mixes from the two geoms at run time.
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <stdexcept>

#include "model.h"

namespace grs {

void build_dev_model(const HostModel& h, DevModel& d, std::vector<float>& hv4, std::vector<int>& adj) {
  std::memset(&d, 0, sizeof d);
  if (h.nq != NQ || h.nv != NV || h.nu != NU)
    throw std::runtime_error("scene does not have the gripper-scene shape nq=14 nv=13 nu=7 (got nq=" + std::to_string(h.nq) + " nv=" + std::to_string(h.nv) +
                             " nu=" + std::to_string(h.nu) + ")");
  if (h.nbody > MAXB || h.njnt > MAXJ || h.ngeom > MAXG || h.npair > MAXPAIR || h.ncam > MAXCAM)
    throw std::runtime_error("scene exceeds the compiled-in limits (bodies/joints/geoms/pairs/cameras)");
  if (h.body_ee < 0 || h.body_object < 0 || h.finger1[0] < 0 || h.finger1[1] < 0 || h.finger2[0] < 0 || h.finger2[1] < 0)
    throw std::runtime_error("scene lacks one of the named bodies ee / object / {left,right}_inner_{knuckle,finger}");
  d.nbody = h.nbody; d.njnt = h.njnt; d.ngeom = h.ngeom; d.npair = h.npair; d.iterations = h.iterations; d.ncam = h.ncam;
  d.timestep = (float)h.timestep; d.impratio = (float)h.impratio; d.meaninertia = (float)h.meaninertia;
  d.solver_scale = (float)(1.0 / (h.meaninertia * std::max(1, h.nv)));
  d.gap_skip = getenv("GRS_GAP_SKIP") ? atoi(getenv("GRS_GAP_SKIP")) : 1;
  d.newton_noise = getenv("GRS_NEWTON_NOISE") ? (float)atof(getenv("GRS_NEWTON_NOISE")) : 3.6e-7f;  // 3 ulps: iteration counts close to the fp64 oracle (tools/iter_compare.py: 1.2 vs 1.1), parity statistics unchanged
  for (int k = 0; k < 3; k++) d.gravity[k] = (float)h.gravity[k];
  d.xfrc_ee_z = (float)(-(0.438 * h.gravity[2]));  // robot_env.py:64-65
  // depth levels
  std::vector<int> depth(h.nbody, 0);
  int maxd = 0;
  for (int b = 1; b < h.nbody; b++) { depth[b] = depth[h.body_parentid[b]] + 1; maxd = std::max(maxd, depth[b]); }
  if (maxd + 1 > MAXLEVEL) throw std::runtime_error("kinematic tree is deeper than the compiled-in limit");
  d.nlevel = maxd + 1;
  int n = 0;
  for (int lv = 0; lv <= maxd; lv++) {
    d.level_start[lv] = n;
    for (int b = 0; b < h.nbody; b++) if (depth[b] == lv) d.level_body[n++] = b;
  }
  for (int lv = maxd + 1; lv <= MAXLEVEL; lv++) d.level_start[lv] = n;
  for (int b = 0; b < h.nbody; b++) {
    d.body_parent[b] = h.body_parentid[b]; d.body_root[b] = h.body_rootid[b];
    d.body_jntadr[b] = h.body_jntadr[b] < 0 ? 0 : h.body_jntadr[b]; d.body_jntnum[b] = h.body_jntnum[b];
    d.body_dofadr[b] = h.body_dofadr[b] < 0 ? 0 : h.body_dofadr[b]; d.body_dofnum[b] = h.body_dofnum[b];
    for (int k = 0; k < 3; k++) { d.body_pos[b][k] = (float)h.body_pos[3 * b + k]; d.body_ipos[b][k] = (float)h.body_ipos[3 * b + k]; d.body_inertia[b][k] = (float)h.body_inertia[3 * b + k]; }
    for (int k = 0; k < 4; k++) { d.body_quat[b][k] = (float)h.body_quat[4 * b + k]; d.body_iquat[b][k] = (float)h.body_iquat[4 * b + k]; }
    d.body_mass[b] = (float)h.body_mass[b];
    d.body_invweight0[b][0] = (float)h.body_invweight0[2 * b]; d.body_invweight0[b][1] = (float)h.body_invweight0[2 * b + 1];
    // subtree mask: every body whose ancestor chain contains b
    unsigned mask = 0;
    for (int c = 0; c < h.nbody; c++) {
      int a = c;
      while (a != b && a > 0) a = h.body_parentid[a];
      if (a == b) mask |= 1u << c;
    }
    d.body_subtree_mask[b] = mask;
    unsigned dm = 0;
    for (int a = b; a > 0; a = h.body_parentid[a])
      for (int k = 0; k < h.body_dofnum[a]; k++) dm |= 1u << (h.body_dofadr[a] + k);
    d.body_dofmask[b] = dm;
  }
  for (int j = 0; j < h.njnt; j++) {
    d.jnt_type[j] = h.jnt_type[j]; d.jnt_body[j] = h.jnt_bodyid[j]; d.jnt_qposadr[j] = h.jnt_qposadr[j];
    d.jnt_dofadr[j] = h.jnt_dofadr[j]; d.jnt_limited[j] = h.jnt_limited[j];
    for (int k = 0; k < 3; k++) { d.jnt_pos[j][k] = (float)h.jnt_pos[3 * j + k]; d.jnt_axis[j][k] = (float)h.jnt_axis[3 * j + k]; }
    d.jnt_range[j][0] = (float)h.jnt_range[2 * j]; d.jnt_range[j][1] = (float)h.jnt_range[2 * j + 1];
    d.jnt_qpos0[j] = (float)h.qpos0[h.jnt_qposadr[j]];
  }
  for (int k = 0; k < 2; k++) d.jnt_solref[k] = (float)h.jnt_solref[k];
  for (int k = 0; k < 5; k++) d.jnt_solimp[k] = (float)h.jnt_solimp[k];
  for (int k = 0; k < NQ; k++) d.qpos0[k] = (float)h.qpos0[k];
  for (int i = 0; i < NV; i++) {
    d.dof_body[i] = h.dof_bodyid[i]; d.dof_jnt[i] = h.dof_jntid[i];
    unsigned am = 0;
    for (int a = i; a >= 0; a = h.dof_parentid[a]) am |= 1u << a;
    d.dof_ancmask[i] = am;
    d.dof_armature[i] = (float)h.dof_armature[i]; d.dof_damping[i] = (float)h.dof_damping[i]; d.dof_invweight0[i] = (float)h.dof_invweight0[i];
  }
  // the fused Cholesky (sim_kernels.cuh chol_factor_solve<true>) relies on M being block diagonal with blocks [0,7) and [7,13)
  for (int i = 0; i < NV; i++) {
    unsigned blk = i < 7 ? 0x7fu : (0x3fu << 7);
    if (d.dof_ancmask[i] & ~blk) throw std::runtime_error("dof tree layout is not 7 gripper dofs followed by 6 free-object dofs");
  }
  hv4.clear(); adj.clear();
  for (int g = 0; g < h.ngeom; g++) {
    d.geom_type[g] = h.geom_type[g]; d.geom_body[g] = h.geom_bodyid[g];
    for (int k = 0; k < 3; k++) d.geom_pos[g][k] = (float)h.geom_pos[3 * g + k];
    for (int k = 0; k < 4; k++) d.geom_quat[g][k] = (float)h.geom_quat[4 * g + k];
    d.geom_rbound[g] = (float)h.geom_rbound[g];
    for (int k = 0; k < 3; k++) d.geom_size[g][k] = (float)h.geom_size[3 * g + k];
    if (h.geom_meshid[g] >= 0) {
      const HostMesh& ms = h.meshes[h.geom_meshid[g]];
      int nvert = (int)ms.hull_verts.size() / 3;
      d.geom_hvadr[g] = (int)hv4.size() / 4; d.geom_hvnum[g] = nvert;
      for (int i = 0; i < nvert; i++) { for (int k = 0; k < 3; k++) hv4.push_back((float)ms.hull_verts[3 * i + k]); hv4.push_back(0.0f); }
      d.geom_adjadr[g] = (int)adj.size();
      adj.insert(adj.end(), ms.adjadr.begin(), ms.adjadr.end());
      adj.insert(adj.end(), ms.adj.begin(), ms.adj.end());
    }
  }
  d.nhv_total = (int)hv4.size() / 4;
  for (int p = 0; p < h.npair; p++) {
    int g1 = h.pair_geom1[p], g2 = h.pair_geom2[p];
    d.pair_g1[p] = g1; d.pair_g2[p] = g2;
    if (std::max(h.geom_condim[g1], h.geom_condim[g2]) != 4)
      throw std::runtime_error("only condim-4 contact pairs are supported (the reference scenes' default geom condim)");
    if (std::max(h.geom_gap[g1], h.geom_gap[g2]) != 0) throw std::runtime_error("geom gap is not supported");
    d.pair_margin[p] = (float)std::max(h.geom_margin[g1], h.geom_margin[g2]);
    for (int k = 0; k < 3; k++) d.pair_fric[p][k] = (float)std::max(h.geom_friction[3 * g1 + k], h.geom_friction[3 * g2 + k]);
    for (int k = 0; k < 2; k++) d.pair_solref[p][k] = (float)(0.5 * (h.geom_solref[2 * g1 + k] + h.geom_solref[2 * g2 + k]));
    for (int k = 0; k < 5; k++) d.pair_solimp[p][k] = (float)(0.5 * (h.geom_solimp[5 * g1 + k] + h.geom_solimp[5 * g2 + k]));
  }
  for (int u = 0; u < NU; u++) {
    d.act_dof[u] = h.act_dofid[u]; d.act_gear[u] = (float)h.act_gear[u];
    d.act_lo[u] = (float)std::max(-1e30, h.act_ctrlrange[2 * u]); d.act_hi[u] = (float)std::min(1e30, h.act_ctrlrange[2 * u + 1]);
  }
  d.body_ee = h.body_ee; d.body_object = h.body_object;
  for (int k = 0; k < 2; k++) { d.finger1[k] = h.finger1[k]; d.finger2[k] = h.finger2[k]; }
  for (int c = 0; c < h.ncam; c++) {
    d.cam_body[c] = h.cam_bodyid[c]; d.cam_mode[c] = h.cam_mode[c]; d.cam_target[c] = h.cam_target[c];
    for (int k = 0; k < 3; k++) d.cam_pos[c][k] = (float)h.cam_pos[3 * c + k];
    for (int k = 0; k < 4; k++) d.cam_quat[c][k] = (float)h.cam_quat[4 * c + k];
    d.cam_fovy[c] = (float)h.cam_fovy[c];
  }
}

std::string scene_mismatch(const HostModel& a, const HostModel& b) {
#define SAME(f) if (!(a.f == b.f)) return #f;
#define SAME_N(f, n) for (int i_ = 0; i_ < (n); i_++) if (!(a.f[i_] == b.f[i_])) return #f;
  SAME(nq) SAME(nv) SAME(nu) SAME(nbody) SAME(njnt) SAME(ngeom) SAME(nmesh) SAME(npair) SAME(ncam) SAME(nlight)
  SAME(body_parentid) SAME(body_jntadr) SAME(body_jntnum) SAME(body_dofadr) SAME(body_dofnum) SAME(body_rootid)
  SAME(jnt_type) SAME(jnt_bodyid) SAME(jnt_qposadr) SAME(jnt_dofadr) SAME(jnt_limited)
  SAME(dof_bodyid) SAME(dof_jntid) SAME(dof_parentid) SAME(act_dofid) SAME(act_gear) SAME(act_ctrlrange)
  SAME(body_ee) SAME(body_object) SAME_N(finger1, 2) SAME_N(finger2, 2)
  SAME(geom_type) SAME(geom_bodyid) SAME(geom_meshid) SAME(pair_geom1) SAME(pair_geom2)
  SAME(geom_rgba) SAME(geom_matprop)
  SAME(timestep) SAME(iterations) SAME(impratio) SAME(cone_elliptic) SAME_N(gravity, 3)
  SAME(cam_names) SAME(cam_fovy)
  SAME(light_bodyid) SAME(light_directional) SAME(light_pos) SAME(light_dir) SAME(light_diffuse) SAME(light_ambient) SAME(light_specular)
  SAME_N(tex_rgb1, 3) SAME_N(tex_rgb2, 3) SAME_N(texrepeat, 2) SAME_N(sky_rgb1, 3) SAME_N(sky_rgb2, 3)
#undef SAME
#undef SAME_N
  // the gripper's collision hulls, render triangles and plane sizes are stored once for all variants
  for (int g = 0; g < a.ngeom; g++) {
    if (a.geom_bodyid[g] == a.body_object) continue;
    for (int k = 0; k < 3; k++) if (a.geom_size[3 * g + k] != b.geom_size[3 * g + k]) return "geom_size";
    if (a.geom_meshid[g] < 0) continue;
    const HostMesh &ma = a.meshes[a.geom_meshid[g]], &mb = b.meshes[b.geom_meshid[g]];
    if (ma.hull_verts != mb.hull_verts) return "hull_verts:" + ma.name;
    if (ma.adjadr != mb.adjadr || ma.adj != mb.adj) return "hull_adj:" + ma.name;
    if (ma.tri != mb.tri) return "mesh_tri:" + ma.name;
  }
  return "";
}

void rebase_hull(const DevModel& d0, DevModel& d, const std::vector<float>& hv4, const std::vector<int>& adj, std::vector<float>& all_hv4,
                 std::vector<int>& all_adj) {
  for (int g = 0; g < d.ngeom; g++) {
    if (d.geom_body[g] != d.body_object) {
      d.geom_hvadr[g] = d0.geom_hvadr[g]; d.geom_adjadr[g] = d0.geom_adjadr[g];
      continue;
    }
    if (d.geom_hvnum[g] == 0) continue;
    int adj_end = (int)adj.size();  // this geom's hull-graph block ends where the next one starts
    for (int o = 0; o < d.ngeom; o++)
      if (d.geom_hvnum[o] > 0 && d.geom_adjadr[o] > d.geom_adjadr[g]) adj_end = std::min(adj_end, d.geom_adjadr[o]);
    const int hv_at = (int)all_hv4.size() / 4, adj_at = (int)all_adj.size();
    all_hv4.insert(all_hv4.end(), hv4.begin() + 4 * d.geom_hvadr[g], hv4.begin() + 4 * (d.geom_hvadr[g] + d.geom_hvnum[g]));
    all_adj.insert(all_adj.end(), adj.begin() + d.geom_adjadr[g], adj.begin() + adj_end);
    d.geom_hvadr[g] = hv_at; d.geom_adjadr[g] = adj_at;
  }
}

}  // namespace grs
