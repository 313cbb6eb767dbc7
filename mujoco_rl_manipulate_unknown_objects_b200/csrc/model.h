// Model structures of the B200 batched gripper simulator.
//
// HostModel : fp64, mjModel-like, produced on the host by mjcf_compiler.cpp from the reference's MJCF
//             scenes (reference xmls/*.xml).  Exported through the C-ABI (grs_model_*) for parity tests.
// DevModel  : fp32 POD copy that lives in HBM, shared read-only by every environment.
//
// Model shape is fixed at compile time for the reference's gripper scenes (SURVEY.md §8: nq=14, nv=13,
// nu=7, nbody=10, ngeom=7): the kernels keep per-dof data in registers with static indexing.
#pragma once
#include <array>
#include <string>
#include <vector>

namespace grs {

constexpr int NQ = 14, NV = 13, NU = 7;
constexpr int MAXB = 10, MAXJ = 8, MAXG = 8, MAXPAIR = 16, MAXMESH = 6, MAXLEVEL = 6;
constexpr int MAXCAM = 4, MAXLIGHT = 4;
constexpr int MAXOBJ = 8;  // scenes (object variants) one simulator can hold

enum GeomType { GEOM_PLANE = 0, GEOM_BOX = 6, GEOM_MESH = 7 };
enum JointType { JNT_FREE = 0, JNT_SLIDE = 2, JNT_HINGE = 3 };

struct HostMesh {
  std::string name;
  std::array<double, 3> pos{};        // CoM offset of the raw mesh (mesh file frame)
  std::array<double, 4> quat{1, 0, 0, 0};
  double volume = 0;
  std::array<double, 3> inertia_unit{};
  std::vector<double> hull_verts;      // nhv x 3, recentred principal frame
  std::vector<int> hull_faces;         // nhf x 3 (hull-local ids, outward)
  std::vector<int> adjadr, adj;        // hull vertex graph (ascending neighbour ids)
  std::vector<float> tri;              // render triangles F x 9, recentred principal frame
};

struct HostModel {
  int nbody = 0, njnt = 0, nq = 0, nv = 0, nu = 0, ngeom = 0, nmesh = 0, npair = 0, ncam = 0, nlight = 0;
  double timestep = 0.002, gravity[3] = {0, 0, -9.81}, impratio = 1, tolerance = 1e-8, znear = 0.01, zfar = 50;
  int iterations = 100, cone_elliptic = 0;
  std::vector<std::string> body_names, geom_names, jnt_names, cam_names;
  std::vector<int> body_parentid, body_weldid, body_jntadr, body_jntnum, body_dofadr, body_dofnum, body_rootid;
  std::vector<double> body_pos, body_quat, body_ipos, body_iquat, body_mass, body_inertia, body_invweight0;
  std::vector<int> jnt_type, jnt_bodyid, jnt_qposadr, jnt_dofadr, jnt_limited;
  std::vector<double> jnt_pos, jnt_axis, jnt_range, qpos0;
  double jnt_solref[2] = {0.02, 1}, jnt_solimp[5] = {0.9, 0.95, 0.001, 0.5, 2};
  std::vector<int> dof_bodyid, dof_jntid, dof_parentid;
  std::vector<double> dof_armature, dof_damping, dof_invweight0;
  std::vector<int> geom_type, geom_bodyid, geom_meshid, geom_condim;
  std::vector<double> geom_pos, geom_quat, geom_friction, geom_margin, geom_gap, geom_solref, geom_solimp,
      geom_rbound, geom_rgba, geom_size, geom_mass, geom_matprop;  // matprop: emission, specular, shininess, textured
  std::vector<HostMesh> meshes;
  std::vector<int> act_dofid;
  std::vector<double> act_gear, act_ctrlrange;
  std::vector<int> pair_geom1, pair_geom2;
  std::vector<int> cam_bodyid, cam_mode, cam_target;
  std::vector<double> cam_pos, cam_quat, cam_fovy;
  std::vector<int> light_bodyid, light_directional;
  std::vector<double> light_pos, light_dir, light_diffuse, light_ambient, light_specular;
  double meaninertia = 1, extent = 1, center[3] = {0, 0, 0};
  double tex_rgb1[3] = {0.1, 0.2, 0.3}, tex_rgb2[3] = {0.2, 0.3, 0.4}, texrepeat[2] = {1, 1};
  double sky_rgb1[3] = {0.3, 0.5, 0.7}, sky_rgb2[3] = {0, 0, 0};
  int body_ee = -1, body_object = -1, finger1[2] = {-1, -1}, finger2[2] = {-1, -1};
};

// Compile an MJCF file (subset used by the reference scenes). Throws std::runtime_error with a message.
HostModel compile_mjcf(const std::string& xml_path);

// ---------------------------------------------------------------- device model (fp32 POD)
struct DevModel {
  int nbody, njnt, ngeom, npair, nlevel, nhv_total, iterations, ncam;
  float timestep, impratio, meaninertia, solver_scale;
  int gap_skip;        // collision: skip convex pairs whose cached separating axis provably still separates them (exact; GRS_GAP_SKIP=0 disables)
  float newton_noise;  // gradient noise floor of the fp32 Newton solver, in units of |Ma| + |fsmooth| + |J^T f| (0 = test disabled)
  float gravity[3], xfrc_ee_z;  // xfrc_ee_z = 0.438*9.81, robot_env.py:64-65
  // bodies, stored in level order is NOT assumed: level_body lists body ids per depth level
  int level_start[MAXLEVEL + 1];
  int level_body[MAXB];
  int body_parent[MAXB], body_root[MAXB], body_jntadr[MAXB], body_jntnum[MAXB], body_dofadr[MAXB], body_dofnum[MAXB];
  unsigned body_subtree_mask[MAXB];  // bit b' set if b' is in the subtree of b (including b)
  unsigned body_dofmask[MAXB];       // dofs on the path from the root to b
  float body_pos[MAXB][3], body_quat[MAXB][4], body_ipos[MAXB][3], body_iquat[MAXB][4];
  float body_mass[MAXB], body_inertia[MAXB][3], body_invweight0[MAXB][2];
  // joints
  int jnt_type[MAXJ], jnt_body[MAXJ], jnt_qposadr[MAXJ], jnt_dofadr[MAXJ], jnt_limited[MAXJ];
  float jnt_pos[MAXJ][3], jnt_axis[MAXJ][3], jnt_range[MAXJ][2], jnt_qpos0[MAXJ];
  float jnt_solref[2], jnt_solimp[5], padj;
  float qpos0[NQ + 2];
  // dofs
  int dof_body[NV + 3], dof_jnt[NV + 3];
  unsigned dof_ancmask[NV + 3];  // ancestors-or-self dofs of dof i
  float dof_armature[NV + 3], dof_damping[NV + 3], dof_invweight0[NV + 3];
  // geoms
  int geom_type[MAXG], geom_body[MAXG], geom_hvadr[MAXG], geom_hvnum[MAXG], geom_adjadr[MAXG];
  float geom_pos[MAXG][3], geom_quat[MAXG][4], geom_rbound[MAXG], geom_size[MAXG][3];
  // candidate pairs with mixed contact parameters (engine_collision_driver.c : mj_contactParam)
  int pair_g1[MAXPAIR], pair_g2[MAXPAIR];
  float pair_margin[MAXPAIR], pair_fric[MAXPAIR][3] /* slide, torsion, roll */, pair_solref[MAXPAIR][2], pair_solimp[MAXPAIR][5];
  // actuators
  int act_dof[NU + 1];
  float act_gear[NU + 1], act_lo[NU + 1], act_hi[NU + 1];
  int body_ee, body_object, finger1[2], finger2[2], pad2, pad3;
  // cameras (fixed, or targetbodycom: look at the subtree CoM of a body)
  int cam_body[MAXCAM], cam_mode[MAXCAM], cam_target[MAXCAM];
  float cam_pos[MAXCAM][3], cam_quat[MAXCAM][4], cam_fovy[MAXCAM];
};

// Flatten a HostModel into the device layout.  hull vertices (float4, w = 0) and the per-geom hull graph
// ([nvert+1 offsets][neighbours], one block per geom) go to separate arrays.
void build_dev_model(const HostModel& h, DevModel& d, std::vector<float>& hull_verts4, std::vector<int>& hull_adj);

// Mixed simulators: several scenes that differ only in the object.  Returns the name of the first shared field (counts, tree,
// joint / dof / actuator layout, named bodies, geoms and pairs, the gripper's hulls and render data, options, cameras' fovy,
// lights and textures) in which `b` differs from `a`, or "" when the two can share one simulator.
std::string scene_mismatch(const HostModel& a, const HostModel& b);

// Appends the object geom's hull of variant `d` to the concatenated arrays and points every other geom of `d` at the hulls of
// variant 0 (`d0`); `hv4` / `adj` are variant d's own arrays from build_dev_model.
void rebase_hull(const DevModel& d0, DevModel& d, const std::vector<float>& hv4, const std::vector<int>& adj, std::vector<float>& all_hv4,
                 std::vector<int>& all_adj);

}  // namespace grs
