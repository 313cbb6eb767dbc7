// Observation builder: a batched software rasteriser for the RGB-D camera images.
//
// Replaces, for every environment at once, RGBDSensor.render_images (reference simulation/controller/sensor.py:56-77:
// two `physics.render` calls = MuJoCo's OpenGL renderer), transform_depth (simulation/utils/utils.py:11-19), the
// observation packing of RobotEnv.get_observation (simulation/environment/robot_env.py:275-293) and the histogram /
// KL part of IntrinsicReward (simulation/environment/reward.py:57-77).
//
// One thread block per (environment, 64x64 pixel tile).  The tile's z-buffer lives in shared memory as 64-bit words
// (depth bits << 32 | primitive id) so that a single atomicMin resolves visibility deterministically:
//   pass 1  every mesh triangle is transformed into the camera frame; triangles with a small pixel footprint are
//           scan-converted by the thread that set them up, large ones are queued and scan-converted by whole warps
//   pass 2  per pixel: floor plane / sky analytically, winner triangle re-fetched for its flat normal, Blinn-Phong
//           shading with the scene's lights + MuJoCo's head light, checker texture, skybox gradient
//   pass 3  (observation path) transform_depth's two reductions, uint8 packing to CHW with the two scalar channels,
//           grey/depth histograms and the KL intrinsic reward, SB3-style terminal observation handling
// Pixel values cannot be pinned against MuJoCo's OpenGL output in the build container; tests compare against
// oracle/render.py, an independent fp64 ray caster of the same scene description (DESIGN.md "observation").
#pragma once
#include <cuda_runtime.h>

#include <cstring>
#include <stdexcept>
#include <vector>

#include "env_kernels.cuh"
#include "model.h"

namespace grs {

constexpr int TILE = 64;
constexpr int RTHREADS = 256;
constexpr int BIGQ = 3072;  // queued large triangles per tile

struct RenderScene {
  const float* tri;  // all mesh triangles, 9 floats each (mesh frame = geom frame)
  int ntri_total;
  int ngeom, plane_geom;
  int geom_triadr[MAXG], geom_trinum[MAXG];
  float geom_rgba[MAXG][4], geom_emission[MAXG], geom_specular[MAXG], geom_shininess[MAXG];
  int geom_textured[MAXG];
  float plane_size[2];
  float tex_rgb1[3], tex_rgb2[3], texrepeat[2], sky_rgb1[3], sky_rgb2[3];
  int nlight;
  int light_directional[MAXLIGHT + 1];
  float light_pos[MAXLIGHT + 1][3], light_dir[MAXLIGHT + 1][3], light_diffuse[MAXLIGHT + 1][3], light_ambient[MAXLIGHT + 1][3], light_specular[MAXLIGHT + 1][3];
  float headlight_ambient[3], headlight_diffuse[3], headlight_specular[3];
  // per variant: the object geom's triangles (variant 0's sit in the geom order, the others' follow every shared triangle) and
  // the clip planes, in metres (scaled by the variant's model extent)
  int obj_geom;
  int obj_triadr[MAXOBJ], obj_trinum[MAXOBJ];
  float znear[MAXOBJ], zfar[MAXOBJ];
};

// triangles of geom g in variant v
__device__ __forceinline__ void geom_tris(const RenderScene& sc, int g, int v, int& adr, int& num) {
  const bool obj = g == sc.obj_geom;
  adr = obj ? sc.obj_triadr[v] : sc.geom_triadr[g];
  num = obj ? sc.obj_trinum[v] : sc.geom_trinum[g];
}

// hs: the variants of one simulator (scene_mismatch found them compatible); everything but the object geom's triangles and the
// clip planes comes from hs[0]
inline void render_scene_upload(const std::vector<HostModel>& hs, RenderScene& sc, std::vector<void*>& owned) {
  const HostModel& h = hs[0];
  std::memset(&sc, 0, sizeof sc);
  std::vector<float> tri;
  sc.ngeom = h.ngeom;
  sc.plane_geom = -1;
  for (int g = 0; g < h.ngeom; g++) {
    sc.geom_triadr[g] = (int)tri.size() / 9;
    if (h.geom_type[g] == GEOM_PLANE) {
      if (sc.plane_geom >= 0) throw std::runtime_error("only one plane geom can be rendered");
      sc.plane_geom = g;
      sc.plane_size[0] = (float)h.geom_size[3 * g]; sc.plane_size[1] = (float)h.geom_size[3 * g + 1];
    } else {
      const auto& t = h.meshes[h.geom_meshid[g]].tri;
      tri.insert(tri.end(), t.begin(), t.end());
    }
    sc.geom_trinum[g] = (int)tri.size() / 9 - sc.geom_triadr[g];
    for (int k = 0; k < 4; k++) sc.geom_rgba[g][k] = (float)h.geom_rgba[4 * g + k];
    sc.geom_emission[g] = (float)h.geom_matprop[4 * g]; sc.geom_specular[g] = (float)h.geom_matprop[4 * g + 1];
    sc.geom_shininess[g] = (float)h.geom_matprop[4 * g + 2]; sc.geom_textured[g] = h.geom_matprop[4 * g + 3] != 0;
  }
  sc.obj_geom = -1;
  for (int g = 0; g < h.ngeom; g++) if (h.geom_bodyid[g] == h.body_object) { sc.obj_geom = g; break; }
  if (sc.obj_geom < 0 || h.geom_meshid[sc.obj_geom] < 0) throw std::runtime_error("the object body has no mesh geom to render");
  for (size_t v = 0; v < hs.size(); v++) {
    if (v == 0) {
      sc.obj_triadr[0] = sc.geom_triadr[sc.obj_geom]; sc.obj_trinum[0] = sc.geom_trinum[sc.obj_geom];
    } else {
      const auto& t = hs[v].meshes[hs[v].geom_meshid[sc.obj_geom]].tri;
      sc.obj_triadr[v] = (int)tri.size() / 9;
      tri.insert(tri.end(), t.begin(), t.end());
      sc.obj_trinum[v] = (int)tri.size() / 9 - sc.obj_triadr[v];
    }
    sc.znear[v] = (float)(hs[v].znear * hs[v].extent); sc.zfar[v] = (float)(hs[v].zfar * hs[v].extent);
  }
  sc.ntri_total = (int)tri.size() / 9;
  if (sc.ntri_total >= (1 << 20)) throw std::runtime_error("too many render triangles");
  float* d = nullptr;
  if (cudaMalloc(&d, (tri.size() + 9) * sizeof(float)) != cudaSuccess) throw std::runtime_error("cudaMalloc(render triangles) failed");
  cudaMemcpy(d, tri.data(), tri.size() * sizeof(float), cudaMemcpyHostToDevice);
  owned.push_back(d);
  sc.tri = d;
  for (int k = 0; k < 3; k++) { sc.tex_rgb1[k] = (float)h.tex_rgb1[k]; sc.tex_rgb2[k] = (float)h.tex_rgb2[k]; sc.sky_rgb1[k] = (float)h.sky_rgb1[k]; sc.sky_rgb2[k] = (float)h.sky_rgb2[k]; }
  sc.texrepeat[0] = (float)h.texrepeat[0]; sc.texrepeat[1] = (float)h.texrepeat[1];
  sc.nlight = std::min(h.nlight, MAXLIGHT);
  for (int l = 0; l < sc.nlight; l++) {
    if (h.light_bodyid[l] != 0) throw std::runtime_error("lights attached to moving bodies are not supported");
    sc.light_directional[l] = h.light_directional[l];
    double dn = 0;
    for (int k = 0; k < 3; k++) dn += h.light_dir[3 * l + k] * h.light_dir[3 * l + k];
    dn = dn > 0 ? 1 / std::sqrt(dn) : 1;
    for (int k = 0; k < 3; k++) {
      sc.light_pos[l][k] = (float)h.light_pos[3 * l + k]; sc.light_dir[l][k] = (float)(h.light_dir[3 * l + k] * dn);
      sc.light_diffuse[l][k] = (float)h.light_diffuse[3 * l + k]; sc.light_ambient[l][k] = (float)h.light_ambient[3 * l + k];
      sc.light_specular[l][k] = (float)h.light_specular[3 * l + k];
    }
  }
  for (int k = 0; k < 3; k++) { sc.headlight_ambient[k] = 0.1f; sc.headlight_diffuse[k] = 0.4f; sc.headlight_specular[k] = 0.5f; }  // mjVisual.headlight defaults
}

// render state of an arbitrary camera for every environment -> first RS_STRIDE floats of each debug row
template <bool MULTI>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32) k_camera_state(SimBuffers s, int cam) {
  stage_models<MULTI>(s);
  WS& w = my_ws(MULTI ? s.nobj : 1);
  const int lane = threadIdx.x & 31;
  for (int env = next_env(s.queue, lane); env < s.n; env = next_env(s.queue, lane)) {
    const DevModel& m = smem_model(MULTI ? s.object[env] : 0);
    EnvFlags f;
    load_state(w, f, s.state + (size_t)env * ST_STRIDE, lane);
    kinematics(m, w, lane);
    com_pos_crb(m, w, lane);
    write_render_state(m, w, cam, s.debug + (size_t)env * DEBUG_STRIDE, lane);
    __syncwarp();
  }
}

struct TileShared {
  unsigned long long zbuf[TILE * TILE];
  float xf[MAXG][12];  // camera-from-geom: R (9) then t (3)
  float cam[12];       // camera pos (3), mat (9) in the world
  int bigq[BIGQ];
  int nbig;
  float red[RTHREADS / 32 + 2];
  unsigned hist[2][256];
  float dxs[TILE], dys[TILE];  // ray-direction components of the tile's pixel columns / rows (camera frame, z = -1)
};

__device__ __forceinline__ unsigned long long pack_frag(float depth, unsigned id) { return ((unsigned long long)__float_as_uint(depth) << 32) | id; }

struct TriSetup { float c0[3], c1[3], c2[3], det; int x0, x1, y0, y1; bool ok; };

// camera-space setup of triangle `t` of geom `g`; pixel bounding box clipped to the tile [tx0, tx0+tw) x [ty0, ty0+th)
__device__ __forceinline__ TriSetup tri_setup(const float* __restrict__ tri, const float* xf, float fx, float fy, int W, int H, int tx0, int ty0, int tw, int th, float znear) {
  TriSetup s;
  float v[3][3];
#pragma unroll
  for (int c = 0; c < 3; c++) {
    float a = __ldg(tri + 3 * c), b = __ldg(tri + 3 * c + 1), d = __ldg(tri + 3 * c + 2);
    v[c][0] = xf[0] * a + xf[1] * b + xf[2] * d + xf[9];
    v[c][1] = xf[3] * a + xf[4] * b + xf[5] * d + xf[10];
    v[c][2] = xf[6] * a + xf[7] * b + xf[8] * d + xf[11];
  }
  s.ok = false;
  float zmax = fmaxf(-v[0][2], fmaxf(-v[1][2], -v[2][2])), zmin = fminf(-v[0][2], fminf(-v[1][2], -v[2][2]));
  if (zmax < znear) return s;  // entirely in front of the near plane / behind the camera
  cross3(s.c0, v[1], v[2]); cross3(s.c1, v[2], v[0]); cross3(s.c2, v[0], v[1]);
  s.det = dot3(v[0], s.c0);
  if (s.det == 0.0f) return s;
  int x0 = tx0, x1 = tx0 + tw - 1, y0 = ty0, y1 = ty0 + th - 1;
  if (zmin > znear) {  // all three vertices project: tight box
    float sxmin = 3e38f, sxmax = -3e38f, symin = 3e38f, symax = -3e38f;
#pragma unroll
    for (int c = 0; c < 3; c++) {
      float iz = 1.0f / (-v[c][2]);
      float px = (v[c][0] * iz * fx + 1.0f) * 0.5f * W - 0.5f, py = (1.0f - v[c][1] * iz * fy) * 0.5f * H - 0.5f;
      sxmin = fminf(sxmin, px); sxmax = fmaxf(sxmax, px); symin = fminf(symin, py); symax = fmaxf(symax, py);
    }
    if (sxmax < (float)tx0 - 1.0f || sxmin > (float)(tx0 + tw) || symax < (float)ty0 - 1.0f || symin > (float)(ty0 + th)) return s;
    x0 = max(x0, (int)floorf(fmaxf(sxmin, -1.0f)));      x1 = min(x1, (int)ceilf(fminf(sxmax, (float)W)));
    y0 = max(y0, (int)floorf(fmaxf(symin, -1.0f)));      y1 = min(y1, (int)ceilf(fminf(symax, (float)H)));
    x0 = max(x0, tx0); y0 = max(y0, ty0);
    if (x1 < x0 || y1 < y0) return s;
  }
  s.x0 = x0; s.x1 = x1; s.y0 = y0; s.y1 = y1; s.ok = true;
  return s;
}

// One fragment.  dx, dy = ray direction of the pixel (from the tile tables), lx, ly = pixel coordinates inside the tile.
__device__ __forceinline__ void raster_pixel(const TriSetup& s, float dx, float dy, int lx, int ly, float znear, float zfar, unsigned id, unsigned long long* zbuf) {
  float e0 = dx * s.c0[0] + dy * s.c0[1] - s.c0[2];
  float e1 = dx * s.c1[0] + dy * s.c1[1] - s.c1[2];
  float e2 = dx * s.c2[0] + dy * s.c2[1] - s.c2[2];
  bool in = (e0 >= 0 && e1 >= 0 && e2 >= 0) || (e0 <= 0 && e1 <= 0 && e2 <= 0);
  if (!in) return;
  float sum = e0 + e1 + e2;
  if (sum == 0.0f) return;
  float t = s.det / sum;
  if (!(t >= znear && t <= zfar)) return;
  atomicMin(&zbuf[ly * TILE + lx], pack_frag(t, id));
}

// Conservative pixel span [lo, hi] of triangle `s` on the row with ray component dy: every edge function is affine in the
// pixel column (e_k = alpha_k * px + beta_k), so each edge bounds the column range from one side.  The span is widened by a
// pixel on both sides and the exact per-pixel test still decides, so the image is identical to testing the whole box.
__device__ __forceinline__ void row_span(const TriSetup& s, float dy, float A, float B, int& lo, int& hi) {
  const float sg = s.det > 0.0f ? 1.0f : -1.0f;
  float flo = (float)s.x0, fhi = (float)s.x1;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const float* c = k == 0 ? s.c0 : k == 1 ? s.c1 : s.c2;
    const float alpha = sg * c[0] * A, beta = sg * (c[0] * B + dy * c[1] - c[2]);
    if (alpha > 0.0f) flo = fmaxf(flo, -beta / alpha - 1.0f);
    else if (alpha < 0.0f) fhi = fminf(fhi, -beta / alpha + 1.0f);
    else if (beta < 0.0f) fhi = flo - 4.0f;  // the whole row is outside this edge
  }
  lo = max(s.x0, (int)floorf(flo));
  hi = min(s.x1, (int)ceilf(fhi));
  if (!(fhi >= flo - 2.0f)) hi = lo - 1;  // also catches NaN
}

struct Shade { float r, g, b; };

// OpenGL fixed-function style lighting evaluated per pixel: emission + sum over lights of ambient + diffuse + Blinn specular
__device__ __forceinline__ Shade shade_point(const RenderScene& sc, int g, const float* p, const float* nrm, const float* eye, const float* view_fwd, const float* tex) {
  float n[3] = {nrm[0], nrm[1], nrm[2]}, vdir[3] = {eye[0] - p[0], eye[1] - p[1], eye[2] - p[2]};
  normalize3(vdir);
  if (dot3(n, vdir) < 0) { n[0] = -n[0]; n[1] = -n[1]; n[2] = -n[2]; }  // two-sided
  const float* rgba = sc.geom_rgba[g];
  float em = sc.geom_emission[g], spec = sc.geom_specular[g], shin = fmaxf(sc.geom_shininess[g] * 128.0f, 1e-3f);
  float col[3] = {em * rgba[0], em * rgba[1], em * rgba[2]};
  for (int l = 0; l <= sc.nlight; l++) {
    float L[3], att = 1.0f;
    const float *amb, *dif, *spc;
    if (l == sc.nlight) {  // head light: directional, along the viewing direction
      L[0] = -view_fwd[0]; L[1] = -view_fwd[1]; L[2] = -view_fwd[2];
      amb = sc.headlight_ambient; dif = sc.headlight_diffuse; spc = sc.headlight_specular;
    } else {
      amb = sc.light_ambient[l]; dif = sc.light_diffuse[l]; spc = sc.light_specular[l];
      if (sc.light_directional[l]) { L[0] = -sc.light_dir[l][0]; L[1] = -sc.light_dir[l][1]; L[2] = -sc.light_dir[l][2]; }
      else {
        for (int k = 0; k < 3; k++) L[k] = sc.light_pos[l][k] - p[k];
        normalize3(L);
        float cs = -(L[0] * sc.light_dir[l][0] + L[1] * sc.light_dir[l][1] + L[2] * sc.light_dir[l][2]);  // spot: cutoff 45 deg, exponent 10 (MJCF defaults)
        att = cs < 0.70710678f ? 0.0f : powf(cs, 10.0f);
      }
    }
    float ndl = fmaxf(dot3(n, L), 0.0f);
    float Hh[3] = {L[0] + vdir[0], L[1] + vdir[1], L[2] + vdir[2]};
    normalize3(Hh);
    float ndh = fmaxf(dot3(n, Hh), 0.0f);
    float sp = ndl > 0 ? spec * powf(ndh, shin) : 0.0f;
    for (int k = 0; k < 3; k++) col[k] += amb[k] * rgba[k] + att * (dif[k] * rgba[k] * ndl + spc[k] * sp);
  }
  Shade o;
  o.r = fminf(col[0], 1.0f) * tex[0]; o.g = fminf(col[1], 1.0f) * tex[1]; o.b = fminf(col[2], 1.0f) * tex[2];
  return o;
}

// Renders one tile into shared memory: after the call zbuf[pix] low word = depth (float bits, metres along the optical axis),
// and rgb8[pix] holds the packed colour.  rs = this environment's render state (geom poses + camera), v = its variant.
static __device__ void render_tile(const RenderScene& sc, const float* __restrict__ rs, int v, TileShared& sh, unsigned* rgb8, int W, int H, int tx0, int ty0, int tw, int th,
                            float fovy) {
  const int tid = threadIdx.x;
  const float znear = sc.znear[v], zfar = sc.zfar[v];
  const float ify = tanf(0.5f * fovy * 0.017453292519943295f) /* MJCF fovy is always in degrees */, ifx = ify * (float)W / (float)H;
  const float fx = 1.0f / ifx, fy = 1.0f / ify;
  for (int i = tid; i < TILE * TILE; i += RTHREADS) sh.zbuf[i] = pack_frag(zfar, 0xffffffffu);
  if (tid < 12) sh.cam[tid] = rs[84 + tid];
  if (tid == 0) sh.nbig = 0;
  if (tid < TILE) sh.dxs[tid] = ((2.0f * ((tx0 + tid) + 0.5f)) / W - 1.0f) * ifx;
  else if (tid < 2 * TILE) sh.dys[tid - TILE] = (1.0f - (2.0f * ((ty0 + tid - TILE) + 0.5f)) / H) * ify;
  __syncthreads();
  if (tid < sc.ngeom * 12) {
    int g = tid / 12, k = tid - g * 12;
    const float* gp = rs + g * 12;      // pos(3), mat(9)
    const float* cp = sh.cam;           // pos(3), mat(9): columns = camera axes in the world
    float v;
    if (k < 9) {  // R = Rc^T Rg
      int r = k / 3, c = k - 3 * r;
      v = cp[3 + r] * gp[3 + c] + cp[3 + 3 + r] * gp[3 + 3 + c] + cp[3 + 6 + r] * gp[3 + 6 + c];
    } else {
      int r = k - 9;
      v = cp[3 + r] * (gp[0] - cp[0]) + cp[3 + 3 + r] * (gp[1] - cp[1]) + cp[3 + 6 + r] * (gp[2] - cp[2]);
    }
    sh.xf[g][k] = v;
  }
  __syncthreads();
  // ---- pass 1a: per-thread triangles
  for (int g = 0; g < sc.ngeom; g++) {
    int n, adr;
    geom_tris(sc, g, v, adr, n);
    for (int t = tid; t < n; t += RTHREADS) {
      TriSetup s = tri_setup(sc.tri + (size_t)(adr + t) * 9, sh.xf[g], fx, fy, W, H, tx0, ty0, tw, th, znear);
      if (!s.ok) continue;
      int area = (s.x1 - s.x0 + 1) * (s.y1 - s.y0 + 1);
      unsigned id = (unsigned)(adr + t);
      if (area > 24) {
        int q = atomicAdd(&sh.nbig, 1);
        if (q < BIGQ) { sh.bigq[q] = (g << 24) | t; continue; }
      }
      for (int py = s.y0; py <= s.y1; py++)
        for (int px = s.x0; px <= s.x1; px++) raster_pixel(s, sh.dxs[px - tx0], sh.dys[py - ty0], px - tx0, py - ty0, znear, zfar, id, sh.zbuf);
    }
  }
  __syncthreads();
  // ---- pass 1b: queued large triangles, one warp each
  {
    const int nb = min(sh.nbig, BIGQ), warp = tid >> 5, lane = tid & 31;
    for (int q = warp; q < nb; q += RTHREADS / 32) {
      int g = sh.bigq[q] >> 24, t = sh.bigq[q] & 0xffffff, adr, n;
      geom_tris(sc, g, v, adr, n);
      TriSetup s = tri_setup(sc.tri + (size_t)(adr + t) * 9, sh.xf[g], fx, fy, W, H, tx0, ty0, tw, th, znear);
      if (!s.ok) continue;
      unsigned id = (unsigned)(adr + t);
      // dx(px) = A * px + B
      const float A = 2.0f * ifx / (float)W, B = (1.0f / (float)W - 1.0f) * ifx;
      for (int py = s.y0 + lane; py <= s.y1; py += 32) {  // one row per lane, only the columns the triangle can cover
        const float dy = sh.dys[py - ty0];
        int lo, hi;
        row_span(s, dy, A, B, lo, hi);
        for (int px = lo; px <= hi; px++) raster_pixel(s, sh.dxs[px - tx0], dy, px - tx0, py - ty0, znear, zfar, id, sh.zbuf);
      }
    }
  }
  __syncthreads();
  // ---- pass 2: shading
  const float* cp = sh.cam;
  const float fwd[3] = {-cp[3 + 2], -cp[3 + 5], -cp[3 + 8]};
  for (int i = tid; i < tw * th; i += RTHREADS) {
    int ly = i / tw, lx = i - ly * tw, px = tx0 + lx, py = ty0 + ly;
    unsigned long long z = sh.zbuf[ly * TILE + lx];
    float depth = __uint_as_float((unsigned)(z >> 32));
    unsigned id = (unsigned)z;
    float dx = sh.dxs[lx], dy = sh.dys[ly];
    // ray direction in the world (not normalised; camera-axis component = 1)
    float dw[3] = {cp[3] * dx + cp[4] * dy - cp[5], cp[6] * dx + cp[7] * dy - cp[8], cp[9] * dx + cp[10] * dy - cp[11]};
    int hit_geom = -1;
    float nrm[3] = {0, 0, 1};
    if (id != 0xffffffffu) {
      int g = 0;
      for (int k = 1; k < sc.ngeom; k++) if (k != sc.obj_geom && (int)id >= sc.geom_triadr[k] && sc.geom_trinum[k] > 0) g = k;
      if ((int)id >= sc.obj_triadr[v] && (int)id < sc.obj_triadr[v] + sc.obj_trinum[v]) g = sc.obj_geom;
      hit_geom = g;
      const float* tp = sc.tri + (size_t)id * 9;
      float a[3] = {__ldg(tp), __ldg(tp + 1), __ldg(tp + 2)}, e1[3] = {__ldg(tp + 3) - a[0], __ldg(tp + 4) - a[1], __ldg(tp + 5) - a[2]},
            e2[3] = {__ldg(tp + 6) - a[0], __ldg(tp + 7) - a[1], __ldg(tp + 8) - a[2]}, nl[3];
      cross3(nl, e1, e2);
      mulmat3vec(nrm, rs + g * 12 + 3, nl);
      normalize3(nrm);
    }
    // floor plane, analytic
    if (sc.plane_geom >= 0) {
      const float* pp = rs + sc.plane_geom * 12;
      const float* pm = pp + 3;
      float pn[3] = {pm[2], pm[5], pm[8]};
      float denom = dot3(pn, dw);
      float num = pn[0] * (pp[0] - cp[0]) + pn[1] * (pp[1] - cp[1]) + pn[2] * (pp[2] - cp[2]);
      if (denom != 0.0f) {
        float t = num / denom;
        if (t >= znear && t < depth) {
          float hp[3] = {cp[0] + t * dw[0] - pp[0], cp[1] + t * dw[1] - pp[1], cp[2] + t * dw[2] - pp[2]};
          float u = hp[0] * pm[0] + hp[1] * pm[3] + hp[2] * pm[6], v = hp[0] * pm[1] + hp[1] * pm[4] + hp[2] * pm[7];
          bool inside = (sc.plane_size[0] <= 0 || fabsf(u) <= sc.plane_size[0]) && (sc.plane_size[1] <= 0 || fabsf(v) <= sc.plane_size[1]);
          if (inside) { depth = t; hit_geom = sc.plane_geom; nrm[0] = pn[0]; nrm[1] = pn[1]; nrm[2] = pn[2]; }
        }
      }
    }
    Shade c;
    if (hit_geom < 0) {  // skybox gradient: rgb1 at the zenith, rgb2 at the nadir, linear in the cube-face height
      float m = fmaxf(fabsf(dw[0]), fmaxf(fabsf(dw[1]), fabsf(dw[2])));
      float f = 0.5f * (dw[2] / m + 1.0f);
      c.r = sc.sky_rgb2[0] + f * (sc.sky_rgb1[0] - sc.sky_rgb2[0]); c.g = sc.sky_rgb2[1] + f * (sc.sky_rgb1[1] - sc.sky_rgb2[1]); c.b = sc.sky_rgb2[2] + f * (sc.sky_rgb1[2] - sc.sky_rgb2[2]);
      depth = zfar;
    } else {
      float p[3] = {cp[0] + depth * dw[0], cp[1] + depth * dw[1], cp[2] + depth * dw[2]};
      float tex[3] = {1, 1, 1};
      if (sc.geom_textured[hit_geom] && hit_geom == sc.plane_geom) {  // builtin 2x2 checker, texuniform: texrepeat tiles per metre
        const float* pp = rs + sc.plane_geom * 12;
        const float* pm = pp + 3;
        float hp[3] = {p[0] - pp[0], p[1] - pp[1], p[2] - pp[2]};
        float u = hp[0] * pm[0] + hp[1] * pm[3] + hp[2] * pm[6], v = hp[0] * pm[1] + hp[1] * pm[4] + hp[2] * pm[7];
        int cu = (int)floorf(u * sc.texrepeat[0] * 2.0f), cv = (int)floorf(v * sc.texrepeat[1] * 2.0f);
        const float* tc = ((cu + cv) & 1) ? sc.tex_rgb2 : sc.tex_rgb1;
        tex[0] = tc[0]; tex[1] = tc[1]; tex[2] = tc[2];
      }
      c = shade_point(sc, hit_geom, p, nrm, cp, fwd, tex);
    }
    unsigned r8 = (unsigned)(fminf(fmaxf(c.r, 0.0f), 1.0f) * 255.0f + 0.5f), g8 = (unsigned)(fminf(fmaxf(c.g, 0.0f), 1.0f) * 255.0f + 0.5f),
             b8 = (unsigned)(fminf(fmaxf(c.b, 0.0f), 1.0f) * 255.0f + 0.5f);
    rgb8[ly * TILE + lx] = r8 | (g8 << 8) | (b8 << 16);
    sh.zbuf[ly * TILE + lx] = (unsigned long long)__float_as_uint(depth);
  }
  __syncthreads();
}

__device__ __forceinline__ float block_reduce(float v, float* red, int op /*0 sum, 1 min*/) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { float u = __shfl_xor_sync(FULL, v, o); v = op ? fminf(v, u) : v + u; }
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  if (warp == 0) {
    float x = lane < RTHREADS / 32 ? red[lane] : (op ? 3.0e38f : 0.0f);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { float u = __shfl_xor_sync(FULL, x, o); x = op ? fminf(x, u) : x + u; }
    if (lane == 0) red[RTHREADS / 32] = x;
  }
  __syncthreads();
  return red[RTHREADS / 32];
}

// Everything the observation builder needs besides the per-step simulator buffers.
struct ObsArgs {
  unsigned char* obs;           // [n][C][H][W] uint8
  unsigned char* terminal_obs;  // likewise (SB3 terminal observation of environments that finished an episode)
  const unsigned char* reset_obs;  // [nobj][C][H][W] observation of a freshly reset environment, per variant
  float* hist_prev;             // [n][2][256] float histograms (grey, depth) of each env's previous observation
  float* hist_reset;            // [nobj][2][256] the reset images' histograms
  const int* object;            // [n] variant of each environment's current episode (the one a reset started)
  int C, H, W;
  float fovy;
  int auto_reset, im_reward;
  // reset randomisation: the observation of a new episode is rendered (reset record's scene with the object geom at its
  // per-environment pose) instead of copied from the constant reset image
  int reset_noise, obj_geom;
  const float* reset_rs;   // [nobj] render states of the reset records, REC_STRIDE apart
  const float* reset_obj;  // [n][12] object geom pose of each environment's current episode
  unsigned char reset_pad0[MAXOBJ], reset_pad1[MAXOBJ];  // pad-channel scalars of a freshly reset environment, per variant
  // host mirrors (grs_step_host with PINNED host buffers): device-visible addresses of the caller's pinned observation /
  // terminal-observation arrays, or NULL.  Each finished observation is stored there by the block that built it, so the
  // device-to-host transfer of the 20 KB images rides under the physics of the environments still integrating.
  unsigned char* obs_host;
  unsigned char* terminal_obs_host;
  // intrinsic reward bookkeeping (reward.py:51-55 adds the KL term to the step reward, which robot_env.py:199 sums into
  // the episode): per-env info rows and state records, with the slots the term has to reach
  float* info;
  float* state;
  int info_stride, state_stride, in_reward, in_ep_return, st_ep_return;
};

// copy `bytes` of an observation this block has just written to global memory into the caller's pinned host array
__device__ __forceinline__ void mirror_to_host(const unsigned char* src, unsigned char* dst_host, int bytes) {
  __syncthreads();  // the block's own stores to `src` are visible to the block
  if ((bytes & 15) == 0) {
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* d4 = reinterpret_cast<uint4*>(dst_host);
    for (int i = threadIdx.x; i < bytes / 16; i += RTHREADS) d4[i] = __ldcg(s4 + i);
  } else {
    for (int i = threadIdx.x; i < bytes; i += RTHREADS) dst_host[i] = __ldcg(src + i);
  }
}

// Observation of ONE environment by one block of RTHREADS threads (the observation is a single tile, W,H <= 64):
// rasterise + shade (render_tile), transform_depth, uint8 CHW packing with the two scalar channels, histograms, intrinsic
// reward, SB3 terminal-observation / reset-observation swap.
//   rs       : this env's render state (geom poses + camera), any address space
//   pad0/1   : grasp / pheromone scalars of the pad channel;  is_done : done flag of the step just taken
//   reward   : per-env reward array (the intrinsic term is added in place), or NULL
// rasterise + shade the scene `rs`, transform_depth, pack uint8 CHW with the two scalar channels into `dst`, histograms of the
// grey image and of the depth channel into sh.hist
__device__ __forceinline__ void render_and_pack(const RenderScene& sc, const ObsArgs& o, const float* rs, int v, unsigned char* dst, unsigned char pad0, unsigned char pad1,
                                                TileShared& sh, unsigned* rgb8) {
  const int tid = threadIdx.x, C = o.C, H = o.H, W = o.W;
  render_tile(sc, rs, v, sh, rgb8, W, H, 0, 0, W, H, o.fovy);
  const int npix = W * H;
  // transform_depth (utils.py:11-19): d -= min(d); d /= 2*mean(d[d <= 1]); 255*clip(d, 0, 1)
  float mn = 3.0e38f;
  for (int i = tid; i < npix; i += RTHREADS) mn = fminf(mn, __uint_as_float((unsigned)sh.zbuf[(i / W) * TILE + i % W]));
  mn = block_reduce(mn, sh.red, 1);
  float sm = 0, cnt = 0;
  for (int i = tid; i < npix; i += RTHREADS) {
    float d = __uint_as_float((unsigned)sh.zbuf[(i / W) * TILE + i % W]) - mn;
    if (d <= 1.0f) { sm += d; cnt += 1.0f; }
  }
  sm = block_reduce(sm, sh.red, 0);
  cnt = block_reduce(cnt, sh.red, 0);
  const float denom = 2.0f * (sm / cnt);  // cnt >= 1: the minimum pixel itself
  for (int i = tid; i < 512; i += RTHREADS) (&sh.hist[0][0])[i] = 0;
  __syncthreads();
  for (int i = tid; i < npix; i += RTHREADS) {
    int y = i / W, x = i - y * W;
    unsigned c = rgb8[y * TILE + x];
    unsigned r8 = c & 255, g8 = (c >> 8) & 255, b8 = (c >> 16) & 255;
    float d = (__uint_as_float((unsigned)sh.zbuf[y * TILE + x]) - mn) / denom;
    float pix = 255.0f * fminf(fmaxf(d, 0.0f), 1.0f);
    unsigned d8 = (pix == pix) ? (unsigned)pix : 0u;  // astype(uint8) truncates
    dst[i] = (unsigned char)r8; dst[npix + i] = (unsigned char)g8; dst[2 * npix + i] = (unsigned char)b8;
    int ch = 3;
    if (C == 5) { dst[3 * npix + i] = (unsigned char)d8; ch = 4; }
    dst[ch * npix + i] = i == 0 ? pad0 : i == 1 ? pad1 : 0;
    // reward.py:63 — cv2.cvtColor(obs[..., :3], COLOR_BGR2GRAY) applied to RGB-ordered data: channel 0 gets the blue weight
    unsigned grey = (r8 * 3735u + g8 * 19235u + b8 * 9798u + 16384u) >> 15;
    atomicAdd(&sh.hist[0][grey], 1u);
    atomicAdd(&sh.hist[1][d8], 1u);
  }
  __syncthreads();
}

// scene of a freshly reset environment of variant v with the object geom at this environment's pose -> rs2 (shared memory,
// RS_STRIDE floats)
__device__ __forceinline__ void build_reset_scene(const ObsArgs& o, int env, int v, float* rs2) {
  const int tid = threadIdx.x;
  __syncthreads();
  if (tid < RS_STRIDE) {
    const int g = tid / 12;
    rs2[tid] = (g == o.obj_geom && tid < 84) ? __ldcg(o.reset_obj + (size_t)env * 12 + (tid - 12 * g)) : o.reset_rs[(size_t)v * REC_STRIDE + tid];
  }
  __syncthreads();
}

// v: the variant of the episode the step belongs to (info IN_OBJECT); an auto-reset's new episode is o.object[env]
__device__ __forceinline__ void render_obs_env(const RenderScene& sc, const ObsArgs& o, const float* rs, int v, int env, unsigned char pad0, unsigned char pad1,
                                               bool is_done, float* reward, TileShared& sh, unsigned* rgb8, float* rs2) {
  const int tid = threadIdx.x, C = o.C, auto_reset = o.auto_reset, im_reward = o.im_reward, npix = o.W * o.H;
  unsigned char* obs = o.obs;
  const unsigned char* reset_obs = o.reset_obs;
  float* hist_prev = o.hist_prev;
  float* hist_reset = o.hist_reset;
  const bool swap = is_done && auto_reset;
  unsigned char* dst = swap ? o.terminal_obs + (size_t)env * C * npix : obs + (size_t)env * C * npix;
  render_and_pack(sc, o, rs, v, dst, pad0, pad1, sh, rgb8);
  {
    unsigned char* hm = swap ? o.terminal_obs_host : o.obs_host;
    if (hm) mirror_to_host(dst, hm + (size_t)env * C * npix, C * npix);
  }
  // intrinsic reward (reward.py:57-77): KL(old || new) of the grey (and depth) histograms, float32 pdfs
  float* hp = hist_prev ? hist_prev + (size_t)env * 512 : nullptr;
  if (im_reward && reward && hp) {
    float kl_g = 0, kl_d = 0;
    for (int i = tid; i < 256; i += RTHREADS) {
      float po = hp[i] / (float)npix, pn = (float)sh.hist[0][i] / (float)npix;
      if (po > 0 && pn > 0) kl_g += po * logf(po / pn);
      float qo = hp[256 + i] / (float)npix, qn = (float)sh.hist[1][i] / (float)npix;
      if (qo > 0 && qn > 0) kl_d += qo * logf(qo / qn);
    }
    kl_g = block_reduce(kl_g, sh.red, 0);
    kl_d = block_reduce(kl_d, sh.red, 0);
    if (tid == 0) {
      const float kl = C == 5 ? 0.5f * (kl_g + kl_d) : kl_g;
      reward[env] = __ldcg(reward + env) + kl;
      if (o.info) {  // the info record's reward / Monitor return and the running episode return carry the term as well
        float* inf = o.info + (size_t)env * o.info_stride;
        inf[o.in_reward] = __ldcg(inf + o.in_reward) + kl;
        inf[o.in_ep_return] = __ldcg(inf + o.in_ep_return) + kl;
        if (o.state && !swap) { float* st = o.state + (size_t)env * o.state_stride; st[o.st_ep_return] = __ldcg(st + o.st_ep_return) + kl; }
      }
    }
  }
  __syncthreads();
  if (is_done && auto_reset) {
    // SB3 VecEnv: the returned observation is the first one of the next episode; the terminal one went to terminal_obs
    const int vn = __ldcg(o.object + env);
    if (o.reset_noise) {
      build_reset_scene(o, env, vn, rs2);
      render_and_pack(sc, o, rs2, vn, obs + (size_t)env * C * npix, o.reset_pad0[vn], o.reset_pad1[vn], sh, rgb8);
      if (o.obs_host) mirror_to_host(obs + (size_t)env * C * npix, o.obs_host + (size_t)env * C * npix, C * npix);
      if (hp) for (int i = tid; i < 512; i += RTHREADS) hp[i] = (float)(&sh.hist[0][0])[i];
    } else {
      reset_obs += (size_t)vn * C * npix;
      hist_reset += (size_t)vn * 512;
      const uint4* src = reinterpret_cast<const uint4*>(reset_obs);
      uint4* o4 = reinterpret_cast<uint4*>(obs + (size_t)env * C * npix);
      if ((C * npix) % 16 == 0) { for (int i = tid; i < C * npix / 16; i += RTHREADS) o4[i] = src[i]; }
      else { for (int i = tid; i < C * npix; i += RTHREADS) obs[(size_t)env * C * npix + i] = reset_obs[i]; }
      if (o.obs_host) {
        unsigned char* oh = o.obs_host + (size_t)env * C * npix;
        if ((C * npix) % 16 == 0) { uint4* h4 = reinterpret_cast<uint4*>(oh); for (int i = tid; i < C * npix / 16; i += RTHREADS) h4[i] = src[i]; }
        else { for (int i = tid; i < C * npix; i += RTHREADS) oh[i] = reset_obs[i]; }
      }
      if (hp) for (int i = tid; i < 512; i += RTHREADS) hp[i] = hist_reset[i];
    }
  } else {
    float* ho = hp ? hp : hist_reset;
    if (ho) for (int i = tid; i < 512; i += RTHREADS) ho[i] = (float)(&sh.hist[0][0])[i];
  }
}

// Standalone observation kernel: one block per environment.  info: per-env info rows; done: per-env done flags (NULL for
// the reset image).  Renders the reset images; the synchronous step builds its observations in the step kernel's observation
// phase (render_phase) and the asynchronous one with k_render_obs_indexed.
static __global__ void __launch_bounds__(RTHREADS) k_render_obs(RenderScene sc, ObsArgs o, const float* __restrict__ render_state, const float* __restrict__ info, int info_stride,
                                                        const unsigned char* __restrict__ done, float* __restrict__ reward) {
  extern __shared__ __align__(16) unsigned char rsm[];
  TileShared& sh = *reinterpret_cast<TileShared*>(rsm);
  unsigned* rgb8 = reinterpret_cast<unsigned*>(rsm + sizeof(TileShared));
  float* rs2 = reinterpret_cast<float*>(rsm + sizeof(TileShared) + TILE * TILE * sizeof(unsigned));
  const int env = blockIdx.x;
  const float* inf = info + (size_t)env * info_stride;
  render_obs_env(sc, o, render_state + (size_t)env * RS_STRIDE, (int)inf[IN_OBJECT], env, (unsigned char)inf[IN_GRASP], (unsigned char)inf[IN_PHEROMONE],
                 done ? done[env] != 0 : false, reward, sh, rgb8, rs2);
}

// The same over a list: block b builds the observation of environment list[b] for b < *count (the asynchronous step renders
// the environments its launch finished; the grid is sized for the largest possible count).
static __global__ void __launch_bounds__(RTHREADS) k_render_obs_indexed(RenderScene sc, ObsArgs o, const float* __restrict__ render_state, const float* __restrict__ info,
                                                                int info_stride, const unsigned char* __restrict__ done, float* __restrict__ reward,
                                                                const int* __restrict__ list, const int* __restrict__ count) {
  if ((int)blockIdx.x >= *count) return;
  extern __shared__ __align__(16) unsigned char rsm[];
  TileShared& sh = *reinterpret_cast<TileShared*>(rsm);
  unsigned* rgb8 = reinterpret_cast<unsigned*>(rsm + sizeof(TileShared));
  float* rs2 = reinterpret_cast<float*>(rsm + sizeof(TileShared) + TILE * TILE * sizeof(unsigned));
  const int env = list[blockIdx.x];
  const float* inf = info + (size_t)env * info_stride;
  render_obs_env(sc, o, render_state + (size_t)env * RS_STRIDE, (int)inf[IN_OBJECT], env, (unsigned char)inf[IN_GRASP], (unsigned char)inf[IN_PHEROMONE], done[env] != 0,
                 reward, sh, rgb8, rs2);
}

// Explicit reset with reset randomisation: observation (and histograms) of the masked environments' new episodes
static __global__ void __launch_bounds__(RTHREADS) k_render_reset(RenderScene sc, ObsArgs o, const unsigned char* __restrict__ mask) {
  extern __shared__ __align__(16) unsigned char rsm[];
  TileShared& sh = *reinterpret_cast<TileShared*>(rsm);
  unsigned* rgb8 = reinterpret_cast<unsigned*>(rsm + sizeof(TileShared));
  float* rs2 = reinterpret_cast<float*>(rsm + sizeof(TileShared) + TILE * TILE * sizeof(unsigned));
  const int env = blockIdx.x, npix = o.W * o.H;
  if (mask && !mask[env]) return;
  const int v = o.object[env];
  build_reset_scene(o, env, v, rs2);
  render_and_pack(sc, o, rs2, v, o.obs + (size_t)env * o.C * npix, o.reset_pad0[v], o.reset_pad1[v], sh, rgb8);
  if (o.hist_prev) for (int i = threadIdx.x; i < 512; i += RTHREADS) o.hist_prev[(size_t)env * 512 + i] = (float)(&sh.hist[0][0])[i];
}

constexpr size_t render_smem_bytes() { return sizeof(TileShared) + TILE * TILE * sizeof(unsigned); }
constexpr size_t render_phase_smem_bytes() { return render_smem_bytes() + RS_STRIDE * sizeof(float); }

// Observation phase of the fused step kernel (env_lockstep.cuh).  A block whose physics work is exhausted turns into an
// observation builder: it takes tickets from a global counter and renders environments in the order in which their
// agent steps finished (s.done_list, published by env_writeback with release semantics), so the rasteriser runs on SMs
// that would otherwise idle while the longest substep chains of the batch complete.  Requires blockDim.x == RTHREADS and
// every block of the grid resident (persistent grid), which the launch code guarantees.  Inputs written by other SMs
// during this same kernel are read through L2 (ld.cg): L1 is not coherent.  sm_busy: see below.
__device__ __forceinline__ void render_phase(const RenderScene& sc, const ObsArgs& o, const SimBuffers& s, unsigned char* smem, int* sm_busy) {
  TileShared& sh = *reinterpret_cast<TileShared*>(smem);
  unsigned* rgb8 = reinterpret_cast<unsigned*>(smem + sizeof(TileShared));
  float* rs = reinterpret_cast<float*>(smem + sizeof(TileShared) + TILE * TILE * sizeof(unsigned));
  __shared__ int cur_env;
  const int tid = threadIdx.x;
  for (;;) {
    __syncthreads();
    if (tid == 0) {
      // yield to a sibling block of this SM that is still integrating substeps: the kernel's duration is the longest substep
      // chain, and rasterising next to it would slow exactly that chain (sm_busy is only meaningful to thread 0's SM)
      while (*reinterpret_cast<volatile int*>(sm_busy) > 0) __nanosleep(2000);
      // Spinning on a ticket is only safe when the environment behind it is being integrated by a RESIDENT block.  The launch
      // sizes the grid to what fits, but should a block still be waiting for an SM (GPU shared with another context), take
      // only tickets whose environment has already finished, and leave when there is none: the late blocks render the rest.
      int ticket;
      if (*reinterpret_cast<volatile int*>(s.queue + 6) >= (int)gridDim.x) {
        ticket = atomicAdd(s.queue + 4, 1);
      } else {
        for (;;) {
          ticket = *reinterpret_cast<volatile int*>(s.queue + 4);
          if (ticket >= *reinterpret_cast<volatile int*>(s.queue + 3)) { ticket = s.n; break; }
          if (atomicCAS(s.queue + 4, ticket, ticket + 1) == ticket) break;
        }
      }
      int env = -1;
      if (ticket < s.n) {
        volatile int* slot = s.done_list + ticket;
        while ((env = *slot) < 0) __nanosleep(200);
        __threadfence();
      }
      cur_env = env;
    }
    __syncthreads();
    const int env = cur_env;
    if (env < 0) break;
    if (tid < RS_STRIDE) rs[tid] = __ldcg(s.render_state + (size_t)env * RS_STRIDE + tid);
    const float* inf = s.info + (size_t)env * IN_STRIDE;
    const unsigned char pad0 = (unsigned char)__ldcg(inf + IN_GRASP), pad1 = (unsigned char)__ldcg(inf + IN_PHEROMONE);
    const int v = (int)__ldcg(inf + IN_OBJECT);
    const bool is_done = __ldcg(s.done + env) != 0;
    __syncthreads();
    render_obs_env(sc, o, rs, v, env, pad0, pad1, is_done, s.reward, sh, rgb8, rs);  // rs is dead once the terminal image is packed
  }
}

// obs == reset image path: done = NULL, n = 1, hist_prev = NULL -> histograms go to hist_reset
inline void launch_render_obs(const RenderScene& sc, const ObsArgs& o, const float* render_state, const float* info, const unsigned char* done, float* reward, int n,
                              cudaStream_t st) {
  static bool attr_dev[64] = {};
  int dev_ = 0;
  cudaGetDevice(&dev_);
  bool& attr = attr_dev[dev_ & 63];  // the attribute is per device: a second simulator on another GPU of this process needs it too
  if (!attr) {
    if (cudaFuncSetAttribute(k_render_obs, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)render_phase_smem_bytes()) != cudaSuccess) throw std::runtime_error("cudaFuncSetAttribute(k_render_obs)");
    if (cudaFuncSetAttribute(k_render_reset, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)render_phase_smem_bytes()) != cudaSuccess) throw std::runtime_error("cudaFuncSetAttribute(k_render_reset)");
    if (cudaFuncSetAttribute(k_render_obs_indexed, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)render_phase_smem_bytes()) != cudaSuccess) throw std::runtime_error("cudaFuncSetAttribute(k_render_obs_indexed)");
    attr = true;
  }
  k_render_obs<<<n, RTHREADS, render_phase_smem_bytes(), st>>>(sc, o, render_state, info, IN_STRIDE, done, reward);
  if (cudaGetLastError() != cudaSuccess) throw std::runtime_error("k_render_obs launch failed");
}

inline void launch_render_reset(const RenderScene& sc, const ObsArgs& o, const unsigned char* mask, int n, cudaStream_t st) {
  k_render_reset<<<n, RTHREADS, render_phase_smem_bytes(), st>>>(sc, o, mask);
  if (cudaGetLastError() != cudaSuccess) throw std::runtime_error("k_render_reset launch failed");
}

// reset path: copy the constant reset image of each masked environment's variant (and its histograms) into it
static __global__ void k_copy_reset_obs(unsigned char* __restrict__ obs, const unsigned char* __restrict__ reset_obs, float* __restrict__ hist, const float* __restrict__ hist_reset,
                                 const int* __restrict__ object, const unsigned char* __restrict__ mask, int bytes) {
  const int env = blockIdx.x;
  if (mask && !mask[env]) return;
  const int v = object[env];
  for (int i = threadIdx.x; i < bytes; i += blockDim.x) obs[(size_t)env * bytes + i] = reset_obs[(size_t)v * bytes + i];
  for (int i = threadIdx.x; i < 512; i += blockDim.x) hist[(size_t)env * 512 + i] = hist_reset[(size_t)v * 512 + i];
}
inline void launch_copy_reset_obs(unsigned char* obs, const unsigned char* reset_obs, float* hist, const float* hist_reset, const int* object, const unsigned char* mask, int n,
                                  int bytes, cudaStream_t st) {
  k_copy_reset_obs<<<n, 256, 0, st>>>(obs, reset_obs, hist, hist_reset, object, mask, bytes);
  if (cudaGetLastError() != cudaSuccess) throw std::runtime_error("k_copy_reset_obs launch failed");
}

// RobotEnv.render / physics.render for any camera and size: rgb u8[n][h][w][3], depth f32[n][h][w] in metres; grid (tiles, n)
static __global__ void __launch_bounds__(RTHREADS) k_render_raw(RenderScene sc, const float* __restrict__ render_state, int rs_stride, const int* __restrict__ object,
                                                        unsigned char* __restrict__ rgb, float* __restrict__ depth, int H, int W, float fovy) {
  extern __shared__ __align__(16) unsigned char rsm[];
  TileShared& sh = *reinterpret_cast<TileShared*>(rsm);
  unsigned* rgb8 = reinterpret_cast<unsigned*>(rsm + sizeof(TileShared));
  const int env = blockIdx.y, tiles_x = (W + TILE - 1) / TILE;
  const int tx0 = (blockIdx.x % tiles_x) * TILE, ty0 = (blockIdx.x / tiles_x) * TILE;
  const int tw = min(TILE, W - tx0), th = min(TILE, H - ty0);
  render_tile(sc, render_state + (size_t)env * rs_stride, object[env], sh, rgb8, W, H, tx0, ty0, tw, th, fovy);
  for (int i = threadIdx.x; i < tw * th; i += RTHREADS) {
    int ly = i / tw, lx = i - ly * tw;
    size_t o = ((size_t)env * H + ty0 + ly) * W + tx0 + lx;
    unsigned c = rgb8[ly * TILE + lx];
    if (rgb) { rgb[3 * o] = c & 255; rgb[3 * o + 1] = (c >> 8) & 255; rgb[3 * o + 2] = (c >> 16) & 255; }
    if (depth) depth[o] = __uint_as_float((unsigned)sh.zbuf[ly * TILE + lx]);
  }
}
inline void launch_render_raw(const RenderScene& sc, const float* render_state, int rs_stride, const int* object, unsigned char* rgb, float* depth, int n, int H, int W,
                              double fovy, cudaStream_t st) {
  static bool attr_dev[64] = {};
  int dev_ = 0;
  cudaGetDevice(&dev_);
  bool& attr = attr_dev[dev_ & 63];
  if (!attr) {
    if (cudaFuncSetAttribute(k_render_raw, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)render_smem_bytes()) != cudaSuccess) throw std::runtime_error("cudaFuncSetAttribute(k_render_raw)");
    attr = true;
  }
  dim3 grid(((W + TILE - 1) / TILE) * ((H + TILE - 1) / TILE), n);
  k_render_raw<<<grid, RTHREADS, render_smem_bytes(), st>>>(sc, render_state, rs_stride, object, rgb, depth, H, W, fovy);
  if (cudaGetLastError() != cudaSuccess) throw std::runtime_error("k_render_raw launch failed");
}

}  // namespace grs
