// ORACLE (test infrastructure, NOT product code). The reference ships no tests; the march, shading and colour blending are pinned
// against the reference's own glsl/tsdf_raymarch.fs + shading.glsl compiled as C++ and run on the CPU (oracle/glsl_host/,
// tests/golden/ref_glsl_raymarch.npz), including the skipSpace branch on depth peels as a rasteriser leaves them
// (oracle/ref_glsl_py.py::depth_peels).
// Scalar restatement of the TSDF raymarcher: ReconIntegration::draw / drawDepthLimits
// (framework/reconstruction/recon_integration.cpp:177-241, 409-429), glsl/tsdf_raymarch.{vs,fs}, glsl/shading.glsl,
// glsl/bricks.{vs,gs,fs}.
//
// Rasterisation -> rays (SURVEY.md §7 "hard parts"): the reference rasterises a unit-cube proxy and, for space
// skipping, the occupied bricks' faces with GL_MIN blending. Here both are analytic per pixel:
//   * a pixel has a fragment iff its ray (through the pixel centre) hits the unit cube [0,1]^3 in volume space;
//   * the ray direction is normalize(P_far - CameraPos) with P_far = screenToVol(frag.xy, 1.0) — any point of the
//     rasterised cube on that pixel's ray gives the same direction up to rounding;
//   * skipSpace: start/end = nearest entry / farthest exit of the ray through the union of occupied bricks (drawn as
//     full brick_size cubes, bricks.vs:19), entry clamped to the camera (front face culled: tsdf_raymarch.fs:395).
// Matrix inverses that the reference evaluates with glm / gloost in float are evaluated in double from the float
// inputs and rounded once (inverse4 below); matrix*vector products are fma chains.
#include "ro_math.h"
#include "ro_sample.h"
#include "rr_oracle.h"

#include <cmath>
#include <vector>

using namespace ro;

namespace {

// column-major 4x4, m[c*4+r]
struct M4 { float m[16]; };
struct M4d { double m[16]; };

// adjugate / determinant, the expansion of Mesa's gluInvertMatrix (public algorithm), in double
bool inverse4(const double* m, double* out) {
  double inv[16];
  inv[0] = m[5] * m[10] * m[15] - m[5] * m[11] * m[14] - m[9] * m[6] * m[15] + m[9] * m[7] * m[14] + m[13] * m[6] * m[11] - m[13] * m[7] * m[10];
  inv[4] = -m[4] * m[10] * m[15] + m[4] * m[11] * m[14] + m[8] * m[6] * m[15] - m[8] * m[7] * m[14] - m[12] * m[6] * m[11] + m[12] * m[7] * m[10];
  inv[8] = m[4] * m[9] * m[15] - m[4] * m[11] * m[13] - m[8] * m[5] * m[15] + m[8] * m[7] * m[13] + m[12] * m[5] * m[11] - m[12] * m[7] * m[9];
  inv[12] = -m[4] * m[9] * m[14] + m[4] * m[10] * m[13] + m[8] * m[5] * m[14] - m[8] * m[6] * m[13] - m[12] * m[5] * m[10] + m[12] * m[6] * m[9];
  inv[1] = -m[1] * m[10] * m[15] + m[1] * m[11] * m[14] + m[9] * m[2] * m[15] - m[9] * m[3] * m[14] - m[13] * m[2] * m[11] + m[13] * m[3] * m[10];
  inv[5] = m[0] * m[10] * m[15] - m[0] * m[11] * m[14] - m[8] * m[2] * m[15] + m[8] * m[3] * m[14] + m[12] * m[2] * m[11] - m[12] * m[3] * m[10];
  inv[9] = -m[0] * m[9] * m[15] + m[0] * m[11] * m[13] + m[8] * m[1] * m[15] - m[8] * m[3] * m[13] - m[12] * m[1] * m[11] + m[12] * m[3] * m[9];
  inv[13] = m[0] * m[9] * m[14] - m[0] * m[10] * m[13] - m[8] * m[1] * m[14] + m[8] * m[2] * m[13] + m[12] * m[1] * m[10] - m[12] * m[2] * m[9];
  inv[2] = m[1] * m[6] * m[15] - m[1] * m[7] * m[14] - m[5] * m[2] * m[15] + m[5] * m[3] * m[14] + m[13] * m[2] * m[7] - m[13] * m[3] * m[6];
  inv[6] = -m[0] * m[6] * m[15] + m[0] * m[7] * m[14] + m[4] * m[2] * m[15] - m[4] * m[3] * m[14] - m[12] * m[2] * m[7] + m[12] * m[3] * m[6];
  inv[10] = m[0] * m[5] * m[15] - m[0] * m[7] * m[13] - m[4] * m[1] * m[15] + m[4] * m[3] * m[13] + m[12] * m[1] * m[7] - m[12] * m[3] * m[5];
  inv[14] = -m[0] * m[5] * m[14] + m[0] * m[6] * m[13] + m[4] * m[1] * m[14] - m[4] * m[2] * m[13] - m[12] * m[1] * m[6] + m[12] * m[2] * m[5];
  inv[3] = -m[1] * m[6] * m[11] + m[1] * m[7] * m[10] + m[5] * m[2] * m[11] - m[5] * m[3] * m[10] - m[9] * m[2] * m[7] + m[9] * m[3] * m[6];
  inv[7] = m[0] * m[6] * m[11] - m[0] * m[7] * m[10] - m[4] * m[2] * m[11] + m[4] * m[3] * m[10] + m[8] * m[2] * m[7] - m[8] * m[3] * m[6];
  inv[11] = -m[0] * m[5] * m[11] + m[0] * m[7] * m[9] + m[4] * m[1] * m[11] - m[4] * m[3] * m[9] - m[8] * m[1] * m[7] + m[8] * m[3] * m[5];
  inv[15] = m[0] * m[5] * m[10] - m[0] * m[6] * m[9] - m[4] * m[1] * m[10] + m[4] * m[2] * m[9] + m[8] * m[1] * m[6] - m[8] * m[2] * m[5];
  double det = m[0] * inv[0] + m[1] * inv[4] + m[2] * inv[8] + m[3] * inv[12];
  if (det == 0.0) return false;
  det = 1.0 / det;
  for (int i = 0; i < 16; ++i) out[i] = inv[i] * det;
  return true;
}

void mul4d(const double* a, const double* b, double* out) {   // out = a * b
  for (int c = 0; c < 4; ++c)
    for (int r = 0; r < 4; ++r) {
      double acc = 0.0;
      for (int k = 0; k < 4; ++k) acc += a[k * 4 + r] * b[c * 4 + k];
      out[c * 4 + r] = acc;
    }
}

inline V4 mulv(const M4& a, V4 v) {
  V4 o;
  o.x = fmaf(a.m[12], v.w, fmaf(a.m[8], v.z, fmaf(a.m[4], v.y, a.m[0] * v.x)));
  o.y = fmaf(a.m[13], v.w, fmaf(a.m[9], v.z, fmaf(a.m[5], v.y, a.m[1] * v.x)));
  o.z = fmaf(a.m[14], v.w, fmaf(a.m[10], v.z, fmaf(a.m[6], v.y, a.m[2] * v.x)));
  o.w = fmaf(a.m[15], v.w, fmaf(a.m[11], v.z, fmaf(a.m[7], v.y, a.m[3] * v.x)));
  return o;
}

struct Frame {
  M4 img_to_eye, inv_mv, inv_v2w, mv_v2w, normal_matrix;
  float mvT3[9];       // transpose of modelview's upper 3x3 (shade mode 2: inverse(gl_NormalMatrix))
  V3 camera_pos;       // volume space
  float proj22, proj32;
};

Frame derive(const float* mv, const float* proj, const float* bmin, const float* bmax, int vw, int vh) {
  Frame f{};
  double MV[16], P[16], V[16] = {0}, t[16], t2[16], inv[16];
  for (int i = 0; i < 16; ++i) { MV[i] = mv[i]; P[i] = proj[i]; }
  const float dx = bmax[0] - bmin[0], dy = bmax[1] - bmin[1], dz = bmax[2] - bmin[2];
  V[0] = dx; V[5] = dy; V[10] = dz; V[12] = bmin[0]; V[13] = bmin[1]; V[14] = bmin[2]; V[15] = 1.0;
  // image_to_eye = inverse(viewport_scale * viewport_translate * projection)  (recon_integration.cpp:183-194)
  double Tr[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 1, 1, 1, 1};
  double Sc[16] = {vw * 0.5, 0, 0, 0, 0, vh * 0.5, 0, 0, 0, 0, 0.5, 0, 0, 0, 0, 1};
  mul4d(Tr, P, t); mul4d(Sc, t, t2);
  inverse4(t2, inv);
  for (int i = 0; i < 16; ++i) f.img_to_eye.m[i] = (float)inv[i];
  inverse4(MV, inv);
  for (int i = 0; i < 16; ++i) f.inv_mv.m[i] = (float)inv[i];
  inverse4(V, inv);
  for (int i = 0; i < 16; ++i) f.inv_v2w.m[i] = (float)inv[i];
  mul4d(MV, V, t);
  for (int i = 0; i < 16; ++i) f.mv_v2w.m[i] = (float)t[i];
  inverse4(t, inv);   // NormalMatrix = inverseTranspose(model_view * vol_to_world)
  for (int c = 0; c < 4; ++c) for (int r = 0; r < 4; ++r) f.normal_matrix.m[c * 4 + r] = (float)inv[r * 4 + c];
  for (int c = 0; c < 3; ++c) for (int r = 0; r < 3; ++r) f.mvT3[c * 3 + r] = mv[r * 4 + c];
  V4 cam_world{f.inv_mv.m[12], f.inv_mv.m[13], f.inv_mv.m[14], f.inv_mv.m[15]};
  V4 cam_vol = mulv(f.inv_v2w, cam_world);
  f.camera_pos = V3{cam_vol.x, cam_vol.y, cam_vol.z};
  f.proj22 = proj[10]; f.proj32 = proj[14];
  return f;
}

// shading.glsl:24-30
const float kCameraColors[5][3] = {{228.f / 255.f, 26.f / 255.f, 28.f / 255.f}, {55.f / 255.f, 126.f / 255.f, 184.f / 255.f},
                                   {77.f / 255.f, 175.f / 255.f, 74.f / 255.f}, {152.f / 255.f, 78.f / 255.f, 163.f / 255.f},
                                   {255.f / 255.f, 127.f / 255.f, 0.f / 255.f}};

// tsdf_raymarch.fs:354-369 with getWeights :159-174
inline V3 blend_cameras(const RM& r, V3 p) {
  V3 tc{0, 0, 0};
  float tw = 0.0f;
  const size_t inv_stride = (size_t)r.IX * r.IY * r.IZ * 4;
  const size_t img = (size_t)r.W * r.H;
  for (int i = 0; i < r.N; ++i) {
    float pc[3];
    tex3d_linear<4>(r.inv + inv_stride * i, r.IX, r.IY, r.IZ, p.x, p.y, p.z, pc, 3);
    float depth = tex2d_nearest(r.depth_b + img * 2 * i, r.W, r.H, 2, 0, pc[0], pc[1]);
    float quality = 0.0f;
    if (fabsf(depth - pc[2]) < r.limit) quality = tex2d_linear(r.quality + img * i, r.W, r.H, 1, 0, pc[0], pc[1]);
    const float* cc = kCameraColors[i < 5 ? i : 4];
    tc.x = fmaf(cc[0], quality, tc.x); tc.y = fmaf(cc[1], quality, tc.y); tc.z = fmaf(cc[2], quality, tc.z);
    tw += quality;
  }
  tc = tc / tw;
  if (tw <= 0.0f) tc = V3{1.0f, 1.0f, 1.0f};
  return tc;
}

// shading.glsl:32-69
inline V3 shade(const RM& r, const Frame& f, V3 view_pos, V3 view_normal, V3 diffuse) {
  if (r.shade_mode == 0) return diffuse;
  if (r.shade_mode == 1) {
    const V3 light_pos{1.5f, 1.0f, 1.0f}, light_diffuse{1.0f, 0.9f, 0.7f};
    const V3 light_ambient = light_diffuse * 0.2f;
    const float ks = 0.5f, n = 20.0f;
    float diff = 0.0f, spec = 0.0f;
    V3 to_light = normalize3(light_pos - view_pos);
    float light_angle = dot3(view_normal, to_light);
    if (!(light_angle <= 0.0f)) {
      diff = gl_max(light_angle, 0.0f);
      V3 to_viewer = normalize3(V3{-view_pos.x, -view_pos.y, -view_pos.z});
      V3 halfway = normalize3(to_light + to_viewer);
      float reflected = dot3(halfway, view_normal);
      spec = gl_pow(reflected, n);
      float a = (1.0f - light_angle) * (1.0f - light_angle);
      spec *= 1.0f - a * a * a;
    }
    const V3 solid{0.5f, 0.5f, 0.5f};
    V3 amb = light_ambient * solid;
    V3 dif = (light_diffuse * solid) * diff;
    float sp = (1.0f * ks) * spec;
    return V3{(amb.x + dif.x) + sp, (amb.y + dif.y) + sp, (amb.z + dif.z) + sp};
  }
  if (r.shade_mode == 2) {
    const float* t = f.mvT3;   // (inverse(gl_NormalMatrix) * vec4(n, 0)).xyz = transpose(mat3(modelview)) * n
    return V3{fmaf(t[6], view_normal.z, fmaf(t[3], view_normal.y, t[0] * view_normal.x)),
              fmaf(t[7], view_normal.z, fmaf(t[4], view_normal.y, t[1] * view_normal.x)),
              fmaf(t[8], view_normal.z, fmaf(t[5], view_normal.y, t[2] * view_normal.x))};
  }
  return V3{1.0f, 1.0f, 1.0f};
}

inline bool slab(V3 o, V3 invd, V3 lo, V3 hi, float& t0, float& t1) {
  const float ax = (lo.x - o.x) * invd.x, bx = (hi.x - o.x) * invd.x;
  const float ay = (lo.y - o.y) * invd.y, by = (hi.y - o.y) * invd.y;
  const float az = (lo.z - o.z) * invd.z, bz = (hi.z - o.z) * invd.z;
  t0 = gl_max(gl_max(gl_min(ax, bx), gl_min(ay, by)), gl_min(az, bz));
  t1 = gl_min(gl_min(gl_max(ax, bx), gl_max(ay, by)), gl_max(az, bz));
  return t0 <= t1;
}

}  // namespace

extern "C" {

// Derived per-frame uniforms, for tests of the host-side matrix code: out = img_to_eye[16], inv_mv[16], inv_v2w[16],
// mv_v2w[16], normal_matrix[16], camera_pos[3]  (83 floats).
void ro_raymarch_uniforms(const float* mv, const float* proj, const float* bmin, const float* bmax, int vw, int vh, float* out) {
  Frame f = derive(mv, proj, bmin, bmax, vw, vh);
  const M4* ms[5] = {&f.img_to_eye, &f.inv_mv, &f.inv_v2w, &f.mv_v2w, &f.normal_matrix};
  for (int k = 0; k < 5; ++k) for (int i = 0; i < 16; ++i) out[k * 16 + i] = ms[k]->m[i];
  out[80] = f.camera_pos.x; out[81] = f.camera_pos.y; out[82] = f.camera_pos.z;
}

// Per pixel: the point screenToVol(vec3(frag.xy, 1.0)) the march aims at (any point of the pixel's ray serves as the
// cube fragment's pass_Position) and whether the ray meets the unit cube in front of the camera, i.e. whether the cube
// proxy produces a fragment there. Used to drive the reference's own tsdf_raymarch.fs on the CPU (oracle/glsl_host).
void ro_raymarch_rays(const float* modelview, const float* projection, const float* bbox_min, const float* bbox_max, int vw, int vh,
                      float limit, float* out_points, uint8_t* out_covered) {
  const Frame f = derive(modelview, projection, bbox_min, bbox_max, vw, vh);
  const float sd = limit * 0.5f;
  for (int py = 0; py < vh; ++py)
    for (int px = 0; px < vw; ++px) {
      const size_t o = (size_t)py * vw + px;
      V4 pc = mulv(f.img_to_eye, V4{(float)px + 0.5f, (float)py + 0.5f, 1.0f, 1.0f});
      V4 es{pc.x / pc.w, pc.y / pc.w, pc.z / pc.w, 1.0f};
      V4 ws = mulv(f.inv_mv, es);
      V4 pv = mulv(f.inv_v2w, ws);
      out_points[o * 3] = pv.x; out_points[o * 3 + 1] = pv.y; out_points[o * 3 + 2] = pv.z;
      const V3 cam = f.camera_pos;
      const V3 step = normalize3(V3{pv.x, pv.y, pv.z} - cam) * sd;
      const V3 invs{1.0f / step.x, 1.0f / step.y, 1.0f / step.z};
      float c0, c1;
      out_covered[o] = (slab(cam, invs, V3{0, 0, 0}, V3{1, 1, 1}, c0, c1) && !(c1 < 0.0f)) ? 1 : 0;
    }
}

void ro_raymarch(const float* tsdf, const uint32_t* res, float limit, int N, const float* inv, const int32_t* inv_res,
                 const float* cv_uv, const int32_t* cv_res, const uint8_t* color, int CW, int CH,
                 const float* depth_b, const float* quality, int W, int H, const float* bbox_min, const float* bbox_max,
                 const float* modelview, const float* projection, int vw, int vh, int shade_mode, int skip_space,
                 const uint32_t* occupied, uint32_t n_occ, const uint32_t* brick_res, float brick_size,
                 float* out_rgba, float* out_depth, float* out_samples, float* out_pos) {
  RM r{tsdf, (int)res[0], (int)res[1], (int)res[2], limit, N, inv, inv_res[0], inv_res[1], inv_res[2],
       cv_uv, cv_res[0], cv_res[1], cv_res[2], color, CW, CH, depth_b, quality, W, H, shade_mode};
  const Frame f = derive(modelview, projection, bbox_min, bbox_max, vw, vh);
  const float sd = limit * 0.5f;
  const V3 dims{bbox_max[0] - bbox_min[0], bbox_max[1] - bbox_min[1], bbox_max[2] - bbox_min[2]};
  std::vector<V3> blo(n_occ), bhi(n_occ);
  for (uint32_t b = 0; b < n_occ; ++b) {
    uint32_t id = occupied[b];
    uint32_t iz = id / (brick_res[0] * brick_res[1]); id %= (brick_res[0] * brick_res[1]);
    uint32_t iy = id / brick_res[0], ix = id % brick_res[0];
    blo[b] = V3{((float)ix * brick_size) / dims.x, ((float)iy * brick_size) / dims.y, ((float)iz * brick_size) / dims.z};
    bhi[b] = V3{((float)(ix + 1) * brick_size) / dims.x, ((float)(iy + 1) * brick_size) / dims.y, ((float)(iz + 1) * brick_size) / dims.z};
  }
#pragma omp parallel for schedule(dynamic, 4)
  for (int py = 0; py < vh; ++py) {
    for (int px = 0; px < vw; ++px) {
      const size_t o = (size_t)py * vw + px;
      out_rgba[o * 4] = out_rgba[o * 4 + 1] = out_rgba[o * 4 + 2] = out_rgba[o * 4 + 3] = 0.0f;
      out_depth[o] = 1.0f;
      out_samples[o] = 0.0f;
      if (out_pos) out_pos[o * 3] = out_pos[o * 3 + 1] = out_pos[o * 3 + 2] = 0.0f;
      // screenToVol(vec3(frag.xy, 1.0))  (tsdf_raymarch.fs:384-390)
      V4 pc = mulv(f.img_to_eye, V4{(float)px + 0.5f, (float)py + 0.5f, 1.0f, 1.0f});
      V4 es{pc.x / pc.w, pc.y / pc.w, pc.z / pc.w, 1.0f};
      V4 ws = mulv(f.inv_mv, es);
      V4 pv = mulv(f.inv_v2w, ws);
      const V3 cam = f.camera_pos;
      const V3 dir = normalize3(V3{pv.x, pv.y, pv.z} - cam);
      const V3 step = dir * sd;
      const V3 invd{1.0f / dir.x, 1.0f / dir.y, 1.0f / dir.z};
      // the cube proxy: intersectBox(CameraPos, sampleStep) (tsdf_raymarch.fs:371-382), t in units of sampleStep
      const V3 invs{1.0f / step.x, 1.0f / step.y, 1.0f / step.z};
      float c0, c1;
      if (!slab(cam, invs, V3{0, 0, 0}, V3{1, 1, 1}, c0, c1) || c1 < 0.0f) continue;   // no cube fragment on this pixel
      V3 sample_pos;
      uint32_t max_num_samples;
      if (skip_space) {
        float T0 = INFINITY, T1 = -INFINITY;
        for (uint32_t b = 0; b < n_occ; ++b) {
          float t0, t1;
          if (!slab(cam, invd, blo[b], bhi[b], t0, t1) || t1 < 0.0f) continue;
          T0 = gl_min(T0, gl_max(t0, 0.0f));
          T1 = gl_max(T1, t1);
        }
        if (!(T0 <= T1)) continue;                                                     // no brick on the ray: zero-length march
        sample_pos = cam + dir * T0;
        max_num_samples = f2u_sat(ceilf((T1 - T0) / sd));
      } else {
        const float t_near = (c0 < 0.0f) ? 0.0f : c0;
        sample_pos = cam + step * t_near;
        max_num_samples = f2u_sat(ceilf(fabsf(c1 - t_near)));
      }
      float prev_density = -limit;
      uint32_t num_samples = 0;
      bool hit = false;
      while (num_samples < max_num_samples) {
        num_samples += 1;
        const float density = sample_tsdf(r, sample_pos);
        if (density > 0.0f) {
          const float ratio = prev_density / (density - prev_density);
          sample_pos = (sample_pos - step) - step * ratio;
          hit = true;
          break;
        }
        prev_density = density;
        sample_pos = sample_pos + step;
      }
      out_samples[o] = (float)num_samples * 0.0027f;
      if (!hit) continue;
      // submitFragment (tsdf_raymarch.fs:116-142)
      V3 grad = get_gradient(r, sample_pos, sd);
      V4 vn4 = mulv(f.normal_matrix, V4{grad.x, grad.y, grad.z, 0.0f});
      V3 view_normal = normalize3(V3{vn4.x, vn4.y, vn4.z});
      V4 vp4 = mulv(f.mv_v2w, V4{sample_pos.x, sample_pos.y, sample_pos.z, 1.0f});
      V3 view_pos{vp4.x, vp4.y, vp4.z};
      V4 outc;
      if (shade_mode == 3) {
        V3 c = blend_cameras(r, sample_pos);
        outc = V4{c.x, c.y, c.z, 1.0f};
      } else {
        V4 diffuse = blend_colors(r, sample_pos);
        V3 c = shade(r, f, view_pos, view_normal, V3{diffuse.x, diffuse.y, diffuse.z});
        outc = V4{c.x, c.y, c.z, diffuse.w};
      }
      out_rgba[o * 4] = outc.x; out_rgba[o * 4 + 1] = outc.y; out_rgba[o * 4 + 2] = outc.z; out_rgba[o * 4 + 3] = outc.w;
      out_depth[o] = (f.proj22 * view_pos.z + f.proj32) / -view_pos.z * 0.5f + 0.5f;
      if (out_pos) { out_pos[o * 3] = sample_pos.x; out_pos[o * 3 + 1] = sample_pos.y; out_pos[o * 3 + 2] = sample_pos.z; }
    }
  }
}

}  // extern "C"
