// ORACLE (test infrastructure, NOT product code): what the raymarch reads from the volume and the stage images at a point of
// volume space (tsdf_raymarch.fs:148-157 getGradient, :303-338 blendColors) for ro_mesh.cpp: the functions of ro_raymarch.cpp,
// restated word for word. The library shares one implementation between its raymarch and its mesh (csrc/rr_sample.cuh), and
// the GPU tests hold the raymarch to ro_raymarch.cpp and the mesh to ro_mesh.cpp, bit for bit, so the two oracle copies
// cannot drift apart without a test failing.
#ifndef RO_SAMPLE_H
#define RO_SAMPLE_H

#include "ro_math.h"

#include <cmath>
#include <cstddef>
#include <cstdint>

namespace {

using namespace ro;

struct RM {
  const float* tsdf; int X, Y, Z;
  float limit;
  int N; const float* inv; int IX, IY, IZ;
  const float* cv_uv; int CX, CY, CZ;
  const uint8_t* color; int CW, CH;
  const float* depth_b; const float* quality; int W, H;
  int shade_mode;
};

inline float sample_tsdf(const RM& r, V3 p) {
  int x0, x1, y0, y1, z0, z1; float a, b, g;
  lin_coord(p.x, r.X, x0, x1, a);
  lin_coord(p.y, r.Y, y0, y1, b);
  lin_coord(p.z, r.Z, z0, z1, g);
  const size_t sy = (size_t)r.X, sz = (size_t)r.X * r.Y;
  const float* T = r.tsdf;
  float c00 = lerpf(T[z0 * sz + y0 * sy + x0], T[z0 * sz + y0 * sy + x1], a);
  float c10 = lerpf(T[z0 * sz + y1 * sy + x0], T[z0 * sz + y1 * sy + x1], a);
  float c01 = lerpf(T[z1 * sz + y0 * sy + x0], T[z1 * sz + y0 * sy + x1], a);
  float c11 = lerpf(T[z1 * sz + y1 * sy + x0], T[z1 * sz + y1 * sy + x1], a);
  return lerpf(lerpf(c00, c10, b), lerpf(c01, c11, b), g);
}

// tsdf_raymarch.fs:148-157
inline V3 get_gradient(const RM& r, V3 p, float sd) {
  V3 gvec{sample_tsdf(r, V3{p.x + sd, p.y, p.z}) - sample_tsdf(r, V3{p.x - sd, p.y, p.z}),
          sample_tsdf(r, V3{p.x, p.y + sd, p.z}) - sample_tsdf(r, V3{p.x, p.y - sd, p.z}),
          sample_tsdf(r, V3{p.x, p.y, p.z + sd}) - sample_tsdf(r, V3{p.x, p.y, p.z - sd})};
  V3 n = normalize3(gvec);
  return V3{-n.x, -n.y, -n.z};
}

inline V3 fetch_rgb8(const uint8_t* img, int W, int H, float s, float t) {
  int x0, x1, y0, y1; float a, b;
  lin_coord(s, W, x0, x1, a);
  lin_coord(t, H, y0, y1, b);
  float o[3];
  for (int c = 0; c < 3; ++c) {
    float v00 = (float)img[((size_t)y0 * W + x0) * 3 + c] / 255.0f, v10 = (float)img[((size_t)y0 * W + x1) * 3 + c] / 255.0f;
    float v01 = (float)img[((size_t)y1 * W + x0) * 3 + c] / 255.0f, v11 = (float)img[((size_t)y1 * W + x1) * 3 + c] / 255.0f;
    o[c] = lerpf(lerpf(v00, v10, a), lerpf(v01, v11, a), b);
  }
  return {o[0], o[1], o[2]};
}

// tsdf_raymarch.fs:303-338
inline V4 blend_colors(const RM& r, V3 p) {
  V3 tc{0, 0, 0}, tc2{0, 0, 0};
  float tw = 0.0f, tw2 = 0.0f;
  const size_t inv_stride = (size_t)r.IX * r.IY * r.IZ * 4, uv_stride = (size_t)r.CX * r.CY * r.CZ * 2;
  const size_t img = (size_t)r.W * r.H;
  for (int i = 0; i < r.N; ++i) {
    float pc[3], uv[2];
    tex3d_linear<4>(r.inv + inv_stride * i, r.IX, r.IY, r.IZ, p.x, p.y, p.z, pc, 3);
    tex3d_linear<2>(r.cv_uv + uv_stride * i, r.CX, r.CY, r.CZ, pc[0], pc[1], pc[2], uv, 2);
    V3 col = fetch_rgb8(r.color + (size_t)r.CW * r.CH * 3 * i, r.CW, r.CH, uv[0], uv[1]);
    float depth = tex2d_nearest(r.depth_b + img * 2 * i, r.W, r.H, 2, 0, pc[0], pc[1]);
    float dist = fabsf(depth - pc[2]);
    float quality = 0.0f;
    if (dist < r.limit) quality = tex2d_linear(r.quality + img * i, r.W, r.H, 1, 0, pc[0], pc[1]);
    const float den = dist + 0.01f;
    tc = tc + (col * quality) / den;
    tw += quality / den;
    tc2 = tc2 + col / dist;
    tw2 += 1.0f / dist;
  }
  if (tw > 0.0f) { tc = tc / tw; return V4{tc.x, tc.y, tc.z, 1.0f}; }
  tc2 = tc2 / tw2;
  return V4{tc2.x, tc2.y, tc2.z, -1.0f};
}

}  // namespace

#endif
