// ORACLE (test infrastructure, NOT product code). Scalar restatement of the point-cloud export (rr_extract_points; contract
// in include/rgbd_recon_b200.h): the vertices ReconPoints::draw keeps before the view transform (recon_points.cpp:46-52
// vertex buffer, glsl/points.gs:39-41 bbox / depth cull, points.fs:38-41 colour-view border cut), in draw order, with the
// attributes at the pixel and the colour points.fs shades with. The lookups are ro_points.cpp's, through the same
// tex3d_linear (ro_math.h) and fetch_rgb8 (ro_draw.h).
#include "rr_oracle.h"

#include "ro_draw.h"
#include "ro_math.h"

#include <cstddef>

using namespace ro;

extern "C" {

void ro_extract_points(int N, int W, int H, const float* depth_b, const float* normal, const float* quality, const uint8_t* color,
                       int CW, int CH, const float* cv_xyz, const float* cv_uv, const int32_t* cv_res, const float* bmin,
                       const float* bmax, uint32_t sensor_mask, uint32_t* out_n, float* positions, float* normals, float* colors,
                       float* quality_out, uint32_t* pixels) {
  const int CX = cv_res[0], CY = cv_res[1], CZ = cv_res[2];
  const size_t cvn = (size_t)CX * CY * CZ, px = (size_t)W * H;
  const float stepX = 1.0f / (float)W, stepY = 1.0f / (float)H;
  size_t n = 0;
  for (int layer = 0; layer < N; ++layer) {
    if (!((sensor_mask >> layer) & 1u)) continue;
    for (int y = 0; y < H; ++y)
      for (int x = 0; x < W; ++x) {
        const size_t id = (size_t)layer * px + (size_t)y * W + x;
        const float sx = (float)(((double)x + 0.5) * (double)stepX), sy = (float)(((double)y + 0.5) * (double)stepY);
        const float depth = depth_b[id * 2];
        float pc[3], tc[2];
        tex3d_linear<3>(cv_xyz + (size_t)layer * cvn * 3, CX, CY, CZ, sx, sy, depth, pc, 3);
        const bool in_box = pc[0] >= bmin[0] && pc[1] >= bmin[1] && pc[2] >= bmin[2] && pc[0] <= bmax[0] && pc[1] <= bmax[1] && pc[2] <= bmax[2];
        if (!in_box || depth <= 0.0f) continue;                            // points.gs:39-41
        tex3d_linear<2>(cv_uv + (size_t)layer * cvn * 2, CX, CY, CZ, sx, sy, depth, tc, 2);
        if (tc[0] > 0.99f || tc[0] < 0.01f || tc[1] > 0.99f || tc[1] < 0.01f) continue;      // points.fs:38-41
        const V3 col = fetch_rgb8(color + (size_t)CW * CH * 3 * layer, CW, CH, tc[0], tc[1]);
        for (int a = 0; a < 3; ++a) {
          positions[n * 3 + a] = pc[a];
          normals[n * 3 + a] = normal[id * 3 + a];
        }
        colors[n * 3] = col.x; colors[n * 3 + 1] = col.y; colors[n * 3 + 2] = col.z;
        quality_out[n] = quality[id];
        pixels[n] = (uint32_t)id;
        ++n;
      }
  }
  *out_n = (uint32_t)n;
}

}  // extern "C"
