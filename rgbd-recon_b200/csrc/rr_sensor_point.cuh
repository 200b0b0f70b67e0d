// A depth pixel lifted to the world: the view-independent half of ReconPoints' vertex stage (points.vs:24-37, the bbox /
// depth cull of points.gs:39-41 and the colour-view border cut of points.fs:38-41). rr_draw_points (rr_points.cu) continues
// from here with the view transform; the point-cloud export (rr_cloud.cu) writes what it returns, so both keep exactly the
// same set of pixels.
#pragma once
#include "rr_context.h"
#include "rr_math.cuh"

namespace rr {

// id = layer * W * H + y * W + x. pos_cs: the trilinear cv_xyz of the layer at (sx, sy, depth_b.x); texcoord: the trilinear
// cv_uv there (written only when the point passed the bbox / depth cull). Returns whether the point is kept.
__device__ __forceinline__ bool sensor_point(const SensorTables& st, const float2* depth_b, int W, int H, const float* bmin,
                                             const float* bmax, uint32_t id, float3& pos_cs, float2& texcoord) {
  const uint32_t px = (uint32_t)(W * H);
  const int layer = (int)(id / px), r = (int)(id - (uint32_t)layer * px), y = r / W, x = r - y * W;
  // the vertex buffer (recon_points.cpp:46-52): (x + 0.5) * stepX in double, rounded to float
  const float stepX = 1.0f / (float)W, stepY = 1.0f / (float)H;
  const float sx = (float)(((double)x + 0.5) * (double)stepX), sy = (float)(((double)y + 0.5) * (double)stepY);
  const float depth = __ldg(depth_b + (size_t)layer * px + (size_t)y * W + x).x;        // a texel centre: the texel itself
  pos_cs = tex3d_xyz(st.xyz[layer], st.cx[layer], st.cy[layer], st.cz[layer], sx, sy, depth);
  const bool in_box = pos_cs.x >= bmin[0] && pos_cs.y >= bmin[1] && pos_cs.z >= bmin[2] &&
                      pos_cs.x <= bmax[0] && pos_cs.y <= bmax[1] && pos_cs.z <= bmax[2];
  if (!in_box || depth <= 0.0f) return false;
  const float zc = depth;
  texcoord = tex3d_uv(st.uv[layer], st.cx[layer], st.cy[layer], st.cz[layer], sx, sy, zc);
  // points.fs:38-41: the border of the colour camera's view is cut away (a flat attribute: the whole point goes)
  if (texcoord.x > 0.99f || texcoord.x < 0.01f || texcoord.y > 0.99f || texcoord.y < 0.01f) return false;
  return true;
}

}  // namespace rr
