// What the raymarcher reads from the volume and the stage images at a point q of volume (texture) space, shared by
// rr_raymarch.cu and rr_mesh.cu so that a mesh vertex and a raymarched pixel at the same q get the same numbers.
// P is the caller's parameter block; it provides
//   tsdf, X, Y, Z, half2                         the volume (R32F, or half2 voxels whose low half is the density)
//   limit, N, inv, IX, IY, IZ, uv[], cx[], cy[], cz[], color, CW, CH, depth_b, quality, W, H   (blend_colors only)
// to_volume and world_normal (the point-sample contract of rr_sample_points, shared by rr_query.cu and rr_simplify.cu) also
// read world (1: positions in metres), bmin[3] and dims[3] = bbox_max - bbox_min.
// Arithmetic as everywhere in the library: see rr_math.cuh.
#pragma once

#include "rr_math.cuh"

#include <cuda_fp16.h>

namespace rr {

// One voxel's density: R32F, or the low half of a half2 (tsdf, weight) voxel widened exactly (warp-uniform branch).
template <class P>
__device__ __forceinline__ float ld_density(const P& p, unsigned i) {
  if (p.half2) {
    const uint32_t u = __ldg(reinterpret_cast<const uint32_t*>(p.tsdf) + i);
    return __half2float(__ushort_as_half((unsigned short)(u & 0xffffu)));
  }
  return __ldg(p.tsdf + i);
}

template <class P>
__device__ __forceinline__ float sample_tsdf(const P& p, float3 q) {
  int x0, x1, y0, y1, z0, z1; float a, b, g;
  lin_coord(q.x, p.X, x0, x1, a);
  lin_coord(q.y, p.Y, y0, y1, b);
  lin_coord(q.z, p.Z, z0, z1, g);
  const unsigned sy = (unsigned)p.X, sz = (unsigned)(p.X * p.Y);
  const float c00 = lerpf(ld_density(p, z0 * sz + y0 * sy + x0), ld_density(p, z0 * sz + y0 * sy + x1), a);
  const float c10 = lerpf(ld_density(p, z0 * sz + y1 * sy + x0), ld_density(p, z0 * sz + y1 * sy + x1), a);
  const float c01 = lerpf(ld_density(p, z1 * sz + y0 * sy + x0), ld_density(p, z1 * sz + y0 * sy + x1), a);
  const float c11 = lerpf(ld_density(p, z1 * sz + y1 * sy + x0), ld_density(p, z1 * sz + y1 * sy + x1), a);
  return lerpf(lerpf(c00, c10, b), lerpf(c01, c11, b), g);
}

// tsdf_raymarch.fs:148-157 getGradient: central differences of sample_tsdf at +-sd, normalised and negated
template <class P>
__device__ __forceinline__ float3 get_gradient(const P& p, float3 q, float sd) {
  const float3 gv = make_float3(sample_tsdf(p, make_float3(q.x + sd, q.y, q.z)) - sample_tsdf(p, make_float3(q.x - sd, q.y, q.z)),
                                sample_tsdf(p, make_float3(q.x, q.y + sd, q.z)) - sample_tsdf(p, make_float3(q.x, q.y - sd, q.z)),
                                sample_tsdf(p, make_float3(q.x, q.y, q.z + sd)) - sample_tsdf(p, make_float3(q.x, q.y, q.z - sd)));
  const float3 gn = normalize3(gv);
  return make_float3(-gn.x, -gn.y, -gn.z);
}

__device__ __forceinline__ float tex_nearest_depth(const float2* img, int W, int H, float s, float t) {
  return __ldg(img + (size_t)near_coord(t, H) * W + near_coord(s, W)).x;
}

__device__ __forceinline__ float tex_linear_1(const float* img, int W, int H, float s, float t) {
  int x0, x1, y0, y1; float a, b;
  lin_coord(s, W, x0, x1, a);
  lin_coord(t, H, y0, y1, b);
  const float v00 = __ldg(img + (size_t)y0 * W + x0), v10 = __ldg(img + (size_t)y0 * W + x1);
  const float v01 = __ldg(img + (size_t)y1 * W + x0), v11 = __ldg(img + (size_t)y1 * W + x1);
  return lerpf(lerpf(v00, v10, a), lerpf(v01, v11, a), b);
}

// tsdf_raymarch.fs:303-338 blendColors: alpha 1 for the quality-weighted colour, -1 for the fallback blend
template <class P>
__device__ float4 blend_colors(const P& p, float3 q) {
  float3 tc = make_float3(0.f, 0.f, 0.f), tc2 = make_float3(0.f, 0.f, 0.f);
  float tw = 0.0f, tw2 = 0.0f;
  const size_t inv_stride = (size_t)p.IX * p.IY * p.IZ, img = (size_t)p.W * p.H;
  for (int i = 0; i < p.N; ++i) {
    const float3 pc = tex3d_xyz(p.inv + inv_stride * i, p.IX, p.IY, p.IZ, q.x, q.y, q.z);
    const float2 uv = tex3d_uv(p.uv[i], p.cx[i], p.cy[i], p.cz[i], pc.x, pc.y, pc.z);
    const float3 col = tex2d_rgb8(p.color + (size_t)p.CW * p.CH * 3 * i, p.CW, p.CH, uv.x, uv.y);
    const float depth = tex_nearest_depth(p.depth_b + img * i, p.W, p.H, pc.x, pc.y);
    const float dist = fabsf(depth - pc.z);
    float quality = 0.0f;
    if (dist < p.limit) quality = tex_linear_1(p.quality + img * i, p.W, p.H, pc.x, pc.y);
    const float den = dist + 0.01f;
    tc = tc + (col * quality) / den;
    tw += quality / den;
    tc2 = tc2 + col / dist;
    tw2 += 1.0f / dist;
  }
  if (tw > 0.0f) { tc = tc / tw; return make_float4(tc.x, tc.y, tc.z, 1.0f); }
  tc2 = tc2 / tw2;
  return make_float4(tc2.x, tc2.y, tc2.z, -1.0f);
}

// q = (p - bbox_min) / (bbox_max - bbox_min): one IEEE division per component (built with --fmad=false: no contraction)
template <class P>
__device__ __forceinline__ float3 to_volume(const P& p, float3 v) {
  if (!p.world) return v;
  return make_float3((v.x - p.bmin[0]) / p.dims[0], (v.y - p.bmin[1]) / p.dims[1], (v.z - p.bmin[2]) / p.dims[2]);
}

// the mesh vertex normal (rr_mesh.cu k_mesh_attributes): the raymarch's gradient, in world space
template <class P>
__device__ __forceinline__ float3 world_normal(const P& p, float3 q) {
  const float3 g = get_gradient(p, q, p.limit * 0.5f);
  return normalize3(make_float3(g.x / p.dims[0], g.y / p.dims[1], g.z / p.dims[2]));
}

__device__ __forceinline__ bool in_unit_cube(float3 q) {   // false for NaN
  return q.x >= 0.0f && q.x <= 1.0f && q.y >= 0.0f && q.y <= 1.0f && q.z >= 0.0f && q.z <= 1.0f;
}

}  // namespace rr
