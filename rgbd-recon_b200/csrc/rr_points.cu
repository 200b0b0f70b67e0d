// The other consumers of the pre-processed maps that draw POINTS (SURVEY.md §8f-4), for sm_100a without a rasteriser:
//   * ReconPoints::draw (framework/reconstruction/recon_points.cpp:71-111; glsl/points.vs, points.gs, points.fs): every depth
//     pixel of every sensor becomes a screen-aligned square of max_size / |pos_eye| pixels, coloured by shade() of the
//     sensor's colour / normal maps, depth-tested (GL_LESS);
//   * ReconCalibs::draw (recon_calibs.cpp:56-66; glsl/calib_vis.vs, calib_vis.fs) over VolumeSampler::sample
//     (rendering/volume_sampler.cpp:9-31,71-73): every voxel centre of the inverse-volume grid becomes a one-pixel point
//     coloured by the TSDF value there (red outside, green inside, blue at +limit, nothing at -limit).
// Two kernels: a splat pass (one thread per vertex: the vertex / geometry shader's arithmetic, clip test, window
// coordinates, then a 64-bit atomicMin of (depth bits << 32 | vertex id) over the pixels whose centres the square covers)
// and a resolve pass (one thread per view pixel: the winner's attributes are recomputed with the same device function and
// the fragment shader's arithmetic is applied). Draw order decides depth ties in GL (an equal depth fails GL_LESS);
// vertex ids ascend in draw order, so the smaller id wins the atomicMin exactly like the first drawn fragment.
// Rasterisation rule (OpenGL 4.4 §14.4.1, point sprites with program point size): a fragment for every pixel whose centre
// lies inside the square of side `size` centred at the point's window position, size clamped to the implementation's range
// (taken as [1, 256]); a point whose centre is outside the clip volume is culled (§13.5).
#include "rr_context.h"
#include "rr_draw.cuh"
#include "rr_math.cuh"
#include "rr_sensor_point.cuh"

#include <cuda_fp16.h>

#include <cmath>

namespace rr {

struct PointParams {
  float mv[16], proj[16], normal_matrix[16], v2w[16];
  float mvT3[9];
  int vw, vh, shade_mode, mode;            // mode 0: ReconPoints, 1: ReconCalibs
  int N, W, H, CW, CH;
  SensorTables st;
  const float2* depth_b; const float4* normal; const uint8_t* color;
  float bmin[3], bmax[3];
  // ReconCalibs
  int IX, IY, IZ;
  const float* tsdf; int X, Y, Z, half2;
  float limit;
  unsigned long long* keys;
  float4* out_rgba; float* out_depth;
};

// what the vertex and geometry stages hand to the rasteriser
struct PointVertex {
  bool alive;
  float xw, yw, zw, size;
  float3 pos_es;             // eye-space position (points) / unused (calibs)
  float2 texcoord;           // colour-image coordinate (points)
  float distance;            // TSDF value at the sample (calibs)
};

__device__ __forceinline__ float pdensity(const PointParams& p, unsigned i) {
  if (p.half2) {
    const uint32_t u = __ldg(reinterpret_cast<const uint32_t*>(p.tsdf) + i);
    return __half2float(__ushort_as_half((unsigned short)(u & 0xffffu)));
  }
  return __ldg(p.tsdf + i);
}
// texture(volume_tsdf, q).r: LINEAR + CLAMP_TO_EDGE, x -> y -> z lerps (the same filter as rr_raymarch.cu::sample_tsdf)
__device__ __forceinline__ float psample_tsdf(const PointParams& p, float3 q) {
  int x0, x1, y0, y1, z0, z1; float a, b, g;
  lin_coord(q.x, p.X, x0, x1, a);
  lin_coord(q.y, p.Y, y0, y1, b);
  lin_coord(q.z, p.Z, z0, z1, g);
  const unsigned sy = (unsigned)p.X, sz = (unsigned)(p.X * p.Y);
  const float c00 = lerpf(pdensity(p, z0 * sz + y0 * sy + x0), pdensity(p, z0 * sz + y0 * sy + x1), a);
  const float c10 = lerpf(pdensity(p, z0 * sz + y1 * sy + x0), pdensity(p, z0 * sz + y1 * sy + x1), a);
  const float c01 = lerpf(pdensity(p, z1 * sz + y0 * sy + x0), pdensity(p, z1 * sz + y0 * sy + x1), a);
  const float c11 = lerpf(pdensity(p, z1 * sz + y1 * sy + x0), pdensity(p, z1 * sz + y1 * sy + x1), a);
  return lerpf(lerpf(c00, c10, b), lerpf(c01, c11, b), g);
}

// clip test, perspective divide, viewport transform (OpenGL 4.4 §13.5, §13.6; depth range [0, 1])
__device__ __forceinline__ bool to_window(const PointParams& p, float4 clip, PointVertex& v) {
  if (!(clip.w > 0.0f) || !(fabsf(clip.x) <= clip.w) || !(fabsf(clip.y) <= clip.w) || !(fabsf(clip.z) <= clip.w)) return false;
  const float nx = clip.x / clip.w, ny = clip.y / clip.w, nz = clip.z / clip.w;
  v.xw = (nx * 0.5f + 0.5f) * (float)p.vw;
  v.yw = (ny * 0.5f + 0.5f) * (float)p.vh;
  v.zw = nz * 0.5f + 0.5f;
  return true;
}

__device__ PointVertex point_vertex(const PointParams& p, uint32_t id) {
  PointVertex v;
  v.alive = false; v.size = 1.0f; v.distance = 0.0f;
  v.pos_es = make_float3(0.f, 0.f, 0.f); v.texcoord = make_float2(0.f, 0.f);
  if (p.mode == 0) {
    // points.vs:24-37 + points.gs:39-60; the view-independent part (up to the border cut of points.fs:38-41) is rr_sensor_point.cuh
    float3 pos_cs;
    if (!sensor_point(p.st, p.depth_b, p.W, p.H, p.bmin, p.bmax, id, pos_cs, v.texcoord)) return v;
    const float4 es = pmulv(p.mv, make_float4(pos_cs.x, pos_cs.y, pos_cs.z, 1.0f));
    v.pos_es = make_float3(es.x, es.y, es.z);
    const float4 clip = pmulv(p.proj, es);
    if (!to_window(p, clip, v)) return v;
    const float dist = sqrtf(dot3(v.pos_es, v.pos_es));
    const float max_size = p.shade_mode == 3 ? 4.0f : 10.0f;
    v.size = gmin(gmax(max_size / dist, 1.0f), 256.0f);       // the implementation's point-size range, taken as [1, 256]
    v.alive = true;
    return v;
  }
  // calib_vis.vs:25-38 over VolumeSampler's voxel centres (volume_sampler.cpp:14-23)
  const uint32_t plane = (uint32_t)(p.IX * p.IY);
  const int z = (int)(id / plane), r = (int)(id - (uint32_t)z * plane), y = r / p.IX, x = r - y * p.IX;
  const float3 q = make_float3(((float)x + 0.5f) * (1.0f / (float)p.IX), ((float)y + 0.5f) * (1.0f / (float)p.IY), ((float)z + 0.5f) * (1.0f / (float)p.IZ));
  v.distance = psample_tsdf(p, q);
  if (v.distance <= -p.limit) return v;            // calib_vis.fs:29 discard (before anything is written)
  const float4 world = pmulv(p.v2w, make_float4(q.x, q.y, q.z, 1.0f));
  const float4 view = pmulv(p.mv, make_float4(world.x, world.y, world.z, 1.0f));
  const float4 clip = pmulv(p.proj, make_float4(view.x, view.y, view.z, 1.0f));
  if (!to_window(p, clip, v)) return v;
  v.alive = true;
  return v;
}

__global__ void __launch_bounds__(256) k_points_clear(unsigned long long* __restrict__ keys, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) keys[i] = ~0ull;
}

__global__ void __launch_bounds__(256) k_points_splat(const __grid_constant__ PointParams p, uint32_t n_vertices) {
  const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= n_vertices) return;
  const PointVertex v = point_vertex(p, id);
  if (!v.alive || !(v.zw < 1.0f)) return;           // GL_LESS against the cleared depth 1
  // pixels whose centres lie in [xw - size/2, xw + size/2) x [yw - size/2, yw + size/2)
  const float h = v.size * 0.5f;
  const int x0 = max(0, (int)ceilf(v.xw - h - 0.5f)), x1 = min(p.vw, (int)ceilf(v.xw + h - 0.5f));
  const int y0 = max(0, (int)ceilf(v.yw - h - 0.5f)), y1 = min(p.vh, (int)ceilf(v.yw + h - 0.5f));
  const unsigned long long key = ((unsigned long long)__float_as_uint(v.zw) << 32) | id;
  for (int y = y0; y < y1; ++y)
    for (int x = x0; x < x1; ++x) atomicMin(p.keys + (size_t)y * p.vw + x, key);
}

__global__ void __launch_bounds__(256) k_points_resolve(const __grid_constant__ PointParams p) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.vw * p.vh) return;
  const unsigned long long key = p.keys[i];
  if (key == ~0ull) { p.out_rgba[i] = make_float4(0.f, 0.f, 0.f, 0.f); p.out_depth[i] = 1.0f; return; }
  const uint32_t id = (uint32_t)(key & 0xffffffffull);
  const PointVertex v = point_vertex(p, id);
  float3 c;
  if (p.mode == 0) {
    // points.fs:64-75
    const uint32_t px = (uint32_t)(p.W * p.H);
    const int layer = (int)(id / px);
    if (p.shade_mode == 3) {
      const float* cc = kPointCameraColors[layer < 5 ? layer : 4];
      c = make_float3(cc[0], cc[1], cc[2]);
    } else {
      const float3 color = tex2d_rgb8(p.color + (size_t)p.CW * p.CH * 3 * layer, p.CW, p.CH, v.texcoord.x, v.texcoord.y);
      const float4 n4 = __ldg(p.normal + id);                               // kinect_normals at the pixel's own centre
      const float4 vn = pmulv(p.normal_matrix, make_float4(n4.x, n4.y, n4.z, 0.0f));
      c = pshade(p.shade_mode, p.mvT3, v.pos_es, make_float3(vn.x, vn.y, vn.z), color);
    }
  } else {
    // calib_vis.fs:17-27
    const float inverted = fabsf(v.distance) / p.limit;
    c = v.distance > 0.0f ? make_float3(1.0f - inverted, 0.0f, 0.0f) : make_float3(0.0f, 1.0f - inverted, 0.0f);
    if (v.distance >= p.limit) c = make_float3(0.0f, 0.0f, 1.0f);
  }
  p.out_rgba[i] = make_float4(c.x, c.y, c.z, 1.0f);
  p.out_depth[i] = v.zw;
}

// mode 0: ReconPoints::draw; mode 1: ReconCalibs::draw (limit: its own m_tsdf_limit, setTsdfLimit). The view images of the
// context (d_rgba, d_zbuf) receive the result, like a raymarch.
int launch_draw_points(rr_ctx* c, const rr_view* v, int mode, float calib_limit) {
  PointParams p{};
  const int vw = v->viewport[2], vh = v->viewport[3];
  double MV[16], inv[16];
  for (int i = 0; i < 16; ++i) { MV[i] = v->modelview[i]; p.mv[i] = v->modelview[i]; p.proj[i] = v->projection[i]; }
  // gl_NormalMatrix: the inverse transpose of the modelview matrix (points.fs:67)
  if (!pinvert4(MV, inv)) return fail(c, RR_ERR_INVALID, "draw points: singular modelview");
  for (int cc = 0; cc < 4; ++cc) for (int r = 0; r < 4; ++r) p.normal_matrix[cc * 4 + r] = (float)inv[r * 4 + cc];
  for (int cc = 0; cc < 3; ++cc) for (int r = 0; r < 3; ++r) p.mvT3[cc * 3 + r] = v->modelview[r * 4 + cc];
  // calib_vis.vs: vol_to_world = translate(bbox_min) * scale(bbox_size) (recon_calibs.cpp:39-46)
  const float dx = c->bbox_max[0] - c->bbox_min[0], dy = c->bbox_max[1] - c->bbox_min[1], dz = c->bbox_max[2] - c->bbox_min[2];
  p.v2w[0] = dx; p.v2w[5] = dy; p.v2w[10] = dz; p.v2w[12] = c->bbox_min[0]; p.v2w[13] = c->bbox_min[1]; p.v2w[14] = c->bbox_min[2]; p.v2w[15] = 1.0f;
  p.vw = vw; p.vh = vh; p.shade_mode = v->shade_mode; p.mode = mode;
  p.N = c->N; p.W = c->W; p.H = c->H; p.CW = c->CW; p.CH = c->CH;
  p.st = sensor_tables(c);
  p.depth_b = c->d_depth_b.ptr; p.normal = c->d_normal.ptr; p.color = c->d_color;
  for (int a = 0; a < 3; ++a) { p.bmin[a] = c->bbox_min[a]; p.bmax[a] = c->bbox_max[a]; }
  p.IX = (int)c->ires[0]; p.IY = (int)c->ires[1]; p.IZ = (int)c->ires[2];
  p.tsdf = c->d_tsdf.ptr; p.X = (int)c->res[0]; p.Y = (int)c->res[1]; p.Z = (int)c->res[2];
  p.half2 = c->cfg.store_weight == RR_VOXELS_HALF2 ? 1 : 0;
  p.limit = calib_limit;
  p.keys = c->d_point_keys.ptr; p.out_rgba = c->d_rgba.ptr; p.out_depth = c->d_zbuf.ptr;
  const uint32_t n_vertices = mode == 0 ? (uint32_t)c->N * c->W * c->H : (uint32_t)(p.IX * p.IY * p.IZ);
  const int npx = vw * vh;
  timer_begin(c, "3recon");
  timer_begin(c, "draw");
  k_points_clear<<<(npx + 255) / 256, 256, 0, c->stream>>>(p.keys, npx);
  RR_LAUNCH_CHECK(c, "k_points_clear");
  if (n_vertices) {
    k_points_splat<<<(n_vertices + 255) / 256, 256, 0, c->stream>>>(p, n_vertices);
    RR_LAUNCH_CHECK(c, "k_points_splat");
  }
  k_points_resolve<<<(npx + 255) / 256, 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_points_resolve");
  timer_end(c, "draw");
  timer_end(c, "3recon");
  return RR_OK;
}

}  // namespace rr
