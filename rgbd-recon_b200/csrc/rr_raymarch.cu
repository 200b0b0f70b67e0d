// TSDF raymarcher for sm_100a: one thread per pixel, replacing ReconIntegration::drawDepthLimits + draw
// (framework/reconstruction/recon_integration.cpp:177-241, 409-429) and glsl/tsdf_raymarch.fs, shading.glsl,
// bricks.{vs,gs,fs}. No rasteriser: the cube proxy and the brick depth limits are analytic per ray; the march itself
// (brick hull, empty-space skipping, z-slab ownership) is rr_march.cuh, shared with rr_cast_rays.
// Filtering is software fp32 (x -> y -> z lerps), see rr_math.cuh.
#include "rr_context.h"
#include "rr_math.cuh"
#include "rr_march.cuh"
#include "rr_sample.cuh"

#include <cmath>

namespace rr {

struct RayParams {
  float img_to_eye[16], inv_mv[16], inv_v2w[16], mv_v2w[16], normal_matrix[16];
  float mvT3[9];
  float cam[3];
  float proj22, proj32;
  const float* tsdf; int X, Y, Z;
  int half2;                      // voxels are half2 (tsdf, weight): the density is the low half
  float limit;
  int N; const float4* inv; int IX, IY, IZ;
  const float2* uv[RR_MAX_SENSORS]; int cx[RR_MAX_SENSORS], cy[RR_MAX_SENSORS], cz[RR_MAX_SENSORS];
  const uint8_t* color; int CW, CH;
  const float2* depth_b; const float* quality; int W, H;
  int vw, vh, shade_mode, skip_space, allow_skip;
  const uint8_t* occ_mask; const uint8_t* near_occ; int rb[3]; float brick_size; float dims[3];
  int z_own0, z_own1;
  float4* out_rgba; float* out_depth; float* out_samples; float4* out_pos; uint32_t* out_step;
};

__device__ __forceinline__ float4 mulv(const float* m, float4 v) {
  float4 o;
  o.x = fmaf(m[12], v.w, fmaf(m[8], v.z, fmaf(m[4], v.y, m[0] * v.x)));
  o.y = fmaf(m[13], v.w, fmaf(m[9], v.z, fmaf(m[5], v.y, m[1] * v.x)));
  o.z = fmaf(m[14], v.w, fmaf(m[10], v.z, fmaf(m[6], v.y, m[2] * v.x)));
  o.w = fmaf(m[15], v.w, fmaf(m[11], v.z, fmaf(m[7], v.y, m[3] * v.x)));
  return o;
}

__constant__ float kCameraColors[5][3] = {{228.f / 255.f, 26.f / 255.f, 28.f / 255.f}, {55.f / 255.f, 126.f / 255.f, 184.f / 255.f},
                                          {77.f / 255.f, 175.f / 255.f, 74.f / 255.f}, {152.f / 255.f, 78.f / 255.f, 163.f / 255.f},
                                          {255.f / 255.f, 127.f / 255.f, 0.f / 255.f}};

// tsdf_raymarch.fs:354-369 blendCameras (+ getWeights :159-174)
__device__ float3 blend_cameras(const RayParams& p, float3 q) {
  float3 tc = make_float3(0.f, 0.f, 0.f);
  float tw = 0.0f;
  const size_t inv_stride = (size_t)p.IX * p.IY * p.IZ, img = (size_t)p.W * p.H;
  for (int i = 0; i < p.N; ++i) {
    const float3 pc = tex3d_xyz(p.inv + inv_stride * i, p.IX, p.IY, p.IZ, q.x, q.y, q.z);
    const float depth = tex_nearest_depth(p.depth_b + img * i, p.W, p.H, pc.x, pc.y);
    float quality = 0.0f;
    if (fabsf(depth - pc.z) < p.limit) quality = tex_linear_1(p.quality + img * i, p.W, p.H, pc.x, pc.y);
    const float* cc = kCameraColors[i < 5 ? i : 4];
    tc.x = fmaf(cc[0], quality, tc.x); tc.y = fmaf(cc[1], quality, tc.y); tc.z = fmaf(cc[2], quality, tc.z);
    tw += quality;
  }
  tc = tc / tw;
  if (tw <= 0.0f) tc = make_float3(1.0f, 1.0f, 1.0f);
  return tc;
}

// shading.glsl:32-69
__device__ float3 shade(const RayParams& p, float3 view_pos, float3 n, float3 diffuse) {
  if (p.shade_mode == 0) return diffuse;
  if (p.shade_mode == 1) {
    const float3 light_pos = make_float3(1.5f, 1.0f, 1.0f), light_diffuse = make_float3(1.0f, 0.9f, 0.7f);
    const float3 light_ambient = light_diffuse * 0.2f;
    float diff = 0.0f, spec = 0.0f;
    const float3 to_light = normalize3(light_pos - view_pos);
    const float light_angle = dot3(n, to_light);
    if (!(light_angle <= 0.0f)) {
      diff = gmax(light_angle, 0.0f);
      const float3 to_viewer = normalize3(make_float3(-view_pos.x, -view_pos.y, -view_pos.z));
      const float3 halfway = normalize3(to_light + to_viewer);
      const float reflected = dot3(halfway, n);
      spec = gpow(reflected, 20.0f);
      const float a = (1.0f - light_angle) * (1.0f - light_angle);
      spec *= 1.0f - a * a * a;
    }
    const float3 amb = light_ambient * 0.5f;
    const float3 dif = (light_diffuse * 0.5f) * diff;
    const float sp = (1.0f * 0.5f) * spec;
    return make_float3((amb.x + dif.x) + sp, (amb.y + dif.y) + sp, (amb.z + dif.z) + sp);
  }
  if (p.shade_mode == 2) {
    const float* t = p.mvT3;
    return make_float3(fmaf(t[6], n.z, fmaf(t[3], n.y, t[0] * n.x)), fmaf(t[7], n.z, fmaf(t[4], n.y, t[1] * n.x)),
                       fmaf(t[8], n.z, fmaf(t[5], n.y, t[2] * n.x)));
  }
  return make_float3(1.0f, 1.0f, 1.0f);
}

__global__ void __launch_bounds__(64) k_raymarch(const __grid_constant__ RayParams p) {
  const int px = blockIdx.x * 8 + threadIdx.x, py = blockIdx.y * 8 + threadIdx.y;
  if (px >= p.vw || py >= p.vh) return;
  const size_t o = (size_t)py * p.vw + px;
  float4 rgba = make_float4(0.f, 0.f, 0.f, 0.f), pos = make_float4(0.f, 0.f, 0.f, 0.f);
  float zbuf = 1.0f, nsamp = 0.0f;
  uint32_t hit_step = 0xFFFFFFFFu;

  // screenToVol(vec3(frag.xy, 1.0)) (tsdf_raymarch.fs:384-390)
  const float4 pc = mulv(p.img_to_eye, make_float4((float)px + 0.5f, (float)py + 0.5f, 1.0f, 1.0f));
  const float4 es = make_float4(pc.x / pc.w, pc.y / pc.w, pc.z / pc.w, 1.0f);
  const float4 ws = mulv(p.inv_mv, es);
  const float4 pv = mulv(p.inv_v2w, ws);
  const float3 cam = make_float3(p.cam[0], p.cam[1], p.cam[2]);
  const float3 dir = normalize3(make_float3(pv.x, pv.y, pv.z) - cam);
  const float sd = p.limit * 0.5f;
  march_ray(p, cam, dir, [&](uint32_t num_samples, bool hit, float3 sample_pos) {
    nsamp = (float)num_samples * 0.0027f;
    if (hit) {
      hit_step = num_samples;
      // submitFragment (tsdf_raymarch.fs:116-142); get_gradient :148-157
      const float3 q = sample_pos;
      const float3 gn = get_gradient(p, q, sd);
      const float4 vn4 = mulv(p.normal_matrix, make_float4(gn.x, gn.y, gn.z, 0.0f));
      const float3 view_normal = normalize3(make_float3(vn4.x, vn4.y, vn4.z));
      const float4 vp4 = mulv(p.mv_v2w, make_float4(q.x, q.y, q.z, 1.0f));
      const float3 view_pos = make_float3(vp4.x, vp4.y, vp4.z);
      if (p.shade_mode == 3) {
        const float3 c = blend_cameras(p, q);
        rgba = make_float4(c.x, c.y, c.z, 1.0f);
      } else {
        const float4 diffuse = blend_colors(p, q);
        const float3 c = shade(p, view_pos, view_normal, make_float3(diffuse.x, diffuse.y, diffuse.z));
        rgba = make_float4(c.x, c.y, c.z, diffuse.w);
      }
      zbuf = (p.proj22 * view_pos.z + p.proj32) / -view_pos.z * 0.5f + 0.5f;
      pos = make_float4(q.x, q.y, q.z, 1.0f);
    }
  });
  p.out_rgba[o] = rgba;
  p.out_depth[o] = zbuf;
  p.out_samples[o] = nsamp;
  p.out_pos[o] = pos;
  p.out_step[o] = hit_step;
}

// ---- multi-GPU: per-slab partial ray records and their composite (SURVEY.md §8e) -------------------------------------
// A slab context marches only the steps whose nearest z texel it owns and reports, per pixel, a 32-byte record
// {rgba; depth, step index of its first hit (0xFFFFFFFF = none), sample count, 0}. After ONE gather the display GPU keeps
// the record with the smallest step index: exactly the hit the single-volume march would have found first.
__global__ void __launch_bounds__(256) k_pack_partial(const float4* __restrict__ rgba, const float* __restrict__ depth,
                                                      const uint32_t* __restrict__ step, const float* __restrict__ nsamp,
                                                      float4* __restrict__ rec, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  rec[2 * i] = rgba[i];
  rec[2 * i + 1] = make_float4(depth[i], __uint_as_float(step[i]), nsamp[i], 0.0f);
}

__global__ void __launch_bounds__(256) k_composite(const float4* __restrict__ rec, int n_parts, int n, float4* __restrict__ rgba,
                                                   float* __restrict__ depth, uint32_t* __restrict__ step, float* __restrict__ nsamp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 best_a = rec[2 * i], best_b = rec[2 * i + 1];
  uint32_t best_step = __float_as_uint(best_b.y);
  for (int p = 1; p < n_parts; ++p) {
    const float4 b = rec[((size_t)p * n + i) * 2 + 1];
    const uint32_t st = __float_as_uint(b.y);
    if (st < best_step) { best_step = st; best_b = b; best_a = rec[((size_t)p * n + i) * 2]; }
  }
  rgba[i] = best_a; depth[i] = best_b.x; step[i] = best_step; nsamp[i] = best_b.z;
}

// Compositing by two reductions instead of a gather (the display GPU would otherwise receive n_parts record images):
//   key = first_hit_step << 8 | rank   ->  MIN all-reduce: the winner of every pixel (smallest step, lowest rank on ties,
//                                          exactly k_composite's choice)
//   records of non-winners zeroed       ->  integer SUM reduce onto the display GPU: x + 0 + ... + 0 is x bit for bit
__global__ void __launch_bounds__(256) k_partial_keys(const float4* __restrict__ rec, long long rank, long long* __restrict__ keys, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  keys[i] = ((long long)__float_as_uint(rec[2 * i + 1].y) << 8) | rank;
}

__global__ void __launch_bounds__(256) k_partial_keep(float4* __restrict__ rec, const long long* __restrict__ keys_min, long long rank, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long mine = ((long long)__float_as_uint(rec[2 * i + 1].y) << 8) | rank;
  if (keys_min[i] != mine) { rec[2 * i] = make_float4(0.f, 0.f, 0.f, 0.f); rec[2 * i + 1] = make_float4(0.f, 0.f, 0.f, 0.f); }
}

int launch_partial_keys(rr_ctx* c, const float4* d_rec, int rank, long long* d_keys) {
  const int n = c->view_w * c->view_h;
  k_partial_keys<<<(n + 255) / 256, 256, 0, c->stream>>>(d_rec, (long long)rank, d_keys, n);
  RR_LAUNCH_CHECK(c, "k_partial_keys");
  return RR_OK;
}

int launch_partial_keep(rr_ctx* c, float4* d_rec, const long long* d_keys_min, int rank) {
  const int n = c->view_w * c->view_h;
  k_partial_keep<<<(n + 255) / 256, 256, 0, c->stream>>>(d_rec, d_keys_min, (long long)rank, n);
  RR_LAUNCH_CHECK(c, "k_partial_keep");
  return RR_OK;
}

int launch_pack_partial(rr_ctx* c, float4* d_rec) {
  const int n = c->view_w * c->view_h;
  k_pack_partial<<<(n + 255) / 256, 256, 0, c->stream>>>(c->d_rgba.ptr, c->d_zbuf.ptr, c->d_step.ptr, c->d_nsamples.ptr, d_rec, n);
  RR_LAUNCH_CHECK(c, "k_pack_partial");
  return RR_OK;
}

int launch_composite(rr_ctx* c, const float4* d_rec, int n_parts) {
  const int n = c->view_w * c->view_h;
  k_composite<<<(n + 255) / 256, 256, 0, c->stream>>>(d_rec, n_parts, n, c->d_rgba.ptr, c->d_zbuf.ptr, c->d_step.ptr, c->d_nsamples.ptr);
  RR_LAUNCH_CHECK(c, "k_composite");
  return RR_OK;
}

// ---- host side: per-frame uniforms of ReconIntegration::draw (recon_integration.cpp:183-206) ----------------------
namespace {

// adjugate / determinant in double from the float inputs (glm::inverse / gloost::Matrix::invert stand-in)
bool invert4(const double* m, double* out) {
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

void matmul4(const double* a, const double* b, double* out) {
  for (int c = 0; c < 4; ++c)
    for (int r = 0; r < 4; ++r) {
      double acc = 0.0;
      for (int k = 0; k < 4; ++k) acc += a[k * 4 + r] * b[c * 4 + k];
      out[c * 4 + r] = acc;
    }
}

}  // namespace

int launch_raymarch(rr_ctx* c, const rr_view* v) {
  RayParams p{};
  const int vw = v->viewport[2], vh = v->viewport[3];
  double MV[16], P[16], V[16] = {0}, t[16], t2[16], inv[16];
  for (int i = 0; i < 16; ++i) { MV[i] = v->modelview[i]; P[i] = v->projection[i]; }
  const float dx = c->bbox_max[0] - c->bbox_min[0], dy = c->bbox_max[1] - c->bbox_min[1], dz = c->bbox_max[2] - c->bbox_min[2];
  V[0] = dx; V[5] = dy; V[10] = dz; V[12] = c->bbox_min[0]; V[13] = c->bbox_min[1]; V[14] = c->bbox_min[2]; V[15] = 1.0;
  const double Tr[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 1, 1, 1, 1};
  const double Sc[16] = {vw * 0.5, 0, 0, 0, 0, vh * 0.5, 0, 0, 0, 0, 0.5, 0, 0, 0, 0, 1};
  matmul4(Tr, P, t); matmul4(Sc, t, t2);
  if (!invert4(t2, inv)) return fail(c, RR_ERR_INVALID, "rr_raymarch: singular projection");
  for (int i = 0; i < 16; ++i) p.img_to_eye[i] = (float)inv[i];
  if (!invert4(MV, inv)) return fail(c, RR_ERR_INVALID, "rr_raymarch: singular modelview");
  for (int i = 0; i < 16; ++i) p.inv_mv[i] = (float)inv[i];
  invert4(V, inv);
  for (int i = 0; i < 16; ++i) p.inv_v2w[i] = (float)inv[i];
  matmul4(MV, V, t);
  for (int i = 0; i < 16; ++i) p.mv_v2w[i] = (float)t[i];
  invert4(t, inv);
  for (int cc = 0; cc < 4; ++cc) for (int r = 0; r < 4; ++r) p.normal_matrix[cc * 4 + r] = (float)inv[r * 4 + cc];
  for (int cc = 0; cc < 3; ++cc) for (int r = 0; r < 3; ++r) p.mvT3[cc * 3 + r] = v->modelview[r * 4 + cc];
  {
    const float cw[4] = {p.inv_mv[12], p.inv_mv[13], p.inv_mv[14], p.inv_mv[15]};
    for (int r = 0; r < 3; ++r)
      p.cam[r] = std::fmaf(p.inv_v2w[12 + r], cw[3], std::fmaf(p.inv_v2w[8 + r], cw[2], std::fmaf(p.inv_v2w[4 + r], cw[1], p.inv_v2w[r] * cw[0])));
  }
  p.proj22 = v->projection[10]; p.proj32 = v->projection[14];
  set_sample_params(p, c);
  p.vw = vw; p.vh = vh; p.shade_mode = v->shade_mode;
  set_march_params(p, c);
  p.out_rgba = c->d_rgba.ptr; p.out_depth = c->d_zbuf.ptr; p.out_samples = c->d_nsamples.ptr; p.out_pos = c->d_pos.ptr; p.out_step = c->d_step.ptr;
  timer_begin(c, "3recon");
  timer_begin(c, "draw");
  const dim3 blk(8, 8, 1), grd((vw + 7) / 8, (vh + 7) / 8, 1);
  k_raymarch<<<grd, blk, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_raymarch");
  timer_end(c, "draw");
  timer_end(c, "3recon");
  return RR_OK;
}

}  // namespace rr
