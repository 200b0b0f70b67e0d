// Queries of the fused volume at rays and points the caller chooses (rr_sample_points / rr_cast_rays and their group
// forms; the contract is stated in include/rgbd_recon_b200.h and DESIGN.md "Beyond the reference: queries"). No reference
// counterpart: a reference user had to render a view and read pixels back, or download the volume.
//   k_sample_points  one thread per point: the density the raymarch reads there, the mesh vertex normal, blendColors
//   k_cast_rays      one thread per ray: the raymarch's own march (rr_march.cuh), then the same three at the refined hit
//   k_query_rays_composite / k_query_points_composite   device group: member 0 keeps each ray's first hit over the
//                    members (smallest step, lowest member on ties) and each point's owner's sample, through peer memory
// Inputs are copied into d_q_in (points [n][3], or origins [n][3] followed by directions [n][3]); every result lands in
// the d_q_* arrays, from which the caller's outputs are copied.
#include "rr_context.h"
#include "rr_march.cuh"

namespace rr {

namespace {

struct QueryParams {
  // the sample block of rr_sample.cuh
  const float* tsdf; int X, Y, Z;
  int half2;
  float limit;
  int N; const float4* inv; int IX, IY, IZ;
  const float2* uv[RR_MAX_SENSORS]; int cx[RR_MAX_SENSORS], cy[RR_MAX_SENSORS], cz[RR_MAX_SENSORS];
  const uint8_t* color; int CW, CH;
  const float2* depth_b; const float* quality; int W, H;
  // the march block of rr_march.cuh (dims = bbox_max - bbox_min)
  int skip_space, allow_skip;
  const uint8_t* occ_mask; const uint8_t* near_occ; int rb[3]; float brick_size; float dims[3];
  int z_own0, z_own1;
  // conversion
  float bmin[3];
  int world;                 // RR_QUERY_WORLD: inputs and positions in metres
  // entries
  const float* in; uint32_t n;
  float* val; float* pos; float* nrm; float4* rgba; uint32_t* step;
};

constexpr uint32_t kNaN = 0x7fc00000u;   // the quiet NaN of outputs without a value

__device__ __forceinline__ bool finite3(float3 v) {
  return fabsf(v.x) <= 3.402823466e38f && fabsf(v.y) <= 3.402823466e38f && fabsf(v.z) <= 3.402823466e38f;
}

__device__ __forceinline__ float3 ld3(const float* a, size_t i) { return make_float3(a[i * 3], a[i * 3 + 1], a[i * 3 + 2]); }
__device__ __forceinline__ void st3(float* a, size_t i, float3 v) { a[i * 3] = v.x; a[i * 3 + 1] = v.y; a[i * 3 + 2] = v.z; }

// Directions are normalised with the raymarch's normalize3 (v * (1 / sqrt(dot(v, v)))). Its dot product overflows for
// |v| beyond ~1.8e19 (the result would be the zero vector, a ray of step 0) and loses precision below ~1e-15 (or becomes NaN),
// so a finite non-zero direction outside that range is first scaled by an exact power of two; ordinary directions keep
// normalize3's bits. In world space the division by the bbox size gets the same treatment when it overflows.
__device__ __forceinline__ float3 dir_to_volume(const QueryParams& p, float3 d) {
  if (p.world) {
    float3 v = make_float3(d.x / p.dims[0], d.y / p.dims[1], d.z / p.dims[2]);
    if (!finite3(v) && finite3(d)) { d = d * 0x1p-70f; v = make_float3(d.x / p.dims[0], d.y / p.dims[1], d.z / p.dims[2]); }
    d = v;
  }
  const float s = dot3(d, d);
  if (s == __int_as_float(0x7f800000)) {
    d = d * 0x1p-70f;
  } else if (s < 0x1p-100f) {                              // also the zero vector, which stays zero (and normalises to NaN)
    d = d * 0x1p64f;
    if (dot3(d, d) < 0x1p-100f) d = d * 0x1p64f;
  }
  return normalize3(d);
}

// The march's sample count is derived in binary32 from the ray parameters of the cube entry and exit; from an origin farther
// than kMaxOrigin bbox sizes their rounding error could reach billions of steps, so such origins are not cast.
constexpr float kMaxOrigin = 0x1p24f;

__device__ __forceinline__ bool castable(float3 q0, float3 dir) {
  return finite3(q0) && fabsf(q0.x) <= kMaxOrigin && fabsf(q0.y) <= kMaxOrigin && fabsf(q0.z) <= kMaxOrigin && finite3(dir) &&
         dot3(dir, dir) > 0.0f;
}

__device__ __forceinline__ float3 from_volume(const QueryParams& p, float3 q) {
  if (!p.world) return q;
  return make_float3(p.bmin[0] + q.x * p.dims[0], p.bmin[1] + q.y * p.dims[1], p.bmin[2] + q.z * p.dims[2]);
}

__global__ void __launch_bounds__(128) k_sample_points(const __grid_constant__ QueryParams p) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  const float3 q = to_volume(p, ld3(p.in, i));
  const bool inside = in_unit_cube(q);
  if (inside && ((p.z_own0 > 0) || (p.z_own1 < p.Z))) {
    const int zi = near_coord(q.z, p.Z);
    if (zi < p.z_own0 || zi >= p.z_own1) return;          // a group member that owns the slice evaluates it
  }
  const float nan = __uint_as_float(kNaN);
  float v = nan;
  float3 n = make_float3(nan, nan, nan);
  float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
  if (inside) {
    v = sample_tsdf(p, q);
    n = world_normal(p, q);
    c = blend_colors(p, q);
  }
  p.val[i] = v;
  st3(p.nrm, i, n);
  p.rgba[i] = c;
}

__global__ void __launch_bounds__(128) k_cast_rays(const __grid_constant__ QueryParams p) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  const float3 cam = to_volume(p, ld3(p.in, i));
  const float3 dir = dir_to_volume(p, ld3(p.in + (size_t)p.n * 3, i));
  const float nan = __uint_as_float(kNaN);
  float3 pos = make_float3(nan, nan, nan), n = pos;
  float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
  uint32_t hit_step = 0xFFFFFFFFu;
  if (castable(cam, dir)) {                                // a zero direction normalises to NaN: no hit
    march_ray(p, cam, dir, [&](uint32_t num_samples, bool hit, float3 q) {
      if (!hit) return;
      hit_step = num_samples;
      n = world_normal(p, q);
      c = blend_colors(p, q);
      pos = from_volume(p, q);
    });
  }
  st3(p.pos, i, pos);
  st3(p.nrm, i, n);
  p.rgba[i] = c;
  p.step[i] = hit_step;
}

// ---- device group: the members' results, read by member 0 through peer memory ----------------------------------------
struct QueryPeers {
  const float* val[RR_MAX_GROUP]; const float* pos[RR_MAX_GROUP]; const float* nrm[RR_MAX_GROUP];
  const float4* rgba[RR_MAX_GROUP]; const uint32_t* step[RR_MAX_GROUP];
  int z1[RR_MAX_GROUP];      // end of member m's slab
  int n;
};

// the first hit along the ray is the smallest step index over the members (lowest member on ties, as k_composite_peers)
__global__ void __launch_bounds__(256) k_query_rays_composite(const __grid_constant__ QueryPeers pq, const __grid_constant__ QueryParams p) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  int best = 0;
  uint32_t best_step = p.step[i];
  for (int m = 1; m < pq.n; ++m) {
    const uint32_t s = pq.step[m][i];
    if (s < best_step) { best_step = s; best = m; }
  }
  if (best == 0) return;                                   // member 0's record already is the output
  st3(p.pos, i, ld3(pq.pos[best], i));
  st3(p.nrm, i, ld3(pq.nrm[best], i));
  p.rgba[i] = pq.rgba[best][i];
  p.step[i] = best_step;
}

// a point inside the volume was evaluated by the member that owns its nearest z slice (k_sample_points)
__global__ void __launch_bounds__(256) k_query_points_composite(const __grid_constant__ QueryPeers pq, const __grid_constant__ QueryParams p) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  const float3 q = to_volume(p, ld3(p.in, i));
  if (!in_unit_cube(q)) return;
  const int zi = near_coord(q.z, p.Z);
  int owner = 0;
  while (owner + 1 < pq.n && zi >= pq.z1[owner]) ++owner;
  if (owner == 0) return;
  p.val[i] = pq.val[owner][i];
  st3(p.nrm, i, ld3(pq.nrm[owner], i));
  p.rgba[i] = pq.rgba[owner][i];
}

QueryParams query_params(const rr_ctx* c, int space, uint32_t count) {
  QueryParams p{};
  set_sample_params(p, c);
  set_march_params(p, c);
  for (int a = 0; a < 3; ++a) p.bmin[a] = c->bbox_min[a];
  p.world = space == RR_QUERY_WORLD ? 1 : 0;
  p.in = c->d_q_in.ptr; p.n = count;
  p.val = c->d_q_val.ptr; p.pos = c->d_q_pos.ptr; p.nrm = c->d_q_nrm.ptr; p.rgba = c->d_q_rgba.ptr; p.step = c->d_q_step.ptr;
  return p;
}

}  // namespace

int query_reserve(rr_ctx* c, uint32_t count) {
  const size_t n = count;
  RR_TRY_RC(c->d_q_in.reserve(c, 6 * n, "query inputs"));
  RR_TRY_RC(c->d_q_val.reserve(c, n, "query values"));
  RR_TRY_RC(c->d_q_pos.reserve(c, 3 * n, "query positions"));
  RR_TRY_RC(c->d_q_nrm.reserve(c, 3 * n, "query normals"));
  RR_TRY_RC(c->d_q_rgba.reserve(c, n, "query colours"));
  return c->d_q_step.reserve(c, n, "query steps");
}

int query_upload(rr_ctx* c, const float* a, const float* b, uint32_t count) {
  RR_TRY_RC(query_reserve(c, count));
  const size_t bytes = (size_t)count * 3 * sizeof(float);
  RR_TRY_RC(check(c, cudaMemcpyAsync(c->d_q_in.ptr, a, bytes, cudaMemcpyDefault, c->stream), "query input copy"));
  if (b) RR_TRY_RC(check(c, cudaMemcpyAsync(c->d_q_in.ptr + (size_t)count * 3, b, bytes, cudaMemcpyDefault, c->stream), "query input copy"));
  return RR_OK;
}

int launch_sample_points(rr_ctx* c, int space, uint32_t count) {
  const QueryParams p = query_params(c, space, count);
  k_sample_points<<<(count + 127) / 128, 128, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_sample_points");
  return RR_OK;
}

int launch_cast_rays(rr_ctx* c, int space, uint32_t count) {
  const QueryParams p = query_params(c, space, count);
  k_cast_rays<<<(count + 127) / 128, 128, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_cast_rays");
  return RR_OK;
}

int launch_query_composite(rr_ctx* const* members, int n, bool rays, int space, uint32_t count) {
  rr_ctx* c0 = members[0];
  QueryPeers pq{};
  pq.n = n;
  for (int m = 0; m < n; ++m) {
    const rr_ctx* c = members[m];
    pq.val[m] = c->d_q_val.ptr; pq.pos[m] = c->d_q_pos.ptr; pq.nrm[m] = c->d_q_nrm.ptr; pq.rgba[m] = c->d_q_rgba.ptr; pq.step[m] = c->d_q_step.ptr;
    pq.z1[m] = (int)c->slab_z1;
  }
  const QueryParams p = query_params(c0, space, count);
  if (rays) {
    k_query_rays_composite<<<(count + 255) / 256, 256, 0, c0->stream>>>(pq, p);
    RR_LAUNCH_CHECK(c0, "k_query_rays_composite");
  } else {
    k_query_points_composite<<<(count + 255) / 256, 256, 0, c0->stream>>>(pq, p);
    RR_LAUNCH_CHECK(c0, "k_query_points_composite");
  }
  return RR_OK;
}

int query_download(rr_ctx* c, uint32_t count, bool rays, float* values_or_positions, float* normals, float* rgba, uint32_t* steps) {
  const size_t n = count;
  if (values_or_positions) {
    const void* src = rays ? (const void*)c->d_q_pos.ptr : (const void*)c->d_q_val.ptr;
    RR_TRY_RC(check(c, cudaMemcpyAsync(values_or_positions, src, n * (rays ? 3 : 1) * sizeof(float), cudaMemcpyDefault, c->stream), "query download"));
  }
  if (normals) RR_TRY_RC(check(c, cudaMemcpyAsync(normals, c->d_q_nrm.ptr, n * 3 * sizeof(float), cudaMemcpyDefault, c->stream), "query download"));
  if (rgba) RR_TRY_RC(check(c, cudaMemcpyAsync(rgba, c->d_q_rgba.ptr, n * sizeof(float4), cudaMemcpyDefault, c->stream), "query download"));
  if (rays && steps) RR_TRY_RC(check(c, cudaMemcpyAsync(steps, c->d_q_step.ptr, n * sizeof(uint32_t), cudaMemcpyDefault, c->stream), "query download"));
  return check(c, cudaStreamSynchronize(c->stream), "query sync");
}

}  // namespace rr
