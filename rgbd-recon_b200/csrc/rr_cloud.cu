// The pre-processed sensor points as a coloured point cloud (rr_extract_points / rr_download_points / rr_group_extract_points;
// the contract is stated in include/rgbd_recon_b200.h and DESIGN.md "Beyond the reference: point clouds"). No reference
// counterpart: a reference user could only draw the points (ReconPoints::draw) and read pixels back.
//   k_cloud_flags  one thread per depth pixel: 1 when its sensor is in the mask and sensor_point (rr_sensor_point.cuh, the
//                  vertex stage rr_draw_points runs) keeps it
//   CUB exclusive scan of the flags: each kept pixel's output slot, ascending pixel id; the total is read back in the call's
//                  single synchronisation
//   k_cloud_write  one thread per depth pixel: a kept pixel writes its position, normal, colour, quality and id at its slot
#include "rr_context.h"
#include "rr_sensor_point.cuh"

#include <cub/device/device_scan.cuh>

namespace rr {

namespace {

struct CloudParams {
  SensorTables st;
  const float2* depth_b; const float4* normal; const float* quality; const uint8_t* color;
  int W, H, CW, CH;
  uint32_t mask, n_px;
  float bmin[3], bmax[3];
  uint32_t* flags; const uint32_t* offsets;
  float* pos; float* nrm; float* rgb; float* q; uint32_t* pix;
};

__device__ __forceinline__ bool cloud_keep(const CloudParams& p, uint32_t id, float3& pos, float2& tc) {
  const uint32_t layer = id / (uint32_t)(p.W * p.H);
  if (!((p.mask >> layer) & 1u)) return false;
  return sensor_point(p.st, p.depth_b, p.W, p.H, p.bmin, p.bmax, id, pos, tc);
}

// flags[n_px] = 0 closes the scan, so offsets[n_px] is the number of points
__global__ void __launch_bounds__(256) k_cloud_flags(const __grid_constant__ CloudParams p) {
  const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id > p.n_px) return;
  float3 pos; float2 tc;
  p.flags[id] = id < p.n_px && cloud_keep(p, id, pos, tc) ? 1u : 0u;
}

__global__ void __launch_bounds__(256) k_cloud_write(const __grid_constant__ CloudParams p) {
  const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= p.n_px || !p.flags[id]) return;
  float3 pos; float2 tc;
  cloud_keep(p, id, pos, tc);                           // kept: the flag pass ran the same function on the same inputs
  const size_t o = p.offsets[id];
  const int layer = (int)(id / (uint32_t)(p.W * p.H));
  // the colour rr_draw_points shades with (points.fs:64-75, k_points_resolve)
  const float3 c = tex2d_rgb8(p.color + (size_t)p.CW * p.CH * 3 * layer, p.CW, p.CH, tc.x, tc.y);
  const float4 n = __ldg(p.normal + id);
  p.pos[o * 3] = pos.x; p.pos[o * 3 + 1] = pos.y; p.pos[o * 3 + 2] = pos.z;
  p.nrm[o * 3] = n.x; p.nrm[o * 3 + 1] = n.y; p.nrm[o * 3 + 2] = n.z;
  p.rgb[o * 3] = c.x; p.rgb[o * 3 + 1] = c.y; p.rgb[o * 3 + 2] = c.z;
  p.q[o] = __ldg(p.quality + id);
  p.pix[o] = id;
}

}  // namespace

int launch_extract_points(rr_ctx* c, uint32_t mask, uint32_t* out_n) {
  c->cloud_valid = false;
  const uint32_t n_px = (uint32_t)((size_t)c->N * c->W * c->H);
  RR_TRY_RC(c->d_cloud_flags.reserve(c, 2 * ((size_t)n_px + 1), "cloud flags"));
  uint32_t* flags = c->d_cloud_flags.ptr;
  uint32_t* offsets = flags + (n_px + 1);
  size_t scan_bytes = 0;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, flags, offsets, (int)(n_px + 1), c->stream), "cloud scan size"));
  RR_TRY_RC(c->d_cloud_scratch.reserve(c, scan_bytes, "cloud scan scratch"));

  CloudParams p{};
  p.st = sensor_tables(c);
  p.depth_b = c->d_depth_b.ptr; p.normal = c->d_normal.ptr; p.quality = c->d_quality.ptr; p.color = c->d_color;
  p.W = c->W; p.H = c->H; p.CW = c->CW; p.CH = c->CH;
  p.mask = mask; p.n_px = n_px;
  for (int a = 0; a < 3; ++a) { p.bmin[a] = c->bbox_min[a]; p.bmax[a] = c->bbox_max[a]; }
  p.flags = flags; p.offsets = offsets;

  k_cloud_flags<<<(n_px + 1 + 255) / 256, 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_cloud_flags");
  size_t bytes = c->d_cloud_scratch.cap;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(c->d_cloud_scratch.ptr, bytes, flags, offsets, (int)(n_px + 1), c->stream), "cloud scan"));
  ++c->launches;
  RR_TRY_RC(check(c, cudaMemcpyAsync(&c->pinned->cloud_count, offsets + n_px, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream), "cloud count"));
  RR_TRY_RC(check(c, cudaStreamSynchronize(c->stream), "cloud count sync"));
  const uint32_t n = c->pinned->cloud_count;
  if (n) {
    RR_TRY_RC(c->d_cloud_pos.reserve(c, 3 * (size_t)n, "cloud positions"));
    RR_TRY_RC(c->d_cloud_nrm.reserve(c, 3 * (size_t)n, "cloud normals"));
    RR_TRY_RC(c->d_cloud_rgb.reserve(c, 3 * (size_t)n, "cloud colours"));
    RR_TRY_RC(c->d_cloud_q.reserve(c, n, "cloud quality"));
    RR_TRY_RC(c->d_cloud_pix.reserve(c, n, "cloud pixel ids"));
    p.pos = c->d_cloud_pos.ptr; p.nrm = c->d_cloud_nrm.ptr; p.rgb = c->d_cloud_rgb.ptr; p.q = c->d_cloud_q.ptr; p.pix = c->d_cloud_pix.ptr;
    k_cloud_write<<<(n_px + 255) / 256, 256, 0, c->stream>>>(p);
    RR_LAUNCH_CHECK(c, "k_cloud_write");
  }
  c->cloud_n = n;
  c->cloud_valid = true;
  *out_n = n;
  return RR_OK;
}

int cloud_download(rr_ctx* c, float* positions, float* normals, float* colors, float* quality, uint32_t* pixels) {
  const size_t n = c->cloud_n;
  if (n) {
    if (positions) RR_TRY_RC(check(c, cudaMemcpyAsync(positions, c->d_cloud_pos.ptr, n * 3 * sizeof(float), cudaMemcpyDefault, c->stream), "cloud download"));
    if (normals) RR_TRY_RC(check(c, cudaMemcpyAsync(normals, c->d_cloud_nrm.ptr, n * 3 * sizeof(float), cudaMemcpyDefault, c->stream), "cloud download"));
    if (colors) RR_TRY_RC(check(c, cudaMemcpyAsync(colors, c->d_cloud_rgb.ptr, n * 3 * sizeof(float), cudaMemcpyDefault, c->stream), "cloud download"));
    if (quality) RR_TRY_RC(check(c, cudaMemcpyAsync(quality, c->d_cloud_q.ptr, n * sizeof(float), cudaMemcpyDefault, c->stream), "cloud download"));
    if (pixels) RR_TRY_RC(check(c, cudaMemcpyAsync(pixels, c->d_cloud_pix.ptr, n * sizeof(uint32_t), cudaMemcpyDefault, c->stream), "cloud download"));
  }
  return check(c, cudaStreamSynchronize(c->stream), "cloud download sync");
}

}  // namespace rr
