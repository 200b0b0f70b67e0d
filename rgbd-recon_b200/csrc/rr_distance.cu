// Distances to the captured surface on the device: the exact nearest-inside-voxel transform of the fused volume and distance
// queries at arbitrary points (rr_distance_field / rr_download_distance_field / rr_sample_distance; the contract is stated in
// include/rgbd_recon_b200.h and DESIGN.md "Beyond the reference: distances"). No reference counterpart.
//
// The field is one uint32 per voxel, the linear index of its nearest inside voxel (v > 0, finite: the inside rule of
// rr_parts.cu) under the integer metric dx^2 + dy^2 + dz^2, ties to the smallest index; 0xFFFFFFFF when nothing is inside.
// No distance is stored: every pass re-derives d^2 from the indices. Three separable passes (Meijster, Roerdink and
// Hesselink, "A general algorithm for computing distance transforms in linear time", 2000), each breaking ties toward the
// smaller coordinate, which gives exactly the smallest-index rule (DESIGN.md):
//   k_dist_rows      A <- per voxel row (warp, lanes along x) the nearest inside x of the row, from ballot masks of the
//                    32-voxel words (lane k holds words k and k + 32) and __clz / __ffs; rows without an inside voxel
//                    (in bricks mode: without a candidate) are written 0xFFFFFFFF without reading the volume
//   k_dist_columns   B <- A along y, then A <- B along z: one thread per column, lanes along x (every load and store of a
//                    column step is coalesced); the lower envelope of the column's parabolas (sites s, boundaries t, 16 bits
//                    each) is a stack kept in the destination column itself, which the backward sweep overwrites only
//                    below the entries it still needs (t[k] >= k)
//   k_sample_distance  one thread per query point
#include "rr_context.h"
#include "rr_rows.cuh"
#include "rr_sample.cuh"

namespace rr {

namespace {

constexpr uint32_t kNone = 0xFFFFFFFFu;
constexpr uint32_t kNaN = 0x7fc00000u;   // the quiet NaN of outputs without a value
// k_dist_rows keeps a row's word masks in two registers per lane (64 words); stack entries hold 16-bit coordinates
constexpr int kDistMaxAxis = 2048;

struct DistParams {
  const float* tsdf; int X, Y, Z;   // the sample block of rr_sample.cuh (ld_density)
  int half2;
  // candidate voxels (use_rows = 0: every voxel): the brick row tables of rr_rows.cuh
  int use_rows, rby, mask_words;
  const uint32_t* rowmask; const uint8_t* rowany; const int16_t* cand_y; const int16_t* cand_z;
  const uint32_t* src; uint32_t* dst;
  uint32_t* count;           // inside voxels (k_dist_rows)
};

__device__ __forceinline__ bool inside_voxel(float v) { return v > 0.0f && v <= 3.402823466e38f; }

__global__ void __launch_bounds__(256) k_dist_rows(const __grid_constant__ DistParams p) {
  const unsigned r = blockIdx.x * 8u + (threadIdx.x >> 5);
  if (r >= (unsigned)p.Y * (unsigned)p.Z) return;
  const unsigned lane = threadIdx.x & 31u;
  const int y = (int)(r % (unsigned)p.Y), z = (int)(r / (unsigned)p.Y);
  const unsigned nw = ((unsigned)p.X + 31u) / 32u;        // at most 64 (X <= 2048, rr_distance_field)
  const uint32_t row = r * (uint32_t)p.X;
  uint32_t lo = 0, hi = 0;                                  // inside masks of words lane and lane + 32
  unsigned long long nz = 0;                                // words holding an inside voxel
  uint32_t inside = 0;
  if (row_any(p, y, z)) {
    for (unsigned w = 0; w < nw; ++w) {
      const uint32_t m = row_word(p, y, z, (int)w);
      if (!m) continue;
      const bool in = ((m >> lane) & 1u) && inside_voxel(ld_density(p, row + w * 32u + lane));
      const uint32_t b = __ballot_sync(0xffffffffu, in);
      if (b) {
        nz |= 1ull << w;
        inside += __popc(b);
        if (lane == (w & 31u)) { if (w < 32u) lo = b; else hi = b; }
      }
    }
    if (lane == 0 && inside) atomicAdd(p.count, inside);
  }
  for (unsigned w = 0; w < nw; ++w) {
    const int x = (int)(w * 32u + lane);
    uint32_t out = kNone;
    if (nz) {                                               // warp-uniform: every lane takes part in the shuffles
      const unsigned long long before = nz & ((1ull << w) - 1ull), after = nz & ~((2ull << w) - 1ull);
      const int pw = before ? 63 - __clzll((long long)before) : -1;
      const int qw = after ? __ffsll((long long)after) - 1 : -1;
      const uint32_t m = __shfl_sync(0xffffffffu, w < 32u ? lo : hi, (int)(w & 31u));
      const int pk = pw < 0 ? 0 : pw, qk = qw < 0 ? 0 : qw;
      const uint32_t pm = __shfl_sync(0xffffffffu, pk < 32 ? lo : hi, pk & 31);
      const uint32_t qm = __shfl_sync(0xffffffffu, qk < 32 ? lo : hi, qk & 31);
      const uint32_t below = m & (0xFFFFFFFFu >> (31u - lane)), above = m & (0xFFFFFFFFu << lane);
      int left = -1, right = -1;
      if (below) left = (int)(w * 32u) + 31 - __clz(below);
      else if (pw >= 0) left = pw * 32 + 31 - __clz(pm);
      if (above) right = (int)(w * 32u) + __ffs(above) - 1;
      else if (qw >= 0) right = qw * 32 + __ffs(qm) - 1;
      out = row + (uint32_t)((left >= 0 && (right < 0 || x - left <= right - x)) ? left : right);   // equal: the left one
    }
    if (x < p.X) p.dst[row + (uint32_t)x] = out;
  }
}

// g of a site: the squared distance from column (x, y) to the site's voxel f in the axes already done (AXIS 1: x; 2: x, y)
template <int AXIS>
__device__ __forceinline__ int site_g(uint32_t f, int x, int y, int X, int Y) {
  const uint32_t t = f / (uint32_t)X;
  const int dx = x - (int)(f - t * (uint32_t)X);
  if (AXIS == 1) return dx * dx;
  const int dy = y - (int)(t % (uint32_t)Y);
  return dx * dx + dy * dy;
}

// floor(num / den) for den > 0
__device__ __forceinline__ int floor_div(int num, int den) { return num >= 0 ? num / den : -((-num + den - 1) / den); }

// One column along AXIS (1: y, 2: z) per thread. Site u (a finite src entry) has the parabola g_u + (v - u)^2 over the
// column's coordinate v; on the stack, site s[k] is the minimum over [t[k], t[k+1]). A new site u removes the top if it is
// strictly below it at t[top] (u > s: it stays below from there on), otherwise it starts at 1 + Sep, the last v at which the
// top is at or below it: equal values keep the smaller coordinate.
template <int AXIS>
__global__ void __launch_bounds__(128) k_dist_columns(const __grid_constant__ DistParams p) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t other = AXIS == 1 ? (uint32_t)p.Z : (uint32_t)p.Y;
  if (t >= (uint32_t)p.X * other) return;
  const int x = (int)(t % (uint32_t)p.X), o = (int)(t / (uint32_t)p.X);
  const int y = AXIS == 2 ? o : 0;
  const uint32_t stride = AXIS == 1 ? (uint32_t)p.X : (uint32_t)p.X * (uint32_t)p.Y;
  const uint32_t base = AXIS == 1 ? (uint32_t)o * (uint32_t)p.X * (uint32_t)p.Y + (uint32_t)x : (uint32_t)o * (uint32_t)p.X + (uint32_t)x;
  const int m = AXIS == 1 ? p.Y : p.Z;
  const uint32_t* src = p.src + base;
  uint32_t* dst = p.dst + base;
  int q = -1, sq = 0, tq = 0, gq = 0;                       // the top entry
  for (int u = 0; u < m; ++u) {
    const uint32_t f = src[(uint32_t)u * stride];
    if (f == kNone) continue;
    const int gu = site_g<AXIS>(f, x, y, p.X, p.Y);
    while (q >= 0) {
      const int a = gq + (tq - sq) * (tq - sq), b = gu + (tq - u) * (tq - u);
      if (a <= b) break;
      if (--q >= 0) {
        const uint32_t e = dst[(uint32_t)q * stride];
        sq = (int)(e & 0xFFFFu); tq = (int)(e >> 16);
        gq = site_g<AXIS>(src[(uint32_t)sq * stride], x, y, p.X, p.Y);
      }
    }
    int w = 0;
    if (q >= 0) {
      w = 1 + floor_div(gu - gq + u * u - sq * sq, 2 * (u - sq));
      if (w >= m) continue;
    }
    ++q; sq = u; tq = w; gq = gu;
    dst[(uint32_t)q * stride] = (uint32_t)sq | ((uint32_t)tq << 16);
  }
  if (q < 0) {
    for (int u = 0; u < m; ++u) dst[(uint32_t)u * stride] = kNone;
    return;
  }
  uint32_t fq = src[(uint32_t)sq * stride];
  for (int u = m - 1; u >= 0; --u) {                        // entry q <= t[q] <= u: the write clobbers no entry still needed
    dst[(uint32_t)u * stride] = fq;
    if (u == tq && --q >= 0) {
      const uint32_t e = dst[(uint32_t)q * stride];
      sq = (int)(e & 0xFFFFu); tq = (int)(e >> 16);
      fq = src[(uint32_t)sq * stride];
    }
  }
}

struct DistQuery {
  const uint32_t* nearest; int X, Y, Z;
  int world;                 // RR_QUERY_WORLD: inputs and nearest points in metres
  float bmin[3], dims[3];    // dims = bbox_max - bbox_min (to_volume of rr_sample.cuh)
  const float* in; uint32_t n;
  float* dist; float* pts; uint32_t* vox;
};

// c_k = bmin_k + (((float)f_k + 0.5f) / (float)R_k) * dims_k and p = bmin + q * dims, binary32 with no fused multiply-add
// (--fmad=false); d = sqrtf((dx*dx + dy*dy) + dz*dz), correctly rounded
__global__ void __launch_bounds__(128) k_sample_distance(const __grid_constant__ DistQuery p) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  const float3 v = make_float3(p.in[(size_t)i * 3], p.in[(size_t)i * 3 + 1], p.in[(size_t)i * 3 + 2]);
  const float3 q = to_volume(p, v);
  const float nan = __uint_as_float(kNaN);
  float d = nan;
  float3 c = make_float3(nan, nan, nan);
  uint32_t f = kNone;
  if (in_unit_cube(q)) {
    const uint32_t a = ((uint32_t)near_coord(q.z, p.Z) * (uint32_t)p.Y + (uint32_t)near_coord(q.y, p.Y)) * (uint32_t)p.X +
                       (uint32_t)near_coord(q.x, p.X);
    f = p.nearest[a];
    if (f == kNone) {
      d = __int_as_float(0x7f800000);
    } else {
      const uint32_t t = f / (uint32_t)p.X;
      const uint32_t fx = f - t * (uint32_t)p.X, fy = t % (uint32_t)p.Y, fz = t / (uint32_t)p.Y;
      const float3 cv = make_float3(((float)fx + 0.5f) / (float)p.X, ((float)fy + 0.5f) / (float)p.Y, ((float)fz + 0.5f) / (float)p.Z);
      const float3 cw = make_float3(p.bmin[0] + cv.x * p.dims[0], p.bmin[1] + cv.y * p.dims[1], p.bmin[2] + cv.z * p.dims[2]);
      const float3 pw = p.world ? v : make_float3(p.bmin[0] + v.x * p.dims[0], p.bmin[1] + v.y * p.dims[1], p.bmin[2] + v.z * p.dims[2]);
      const float dx = pw.x - cw.x, dy = pw.y - cw.y, dz = pw.z - cw.z;
      d = sqrtf((dx * dx + dy * dy) + dz * dz);
      c = p.world ? cw : cv;
    }
  }
  p.dist[i] = d;
  p.pts[(size_t)i * 3] = c.x; p.pts[(size_t)i * 3 + 1] = c.y; p.pts[(size_t)i * 3 + 2] = c.z;
  p.vox[i] = f;
}

}  // namespace

int launch_distance_field(rr_ctx* c, uint32_t* out_num_inside) {
  const int X = (int)c->res[0], Y = (int)c->res[1], Z = (int)c->res[2];
  if (X > kDistMaxAxis || Y > kDistMaxAxis || Z > kDistMaxAxis)
    return fail(c, RR_ERR_UNSUPPORTED, "rr_distance_field: volumes with an axis of more than 2048 voxels are not supported");
  const size_t nvox = (size_t)X * Y * Z, rows = (size_t)Y * Z;
  c->dist_valid = false;
  for (int k = 0; k < 2; ++k)                               // exactly a volume each; released by a new volume allocation
    if (c->d_dist[k].cap != nvox) RR_TRY_RC(c->d_dist[k].allocate(c, nvox, "distance field"));
  if (!c->d_dist_count.ptr) RR_TRY_RC(c->d_dist_count.allocate(c, 1, "inside count"));

  DistParams p{};
  p.tsdf = c->d_tsdf.ptr; p.X = X; p.Y = Y; p.Z = Z;
  p.half2 = c->cfg.store_weight == RR_VOXELS_HALF2 ? 1 : 0;
  p.use_rows = c->mesh_rows_ok ? 1 : 0;
  p.rby = (int)c->bricks.res[1]; p.mask_words = c->mask_words;
  p.rowmask = c->d_rowmask.ptr; p.rowany = c->d_rowany.ptr; p.cand_y = c->d_cand_y.ptr; p.cand_z = c->d_cand_z.ptr;
  p.count = c->d_dist_count.ptr;
  uint32_t* A = c->d_dist[0].ptr;
  uint32_t* B = c->d_dist[1].ptr;

  RR_TRY_RC(check(c, cudaMemsetAsync(p.count, 0, sizeof(uint32_t), c->stream), "inside count"));
  p.dst = A;
  k_dist_rows<<<(unsigned)((rows + 7) / 8), 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_dist_rows");
  p.src = A; p.dst = B;
  k_dist_columns<1><<<(unsigned)(((size_t)X * Z + 127) / 128), 128, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_dist_columns<y>");
  p.src = B; p.dst = A;
  k_dist_columns<2><<<(unsigned)(((size_t)X * Y + 127) / 128), 128, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_dist_columns<z>");
  RR_TRY_RC(check(c, cudaMemcpyAsync(&c->pinned->dist_inside, p.count, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream), "inside count"));
  RR_TRY_RC(check(c, cudaStreamSynchronize(c->stream), "distance field sync"));
  c->dist_epoch = c->volume_epoch;
  c->dist_valid = true;
  *out_num_inside = c->pinned->dist_inside;
  return RR_OK;
}

int distance_download(rr_ctx* c, uint32_t* nearest) {
  const size_t nvox = (size_t)c->res[0] * c->res[1] * c->res[2];
  if (nearest) RR_TRY_RC(check(c, cudaMemcpyAsync(nearest, c->d_dist[0].ptr, nvox * sizeof(uint32_t), cudaMemcpyDefault, c->stream), "distance field download"));
  return check(c, cudaStreamSynchronize(c->stream), "distance field download sync");
}

int sample_distance(rr_ctx* c, int space, const float* points, uint32_t count, float* distances, float* nearest_points,
                    uint32_t* nearest_voxels) {
  const size_t n = count;
  RR_TRY_RC(c->d_dq.reserve(c, 7 * n, "distance query buffers"));
  RR_TRY_RC(c->d_dq_vox.reserve(c, n, "distance query voxels"));
  DistQuery p{};
  p.nearest = c->d_dist[0].ptr; p.X = (int)c->res[0]; p.Y = (int)c->res[1]; p.Z = (int)c->res[2];
  p.world = space == RR_QUERY_WORLD ? 1 : 0;
  for (int a = 0; a < 3; ++a) { p.bmin[a] = c->bbox_min[a]; p.dims[a] = c->bbox_max[a] - c->bbox_min[a]; }
  p.in = c->d_dq.ptr; p.n = count;
  p.dist = c->d_dq.ptr + 3 * n; p.pts = c->d_dq.ptr + 4 * n; p.vox = c->d_dq_vox.ptr;
  RR_TRY_RC(check(c, cudaMemcpyAsync(c->d_dq.ptr, points, n * 3 * sizeof(float), cudaMemcpyDefault, c->stream), "distance query input copy"));
  k_sample_distance<<<(count + 127) / 128, 128, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_sample_distance");
  if (distances) RR_TRY_RC(check(c, cudaMemcpyAsync(distances, p.dist, n * sizeof(float), cudaMemcpyDefault, c->stream), "distance query download"));
  if (nearest_points) RR_TRY_RC(check(c, cudaMemcpyAsync(nearest_points, p.pts, n * 3 * sizeof(float), cudaMemcpyDefault, c->stream), "distance query download"));
  if (nearest_voxels) RR_TRY_RC(check(c, cudaMemcpyAsync(nearest_voxels, p.vox, n * sizeof(uint32_t), cudaMemcpyDefault, c->stream), "distance query download"));
  return check(c, cudaStreamSynchronize(c->stream), "distance query sync");
}

}  // namespace rr
