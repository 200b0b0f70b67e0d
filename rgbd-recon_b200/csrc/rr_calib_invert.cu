// Calibration-volume inversion for sm_100a: CalibrationInverter::calculateInverseVolumes for one sensor
// (framework/calibration/calibration_inverter.cpp:99-155) with getXyzSamples (:38-53), inverseDistance (:55-69),
// Frustum::inside (frustum.cpp:36-43) and NearestNeighbourSearch::search (nearest_neighbour_search.cpp:32-43, i.e.
// CGAL Orthogonal_k_neighbor_search: exact k = 8 nearest samples, squared distances in double on float-promoted
// coordinates, ascending; ties broken by the sample's linear index x*Y*Z + y*Z + z).
//
// Shape: the C samples are binned once into a uniform world-space cell grid (count -> exclusive scan -> scatter,
// float4 = position + sample index so a candidate is one LDG.128). One thread owns one output voxel (x fastest, so
// stores are coalesced and neighbouring lanes walk the same cells -> L1 reuse) and searches Chebyshev rings of
// cells around its own cell until the 8th-best distance is provably inside the ring (exact, not approximate).
// Candidates are pre-screened with an fp32 distance against a conservatively widened bound; only survivors pay the
// fp64 distance that decides rank, so results equal a brute-force scan bit for bit. Gather/latency-bound integer and
// fp work: no tensor-core path applies.
#include "rr_context.h"
#include "rr_math.cuh"

#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <cmath>
#include <cstdlib>

namespace rr {

struct CellGrid {
  double gmin[3];
  double cell, inv_cell;
  int dim[3];
};

__device__ __forceinline__ int axis_cell(const CellGrid& g, double v, int a) {
  const int c = (int)floor((v - g.gmin[a]) * g.inv_cell);
  return c < 0 ? 0 : (c >= g.dim[a] ? g.dim[a] - 1 : c);
}

// pass 1/2 of the counting sort: samples enumerated in getXyzSamples order (x outer, z inner) only to derive idx
__global__ void __launch_bounds__(256) k_invert_bin(const float4* __restrict__ xyz, int X, int Y, int Z, const __grid_constant__ CellGrid g,
                                                    uint32_t* __restrict__ cursor, float4* __restrict__ sorted) {
  const size_t n = (size_t)X * Y * Z;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int x = (int)(t % X), y = (int)((t / X) % Y), z = (int)(t / ((size_t)X * Y));
  const float4 p = xyz[t];
  const uint32_t ci = ((uint32_t)axis_cell(g, (double)p.z, 2) * g.dim[1] + axis_cell(g, (double)p.y, 1)) * g.dim[0] + axis_cell(g, (double)p.x, 0);
  const uint32_t slot = atomicAdd(cursor + ci, 1u);
  if (sorted) {
    const uint32_t idx = ((uint32_t)x * Y + y) * Z + z;
    sorted[slot] = make_float4(p.x, p.y, p.z, __uint_as_float(idx));
  }
}

struct InvertParams {
  const float4* sorted;        // binned samples
  const uint32_t* cell_start;  // [ncell + 1]
  CellGrid g;
  float planes[6][4];
  float start[3], step[3];     // sample_start, sample_step (calibration_inverter.cpp:105-108)
  float calib_dims[3];
  const float4* xyz;           // the calibration volume itself, [Z][Y][X] (winners' positions are re-read from it)
  int cX, cY, cZ;
  int ox, oy, oz;
  float4* out;
};

struct Best {
  double d2[8];
  uint32_t idx[8];
};

__device__ __forceinline__ bool cand_less(double d2, uint32_t idx, double bd2, uint32_t bidx) {
  return d2 < bd2 || (d2 == bd2 && idx < bidx);
}

__global__ void __launch_bounds__(128) k_invert(const __grid_constant__ InvertParams p) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y, z = blockIdx.z;
  if (x >= p.ox) return;
  const size_t o = ((size_t)z * p.oy + y) * p.ox + x;
  // glm::fvec3 sample_pos = sample_start + glm::fvec3{x,y,z} * sample_step
  const float sx = p.start[0] + (float)x * p.step[0], sy = p.start[1] + (float)y * p.step[1], sz = p.start[2] + (float)z * p.step[2];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const float d = (p.planes[i][0] * sx + p.planes[i][1] * sy) + (p.planes[i][2] * sz + p.planes[i][3] * 1.0f);
    if (d < 0.0f) { p.out[o] = make_float4(-1.0f, -1.0f, -1.0f, -1.0f); return; }
  }
  const double qx = (double)sx, qy = (double)sy, qz = (double)sz;
  const int cx = axis_cell(p.g, qx, 0), cy = axis_cell(p.g, qy, 1), cz = axis_cell(p.g, qz, 2);
  Best b;
#pragma unroll
  for (int k = 0; k < 8; ++k) { b.d2[k] = __longlong_as_double(0x7ff0000000000000LL); b.idx[k] = 0xFFFFFFFFu; }
  float screen = __int_as_float(0x7f800000);   // fp32 rejection bound: worst kept d2, widened
  const int rmax = max(p.g.dim[0], max(p.g.dim[1], p.g.dim[2]));
  for (int r = 0; r <= rmax; ++r) {
    const int z0 = max(cz - r, 0), z1 = min(cz + r, p.g.dim[2] - 1);
    const int y0 = max(cy - r, 0), y1 = min(cy + r, p.g.dim[1] - 1);
    const int x0 = max(cx - r, 0), x1 = min(cx + r, p.g.dim[0] - 1);
    for (int zz = z0; zz <= z1; ++zz) {
      const bool z_shell = (abs(zz - cz) == r);
      for (int yy = y0; yy <= y1; ++yy) {
        const bool yz_shell = z_shell || (abs(yy - cy) == r);
        const uint32_t row = ((uint32_t)zz * p.g.dim[1] + yy) * p.g.dim[0];
        // shell cells of this row: the whole x span on a y/z face, else only the two end cells (if inside the grid)
        for (int pass = 0; pass < 2; ++pass) {
          int xa, xb;
          if (yz_shell) { if (pass) break; xa = x0; xb = x1; }
          else if (pass == 0) { if (cx - r < 0) continue; xa = xb = cx - r; }
          else { if (r == 0 || cx + r >= p.g.dim[0]) break; xa = xb = cx + r; }
          const uint32_t s0 = __ldg(p.cell_start + row + xa), s1 = __ldg(p.cell_start + row + xb + 1);
          for (uint32_t s = s0; s < s1; ++s) {
            const float4 c = __ldg(p.sorted + s);
            const float fx = sx - c.x, fy = sy - c.y, fz = sz - c.z;
            const float f2 = fmaf(fz, fz, fmaf(fy, fy, fx * fx));
            if (f2 > screen) continue;
            const double dx = qx - (double)c.x, dy = qy - (double)c.y, dz = qz - (double)c.z;
            const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
            const uint32_t idx = __float_as_uint(c.w);
            if (!cand_less(d2, idx, b.d2[7], b.idx[7])) continue;
            // insert into the ascending list (registers only: fully unrolled bubble from the tail)
            b.d2[7] = d2; b.idx[7] = idx;
#pragma unroll
            for (int k = 7; k > 0; --k) {
              if (cand_less(b.d2[k], b.idx[k], b.d2[k - 1], b.idx[k - 1])) {
                const double td = b.d2[k]; b.d2[k] = b.d2[k - 1]; b.d2[k - 1] = td;
                const uint32_t ti = b.idx[k]; b.idx[k] = b.idx[k - 1]; b.idx[k - 1] = ti;
              }
            }
            // fp32 screen: anything with an fp32 distance above this cannot beat the 8th best in fp64
            screen = (b.idx[7] == 0xFFFFFFFFu) ? __int_as_float(0x7f800000) : __double2float_ru(b.d2[7]) * 1.0001f + 1e-30f;
          }
        }
      }
    }
    if (b.idx[7] != 0xFFFFFFFFu) {
      // distance from the query to the nearest face of the visited cell cube that still has cells behind it
      double dout = 1e300;
      if (cx - r > 0) dout = fmin(dout, qx - (p.g.gmin[0] + (double)(cx - r) * p.g.cell));
      if (cx + r < p.g.dim[0] - 1) dout = fmin(dout, (p.g.gmin[0] + (double)(cx + r + 1) * p.g.cell) - qx);
      if (cy - r > 0) dout = fmin(dout, qy - (p.g.gmin[1] + (double)(cy - r) * p.g.cell));
      if (cy + r < p.g.dim[1] - 1) dout = fmin(dout, (p.g.gmin[1] + (double)(cy + r + 1) * p.g.cell) - qy);
      if (cz - r > 0) dout = fmin(dout, qz - (p.g.gmin[2] + (double)(cz - r) * p.g.cell));
      if (cz + r < p.g.dim[2] - 1) dout = fmin(dout, (p.g.gmin[2] + (double)(cz + r + 1) * p.g.cell) - qz);
      if (dout == 1e300) break;                 // whole grid visited
      dout -= 1e-7 * p.g.cell;                  // guard the cell-boundary rounding of the binning pass
      if (dout > 0.0 && b.d2[7] < dout * dout) break;
    }
  }
  // inverseDistance (calibration_inverter.cpp:55-69), fp32, neighbours in ascending distance; the winners' positions
  // are re-read from the calibration volume through their decoded (x, y, z) index
  float total_weight = 0.0f, wx = 0.0f, wy = 0.0f, wz = 0.0f;
  const uint32_t uZ = (uint32_t)p.cZ, uY = (uint32_t)p.cY;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const uint32_t i = b.idx[k];
    if (i == 0xFFFFFFFFu) continue;
    const uint32_t iz = i % uZ, iy = (i / uZ) % uY, ix = i / (uZ * uY);
    const float4 s = __ldg(p.xyz + ((size_t)iz * uY + iy) * (uint32_t)p.cX + ix);
    const float dx = s.x - sx, dy = s.y - sy, dz = s.z - sz;
    const float weight = 1.0f / sqrtf((dx * dx + dy * dy) + dz * dz);
    wx = wx + (float)ix * weight; wy = wy + (float)iy * weight; wz = wz + (float)iz * weight;
    total_weight += weight;
  }
  wx = wx / total_weight; wy = wy / total_weight; wz = wz / total_weight;
  p.out[o] = make_float4((wx + 0.5f) / p.calib_dims[0], (wy + 0.5f) / p.calib_dims[1], (wz + 0.5f) / p.calib_dims[2], 1.0f);
}

// ---------------------------------------------------------------------------------------------------------- host
int launch_calib_invert(rr_ctx* c, int sensor, const uint32_t out_res[3], float4* d_out) {
  const int X = (int)c->cres[sensor][0], Y = (int)c->cres[sensor][1], Z = (int)c->cres[sensor][2];
  const size_t n = (size_t)X * Y * Z;
  if (n >= 0xFFFFFFFFull) return fail(c, RR_ERR_UNSUPPORTED, "rr_calib_invert: calibration volume too large for 32-bit sample ids");
  // cell grid over the samples' bounding box (computed at rr_calib_upload): ~RR_INVERT_PTS_PER_CELL samples per cell on average
  CellGrid g{};
  static const double target = getenv("RR_INVERT_PTS_PER_CELL") ? atof(getenv("RR_INVERT_PTS_PER_CELL")) : 1.0;
  double vol = 1.0;
  for (int a = 0; a < 3; ++a) vol *= std::max((double)c->xyz_max[sensor][a] - (double)c->xyz_min[sensor][a], 1e-9);
  g.cell = std::cbrt(vol / std::max(1.0, (double)n / target));
  for (;;) {
    double cells = 1.0;
    for (int a = 0; a < 3; ++a) {
      g.gmin[a] = (double)c->xyz_min[sensor][a];
      g.dim[a] = (int)std::max(1.0, std::ceil(((double)c->xyz_max[sensor][a] - g.gmin[a]) / g.cell + 1e-9));
      cells *= g.dim[a];
    }
    if (cells <= 64.0 * 1024 * 1024) break;
    g.cell *= 1.26;
  }
  g.inv_cell = 1.0 / g.cell;
  const size_t ncell = (size_t)g.dim[0] * g.dim[1] * g.dim[2];

  DeviceArray<uint32_t> count, start;
  DeviceArray<float4> sorted;
  DeviceArray<uint8_t> tmp;
  size_t tmp_bytes = 0;
  cudaStream_t s = c->stream;
  RR_TRY_RC(count.allocate(c, ncell + 1, "invert: cell counters"));
  RR_TRY_RC(start.allocate(c, ncell + 1, "invert: cell starts"));
  RR_TRY_RC(sorted.allocate(c, n, "invert: binned samples"));
  uint32_t *d_count = count.ptr, *d_start = start.ptr;
  cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_count, d_start, (int)(ncell + 1), s);
  RR_TRY_RC(tmp.allocate(c, tmp_bytes, "invert: scan scratch"));

  timer_begin(c, "calib_invert");
  cudaMemsetAsync(d_count, 0, (ncell + 1) * sizeof(uint32_t), s);
  const unsigned nb = (unsigned)((n + 255) / 256);
  k_invert_bin<<<nb, 256, 0, s>>>(c->d_xyz[sensor].ptr, X, Y, Z, g, d_count, nullptr);
  ++c->launches;
  cub::DeviceScan::ExclusiveSum(tmp.ptr, tmp_bytes, d_count, d_start, (int)(ncell + 1), s);
  ++c->launches;
  cudaMemcpyAsync(d_count, d_start, (ncell + 1) * sizeof(uint32_t), cudaMemcpyDeviceToDevice, s);   // scatter cursors
  k_invert_bin<<<nb, 256, 0, s>>>(c->d_xyz[sensor].ptr, X, Y, Z, g, d_count, sorted.ptr);
  ++c->launches;

  InvertParams p{};
  p.sorted = sorted.ptr; p.cell_start = d_start; p.g = g; p.xyz = c->d_xyz[sensor].ptr;
  for (int i = 0; i < 6; ++i) for (int k = 0; k < 4; ++k) p.planes[i][k] = c->planes[sensor][i][k];
  for (int a = 0; a < 3; ++a) {
    // calibration_inverter.cpp:100-108, single precision as written
    const float dim = c->bbox_max[a] - c->bbox_min[a];
    const float volume_step = 1.0f / (float)out_res[a];
    p.step[a] = dim * volume_step;
    p.start[a] = c->bbox_min[a] + p.step[a] * 0.5f;
    p.calib_dims[a] = (float)c->cres[sensor][a];
  }
  p.cX = X; p.cY = Y; p.cZ = Z;
  p.ox = (int)out_res[0]; p.oy = (int)out_res[1]; p.oz = (int)out_res[2];
  p.out = d_out;
  if (p.oy > 65535 || p.oz > 65535) return fail(c, RR_ERR_UNSUPPORTED, "rr_calib_invert: output resolution too large");
  const dim3 grd((p.ox + 127) / 128, p.oy, p.oz);
  k_invert<<<grd, 128, 0, s>>>(p);
  ++c->launches;
  timer_end(c, "calib_invert");
  RR_TRY_RC(check(c, cudaGetLastError(), "k_invert"));
  return check(c, cudaStreamSynchronize(s), "invert sync");
}

}  // namespace rr
