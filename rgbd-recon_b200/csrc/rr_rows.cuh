// One warp per voxel row (y, z), lanes along x: the work domain of the passes over the whole volume that rr_parts.cu and
// rr_track.cu share. In bricks mode only the voxels inside occupied bricks are visited (each once: the x masks of the brick
// rows that contain the row), otherwise every voxel.
// P is the caller's parameter block; it provides
//   X, Y                                           the volume's row length and rows per slice
//   use_rows (0: every voxel), rby, mask_words,    the brick row tables of the last integrate (rr_context.h)
//   rowmask, rowany, cand_y, cand_z
#pragma once

#include <stdint.h>

namespace rr {

// the candidate voxels of word w (x = 32 w + lane) of row (y, z)
template <class P>
__device__ __forceinline__ uint32_t row_word(const P& p, int y, int z, int w) {
  const int rem = p.X - 32 * w;
  const uint32_t all = rem >= 32 ? 0xFFFFFFFFu : ((1u << rem) - 1u);
  if (!p.use_rows) return all;
  uint32_t m = 0;
  for (int a = 0; a < 2; ++a) {
    const int by = p.cand_y[2 * y + a];
    if (by < 0) continue;
    for (int b = 0; b < 2; ++b) {
      const int bz = p.cand_z[2 * z + b];
      if (bz >= 0) m |= p.rowmask[((size_t)bz * p.rby + by) * p.mask_words + w];
    }
  }
  return m & all;
}

template <class P>
__device__ __forceinline__ bool row_any(const P& p, int y, int z) {
  if (!p.use_rows) return true;
  for (int a = 0; a < 2; ++a) {
    const int by = p.cand_y[2 * y + a];
    if (by < 0) continue;
    for (int b = 0; b < 2; ++b) {
      const int bz = p.cand_z[2 * z + b];
      if (bz >= 0 && p.rowany[bz * p.rby + by]) return true;
    }
  }
  return false;
}

// Each pass: warp = row r, the body runs for every lane (all 32 lanes, uniform control flow) with the lane's voxel and
// whether it is a candidate.
template <class P, class F>
__device__ __forceinline__ void walk_row(const P& p, unsigned r, F&& body) {
  const unsigned lane = threadIdx.x & 31u;
  const int y = (int)(r % (unsigned)p.Y), z = (int)(r / (unsigned)p.Y);
  if (!row_any(p, y, z)) return;
  const unsigned nw = ((unsigned)p.X + 31u) / 32u;
  for (unsigned w = 0; w < nw; ++w) {
    const uint32_t m = row_word(p, y, z, (int)w);
    if (!m) continue;
    const int x = (int)(w * 32u + lane);
    body(x, y, z, ((unsigned)z * (unsigned)p.Y + (unsigned)y) * (unsigned)p.X + (unsigned)x, ((m >> lane) & 1u) != 0, w * 32u);
  }
}

}  // namespace rr
