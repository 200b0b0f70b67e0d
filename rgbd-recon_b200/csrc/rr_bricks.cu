// Brick occupancy on the device: ReconIntegration::clearOccupiedBricks / updateOccupiedBricks
// (framework/reconstruction/recon_integration.cpp:272-278, 431-446) without the GPU->CPU->GPU round trip.
// The occupied list must equal the CPU loop's order (ascending brick id), so the compaction is an ORDERED
// ballot + prefix scan by a single 1024-thread block (a brick grid is ~10^4 counters: one block is latency-optimal).
#include "rr_integrate.cuh"

namespace rr {

// Ordered compaction by one 1024-thread block: every thread owns a contiguous run of brick ids, counts its occupied
// ones, a block-wide exclusive scan (warp shuffles + one shared-memory hop) gives its output offset, and it writes its ids
// in ascending order. One pass over the counters, two barriers.
__device__ void bricks_compact_block(const uint32_t* __restrict__ counters, uint32_t num_bricks, uint32_t min_voxels,
                                     uint32_t* __restrict__ occupied, uint32_t* __restrict__ num_occupied) {
  __shared__ uint32_t warp_sums[32];
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t per = (num_bricks + 1023u) / 1024u;
  const uint32_t i0 = min(threadIdx.x * per, num_bricks), i1 = min(i0 + per, num_bricks);
  uint32_t mine = 0;
  for (uint32_t i = i0; i < i1; ++i) mine += (counters[i] >= min_voxels) ? 1u : 0u;
  uint32_t incl = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
    if ((int)lane >= d) incl += v;
  }
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = warp_sums[lane];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, w, d);
      if ((int)lane >= d) w += v;
    }
    warp_sums[lane] = w;                      // inclusive sums of the warp totals
  }
  __syncthreads();
  uint32_t out = (warp ? warp_sums[warp - 1] : 0u) + incl - mine;
  for (uint32_t i = i0; i < i1; ++i)
    if (counters[i] >= min_voxels) occupied[out++] = i;
  if (threadIdx.x == 1023) *num_occupied = warp_sums[31];
}

// Per-brick and per-brick-row masks derived from the counters (one launch):
//   near_occ[b] = 1 if brick b or any of its 26 neighbours is occupied: the raymarcher may skip the TSDF fetches of
//     samples inside bricks with near_occ == 0 (every trilinear tap there still holds the cleared value -limit);
//   occ_mask[b] = brick b is occupied;
//   rowmask[bz][by][w] = bit x set iff voxel column x lies inside the x range of an occupied brick of row (by, bz);
//   rowany[bz][by]     = the row has an occupied brick  (both read by the fused clear+integrate kernel).
// Block 0 performs the ordered compaction (updateOccupiedBricks), the other blocks build the masks: one launch.
__global__ void __launch_bounds__(1024) k_bricks_update(const uint32_t* __restrict__ counters, uint32_t num_bricks, uint32_t rx, uint32_t ry,
                                                        uint32_t rz, uint32_t min_voxels, const int32_t* __restrict__ ranges, int mask_words,
                                                        uint32_t* __restrict__ occupied, uint32_t* __restrict__ num_occupied,
                                                        uint8_t* __restrict__ near_occ, uint8_t* __restrict__ occ_mask,
                                                        uint32_t* __restrict__ rowmask, uint8_t* __restrict__ rowany,
                                                        uint32_t* __restrict__ work, uint32_t mask_blocks, const __grid_constant__ ClassifyParams cq) {
  if (blockIdx.x == 0) {
    if (threadIdx.x < 4) work[threadIdx.x] = 0;          // work counters of the persistent integrators (this frame's launch)
    bricks_compact_block(counters, num_bricks, min_voxels, occupied, num_occupied);
    return;
  }
  if (blockIdx.x > mask_blocks) {
    // verdict blocks (staged integrator): one warp per work item of every brick, idle unless the brick is occupied
    const uint32_t w = (blockIdx.x - 1 - mask_blocks) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t brick = w / (uint32_t)cq.per_brick;
    if (brick >= num_bricks || counters[brick] < min_voxels) return;
    classify_item(cq, brick, w - brick * (uint32_t)cq.per_brick, threadIdx.x & 31);
    return;
  }
  if (near_occ == nullptr) return;
  const uint32_t i = (blockIdx.x - 1) * blockDim.x + threadIdx.x;
  if (i < rx * ry * rz) {
    const int bx = (int)(i % rx), by = (int)((i / rx) % ry), bz = (int)(i / (rx * ry));
    uint8_t any = 0;
    for (int dz = -1; dz <= 1; ++dz)
      for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx) {
          const int x = bx + dx, y = by + dy, z = bz + dz;
          if (x < 0 || y < 0 || z < 0 || x >= (int)rx || y >= (int)ry || z >= (int)rz) continue;
          if (counters[((size_t)z * ry + y) * rx + x] >= min_voxels) any = 1;
        }
    near_occ[i] = any;
    occ_mask[i] = counters[i] >= min_voxels ? 1 : 0;
  }
  if (rowmask && i < ry * rz * (uint32_t)mask_words) {
    const uint32_t row = i / (uint32_t)mask_words, w = i - row * (uint32_t)mask_words;
    const int w0 = (int)(w * 32u);
    uint32_t m = 0, any = 0;
    for (uint32_t bx = 0; bx < rx; ++bx) {
      if (counters[(size_t)row * rx + bx] < min_voxels) continue;
      any = 1;
      const int lo = max(ranges[bx * 6] - w0, 0), hi = min(ranges[bx * 6 + 1] - w0, 32);   // x range of brick (bx, 0, 0)
      if (lo < hi) m |= (hi - lo == 32) ? 0xFFFFFFFFu : (((1u << (hi - lo)) - 1u) << lo);
    }
    rowmask[i] = m;
    if (w == 0) rowany[row] = (uint8_t)any;
  }
}

int launch_bricks_clear(rr_ctx* c) {
  cudaError_t e = cudaMemsetAsync(c->d_counters.ptr, 0, sizeof(uint32_t) * ((size_t)c->bricks.num + RR_CLASS_COUNTERS), c->stream);
  c->sti.lists_key = 0;
  return check(c, e, "bricks clear");
}

int launch_bricks_update(rr_ctx* c) {
  const uint32_t nb = c->bricks.num;
  const bool grid_ok = nb == c->bricks.res[0] * c->bricks.res[1] * c->bricks.res[2];
  const uint32_t rows_words = (grid_ok && c->fused_ok) ? c->bricks.res[1] * c->bricks.res[2] * (uint32_t)c->mask_words : 0u;
  const uint32_t threads = grid_ok ? (nb > rows_words ? nb : rows_words) : 0u;
  const uint32_t mask_blocks = (threads + 1023) / 1024;
  // the staged integrator's per-frame verdicts ride along (the pair image is complete: k_quality ran before this)
  ClassifyParams cq{};
  RR_TRY_RC(staged_prepare(c));
  const bool classify = staged_classify_params(c, cq);
  const uint32_t cls_blocks = classify ? (nb * (uint32_t)cq.per_brick + 31u) / 32u : 0u;
  timer_begin(c, "bricks");
  k_bricks_update<<<1 + mask_blocks + cls_blocks, 1024, 0, c->stream>>>(
      c->d_counters.ptr, nb, c->bricks.res[0], c->bricks.res[1], c->bricks.res[2], c->cfg.min_voxels_per_brick, c->d_ranges.ptr, c->mask_words,
      c->d_occupied.ptr, c->d_num_occ.ptr, grid_ok ? c->d_near_occ.ptr : nullptr, c->d_occ_mask.ptr, (grid_ok && c->fused_ok) ? c->d_rowmask.ptr : nullptr, c->d_rowany.ptr,
      c->d_work.ptr, mask_blocks, cq);
  RR_LAUNCH_CHECK(c, "k_bricks_update");
  timer_end(c, "bricks");
  c->work_fresh = true;
  c->mesh_rows_ok = false;     // new row tables: the volume was cleared by the previous ones
  if (classify) c->sti.lists_key = staged_lists_key(c);
  cudaError_t e = cudaMemcpyAsync(&c->pinned->num_occ, c->d_num_occ.ptr, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream);
  return check(c, e, "bricks count copy");
}

}  // namespace rr
