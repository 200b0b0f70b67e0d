// Removing connected parts from the fused volume on the device (rr_remove_parts / rr_group_remove_parts; the contract is
// stated in include/rgbd_recon_b200.h and DESIGN.md "Beyond the reference: removing parts"). No reference counterpart.
//
// The call rewrites the voxels of the chosen parts of the last labelling (rr_parts.cu) to the voxel the bricks-mode clear
// writes, so every consumer of the volume sees the cleaned volume through its own code path:
//   memset            the counters
//   k_remove_flags    per part p: removed iff voxels[p] < min_voxels or keep[p] == 0; the rows of a removed part's box
//                     (0 for a kept part); warp-aggregated counts of the removed parts and their voxels
//   CUB scan          the rows' exclusive offsets over P + 1 entries: work item w is row w - off[p] of part p's box
//   k_remove_voxels   per destination volume (a group member's slab and halo rows [z0, z1)): a warp per work item, lanes
//                     along x, stores the cleared voxel where label == p
// The work follows the removed parts' boxes, not the volume: a box holds every voxel of its part, so walking the boxes finds
// every removed voxel whatever their size (a box can never be larger than the volume; only overlapping boxes of many large
// removed parts could add up to more than one pass over it). Every store writes the same value, so overlapping boxes and
// the order of the warps do not change the result. The counts are read back with the call's one synchronisation.
#include "rr_context.h"
#include "rr_integrate.cuh"

#include <cub/device/device_scan.cuh>

#include <cstring>

namespace rr {

namespace {

constexpr unsigned kRemoveWarps = 8;   // warps per CTA of k_remove_voxels

// counts[0] removed parts, [1] their voxels (the volume holds fewer than 2^31 voxels)
__global__ void __launch_bounds__(256) k_remove_flags(uint32_t P, const uint32_t* __restrict__ voxels,
                                                      const int32_t* __restrict__ boxes, const uint8_t* __restrict__ keep,
                                                      uint32_t min_voxels, unsigned long long* __restrict__ rows,
                                                      uint32_t* __restrict__ counts) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t n = 0;
  unsigned long long box_rows = 0;
  bool removed = false;
  if (k < P) {
    n = voxels[k];
    removed = n < min_voxels || (keep && keep[k] == 0);
    if (removed) {
      const int32_t* b = boxes + (size_t)k * 6;
      box_rows = (unsigned long long)(b[3] - b[2]) * (unsigned long long)(b[5] - b[4]);
    } else {
      n = 0;
    }
  }
  if (k < P + 1) rows[k] = box_rows;   // rows[P] = 0: the scan's last entry is the item count
  const unsigned parts = __reduce_add_sync(0xffffffffu, removed ? 1u : 0u);
  const unsigned vox = __reduce_add_sync(0xffffffffu, n);
  if ((threadIdx.x & 31u) == 0 && parts) {
    atomicAdd(counts + 0, parts);
    atomicAdd(counts + 1, vox);
  }
}

struct RemoveParams {
  int X, Y;
  const uint32_t* L;                   // labels
  uint32_t P;
  const unsigned long long* off;       // per part, exclusive offsets of the removed box rows, P + 1 entries (64-bit: the
                                       // boxes of many removed parts may hold more rows than 2^32 together)
  const int32_t* boxes;
  int z0, z1;                          // destination rows
  uint32_t* tsdf;                      // destination volume: the cleared voxel's 4 bytes
  float* weight;                       // destination weight volume (F32_WEIGHT), or null: 0
  uint32_t fill;
};

__global__ void __launch_bounds__(256) k_remove_voxels(const __grid_constant__ RemoveParams p) {
  const unsigned lane = threadIdx.x & 31u;
  const unsigned warp = blockIdx.x * kRemoveWarps + (threadIdx.x >> 5), nwarps = gridDim.x * kRemoveWarps;
  const unsigned long long items = p.off[p.P];
  for (unsigned long long w = warp; w < items; w += nwarps) {
    uint32_t lo = 0, hi = p.P;            // the part whose rows hold item w: the last p with off[p] <= w
    while (hi - lo > 1) {
      const uint32_t mid = (lo + hi) >> 1;
      if (p.off[mid] <= w) lo = mid; else hi = mid;
    }
    const int32_t* b = p.boxes + (size_t)lo * 6;
    const unsigned long long k = w - p.off[lo], by = (unsigned long long)(b[3] - b[2]);
    const int y = b[2] + (int)(k % by), z = b[4] + (int)(k / by);
    if (z < p.z0 || z >= p.z1) continue;
    const uint32_t row = ((uint32_t)z * (uint32_t)p.Y + (uint32_t)y) * (uint32_t)p.X;
    for (int x = b[0] + (int)lane; x < b[1]; x += 32) {
      const uint32_t i = row + (uint32_t)x;
      if (p.L[i] == lo) {
        p.tsdf[i] = p.fill;
        if (p.weight) p.weight[i] = 0.0f;
      }
    }
  }
}

}  // namespace

int remove_parts(rr_ctx* c, rr_ctx* const* members, int n, uint32_t min_voxels, const uint8_t* keep, uint32_t* out_parts,
                 uint32_t* out_voxels) {
  const uint32_t P = c->parts_n;
  RR_TRY_RC(c->d_remove_rows.reserve(c, 2 * ((size_t)P + 1), "removal rows"));
  if (!c->d_remove_counts.ptr) RR_TRY_RC(c->d_remove_counts.allocate(c, 2, "removal counts"));
  unsigned long long* rows = c->d_remove_rows.ptr;
  unsigned long long* off = rows + (P + 1);
  size_t scan_bytes = 0;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, rows, off, (int)(P + 1), c->stream), "removal scan size"));
  RR_TRY_RC(c->d_remove_scratch.reserve(c, scan_bytes, "removal scan scratch"));
  const uint8_t* d_keep = nullptr;
  if (keep && P) {
    RR_TRY_RC(c->d_remove_keep.reserve(c, P, "keep flags"));
    RR_TRY_RC(check(c, cudaMemcpyAsync(c->d_remove_keep.ptr, keep, P, cudaMemcpyDefault, c->stream), "keep flags copy"));
    d_keep = c->d_remove_keep.ptr;
  }
  RR_TRY_RC(check(c, cudaMemsetAsync(c->d_remove_counts.ptr, 0, 2 * sizeof(uint32_t), c->stream), "removal counts"));
  k_remove_flags<<<(P + 256) / 256, 256, 0, c->stream>>>(P, c->d_parts_voxels.ptr, c->d_parts_boxes.ptr, d_keep, min_voxels,
                                                         rows, c->d_remove_counts.ptr);
  RR_LAUNCH_CHECK(c, "k_remove_flags");
  size_t bytes = c->d_remove_scratch.cap;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(c->d_remove_scratch.ptr, bytes, rows, off, (int)(P + 1), c->stream), "removal scan"));
  c->launches += 1;

  RemoveParams p{};
  p.X = (int)c->res[0]; p.Y = (int)c->res[1];
  p.L = c->d_parts_labels[c->parts_cur].ptr;
  p.P = P; p.off = off; p.boxes = c->d_parts_boxes.ptr;
  for (int i = 0; i < n && P; ++i) {
    const rr_ctx* m = members[i];
    const ClearState rowset = integrate_clear_key(m);   // the rows the member's integrate writes: its slab and halo
    p.z0 = rowset.z0; p.z1 = rowset.z1;
    p.tsdf = reinterpret_cast<uint32_t*>(m->d_tsdf.ptr);
    p.weight = m->d_weight.ptr;
    const float f = cleared_voxel(rowset.mode, m->cfg.limit);
    std::memcpy(&p.fill, &f, sizeof(f));
    k_remove_voxels<<<(unsigned)c->num_sms * 8u, 256, 0, c->stream>>>(p);
    RR_LAUNCH_CHECK(c, "k_remove_voxels");
  }
  RR_TRY_RC(check(c, cudaMemcpyAsync(c->pinned->remove_counts, c->d_remove_counts.ptr, 2 * sizeof(uint32_t),
                                     cudaMemcpyDeviceToHost, c->stream), "removal counts"));
  RR_TRY_RC(check(c, cudaStreamSynchronize(c->stream), "removal sync"));
  *out_parts = c->pinned->remove_counts[0];
  *out_voxels = c->pinned->remove_counts[1];
  // a new volume state when anything changed: the mesh, labelling and distance field taken before are of the old one
  if (*out_parts)
    for (int i = 0; i < n; ++i) ++members[i]->volume_epoch;
  return RR_OK;
}

}  // namespace rr
