// Connected parts of the fused surface on the device: 6-connected labelling of the inside voxels (v > 0, finite) with
// per-part statistics, and the part of every vertex and triangle of the last mesh (rr_label_parts / rr_download_parts /
// rr_download_mesh_parts; the contract is stated in include/rgbd_recon_b200.h and DESIGN.md "Beyond the reference:
// connected parts"). No reference counterpart.
//
// The label array L (uint32 [Z][Y][X]) is a union-find forest over linear voxel indices in which every link points to a
// smaller index (Playne & Hawick, "A new algorithm for parallel connected-component labelling on GPUs", 2018): a root is
// hooked to the smaller root with atomicMin, so a finished root is its part's smallest index, the part's key. Every pass
// is one voxel row (y, z) per warp, lanes along x; in bricks mode only the voxels inside occupied bricks are visited (each
// once: the x masks of the brick rows that contain the row; rr_rows.cuh), otherwise every voxel:
//   memset             L = 0xFFFFFFFF (outside)
//   k_parts_init       L[i] = i for every inside voxel
//   k_parts_merge      union with the inside -x, -y and -z neighbours
//   k_parts_compress   L[i] = root; per row: the roots it holds
//   CUB scan           per-row root offsets and the part count; one read-back, one synchronisation
//   k_parts_number     L[root] = part | 0x80000000 in ascending key order; the part's statistics are reset
//   k_parts_relabel    L[i] = part; counts, boxes and index sums by integer atomics (warp-aggregated)
//   k_parts_finish     per part: half-open box and the centroid in binary64
// Volumes hold fewer than 2^31 voxels (rr_configure), so bit 31 of an index is free for the root mark.
#include "rr_context.h"
#include "rr_rows.cuh"
#include "rr_sample.cuh"

#include <cub/device/device_scan.cuh>

#include <climits>

namespace rr {

namespace {

constexpr uint32_t kOutside = 0xFFFFFFFFu;
constexpr uint32_t kRootMark = 0x80000000u;

struct PartsParams {
  const float* tsdf; int X, Y, Z;   // the sample block of rr_sample.cuh (ld_density)
  int half2;
  uint32_t* L;
  // candidate voxels (use_rows = 0: every voxel): the x masks of the brick rows that contain the voxel row
  int use_rows, rby, mask_words;
  const uint32_t* rowmask; const uint8_t* rowany; const int16_t* cand_y; const int16_t* cand_z;
  // per row (z * Y + y): roots, then their exclusive offsets over rows + 1 entries
  uint32_t* cnt; const uint32_t* off;
  // per part
  uint32_t P;
  uint32_t* voxels; int32_t* boxes; unsigned long long* sums; float* centroids;
  double bmin[3], size[3];
};

__device__ __forceinline__ bool inside_voxel(float v) { return v > 0.0f && v <= 3.402823466e38f; }

__device__ __forceinline__ uint32_t find_root(const uint32_t* L, uint32_t i) {
  uint32_t n = L[i];
  while (n != i) { i = n; n = L[i]; }
  return i;
}

// hook the larger of the two roots to the smaller until both are in one tree
__device__ void unite(uint32_t* L, uint32_t a, uint32_t b) {
  a = find_root(L, a); b = find_root(L, b);
  while (a != b) {
    if (a < b) { const uint32_t t = a; a = b; b = t; }
    const uint32_t old = atomicMin(L + a, b);
    if (old == a) return;
    a = find_root(L, old); b = find_root(L, b);
  }
}

#define RR_PARTS_ROW                                                   \
  const unsigned r = blockIdx.x * 8u + (threadIdx.x >> 5);             \
  if (r >= (unsigned)p.Y * (unsigned)p.Z) return;

__global__ void __launch_bounds__(256) k_parts_init(const __grid_constant__ PartsParams p) {
  RR_PARTS_ROW
  walk_row(p, r, [&](int, int, int, uint32_t i, bool cand, unsigned) {
    if (cand && inside_voxel(ld_density(p, i))) p.L[i] = i;
  });
}

__global__ void __launch_bounds__(256) k_parts_merge(const __grid_constant__ PartsParams p) {
  RR_PARTS_ROW
  const uint32_t sy = (uint32_t)p.X, sz = (uint32_t)p.X * (uint32_t)p.Y;
  walk_row(p, r, [&](int x, int y, int z, uint32_t i, bool cand, unsigned) {
    if (!cand || p.L[i] == kOutside) return;
    // an outside neighbour is 0xFFFFFFFF for good (outside every occupied brick too), an inside one is initialised
    if (x > 0 && p.L[i - 1] != kOutside) unite(p.L, i, i - 1);
    if (y > 0 && p.L[i - sy] != kOutside) unite(p.L, i, i - sy);
    if (z > 0 && p.L[i - sz] != kOutside) unite(p.L, i, i - sz);
  });
}

__global__ void __launch_bounds__(256) k_parts_compress(const __grid_constant__ PartsParams p) {
  RR_PARTS_ROW
  unsigned roots = 0;
  walk_row(p, r, [&](int, int, int, uint32_t i, bool cand, unsigned) {
    bool root = false;
    if (cand && p.L[i] != kOutside) {
      const uint32_t k = find_root(p.L, i);
      p.L[i] = k;
      root = k == i;
    }
    roots += __popc(__ballot_sync(0xffffffffu, root));
  });
  if ((threadIdx.x & 31u) == 0) p.cnt[r] = roots;
}

__global__ void __launch_bounds__(256) k_parts_number(const __grid_constant__ PartsParams p) {
  RR_PARTS_ROW
  uint32_t base = p.off[r];
  if (p.off[r + 1] == base) return;
  const unsigned lane = threadIdx.x & 31u;
  walk_row(p, r, [&](int, int, int, uint32_t i, bool cand, unsigned) {
    const bool root = cand && p.L[i] == i;
    const uint32_t b = __ballot_sync(0xffffffffu, root);
    if (root) {
      const uint32_t part = base + __popc(b & ((1u << lane) - 1u));
      p.L[i] = part | kRootMark;
      p.voxels[part] = 0;
      int32_t* bx = p.boxes + (size_t)part * 6;
      bx[0] = bx[2] = bx[4] = INT_MAX; bx[1] = bx[3] = bx[5] = INT_MIN;
      unsigned long long* s = p.sums + (size_t)part * 3;
      s[0] = s[1] = s[2] = 0ull;
    }
    base += __popc(b);
  });
}

struct PartAcc {
  uint32_t part, n;
  int x0, x1, y0, y1, z0, z1;
  unsigned long long sx, sy, sz;
};

__device__ __forceinline__ void flush(const PartsParams& p, const PartAcc& a) {
  atomicAdd(p.voxels + a.part, a.n);
  int32_t* bx = p.boxes + (size_t)a.part * 6;
  atomicMin(bx + 0, a.x0); atomicMax(bx + 1, a.x1);
  atomicMin(bx + 2, a.y0); atomicMax(bx + 3, a.y1);
  atomicMin(bx + 4, a.z0); atomicMax(bx + 5, a.z1);
  unsigned long long* s = p.sums + (size_t)a.part * 3;
  atomicAdd(s + 0, a.sx); atomicAdd(s + 1, a.sy); atomicAdd(s + 2, a.sz);
}

// Statistics are gathered per warp: the lanes of one part in a 32-voxel word are reduced by ballots, and the warp keeps a
// running sum for the last part it saw, flushed by lane 0 when another part comes up (integer atomics only: the totals do
// not depend on the order).
__global__ void __launch_bounds__(256) k_parts_relabel(const __grid_constant__ PartsParams p) {
  RR_PARTS_ROW
  const unsigned lane = threadIdx.x & 31u;
  PartAcc acc{kOutside, 0, 0, 0, 0, 0, 0, 0, 0ull, 0ull, 0ull};
  walk_row(p, r, [&](int, int y, int z, uint32_t i, bool cand, unsigned x0) {
    uint32_t part = kOutside;
    if (cand) {
      const uint32_t v = p.L[i];
      if (v != kOutside) {
        part = (v & kRootMark) ? (v & ~kRootMark) : (p.L[v] & ~kRootMark);   // a root's mark is read with or without it
        p.L[i] = part;
      }
    }
    uint32_t todo = __ballot_sync(0xffffffffu, part != kOutside);
    while (todo) {
      const uint32_t q = __shfl_sync(0xffffffffu, part, __ffs(todo) - 1);
      const uint32_t grp = __ballot_sync(0xffffffffu, part == q);
      todo &= ~grp;
      if (q != acc.part) {
        if (acc.part != kOutside && lane == 0) flush(p, acc);
        acc = PartAcc{q, 0, INT_MAX, INT_MIN, INT_MAX, INT_MIN, INT_MAX, INT_MIN, 0ull, 0ull, 0ull};
      }
      const uint32_t n = __popc(grp);
      const unsigned lo = __ffs(grp) - 1, hi = 31 - __clz(grp);
      const unsigned lanesum = __reduce_add_sync(0xffffffffu, (grp >> lane) & 1u ? lane : 0u);
      acc.n += n;
      acc.x0 = min(acc.x0, (int)(x0 + lo)); acc.x1 = max(acc.x1, (int)(x0 + hi));
      acc.y0 = min(acc.y0, y); acc.y1 = max(acc.y1, y);
      acc.z0 = min(acc.z0, z); acc.z1 = max(acc.z1, z);
      acc.sx += (unsigned long long)n * x0 + lanesum;
      acc.sy += (unsigned long long)n * (unsigned)y;
      acc.sz += (unsigned long long)n * (unsigned)z;
    }
  });
  if (acc.part != kOutside && lane == 0) flush(p, acc);
}

// c_k = (float)(bmin_k + ((S_k / n) + 0.5) / R_k * (bmax_k - bmin_k)) in binary64, no fused multiply-add (--fmad=false)
__global__ void __launch_bounds__(128) k_parts_finish(const __grid_constant__ PartsParams p) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= p.P) return;
  const double n = (double)p.voxels[k];
  const int R[3] = {p.X, p.Y, p.Z};
  int32_t* bx = p.boxes + (size_t)k * 6;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    bx[2 * a + 1] += 1;
    const double s = (double)p.sums[(size_t)k * 3 + a];
    p.centroids[(size_t)k * 3 + a] = (float)(p.bmin[a] + ((s / n) + 0.5) / (double)R[a] * p.size[a]);
  }
}

__global__ void __launch_bounds__(128) k_mesh_vertex_parts(const unsigned long long* __restrict__ keys, uint32_t nv, int X, int Y,
                                                           const uint32_t* __restrict__ L, uint32_t* __restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nv) return;
  const unsigned long long key = keys[i];
  const uint32_t a = (uint32_t)(key / 3ull);
  const int k = (int)(key - (unsigned long long)a * 3ull);
  const uint32_t b = a + (k == 0 ? 1u : (k == 1 ? (uint32_t)X : (uint32_t)X * (uint32_t)Y));
  const uint32_t la = L[a];
  out[i] = la != kOutside ? la : L[b];   // exactly one end is inside (the mesh's vertex rule)
}

__global__ void __launch_bounds__(128) k_mesh_triangle_parts(const uint32_t* __restrict__ tri, uint32_t nt,
                                                             const uint32_t* __restrict__ vparts, uint32_t* __restrict__ out) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < nt) out[t] = vparts[tri[(size_t)t * 3]];
}

}  // namespace

int launch_label_parts(rr_ctx* c, int dest, uint32_t* out_num_parts) {
  const int X = (int)c->res[0], Y = (int)c->res[1], Z = (int)c->res[2];
  const size_t nvox = (size_t)X * Y * Z, rows = (size_t)Y * Z;
  c->parts_valid = false;
  RR_TRY_RC(c->d_parts_labels[dest].reserve(c, nvox, "part labels"));
  RR_TRY_RC(c->d_parts_rows.reserve(c, 2 * (rows + 1), "part row counts"));
  uint32_t* cnt = c->d_parts_rows.ptr;
  uint32_t* off = cnt + (rows + 1);
  size_t scan_bytes = 0;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, cnt, off, (int)(rows + 1), c->stream), "part scan size"));
  RR_TRY_RC(c->d_parts_scratch.reserve(c, scan_bytes, "part scan scratch"));

  PartsParams p{};
  p.tsdf = c->d_tsdf.ptr; p.X = X; p.Y = Y; p.Z = Z;
  p.half2 = c->cfg.store_weight == RR_VOXELS_HALF2 ? 1 : 0;
  p.L = c->d_parts_labels[dest].ptr;
  p.use_rows = c->mesh_rows_ok ? 1 : 0;
  p.rby = (int)c->bricks.res[1]; p.mask_words = c->mask_words;
  p.rowmask = c->d_rowmask.ptr; p.rowany = c->d_rowany.ptr; p.cand_y = c->d_cand_y.ptr; p.cand_z = c->d_cand_z.ptr;
  p.cnt = cnt; p.off = off;
  for (int a = 0; a < 3; ++a) {
    p.bmin[a] = (double)c->bbox_min[a];
    p.size[a] = (double)c->bbox_max[a] - (double)c->bbox_min[a];
  }

  const unsigned row_blocks = (unsigned)((rows + 7) / 8);
  RR_TRY_RC(check(c, cudaMemsetAsync(p.L, 0xFF, nvox * sizeof(uint32_t), c->stream), "part labels reset"));
  RR_TRY_RC(check(c, cudaMemsetAsync(cnt + rows, 0, sizeof(uint32_t), c->stream), "part counts"));
  k_parts_init<<<row_blocks, 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_parts_init");
  k_parts_merge<<<row_blocks, 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_parts_merge");
  k_parts_compress<<<row_blocks, 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_parts_compress");
  size_t bytes = c->d_parts_scratch.cap;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(c->d_parts_scratch.ptr, bytes, cnt, off, (int)(rows + 1), c->stream), "part scan"));
  c->launches += 1;
  RR_TRY_RC(check(c, cudaMemcpyAsync(&c->pinned->parts_count, off + rows, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream), "part count"));
  RR_TRY_RC(check(c, cudaStreamSynchronize(c->stream), "part count sync"));
  const uint32_t np = c->pinned->parts_count;
  RR_TRY_RC(c->d_parts_voxels.reserve(c, np, "part voxel counts"));
  RR_TRY_RC(c->d_parts_boxes.reserve(c, 6 * (size_t)np, "part boxes"));
  RR_TRY_RC(c->d_parts_sums.reserve(c, 3 * (size_t)np, "part index sums"));
  RR_TRY_RC(c->d_parts_centroids.reserve(c, 3 * (size_t)np, "part centroids"));
  p.P = np;
  p.voxels = c->d_parts_voxels.ptr; p.boxes = c->d_parts_boxes.ptr; p.sums = c->d_parts_sums.ptr; p.centroids = c->d_parts_centroids.ptr;
  if (np) {
    k_parts_number<<<row_blocks, 256, 0, c->stream>>>(p);
    RR_LAUNCH_CHECK(c, "k_parts_number");
    k_parts_relabel<<<row_blocks, 256, 0, c->stream>>>(p);
    RR_LAUNCH_CHECK(c, "k_parts_relabel");
    k_parts_finish<<<(np + 127) / 128, 128, 0, c->stream>>>(p);
    RR_LAUNCH_CHECK(c, "k_parts_finish");
  }
  c->parts_n = np;
  c->parts_cur = dest;
  c->parts_epoch = c->volume_epoch;
  c->parts_valid = true;
  *out_num_parts = np;
  return RR_OK;
}

int parts_download(rr_ctx* c, uint32_t* voxels, int32_t* boxes, float* centroids, uint32_t* labels) {
  const size_t np = c->parts_n, nvox = (size_t)c->res[0] * c->res[1] * c->res[2];
  if (voxels && np) RR_TRY_RC(check(c, cudaMemcpyAsync(voxels, c->d_parts_voxels.ptr, np * sizeof(uint32_t), cudaMemcpyDefault, c->stream), "part download"));
  if (boxes && np) RR_TRY_RC(check(c, cudaMemcpyAsync(boxes, c->d_parts_boxes.ptr, np * 6 * sizeof(int32_t), cudaMemcpyDefault, c->stream), "part download"));
  if (centroids && np) RR_TRY_RC(check(c, cudaMemcpyAsync(centroids, c->d_parts_centroids.ptr, np * 3 * sizeof(float), cudaMemcpyDefault, c->stream), "part download"));
  if (labels) RR_TRY_RC(check(c, cudaMemcpyAsync(labels, c->d_parts_labels[c->parts_cur].ptr, nvox * sizeof(uint32_t), cudaMemcpyDefault, c->stream), "label download"));
  return check(c, cudaStreamSynchronize(c->stream), "part download sync");
}

int mesh_parts_download(rr_ctx* c, uint32_t* vertex_parts, uint32_t* triangle_parts) {
  const uint32_t nv = c->mesh_nv, nt = c->mesh_nt;
  RR_TRY_RC(c->d_mesh_parts.reserve(c, (size_t)nv + nt, "mesh part buffers"));
  uint32_t* vp = c->d_mesh_parts.ptr;
  uint32_t* tp = vp + nv;
  if (nv) {
    k_mesh_vertex_parts<<<(nv + 127) / 128, 128, 0, c->stream>>>(c->d_mesh_keys.ptr, nv, (int)c->res[0], (int)c->res[1],
                                                                 c->d_parts_labels[c->parts_cur].ptr, vp);
    RR_LAUNCH_CHECK(c, "k_mesh_vertex_parts");
  }
  if (nt) {
    k_mesh_triangle_parts<<<(nt + 127) / 128, 128, 0, c->stream>>>(c->d_mesh_tri.ptr, nt, vp, tp);
    RR_LAUNCH_CHECK(c, "k_mesh_triangle_parts");
  }
  if (vertex_parts && nv) RR_TRY_RC(check(c, cudaMemcpyAsync(vertex_parts, vp, (size_t)nv * sizeof(uint32_t), cudaMemcpyDefault, c->stream), "mesh part download"));
  if (triangle_parts && nt) RR_TRY_RC(check(c, cudaMemcpyAsync(triangle_parts, tp, (size_t)nt * sizeof(uint32_t), cudaMemcpyDefault, c->stream), "mesh part download"));
  return check(c, cudaStreamSynchronize(c->stream), "mesh part download sync");
}

}  // namespace rr
