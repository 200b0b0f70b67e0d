// Surface extraction on the device: marching cubes over the TSDF volume into an indexed, coloured triangle mesh
// (rr_extract_mesh / rr_download_mesh; the contract is stated in include/rgbd_recon_b200.h and DESIGN.md "Beyond the
// reference: surface extraction"). No reference counterpart: the reference only raymarches the volume.
//
// Work is one voxel row (y, z) per warp, lanes along x. A row owns the vertices on the edges whose lower corner lies in it
// and the triangles of the cells whose lower corner lies in it, so every count, scan and write is in the canonical order
// (vertices by edge key, triangles by cell, then table order) whatever the scheduling:
//   k_mesh_count       per row: owned vertices and triangles (rows no occupied brick reaches are skipped when the brick
//                      row tables are the ones the volume was integrated with)
//   two CUB scans      per-row offsets and the totals; one 16-byte read-back, one synchronisation
//   k_mesh_vertices    per row: edge keys and positions
//   k_mesh_attributes  per vertex: gradient normal (6 trilinear taps) and blendColors (N sensor lookups)
//   k_mesh_triangles   per row: vertex indices by binary search of the owning row's key segment
#include "rr_context.h"
#include "rr_sample.cuh"

#include <cub/device/device_scan.cuh>

#include <cmath>
#include <cstring>

namespace rr {

namespace {

constexpr int kMaxCellTris = 5;      // most triangles any case of the table needs (checked when the table is built)

struct MeshTable {
  uint8_t ntri[256];
  uint8_t tri[256][kMaxCellTris * 3];   // cube edges, three per triangle
};

__constant__ MeshTable kMesh;

// Cube corner c = (c & 1, c >> 1 & 1, c >> 2 & 1). Edge e runs along axis k = e / 4 from the corner whose other two
// coordinates (u, w) are (e & 1, e >> 1 & 1), u < w being the two other axes in x, y, z order.
__host__ __device__ inline int edge_lower_corner(int e) {
  const int k = e >> 2, j = e & 3;
  const int u = k == 0 ? 1 : 0, w = k == 2 ? 1 : 2;
  return ((j & 1) << u) | ((j >> 1) << w);
}

// The case table, generated from the face rule (DESIGN.md): on every cube face, two crossed edges give one segment and
// four crossed edges give the two segments that cut off the inside corners; segments are oriented so that the loop runs
// counter-clockwise seen from the outside (v <= 0) side, chained into loops and fanned from each loop's lowest edge.
bool build_case_table(MeshTable& t) {
  std::memset(&t, 0, sizeof(t));
  for (int cs = 0; cs < 256; ++cs) {
    auto inside = [&](int c) { return (cs >> c) & 1; };
    auto pos = [](int c, int a) { return (double)((c >> a) & 1); };
    int edge_of[8][8];
    for (int e = 0; e < 12; ++e) {
      const int a = edge_lower_corner(e), b = a | (1 << (e >> 2));
      edge_of[a][b] = edge_of[b][a] = e;
    }
    auto mid = [&](int e, double* m) {
      const int a = edge_lower_corner(e);
      for (int ax = 0; ax < 3; ++ax) m[ax] = pos(a, ax) + (ax == (e >> 2) ? 0.5 : 0.0);
    };
    int next[12], nin[12];
    for (int e = 0; e < 12; ++e) { next[e] = -1; nin[e] = 0; }
    for (int k = 0; k < 3; ++k)
      for (int s = 0; s < 2; ++s) {
        const int u = k == 0 ? 1 : 0, w = k == 2 ? 1 : 2;
        const int base = s << k;
        const int cyc[4] = {base, base | (1 << u), base | (1 << u) | (1 << w), base | (1 << w)};
        int crossed = 0;
        for (int i = 0; i < 4; ++i) crossed += inside(cyc[i]) != inside(cyc[(i + 1) & 3]);
        // segments as (edge a, edge b, inside reference point)
        int seg[2][2]; double ref[2][3]; int nseg = 0;
        if (crossed == 2) {
          int ce[2], n = 0;
          for (int i = 0; i < 4; ++i)
            if (inside(cyc[i]) != inside(cyc[(i + 1) & 3])) ce[n++] = edge_of[cyc[i]][cyc[(i + 1) & 3]];
          double r[3] = {0, 0, 0}; int ni = 0;
          for (int i = 0; i < 4; ++i)
            if (inside(cyc[i])) { for (int ax = 0; ax < 3; ++ax) r[ax] += pos(cyc[i], ax); ++ni; }
          for (int ax = 0; ax < 3; ++ax) ref[0][ax] = r[ax] / ni;
          seg[0][0] = ce[0]; seg[0][1] = ce[1]; nseg = 1;
        } else if (crossed == 4) {
          for (int i = 0; i < 4; ++i) {
            if (!inside(cyc[i])) continue;
            seg[nseg][0] = edge_of[cyc[(i + 3) & 3]][cyc[i]];
            seg[nseg][1] = edge_of[cyc[i]][cyc[(i + 1) & 3]];
            for (int ax = 0; ax < 3; ++ax) ref[nseg][ax] = pos(cyc[i], ax);
            ++nseg;
          }
        }
        for (int q = 0; q < nseg; ++q) {
          double ma[3], mb[3], d[3], r[3];
          mid(seg[q][0], ma); mid(seg[q][1], mb);
          for (int ax = 0; ax < 3; ++ax) { d[ax] = mb[ax] - ma[ax]; r[ax] = ref[q][ax] - 0.5 * (ma[ax] + mb[ax]); }
          const double cr[3] = {d[1] * r[2] - d[2] * r[1], d[2] * r[0] - d[0] * r[2], d[0] * r[1] - d[1] * r[0]};
          // (d x r) . n_face < 0, n_face = the face's outward normal: the inside corners lie right of the direction of travel
          const double side = cr[k] * (s ? 1.0 : -1.0);
          if (side == 0.0) return false;
          int a = seg[q][0], b = seg[q][1];
          if (side > 0.0) { const int x = a; a = b; b = x; }
          if (next[a] != -1) return false;
          next[a] = b; ++nin[b];
        }
      }
    int n = 0;
    bool used[12] = {};
    for (int e = 0; e < 12; ++e) {
      const bool crossed = inside(edge_lower_corner(e)) != inside(edge_lower_corner(e) | (1 << (e >> 2)));
      if (crossed != (next[e] != -1) || nin[e] != (crossed ? 1 : 0)) return false;
    }
    for (int e0 = 0; e0 < 12; ++e0) {
      if (next[e0] == -1 || used[e0]) continue;
      int loop[12], len = 0;
      for (int e = e0; !used[e]; e = next[e]) { used[e] = true; loop[len++] = e; }
      if (loop[0] != e0 || next[loop[len - 1]] != e0) return false;
      for (int i = 1; i + 1 < len; ++i) {
        if (n >= kMaxCellTris) return false;
        t.tri[cs][n * 3] = (uint8_t)loop[0]; t.tri[cs][n * 3 + 1] = (uint8_t)loop[i]; t.tri[cs][n * 3 + 2] = (uint8_t)loop[i + 1];
        ++n;
      }
    }
    t.ntri[cs] = (uint8_t)n;
  }
  return true;
}

struct MeshParams {
  // the sample block of rr_sample.cuh
  const float* tsdf; int X, Y, Z;
  int half2;
  float limit;
  int N; const float4* inv; int IX, IY, IZ;
  const float2* uv[RR_MAX_SENSORS]; int cx[RR_MAX_SENSORS], cy[RR_MAX_SENSORS], cz[RR_MAX_SENSORS];
  const uint8_t* color; int CW, CH;
  const float2* depth_b; const float* quality; int W, H;
  // geometry
  float bmin[3], size[3];
  // candidate rows (use_rows = 0: every row)
  int use_rows, rby;
  const uint8_t* rowany; const int16_t* cand_y; const int16_t* cand_z;
  // per row (z * Y + y): counts, then exclusive offsets over rows + 1 entries
  unsigned long long* cnt_v; unsigned long long* cnt_t;
  const unsigned long long* off_v; const unsigned long long* off_t;
  // outputs
  unsigned long long* keys; float* pos; float* nrm; float4* rgba; uint32_t* tri;
  uint32_t nv;
};

__device__ __forceinline__ float vox(const MeshParams& p, int x, int y, int z) {
  return ld_density(p, ((unsigned)z * (unsigned)p.Y + (unsigned)y) * (unsigned)p.X + (unsigned)x);
}

__device__ __forceinline__ bool is_finite(float v) { return fabsf(v) <= 3.402823466e38f; }

// bit c: corner c is inside (v > 0); -1 when a corner is not finite (the cell emits nothing)
__device__ __forceinline__ int cell_case(const MeshParams& p, int x, int y, int z) {
  int cs = 0;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const float v = vox(p, x + (c & 1), y + ((c >> 1) & 1), z + ((c >> 2) & 1));
    if (!is_finite(v)) return -1;
    cs |= (v > 0.0f ? 1 : 0) << c;
  }
  return cs;
}

__device__ __forceinline__ bool cell_finite(const MeshParams& p, int x, int y, int z) {
  if (x < 0 || y < 0 || z < 0 || x >= p.X - 1 || y >= p.Y - 1 || z >= p.Z - 1) return false;
  return cell_case(p, x, y, z) >= 0;
}

// Bit k: the edge from (x, y, z) along axis k carries a vertex (crossed, both ends finite, on at least one emitting cell).
__device__ int owned_edges(const MeshParams& p, int x, int y, int z) {
  const float a = vox(p, x, y, z);
  if (!is_finite(a)) return 0;
  int mask = 0;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int bx = x + (k == 0), by = y + (k == 1), bz = z + (k == 2);
    if (bx >= p.X || by >= p.Y || bz >= p.Z) continue;
    const float b = vox(p, bx, by, bz);
    if (!is_finite(b) || (a > 0.0f) == (b > 0.0f)) continue;
    // the up to four cells around the edge: step back by 0 / 1 along the two other axes
    bool any = false;
    for (int m = 0; m < 4 && !any; ++m) {
      const int du = m & 1, dw = m >> 1;
      const int cx = x - (k != 0 ? du : 0);
      const int cy = y - (k == 0 ? du : (k == 2 ? dw : 0));
      const int cz = z - (k != 2 ? dw : 0);
      any = cell_finite(p, cx, cy, cz);
    }
    if (any) mask |= 1 << k;
  }
  return mask;
}

// a voxel row's rows (y..y+1, z..z+1) meet a brick row with an occupied brick (brick ranges may overlap by a voxel: both
// candidate bricks of an index are tested)
__device__ bool row_candidate(const MeshParams& p, int y, int z) {
  if (!p.use_rows) return true;
  for (int dz = 0; dz < 2; ++dz)
    for (int dy = 0; dy < 2; ++dy) {
      const int yy = min(y + dy, p.Y - 1), zz = min(z + dz, p.Z - 1);
      for (int a = 0; a < 2; ++a) {
        const int by = p.cand_y[2 * yy + a];
        if (by < 0) continue;
        for (int b = 0; b < 2; ++b) {
          const int bz = p.cand_z[2 * zz + b];
          if (bz >= 0 && p.rowany[bz * p.rby + by]) return true;
        }
      }
    }
  return false;
}

__device__ __forceinline__ unsigned warp_excl_scan(unsigned v, unsigned lane, unsigned& total) {
  unsigned incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned o = __shfl_up_sync(0xffffffffu, incl, d);
    if ((int)lane >= d) incl += o;
  }
  total = __shfl_sync(0xffffffffu, incl, 31);
  return incl - v;
}

// texture coordinate of the vertex on the edge from (x, y, z) along axis k (the caller knows the edge is crossed)
__device__ __forceinline__ float3 edge_q(const MeshParams& p, int x, int y, int z, int k) {
  const float va = vox(p, x, y, z), vb = vox(p, x + (k == 0), y + (k == 1), z + (k == 2));
  const float t = va / (va - vb);
  float3 q = make_float3(((float)x + 0.5f) * (1.0f / (float)p.X), ((float)y + 0.5f) * (1.0f / (float)p.Y),
                         ((float)z + 0.5f) * (1.0f / (float)p.Z));
  if (k == 0) q.x = ((float)x + 0.5f + t) / (float)p.X;
  else if (k == 1) q.y = ((float)y + 0.5f + t) / (float)p.Y;
  else q.z = ((float)z + 0.5f + t) / (float)p.Z;
  return q;
}

__global__ void __launch_bounds__(256) k_mesh_count(const __grid_constant__ MeshParams p) {
  const unsigned lane = threadIdx.x & 31u;
  const unsigned r = blockIdx.x * 8u + (threadIdx.x >> 5);
  if (r >= (unsigned)p.Y * (unsigned)p.Z) return;
  const int y = (int)(r % (unsigned)p.Y), z = (int)(r / (unsigned)p.Y);
  unsigned nv = 0, nt = 0;
  if (row_candidate(p, y, z)) {
    const bool cells = y < p.Y - 1 && z < p.Z - 1;
    for (int x0 = 0; x0 < p.X; x0 += 32) {
      const int x = x0 + (int)lane;
      if (x >= p.X) continue;
      nv += __popc(owned_edges(p, x, y, z));
      if (cells && x < p.X - 1) {
        const int cs = cell_case(p, x, y, z);
        if (cs >= 0) nt += kMesh.ntri[cs];
      }
    }
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) { nv += __shfl_down_sync(0xffffffffu, nv, d); nt += __shfl_down_sync(0xffffffffu, nt, d); }
  if (lane == 0) { p.cnt_v[r] = nv; p.cnt_t[r] = nt; }
}

__global__ void __launch_bounds__(256) k_mesh_vertices(const __grid_constant__ MeshParams p) {
  const unsigned lane = threadIdx.x & 31u;
  const unsigned r = blockIdx.x * 8u + (threadIdx.x >> 5);
  if (r >= (unsigned)p.Y * (unsigned)p.Z) return;
  unsigned long long base = p.off_v[r];
  if (p.off_v[r + 1] == base) return;
  const int y = (int)(r % (unsigned)p.Y), z = (int)(r / (unsigned)p.Y);
  for (int x0 = 0; x0 < p.X; x0 += 32) {
    const int x = x0 + (int)lane;
    const int mask = x < p.X ? owned_edges(p, x, y, z) : 0;
    unsigned total;
    unsigned at = warp_excl_scan((unsigned)__popc(mask), lane, total);
    for (int k = 0; k < 3; ++k) {
      if (!((mask >> k) & 1)) continue;
      const unsigned long long i = base + at++;
      p.keys[i] = ((unsigned long long)r * (unsigned)p.X + (unsigned)x) * 3ull + (unsigned)k;
      const float3 q = edge_q(p, x, y, z, k);
      p.pos[i * 3] = p.bmin[0] + q.x * p.size[0];
      p.pos[i * 3 + 1] = p.bmin[1] + q.y * p.size[1];
      p.pos[i * 3 + 2] = p.bmin[2] + q.z * p.size[2];
    }
    base += total;
  }
}

__global__ void __launch_bounds__(128) k_mesh_attributes(const __grid_constant__ MeshParams p) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.nv) return;
  const unsigned long long key = p.keys[i];
  const unsigned long long lin = key / 3ull;
  const int k = (int)(key - lin * 3ull);
  const int x = (int)(lin % (unsigned)p.X);
  const unsigned long long r = lin / (unsigned)p.X;
  const int y = (int)(r % (unsigned)p.Y), z = (int)(r / (unsigned)p.Y);
  const float3 q = edge_q(p, x, y, z, k);
  const float3 g = get_gradient(p, q, p.limit * 0.5f);
  const float3 n = normalize3(make_float3(g.x / p.size[0], g.y / p.size[1], g.z / p.size[2]));
  p.nrm[(size_t)i * 3] = n.x; p.nrm[(size_t)i * 3 + 1] = n.y; p.nrm[(size_t)i * 3 + 2] = n.z;
  p.rgba[i] = blend_colors(p, q);
}

__global__ void __launch_bounds__(256) k_mesh_triangles(const __grid_constant__ MeshParams p) {
  const unsigned lane = threadIdx.x & 31u;
  const unsigned r = blockIdx.x * 8u + (threadIdx.x >> 5);
  if (r >= (unsigned)p.Y * (unsigned)p.Z) return;
  unsigned long long base = p.off_t[r];
  if (p.off_t[r + 1] == base) return;
  const int y = (int)(r % (unsigned)p.Y), z = (int)(r / (unsigned)p.Y);
  for (int x0 = 0; x0 < p.X - 1; x0 += 32) {
    const int x = x0 + (int)lane;
    const int cs = x < p.X - 1 ? cell_case(p, x, y, z) : -1;
    const int nt = cs >= 0 ? kMesh.ntri[cs] : 0;
    unsigned total;
    const unsigned at = warp_excl_scan((unsigned)nt, lane, total);
    for (int j = 0; j < nt * 3; ++j) {
      const int e = kMesh.tri[cs][j];
      const int lc = edge_lower_corner(e), k = e >> 2;
      const int ex = x + (lc & 1), ey = y + ((lc >> 1) & 1), ez = z + ((lc >> 2) & 1);
      const unsigned ro = (unsigned)ez * (unsigned)p.Y + (unsigned)ey;
      const unsigned long long key = ((unsigned long long)ro * (unsigned)p.X + (unsigned)ex) * 3ull + (unsigned)k;
      unsigned long long lo = p.off_v[ro], hi = p.off_v[ro + 1];   // the owning row's keys are sorted: binary search
      while (lo < hi) {
        const unsigned long long mid = (lo + hi) >> 1;
        if (p.keys[mid] < key) lo = mid + 1; else hi = mid;
      }
      p.tri[(base + at) * 3 + j] = (uint32_t)lo;
    }
    base += total;
  }
}

}  // namespace

bool mesh_rows_usable(const rr_ctx* c) {
  const bool grid_ok = c->bricks.num == c->bricks.res[0] * c->bricks.res[1] * c->bricks.res[2];
  const uint32_t path = c->last_integrate[0];
  return c->cfg.use_bricks && grid_ok && c->fused_ok && c->d_rowany && c->d_cand_y && c->d_cand_z && path >= 1 && path <= 3;
}

int launch_extract_mesh(rr_ctx* c, uint32_t* out_nv, uint32_t* out_nt) {
  if (!c->mesh_table) {
    MeshTable t;
    if (!build_case_table(t)) return fail(c, RR_ERR_INVALID, "rr_extract_mesh: case table generation failed");
    RR_TRY_RC(check(c, cudaMemcpyToSymbolAsync(kMesh, &t, sizeof(t), 0, cudaMemcpyHostToDevice, c->stream), "mesh case table"));
    c->mesh_table = true;
  }
  const int X = (int)c->res[0], Y = (int)c->res[1], Z = (int)c->res[2];
  const size_t rows = (size_t)Y * Z;
  RR_TRY_RC(c->d_mesh_rows.reserve(c, 4 * (rows + 1), "mesh row counts"));
  unsigned long long* cnt_v = c->d_mesh_rows.ptr;
  unsigned long long* cnt_t = cnt_v + (rows + 1);
  unsigned long long* off_v = cnt_t + (rows + 1);
  unsigned long long* off_t = off_v + (rows + 1);
  size_t scan_bytes = 0;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, cnt_v, off_v, (int)(rows + 1), c->stream), "mesh scan size"));
  RR_TRY_RC(c->d_mesh_scratch.reserve(c, scan_bytes, "mesh scan scratch"));

  MeshParams p{};
  p.tsdf = c->d_tsdf; p.X = X; p.Y = Y; p.Z = Z;
  p.half2 = c->cfg.store_weight == RR_VOXELS_HALF2 ? 1 : 0;
  p.limit = c->cfg.limit;
  p.N = c->N; p.inv = c->d_inv; p.IX = (int)c->ires[0]; p.IY = (int)c->ires[1]; p.IZ = (int)c->ires[2];
  for (int i = 0; i < c->N; ++i) { p.uv[i] = c->d_uv[i]; p.cx[i] = (int)c->cres[i][0]; p.cy[i] = (int)c->cres[i][1]; p.cz[i] = (int)c->cres[i][2]; }
  p.color = c->d_color; p.CW = c->CW; p.CH = c->CH;
  p.depth_b = c->d_depth_b; p.quality = c->d_quality; p.W = c->W; p.H = c->H;
  for (int a = 0; a < 3; ++a) { p.bmin[a] = c->bbox_min[a]; p.size[a] = c->bbox_max[a] - c->bbox_min[a]; }
  p.use_rows = c->mesh_rows_ok ? 1 : 0;
  p.rby = (int)c->bricks.res[1];
  p.rowany = c->d_rowany; p.cand_y = c->d_cand_y; p.cand_z = c->d_cand_z;
  p.cnt_v = cnt_v; p.cnt_t = cnt_t; p.off_v = off_v; p.off_t = off_t;

  const unsigned row_blocks = (unsigned)((rows + 7) / 8);
  RR_TRY_RC(check(c, cudaMemsetAsync(cnt_v + rows, 0, sizeof(unsigned long long), c->stream), "mesh counts"));
  RR_TRY_RC(check(c, cudaMemsetAsync(cnt_t + rows, 0, sizeof(unsigned long long), c->stream), "mesh counts"));
  k_mesh_count<<<row_blocks, 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_mesh_count");
  size_t bytes = c->d_mesh_scratch.cap;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(c->d_mesh_scratch.ptr, bytes, cnt_v, off_v, (int)(rows + 1), c->stream), "mesh vertex scan"));
  bytes = c->d_mesh_scratch.cap;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(c->d_mesh_scratch.ptr, bytes, cnt_t, off_t, (int)(rows + 1), c->stream), "mesh triangle scan"));
  c->launches += 2;
  unsigned long long* totals = c->pinned->mesh_totals;
  RR_TRY_RC(check(c, cudaMemcpyAsync(totals, off_v + rows, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream), "mesh totals"));
  RR_TRY_RC(check(c, cudaMemcpyAsync(totals + 1, off_t + rows, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream), "mesh totals"));
  RR_TRY_RC(check(c, cudaStreamSynchronize(c->stream), "mesh count sync"));
  const unsigned long long nv = totals[0], nt = totals[1];
  c->mesh_valid = false;
  // vertex and triangle indices are uint32 in the output and int-sized in the launches
  if (nv >= (1ull << 31) || nt >= (1ull << 31))
    return fail(c, RR_ERR_UNSUPPORTED, "rr_extract_mesh: meshes of 2^31 or more vertices or triangles are not supported");
  RR_TRY_RC(c->d_mesh_keys.reserve(c, nv, "mesh keys"));
  RR_TRY_RC(c->d_mesh_pos.reserve(c, 3 * nv, "mesh positions"));
  RR_TRY_RC(c->d_mesh_nrm.reserve(c, 3 * nv, "mesh normals"));
  RR_TRY_RC(c->d_mesh_rgba.reserve(c, nv, "mesh colours"));
  if (nt) RR_TRY_RC(c->d_mesh_tri.reserve(c, 3 * nt, "mesh triangles"));
  p.keys = c->d_mesh_keys.ptr; p.pos = c->d_mesh_pos.ptr; p.nrm = c->d_mesh_nrm.ptr; p.rgba = c->d_mesh_rgba.ptr; p.tri = c->d_mesh_tri.ptr;
  p.nv = (uint32_t)nv;
  if (nv) {
    k_mesh_vertices<<<row_blocks, 256, 0, c->stream>>>(p);
    RR_LAUNCH_CHECK(c, "k_mesh_vertices");
    k_mesh_attributes<<<(unsigned)((nv + 127) / 128), 128, 0, c->stream>>>(p);
    RR_LAUNCH_CHECK(c, "k_mesh_attributes");
  }
  if (nt) {
    k_mesh_triangles<<<row_blocks, 256, 0, c->stream>>>(p);
    RR_LAUNCH_CHECK(c, "k_mesh_triangles");
  }
  c->mesh_nv = (uint32_t)nv; c->mesh_nt = (uint32_t)nt;
  c->mesh_epoch = c->volume_epoch;
  c->mesh_valid = true;
  if (out_nv) *out_nv = c->mesh_nv;
  if (out_nt) *out_nt = c->mesh_nt;
  return RR_OK;
}

}  // namespace rr
