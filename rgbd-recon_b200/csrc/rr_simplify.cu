// Mesh simplification by vertex clustering on the device (rr_simplify_mesh / rr_download_simplified_mesh /
// rr_group_simplify_mesh; the contract is stated in include/rgbd_recon_b200.h and DESIGN.md "Beyond the reference: mesh
// simplification"). No reference counterpart. Input: the last mesh of rr_extract_mesh, whose vertices are in edge-key order.
//   k_simp_cluster     one thread per vertex: its cluster id from the lower corner of its edge key
//   CUB radix sort     (cluster id, vertex) pairs over the bits the ids need; stable, so a cluster's members stay in
//                      ascending edge-key order
//   k_simp_heads       one thread per sorted vertex: 1 where a cluster starts; CUB inclusive scan -> each vertex's cluster
//                      rank (rank = position among the clusters that hold a vertex, in ascending cluster id)
//   k_simp_rank        per sorted vertex: the rank of every vertex, the first member of every cluster
//   k_simp_tri_map     one thread per triangle: ranks of its corners; degenerate -> sentinel, otherwise rotated so that the
//                      smallest rank comes first; flags the clusters it references
//   two CUB radix sorts  (third rank, triangle), then (first two ranks as 64 bits, triangle): equal triples end up next to
//                      each other in ascending triangle index
//   k_simp_tri_keep    one thread per sorted triangle: the head of each run of equal triples is kept
//   two CUB exclusive scans  output slots of the kept triangles and of the referenced clusters; both totals are read back in
//                      the call's single synchronisation
//   k_simp_vertices    one thread per referenced cluster: the binary64 mean of its members in edge-key order, then the
//                      sample contract of rr_sample_points(RR_QUERY_WORLD) at the mean (rr_sample.cuh)
//   k_simp_triangles   one thread per kept triangle: the new vertex indices and the source triangle
// Every kernel is launched with a grid for the input's V or T and returns past the device-side counts.
#include "rr_context.h"
#include "rr_march.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>

namespace rr {

namespace {

struct SimplifyParams {
  // the sample block of rr_sample.cuh
  const float* tsdf; int X, Y, Z;
  int half2;
  float limit;
  int N; const float4* inv; int IX, IY, IZ;
  const float2* uv[RR_MAX_SENSORS]; int cx[RR_MAX_SENSORS], cy[RR_MAX_SENSORS], cz[RR_MAX_SENSORS];
  const uint8_t* color; int CW, CH;
  const float2* depth_b; const float* quality; int W, H;
  // world <-> volume (to_volume / world_normal of rr_sample.cuh)
  float bmin[3], dims[3];
  int world;                 // always 1: the mean is in metres
  // clusters
  uint32_t cs;               // cluster edge in voxels
  uint32_t CX, CY;           // clusters along x and y
  uint32_t V, T;             // the input mesh's vertices and triangles
  uint32_t S;                // sentinel rank of a dropped triangle, above every cluster rank
  int rb;                    // bits of a rank (S < 2^rb)
  // input mesh
  const unsigned long long* keys; const float* pos; const uint32_t* tri;
  // per vertex
  uint32_t* cid; uint32_t* vid; uint32_t* cid_s; uint32_t* perm;   // cluster ids and vertex indices, before and after the sort
  uint32_t* head; uint32_t* incl;                                   // cluster starts in sorted order, their inclusive scan
  uint32_t* vrank;                                                  // [V] cluster rank of each vertex
  uint32_t* start;                                                  // [V + 1] first sorted member of each rank (start[U] = V)
  uint32_t* ref; uint32_t* vnew;                                    // [V + 1] rank referenced by a kept triangle, its scan
  // per triangle
  uint32_t* trip;                                                   // [T][3] rotated ranks (S, S, S: dropped)
  uint32_t* key3; uint32_t* idx0; uint32_t* key3_s; uint32_t* idx1; uint32_t* idx2;
  unsigned long long* k64; unsigned long long* k64_s;
  uint32_t* keep; uint32_t* toff;                                   // [T + 1] kept flag by source triangle, its scan
  // outputs
  float* out_pos; float* out_nrm; float4* out_rgba; uint32_t* out_tri; uint32_t* out_src;
};

constexpr uint32_t kNaN = 0x7fc00000u;   // the quiet NaN of rr_sample_points outside the unit cube

__global__ void __launch_bounds__(256) k_simp_cluster(const __grid_constant__ SimplifyParams p) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.V) return;
  const unsigned long long lin = p.keys[i] / 3ull;
  const uint32_t x = (uint32_t)(lin % (uint32_t)p.X);
  const unsigned long long r = lin / (uint32_t)p.X;
  const uint32_t y = (uint32_t)(r % (uint32_t)p.Y), z = (uint32_t)(r / (uint32_t)p.Y);
  p.cid[i] = ((z / p.cs) * p.CY + y / p.cs) * p.CX + x / p.cs;   // < X*Y*Z < 2^31
  p.vid[i] = i;
}

__global__ void __launch_bounds__(256) k_simp_heads(const __grid_constant__ SimplifyParams p) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= p.V) return;
  p.head[j] = (j == 0 || p.cid_s[j] != p.cid_s[j - 1]) ? 1u : 0u;
}

__global__ void __launch_bounds__(256) k_simp_rank(const __grid_constant__ SimplifyParams p) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= p.V) return;
  const uint32_t u = p.incl[j] - 1u;
  p.vrank[p.perm[j]] = u;
  if (p.head[j]) p.start[u] = j;
  if (j == p.V - 1) p.start[u + 1] = p.V;
}

__global__ void __launch_bounds__(256) k_simp_tri_map(const __grid_constant__ SimplifyParams p) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= p.T) return;
  uint32_t a = p.vrank[p.tri[(size_t)t * 3]], b = p.vrank[p.tri[(size_t)t * 3 + 1]], c = p.vrank[p.tri[(size_t)t * 3 + 2]];
  if (a == b || b == c || a == c) {
    a = b = c = p.S;
  } else {
    // rotate (a, b, c) -> (b, c, a) or (c, a, b): the cyclic order, and so the orientation, is kept
    if (b < a && b < c) { const uint32_t x = a; a = b; b = c; c = x; }
    else if (c < a && c < b) { const uint32_t x = c; c = b; b = a; a = x; }
    // every triangle that maps to this triple references the same clusters, the kept one among them
    p.ref[a] = 1u; p.ref[b] = 1u; p.ref[c] = 1u;
  }
  p.trip[(size_t)t * 3] = a; p.trip[(size_t)t * 3 + 1] = b; p.trip[(size_t)t * 3 + 2] = c;
  p.key3[t] = c;
  p.idx0[t] = t;
}

__global__ void __launch_bounds__(256) k_simp_tri_key(const __grid_constant__ SimplifyParams p) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= p.T) return;
  const uint32_t t = p.idx1[j];
  p.k64[j] = ((unsigned long long)p.trip[(size_t)t * 3] << p.rb) | p.trip[(size_t)t * 3 + 1];
}

// keep[T] = 0 closes the scan, so toff[T] is the number of kept triangles
__global__ void __launch_bounds__(256) k_simp_tri_keep(const __grid_constant__ SimplifyParams p) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j > p.T) return;
  if (j == p.T) { p.keep[p.T] = 0u; return; }
  const uint32_t t = p.idx2[j];
  const bool valid = p.trip[(size_t)t * 3] != p.S;
  const bool first = j == 0 || p.k64_s[j] != p.k64_s[j - 1] ||
                     p.trip[(size_t)t * 3 + 2] != p.trip[(size_t)p.idx2[j - 1] * 3 + 2];
  p.keep[t] = valid && first ? 1u : 0u;
}

__device__ __forceinline__ float3 ld3(const float* a, size_t i) { return make_float3(a[i * 3], a[i * 3 + 1], a[i * 3 + 2]); }
__device__ __forceinline__ void st3(float* a, size_t i, float3 v) { a[i * 3] = v.x; a[i * 3 + 1] = v.y; a[i * 3 + 2] = v.z; }

__global__ void __launch_bounds__(128) k_simp_vertices(const __grid_constant__ SimplifyParams p) {
  const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= p.incl[p.V - 1] || !p.ref[u]) return;
  const uint32_t j0 = p.start[u], j1 = p.start[u + 1];
  double s0 = 0.0, s1 = 0.0, s2 = 0.0;
  for (uint32_t j = j0; j < j1; ++j) {                     // ascending edge key
    const float3 v = ld3(p.pos, p.perm[j]);
    s0 = s0 + (double)v.x; s1 = s1 + (double)v.y; s2 = s2 + (double)v.z;
  }
  const double n = (double)(j1 - j0);
  const float3 m = make_float3((float)(s0 / n), (float)(s1 / n), (float)(s2 / n));
  // k_sample_points (rr_query.cu) at m in world space, over the whole volume
  const float3 q = to_volume(p, m);
  const float nan = __uint_as_float(kNaN);
  float3 nrm = make_float3(nan, nan, nan);
  float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
  if (in_unit_cube(q)) {
    nrm = world_normal(p, q);
    c = blend_colors(p, q);
  }
  const uint32_t o = p.vnew[u];
  st3(p.out_pos, o, m);
  st3(p.out_nrm, o, nrm);
  p.out_rgba[o] = c;
}

__global__ void __launch_bounds__(256) k_simp_triangles(const __grid_constant__ SimplifyParams p) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= p.T || !p.keep[t]) return;
  const size_t o = p.toff[t];
  for (int k = 0; k < 3; ++k) p.out_tri[o * 3 + k] = p.vnew[p.trip[(size_t)t * 3 + k]];
  p.out_src[o] = t;
}

int bit_width(uint32_t v) { int b = 0; while (v) { ++b; v >>= 1; } return b; }

}  // namespace

int launch_simplify_mesh(rr_ctx* c, uint32_t cluster_voxels, uint32_t* out_nv, uint32_t* out_nt) {
  c->simp_valid = false;
  const uint32_t V = c->mesh_nv, T = c->mesh_nt;
  const uint32_t X = c->res[0], Y = c->res[1], Z = c->res[2], cs = cluster_voxels;
  const uint32_t CX = X / cs + (X % cs != 0), CY = Y / cs + (Y % cs != 0), CZ = Z / cs + (Z % cs != 0);
  if (V == 0 || T == 0) {                                  // no triangle: no vertex either
    c->simp_nv = c->simp_nt = 0;
    c->simp_valid = true;
    *out_nv = *out_nt = 0;
    return RR_OK;
  }
  const uint32_t ncl = CX * CY * CZ;                       // <= X*Y*Z < 2^31
  const int cid_bits = std::max(1, bit_width(ncl - 1));
  const uint32_t S = std::min(V, ncl);                     // ranks are below the number of non-empty clusters <= S
  const int rb = bit_width(S);

  // per vertex: cid, vid, cid_s, perm, head, incl, vrank [V]; start, ref, vnew [V + 1]
  const size_t v1 = (size_t)V + 1, t1 = (size_t)T + 1;
  RR_TRY_RC(c->d_simp_v.reserve(c, 10 * v1, "simplification vertex scratch"));
  // per triangle: trip [3T]; key3, idx0, key3_s, idx1, idx2 [T]; keep, toff [T + 1]
  RR_TRY_RC(c->d_simp_t.reserve(c, 10 * t1, "simplification triangle scratch"));
  RR_TRY_RC(c->d_simp_k64.reserve(c, 2 * (size_t)T, "simplification triangle keys"));
  SimplifyParams p{};
  set_sample_params(p, c);
  for (int a = 0; a < 3; ++a) { p.bmin[a] = c->bbox_min[a]; p.dims[a] = c->bbox_max[a] - c->bbox_min[a]; }
  p.world = 1;
  p.cs = cs; p.CX = CX; p.CY = CY; p.V = V; p.T = T; p.S = S; p.rb = rb;
  p.keys = c->d_mesh_keys.ptr; p.pos = c->d_mesh_pos.ptr; p.tri = c->d_mesh_tri.ptr;
  uint32_t* w = c->d_simp_v.ptr;
  p.cid = w; p.vid = w + v1; p.cid_s = w + 2 * v1; p.perm = w + 3 * v1; p.head = w + 4 * v1; p.incl = w + 5 * v1;
  p.vrank = w + 6 * v1; p.start = w + 7 * v1; p.ref = w + 8 * v1; p.vnew = w + 9 * v1;
  uint32_t* tw = c->d_simp_t.ptr;
  p.trip = tw; p.key3 = tw + 3 * t1; p.idx0 = tw + 4 * t1; p.key3_s = tw + 5 * t1; p.idx1 = tw + 6 * t1; p.idx2 = tw + 7 * t1;
  p.keep = tw + 8 * t1; p.toff = tw + 9 * t1;
  p.k64 = c->d_simp_k64.ptr; p.k64_s = c->d_simp_k64.ptr + T;

  size_t need = 0, b = 0;
  RR_TRY_RC(check(c, cub::DeviceRadixSort::SortPairs(nullptr, b, p.cid, p.cid_s, p.vid, p.perm, (int)V, 0, cid_bits, c->stream), "simplification sort size"));
  need = std::max(need, b);
  RR_TRY_RC(check(c, cub::DeviceRadixSort::SortPairs(nullptr, b, p.key3, p.key3_s, p.idx0, p.idx1, (int)T, 0, rb, c->stream), "simplification sort size"));
  need = std::max(need, b);
  RR_TRY_RC(check(c, cub::DeviceRadixSort::SortPairs(nullptr, b, p.k64, p.k64_s, p.idx1, p.idx2, (int)T, 0, 2 * rb, c->stream), "simplification sort size"));
  need = std::max(need, b);
  RR_TRY_RC(check(c, cub::DeviceScan::InclusiveSum(nullptr, b, p.head, p.incl, (int)V, c->stream), "simplification scan size"));
  need = std::max(need, b);
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(nullptr, b, p.ref, p.vnew, (int)v1, c->stream), "simplification scan size"));
  need = std::max(need, b);
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(nullptr, b, p.keep, p.toff, (int)t1, c->stream), "simplification scan size"));
  need = std::max(need, b);
  RR_TRY_RC(c->d_simp_scratch.reserve(c, need, "simplification sort scratch"));
  // the output is never larger than the input
  RR_TRY_RC(c->d_simp_pos.reserve(c, 3 * (size_t)V, "simplified positions"));
  RR_TRY_RC(c->d_simp_nrm.reserve(c, 3 * (size_t)V, "simplified normals"));
  RR_TRY_RC(c->d_simp_rgba.reserve(c, V, "simplified colours"));
  RR_TRY_RC(c->d_simp_tri.reserve(c, 3 * (size_t)T, "simplified triangles"));
  RR_TRY_RC(c->d_simp_src.reserve(c, T, "simplified sources"));
  p.out_pos = c->d_simp_pos.ptr; p.out_nrm = c->d_simp_nrm.ptr; p.out_rgba = c->d_simp_rgba.ptr;
  p.out_tri = c->d_simp_tri.ptr; p.out_src = c->d_simp_src.ptr;
  void* scratch = c->d_simp_scratch.ptr;

  const unsigned vb = (V + 255) / 256, tb = (T + 255) / 256;
  RR_TRY_RC(check(c, cudaMemsetAsync(p.ref, 0, v1 * sizeof(uint32_t), c->stream), "simplification flags"));
  k_simp_cluster<<<vb, 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_simp_cluster");
  b = need;
  RR_TRY_RC(check(c, cub::DeviceRadixSort::SortPairs(scratch, b, p.cid, p.cid_s, p.vid, p.perm, (int)V, 0, cid_bits, c->stream), "cluster sort"));
  k_simp_heads<<<vb, 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_simp_heads");
  b = need;
  RR_TRY_RC(check(c, cub::DeviceScan::InclusiveSum(scratch, b, p.head, p.incl, (int)V, c->stream), "cluster scan"));
  k_simp_rank<<<vb, 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_simp_rank");
  k_simp_tri_map<<<tb, 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_simp_tri_map");
  b = need;
  RR_TRY_RC(check(c, cub::DeviceRadixSort::SortPairs(scratch, b, p.key3, p.key3_s, p.idx0, p.idx1, (int)T, 0, rb, c->stream), "triangle sort"));
  k_simp_tri_key<<<tb, 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_simp_tri_key");
  b = need;
  RR_TRY_RC(check(c, cub::DeviceRadixSort::SortPairs(scratch, b, p.k64, p.k64_s, p.idx1, p.idx2, (int)T, 0, 2 * rb, c->stream), "triangle sort"));
  k_simp_tri_keep<<<(T + 1 + 255) / 256, 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_simp_tri_keep");
  b = need;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(scratch, b, p.keep, p.toff, (int)t1, c->stream), "triangle scan"));
  b = need;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(scratch, b, p.ref, p.vnew, (int)v1, c->stream), "vertex scan"));
  c->launches += 5;
  uint32_t* counts = c->pinned->simplify_counts;
  RR_TRY_RC(check(c, cudaMemcpyAsync(counts, p.vnew + V, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream), "simplification counts"));
  RR_TRY_RC(check(c, cudaMemcpyAsync(counts + 1, p.toff + T, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream), "simplification counts"));
  k_simp_vertices<<<(V + 127) / 128, 128, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_simp_vertices");
  k_simp_triangles<<<tb, 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_simp_triangles");
  RR_TRY_RC(check(c, cudaStreamSynchronize(c->stream), "simplification sync"));
  c->simp_nv = counts[0]; c->simp_nt = counts[1];
  c->simp_valid = true;
  *out_nv = c->simp_nv;
  *out_nt = c->simp_nt;
  return RR_OK;
}

int simplified_download(rr_ctx* c, float* positions, float* normals, float* rgba, uint32_t* triangles, uint32_t* sources) {
  const size_t nv = c->simp_nv, nt = c->simp_nt;
  if (positions && nv) RR_TRY_RC(check(c, cudaMemcpyAsync(positions, c->d_simp_pos.ptr, nv * 3 * sizeof(float), cudaMemcpyDefault, c->stream), "simplified mesh download"));
  if (normals && nv) RR_TRY_RC(check(c, cudaMemcpyAsync(normals, c->d_simp_nrm.ptr, nv * 3 * sizeof(float), cudaMemcpyDefault, c->stream), "simplified mesh download"));
  if (rgba && nv) RR_TRY_RC(check(c, cudaMemcpyAsync(rgba, c->d_simp_rgba.ptr, nv * sizeof(float4), cudaMemcpyDefault, c->stream), "simplified mesh download"));
  if (triangles && nt) RR_TRY_RC(check(c, cudaMemcpyAsync(triangles, c->d_simp_tri.ptr, nt * 3 * sizeof(uint32_t), cudaMemcpyDefault, c->stream), "simplified mesh download"));
  if (sources && nt) RR_TRY_RC(check(c, cudaMemcpyAsync(sources, c->d_simp_src.ptr, nt * sizeof(uint32_t), cudaMemcpyDefault, c->stream), "simplified mesh download"));
  return check(c, cudaStreamSynchronize(c->stream), "simplified mesh download sync");
}

}  // namespace rr
