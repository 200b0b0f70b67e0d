// TSDF integration for sm_100a: the per-voxel work of glsl/tsdf_integration.vs:23-59, driven like
// ReconIntegration::integrate (framework/reconstruction/recon_integration.cpp:243-270): clear to -limit, then either
// every voxel (dense) or the voxels of every occupied brick.
//
// Kernel shape (DESIGN.md "integrate"): one thread owns an (x, y) column of the volume and marches z. The x/y part of
// the trilinear inverse-calibration lookup (cv_xyz_inv, LINEAR filtering restated in fp32) is reduced once per coarse
// z-plane and kept in registers for all N sensors, so the 8-corner gather of the shader becomes 4 corner loads per
// coarse plane per sensor; consecutive lanes are consecutive x, so the R32F stores are 128-byte coalesced rows.
// Silhouette (bilinear), depth (nearest) and quality (bilinear) come from ONE 32-byte gather texel per voxel-sensor
// (see k_pack_gather). HBM-bound integer/float gather work: no tensor-core path applies.
#include "rr_integrate.cuh"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

namespace rr {

// lin_coord of every fine z against the inverse volume's z axis, evaluated once per (Z, IZ) pair with the same
// float operations march_column used to repeat per voxel (identical results, ~25 instructions saved per voxel).
__global__ void k_build_ztab(float4* __restrict__ ztab, int Z, int IZ) {
  const int z = blockIdx.x * blockDim.x + threadIdx.x;
  if (z >= Z) return;
  const float stepZ = 1.0f / (float)Z;
  const float pz = ((float)z + 0.5f) * stepZ;
  int k0, k1; float g;
  lin_coord(pz, IZ, k0, k1, g);
  ztab[z] = make_float4(__int_as_float(k0), __int_as_float(k1), g, 1.0f - g);
}

template <int N, int MODE>
__global__ void __launch_bounds__(256) k_integrate_dense(const __grid_constant__ IntegrateParams p) {
  const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
  if (x >= p.X || y >= p.Y) return;
  const int zb = p.z_begin + blockIdx.z * p.z_chunk;
  const int ze = min(zb + p.z_chunk, p.z_end);
  march_column<N, MODE>(p, x, y, zb, ze);
}

// Occupied bricks only (VolumeSampler::sample(indices), volume_sampler.cpp:74-76). Persistent kernel: a fixed grid
// (a multiple of the 148 SMs) strides over work items = (occupied brick, z-chunk, block of BRICK_COLS columns); the
// item count comes from the device-side occupied count, so no host round trip and no empty blocks.
// Bricks may overlap or leave one-voxel gaps (float rounding in divideBox/containedVoxels): overlapping voxels are
// written twice with the same value, gaps keep the cleared -limit.
#define BRICK_MAX_THREADS 320
template <int N, int MODE, int MINB>
__global__ void __launch_bounds__(BRICK_MAX_THREADS, MINB) k_integrate_bricks(const __grid_constant__ IntegrateParams p, int max_cols, int max_nz, int BRICK_ZCHUNK) {
  const unsigned n_occ = *p.num_occupied;
  const unsigned col_blocks = ((unsigned)max_cols + blockDim.x - 1u) / blockDim.x;
  const unsigned z_blocks = (unsigned)(max_nz + BRICK_ZCHUNK - 1) / BRICK_ZCHUNK;
  const unsigned per_brick = col_blocks * z_blocks;
  const unsigned items = n_occ * per_brick;
  for (unsigned w = blockIdx.x; w < items; w += gridDim.x) {
    const unsigned b = w / per_brick, r = w - b * per_brick;
    const unsigned zc = r / col_blocks, cc = r - zc * col_blocks;
    const int32_t* rg = p.ranges + (size_t)p.occupied[b] * 6;
    const int x0 = rg[0], nx = rg[1] - rg[0], y0 = rg[2], ny = rg[3] - rg[2];
    const int zb = max(rg[4] + (int)zc * BRICK_ZCHUNK, p.z_begin);
    const int ze = min(min(rg[4] + (int)(zc + 1) * BRICK_ZCHUNK, rg[5]), p.z_end);
    const int ci = (int)(cc * blockDim.x + threadIdx.x);
    if (zb >= ze || ci >= nx * ny) continue;
    const int cy = ci / nx, cx = ci - cy * nx;
    march_column<N, MODE>(p, x0 + cx, y0 + cy, zb, ze);
  }
}

// ---- fused clear + integrate (bricks mode) ----------------------------------------------------------------------
// ReconIntegration::integrate clears the whole volume to -limit and then overwrites the voxels of the occupied bricks
// (recon_integration.cpp:248-259). Here ONE persistent kernel writes every voxel of the slab exactly once: the clear is
// an HBM-bound stream of 16-byte stores (4 bytes per voxel), the brick evaluation is issue/latency-bound gather work,
// so warps of both kinds share each SM and overlap. Work is handed out per WARP from two device counters:
//   fill item    = FILL_ROWS consecutive (y, z) voxel rows; voxels inside an occupied brick are skipped (row bitmask
//                  built by k_bricks_masks), everything else gets -limit (and weight 0);
//   compute item = 32 consecutive columns of the flattened (occupied brick, column) space x one z-chunk.
// The first `fill_warps` warps of a CTA start on fill items, the others on compute items; a warp that runs out of its
// own kind helps with the other, so the kernel ends when both counters are exhausted.
// Compute items are handed out to a CTA in chunks of `chunk` consecutive items (one global atomic per chunk) and to
// its warps one at a time from a shared counter, so the warps of a CTA work on neighbouring column blocks of the same
// brick at the same time: their inverse-volume corners and gather texels hit the SM's L1 instead of L2.
// Slot protocol: the warp that draws the first index of a chunk fetches the chunk base from the global counter and
// publishes (chunk number + 1, base) as one 64-bit word; the other warps of that chunk spin on the word.
#define FUSED_SLOTS 8
// THREADS = 512 caps the kernel at 64 registers (32 warps/SM), 384 at 85 registers (24 warps/SM).
template <int N, int MODE, int THREADS>
__global__ void __launch_bounds__(THREADS, 2) k_integrate_fused(const __grid_constant__ FusedParams p) {
  __shared__ unsigned s_taken;
  __shared__ unsigned long long s_slot[FUSED_SLOTS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_taken = 0;
  if (threadIdx.x < FUSED_SLOTS) s_slot[threadIdx.x] = 0ull;
  __syncthreads();
  const unsigned n_occ = *p.ip.num_occupied;
  const unsigned cbpb = ((unsigned)p.max_cols + 31u) / 32u;          // 32-column blocks per brick (a warp never straddles bricks)
  const unsigned per_brick = cbpb * (unsigned)p.n_zchunks;
  const unsigned citems = n_occ * per_brick;
  const unsigned chunk = (unsigned)p.chunk;
  bool filling = warp < p.fill_warps;
  for (int phase = 0; phase < 2; ++phase, filling = !filling) {
    if (filling) {
      for (;;) {
        unsigned it = 0;
        if (lane == 0) it = atomicAdd(p.work + 1, 1u);
        it = __shfl_sync(0xffffffffu, it, 0);
        if (it >= p.fill_items) break;
        const uint32_t r0 = p.row_begin + it * (uint32_t)p.fill_rows;
        fill_rows<MODE == 1>(p, FillTables{p.cand_y, p.cand_z, p.rowany}, r0, min(r0 + (uint32_t)p.fill_rows, p.row_end), lane);
      }
    } else {
      for (;;) {
        unsigned it = 0;
        if (lane == 0) {
          if (chunk <= 1u) {
            it = atomicAdd(p.work, 1u);
          } else {
            const unsigned i = atomicAdd(&s_taken, 1u);
            const unsigned c = i / chunk, j = i - c * chunk;
            volatile unsigned long long* slot = s_slot + (c % FUSED_SLOTS);
            if (j == 0) {
              const unsigned g = atomicAdd(p.work, chunk);
              *slot = ((unsigned long long)(c + 1u) << 32) | g;
              it = g;
            } else {
              unsigned long long v;
              do { v = *slot; } while ((unsigned)(v >> 32) != c + 1u);
              it = (unsigned)v + j;
            }
          }
        }
        it = __shfl_sync(0xffffffffu, it, 0);
        if (it >= citems) break;
        const unsigned b = it / per_brick, rem = it - b * per_brick;
        const unsigned zc = rem / cbpb, col = (rem - zc * cbpb) * 32u + (unsigned)lane;
        const int32_t* rg = p.ip.ranges + (size_t)p.ip.occupied[b] * 6;
        const int x0 = rg[0], nx = rg[1] - rg[0], y0 = rg[2], ny = rg[3] - rg[2];
        const int zb = max(rg[4] + (int)zc * p.zchunk, p.ip.z_begin);
        const int ze = min(min(rg[4] + (int)(zc + 1) * p.zchunk, rg[5]), p.ip.z_end);
        if (zb >= ze || (int)col >= nx * ny) continue;
        const int cy = (int)col / nx, cx = (int)col - cy * nx;
        march_column<N, MODE>(p.ip, x0 + cx, y0 + cy, zb, ze);
      }
    }
  }
}

// glClearTexImage(-limit) (recon_integration.cpp:250-251): 16-byte streaming stores over the slab.
// A slab may start at any voxel (odd plane sizes): scalar stores up to the first 16-byte boundary, vectors after it.
__global__ void __launch_bounds__(256) k_fill(float* __restrict__ dst, size_t n, float value) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t head = min(n, (size_t)((4u - (unsigned)((reinterpret_cast<uintptr_t>(dst) >> 2) & 3u)) & 3u));
  if (i < head) dst[i] = value;
  float* body = dst + head;
  const size_t nb = n - head, n4 = nb / 4;
  float4* d4 = reinterpret_cast<float4*>(body);
  const float4 v = make_float4(value, value, value, value);
  for (size_t j = i; j < n4; j += stride) __stcs(d4 + j, v);
  for (size_t j = n4 * 4 + i; j < nb; j += stride) body[j] = value;
}

// The cleared voxel as the 4 bytes the fill stores write: -limit (R32F), or half2(-limit, 0) for half2 voxels.
float cleared_voxel(int mode, float limit) {
  if (mode != 2) return -limit;
  const __half2 h = __floats2half2_rn(-limit, 0.0f);
  float f;
  std::memcpy(&f, &h, sizeof(f));
  return f;
}

// Launch-shape knobs of the integrator (rr_set_tunable; environment RR_<NAME> gives the initial value).
Tunables& tunables() {
  static Tunables t = [] {
    Tunables v;
    auto env = [](const char* n, int d) { const char* e = getenv(n); return e ? atoi(e) : d; };
    v.fused = env("RR_INTEGRATE_FUSED", v.fused);
    v.zchunk = env("RR_BRICK_ZCHUNK", v.zchunk);
    v.fill_rows = env("RR_FUSED_FILL_ROWS", v.fill_rows);
    v.fill_warps = env("RR_FUSED_FILL_WARPS", v.fill_warps);
    v.ctas = env("RR_FUSED_CTAS", v.ctas);
    v.threads = env("RR_FUSED_THREADS", v.threads);
    v.chunk = env("RR_FUSED_CHUNK", v.chunk);
    v.brick_grid = env("RR_BRICK_GRID", v.brick_grid);
    v.ldg256 = env("RR_LDG256", v.ldg256);
    v.graph = env("RR_GRAPH", v.graph);
    v.staged = env("RR_STAGED", v.staged);
    v.stage_zchunk = env("RR_STAGE_ZCHUNK", v.stage_zchunk);
    v.stage_ychunk = env("RR_STAGE_YCHUNK", v.stage_ychunk);
    v.stage_tile = env("RR_STAGE_TILE", v.stage_tile);
    v.stage_fill_rows = env("RR_STAGE_FILL_ROWS", v.stage_fill_rows);
    return v;
  }();
  return t;
}

void setup_fill(const rr_ctx* c, const IntegrateParams& p, int mode, int fill_rows, FusedParams& f) {
  f.ip = p;
  f.rowmask = c->d_rowmask.ptr; f.rowany = c->d_rowany.ptr; f.cand_y = c->d_cand_y.ptr; f.cand_z = c->d_cand_z.ptr;
  f.mask_words = c->mask_words; f.nby = (int)c->bricks.res[1];
  f.work = c->d_work.ptr;
  f.fill_rows = std::min(32, std::max(1, fill_rows));
  f.row_begin = (uint32_t)p.z_begin * (uint32_t)p.Y; f.row_end = (uint32_t)p.z_end * (uint32_t)p.Y;
  f.fill_items = (f.row_end - f.row_begin + (uint32_t)f.fill_rows - 1u) / (uint32_t)f.fill_rows;
  f.fill_value = cleared_voxel(mode, p.limit);
}

static void brick_extents(const rr_ctx* c, int& max_cols, int& max_nz) {
  max_cols = max_nz = 0;
  for (size_t i = 0; i + 5 < c->h_ranges.size(); i += 6) {
    max_cols = std::max(max_cols, (c->h_ranges[i + 1] - c->h_ranges[i]) * (c->h_ranges[i + 3] - c->h_ranges[i + 2]));
    max_nz = std::max(max_nz, c->h_ranges[i + 5] - c->h_ranges[i + 4]);
  }
}

template <int N>
static int launch_bricks_n(rr_ctx* c, const IntegrateParams& p, int mode) {
  int max_cols, max_nz;
  brick_extents(c, max_cols, max_nz);
  if (max_cols == 0 || max_nz == 0) return RR_OK;
  // block size: the multiple of 32 (128..320) that wastes the fewest lanes on a brick's column count
  int threads = 256;
  double best = 1e9;
  for (int t = 128; t <= BRICK_MAX_THREADS; t += 32) {
    const double waste = double((max_cols + t - 1) / t * t) / double(max_cols);
    if (waste < best - 1e-9 || (waste < best + 1e-9 && t > threads)) { best = waste; threads = t; }
  }
  const int zchunk = 9;
  const dim3 grd(148 * std::max(1, tunables().brick_grid), 1, 1);
  c->last_integrate[0] = 3; c->last_integrate[3] = (uint32_t)threads;
  if (mode == 1) k_integrate_bricks<N, 1, 2><<<grd, threads, 0, c->stream>>>(p, max_cols, max_nz, zchunk);
  else if (mode == 2) k_integrate_bricks<N, 2, 2><<<grd, threads, 0, c->stream>>>(p, max_cols, max_nz, zchunk);
  else k_integrate_bricks<N, 0, 2><<<grd, threads, 0, c->stream>>>(p, max_cols, max_nz, zchunk);
  RR_LAUNCH_CHECK(c, "k_integrate_bricks");
  return RR_OK;
}

template <int N>
static int launch_n(rr_ctx* c, const IntegrateParams& p, bool bricks, int mode, bool fused) {
  const dim3 blk(32, 8, 1);
  const Tunables& tn = tunables();
  if (bricks) {
    int max_cols, max_nz;
    brick_extents(c, max_cols, max_nz);
    if (max_cols == 0 || max_nz == 0) return RR_OK;
    if (fused) {
      // z-chunks: split a brick's z extent into pieces of ~zchunk voxels of equal size
      const int want = std::max(1, tn.zchunk);
      const int n_zchunks = std::max(1, (max_nz + want - 1) / want);
      FusedParams f{};
      setup_fill(c, p, mode, tn.fill_rows, f);
      f.max_cols = max_cols; f.max_nz = max_nz; f.n_zchunks = n_zchunks; f.zchunk = (max_nz + n_zchunks - 1) / n_zchunks;
      f.fill_warps = tn.fill_warps;
      // chunk <= 0: one z-chunk of one brick (all its column blocks) per draw
      f.chunk = tn.chunk > 0 ? tn.chunk : (max_cols + 31) / 32;
      cudaMemsetAsync(c->d_work.ptr, 0, 4 * sizeof(uint32_t), c->stream);
      const dim3 grd(148 * std::min(2, std::max(1, tn.ctas)), 1, 1);
      c->last_integrate[0] = 2;
      c->last_integrate[3] = N > 4 ? 256u : (mode == 0 && tn.threads != 384 ? 512u : 384u);
      if constexpr (N > 4) {
        // 6 registers of plane state per sensor: more than 4 sensors get 256-thread CTAs (128 registers)
        if (mode == 1) k_integrate_fused<N, 1, 256><<<grd, 256, 0, c->stream>>>(f);
        else if (mode == 2) k_integrate_fused<N, 2, 256><<<grd, 256, 0, c->stream>>>(f);
        else k_integrate_fused<N, 0, 256><<<grd, 256, 0, c->stream>>>(f);
      } else {
        if (mode == 1) k_integrate_fused<N, 1, 384><<<grd, 384, 0, c->stream>>>(f);
        else if (mode == 2) k_integrate_fused<N, 2, 384><<<grd, 384, 0, c->stream>>>(f);
        else if (tn.threads == 384) k_integrate_fused<N, 0, 384><<<grd, 384, 0, c->stream>>>(f);
        else k_integrate_fused<N, 0, 512><<<grd, 512, 0, c->stream>>>(f);
      }
      RR_LAUNCH_CHECK(c, "k_integrate_fused");
      return RR_OK;
    }
    return launch_bricks_n<N>(c, p, mode);
  } else {
    const int nz = p.z_end - p.z_begin;
    const dim3 grd((p.X + 31) / 32, (p.Y + 7) / 8, (nz + p.z_chunk - 1) / p.z_chunk);
    c->last_integrate[0] = 4; c->last_integrate[3] = blk.x * blk.y;
    if (mode == 1) k_integrate_dense<N, 1><<<grd, blk, 0, c->stream>>>(p);
    else if (mode == 2) k_integrate_dense<N, 2><<<grd, blk, 0, c->stream>>>(p);
    else k_integrate_dense<N, 0><<<grd, blk, 0, c->stream>>>(p);
  }
  RR_LAUNCH_CHECK(c, "k_integrate");
  return RR_OK;
}

// (k0, k1, g, 1-g) of every fine z against the inverse volume's z axis; rebuilt when either resolution changes
int build_ztab(rr_ctx* c) {
  const int Z = (int)c->res[2], IZ = (int)c->ires[2];
  if (c->d_ztab.ptr && c->ztab_Z == Z && c->ztab_IZ == IZ) return RR_OK;
  RR_TRY_RC(c->d_ztab.allocate(c, (size_t)Z, "integrate: z table"));
  k_build_ztab<<<(Z + 127) / 128, 128, 0, c->stream>>>(c->d_ztab.ptr, Z, IZ);
  RR_LAUNCH_CHECK(c, "k_build_ztab");
  c->ztab_Z = Z; c->ztab_IZ = IZ;
  return RR_OK;
}

int launch_integrate(rr_ctx* c) {
  IntegrateParams p{};
  p.inv = c->d_inv.ptr; p.gather = c->d_gather.ptr; p.tsdf = c->d_tsdf.ptr; p.weight = c->d_weight.ptr;
  p.ranges = c->d_ranges.ptr; p.occupied = c->d_occupied.ptr; p.num_occupied = c->d_num_occ.ptr;
  p.IX = (int)c->ires[0]; p.IY = (int)c->ires[1]; p.IZ = (int)c->ires[2];
  p.W = c->W; p.H = c->H; p.X = (int)c->res[0]; p.Y = (int)c->res[1]; p.Z = (int)c->res[2];
  p.z_begin = (int)c->slab_z0; p.z_end = (int)c->slab_z1;
  p.plane_elems = (unsigned)(c->res[0] * c->res[1]);
  if (c->slab_z0 > 0 || c->slab_z1 < c->res[2]) {
    // a slab owner also computes a read-only halo: the raymarcher's refinement and gradient taps reach at most
    // 2 * (limit/2) * Z voxels (+1 for the trilinear tap) past the owned samples; integration is pure, so the halo is
    // recomputed locally instead of exchanged
    const int halo = (int)std::ceil(c->cfg.limit * (float)c->res[2]) + 2;
    p.z_begin = std::max(0, p.z_begin - halo);
    p.z_end = std::min((int)c->res[2], p.z_end + halo);
  }
  p.z_chunk = 32;
  p.fW = (float)c->W; p.fH = (float)c->H; p.exmax = (float)(c->W - 1); p.eymax = (float)(c->H - 1);
  RR_TRY_RC(build_ztab(c));
  p.ztab = c->d_ztab.ptr;
  p.pairs = c->d_pairs.ptr; p.pair_pitch = c->pair_pitch;
  p.limit = c->cfg.limit;
  p.wide_loads = tunables().ldg256;
  const int mode = c->cfg.store_weight == RR_VOXELS_HALF2 ? 2 : (c->cfg.store_weight != 0 ? 1 : 0);
  const bool weight = mode == 1;
  const bool bricks = c->cfg.use_bricks != 0;
  std::memset(c->last_integrate, 0, sizeof(c->last_integrate));
  c->last_integrate[1] = (uint32_t)c->N; c->last_integrate[2] = (uint32_t)mode;
  timer_begin(c, "2integrate");
  const size_t plane = (size_t)p.X * p.Y;
  const size_t nslab = plane * (size_t)(p.z_end - p.z_begin);
  // tunable fused=0 selects the two-kernel path (k_fill, then k_integrate_bricks) for A/B measurements
  const bool fused = bricks && tunables().fused != 0 && c->fused_ok;
  int rc = RR_OK;
  bool done = false;
  // first choice in bricks mode: the TMA-staged persistent kernel (rr_integrate_staged.cu); it declines (done = false) when
  // the configuration does not fit its shared-memory stages or its item lists are stale, and the direct kernels below take over
  if (fused && nslab && tunables().staged != 0) rc = launch_integrate_staged(c, p, mode, &done);
  if (!done && rc == RR_OK && nslab && !c->gather_packed) {
    // the last pre-process left the gather texels to the staged kernel, which is not the one running now
    rc = launch_pack_gather(c);
    c->last_integrate[4] |= 2u;
  }
  if (!done && rc == RR_OK) {
    if (bricks && !fused && nslab) {
      // dense mode overwrites every voxel, so only the brick path needs the clear
      float* t0 = c->d_tsdf.ptr + plane * p.z_begin;
      k_fill<<<148 * 8, 256, 0, c->stream>>>(t0, nslab, cleared_voxel(mode, p.limit));
      RR_LAUNCH_CHECK(c, "k_fill");
      if (weight) {
        k_fill<<<148 * 8, 256, 0, c->stream>>>(c->d_weight.ptr + plane * p.z_begin, nslab, 0.0f);
        RR_LAUNCH_CHECK(c, "k_fill");
      }
    }
    if (nslab) {
      switch (c->N) {
        case 1: rc = launch_n<1>(c, p, bricks, mode, fused); break;
        case 2: rc = launch_n<2>(c, p, bricks, mode, fused); break;
        case 3: rc = launch_n<3>(c, p, bricks, mode, fused); break;
        case 4: rc = launch_n<4>(c, p, bricks, mode, fused); break;
        case 5: rc = launch_n<5>(c, p, bricks, mode, fused); break;
        case 6: rc = launch_n<6>(c, p, bricks, mode, fused); break;
        case 7: rc = launch_n<7>(c, p, bricks, mode, fused); break;
        case 8: rc = launch_n<8>(c, p, bricks, mode, fused); break;
        default: return fail(c, RR_ERR_UNSUPPORTED, "integrate: 1..8 sensors supported");
      }
    }
    c->work_fresh = false;   // the fused kernel draws from the work counters too
  }
  timer_end(c, "2integrate");
  if (rc == RR_OK) { c->volume_integrated = true; ++c->volume_epoch; c->mesh_rows_ok = mesh_rows_usable(c); }
  return rc;
}

}  // namespace rr
