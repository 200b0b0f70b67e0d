// TSDF integration of the occupied bricks with TMA-staged operands (sm_100a): the per-voxel work of
// glsl/tsdf_integration.vs:23-59 driven like ReconIntegration::integrate (recon_integration.cpp:243-270), fused with the
// clear of the volume (glClearTexImage, :250-251) as in rr_integrate.cu's k_integrate_fused - same arithmetic (the device
// functions of rr_integrate.cuh), same results bit for bit, different data movement.
//
// Both operands of a voxel-sensor evaluation have addresses that do not depend on frame data:
//   * the inverse calibration volume (cv_xyz_inv) is sampled at the voxel centre: for a box of voxels the eight-corner
//     gathers cover an axis-aligned box of coarse texels, an affine function of the voxel range;
//   * the depth / quality / silhouette taps sit where the calibration projects the voxel: for a box of voxels they cover a
//     small rectangle of each sensor's image, fixed by calibration + brick grid and computed once (k_footprints).
// So a work item = (occupied brick, y-chunk, z-chunk) is served by 1 + N bulk tensor copies (cp.async.bulk.tensor, TMA):
// a 5-D box {xyzw, BX, BY, BZ, N} of the inverse volumes and one T x T tile per sensor of the "pair image"
// (depth_b.x, quality | silhouette sign; 8 bytes per pixel, border replicated so CLAMP_TO_EDGE needs no clamping).
// A persistent CTA per SM runs a two-stage mbarrier pipeline: one producer thread draws items from a global counter and
// issues the copies for item i+1 while CWARPS consumer warps evaluate item i out of shared memory (LDS only, no global
// loads in the voxel loop); FWARPS warps stream the clear (-limit) over every voxel outside the occupied bricks the whole
// time, and every warp that runs out of its own work helps with the clear.
#include "rr_integrate.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <utility>
#include <vector>

// Role-level cycle counters (rr_integrator_profile): compiled in only for `make prof` (librr_b200_prof.so), so that the
// shipped kernel's register allocation is not shaped by them.
#ifdef RR_STAGE_PROF
#define RR_PROF(...) __VA_ARGS__
#else
#define RR_PROF(...)
#endif

namespace rr {

struct StagedParams {
  FusedParams f;            // integrate parameters + clear stream
  int cy, cz, n_yc, n_zc;   // work item = brick x y-chunk x z-chunk (voxels per chunk, chunks per brick)
  int BX, BY, BZ, T;        // staged inverse-volume box per sensor (coarse texels) and pair-image tile edge (pixels)
  const uint2* fp;          // [bricks * n_yc * n_zc][N]: .x = tile origin tx0 | ty0 << 16, .y = footprint rectangle (bit 7: exceeds the tile)
  const uint2* list;        // [N + 1][list_stride]: this frame's items by cost class (.x item, .y verdict), written by k_bricks_update
  const uint32_t* class_count;   // [N + 1]
  uint32_t list_stride;
  uint32_t inv_bytes, tile_bytes;    // bytes one sensor's copies deliver (box, tile)
  uint32_t inv_span;        // offset of the tile inside a slot (TMA destinations are 128-byte aligned)
  uint32_t slot_bytes, n_slots, slots_off;   // ring of per-sensor operand slots behind the item headers
  uint32_t fill_src_off, fill_src_bytes;   // buffer of cleared voxels (source of the clear's bulk stores)
  uint32_t tables_off;      // shared-memory copies of cand_y [2Y], cand_z [2Z] (int16) and rowany [nby*nbz] behind that
  uint32_t n_rowany;
  uint32_t* err;            // [0] box overflow, [1] barrier time-out
  int fill_depth, fill_lsu; // tunables stage_fill_depth / stage_fill_lsu (FillSource)
  int tail_cap;             // tunable stage_tail_cap: items in flight per CTA once the list runs out (0: no limit)
  unsigned long long* prof; // stage_debug bit 7: cycle counters per role (rr_integrator_profile), else nullptr
  int debug;
};

// An item in flight = one header of the header ring + one operand slot per sensor that is evaluated voxel by voxel.
// The first 128 bytes of a header are written by the producer before it arms the header's full barrier; the item's slice
// of the z table follows (bulk copy).
struct ItemHdr {
  int valid;                // 0: no more items, 1: staged item, 2: direct item (operands stay in global memory)
  int x0, nx, y0, ny, zb, ze;
  // Per-sensor verdict of k_bricks_update for this frame: bit s of `skip` = every voxel of the item lies at least `limit`
  // behind everything sensor s sees in its footprint (tsdf_integration.vs:45 "do nothing"), bit s of `front` = at least
  // `limit` in front of it (:41 weighted_tsd = -limit); neither = evaluate voxel by voxel.
  uint32_t skip, front;
  uint32_t nslots;          // operand slots the item holds (returned to the ring when every consumer warp has left it)
  uint32_t ib[RR_MAX_SENSORS];   // byte offset (from the dynamic smem base) of inverse-volume texel (0, 0, 0) of sensor s, were the whole volume staged
  uint32_t tb[RR_MAX_SENSORS];   // ... and of pair texel (-1, -1) of sensor s: tile start - tile origin
};
#define ITEM_HDR_BYTES 128
#define ZT_MAX 56
#define HDR_BYTES (ITEM_HDR_BYTES + 16 * ZT_MAX)
#define NH 8                // headers = items in flight per CTA at most
static_assert(sizeof(ItemHdr) <= ITEM_HDR_BYTES, "item header must fit its slot");
static_assert(HDR_BYTES % 128 == 0, "TMA destinations are 128-byte aligned");

// ---- PTX: mbarrier + TMA ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
// try_wait suspends the thread in hardware until the phase completes or the time hint (ns) runs out: a waiting warp
// issues one instruction per hint period instead of spinning
__device__ __forceinline__ bool mbar_try_wait(uint64_t* b, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.b32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(smem_u32(b)), "r"(parity), "r"(100000u) : "memory");
  return ok != 0;
}
// A wait that never completes would hang the GPU, so a pipeline bug gives up after ~0.3 s of wall time, raises err[1]
// (rr_integrator_info reports it) and lets the role run out instead.
__device__ __forceinline__ bool mbar_wait(uint64_t* b, uint32_t parity, uint32_t* err) {
  if (mbar_try_wait(b, parity)) return true;
  unsigned long long t0, t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  while (!mbar_try_wait(b, parity)) {
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    if (t - t0 > 300000000ull) {
      atomicOr(err + 1, 1u);
      return false;
    }
  }
  return true;
}
// plain bulk copy global -> shared (1-D TMA): src, dst and size multiples of 16 bytes
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// L2 policies: the integrator's operands (a few tens of MB per frame) are re-read every frame and should survive the
// 0.5 GB of clear traffic that streams through L2 in the same kernel, so loads ask for evict_last, the clear for evict_first.
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3, int c4, uint64_t policy) {
  asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5, %6, %7}], [%2], %8;"
               ::"r"(dst), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "l"(policy) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, uint64_t policy) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
               ::"r"(dst), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "l"(policy) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)map) : "memory");
}

// ---- one (x, y) column of a staged item ---------------------------------------------------------------------------
// Same plane / tap / decision arithmetic as march_column (rr_integrate.cuh), operands read from the item's slots:
//   inverse-volume corners: float4 at ib[s] + ((k*BY + y)*BX + x) * 16
//   pair texels of the footprint (ex, ey): float2 at tb[s] + (ey*T + ex)*8, +8, +T*8, +T*8+8
template <int N, int MODE>
__device__ __forceinline__ void march_staged(const IntegrateParams& p, const uint8_t* __restrict__ smem, const ItemHdr* __restrict__ h,
                                             int BX, uint32_t ps, int T, int x, int y) {
  // Register budget: 72 per thread with 22 consumer warps. Everything warp-uniform that is needed once per voxel or less
  // (slot bases, z range, verdict masks) stays in the item header and is re-read by LDS (a broadcast) where it is used.
  float a, b;
  uint32_t cxy, dX, dY;            // byte offset of the (x0, y0) corner inside a coarse plane; +dX: x1, +dY: y1
  {
    const float stepX = 1.0f / (float)p.X, stepY = 1.0f / (float)p.Y;
    const float px = ((float)x + 0.5f) * stepX, py = ((float)y + 0.5f) * stepY;
    int x0, x1, y0, y1;
    lin_coord(px, p.IX, x0, x1, a);
    lin_coord(py, p.IY, y0, y1, b);
    cxy = (uint32_t)(y0 * BX + x0) << 4;
    dX = (uint32_t)(x1 - x0) << 4;
    dY = (uint32_t)((y1 - y0) * BX) << 4;
  }
  const uint32_t masks = h->skip | h->front | (h->front << 8);     // bits 0-7: no per-voxel work, bits 8-15: front
  float3 A[N], B[N];
#pragma unroll
  for (int s = 0; s < N; ++s) A[s] = B[s] = make_float3(0.f, 0.f, 0.f);
  int ck0 = -1, ck1 = -1;

  auto plane = [&](int s, int k) -> float3 {
    if ((masks >> s) & 1u) return make_float3(0.f, 0.f, 0.f);
    const uint8_t* q = smem + (h->ib[s] + (uint32_t)k * ps + cxy);
    const float4 p00 = *reinterpret_cast<const float4*>(q), p10 = *reinterpret_cast<const float4*>(q + dX);
    const float4 p01 = *reinterpret_cast<const float4*>(q + dY), p11 = *reinterpret_cast<const float4*>(q + dY + dX);
    return plane_reduce(p00, p10, p01, p11, a, 1.0f - a, b, 1.0f - b);
  };

  const int zb = h->zb;
  unsigned o = (unsigned)((zb * p.Y + y) * p.X + x);
  const float4* zt_ptr = reinterpret_cast<const float4*>(reinterpret_cast<const uint8_t*>(h) + ITEM_HDR_BYTES);   // the item's slice of the z table
  const float4* zt_end = zt_ptr + (h->ze - zb);
  for (; zt_ptr < zt_end; ++zt_ptr, o += p.plane_elems) {
    const float4 zt = *zt_ptr;
    const int k0 = __float_as_int(zt.x), k1 = __float_as_int(zt.y);
    const float g = zt.z, omg = zt.w;
    if (k0 != ck0) {
      if (k0 == ck1) {
#pragma unroll
        for (int s = 0; s < N; ++s) A[s] = B[s];
      } else {
#pragma unroll
        for (int s = 0; s < N; ++s) A[s] = plane(s, k0);
      }
      ck0 = k0;
    }
    if (k1 != ck1) {
      if (k1 == k0) {
#pragma unroll
        for (int s = 0; s < N; ++s) B[s] = A[s];
      } else {
#pragma unroll
        for (int s = 0; s < N; ++s) B[s] = plane(s, k1);
      }
      ck1 = k1;
    }
    float weighted_tsd = p.limit, total_weight = 0.0f;
#pragma unroll
    for (int s = 0; s < N; ++s) {
      if (!((masks >> s) & 1u)) {
        float wa, wb, d;
        int ex, ey;                // lower-left texel clamped to [-1, W-1]; the + 1 of the footprint index lives in tb[s]
        tap_coords(A[s], B[s], g, omg, p.fW, p.fH, p.exmax, p.eymax, wa, wb, d, ex, ey);
        const uint8_t* q = smem + (h->tb[s] + ((uint32_t)(ey * T + ex) << 3));
        const float2 t00 = *reinterpret_cast<const float2*>(q), t10 = *reinterpret_cast<const float2*>(q + 8);
        const float2 t01 = *reinterpret_cast<const float2*>(q + (T << 3)), t11 = *reinterpret_cast<const float2*>(q + (T << 3) + 8);
        fuse_tap(wa, wb, d, t00.x, t10.x, t01.x, t11.x, t00.y, t10.y, t01.y, t11.y, p.limit, -p.limit, weighted_tsd, total_weight);
      } else if ((masks >> (8 + s)) & 1u) {
        weighted_tsd = -p.limit;
      }
    }
    store_voxel<MODE>(p, o, weighted_tsd, total_weight);
  }
}

// Cold path of the kernel below, kept out of line so that its register needs do not shape the staged loop's allocation.
template <int N, int MODE>
__device__ __noinline__ void march_direct(const IntegrateParams& p, int x, int y, int zb, int ze) {
  march_column<N, MODE, true>(p, x, y, zb, ze);
}

// ---- the kernel ------------------------------------------------------------------------------------------------------
// The CTA is launched as whole warpgroups: the CWARPS consumer warps rounded up to warpgroups, then two auxiliary
// warpgroups = the producer warp + seven clear warps. It starts at 65536 / threads registers per thread; the auxiliary
// warpgroups then give registers back (setmaxnreg.dec to 40) and the consumer warpgroups take them (setmaxnreg.inc to 72
// with 22 consumer warps, 144 with 11): the clear gets enough warps to keep HBM busy while the brick evaluation keeps its
// register budget.
//
// Items flow through a ring of NH headers and a ring of operand slots (one slot = one sensor's inverse-volume box + its
// pair-image tile). The producer (one thread) draws an item from this frame's class-sorted list, takes a header and as
// many slots as the item has sensors to evaluate voxel by voxel - sensors a verdict has settled need no operands - and
// issues the copies against the header's `full` barrier without waiting for them: an average item of the bench workload
// holds 3 of 10 slots, so three to four items are in flight and a consumer warp that finishes early runs ahead instead of
// waiting. Consumer warps walk the headers in order; the last one to leave an item completes its `empty` barrier, which
// is what the producer waits on (oldest item first) when it needs a header or slots back.
template <int CWARPS> struct StagedShape {
  static constexpr int kConsumerWG = (CWARPS + 3) / 4;
  static constexpr int kThreads = (kConsumerWG + 2) * 128;
  static constexpr int kProducerWarp = kConsumerWG * 4;
  static constexpr int kAuxRegs = 40;
  // setmaxnreg needs the kernel's register count declared (.maxnreg)
  static constexpr int kLaunchRegs = (65536 / kThreads) / 8 * 8;
  // the CTA's pool is what it was launched with: the consumers can take what the auxiliary warpgroups give back, no more
  // (asking for more would block forever)
  static constexpr int kConsumerRegs = ((kThreads * kLaunchRegs - 256 * kAuxRegs) / (kConsumerWG * 128)) / 8 * 8;
  static_assert(kConsumerRegs >= kLaunchRegs && kConsumerRegs <= 255 && kAuxRegs <= kLaunchRegs, "register reallocation plan");
};

template <int N, int MODE, int CWARPS>
__global__ void __maxnreg__((StagedShape<CWARPS>::kLaunchRegs))
k_integrate_staged(const __grid_constant__ StagedParams p, const __grid_constant__ CUtensorMap map_inv, const __grid_constant__ CUtensorMap map_pairs) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t s_full[NH], s_empty[NH];
  // TMA destinations must be 128-byte aligned; the dynamic window's own alignment is only guaranteed to 16
  uint8_t* smem = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < NH; ++i) { mbar_init(&s_full[i], 1); mbar_init(&s_empty[i], CWARPS); }
    mbar_fence_init();
  }
  // the clear's bulk-store source: fill_src_bytes of cleared voxels (then as many zero bytes for a separate weight volume)
  for (uint32_t i = threadIdx.x * 4u; i < p.fill_src_bytes * (MODE == 1 ? 2u : 1u); i += blockDim.x * 4u)
    *reinterpret_cast<float*>(smem + p.fill_src_off + i) = i < p.fill_src_bytes ? p.f.fill_value : 0.0f;
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic-proxy writes -> visible to the async proxy (TMA reads)
  // the clear's row tables, once per CTA
  int16_t* s_cand_y = reinterpret_cast<int16_t*>(smem + p.tables_off);
  int16_t* s_cand_z = s_cand_y + 2 * p.f.ip.Y;
  uint8_t* s_rowany = reinterpret_cast<uint8_t*>(s_cand_z + 2 * p.f.ip.Z);
  for (int i = threadIdx.x; i < 2 * p.f.ip.Y; i += blockDim.x) s_cand_y[i] = p.f.cand_y[i];
  for (int i = threadIdx.x; i < 2 * p.f.ip.Z; i += blockDim.x) s_cand_z[i] = p.f.cand_z[i];
  for (uint32_t i = threadIdx.x; i < p.n_rowany; i += blockDim.x) s_rowany[i] = p.f.rowany[i];
  __syncthreads();
  RR_PROF(const long long t_start = clock64();)
  const FillTables ft{s_cand_y, s_cand_z, s_rowany};
  const IntegrateParams& ip = p.f.ip;
  using Shape = StagedShape<CWARPS>;
  constexpr int PWARP = Shape::kProducerWarp;
  const FillSource fs{smem_u32(smem + p.fill_src_off), p.fill_src_bytes, (p.debug & 32) != 0, l2_policy_evict_first(), p.fill_depth, p.fill_lsu != 0};

  // ---- producer (one thread)
  auto producer = [&]() {
    tma_prefetch_desc(&map_inv);
    tma_prefetch_desc(&map_pairs);
    const uint64_t keep = l2_policy_evict_last();
    uint32_t cnt[N + 1];
#pragma unroll
    for (int k = 0; k <= N; ++k) cnt[k] = (p.debug & 2) ? 0u : min(p.class_count[k], p.list_stride);
    const uint32_t per_brick = (uint32_t)(p.n_yc * p.n_zc);
    const float stepX = 1.0f / (float)ip.X, stepY = 1.0f / (float)ip.Y;
    uint32_t j = 0, tail = 0, slots_free = p.n_slots, slot_head = 0;      // items pushed / retired, the slot ring
    auto hdr = [&](uint32_t k) { return reinterpret_cast<ItemHdr*>(smem + (k % NH) * HDR_BYTES); };
    // wait until the oldest item in flight has been consumed; its slots return to the ring
    auto retire = [&]() -> bool {
      if (!mbar_wait(&s_empty[tail % NH], (tail / NH) & 1u, p.err)) return false;
      slots_free += hdr(tail)->nslots;
      ++tail;
      return true;
    };
    RR_PROF(long long tp0 = clock64(); long long tp1 = 0; long long t_meta = 0; long long t_empty = 0; long long n_staged = 0; long long n_direct = 0;)
    uint32_t total = 0, seen = 0;             // items of this frame, and the last index this producer drew
#pragma unroll
    for (int k = 0; k <= N; ++k) total += cnt[k];
    for (;;) {
      // Items drawn early are items other CTAs cannot take: towards the end of the list the run-ahead shrinks with what is
      // left per CTA (down to one item at a time), so that the last items spread over all SMs instead of queueing in a few.
      if (p.tail_cap > 0) {
        const uint32_t left = total > seen ? (total - seen) / gridDim.x : 0u;
        const uint32_t cap = min(max(left, (uint32_t)p.tail_cap), (uint32_t)NH);
        while (j - tail >= cap) if (!retire()) return;
      }
      const uint32_t it = atomicAdd(p.f.work, 1u);
      seen = it;
      // the most expensive class first
      int cls = -1;
      uint32_t idx = it;
#pragma unroll
      for (int k = N; k >= 0; --k)
        if (cls < 0) { if (idx < cnt[k]) cls = k; else idx -= cnt[k]; }
      if (cls < 0) {
        while (j - tail >= NH) if (!retire()) return;
        ItemHdr* h = hdr(j);
        h->valid = 0; h->nslots = 0;
        mbar_arrive(&s_full[j % NH]);
        RR_PROF(if (p.prof) {
          atomicAdd(p.prof + 4, (unsigned long long)t_meta); atomicAdd(p.prof + 5, (unsigned long long)t_empty);
          atomicAdd(p.prof + 7, (unsigned long long)n_staged); atomicAdd(p.prof + 8, (unsigned long long)n_direct);
        })
        return;
      }
      const uint2 e = p.list[(size_t)cls * p.list_stride + idx];
      const uint32_t item = e.x;
      const uint32_t brick = item / per_brick, r = item - brick * per_brick;
      const int yc = (int)(r / (uint32_t)p.n_zc), zc = (int)(r - (uint32_t)yc * (uint32_t)p.n_zc);
      const int32_t* rg = ip.ranges + (size_t)brick * 6;
      const int x0 = rg[0], x1 = rg[1];
      const int yb = rg[2] + yc * p.cy, ye = min(yb + p.cy, rg[3]);
      const int zb = max(rg[4] + zc * p.cz, ip.z_begin), ze = min(min(rg[4] + (zc + 1) * p.cz, rg[5]), ip.z_end);
      if (x0 >= x1 || yb >= ye || zb >= ze) continue;
      const uint32_t verdict = (p.debug & 4) ? 0u : e.y;
      const uint32_t off = (verdict | (verdict >> 8)) & ((1u << N) - 1u);      // sensors a verdict has settled
      const uint2* fp = p.fp + (size_t)item * N;
      uint2 f[N];
#pragma unroll
      for (int s = 0; s < N; ++s) f[s] = fp[s];
      bool direct = false;                     // a footprint that has to be read exceeds the tile: global-memory path
#pragma unroll
      for (int s = 0; s < N; ++s) direct = direct || (!((off >> s) & 1u) && (f[s].y & 128u));
      const uint32_t act = direct ? 0u : (uint32_t)N - (uint32_t)__popc(off);
      // coarse box of the item: lin_coord is monotone, so the first / last voxel bound every corner index
      int ixlo = 0, iylo = 0, izlo = 0;
      if (!direct) {
        int i0, i1, ixhi, iyhi; float w;
        lin_coord(((float)x0 + 0.5f) * stepX, ip.IX, ixlo, i1, w);
        lin_coord(((float)(x1 - 1) + 0.5f) * stepX, ip.IX, i0, ixhi, w);
        lin_coord(((float)yb + 0.5f) * stepY, ip.IY, iylo, i1, w);
        lin_coord(((float)(ye - 1) + 0.5f) * stepY, ip.IY, i0, iyhi, w);
        izlo = __float_as_int(ip.ztab[zb].x);
        const int izhi = __float_as_int(ip.ztab[ze - 1].y);
        if (ixhi - ixlo >= p.BX || iyhi - iylo >= p.BY || izhi - izlo >= p.BZ) { atomicOr(p.err, 1u); continue; }
      }
      // everything above overlapped the consumers' work; now a header and the item's slots are needed
      RR_PROF(tp1 = clock64(); t_meta += tp1 - tp0;)
      while (j - tail >= NH || slots_free < act) if (!retire()) return;
      RR_PROF(tp0 = clock64(); t_empty += tp0 - tp1;)
      const uint32_t hs = j % NH;
      ItemHdr* h = hdr(j);
      h->valid = direct ? 2 : 1;
      h->x0 = x0; h->nx = x1 - x0; h->y0 = yb; h->ny = ye - yb; h->zb = zb; h->ze = ze;
      h->skip = verdict & 255u; h->front = (verdict >> 8) & 255u;
      h->nslots = act;
      if (direct) {
        mbar_arrive(&s_full[hs]);              // nothing to copy
        RR_PROF(++n_direct;)
      } else {
        const uint32_t first = slot_head;
        const uint32_t vol0 = (uint32_t)((izlo * p.BY + iylo) * p.BX + ixlo) << 4;
#pragma unroll
        for (int s = 0; s < N; ++s) {
          if ((off >> s) & 1u) continue;
          const uint32_t slot = p.slots_off + slot_head * p.slot_bytes;
          slot_head = slot_head + 1u == p.n_slots ? 0u : slot_head + 1u;
          h->ib[s] = slot - vol0;
          h->tb[s] = slot + p.inv_span + ((uint32_t)(p.T + 1) << 3) - ((((f[s].x >> 16) * (uint32_t)p.T) + (f[s].x & 0xffffu)) << 3);
        }
        const uint32_t zt_bytes = (uint32_t)(ze - zb) * 16u;
        mbar_expect_tx(&s_full[hs], zt_bytes + act * (p.inv_bytes + p.tile_bytes));
        const uint32_t base = smem_u32(smem);
        bulk_load(base + hs * HDR_BYTES + ITEM_HDR_BYTES, ip.ztab + zb, zt_bytes, &s_full[hs]);
        uint32_t sl = first;
#pragma unroll
        for (int s = 0; s < N; ++s) {
          if ((off >> s) & 1u) continue;
          const uint32_t dst = base + p.slots_off + sl * p.slot_bytes;
          sl = sl + 1u == p.n_slots ? 0u : sl + 1u;
          tma_load_5d(dst, &map_inv, &s_full[hs], 0, ixlo, iylo, izlo, s, keep);
          tma_load_3d(dst + p.inv_span, &map_pairs, &s_full[hs], (int)(f[s].x & 0xffffu), (int)(f[s].x >> 16), s, keep);
        }
        RR_PROF(++n_staged; if (p.prof) {
          uint32_t need = 0;
          for (int s = 0; s < N; ++s)
            if (!((off >> s) & 1u)) need = max(need, max((f[s].y & 127u) + ((f[s].y >> 8) & 4095u), f[s].y >> 20));
          atomicMax(p.prof + 13, (unsigned long long)need); atomicAdd(p.prof + 3, (unsigned long long)act);
          if (need <= 30u) atomicAdd(p.prof + 14, 1ull);
          if (need <= 36u) atomicAdd(p.prof + 15, 1ull);
        })
      }
      slots_free -= act;
      ++j;
      RR_PROF(tp0 = clock64();)
    }
  };
  // ---- consumers: the headers in order, until the producer signals the end
  auto consumer = [&]() {
    const uint32_t ps = (uint32_t)(p.BX * p.BY) << 4;
    RR_PROF(long long tc0 = clock64(); long long t_wait = 0; long long t_work = 0; long long t_idle = 0;)
    for (uint32_t j = 0;; ++j) {
      const uint32_t hs = j % NH;
      if (!mbar_wait(&s_full[hs], (j / NH) & 1u, p.err)) return;
      RR_PROF({ const long long t = clock64(); t_wait += t - tc0; tc0 = t; })
      const ItemHdr* h = reinterpret_cast<const ItemHdr*>(smem + hs * HDR_BYTES);
      if (!h->valid) break;
      // one column per thread: the host sizes the y-chunk so that an item's columns fit the consumer threads
      const int nx = h->nx, col = (int)threadIdx.x;
      if (col < nx * h->ny) {
        const int cyv = col / nx, x = h->x0 + (col - cyv * nx), y = h->y0 + cyv;
        if (h->valid == 2) march_direct<N, MODE>(ip, x, y, h->zb, h->ze);      // oversize footprint: operands from global memory
        else march_staged<N, MODE>(ip, smem, h, p.BX, ps, p.T, x, y);
      }
      __syncwarp();
      RR_PROF({ const long long t = clock64(); if (col - lane < nx * h->ny) t_work += t - tc0; else t_idle += 1; tc0 = t; })
      if (lane == 0) mbar_arrive(&s_empty[hs]);
    }
    RR_PROF(if (p.prof && lane == 0) {
      atomicAdd(p.prof + 0, (unsigned long long)t_wait); atomicAdd(p.prof + 1, (unsigned long long)t_work);
      atomicAdd(p.prof + 2, (unsigned long long)t_idle);
    })
  };
  // ---- clear stream: the clear warps from the start, everybody else once their own work is done
  auto clear = [&]() {
    RR_PROF(const long long t0 = clock64();)
    fill_loop_bulk<MODE == 1>(p.f, ft, lane, fs);
    RR_PROF(if (p.prof && lane == 0) {
      atomicAdd(p.prof + (warp > PWARP ? 9 : 10), (unsigned long long)(clock64() - t0));
      atomicMax(p.prof + 11, (unsigned long long)(clock64() - t_start));
      atomicAdd(p.prof + 12, (unsigned long long)(clock64() - t_start));
    })
  };
  const bool helpers_clear = !(p.debug & 16);
  // each role's code sits behind its own setmaxnreg, so that ptxas allocates it against that budget
  if (warp < PWARP) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(Shape::kConsumerRegs));
    if (warp < CWARPS) consumer();
    if (helpers_clear) clear();
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(Shape::kAuxRegs));
    if (warp == PWARP) {
      if (lane == 0) producer();
      __syncwarp();
      if (helpers_clear) clear();
    } else {
      clear();
    }
  }
}

// ---- footprints ------------------------------------------------------------------------------------------------------
// One block per (brick, y-chunk, z-chunk) of the WHOLE brick grid (occupancy changes per frame, the footprints do not):
// every voxel of the item runs the plane / tap arithmetic of the integrator and the block reduces the footprint indices
// (ex, ey) per sensor to their bounding rectangle. out[item][s] = (exmin, eymin, exmax, eymax); empty item: exmax < exmin.
template <int N>
__global__ void __launch_bounds__(256) k_footprints(const __grid_constant__ IntegrateParams p, int cy, int cz, int n_yc, int n_zc, int4* __restrict__ out,
                                                    float2* __restrict__ out_z) {
  __shared__ int s_red[8][RR_MAX_SENSORS][4];
  __shared__ float s_redz[8][RR_MAX_SENSORS][2];
  const uint32_t item = blockIdx.x;
  const uint32_t per_brick = (uint32_t)(n_yc * n_zc);
  const uint32_t brick = item / per_brick, r = item - brick * per_brick;
  const int yc = (int)(r / (uint32_t)n_zc), zc = (int)(r - (uint32_t)yc * (uint32_t)n_zc);
  const int32_t* rg = p.ranges + (size_t)brick * 6;
  const int x0 = rg[0], nx = rg[1] - rg[0];
  const int yb = rg[2] + yc * cy, ye = min(yb + cy, rg[3]);
  const int zb = rg[4] + zc * cz, ze = min(zb + cz, rg[5]);
  int mn_x[N], mn_y[N], mx_x[N], mx_y[N];
  float zlo[N], zhi[N];              // range of pos_calib.z over the item; any non-finite value widens it to (-inf, inf)
  const float inf = __int_as_float(0x7f800000);
#pragma unroll
  for (int s = 0; s < N; ++s) { mn_x[s] = mn_y[s] = 0x7fffffff; mx_x[s] = mx_y[s] = -1; zlo[s] = inf; zhi[s] = -inf; }
  const int cols = (nx > 0 && ye > yb && ze > zb) ? nx * (ye - yb) : 0;
  const float stepX = 1.0f / (float)p.X, stepY = 1.0f / (float)p.Y;
  const unsigned plane_sz = (unsigned)(p.IX * p.IY);
  for (int col = (int)threadIdx.x; col < cols; col += (int)blockDim.x) {
    const int cyv = col / nx, cxv = col - cyv * nx;
    const float px = ((float)(x0 + cxv) + 0.5f) * stepX, py = ((float)(yb + cyv) + 0.5f) * stepY;
    int cx0, cx1, cy0, cy1; float a, b;
    lin_coord(px, p.IX, cx0, cx1, a);
    lin_coord(py, p.IY, cy0, cy1, b);
    const float oma = 1.0f - a, omb = 1.0f - b;
    const unsigned o00 = cy0 * p.IX + cx0, o10 = cy0 * p.IX + cx1, o01 = cy1 * p.IX + cx0, o11 = cy1 * p.IX + cx1;
    for (int z = zb; z < ze; ++z) {
      const float4 zt = __ldg(p.ztab + z);
      const int k0 = __float_as_int(zt.x), k1 = __float_as_int(zt.y);
#pragma unroll
      for (int s = 0; s < N; ++s) {
        const float4* b0 = p.inv + (unsigned)(s * p.IZ + k0) * plane_sz;
        const float4* b1 = p.inv + (unsigned)(s * p.IZ + k1) * plane_sz;
        const float3 A = plane_reduce(__ldg(b0 + o00), __ldg(b0 + o10), __ldg(b0 + o01), __ldg(b0 + o11), a, oma, b, omb);
        const float3 B = plane_reduce(__ldg(b1 + o00), __ldg(b1 + o10), __ldg(b1 + o01), __ldg(b1 + o11), a, oma, b, omb);
        float wa, wb, d; int ex, ey;
        tap_coords(A, B, zt.z, zt.w, p.fW, p.fH, p.exmax, p.eymax, wa, wb, d, ex, ey);
        ex += 1; ey += 1;
        mn_x[s] = min(mn_x[s], ex); mx_x[s] = max(mx_x[s], ex);
        mn_y[s] = min(mn_y[s], ey); mx_y[s] = max(mx_y[s], ey);
        if (fabsf(d) < inf) { zlo[s] = fminf(zlo[s], d); zhi[s] = fmaxf(zhi[s], d); } else { zlo[s] = -inf; zhi[s] = inf; }
      }
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int s = 0; s < N; ++s) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      mn_x[s] = min(mn_x[s], __shfl_xor_sync(0xffffffffu, mn_x[s], d)); mn_y[s] = min(mn_y[s], __shfl_xor_sync(0xffffffffu, mn_y[s], d));
      mx_x[s] = max(mx_x[s], __shfl_xor_sync(0xffffffffu, mx_x[s], d)); mx_y[s] = max(mx_y[s], __shfl_xor_sync(0xffffffffu, mx_y[s], d));
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      zlo[s] = fminf(zlo[s], __shfl_xor_sync(0xffffffffu, zlo[s], d)); zhi[s] = fmaxf(zhi[s], __shfl_xor_sync(0xffffffffu, zhi[s], d));
    }
    if (lane == 0) {
      s_red[warp][s][0] = mn_x[s]; s_red[warp][s][1] = mn_y[s]; s_red[warp][s][2] = mx_x[s]; s_red[warp][s][3] = mx_y[s];
      s_redz[warp][s][0] = zlo[s]; s_redz[warp][s][1] = zhi[s];
    }
  }
  __syncthreads();
  if (threadIdx.x < N) {
    const int s = threadIdx.x;
    int4 v = make_int4(0x7fffffff, 0x7fffffff, -1, -1);
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
      v.x = min(v.x, s_red[w][s][0]); v.y = min(v.y, s_red[w][s][1]); v.z = max(v.z, s_red[w][s][2]); v.w = max(v.w, s_red[w][s][3]);
    }
    out[(size_t)item * N + s] = v;
    float2 zr = make_float2(inf, -inf);
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { zr.x = fminf(zr.x, s_redz[w][s][0]); zr.y = fmaxf(zr.y, s_redz[w][s][1]); }
    out_z[(size_t)item * N + s] = zr;
  }
}

// ---- host ------------------------------------------------------------------------------------------------------------
// lin_coord (rr_math.cuh) on the host: same float operations (this file is compiled with -ffp-contract=off)
static void h_lin_coord(float s, int W, int& i0, int& i1) {
  const float u = s * (float)W - 0.5f;
  const float f = floorf(u);
  auto cl = [&](float v) { return !(v >= 0.0f) ? 0 : (v >= (float)(W - 1) ? W - 1 : (int)v); };
  i0 = cl(f);
  i1 = cl(f + 1.0f);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) f = nullptr;
    cudaGetLastError();
    return (EncodeTiledFn)f;
  }();
  return fn;
}

template <int N, int CWARPS>
static int launch_staged_n(rr_ctx* c, const StagedParams& sp, int mode) {
  const auto& st = c->sti;
  // one persistent CTA per SM; tunable stage_ctas leaves SMs free (a collective library's kernels cannot share an SM with
  // a CTA that holds its whole register file and shared memory)
  const int ctas = tunables().stage_ctas > 0 ? std::min(tunables().stage_ctas, c->num_sms) : c->num_sms;
  const dim3 grd((unsigned)std::max(1, ctas), 1, 1), blk(StagedShape<CWARPS>::kThreads, 1, 1);
  auto go = [&](auto kern) -> int {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)st.smem_bytes);
    if (e != cudaSuccess) return check(c, e, "k_integrate_staged shared memory");
    kern<<<grd, blk, st.smem_bytes, c->stream>>>(sp, st.map_inv, st.map_pairs);
    return RR_OK;
  };
  int rc;
  if (mode == 1) rc = go(k_integrate_staged<N, 1, CWARPS>);
  else if (mode == 2) rc = go(k_integrate_staged<N, 2, CWARPS>);
  else rc = go(k_integrate_staged<N, 0, CWARPS>);
  if (rc != RR_OK) return rc;
  RR_LAUNCH_CHECK(c, "k_integrate_staged");
  return RR_OK;
}

// consumer warps per CTA: up to four sensors run 22 warps (a 26 x 26 brick's 676 columns in one pass) at 72 registers;
// more sensors keep 6 more registers of plane state each: 16 warps at 96 registers (tunable stage_cwarps = 11: 11 at 144).
// Measured on 8 sensors / 1024^3 (profiles/r2_g_c5.log): 11 warps 2.50 ms, 16 warps 1.86 ms, 20 warps at 80 registers 2.25 ms
// (spills), pairs of sensors in flight 2.87 ms (spills).
static int consumer_warps(int N) {
  if (tunables().stage_cwarps == 11) return 11;
  return N <= 4 ? 22 : 16;
}

static int footprints(rr_ctx* c, const IntegrateParams& p, int cy, int cz, int n_yc, int n_zc, int4* d_out, float2* d_z, uint32_t items) {
  switch (c->N) {
    case 1: k_footprints<1><<<items, 256, 0, c->stream>>>(p, cy, cz, n_yc, n_zc, d_out, d_z); break;
    case 2: k_footprints<2><<<items, 256, 0, c->stream>>>(p, cy, cz, n_yc, n_zc, d_out, d_z); break;
    case 3: k_footprints<3><<<items, 256, 0, c->stream>>>(p, cy, cz, n_yc, n_zc, d_out, d_z); break;
    case 4: k_footprints<4><<<items, 256, 0, c->stream>>>(p, cy, cz, n_yc, n_zc, d_out, d_z); break;
    case 5: k_footprints<5><<<items, 256, 0, c->stream>>>(p, cy, cz, n_yc, n_zc, d_out, d_z); break;
    case 6: k_footprints<6><<<items, 256, 0, c->stream>>>(p, cy, cz, n_yc, n_zc, d_out, d_z); break;
    case 7: k_footprints<7><<<items, 256, 0, c->stream>>>(p, cy, cz, n_yc, n_zc, d_out, d_z); break;
    case 8: k_footprints<8><<<items, 256, 0, c->stream>>>(p, cy, cz, n_yc, n_zc, d_out, d_z); break;
    default: return fail(c, RR_ERR_UNSUPPORTED, "integrate: 1..8 sensors supported");
  }
  RR_LAUNCH_CHECK(c, "k_footprints");
  return RR_OK;
}

uint64_t staged_lists_key(const rr_ctx* c) {
  uint32_t limit;
  std::memcpy(&limit, &c->cfg.limit, sizeof(limit));
  return ((uint64_t)c->sti.tables << 32) | limit;
}

// the tunables the staged tables depend on, as one key (other knobs change launch shapes of the direct kernels only)
static unsigned staged_key() {
  const Tunables& tn = tunables();
  unsigned k = 2166136261u;
  for (int v : {tn.staged, tn.fused, tn.stage_zchunk, tn.stage_ychunk, tn.stage_tile, tn.stage_cwarps, tn.stage_bulk_fill}) k = (k ^ (unsigned)v) * 16777619u;
  return k;
}

bool staged_selected(const rr_ctx* c) {
  const Tunables& tn = tunables();
  return c->configured && c->cfg.use_bricks && c->fused_ok && tn.fused && tn.staged && c->sti.ok && !c->sti.dirty &&
         c->sti.generation == staged_key();
}

bool staged_classify_params(const rr_ctx* c, ClassifyParams& q) {
  if (!staged_selected(c)) return false;
  const auto& st = c->sti;
  q.fp = st.d_fp.ptr; q.zr = st.d_zr.ptr; q.pairs = c->d_pairs.ptr; q.pair_pitch = c->pair_pitch; q.H2 = c->H + 2;
  q.list = st.d_list.ptr; q.class_count = c->d_counters.ptr + c->bricks.num; q.list_stride = st.list_stride;
  q.per_brick = st.n_yc * st.n_zc; q.N = c->N; q.limit = c->cfg.limit;
  return true;
}

int build_ztab(rr_ctx* c);   // rr_integrate.cu

// Everything the staged kernel needs that depends only on calibration + configuration: item geometry, box and tile sizes,
// the footprint table, the tensor maps. Synchronises the stream (never called inside a graph capture: rr_fuse_frame runs
// it before capturing).
int staged_prepare(rr_ctx* c) {
  auto& st = c->sti;
  const Tunables& tn = tunables();
  if (!st.dirty && st.generation == staged_key()) return RR_OK;
  st.ok = false;
  st.n_oversize = 0;
  // declined before any table is built: stay dirty, so that returning to the current tunables rebuilds the tables
  st.dirty = true;
  if (!c->configured || !c->cfg.use_bricks || !c->fused_ok || !tn.staged || !tn.fused || !c->d_inv.ptr) return RR_OK;
  for (int i = 0; i < c->N; ++i) if (!c->have_inv[i]) return RR_OK;
  st.dirty = false;
  st.generation = staged_key();
  EncodeTiledFn enc = encode_tiled();
  if (!enc) return RR_OK;                       // driver without tensor maps: the direct kernels run
  const int N = c->N, X = (int)c->res[0], Y = (int)c->res[1], Z = (int)c->res[2];
  const int IX = (int)c->ires[0], IY = (int)c->ires[1], IZ = (int)c->ires[2];
  int max_nx = 0, max_ny = 0, max_nz = 0;
  const size_t nb = c->h_ranges.size() / 6;
  for (size_t i = 0; i < nb; ++i) {
    const int32_t* r = c->h_ranges.data() + i * 6;
    max_nx = std::max(max_nx, r[1] - r[0]); max_ny = std::max(max_ny, r[3] - r[2]); max_nz = std::max(max_nz, r[5] - r[4]);
  }
  if (max_nx <= 0 || max_ny <= 0 || max_nz <= 0) return RR_OK;
  // the clear's bulk stores need 16-byte aligned rows, a row mask of at most 32 words and a buffer of at least one row
  const long fill_buf = std::max(4L, (long)tn.stage_bulk_fill) * 1024;
  if ((X & 3) != 0 || X > 1024 || (long)X * 4 > fill_buf || c->W > 0xffff || c->H > 0xffff) return RR_OK;
  st.cwarps = consumer_warps(N);
  st.fwarps = 7;
  const int CT = st.cwarps * 32;
  // y-chunk: as many brick rows as fill the consumer threads best (ties: the larger chunk, fewer items)
  int cy = tn.stage_ychunk > 0 ? std::min(tn.stage_ychunk, max_ny) : 0;
  if (cy == 0) {
    double best = -1.0;
    for (int t = 1; t <= max_ny; ++t) {
      const int cols = max_nx * t;
      const double eff = double(cols) / double((cols + CT - 1) / CT * CT);
      if (eff >= best - 0.02) { if (eff > best) best = eff; cy = t; }
    }
  }
  while (cy > 1 && max_nx * cy > CT) --cy;
  if (max_nx * cy > CT) return RR_OK;           // a single brick row exceeds the consumer threads: the direct kernels run
  const int n_yc = (max_ny + cy - 1) / cy;
  const int n_zc = std::max(1, (max_nz + std::max(1, tn.stage_zchunk) - 1) / std::max(1, tn.stage_zchunk));
  const int cz = (max_nz + n_zc - 1) / n_zc;
  // staged inverse-volume box: the largest coarse extent any item needs, from the same coordinate arithmetic as the device
  int BX = 1, BY = 1, BZ = 1;
  const float stepX = 1.0f / (float)X, stepY = 1.0f / (float)Y, stepZ = 1.0f / (float)Z;
  for (size_t i = 0; i < nb; ++i) {
    const int32_t* r = c->h_ranges.data() + i * 6;
    int lo, hi, t;
    if (r[1] > r[0]) {
      h_lin_coord(((float)r[0] + 0.5f) * stepX, IX, lo, t); h_lin_coord(((float)(r[1] - 1) + 0.5f) * stepX, IX, t, hi);
      BX = std::max(BX, hi - lo + 1);
    }
    for (int yb = r[2]; yb < r[3]; yb += cy) {
      const int ye = std::min(yb + cy, r[3]);
      h_lin_coord(((float)yb + 0.5f) * stepY, IY, lo, t); h_lin_coord(((float)(ye - 1) + 0.5f) * stepY, IY, t, hi);
      BY = std::max(BY, hi - lo + 1);
    }
    for (int zb = r[4]; zb < r[5]; zb += cz) {
      const int ze = std::min(zb + cz, r[5]);
      h_lin_coord(((float)zb + 0.5f) * stepZ, IZ, lo, t); h_lin_coord(((float)(ze - 1) + 0.5f) * stepZ, IZ, t, hi);
      BZ = std::max(BZ, hi - lo + 1);
    }
  }
  if (BX > 256 || BY > 256 || BZ > 256 || cz > ZT_MAX) return RR_OK;
  int smem_max = 0;
  cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->device);
  const int weight_mode = c->cfg.store_weight == RR_VOXELS_F32_WEIGHT ? 2 : 1;
  const long tables = ((long)(4 * (Y + Z)) + (long)c->bricks.res[1] * c->bricks.res[2] + 127) & ~127L;      // cand_y, cand_z, rowany
  const long budget = (long)smem_max - 1024 - (long)NH * HDR_BYTES - fill_buf * weight_mode - tables;       // the slot ring
  const long inv_bytes = (long)BZ * BY * BX * 16, inv_span = (inv_bytes + 127) & ~127L;
  auto slot_bytes_for = [&](long T) { return inv_span + ((T * T * 8 + 127) & ~127L); };
  // largest tile that still leaves `slots` slots
  auto tile_for_slots = [&](long slots) {
    long T = 256;
    while (T >= 8 && slot_bytes_for(T) * slots > budget) T -= 2;
    return T;
  };
  const long t_min_slots = tile_for_slots(N);            // every sensor of one item must fit the ring
  if (t_min_slots < 8) return RR_OK;

  // footprints of every item of the brick grid
  IntegrateParams p{};
  p.inv = c->d_inv.ptr; p.ranges = c->d_ranges.ptr;
  p.IX = IX; p.IY = IY; p.IZ = IZ; p.W = c->W; p.H = c->H; p.X = X; p.Y = Y; p.Z = Z;
  p.fW = (float)c->W; p.fH = (float)c->H; p.exmax = (float)(c->W - 1); p.eymax = (float)(c->H - 1);
  RR_TRY_RC(build_ztab(c));
  p.ztab = c->d_ztab.ptr;
  const size_t items = nb * (size_t)n_yc * n_zc;
  if (items == 0 || items > 0x3fffffffull) return RR_OK;
  std::vector<int4> ext(items * N);
  DeviceArray<float2> d_zr;
  {
    DeviceArray<int4> d_ext;
    // a failed allocation declines: the direct kernels run
    if (d_ext.allocate(c, items * N, "footprint extents") != RR_OK || d_zr.allocate(c, items * N, "footprint z ranges") != RR_OK) {
      cudaGetLastError();
      return RR_OK;
    }
    RR_TRY_RC(footprints(c, p, cy, cz, n_yc, n_zc, d_ext.ptr, d_zr.ptr, (uint32_t)items));
    RR_TRY_RC(check(c, cudaMemcpyAsync(ext.data(), d_ext.ptr, ext.size() * sizeof(int4), cudaMemcpyDeviceToHost, c->stream), "footprint download"));
    RR_TRY_RC(check(c, cudaStreamSynchronize(c->stream), "footprint sync"));
  }
  // Tile edge: a smaller tile leaves more slots in the ring (more items in flight), a larger one sends fewer (item, sensor)
  // pairs to the global-memory path, which costs several times a staged item: the largest tile that keeps two items' worth
  // of slots plus one, and no larger than the largest footprint of the grid.
  std::vector<int> need;
  need.reserve(ext.size());
  for (const int4& e : ext)
    if (e.z >= e.x) need.push_back(std::max(e.z - (e.x & ~1), e.w - e.y) + 2);
  if (need.empty()) return RR_OK;
  std::sort(need.begin(), need.end());
  auto even = [](long v) { return (v + 1) & ~1L; };
  long T;
  if (tn.stage_tile > 0) {
    T = std::min<long>(even(tn.stage_tile), t_min_slots);
  } else {
    T = std::min(even(need.back()), std::max(tile_for_slots(2 * N + 1), std::min(t_min_slots, 24L)));
  }
  T = std::max(T, 8L);
  const long slot_bytes = slot_bytes_for(T);
  const long n_slots = std::min(budget / slot_bytes, 64L);
  if (n_slots < N) return RR_OK;
  std::vector<uint2> fp(items * N, make_uint2(0u, 0u));
  for (size_t i = 0; i < items; ++i)
    for (int s = 0; s < N; ++s) {
      const int4& e = ext[i * N + s];
      if (e.z < e.x) continue;
      // tile origin (even x: TMA start coordinates are multiples of 16 bytes) and the footprint rectangle inside the tile;
      // bit 7: the footprint exceeds the tile (the item then reads its operands from global memory, if this sensor is read at all)
      const uint32_t over = std::max(e.z - (e.x & ~1), e.w - e.y) + 2 > T ? 128u : 0u;
      const uint32_t rx = (uint32_t)(e.x & 1), rw = (uint32_t)std::min(e.z - e.x + 2, 4095), rh = (uint32_t)std::min(e.w - e.y + 2, 4095);
      fp[i * N + s] = make_uint2((uint32_t)(e.x & ~1) | ((uint32_t)e.y << 16), rx | over | (rw << 8) | (rh << 20));
      st.n_oversize += over ? 1u : 0u;
    }
  st.lists_key = 0;
  ++st.tables;
  st.d_zr = std::move(d_zr);
  st.list_stride = (uint32_t)items;
  RR_TRY_RC(st.d_list.allocate(c, (size_t)(N + 1) * items, "item lists"));
  RR_TRY_RC(st.d_fp.allocate(c, fp.size(), "footprint table"));
  RR_TRY_RC(st.d_err.allocate(c, 4 + 16 * sizeof(unsigned long long) / sizeof(uint32_t), "staged flags"));
  cudaMemcpyAsync(st.d_fp.ptr, fp.data(), fp.size() * sizeof(uint2), cudaMemcpyHostToDevice, c->stream);
  cudaMemsetAsync(st.d_err.ptr, 0, 4 * sizeof(uint32_t) + 16 * sizeof(unsigned long long), c->stream);
  cudaMemsetAsync(c->d_counters.ptr + nb, 0, RR_CLASS_COUNTERS * sizeof(uint32_t), c->stream);
  RR_TRY_RC(check(c, cudaStreamSynchronize(c->stream), "staged tables upload"));

  // tensor maps: inverse volumes as (xyzw, IX, IY, IZ, N) float32 with a one-sensor box, pair image as (pitch, H+2, N) 8-byte pixels.
  // The innermost start coordinate of a tile must be a multiple of 16 bytes (measured: tools/tma_probe.cu), so tile origins are even pixels.
  {
    const cuuint64_t dims[5] = {4, (cuuint64_t)IX, (cuuint64_t)IY, (cuuint64_t)IZ, (cuuint64_t)N};
    const cuuint64_t strides[4] = {16, (cuuint64_t)IX * 16, (cuuint64_t)IX * IY * 16, (cuuint64_t)IX * IY * IZ * 16};
    const cuuint32_t box[5] = {4, (cuuint32_t)BX, (cuuint32_t)BY, (cuuint32_t)BZ, 1};
    const cuuint32_t es[5] = {1, 1, 1, 1, 1};
    if (enc(&st.map_inv, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, c->d_inv.ptr, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) return RR_OK;
  }
  {
    const cuuint64_t dims[3] = {(cuuint64_t)c->pair_pitch, (cuuint64_t)(c->H + 2), (cuuint64_t)N};
    const cuuint64_t strides[2] = {(cuuint64_t)c->pair_pitch * 8, (cuuint64_t)c->pair_pitch * (c->H + 2) * 8};
    const cuuint32_t box[3] = {(cuuint32_t)T, (cuuint32_t)T, 1};
    const cuuint32_t es[3] = {1, 1, 1};
    if (enc(&st.map_pairs, CU_TENSOR_MAP_DATA_TYPE_INT64, 3, c->d_pairs.ptr, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) return RR_OK;
  }
  st.cy = cy; st.cz = cz; st.n_yc = n_yc; st.n_zc = n_zc;
  st.BX = BX; st.BY = BY; st.BZ = BZ; st.T = (int)T;
  st.inv_bytes = (uint32_t)inv_bytes;
  st.tile_bytes = (uint32_t)(T * T * 8);
  st.inv_span = (uint32_t)inv_span;
  st.slot_bytes = (uint32_t)slot_bytes;
  st.n_slots = (uint32_t)n_slots;
  st.slots_off = (uint32_t)NH * HDR_BYTES;
  st.fill_src_bytes = (uint32_t)fill_buf;
  st.fill_src_off = st.slots_off + st.n_slots * st.slot_bytes;
  st.tables_off = st.fill_src_off + (uint32_t)(fill_buf * weight_mode);
  st.smem_bytes = st.tables_off + (uint32_t)tables + 128;
  st.ok = true;
  return RR_OK;
}

int launch_integrate_staged(rr_ctx* c, const IntegrateParams& p, int mode, bool* done) {
  *done = false;
  RR_TRY_RC(staged_prepare(c));
  const auto& st = c->sti;
  if (!staged_selected(c)) return RR_OK;
  // The item lists hold the verdicts of the last rr_bricks_update. Tables rebuilt since, a limit changed since, a newer
  // pre-process (the verdicts describe the pair image they were classified on) or rr_bricks_clear (it zeroes the class
  // counters) leave them stale: the direct kernels integrate the occupied list instead.
  if (st.lists_key != staged_lists_key(c)) { c->last_integrate[4] |= 1u; return RR_OK; }
  StagedParams sp{};
  setup_fill(c, p, mode, tunables().stage_fill_rows, sp.f);
  sp.cy = st.cy; sp.cz = st.cz; sp.n_yc = st.n_yc; sp.n_zc = st.n_zc;
  sp.BX = st.BX; sp.BY = st.BY; sp.BZ = st.BZ; sp.T = st.T;
  sp.fp = st.d_fp.ptr;
  sp.list = st.d_list.ptr; sp.class_count = c->d_counters.ptr + c->bricks.num; sp.list_stride = st.list_stride;
  sp.inv_bytes = st.inv_bytes; sp.tile_bytes = st.tile_bytes; sp.inv_span = st.inv_span;
  sp.slot_bytes = st.slot_bytes; sp.n_slots = st.n_slots; sp.slots_off = st.slots_off;
  sp.err = st.d_err.ptr;
  sp.prof = (tunables().stage_debug & 128) ? reinterpret_cast<unsigned long long*>(st.d_err.ptr + 4) : nullptr;
  sp.fill_src_off = st.fill_src_off; sp.fill_src_bytes = st.fill_src_bytes;
  sp.tables_off = st.tables_off; sp.n_rowany = c->bricks.res[1] * c->bricks.res[2];
  if (tunables().stage_debug & 1) sp.f.fill_items = 0;
  sp.debug = tunables().stage_debug;
  sp.fill_depth = tunables().stage_fill_depth; sp.fill_lsu = tunables().stage_fill_lsu;
  sp.tail_cap = tunables().stage_tail_cap;
  // The work counters are reset and this frame's item lists written by k_bricks_update; a second integrate of the same
  // frame set (another slab, a repeated call) finds the lists intact and only needs fresh counters.
  if (!c->work_fresh) cudaMemsetAsync(c->d_work.ptr, 0, 4 * sizeof(uint32_t), c->stream);
  c->work_fresh = false;
  int rc;
  switch (c->N) {
    case 1: rc = launch_staged_n<1, 22>(c, sp, mode); break;
    case 2: rc = launch_staged_n<2, 22>(c, sp, mode); break;
    case 3: rc = launch_staged_n<3, 22>(c, sp, mode); break;
    case 4: rc = st.cwarps == 11 ? launch_staged_n<4, 11>(c, sp, mode) : launch_staged_n<4, 22>(c, sp, mode); break;
    case 5: rc = st.cwarps == 11 ? launch_staged_n<5, 11>(c, sp, mode) : launch_staged_n<5, 16>(c, sp, mode); break;
    case 6: rc = st.cwarps == 11 ? launch_staged_n<6, 11>(c, sp, mode) : launch_staged_n<6, 16>(c, sp, mode); break;
    case 7: rc = st.cwarps == 11 ? launch_staged_n<7, 11>(c, sp, mode) : launch_staged_n<7, 16>(c, sp, mode); break;
    case 8: rc = st.cwarps == 11 ? launch_staged_n<8, 11>(c, sp, mode) : launch_staged_n<8, 16>(c, sp, mode); break;
    default: return fail(c, RR_ERR_UNSUPPORTED, "integrate: 1..8 sensors supported");
  }
  if (rc != RR_OK) return rc;
  c->last_integrate[0] = 1; c->last_integrate[3] = (uint32_t)st.cwarps;
  *done = true;
  return RR_OK;
}

}  // namespace rr
