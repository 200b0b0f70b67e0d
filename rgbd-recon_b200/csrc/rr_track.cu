// Part tracking on the device: persistent identities for the connected parts of consecutive labellings, matched by voxel
// overlap (rr_track_parts / rr_download_part_tracks / rr_reset_part_tracks; the contract is stated in
// include/rgbd_recon_b200.h and DESIGN.md "Beyond the reference: tracking parts"). No reference counterpart.
//
// The call labels the volume exactly as rr_label_parts does (rr_parts.cu), into the label array that does not hold the
// tracked labelling, then compares the two arrays voxel by voxel:
//   k_track_init         per current part: no track yet; per previous part: not accepted
//   k_track_pairs<0>     per row: the (q, p) pair records it emits (q candidate, p tracked, equal pairs aggregated per warp)
//   CUB scan             per-row record offsets; the record count is read back (synchronisation 2 of 3)
//   k_track_pairs<1>     the records, key q << 32 | p and voxel count
//   CUB sort + reduce    distinct pairs in ascending key with their overlap O (the count of distinct pairs stays on the device)
//   CUB sort descending  stable by O: the contract's order (O descending, q ascending, p ascending)
//   k_track_match        one thread walks the ordered pairs: the greedy matching
//   k_track_flags        per current part: tracked and unmatched; per previous part: candidate and not accepted
//   CUB scans x2         new-id ranks and ended slots; the new-id and ended counts are read back (synchronisation 3)
//   k_track_finish       new ids next_id + rank, the ended track ids
// Synchronisations: one for the part count (the labelling), one for the record count when both labellings have parts, one
// for the counts the call returns. The per-part outputs go to the slot of the new labelling, so a refused call
// (RR_ERR_UNSUPPORTED) leaves the last call's outputs and the tracked labelling as they were.
#include "rr_context.h"
#include "rr_rows.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_reduce.cuh>
#include <cub/device/device_scan.cuh>
#include <cuda/std/functional>

#include <algorithm>

namespace rr {

namespace {

constexpr uint32_t kNone = 0xFFFFFFFFu;            // outside voxel, untracked part, no previous part
constexpr unsigned long long kNoPair = ~0ull;      // q = 0xFFFFFFFF never names a part

struct TrackParams {
  int X, Y, Z;
  // candidate voxels: the work domain of the labelling (rr_rows.cuh)
  int use_rows, rby, mask_words;
  const uint32_t* rowmask; const uint8_t* rowany; const int16_t* cand_y; const int16_t* cand_z;
  const uint32_t* L;          // labels of this call
  const uint32_t* L_prev;     // the tracked labelling
  const uint32_t* voxels;     // per current part
  const uint32_t* ids_prev;   // per previous part: its track id, 0xFFFFFFFF for none (not a candidate)
  uint32_t min_voxels;
  uint32_t* cnt; const uint32_t* off;   // per row: records, their exclusive offsets over rows + 1 entries
  unsigned long long* keys; uint32_t* counts;
};

#define RR_TRACK_ROW                                                   \
  const unsigned r = blockIdx.x * 8u + (threadIdx.x >> 5);             \
  if (r >= (unsigned)p.Y * (unsigned)p.Z) return;

// The lanes of one pair in a 32-voxel word are grouped by ballots, and the warp keeps a running count for the last pair it
// saw, closed into a record when another pair comes up: the same records, in the same order, in both instances.
template <bool kEmit>
__global__ void __launch_bounds__(256) k_track_pairs(const __grid_constant__ TrackParams p) {
  RR_TRACK_ROW
  const unsigned lane = threadIdx.x & 31u;
  const uint32_t base = kEmit ? p.off[r] : 0u;
  if (kEmit && p.off[r + 1] == base) return;
  unsigned long long acc = kNoPair;
  uint32_t n = 0, rec = 0;
  walk_row(p, r, [&](int, int, int, uint32_t i, bool cand, unsigned) {
    unsigned long long key = kNoPair;
    if (cand) {
      const uint32_t b = p.L[i];
      if (b != kNone && p.voxels[b] >= p.min_voxels) {
        const uint32_t a = p.L_prev[i];
        if (a != kNone && p.ids_prev[a] != kNone) key = ((unsigned long long)a << 32) | b;
      }
    }
    uint32_t todo = __ballot_sync(0xffffffffu, key != kNoPair);
    while (todo) {
      const unsigned long long k = __shfl_sync(0xffffffffu, key, __ffs(todo) - 1);
      const uint32_t grp = __ballot_sync(0xffffffffu, key == k);
      todo &= ~grp;
      if (k != acc) {
        if (n) {
          if (kEmit && lane == 0) { p.keys[base + rec] = acc; p.counts[base + rec] = n; }
          ++rec;
        }
        acc = k; n = 0;
      }
      n += __popc(grp);
    }
  });
  if (n) {
    if (kEmit && lane == 0) { p.keys[base + rec] = acc; p.counts[base + rec] = n; }
    ++rec;
  }
  if (!kEmit && lane == 0) p.cnt[r] = rec;
}

__global__ void __launch_bounds__(128) k_track_init(uint32_t P, uint32_t P_prev, uint32_t* __restrict__ ids,
                                                    uint32_t* __restrict__ prev, uint32_t* __restrict__ overlaps,
                                                    uint32_t* __restrict__ accepted) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < P) { ids[k] = kNone; prev[k] = kNone; overlaps[k] = 0; }
  if (k < P_prev) accepted[k] = 0;
}

// The contract's greedy, sequentially: a pair is accepted iff neither its previous nor its current part is taken yet.
__global__ void __launch_bounds__(32) k_track_match(const unsigned long long* __restrict__ order, const uint32_t* __restrict__ order_o,
                                                    const uint32_t* __restrict__ num_pairs, const uint32_t* __restrict__ ids_prev,
                                                    uint32_t* accepted, uint32_t* ids, uint32_t* prev, uint32_t* overlaps) {
  if (threadIdx.x != 0) return;
  const uint32_t D = *num_pairs;
  for (uint32_t k = 0; k < D; ++k) {
    const unsigned long long key = order[k];
    const uint32_t q = (uint32_t)(key >> 32), pp = (uint32_t)key;
    if (accepted[q] || prev[pp] != kNone) continue;
    accepted[q] = 1;
    prev[pp] = q;
    overlaps[pp] = order_o[k];
    ids[pp] = ids_prev[q];
  }
}

__global__ void __launch_bounds__(128) k_track_flags(uint32_t P, uint32_t P_prev, uint32_t min_voxels,
                                                     const uint32_t* __restrict__ voxels, const uint32_t* __restrict__ prev,
                                                     const uint32_t* __restrict__ ids_prev, const uint32_t* __restrict__ accepted,
                                                     uint32_t* __restrict__ new_flag, uint32_t* __restrict__ end_flag) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k <= P) new_flag[k] = k < P && voxels[k] >= min_voxels && prev[k] == kNone;
  if (k <= P_prev) end_flag[k] = k < P_prev && ids_prev[k] != kNone && !accepted[k];
}

__global__ void __launch_bounds__(128) k_track_finish(uint32_t P, uint32_t P_prev, uint32_t next_id,
                                                      const uint32_t* __restrict__ new_flag, const uint32_t* __restrict__ new_off,
                                                      const uint32_t* __restrict__ end_flag, const uint32_t* __restrict__ end_off,
                                                      const uint32_t* __restrict__ ids_prev, uint32_t* __restrict__ ids,
                                                      uint32_t* __restrict__ ended) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < P && new_flag[k]) ids[k] = next_id + new_off[k];   // wraps only in a call that is refused
  if (k < P_prev && end_flag[k]) ended[end_off[k]] = ids_prev[k];
}

unsigned blocks128(size_t n) { return (unsigned)((n + 127) / 128); }

}  // namespace

int label_dest(const rr_ctx* c) { return c->track_slot == 0 ? 1 : 0; }

void track_reset(rr_ctx* c) {
  c->track_slot = -1;
  c->track_valid = false;
  c->track_next_id = 0;
}

int launch_track_parts(rr_ctx* c, uint32_t min_voxels, uint32_t* out_num_parts, uint32_t* out_num_ended) {
  const size_t nvox = (size_t)c->res[0] * c->res[1] * c->res[2], rows = (size_t)c->res[1] * c->res[2];
  // the second label array is reserved here, so that no later labelling allocates in the middle of a tracked sequence
  RR_TRY_RC(c->d_parts_labels[0].reserve(c, nvox, "part labels"));
  RR_TRY_RC(c->d_parts_labels[1].reserve(c, nvox, "part labels"));
  const int dest = label_dest(c), src = c->track_slot;
  uint32_t P = 0;
  RR_TRY_RC(launch_label_parts(c, dest, &P));                      // synchronisation 1
  const uint32_t P_prev = src >= 0 ? c->track_n[src] : 0u;
  const uint32_t* ids_prev = src >= 0 ? c->d_track_ids[src].ptr : nullptr;

  RR_TRY_RC(c->d_track_ids[dest].reserve(c, P, "track ids"));
  RR_TRY_RC(c->d_track_prev[dest].reserve(c, P, "track previous parts"));
  RR_TRY_RC(c->d_track_overlaps[dest].reserve(c, P, "track overlaps"));
  RR_TRY_RC(c->d_track_ended[dest].reserve(c, P_prev, "ended tracks"));
  RR_TRY_RC(c->d_track_flags.reserve(c, 2 * ((size_t)P + 1) + 3 * (size_t)P_prev + 3, "track flags"));
  uint32_t* new_flag = c->d_track_flags.ptr;
  uint32_t* new_off = new_flag + (P + 1);
  uint32_t* end_flag = new_off + (P + 1);
  uint32_t* end_off = end_flag + (P_prev + 1);
  uint32_t* accepted = end_off + (P_prev + 1);
  uint32_t* num_pairs = accepted + P_prev;
  uint32_t* ids = c->d_track_ids[dest].ptr;
  uint32_t* prev = c->d_track_prev[dest].ptr;
  uint32_t* overlaps = c->d_track_overlaps[dest].ptr;
  const uint32_t n_init = std::max(P, P_prev);
  if (n_init) {
    k_track_init<<<blocks128(n_init), 128, 0, c->stream>>>(P, P_prev, ids, prev, overlaps, accepted);
    RR_LAUNCH_CHECK(c, "k_track_init");
  }

  if (P && P_prev) {   // overlap pairs, their order, the matching
    uint32_t* cnt = c->d_parts_rows.ptr;   // the labelling's per-row scratch, free again
    uint32_t* off = cnt + (rows + 1);
    TrackParams p{};
    p.X = (int)c->res[0]; p.Y = (int)c->res[1]; p.Z = (int)c->res[2];
    p.use_rows = c->mesh_rows_ok ? 1 : 0;
    p.rby = (int)c->bricks.res[1]; p.mask_words = c->mask_words;
    p.rowmask = c->d_rowmask.ptr; p.rowany = c->d_rowany.ptr; p.cand_y = c->d_cand_y.ptr; p.cand_z = c->d_cand_z.ptr;
    p.L = c->d_parts_labels[dest].ptr; p.L_prev = c->d_parts_labels[src].ptr;
    p.voxels = c->d_parts_voxels.ptr; p.ids_prev = ids_prev; p.min_voxels = min_voxels;
    p.cnt = cnt; p.off = off;
    const unsigned row_blocks = (unsigned)((rows + 7) / 8);
    RR_TRY_RC(check(c, cudaMemsetAsync(cnt + rows, 0, sizeof(uint32_t), c->stream), "track record counts"));
    k_track_pairs<false><<<row_blocks, 256, 0, c->stream>>>(p);
    RR_LAUNCH_CHECK(c, "k_track_pairs<count>");
    size_t bytes = c->d_parts_scratch.cap;   // sized by the labelling for this very scan
    RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(c->d_parts_scratch.ptr, bytes, cnt, off, (int)(rows + 1), c->stream), "track record scan"));
    c->launches += 1;
    RR_TRY_RC(check(c, cudaMemcpyAsync(&c->pinned->track_counts[0], off + rows, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream), "track record count"));
    RR_TRY_RC(check(c, cudaStreamSynchronize(c->stream), "track record count sync"));   // synchronisation 2
    const uint32_t R = c->pinned->track_counts[0];
    if (R) {
      RR_TRY_RC(c->d_track_keys.reserve(c, 4 * (size_t)R, "track pair keys"));
      RR_TRY_RC(c->d_track_counts.reserve(c, 4 * (size_t)R, "track pair counts"));
      unsigned long long* k_rec = c->d_track_keys.ptr;
      unsigned long long* k_sorted = k_rec + R;
      unsigned long long* k_pair = k_sorted + R;
      unsigned long long* k_order = k_pair + R;
      uint32_t* c_rec = c->d_track_counts.ptr;
      uint32_t* c_sorted = c_rec + R;
      uint32_t* o_pair = c_sorted + R;
      uint32_t* o_order = o_pair + R;
      int qbits = 1;
      while (qbits < 32 && ((P_prev - 1) >> qbits)) ++qbits;
      const int end_bit = 32 + qbits;
      size_t need = 0, b = 0;
      RR_TRY_RC(check(c, cub::DeviceRadixSort::SortPairs(nullptr, b, k_rec, k_sorted, c_rec, c_sorted, (int)R, 0, end_bit, c->stream), "track sort size"));
      need = std::max(need, b);
      RR_TRY_RC(check(c, cub::DeviceReduce::ReduceByKey(nullptr, b, k_sorted, k_pair, c_sorted, o_pair, num_pairs, cuda::std::plus<uint32_t>{}, (int)R, c->stream), "track reduce size"));
      need = std::max(need, b);
      RR_TRY_RC(check(c, cub::DeviceRadixSort::SortPairsDescending(nullptr, b, o_pair, o_order, k_pair, k_order, (int)R, 0, 32, c->stream), "track order size"));
      need = std::max(need, b);
      RR_TRY_RC(c->d_track_scratch.reserve(c, need, "track sort scratch"));
      p.keys = k_rec; p.counts = c_rec;
      k_track_pairs<true><<<row_blocks, 256, 0, c->stream>>>(p);
      RR_LAUNCH_CHECK(c, "k_track_pairs<emit>");
      void* scratch = c->d_track_scratch.ptr;
      b = c->d_track_scratch.cap;
      RR_TRY_RC(check(c, cub::DeviceRadixSort::SortPairs(scratch, b, k_rec, k_sorted, c_rec, c_sorted, (int)R, 0, end_bit, c->stream), "track pair sort"));
      // entries past the distinct pairs keep O = 0 and sort behind every pair (O >= 1)
      RR_TRY_RC(check(c, cudaMemsetAsync(o_pair, 0, (size_t)R * sizeof(uint32_t), c->stream), "track overlaps reset"));
      b = c->d_track_scratch.cap;
      RR_TRY_RC(check(c, cub::DeviceReduce::ReduceByKey(scratch, b, k_sorted, k_pair, c_sorted, o_pair, num_pairs, cuda::std::plus<uint32_t>{}, (int)R, c->stream), "track pair reduce"));
      b = c->d_track_scratch.cap;
      RR_TRY_RC(check(c, cub::DeviceRadixSort::SortPairsDescending(scratch, b, o_pair, o_order, k_pair, k_order, (int)R, 0, 32, c->stream), "track pair order"));
      c->launches += 3;
      k_track_match<<<1, 32, 0, c->stream>>>(k_order, o_order, num_pairs, ids_prev, accepted, ids, prev, overlaps);
      RR_LAUNCH_CHECK(c, "k_track_match");
    }
  }

  // new ids over the unmatched tracked parts, ended tracks over the unaccepted candidates
  size_t scan_bytes = 0, b = 0;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(nullptr, b, new_flag, new_off, (int)(P + 1), c->stream), "track scan size"));
  scan_bytes = b;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(nullptr, b, end_flag, end_off, (int)(P_prev + 1), c->stream), "track scan size"));
  RR_TRY_RC(c->d_track_scratch.reserve(c, std::max(scan_bytes, b), "track scan scratch"));
  k_track_flags<<<blocks128((size_t)n_init + 1), 128, 0, c->stream>>>(P, P_prev, min_voxels, c->d_parts_voxels.ptr, prev, ids_prev,
                                                                       accepted, new_flag, end_flag);
  RR_LAUNCH_CHECK(c, "k_track_flags");
  b = c->d_track_scratch.cap;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(c->d_track_scratch.ptr, b, new_flag, new_off, (int)(P + 1), c->stream), "track id scan"));
  b = c->d_track_scratch.cap;
  RR_TRY_RC(check(c, cub::DeviceScan::ExclusiveSum(c->d_track_scratch.ptr, b, end_flag, end_off, (int)(P_prev + 1), c->stream), "ended scan"));
  c->launches += 2;
  if (n_init) {
    k_track_finish<<<blocks128(n_init), 128, 0, c->stream>>>(P, P_prev, (uint32_t)c->track_next_id, new_flag, new_off, end_flag, end_off,
                                                            ids_prev, ids, c->d_track_ended[dest].ptr);
    RR_LAUNCH_CHECK(c, "k_track_finish");
  }
  RR_TRY_RC(check(c, cudaMemcpyAsync(&c->pinned->track_counts[1], new_off + P, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream), "track counts"));
  RR_TRY_RC(check(c, cudaMemcpyAsync(&c->pinned->track_counts[2], end_off + P_prev, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream), "track counts"));
  RR_TRY_RC(check(c, cudaStreamSynchronize(c->stream), "track counts sync"));   // synchronisation 3
  const uint32_t n_new = c->pinned->track_counts[1], E = c->pinned->track_counts[2];
  if (c->track_next_id + n_new > (uint64_t)kNone)
    return fail(c, RR_ERR_UNSUPPORTED, "rr_track_parts: the track ids are used up (rr_reset_part_tracks starts them at 0 again)");
  c->track_next_id += n_new;
  c->track_n[dest] = P;
  c->track_e[dest] = E;
  c->track_slot = dest;
  c->track_valid = true;
  *out_num_parts = P;
  *out_num_ended = E;
  return RR_OK;
}

int track_download(rr_ctx* c, uint32_t* track_ids, uint32_t* prev_parts, uint32_t* overlaps, uint32_t* ended) {
  const int s = c->track_slot;
  const size_t P = c->track_n[s], E = c->track_e[s];
  if (track_ids && P) RR_TRY_RC(check(c, cudaMemcpyAsync(track_ids, c->d_track_ids[s].ptr, P * sizeof(uint32_t), cudaMemcpyDefault, c->stream), "track download"));
  if (prev_parts && P) RR_TRY_RC(check(c, cudaMemcpyAsync(prev_parts, c->d_track_prev[s].ptr, P * sizeof(uint32_t), cudaMemcpyDefault, c->stream), "track download"));
  if (overlaps && P) RR_TRY_RC(check(c, cudaMemcpyAsync(overlaps, c->d_track_overlaps[s].ptr, P * sizeof(uint32_t), cudaMemcpyDefault, c->stream), "track download"));
  if (ended && E) RR_TRY_RC(check(c, cudaMemcpyAsync(ended, c->d_track_ended[s].ptr, E * sizeof(uint32_t), cudaMemcpyDefault, c->stream), "track download"));
  return check(c, cudaStreamSynchronize(c->stream), "track download sync");
}

}  // namespace rr
