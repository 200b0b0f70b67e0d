// Compressed frame ingest for sm_100a (SURVEY.md §8f-2). The reference hands DXT1 colour blocks and 8-bit depth texels to
// OpenGL, whose sampler decodes them (framework/NetKinectArray.cpp:120-131,149-151,170-172); here the packed frame set is
// copied host->device as it arrives (6.2 MB instead of 20 MB per 4-sensor frame set) and expanded once, on the device,
// into the RGB8 / float32 layers every later kernel reads. HBM-bound byte work: one thread per 4x4 block / per texel.
#include "rr_context.h"

namespace rr {

// S3TC DXT1 (BC1) block -> 4x4 RGB8 texels; same integer arithmetic as the reference's CPU codec external/squish
// (colourblock.cpp:160-214): 565 endpoints expanded by bit replication, (2a+b)/3 and (a+2b)/3 in four-colour mode,
// (a+b)/2 and black in three-colour mode (endpoint0 <= endpoint1). Alpha is not sampled downstream.
// DXT5 (BC3, GL_COMPRESSED_RGBA_S3TC_DXT5_EXT, NetKinectArray.cpp:125-128,153-156): 16-byte blocks, the colour block sits
// behind 8 bytes of alpha and is always in four-colour mode (squish DecompressColour with isDxt1 = false).
template <bool DXT5>
__global__ void __launch_bounds__(256) k_decode_dxt(const uint2* __restrict__ blocks, uint8_t* __restrict__ rgb, int W, int H) {
  const int bw = W >> 2, bh = H >> 2;
  const int bx = blockIdx.x * 32 + threadIdx.x, by = blockIdx.y * 8 + threadIdx.y;
  if (bx >= bw || by >= bh) return;
  const size_t layer = blockIdx.z;
  const uint2 blk = __ldg(blocks + ((layer * bh + by) * bw + bx) * (DXT5 ? 2 : 1) + (DXT5 ? 1 : 0));
  const int a = (int)(blk.x & 0xffffu), b = (int)(blk.x >> 16);
  int code[4][3];
  code[0][0] = ((a >> 11) << 3) | (a >> 13);            code[1][0] = ((b >> 11) << 3) | (b >> 13);
  code[0][1] = (((a >> 5) & 63) << 2) | ((a >> 9) & 3); code[1][1] = (((b >> 5) & 63) << 2) | ((b >> 9) & 3);
  code[0][2] = ((a & 31) << 3) | ((a & 31) >> 2);       code[1][2] = ((b & 31) << 3) | ((b & 31) >> 2);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int c = code[0][i], d = code[1][i];
    if (!DXT5 && a <= b) { code[2][i] = (c + d) / 2; code[3][i] = 0; }
    else { code[2][i] = (2 * c + d) / 3; code[3][i] = (c + 2 * d) / 3; }
  }
  uint8_t* img = rgb + layer * (size_t)W * H * 3;
#pragma unroll
  for (int py = 0; py < 4; ++py) {
    const uint32_t packed = (blk.y >> (8 * py)) & 0xffu;
    // 4 texels x 3 bytes = 12 bytes = three aligned 32-bit stores (rows start at multiples of 12 bytes: W % 4 == 0)
    uint32_t bytes[12];
#pragma unroll
    for (int px = 0; px < 4; ++px) {
      const int idx = (packed >> (2 * px)) & 3;
      bytes[px * 3] = (uint32_t)code[idx][0]; bytes[px * 3 + 1] = (uint32_t)code[idx][1]; bytes[px * 3 + 2] = (uint32_t)code[idx][2];
    }
    uint32_t* o = reinterpret_cast<uint32_t*>(img + ((size_t)(by * 4 + py) * W + bx * 4) * 3);
#pragma unroll
    for (int w = 0; w < 3; ++w)
      o[w] = bytes[w * 4] | (bytes[w * 4 + 1] << 8) | (bytes[w * 4 + 2] << 16) | (bytes[w * 4 + 3] << 24);
  }
}

// 8-bit GL_LUMINANCE texel -> normalised fixed point byte / 255 (one IEEE division, as the sampler returns it);
// pre_depth.fs uncompress() (:51-61) is applied later, inside k_bilateral
__global__ void __launch_bounds__(256) k_depth8(const uint8_t* __restrict__ in, float* __restrict__ out, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (float)in[i] / 255.0f;
}

// expand the packed layers of frame slot `slot` into its RGB8 / float32 buffers, on the compute stream
int launch_unpack_frames(rr_ctx* c, int slot) {
  if (c->color_format == RR_COLOR_DXT1 || c->color_format == RR_COLOR_DXT5) {
    const dim3 blk(32, 8, 1), grd((c->CW / 4 + 31) / 32, (c->CH / 4 + 7) / 8, c->N);
    const uint2* src = reinterpret_cast<const uint2*>(c->d_color_packed[slot].ptr);
    if (c->color_format == RR_COLOR_DXT5) k_decode_dxt<true><<<grd, blk, 0, c->stream>>>(src, c->d_color_slot[slot].ptr, c->CW, c->CH);
    else k_decode_dxt<false><<<grd, blk, 0, c->stream>>>(src, c->d_color_slot[slot].ptr, c->CW, c->CH);
    RR_LAUNCH_CHECK(c, "k_decode_dxt");
  }
  if (c->depth_format == RR_DEPTH_U8) {
    const size_t n = (size_t)c->N * c->W * c->H;
    k_depth8<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->d_depth_packed[slot].ptr, c->d_depth_slot[slot].ptr, n);
    RR_LAUNCH_CHECK(c, "k_depth8");
  }
  return RR_OK;
}

}  // namespace rr
