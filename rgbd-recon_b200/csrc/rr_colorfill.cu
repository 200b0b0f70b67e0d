// Colour hole filling after the raymarch for sm_100a: ReconIntegration::fillColors
// (framework/reconstruction/recon_integration.cpp:280-339) over the ViewLod mip atlas (framework/rendering/view_lod.cpp:
// 24-61) with glsl/framebuffer_transfer.fs, glsl/tsdf_inpaint.fs and glsl/tsdf_colorfill.fs.
//
// The reference ping-pongs two 1.5W x H framebuffers through 2L-1 full-screen passes (L = number of lods): every
// "transfer" squeezes the WHOLE atlas into the W x H viewport of the other buffer (source column = texcoord.x * 1.5W),
// every "inpaint" renders one lod from the squeezed copy. Only one lod changes between two transfers, so here
//   F = the atlas: its lod-0 part is the raymarch output itself, the part right of column W is d_fill_fc / d_fill_fd;
//   S = the squeezed copy (W x H; the cleared columns W..1.5W are implied),
// and each level kernel writes its lod into F AND refreshes exactly the squeezed pixels whose source lies in that lod.
// A squeezed pixel whose source lies in a lod that is not finished yet reads as the cleared value it has in the
// reference at that moment, so levels never race with their own output. Lods of <= TAIL_PIXELS pixels run back to back
// in one CTA. Result: 7 launches at 1280x720 instead of 20 draw calls, same pixels (tests/test_colorfill_gpu.py).
#include "rr_context.h"
#include "rr_math.cuh"

#include <algorithm>
#include <cmath>

namespace rr {

#define FILL_MAX_LODS 20
#define TAIL_PIXELS 1024

struct FillParams {
  int n;                                   // number of lods
  int off[FILL_MAX_LODS][2], res[FILL_MAX_LODS][2];   // elements past n stay zero (unset uniform array elements)
  int W, H, FW;
  const float4* rgba;                      // raymarch output (lod 0 of F)
  const float* zbuf;
  float4* fc; float* fd;                   // F right of column W: [H][FW - W]
  float4* sc; float* sd;                   // S: [H][W]
  float4* out;                             // filled colour [H][W]
};

__device__ __forceinline__ float4 clear_color() { return make_float4(0.0f, 1.0f, 0.0f, 0.0f); }

// lod 0 of F: a pixel the raymarch discarded (alpha 0), or whose fragment failed GL_LESS against the cleared 1.0,
// keeps the cleared framebuffer value
__device__ __forceinline__ void fetch_lod0(const FillParams& p, int x, int y, float4& c, float& d) {
  const float4 v = __ldg(p.rgba + (size_t)y * p.W + x);
  const float z = __ldg(p.zbuf + (size_t)y * p.W + x);
  const bool drawn = (v.w != 0.0f) && (z < 1.0f);
  c = drawn ? v : clear_color();
  d = drawn ? z : 1.0f;
}

// texelFetch on F; outside the texture -> zeros
__device__ __forceinline__ void fetch_F(const FillParams& p, int x, int y, float4& c, float& d) {
  if (x < 0 || y < 0 || x >= p.FW || y >= p.H) { c = make_float4(0.f, 0.f, 0.f, 0.f); d = 0.0f; return; }
  if (x < p.W) { fetch_lod0(p, x, y, c, d); return; }
  const size_t i = (size_t)y * (p.FW - p.W) + (x - p.W);
  c = p.fc[i]; d = p.fd[i];
}

// source column of squeezed pixel px (framebuffer_transfer.fs:14: ivec2(pass_TexCoord * resolution_tex))
__device__ __forceinline__ int squeeze_src(const FillParams& p, int px) {
  const float tx = ((float)px + 0.5f) / (float)p.W;
  return (int)(tx * (float)p.FW);
}

// texelFetch on S as it is while lod `level` is being rendered (lods < level finished, the others still cleared)
__device__ __forceinline__ void fetch_S(const FillParams& p, int level, int x, int y, float4& c, float& d) {
  // Branch-free: the two loads are issued unconditionally from a clamped address and the special cases select afterwards, so
  // the sixteen fetches of an inpaint fragment are in flight together instead of one L2 round trip after the other.
  const bool outside = (x < 0 || y < 0 || x >= p.FW || y >= p.H);
  const bool right = x >= p.W;                         // F's lod columns: S holds the clear colour there
  // rows of the lods that are not finished yet: everything above lod level-1's rows (all rows for level 1)
  const int unfinished_below = (level == 1) ? p.H : p.off[level - 1][1];
  const bool cleared = right || (y < unfinished_below && squeeze_src(p, x) >= p.W);
  const bool load = !outside && !cleared;
  const size_t i = load ? (size_t)y * p.W + x : 0;
  const float4 cv = __ldcg(p.sc + i);                  // L2 reads: the tail kernel reads what earlier levels of the same CTA wrote
  const float dv = __ldcg(p.sd + i);
  c = outside ? make_float4(0.f, 0.f, 0.f, 0.f) : (cleared ? clear_color() : cv);
  d = outside ? 0.0f : (cleared ? 1.0f : dv);
}

// tsdf_inpaint.fs:34-88 for fragment (fx, fy) of lod `level` (shader uniform lod = level - 1)
__device__ void inpaint_pixel(const FillParams& p, int level, int fx, int fy) {
  const int l = level - 1;
  const int ox = p.off[level][0], oy = p.off[level][1], rx = p.res[level][0], ry = p.res[level][1];
  const float tcx = ((float)fx - (float)ox) / (float)rx, tcy = ((float)fy - (float)oy) / (float)ry;
  const int lx = (int)((float)p.off[l][0] + (float)p.res[l][0] * tcx), ly = (int)((float)p.off[l][1] + (float)p.res[l][1] * tcy);
  const int pix = (int)((float)lx * (2.0f / 3.0f)), piy = (int)((float)ly * 1.0f);
  float depth_av = 0.0f;
  int num_samples = 0;
  float4 samples[16];
#pragma unroll
  for (int x = 0; x < 4; ++x)
#pragma unroll
    for (int y = 0; y < 4; ++y) {
      float4 color; float depth;
      fetch_S(p, level, pix + x - 1, piy + y - 1, color, depth);
      if (color.w <= 0.0f) color.x = -1.0f;
      else { depth_av += depth; ++num_samples; }
      samples[x + y * 4] = make_float4(color.x, color.y, color.z, depth);
    }
  float4 out;
  float out_depth;
  if (num_samples == 0) {
    float4 c;
    fetch_S(p, level, pix, piy, c, out_depth);
    out = (out_depth < 1.0f) ? make_float4(0.f, 0.f, 0.f, -1.f) : clear_color();
  } else {
    depth_av /= (float)num_samples;
    float t0 = 0.f, t1 = 0.f, t2 = 0.f, total_depth = 0.0f, total_weight = 0.0f;
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (samples[i].x >= 0.0f && samples[i].w >= depth_av) {
        t0 += samples[i].x * 1.0f; t1 += samples[i].y * 1.0f; t2 += samples[i].z * 1.0f;
        total_depth += samples[i].w * 1.0f;
        total_weight += 1.0f;
      }
    out = make_float4(t0 / total_weight, t1 / total_weight, t2 / total_weight, 1.0f);
    out_depth = total_depth / total_weight;
  }
  if (fx < p.FW && fy < p.H) {                       // GL clips the viewport to the framebuffer
    const size_t i = (size_t)fy * (p.FW - p.W) + (fx - p.W);
    p.fc[i] = out; p.fd[i] = out_depth;
    // the next transfer copies this texel to the squeezed pixel whose source column it is (at most one)
    const int c0 = (int)((float)fx / 1.5f);
    for (int px = max(0, c0 - 1); px <= min(p.W - 1, c0 + 1); ++px)
      if (squeeze_src(p, px) == fx) { p.sc[(size_t)fy * p.W + px] = out; p.sd[(size_t)fy * p.W + px] = out_depth; }
  }
}

// first transfer: S = squeeze(F) with only lod 0 drawn; also clears F right of column W
__global__ void __launch_bounds__(256) k_fill_init(const __grid_constant__ FillParams p) {
  const int px = blockIdx.x * 32 + threadIdx.x, py = blockIdx.y * 8 + threadIdx.y;
  if (px >= p.W || py >= p.H) return;
  const int sx = squeeze_src(p, px);
  float4 c = clear_color(); float d = 1.0f;
  if (sx < p.W) fetch_lod0(p, sx, py, c, d);
  p.sc[(size_t)py * p.W + px] = c; p.sd[(size_t)py * p.W + px] = d;
  if (px < p.FW - p.W) { p.fc[(size_t)py * (p.FW - p.W) + px] = clear_color(); p.fd[(size_t)py * (p.FW - p.W) + px] = 1.0f; }
}

__global__ void __launch_bounds__(256) k_fill_level(const __grid_constant__ FillParams p, int level) {
  const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
  if (x >= p.res[level][0] || y >= p.res[level][1]) return;
  inpaint_pixel(p, level, p.off[level][0] + x, p.off[level][1] + y);
}

// lods first..n-1 in one CTA, one after the other
__global__ void __launch_bounds__(512) k_fill_tail(const __grid_constant__ FillParams p, int first) {
  for (int level = first; level < p.n; ++level) {
    const int rx = p.res[level][0], n = rx * p.res[level][1];
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const int y = i / rx, x = i - y * rx;
      inpaint_pixel(p, level, p.off[level][0] + x, p.off[level][1] + y);
    }
    __syncthreads();
  }
}

// GL 4.4 §8.14.2 MIRRORED_REPEAT
__device__ __forceinline__ int mirror_wrap(int i, int size) {
  int m = i % (2 * size);
  if (m < 0) m += 2 * size;
  int a = m - size;
  if (a < 0) a = -(1 + a);
  return (size - 1) - a;
}

__device__ float4 texture_F(const FillParams& p, float s, float r) {
  const float u = s * (float)p.FW - 0.5f, v = r * (float)p.H - 0.5f;
  const float fu = floorf(u), fv = floorf(v);
  const float a = u - fu, b = v - fv;
  const int i0 = mirror_wrap((int)fu, p.FW), i1 = mirror_wrap((int)fu + 1, p.FW);
  const int j0 = mirror_wrap((int)fv, p.H), j1 = mirror_wrap((int)fv + 1, p.H);
  float4 c00, c10, c01, c11; float d;
  fetch_F(p, i0, j0, c00, d); fetch_F(p, i1, j0, c10, d); fetch_F(p, i0, j1, c01, d); fetch_F(p, i1, j1, c11, d);
  float4 o;
  o.x = lerpf(lerpf(c00.x, c10.x, a), lerpf(c01.x, c11.x, a), b);
  o.y = lerpf(lerpf(c00.y, c10.y, a), lerpf(c01.y, c11.y, a), b);
  o.z = lerpf(lerpf(c00.z, c10.z, a), lerpf(c01.z, c11.z, a), b);
  o.w = lerpf(lerpf(c00.w, c10.w, a), lerpf(c01.w, c11.w, a), b);
  return o;
}

// tsdf_colorfill.fs:30-55 + the GL_LESS depth test against the cleared default framebuffer
__global__ void __launch_bounds__(256) k_fill_final(const __grid_constant__ FillParams p) {
  const int px = blockIdx.x * 32 + threadIdx.x, py = blockIdx.y * 8 + threadIdx.y;
  if (px >= p.W || py >= p.H) return;
  const float tcx = (float)px / (float)p.res[0][0], tcy = (float)py / (float)p.res[0][1];
  const float ptx = ((float)px + 0.5f) / (float)p.W, pty = ((float)py + 0.5f) / (float)p.H;
  // the fragment only survives GL_LESS if the raymarch drew the texel its depth comes from: decide that first, the
  // colour of a discarded fragment is never seen
  float4 c0; float frag_depth;
  const int dx0 = (int)((float)p.off[0][0] + (float)p.res[0][0] * tcx), dy0 = (int)((float)p.off[0][1] + (float)p.res[0][1] * tcy);
  fetch_F(p, dx0, dy0, c0, frag_depth);
  if (!(frag_depth < 1.0f)) { p.out[(size_t)py * p.W + px] = __ldg(p.rgba + (size_t)py * p.W + px); return; }
  float4 out = make_float4(0.f, 0.f, 0.f, 0.f);
  float d;
  int level = 0;
  for (; level < p.n; ++level) {
    const int cx = (int)((float)p.off[level][0] + (float)p.res[level][0] * tcx);
    const int cy = (int)((float)p.off[level][1] + (float)p.res[level][1] * tcy);
    fetch_F(p, cx, cy, out, d);
    if (out.w > 0.0f) break;
  }
  if (level > 0) {
    const float inv_fw = 1.0f / (float)p.FW, inv_h = 1.0f / (float)p.H;
    float px_[2], py_[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int lod = min(level + 1 + k, FILL_MAX_LODS - 1);
      const float o0 = (float)p.off[lod][0], o1 = (float)p.off[lod][1], r0 = (float)p.res[lod][0], r1 = (float)p.res[lod][1];
      px_[k] = gmin(gmax(o0 + r0 * ptx, o0 + 0.5f), (float)(p.off[lod][0] + p.res[lod][0]) - 0.5f);
      py_[k] = gmin(gmax(o1 + r1 * pty, o1 + 0.5f), (float)(p.off[lod][1] + p.res[lod][1]) - 0.5f);
    }
    const float4 c1 = texture_F(p, px_[0] * inv_fw, py_[0] * inv_h);
    const float4 c2 = texture_F(p, px_[1] * inv_fw, py_[1] * inv_h);
    const float dx = ptx - floorf(ptx), dy = pty - floorf(pty);
    const float w1 = sqrtf(fmaf(dy, dy, dx * dx));
    const float w2 = 1.0f - w1;
    const float ws = w1 + w2;
    out = make_float4((c1.x * w1 + c2.x * w2) / ws, (c1.y * w1 + c2.y * w2) / ws, (c1.z * w1 + c2.z * w2) / ws, (c1.w * w1 + c2.w * w2) / ws);
  }
  p.out[(size_t)py * p.W + px] = out;
}

// ViewLod::setResolution (view_lod.cpp:24-52)
static void make_lods(FillParams& p, int W, int H) {
  p.W = W; p.H = H; p.FW = (int)((float)W * 1.5f);
  p.n = std::min(FILL_MAX_LODS, 1 + (int)std::floor(std::log2((float)std::min(W, H))));
  int oy = H;
  for (int i = 0; i < p.n; ++i) {
    p.res[i][0] = (int)std::floor((float)W / std::pow(2.0f, (float)i));
    p.res[i][1] = (int)std::floor((float)H / std::pow(2.0f, (float)i));
    if (i > 0) { oy -= p.res[i][1]; p.off[i][0] = W; p.off[i][1] = oy; }
  }
}

int launch_fill_colors(rr_ctx* c) {
  const int W = c->view_w, H = c->view_h;
  FillParams p{};
  make_lods(p, W, H);
  if (p.FW <= W) return fail(c, RR_ERR_INVALID, "fill colours: view too small");
  if (c->fill_w != W || c->fill_h != H) {
    c->fill_w = c->fill_h = 0;
    const size_t nf = (size_t)(p.FW - W) * H, ns = (size_t)W * H;
    const char* what = "fill colours";
    if (c->d_fill_fc.allocate(c, nf, what) != RR_OK || c->d_fill_fd.allocate(c, nf, what) != RR_OK ||
        c->d_fill_sc.allocate(c, ns, what) != RR_OK || c->d_fill_sd.allocate(c, ns, what) != RR_OK ||
        c->d_filled.allocate(c, ns, what) != RR_OK)
      return fail(c, RR_ERR_CUDA, "fill colours: allocation failed");
    c->fill_w = W; c->fill_h = H;
  }
  p.rgba = c->d_rgba.ptr; p.zbuf = c->d_zbuf.ptr;
  p.fc = c->d_fill_fc.ptr; p.fd = c->d_fill_fd.ptr; p.sc = c->d_fill_sc.ptr; p.sd = c->d_fill_sd.ptr; p.out = c->d_filled.ptr;
  timer_begin(c, "holefill");
  const dim3 blk(32, 8, 1);
  const dim3 grd((W + 31) / 32, (H + 7) / 8, 1);
  k_fill_init<<<grd, blk, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_fill_init");
  int level = 1;
  for (; level < p.n && p.res[level][0] * p.res[level][1] > TAIL_PIXELS; ++level) {
    const dim3 g((p.res[level][0] + 31) / 32, (p.res[level][1] + 7) / 8, 1);
    k_fill_level<<<g, blk, 0, c->stream>>>(p, level);
    RR_LAUNCH_CHECK(c, "k_fill_level");
  }
  if (level < p.n) {
    k_fill_tail<<<1, 512, 0, c->stream>>>(p, level);
    RR_LAUNCH_CHECK(c, "k_fill_tail");
  }
  k_fill_final<<<grd, blk, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_fill_final");
  timer_end(c, "holefill");
  return RR_OK;
}

}  // namespace rr
