// ReconTrigrid::draw (SURVEY.md §8f-4; framework/reconstruction/recon_trigrid.cpp:82-149 with glsl/trigrid_accum.{vs,gs,fs} and
// trigrid_normalize.fs) for sm_100a without a rasteriser: every depth pixel of every sensor spans two triangles of a grid mesh
// (:48-61); pass 1 renders their depth (GL_LESS), pass 2 adds shade() * quality, quality of every fragment within `epsilon` of
// the pass-1 surface (additive blending, no depth test), pass 3 divides by the summed quality.
// Kernels:
//   k_tg_vertices   one thread per grid vertex: trigrid_accum.vs once per vertex instead of six times (64-byte records);
//   k_tg_raster     one thread per triangle, ONE walk for both passes: trigrid_accum.gs (validSurface, flat normal), the
//                   fixed-function stages below, the fragment tests both stages share; every surviving fragment lowers the
//                   pixel's window depth (atomicMin of the bits: order-independent, like GL_LESS's result) AND is appended,
//                   with its eye-space position, its colour * quality and its triangle id, to the pixel's list (A-buffer:
//                   one atomic counter, one atomicExch per fragment);
//   k_tg_resolve    one thread per pixel: pass 2's epsilon test of every listed fragment against the FINAL depth of pass 1,
//                   the survivors summed in ascending triangle id - binary32 additions in exactly the order in-order
//                   blending performs them, so the sums do not depend on the scheduling - then trigrid_normalize.fs.
// Fixed-function stages (OpenGL 4.4), fp64 from the binary32 clip coordinates: near / far clipping in clip space (§13.5; new
// vertices carry barycentric coordinates of the original triangle), perspective divide and viewport transform with depth range
// [0, 1] (§13.6.1), a fragment for every pixel centre inside the (fanned) polygon (§14.6.1), window z interpolated affinely and
// every other attribute perspective-correct (eq. 14.9 / 14.10). Every edge function is evaluated with its end points in one
// canonical order, so the two triangles sharing an edge compute bit-identical values of opposite sign and a pixel centre belongs
// to exactly one of them - with additive blending a doubly drawn seam pixel would show.
// The grid is the reference's as written: cells x < H, y < W (recon_trigrid.cpp:51-52 loops y to tex_width and x to tex_height).
#include "rr_context.h"
#include "rr_draw.cuh"
#include "rr_math.cuh"

#include <algorithm>
#include <cmath>

namespace rr {

struct TrigridParams {
  float mv[16], proj[16], img_to_eye[16];
  float mvT3[9];
  int vw, vh, shade_mode;
  int N, W, H, CW, CH;
  SensorTables st;
  const float2* depth_b; const float* quality; const uint8_t* color;
  float bmin[3], bmax[3];
  float min_length, epsilon;
  float4* verts;                 // [N][W + 1][H + 1][4]
  uint32_t* depth1;              // [vh][vw] bits of the pass-1 window depth (non-negative floats order like their bits)
  uint32_t* head;                // [vh][vw] newest fragment of the pixel's list, 0xFFFFFFFF = none
  float4* frag_rgba; float4* frag_pos; uint2* frag_link;     // colour * quality | quality; eye-space position; (triangle id, next)
  uint32_t frag_cap; uint32_t* frag_count;
  float4* out_rgba; float* out_depth;
};

// bilinear fetch of a one-channel float image, LINEAR + CLAMP_TO_EDGE (kinect_qualities)
__device__ __forceinline__ float tg_tex2d(const float* __restrict__ T, int W, int H, float s, float t) {
  int x0, x1, y0, y1; float a, b;
  lin_coord(s, W, x0, x1, a);
  lin_coord(t, H, y0, y1, b);
  const float v00 = __ldg(T + (size_t)y0 * W + x0), v10 = __ldg(T + (size_t)y0 * W + x1);
  const float v01 = __ldg(T + (size_t)y1 * W + x0), v11 = __ldg(T + (size_t)y1 * W + x1);
  return lerpf(lerpf(v00, v10, a), lerpf(v01, v11, a), b);
}

__global__ void __launch_bounds__(256) k_tg_clear(uint32_t* __restrict__ depth1, uint32_t* __restrict__ head, uint32_t* __restrict__ count, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) *count = 0u;
  if (i < n) { depth1[i] = 0x3f800000u; head[i] = 0xFFFFFFFFu; }
}
__global__ void __launch_bounds__(256) k_tg_clear_lists(uint32_t* __restrict__ head, uint32_t* __restrict__ count, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) *count = 0u;
  if (i < n) head[i] = 0xFFFFFFFFu;
}

// trigrid_accum.vs:22-35
__global__ void __launch_bounds__(256) k_tg_vertices(const __grid_constant__ TrigridParams p, uint32_t n_vertices) {
  const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= n_vertices) return;
  const int GW = p.H + 1, GH = p.W + 1;
  const int layer = (int)(id / (uint32_t)(GW * GH)), r = (int)(id - (uint32_t)layer * (uint32_t)(GW * GH)), j = r / GW, i = r - j * GW;
  const float stepX = 1.0f / (float)p.W, stepY = 1.0f / (float)p.H;
  const float sx = (float)(((double)i + 0.5) * (double)stepX), sy = (float)(((double)j + 0.5) * (double)stepY);
  const size_t px = (size_t)p.W * p.H;
  const float depth = __ldg(p.depth_b + (size_t)layer * px + (size_t)near_coord(sy, p.H) * p.W + near_coord(sx, p.W)).x;   // NEAREST
  const float3 pos_cs = tex3d_xyz(p.st.xyz[layer], p.st.cx[layer], p.st.cy[layer], p.st.cz[layer], sx, sy, depth);
  const float2 tc = tex3d_uv(p.st.uv[layer], p.st.cx[layer], p.st.cy[layer], p.st.cz[layer], sx, sy, depth);
  const float4 es = pmulv(p.mv, make_float4(pos_cs.x, pos_cs.y, pos_cs.z, 1.0f));
  const float4 clip = pmulv(p.proj, es);
  const float q = tg_tex2d(p.quality + (size_t)layer * px, p.W, p.H, sx, sy);
  float4* o = p.verts + (size_t)id * 4;
  o[0] = clip;
  o[1] = make_float4(es.x, es.y, es.z, depth);
  o[2] = make_float4(pos_cs.x, pos_cs.y, pos_cs.z, q);
  o[3] = make_float4(tc.x, tc.y, 0.0f, 0.0f);
}

struct TgVert { double x, y, z, w; double b[3]; };

__device__ __forceinline__ TgVert tg_lerp(const TgVert& A, const TgVert& B, double t) {
  TgVert o;
  o.x = A.x + (B.x - A.x) * t; o.y = A.y + (B.y - A.y) * t; o.z = A.z + (B.z - A.z) * t; o.w = A.w + (B.w - A.w) * t;
#pragma unroll
  for (int k = 0; k < 3; ++k) o.b[k] = A.b[k] + (B.b[k] - A.b[k]) * t;
  return o;
}

// the edge A -> B at P with the end points in canonical (lexicographic x, y) order; s = orientation of the triangle
__device__ __forceinline__ bool tg_edge_inside(double ax, double ay, double bx, double by, double px, double py, double s) {
  const bool flip = (bx < ax) || (bx == ax && by < ay);
  if (flip) { double t = ax; ax = bx; bx = t; t = ay; ay = by; by = t; }
  const double e = (bx - ax) * (py - ay) - (by - ay) * (px - ax);
  const double sigma = flip ? -s : s;
  return sigma > 0.0 ? e >= 0.0 : e < 0.0;
}

__device__ __forceinline__ float tg_interp(const double* B, float a0, float a1, float a2) {
  return (float)((B[0] * (double)a0 + B[1] * (double)a1) + B[2] * (double)a2);
}

__global__ void __launch_bounds__(128) k_tg_raster(const __grid_constant__ TrigridParams p, uint32_t n_triangles) {
  const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= n_triangles) return;
  const int GW = p.H + 1, GH = p.W + 1;
  const uint32_t per_layer = (uint32_t)p.W * p.H * 2u;
  const int layer = (int)(id / per_layer);
  const uint32_t r = id - (uint32_t)layer * per_layer, cell = r >> 1;
  const int k = (int)(r & 1u), y = (int)(cell / (uint32_t)p.H), x = (int)(cell - (uint32_t)y * p.H);
  const float4* g = p.verts + (size_t)layer * GW * GH * 4;
  const float4* a0 = g + ((size_t)y * GW + (k == 0 ? x : x + 1)) * 4;                  // (x, y) | (x + 1, y)
  const float4* a1 = g + ((size_t)(k == 0 ? y : y + 1) * GW + x + 1) * 4;              // (x + 1, y) | (x + 1, y + 1)
  const float4* a2 = g + ((size_t)(y + 1) * GW + x) * 4;                               // (x, y + 1)
  const float4 e0 = __ldg(a0 + 1), e1 = __ldg(a1 + 1), e2 = __ldg(a2 + 1);            // pos_es, depth
  // trigrid_accum.gs:27-37,44-55
  if (e0.w < 0.0f || e1.w < 0.0f || e2.w < 0.0f) return;
  const float4 c0 = __ldg(a0 + 2), c1 = __ldg(a1 + 2), c2 = __ldg(a2 + 2);            // pos_cs, quality
  const float avg_depth = (e0.w + e1.w + e2.w) / 3.0f;
  const float l = p.min_length * avg_depth * 4.0f;
  const float3 pc0 = make_float3(c0.x, c0.y, c0.z), pc1 = make_float3(c1.x, c1.y, c1.z), pc2 = make_float3(c2.x, c2.y, c2.z);
  if (!(length3(pc1 - pc0) < l) || !(length3(pc2 - pc0) < l) || !(length3(pc2 - pc1) < l)) return;
  const float3 pe0 = make_float3(e0.x, e0.y, e0.z), pe1 = make_float3(e1.x, e1.y, e1.z), pe2 = make_float3(e2.x, e2.y, e2.z);
  const float3 tri_normal = normalize3(cross3(pe1 - pe0, pe2 - pe0));
  const float3 nn = normalize3(tri_normal);
  const float3 normal = make_float3(-nn.x, -nn.y, -nn.z);
  const float4 t0 = __ldg(a0 + 3), t1 = __ldg(a1 + 3), t2 = __ldg(a2 + 3);            // texcoord

  // ---- clipping against the near (z >= -w) and far (z <= w) planes ----
  TgVert poly[8];
  int n = 3;
  {
    const float4 k0 = __ldg(a0), k1 = __ldg(a1), k2 = __ldg(a2);
    poly[0].x = k0.x; poly[0].y = k0.y; poly[0].z = k0.z; poly[0].w = k0.w; poly[0].b[0] = 1.0; poly[0].b[1] = 0.0; poly[0].b[2] = 0.0;
    poly[1].x = k1.x; poly[1].y = k1.y; poly[1].z = k1.z; poly[1].w = k1.w; poly[1].b[0] = 0.0; poly[1].b[1] = 1.0; poly[1].b[2] = 0.0;
    poly[2].x = k2.x; poly[2].y = k2.y; poly[2].z = k2.z; poly[2].w = k2.w; poly[2].b[0] = 0.0; poly[2].b[1] = 0.0; poly[2].b[2] = 1.0;
    bool all_in = true;
#pragma unroll
    for (int i = 0; i < 3; ++i) all_in = all_in && (poly[i].z + poly[i].w >= 0.0) && (poly[i].w - poly[i].z >= 0.0);
    if (!all_in) {                                   // Sutherland-Hodgman; an untouched triangle comes out as it went in
      TgVert tmp[8];
      for (int plane = 0; plane < 2; ++plane) {
        int m = 0;
        for (int i = 0; i < n; ++i) {
          const TgVert& A = poly[i]; const TgVert& B = poly[(i + 1) % n];
          const double da = plane == 0 ? A.z + A.w : A.w - A.z, db = plane == 0 ? B.z + B.w : B.w - B.z;
          const bool ia = da >= 0.0, ib = db >= 0.0;
          if (ia) tmp[m++] = A;
          if (ia != ib) tmp[m++] = tg_lerp(A, B, da / (da - db));
        }
        n = m;
        for (int i = 0; i < n; ++i) poly[i] = tmp[i];
        if (n < 3) return;
      }
    }
  }
  double wx[8], wy[8], wz[8], iw[8];
  for (int i = 0; i < n; ++i) {
    if (!(poly[i].w > 0.0)) return;
    wx[i] = (poly[i].x / poly[i].w + 1.0) * 0.5 * (double)p.vw;
    wy[i] = (poly[i].y / poly[i].w + 1.0) * 0.5 * (double)p.vh;
    wz[i] = (poly[i].z / poly[i].w + 1.0) * 0.5;
    iw[i] = 1.0 / poly[i].w;
    if (!isfinite(wx[i]) || !isfinite(wy[i]) || !isfinite(wz[i])) return;
  }
  for (int f = 1; f + 1 < n; ++f) {
    const int i0 = 0, i1 = f, i2 = f + 1;
    const double x0 = wx[i0], y0 = wy[i0], x1 = wx[i1], y1 = wy[i1], x2 = wx[i2], y2 = wy[i2];
    const double den = (x1 - x0) * (y2 - y0) - (x2 - x0) * (y1 - y0);
    if (den == 0.0 || !isfinite(den)) continue;
    const double s = den > 0.0 ? 1.0 : -1.0;
    double lox = fmin(x0, fmin(x1, x2)), hix = fmax(x0, fmax(x1, x2));
    double loy = fmin(y0, fmin(y1, y2)), hiy = fmax(y0, fmax(y1, y2));
    if (hix < 0.0 || hiy < 0.0 || lox > (double)p.vw || loy > (double)p.vh) continue;
    lox = fmax(lox, 0.0); loy = fmax(loy, 0.0); hix = fmin(hix, (double)p.vw); hiy = fmin(hiy, (double)p.vh);
    const int px0 = max(0, (int)floor(lox - 0.5)), px1 = min(p.vw - 1, (int)ceil(hix - 0.5));
    const int py0 = max(0, (int)floor(loy - 0.5)), py1 = min(p.vh - 1, (int)ceil(hiy - 0.5));
    for (int py = py0; py <= py1; ++py)
      for (int px = px0; px <= px1; ++px) {
        const double cx = (double)px + 0.5, cy = (double)py + 0.5;
        if (!tg_edge_inside(x0, y0, x1, y1, cx, cy, s) || !tg_edge_inside(x1, y1, x2, y2, cx, cy, s) || !tg_edge_inside(x2, y2, x0, y0, cx, cy, s)) continue;
        const double b1 = ((cx - x0) * (y2 - y0) - (x2 - x0) * (cy - y0)) / den;
        const double b2 = ((x1 - x0) * (cy - y0) - (cx - x0) * (y1 - y0)) / den;
        const double b0 = (1.0 - b1) - b2;
        float zw = (float)((b0 * wz[i0] + b1 * wz[i1]) + b2 * wz[i2]);
        if (!(zw > 0.0f)) zw = 0.0f;                                 // the depth range is [0, 1]
        if (zw > 1.0f) zw = 1.0f;
        const double q0 = b0 * iw[i0], q1 = b1 * iw[i1], q2 = b2 * iw[i2];
        const double qs = (q0 + q1) + q2;
        const double p0 = q0 / qs, p1 = q1 / qs, p2 = q2 / qs;
        double B[3];
#pragma unroll
        for (int kk = 0; kk < 3; ++kk) B[kk] = (p0 * poly[i0].b[kk] + p1 * poly[i1].b[kk]) + p2 * poly[i2].b[kk];

        // ---- trigrid_accum.fs:41-80 ----
        const float3 pos_cs = make_float3(tg_interp(B, c0.x, c1.x, c2.x), tg_interp(B, c0.y, c1.y, c2.y), tg_interp(B, c0.z, c1.z, c2.z));
        if (!(pos_cs.x >= p.bmin[0] && pos_cs.y >= p.bmin[1] && pos_cs.z >= p.bmin[2] && pos_cs.x <= p.bmax[0] && pos_cs.y <= p.bmax[1] && pos_cs.z <= p.bmax[2])) continue;
        const float ts = tg_interp(B, t0.x, t1.x, t2.x), tt = tg_interp(B, t0.y, t1.y, t2.y);
        if (ts > 0.99f || ts < 0.01f || tt > 0.99f || tt < 0.01f) continue;
        const float3 pos_es = make_float3(tg_interp(B, e0.x, e1.x, e2.x), tg_interp(B, e0.y, e1.y, e2.y), tg_interp(B, e0.z, e1.z, e2.z));
        if (dot3(normal, normalize3(pos_es)) > 0.0f) continue;
        const size_t o = (size_t)py * p.vw + px;
        atomicMin(p.depth1 + o, __float_as_uint(zw));                // pass 1 (stage 0): GL_LESS, depth writes on
        // pass 2 (stage 1) up to its epsilon test, which needs the final depth of pass 1 and is applied by k_tg_resolve
        const float q = tg_interp(B, c0.w, c1.w, c2.w);
        float3 c;
        if (p.shade_mode == 3) {
          const float* cc = kPointCameraColors[layer < 5 ? layer : 4];
          c = make_float3(cc[0], cc[1], cc[2]);
        } else {
          c = pshade(p.shade_mode, p.mvT3, pos_es, normal, tex2d_rgb8(p.color + (size_t)p.CW * p.CH * 3 * layer, p.CW, p.CH, ts, tt));
        }
        const uint32_t slot = atomicAdd(p.frag_count, 1u);
        if (slot < p.frag_cap) {
          p.frag_rgba[slot] = make_float4(c.x * q, c.y * q, c.z * q, q);
          p.frag_pos[slot] = make_float4(pos_es.x, pos_es.y, pos_es.z, 0.0f);
          p.frag_link[slot] = make_uint2(id, atomicExch(p.head + o, slot));
        }
      }
  }
}

// trigrid_accum.fs:60-69 (the epsilon test against pass 1's depth), the additive blend in draw order, trigrid_normalize.fs:13-31
__global__ void __launch_bounds__(256) k_tg_resolve(const __grid_constant__ TrigridParams p) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.vw * p.vh) return;
  const uint32_t head = p.head[i];
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (head != 0xFFFFFFFFu) {
    const int py = i / p.vw, px = i - py * p.vw;
    const float depth_curr = __uint_as_float(p.depth1[i]);
    const float4 pc = pmulv(p.img_to_eye, make_float4(((float)px + 0.5f) + 0.5f, ((float)py + 0.5f) + 0.5f, depth_curr, 1.0f));
    const float3 cur = make_float3(pc.x / pc.w, pc.y / pc.w, pc.z / pc.w);
    long long last = -1;
    for (;;) {                                      // selection by ascending triangle id: lists are a handful of entries long
      long long best = 0x7fffffffffffffffll; uint32_t best_slot = 0xFFFFFFFFu;
      for (uint32_t s = head; s != 0xFFFFFFFFu;) {
        const uint2 lk = p.frag_link[s];
        if ((long long)lk.x > last && (long long)lk.x < best) { best = (long long)lk.x; best_slot = s; }
        s = lk.y;
      }
      if (best_slot == 0xFFFFFFFFu) break;
      last = best;
      const float4 pe = p.frag_pos[best_slot];
      if (p.epsilon < length3(cur - make_float3(pe.x, pe.y, pe.z))) continue;      // occluded by the triangles in front
      const float4 v = p.frag_rgba[best_slot];
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  }
  if (acc.w > 0.0f) {
    p.out_rgba[i] = make_float4(acc.x / acc.w, acc.y / acc.w, acc.z / acc.w, acc.w / acc.w);
    p.out_depth[i] = __uint_as_float(p.depth1[i]);
  } else {
    p.out_rgba[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    p.out_depth[i] = 1.0f;
  }
}

static void tg_matmul4(const double* a, const double* b, double* out) {
  for (int c = 0; c < 4; ++c)
    for (int r = 0; r < 4; ++r) {
      double acc = 0.0;
      for (int k = 0; k < 4; ++k) acc += a[k * 4 + r] * b[c * 4 + k];
      out[c * 4 + r] = acc;
    }
}

// The view images of the context (d_rgba, d_zbuf) receive the result, like a raymarch. One host synchronisation per draw: the
// fragment count is read back, and the walk is repeated with a larger pool if the lists did not fit.
int launch_draw_trigrid(rr_ctx* c, const rr_view* v, float min_length) {
  TrigridParams p{};
  const int vw = v->viewport[2], vh = v->viewport[3], npx = vw * vh;
  double P[16], t[16], t2[16], inv[16];
  for (int i = 0; i < 16; ++i) { P[i] = v->projection[i]; p.mv[i] = v->modelview[i]; p.proj[i] = v->projection[i]; }
  // image_to_eye = inverse(viewport_scale * viewport_translate * projection) (recon_trigrid.cpp:84-95)
  const double Tr[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 1, 1, 1, 1};
  const double Sc[16] = {vw * 0.5, 0, 0, 0, 0, vh * 0.5, 0, 0, 0, 0, 0.5, 0, 0, 0, 0, 1};
  tg_matmul4(Tr, P, t); tg_matmul4(Sc, t, t2);
  if (!pinvert4(t2, inv)) return fail(c, RR_ERR_INVALID, "rr_draw_trigrid: singular projection");
  for (int i = 0; i < 16; ++i) p.img_to_eye[i] = (float)inv[i];
  for (int cc = 0; cc < 3; ++cc) for (int r = 0; r < 3; ++r) p.mvT3[cc * 3 + r] = v->modelview[r * 4 + cc];
  p.vw = vw; p.vh = vh; p.shade_mode = v->shade_mode;
  p.N = c->N; p.W = c->W; p.H = c->H; p.CW = c->CW; p.CH = c->CH;
  p.st = sensor_tables(c);
  p.depth_b = c->d_depth_b.ptr; p.quality = c->d_quality.ptr; p.color = c->d_color;
  for (int a = 0; a < 3; ++a) { p.bmin[a] = c->bbox_min[a]; p.bmax[a] = c->bbox_max[a]; }
  p.min_length = min_length; p.epsilon = 0.075f;                       // recon_trigrid.cpp:35
  const size_t n_vertices = (size_t)c->N * (c->W + 1) * (c->H + 1), n_triangles = (size_t)c->N * c->W * c->H * 2;
  if (n_triangles >= 0xFFFFFFFFull) return fail(c, RR_ERR_UNSUPPORTED, "rr_draw_trigrid: too many triangles");
  RR_TRY_RC(c->d_tg_verts.reserve(c, n_vertices * 4, "trigrid vertices"));
  RR_TRY_RC(c->d_tg_depth.reserve(c, (size_t)npx, "trigrid depth"));
  RR_TRY_RC(c->d_tg_head.reserve(c, (size_t)npx, "trigrid list heads"));
  RR_TRY_RC(c->d_tg_count.reserve(c, 1, "trigrid counter"));
  p.verts = c->d_tg_verts.ptr; p.depth1 = c->d_tg_depth.ptr; p.head = c->d_tg_head.ptr; p.frag_count = c->d_tg_count.ptr;
  p.out_rgba = c->d_rgba.ptr; p.out_depth = c->d_zbuf.ptr;
  timer_begin(c, "3recon");
  timer_begin(c, "draw");
  k_tg_clear<<<(npx + 255) / 256, 256, 0, c->stream>>>(p.depth1, p.head, p.frag_count, npx);
  RR_LAUNCH_CHECK(c, "k_tg_clear");
  k_tg_vertices<<<(unsigned)((n_vertices + 255) / 256), 256, 0, c->stream>>>(p, (uint32_t)n_vertices);
  RR_LAUNCH_CHECK(c, "k_tg_vertices");
  // the fragment pool (colour contributions + list links) holds at least `pool` fragments
  size_t pool = (size_t)npx * (size_t)(tunables().trigrid_pool > 0 ? tunables().trigrid_pool : 1) / 16 + 16;
  for (int attempt = 0;; ++attempt) {
    RR_TRY_RC(c->d_tg_frag_rgba.reserve(c, pool, "trigrid fragments"));
    RR_TRY_RC(c->d_tg_frag_pos.reserve(c, pool, "trigrid fragment positions"));
    RR_TRY_RC(c->d_tg_frag_link.reserve(c, pool, "trigrid fragment links"));
    p.frag_rgba = c->d_tg_frag_rgba.ptr; p.frag_pos = c->d_tg_frag_pos.ptr; p.frag_link = c->d_tg_frag_link.ptr;
    // the capacities are equal unless an earlier reserve failed part way
    const size_t cap = std::min({c->d_tg_frag_rgba.cap, c->d_tg_frag_pos.cap, c->d_tg_frag_link.cap});
    p.frag_cap = (uint32_t)(cap > 0xFFFFFFF0ull ? 0xFFFFFFF0ull : cap);
    k_tg_raster<<<(unsigned)((n_triangles + 127) / 128), 128, 0, c->stream>>>(p, (uint32_t)n_triangles);
    RR_LAUNCH_CHECK(c, "k_tg_raster");
    uint32_t count = 0;
    RR_TRY_RC(check(c, cudaMemcpyAsync(&count, p.frag_count, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream), "trigrid fragment count"));
    RR_TRY_RC(check(c, cudaStreamSynchronize(c->stream), "trigrid fragment count"));
    if (count <= p.frag_cap) break;
    if (attempt > 0 || count >= 0xFFFFFFF0u) return fail(c, RR_ERR_UNSUPPORTED, "rr_draw_trigrid: fragment lists do not fit");
    // the lists did not fit: grow the pool to what this view needs (+ 1/8) and walk the triangles again (the depths the first
    // walk left are the final ones already: lowering them again changes nothing)
    pool = (size_t)count + (size_t)count / 8 + 1024;
    k_tg_clear_lists<<<(npx + 255) / 256, 256, 0, c->stream>>>(p.head, p.frag_count, npx);
    RR_LAUNCH_CHECK(c, "k_tg_clear_lists");
  }
  k_tg_resolve<<<(npx + 255) / 256, 256, 0, c->stream>>>(p);
  RR_LAUNCH_CHECK(c, "k_tg_resolve");
  timer_end(c, "draw");
  timer_end(c, "3recon");
  return RR_OK;
}

}  // namespace rr
