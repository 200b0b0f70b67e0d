// ORACLE (test infrastructure, NOT product code): plain sequential restatement of the nearest-inside-voxel transform
// (rr_distance_field, rgbd-recon_b200/csrc/rr_distance.cu; the contract is stated in include/rgbd_recon_b200.h and
// DESIGN.md "Beyond the reference: distances"). Meijster, Roerdink and Hesselink's separable transform, one axis at a
// time, every tie to the smaller coordinate, which together give the smallest linear index among the nearest voxels.
#include <stdint.h>

#include <vector>

namespace {

const uint32_t kNone = 0xFFFFFFFFu;

// squared distance from (x, y, z) to voxel f, over the axes up to `axis` (0: x; 1: x, y)
long long g_of(uint32_t f, int x, int y, int X, int Y, int axis) {
  const long long fx = f % (uint32_t)X, fy = (f / (uint32_t)X) % (uint32_t)Y;
  const long long dx = x - fx, dy = y - fy;
  return axis == 0 ? dx * dx : dx * dx + dy * dy;
}

// floor(a / b), b > 0
long long floor_div(long long a, long long b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

// One column of length m: in[k] are the sites (kNone: none) with costs g[k]; out[v] = in[s] for the site s minimising
// g[s] + (v - s)^2, the smallest s on ties.
void envelope(const std::vector<uint32_t>& in, const std::vector<long long>& g, std::vector<uint32_t>& out,
              std::vector<int>& s, std::vector<int>& t) {
  const int m = (int)in.size();
  int q = -1;
  for (int u = 0; u < m; ++u) {
    if (in[u] == kNone) continue;
    // pop the top while u is strictly below it where the top starts
    while (q >= 0) {
      const long long a = g[s[q]] + (long long)(t[q] - s[q]) * (t[q] - s[q]);
      const long long b = g[u] + (long long)(t[q] - u) * (t[q] - u);
      if (a <= b) break;
      --q;
    }
    if (q < 0) {
      q = 0; s[0] = u; t[0] = 0;
      continue;
    }
    // the last v at which the top is at or below u: g[s] + (v-s)^2 <= g[u] + (v-u)^2  <=>  v <= (g[u]-g[s]+u^2-s^2) / (2(u-s))
    const long long w = 1 + floor_div(g[u] - g[s[q]] + (long long)u * u - (long long)s[q] * s[q], 2LL * (u - s[q]));
    if (w < m) { ++q; s[q] = u; t[q] = (int)w; }
  }
  for (int v = m - 1; v >= 0; --v) {
    if (q < 0) { out[v] = kNone; continue; }
    out[v] = in[s[q]];
    if (v == t[q]) --q;
  }
}

}  // namespace

extern "C" {

// inside uint8 [Z][Y][X] (1: inside) -> nearest uint32 [Z][Y][X]
void ro_distance_field(const uint8_t* inside, int X, int Y, int Z, uint32_t* nearest) {
  const size_t sy = (size_t)X, sz = (size_t)X * Y;
  std::vector<uint32_t> tmp((size_t)X * Y * Z);
  // x: per row the nearest inside x, the left one on ties
#pragma omp parallel for
  for (long long r = 0; r < (long long)Y * Z; ++r) {
    const size_t row = (size_t)r * X;
    std::vector<int> left(X, -1);
    int last = -1;
    for (int x = 0; x < X; ++x) { if (inside[row + x]) last = x; left[x] = last; }
    int next = -1;
    for (int x = X - 1; x >= 0; --x) {
      if (inside[row + x]) next = x;
      const int l = left[x];
      int best = -1;
      if (l >= 0 && (next < 0 || x - l <= next - x)) best = l;
      else best = next;
      nearest[row + x] = best < 0 ? kNone : (uint32_t)(row + best);
    }
  }
  // y, then z: per column the lower envelope of the parabolas g[s] + (v - s)^2
  for (int axis = 1; axis <= 2; ++axis) {
    const uint32_t* src = axis == 1 ? nearest : tmp.data();
    uint32_t* dst = axis == 1 ? tmp.data() : nearest;
    const int m = axis == 1 ? Y : Z, other = axis == 1 ? Z : Y;
    const size_t stride = axis == 1 ? sy : sz;
#pragma omp parallel for
    for (long long c = 0; c < (long long)X * other; ++c) {
      const int x = (int)(c % X), o = (int)(c / X);
      const int y = axis == 2 ? o : 0;
      const size_t base = axis == 1 ? (size_t)o * sz + x : (size_t)o * sy + x;
      std::vector<uint32_t> in(m), out(m);
      std::vector<long long> g(m);
      std::vector<int> s(m), t(m);
      for (int k = 0; k < m; ++k) {
        in[k] = src[base + k * stride];
        g[k] = in[k] == kNone ? 0 : g_of(in[k], x, y, X, Y, axis - 1);
      }
      envelope(in, g, out, s, t);
      for (int k = 0; k < m; ++k) dst[base + k * stride] = out[k];
    }
  }
}

}  // extern "C"
