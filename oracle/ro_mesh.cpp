// ORACLE (test infrastructure, NOT product code): scalar restatement of the library's surface extraction (rr_extract_mesh,
// rgbd-recon_b200/csrc/rr_mesh.cu; the contract is stated in include/rgbd_recon_b200.h). Marching cubes over every cell in
// canonical order, with its own generator of the case table. The sample functions are the raymarch oracle's (ro_sample.h). Built
// into its own library (mesh.mk, oracle_mesh.py).
#include "ro_math.h"
#include "ro_sample.h"
#include "ro_mesh.h"

#include <algorithm>
#include <cmath>
#include <vector>

namespace {

const int kTableTris = 10;   // the most a case could need: twelve crossed edges in one loop

struct Table { int ntri[256]; int tri[256][kTableTris * 3]; };

// cube corner c has coordinates (c & 1, c >> 1 & 1, c >> 2 & 1); edge e runs along axis e / 4 from the corner whose two
// other coordinates, in x, y, z order, are (e & 1, e >> 1 & 1)
int corner_of_edge(int e) {
  const int axis = e / 4, bits = e % 4;
  int other[2], n = 0;
  for (int a = 0; a < 3; ++a) if (a != axis) other[n++] = a;
  return ((bits & 1) << other[0]) | (((bits >> 1) & 1) << other[1]);
}

int edge_between(int c0, int c1) {
  const int d = c0 ^ c1, lo = c0 < c1 ? c0 : c1;
  const int axis = d == 1 ? 0 : (d == 2 ? 1 : 2);
  for (int e = axis * 4; e < axis * 4 + 4; ++e) if (corner_of_edge(e) == lo) return e;
  return -1;
}

// twice the coordinates, so midpoints stay integral
void corner2(int c, int* p) { for (int a = 0; a < 3; ++a) p[a] = 2 * ((c >> a) & 1); }
void mid2(int e, int* p) { corner2(corner_of_edge(e), p); p[e / 4] += 1; }

bool make_table(Table& T) {
  for (int cs = 0; cs < 256; ++cs) {
    int succ[12], pred[12];
    for (int e = 0; e < 12; ++e) succ[e] = pred[e] = -1;
    for (int axis = 0; axis < 3; ++axis)
      for (int side = 0; side < 2; ++side) {
        int a1 = -1, a2 = -1;
        for (int a = 0; a < 3; ++a) if (a != axis) { if (a1 < 0) a1 = a; else a2 = a; }
        const int c0 = side << axis;
        const int ring[4] = {c0, c0 | (1 << a1), c0 | (1 << a1) | (1 << a2), c0 | (1 << a2)};
        bool in[4];
        int ncross = 0;
        for (int i = 0; i < 4; ++i) in[i] = (cs >> ring[i]) & 1;
        for (int i = 0; i < 4; ++i) ncross += in[i] != in[(i + 1) % 4];
        std::vector<std::pair<int, int>> segs;     // (edge, edge)
        std::vector<std::vector<int>> keep;        // the inside corners each segment separates
        if (ncross == 2) {
          std::vector<int> ce, ins;
          for (int i = 0; i < 4; ++i) {
            if (in[i] != in[(i + 1) % 4]) ce.push_back(edge_between(ring[i], ring[(i + 1) % 4]));
            if (in[i]) ins.push_back(ring[i]);
          }
          segs.push_back({ce[0], ce[1]});
          keep.push_back(ins);
        } else if (ncross == 4) {
          for (int i = 0; i < 4; ++i)
            if (in[i]) {
              segs.push_back({edge_between(ring[(i + 3) % 4], ring[i]), edge_between(ring[i], ring[(i + 1) % 4])});
              keep.push_back({ring[i]});
            }
        }
        for (size_t s = 0; s < segs.size(); ++s) {
          int pa[3], pb[3];
          mid2(segs[s].first, pa); mid2(segs[s].second, pb);
          // r = (inside centroid - segment midpoint) * 2k in doubled coordinates: exact integers
          long long cen[3] = {0, 0, 0};
          for (int c : keep[s]) { int pc[3]; corner2(c, pc); for (int a = 0; a < 3; ++a) cen[a] += pc[a]; }
          const long long k = (long long)keep[s].size();
          long long d[3], r[3];
          for (int a = 0; a < 3; ++a) { d[a] = pb[a] - pa[a]; r[a] = 2 * cen[a] - k * (pa[a] + pb[a]); }
          // the face's outward normal is +-axis: seen from outside the cube, the inside corners must lie to the right of
          // the direction of travel, i.e. (d x r) . n < 0
          const long long cz = (axis == 0) ? d[1] * r[2] - d[2] * r[1] : (axis == 1) ? d[2] * r[0] - d[0] * r[2] : d[0] * r[1] - d[1] * r[0];
          const long long dn = side ? cz : -cz;
          if (dn == 0) return false;
          const int from = dn < 0 ? segs[s].first : segs[s].second, to = dn < 0 ? segs[s].second : segs[s].first;
          if (succ[from] >= 0 || pred[to] >= 0) return false;
          succ[from] = to; pred[to] = from;
        }
      }
    int n = 0;
    bool seen[12] = {false};
    for (int e = 0; e < 12; ++e) {
      if (succ[e] < 0 || seen[e]) continue;
      std::vector<int> loop;
      for (int f = e; !seen[f]; f = succ[f]) { seen[f] = true; loop.push_back(f); }
      for (size_t i = 1; i + 1 < loop.size(); ++i) {
        if (n >= kTableTris) return false;
        T.tri[cs][3 * n] = loop[0]; T.tri[cs][3 * n + 1] = loop[i]; T.tri[cs][3 * n + 2] = loop[i + 1];
        ++n;
      }
    }
    T.ntri[cs] = n;
  }
  return true;
}

const Table& table() {
  static Table T;
  static const bool ok = make_table(T);
  (void)ok;
  return T;
}

struct Vol {
  const float* v; int X, Y, Z;
  float at(int x, int y, int z) const { return v[((size_t)z * Y + y) * X + x]; }
};

bool fin(float f) { return std::isfinite(f); }

// case of the cell at (x, y, z), -1 with a non-finite corner
int cell_case(const Vol& V, int x, int y, int z) {
  int cs = 0;
  for (int c = 0; c < 8; ++c) {
    const float f = V.at(x + (c & 1), y + ((c >> 1) & 1), z + ((c >> 2) & 1));
    if (!fin(f)) return -1;
    if (f > 0.0f) cs |= 1 << c;
  }
  return cs;
}

bool emitting(const Vol& V, int x, int y, int z) {
  return x >= 0 && y >= 0 && z >= 0 && x < V.X - 1 && y < V.Y - 1 && z < V.Z - 1 && cell_case(V, x, y, z) >= 0;
}

bool has_vertex(const Vol& V, int x, int y, int z, int axis) {
  const int o[3] = {axis == 0, axis == 1, axis == 2};
  if (x + o[0] >= V.X || y + o[1] >= V.Y || z + o[2] >= V.Z) return false;
  const float a = V.at(x, y, z), b = V.at(x + o[0], y + o[1], z + o[2]);
  if (!fin(a) || !fin(b) || (a > 0.0f) == (b > 0.0f)) return false;
  for (int i = 0; i < 2; ++i)
    for (int j = 0; j < 2; ++j) {
      int c[3] = {x, y, z}, n = 0;
      for (int ax = 0; ax < 3; ++ax) {
        if (ax == axis) continue;
        c[ax] -= (n++ == 0) ? i : j;
      }
      if (emitting(V, c[0], c[1], c[2])) return true;
    }
  return false;
}

V3 vertex_q(const Vol& V, int x, int y, int z, int axis) {
  const int i[3] = {x, y, z}, R[3] = {V.X, V.Y, V.Z};
  const float a = V.at(x, y, z), b = V.at(x + (axis == 0), y + (axis == 1), z + (axis == 2));
  const float t = a / (a - b);
  float q[3];
  for (int k = 0; k < 3; ++k) {
    const float step = 1.0f / (float)R[k];
    q[k] = ((float)i[k] + 0.5f) * step;            // voxel centre (volume_sampler.cpp:36-42)
  }
  q[axis] = ((float)i[axis] + 0.5f + t) / (float)R[axis];
  return V3{q[0], q[1], q[2]};
}

}  // namespace

extern "C" {

int ro_mesh_case_table(int32_t* ntri, int32_t* tri) {
  Table T;
  if (!make_table(T)) return -1;
  int most = 0;
  for (int cs = 0; cs < 256; ++cs) {
    ntri[cs] = T.ntri[cs];
    most = std::max(most, T.ntri[cs]);
    for (int j = 0; j < kTableTris * 3; ++j) tri[cs * kTableTris * 3 + j] = j < 3 * T.ntri[cs] ? T.tri[cs][j] : -1;
  }
  return most;
}

void ro_extract_mesh(const float* tsdf, const uint32_t* res, float limit, int N, const float* inv, const int32_t* inv_res,
                     const float* cv_uv, const int32_t* cv_res, const uint8_t* color, int CW, int CH,
                     const float* depth_b, const float* quality, int W, int H, const float* bbox_min, const float* bbox_max,
                     uint64_t* counts, float* positions, float* normals, float* rgba, uint32_t* triangles) {
  const Table& T = table();
  const Vol V{tsdf, (int)res[0], (int)res[1], (int)res[2]};
  const int X = V.X, Y = V.Y, Z = V.Z;
  // vertices: keys per z slice, concatenated in z order
  std::vector<std::vector<uint64_t>> kz(Z);
#pragma omp parallel for schedule(dynamic, 1)
  for (int z = 0; z < Z; ++z)
    for (int y = 0; y < Y; ++y)
      for (int x = 0; x < X; ++x)
        for (int axis = 0; axis < 3; ++axis)
          if (has_vertex(V, x, y, z, axis)) kz[z].push_back((((uint64_t)z * Y + y) * X + x) * 3 + axis);
  std::vector<uint64_t> keys;
  for (auto& k : kz) keys.insert(keys.end(), k.begin(), k.end());
  std::vector<std::vector<uint32_t>> tz(Z > 1 ? Z - 1 : 0);
#pragma omp parallel for schedule(dynamic, 1)
  for (int z = 0; z < Z - 1; ++z)
    for (int y = 0; y < Y - 1; ++y)
      for (int x = 0; x < X - 1; ++x) {
        const int cs = cell_case(V, x, y, z);
        if (cs < 0) continue;
        for (int j = 0; j < 3 * T.ntri[cs]; ++j) {
          const int e = T.tri[cs][j], c = corner_of_edge(e);
          const uint64_t key = (((uint64_t)(z + ((c >> 2) & 1)) * Y + (y + ((c >> 1) & 1))) * X + (x + (c & 1))) * 3 + e / 4;
          tz[z].push_back((uint32_t)(std::lower_bound(keys.begin(), keys.end(), key) - keys.begin()));
        }
      }
  size_t nt = 0;
  for (auto& t : tz) nt += t.size() / 3;
  counts[0] = keys.size();
  counts[1] = nt;
  if (triangles) {
    size_t o = 0;
    for (auto& t : tz) { std::copy(t.begin(), t.end(), triangles + o); o += t.size(); }
  }
  if (!positions && !normals && !rgba) return;
  const RM r{tsdf, X, Y, Z, limit, N, inv, inv_res[0], inv_res[1], inv_res[2], cv_uv, cv_res[0], cv_res[1], cv_res[2],
             color, CW, CH, depth_b, quality, W, H, 0};
  const float size[3] = {bbox_max[0] - bbox_min[0], bbox_max[1] - bbox_min[1], bbox_max[2] - bbox_min[2]};
#pragma omp parallel for schedule(dynamic, 256)
  for (long long i = 0; i < (long long)keys.size(); ++i) {
    const uint64_t lin = keys[i] / 3;
    const int axis = (int)(keys[i] % 3);
    const int x = (int)(lin % X), y = (int)((lin / X) % Y), z = (int)(lin / ((uint64_t)X * Y));
    const V3 q = vertex_q(V, x, y, z, axis);
    if (positions) {
      positions[i * 3] = bbox_min[0] + q.x * size[0];
      positions[i * 3 + 1] = bbox_min[1] + q.y * size[1];
      positions[i * 3 + 2] = bbox_min[2] + q.z * size[2];
    }
    if (normals) {
      const V3 g = get_gradient(r, q, limit * 0.5f);
      const V3 n = normalize3(V3{g.x / size[0], g.y / size[1], g.z / size[2]});
      normals[i * 3] = n.x; normals[i * 3 + 1] = n.y; normals[i * 3 + 2] = n.z;
    }
    if (rgba) {
      const V4 c = blend_colors(r, q);
      rgba[i * 4] = c.x; rgba[i * 4 + 1] = c.y; rgba[i * 4 + 2] = c.z; rgba[i * 4 + 3] = c.w;
    }
  }
}

}  // extern "C"
