// fusion_playback — headless equivalent of kinect_client's init() + frame loop (source/kinect_client.cpp:194-279,
// 572-617) for the TSDF-integration mode: plays .stream files through NetKinectArray, fuses every frame set and
// raymarches it. Prints the TimerDatabase stage means; optionally dumps the last TSDF volume, image and surface mesh.
//   fusion_playback <file.ks> (--streams "s0;s1;..." | --messages file) [--depth W H --color CW CH] [--frames K] [--voxel m]
//                   [--limit l] [--eye x y z | --matrices file] [--view W H] [--shade m] [--dump-tsdf file] [--dump-image file] [--dense]
//                   [--dump-mesh file.ply [--simplify C] [--min-part-voxels N]] [--dump-points file.ply] [--pick PX PY] [--parts]
//                   [--track-parts N] [--distance X Y Z] [--remove-parts N]
//                   [--gpus N | --devices a,b,...] [--recon points|trigrid|calibs [--min-length m] [--dump-recon file]]
// --recon: like kinect_client's reconstruction list (source/kinect_client.cpp:251-257, key-selected g_recon_mode), one of the
// other reconstructions also draws the last frame set's maps - ReconPoints, ReconTrigrid (min_length from the sensor .yml
// unless --min-length is given) or ReconCalibs - and --dump-recon writes its image (rgba float32 [h][w][4], then depth [h][w]).
// --gpus N / --devices: the volume is split into z-slabs over several devices in this one process (rr_group: frame sets by
// peer copies from the first device, per-slab integration, the view composited on the first device); after the first frame
// the slabs are re-cut to equal integrate cost. A device may be named more than once (slabs sharing a GPU).
// --dump-mesh: the last frame set's fused surface (ReconIntegration::extractMesh) as a binary PLY with normals and colours.
// --simplify C: with --dump-mesh, the mesh simplified by vertex clustering with clusters of C voxels per side
//   (ReconIntegration::simplifyMesh) instead of the full one.
// --min-part-voxels N: with --dump-mesh, only the triangles of connected parts of at least N voxels, and the vertices they
//   use, in their original order and re-indexed (drops the small floating blobs sensor noise leaves in front of the surface).
//   With --simplify, a simplified triangle is in the part of its source triangle.
// --remove-parts N: after every frame set's fuse, before anything reads the volume (the view, --recon, the dumps, --pick,
//   --parts, --track-parts, --distance), its connected parts of fewer than N voxels are taken out of the volume
//   (ReconIntegration::labelParts, then removeParts): one line "frame F removed K parts V voxels" per frame set.
// --parts: one line per connected part of the last frame set's volume (ReconIntegration::labelParts): index, voxels, box
//   (x0 x1 y0 y1 z0 z1, half-open voxel ranges) and centroid (metres).
// --track-parts N: after every frame set, its connected parts with track ids that persist across frame sets
//   (ReconIntegration::trackParts with min_voxels N, matched by voxel overlap): one line "frame F part K track T voxels V
//   prev Q overlap O" per part of at least N voxels (Q = 4294967295 and O = 0 for a new track), then one line
//   "frame F ended T" per track that ended; F counts frame sets from 0.
// --distance X Y Z: after every frame set, how far the world point (X, Y, Z) (metres) is from the fused surface
//   (ReconIntegration::distanceField, then sampleDistance): one line "frame F distance D nearest x y z voxel V" (%.9g, so
//   every binary32 value is exact; D = inf when nothing is inside, nan with voxel 4294967295 outside the bbox).
// --dump-points: the last frame set's pre-processed sensor points (ReconPoints::extractPoints) as a binary PLY with normals,
// colours and quality (with --gpus N through the group call: pre-processing is replicated on every member).
// --pick PX PY: picking as kinect_client's view would do it - the world ray through the centre of view pixel (PX, PY) (GL window
// coordinates, row 0 = bottom) of the playback camera, cast into the last frame set's volume (ReconIntegration::castRays).
// Prints one line: "pick origin x y z direction x y z hit x y z normal x y z rgba r g b a step s", %.9g so every binary32
// value round-trips (NaN hit and normal, rgba 0 and step 4294967295 when the ray hits nothing).
// Without --depth/--color the sizes and stream formats (DXT1 colour, 8-bit depth, near/far) come from the sensors' .yml
// files like in the reference (CalibrationFiles, calibration_files.cpp:7-34). --messages plays a file of back-to-back
// server messages (the ZMQ payload layout of NetKinectArray::readLoop, :511-538) through NetKinectArray::pushMessage.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <utility>

#include "rr_host.hpp"

static void look_at(const float eye[3], const float at[3], float m[16]) {          // gluLookAt, column-major
  float f[3] = {at[0] - eye[0], at[1] - eye[1], at[2] - eye[2]};
  float fl = std::sqrt(f[0] * f[0] + f[1] * f[1] + f[2] * f[2]);
  for (float& v : f) v /= fl;
  const float up[3] = {0.f, 1.f, 0.f};
  float s[3] = {f[1] * up[2] - f[2] * up[1], f[2] * up[0] - f[0] * up[2], f[0] * up[1] - f[1] * up[0]};
  float sl = std::sqrt(s[0] * s[0] + s[1] * s[1] + s[2] * s[2]);
  for (float& v : s) v /= sl;
  const float u[3] = {s[1] * f[2] - s[2] * f[1], s[2] * f[0] - s[0] * f[2], s[0] * f[1] - s[1] * f[0]};
  const float r[3][3] = {{s[0], s[1], s[2]}, {u[0], u[1], u[2]}, {-f[0], -f[1], -f[2]}};
  for (int row = 0; row < 3; ++row) {
    for (int c = 0; c < 3; ++c) m[c * 4 + row] = r[row][c];
    m[12 + row] = -(r[row][0] * eye[0] + r[row][1] * eye[1] + r[row][2] * eye[2]);
  }
  m[3] = m[7] = m[11] = 0.f; m[15] = 1.f;
}
static void perspective(float fovy_deg, float aspect, float n, float f, float m[16]) {   // gluPerspective
  std::memset(m, 0, sizeof(float) * 16);
  const float t = 1.0f / std::tan(fovy_deg * 3.14159265358979f / 360.0f);
  m[0] = t / aspect; m[5] = t; m[10] = (f + n) / (n - f); m[11] = -1.f; m[14] = 2.f * f * n / (n - f);
}

// inverse of a column-major 4x4 matrix by Gauss-Jordan elimination with partial pivoting, in double
static bool invert4(const double* m, double* out) {
  double a[4][8];
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c) { a[r][c] = m[c * 4 + r]; a[r][c + 4] = r == c ? 1.0 : 0.0; }
  for (int c = 0; c < 4; ++c) {
    int p = c;
    for (int r = c + 1; r < 4; ++r) if (std::fabs(a[r][c]) > std::fabs(a[p][c])) p = r;
    if (a[p][c] == 0.0) return false;
    for (int k = 0; k < 8; ++k) std::swap(a[c][k], a[p][k]);
    const double d = a[c][c];
    for (int k = 0; k < 8; ++k) a[c][k] /= d;
    for (int r = 0; r < 4; ++r)
      if (r != c) { const double f = a[r][c]; for (int k = 0; k < 8; ++k) a[r][k] -= f * a[c][k]; }
  }
  for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) out[c * 4 + r] = a[r][c + 4];
  return true;
}

// The world ray through the centre of window pixel (px, py) of a vw x vh view: from the eye (inverse modelview applied to the
// origin) towards the pixel's point on the far plane (inverse projection, then inverse modelview), in double, rounded once.
static void pick_ray(const float* mv, const float* pr, unsigned vw, unsigned vh, int px, int py, std::vector<float>& origin,
                     std::vector<float>& direction) {
  double M[16], P[16], iM[16], iP[16];
  for (int i = 0; i < 16; ++i) { M[i] = mv[i]; P[i] = pr[i]; }
  if (!invert4(M, iM) || !invert4(P, iP)) throw std::runtime_error("--pick: singular view matrices");
  const double ndc[4] = {(px + 0.5) / vw * 2.0 - 1.0, (py + 0.5) / vh * 2.0 - 1.0, 1.0, 1.0};
  double eye[4], world[4];
  for (int r = 0; r < 4; ++r) eye[r] = iP[r] * ndc[0] + iP[4 + r] * ndc[1] + iP[8 + r] * ndc[2] + iP[12 + r] * ndc[3];
  for (int r = 0; r < 4; ++r) world[r] = iM[r] * eye[0] + iM[4 + r] * eye[1] + iM[8 + r] * eye[2] + iM[12 + r] * eye[3];
  origin.assign(3, 0.0f); direction.assign(3, 0.0f);
  for (int a = 0; a < 3; ++a) {
    const double o = iM[12 + a] / iM[15];
    origin[a] = (float)o;
    direction[a] = (float)(world[a] / world[3] - o);
  }
}

int main(int argc, char** argv) {
  std::string ks, streams, messages, dump_tsdf, dump_image, dump_mesh, dump_points, matrices, recon_mode, dump_recon;
  int pick[2] = {-1, -1};
  float min_length = 0.0f;
  bool explicit_sizes = false;
  unsigned W = 512, H = 424, CW = 1280, CH = 1080, VW = 1280, VH = 720;
  int frames = 10, shade = 1;
  float voxel = 0.01f, limit = 0.01f, eye[3] = {1.6f, 1.5f, 2.2f};
  bool dense = false;
  std::vector<int> devices(1, 0);
  bool print_parts = false;
  long long min_part_voxels = -1;
  long long simplify = 0;
  long long track_min_voxels = 0;
  long long remove_min_voxels = -1;
  std::vector<float> distance_point;
  for (int i = 1; i < argc; ++i) {
    auto next = [&](int k) { return std::atof(argv[i + k]); };
    if (!std::strcmp(argv[i], "--depth")) { W = (unsigned)next(1); H = (unsigned)next(2); i += 2; explicit_sizes = true; }
    else if (!std::strcmp(argv[i], "--color")) { CW = (unsigned)next(1); CH = (unsigned)next(2); i += 2; explicit_sizes = true; }
    else if (!std::strcmp(argv[i], "--messages")) messages = argv[++i];
    else if (!std::strcmp(argv[i], "--view")) { VW = (unsigned)next(1); VH = (unsigned)next(2); i += 2; }
    else if (!std::strcmp(argv[i], "--eye")) { eye[0] = (float)next(1); eye[1] = (float)next(2); eye[2] = (float)next(3); i += 3; }
    else if (!std::strcmp(argv[i], "--streams")) streams = argv[++i];
    else if (!std::strcmp(argv[i], "--frames")) frames = std::atoi(argv[++i]);
    else if (!std::strcmp(argv[i], "--voxel")) voxel = (float)std::atof(argv[++i]);
    else if (!std::strcmp(argv[i], "--limit")) limit = (float)std::atof(argv[++i]);
    else if (!std::strcmp(argv[i], "--shade")) shade = std::atoi(argv[++i]);
    else if (!std::strcmp(argv[i], "--dump-tsdf")) dump_tsdf = argv[++i];
    else if (!std::strcmp(argv[i], "--dump-image")) dump_image = argv[++i];
    else if (!std::strcmp(argv[i], "--dump-mesh")) dump_mesh = argv[++i];
    else if (!std::strcmp(argv[i], "--dump-points")) dump_points = argv[++i];
    else if (!std::strcmp(argv[i], "--pick")) { pick[0] = std::atoi(argv[i + 1]); pick[1] = std::atoi(argv[i + 2]); i += 2; }
    else if (!std::strcmp(argv[i], "--dense")) dense = true;
    else if (!std::strcmp(argv[i], "--parts")) print_parts = true;
    else if (!std::strcmp(argv[i], "--min-part-voxels")) min_part_voxels = std::atoll(argv[++i]);
    else if (!std::strcmp(argv[i], "--simplify")) simplify = std::atoll(argv[++i]);
    else if (!std::strcmp(argv[i], "--track-parts")) track_min_voxels = std::atoll(argv[++i]);
    else if (!std::strcmp(argv[i], "--remove-parts")) remove_min_voxels = std::atoll(argv[++i]);
    else if (!std::strcmp(argv[i], "--distance")) { distance_point = {(float)next(1), (float)next(2), (float)next(3)}; i += 3; }
    else if (!std::strcmp(argv[i], "--gpus")) { devices.clear(); for (int d = 0, n = std::atoi(argv[++i]); d < n; ++d) devices.push_back(d); }
    else if (!std::strcmp(argv[i], "--devices")) {
      devices.clear();
      for (char* tok = std::strtok(argv[++i], ","); tok; tok = std::strtok(nullptr, ",")) devices.push_back(std::atoi(tok));
    }
    else if (!std::strcmp(argv[i], "--recon")) recon_mode = argv[++i];
    else if (!std::strcmp(argv[i], "--min-length")) min_length = (float)std::atof(argv[++i]);
    else if (!std::strcmp(argv[i], "--dump-recon")) dump_recon = argv[++i];
    else if (!std::strcmp(argv[i], "--matrices")) matrices = argv[++i];     // 32 floats: modelview, projection (column-major)
    else ks = argv[i];
  }
  if (ks.empty() || (streams.empty() == messages.empty())) { std::cerr << "usage: fusion_playback <file.ks> (--streams \"a;b\" | --messages file) [...]" << std::endl; return 1; }
  try {
    using namespace kinect;
    SceneFile sc = readSceneFile(ks);                                                  // init(): kinect_client.cpp:213-234
    CalibrationFiles calib_files = explicit_sizes ? CalibrationFiles(sc.calib_filenames, W, H, CW, CH) : CalibrationFiles(sc.calib_filenames);
    if (!explicit_sizes)
      std::cout << "streams: depth " << calib_files.getWidth() << "x" << calib_files.getHeight() << (calib_files.isCompressedDepth() ? " 8-bit" : " float32")
                << ", colour " << calib_files.getWidthC() << "x" << calib_files.getHeightC() << (calib_files.isCompressedRGB() == 1 ? " DXT1" : " RGB8")
                << ", near/far " << calib_files.getNear() << " " << calib_files.getFar() << std::endl;
    if (devices.empty()) throw std::runtime_error("--gpus / --devices name no device");
    gpu::Context gpu(devices, calib_files);                                            // stands where the GL context stood
    if (devices.size() > 1) std::cout << "z-slabs over " << devices.size() << " devices" << std::endl;
    CalibVolumes cv(sc.calib_filenames, sc.bbox);                                      // :241
    NetKinectArray nka(streams, "", &calib_files, &cv, !streams.empty());              // :242
    std::ifstream msg_file;
    std::vector<char> msg;
    if (!messages.empty()) {
      msg_file.open(messages, std::ios::binary);
      if (!msg_file) throw std::runtime_error("cannot open message file " + messages);
      const std::size_t csz = calib_files.isCompressedRGB() == 1 ? (std::size_t)calib_files.getWidthC() * calib_files.getHeightC() / 2
                                                                  : (std::size_t)calib_files.getWidthC() * calib_files.getHeightC() * 3;
      const std::size_t dsz = (std::size_t)calib_files.getWidth() * calib_files.getHeight() * (calib_files.isCompressedDepth() ? 1 : sizeof(float));
      msg.resize((csz + dsz) * calib_files.num());
    }
    cv.loadInverseCalibs(sc.resource_path);                                            // :248
    ReconIntegration recon(calib_files, &cv, sc.bbox, limit, voxel);                   // :252
    recon.setUseBricks(!dense);
    recon.setShadeMode(shade);
    recon.resize(VW, VH);
    if (calib_files.isCompressedDepth()) nka.useProcessedDepths(false);                // pre_morph.fs validates metres: 8-bit streams skip it
    float mv[16], pr[16];
    const float at[3] = {0.5f * (sc.bbox.getPMin()[0] + sc.bbox.getPMax()[0]), 1.1f, 0.5f * (sc.bbox.getPMin()[2] + sc.bbox.getPMax()[2])};
    look_at(eye, at, mv);
    perspective(50.0f, float(VW) / float(VH), 0.1f, 10.0f, pr);
    if (!matrices.empty()) {
      std::ifstream m(matrices, std::ios::binary);
      m.read(reinterpret_cast<char*>(mv), sizeof(mv));
      m.read(reinterpret_cast<char*>(pr), sizeof(pr));
      if (!m) throw std::runtime_error("cannot read 32 floats from " + matrices);
    }
    recon.setViewMatrices(mv, pr);
    TimerDatabase::instance().enable(1);
    int done = 0;
    while (done < frames) {                                                            // draw3d(): :583-617
      if (!messages.empty()) {                                                         // what readLoop does per recv()
        msg_file.read(msg.data(), (std::streamsize)msg.size());
        if (!msg_file) { msg_file.clear(); msg_file.seekg(0); msg_file.read(msg.data(), (std::streamsize)msg.size()); }
        if (!msg_file) throw std::runtime_error("message file holds no complete message");
        nka.pushMessage(msg.data(), msg.size());
      }
      if (!nka.update()) continue;
      recon.clearOccupiedBricks();                                                     // process_textures(): :572-580
      nka.processTextures();
      recon.updateOccupiedBricks();
      recon.integrate();
      if (remove_min_voxels >= 0) {                                                    // floaters out of the volume, per frame set
        Parts labelled;
        recon.labelParts(labelled);
        const std::pair<uint32_t, uint32_t> removed = recon.removeParts((uint32_t)remove_min_voxels);
        std::printf("frame %d removed %u parts %u voxels\n", done, (unsigned)removed.first, (unsigned)removed.second);
      }
      recon.drawF();
      if (done == 0 && devices.size() > 1) gpu.balanceSlabs();                        // occupied bricks cluster around the subject
      if (track_min_voxels > 0) {                                                      // persistent part ids, per frame set
        Parts parts;
        PartTracks tracks;
        recon.trackParts((uint32_t)track_min_voxels, parts, tracks);
        for (std::size_t k = 0; k < parts.voxels.size(); ++k)
          if (tracks.track_ids[k] != 0xFFFFFFFFu)
            std::printf("frame %d part %zu track %u voxels %u prev %u overlap %u\n", done, k, (unsigned)tracks.track_ids[k],
                        (unsigned)parts.voxels[k], (unsigned)tracks.prev_parts[k], (unsigned)tracks.overlaps[k]);
        for (uint32_t t : tracks.ended) std::printf("frame %d ended %u\n", done, (unsigned)t);
      }
      if (!distance_point.empty()) {                                                   // distance to the surface, per frame set
        std::vector<float> dist, nearest;
        std::vector<uint32_t> voxel;
        recon.distanceField();
        recon.sampleDistance(distance_point, dist, nearest, voxel);
        std::printf("frame %d distance %.9g nearest %.9g %.9g %.9g voxel %u\n", done, dist[0], nearest[0], nearest[1], nearest[2],
                    (unsigned)voxel[0]);
      }
      ++done;
    }
    if (!messages.empty()) std::cout << "last frame time " << nka.getCurrentFrameTime() << std::endl;
    std::cout << "frames " << done << " bricks " << recon.numBricks() << " occupied ratio " << recon.occupiedRatio() << " brick size " << recon.getBrickSize() << std::endl;
    for (char const* name : {"1preprocess", "2integrate", "3recon"})
      std::cout << name << " mean ms " << TimerDatabase::instance().mean(name) << std::endl;
    if (!dump_tsdf.empty()) {
      std::vector<float> tsdf;
      recon.downloadTsdf(tsdf);
      std::ofstream(dump_tsdf, std::ios::binary).write(reinterpret_cast<char const*>(tsdf.data()), (std::streamsize)(tsdf.size() * sizeof(float)));
    }
    Parts parts;
    if (print_parts || (!dump_mesh.empty() && min_part_voxels >= 0)) recon.labelParts(parts);
    if (print_parts)
      for (std::size_t k = 0; k < parts.voxels.size(); ++k) {
        const int32_t* b = &parts.boxes[k * 6];
        const float* c = &parts.centroids[k * 3];
        std::printf("part %zu voxels %u box %d %d %d %d %d %d centroid %.9g %.9g %.9g\n", k, (unsigned)parts.voxels[k], b[0], b[1], b[2],
                    b[3], b[4], b[5], c[0], c[1], c[2]);
      }
    std::fflush(stdout);
    if (!dump_mesh.empty()) {
      Mesh mesh;
      recon.extractMesh(mesh);
      std::vector<uint32_t> tparts;   // the part of each triangle of `mesh`
      if (min_part_voxels >= 0) {
        std::vector<uint32_t> vparts;
        recon.meshParts(vparts, tparts);
      }
      if (simplify > 0) {
        Mesh simple;
        std::vector<uint32_t> sources;
        recon.simplifyMesh((uint32_t)simplify, simple, &sources);
        if (min_part_voxels >= 0) {   // a simplified triangle is in its source triangle's part
          std::vector<uint32_t> sparts(sources.size());
          for (std::size_t t = 0; t < sources.size(); ++t) sparts[t] = tparts[sources[t]];
          tparts.swap(sparts);
        }
        std::swap(mesh, simple);
      }
      if (min_part_voxels >= 0) {
        const std::size_t nv = mesh.positions.size() / 3;
        Mesh kept;
        std::vector<uint32_t> index(nv, 0xFFFFFFFFu);
        std::vector<char> used(nv, 0);
        for (std::size_t t = 0; t < tparts.size(); ++t)
          if (parts.voxels[tparts[t]] >= (unsigned long long)min_part_voxels)
            for (int j = 0; j < 3; ++j) used[mesh.triangles[t * 3 + j]] = 1;
        for (std::size_t v = 0; v < used.size(); ++v) {
          if (!used[v]) continue;
          index[v] = (uint32_t)(kept.positions.size() / 3);
          kept.positions.insert(kept.positions.end(), &mesh.positions[v * 3], &mesh.positions[v * 3] + 3);
          kept.normals.insert(kept.normals.end(), &mesh.normals[v * 3], &mesh.normals[v * 3] + 3);
          kept.rgba.insert(kept.rgba.end(), &mesh.rgba[v * 4], &mesh.rgba[v * 4] + 4);
        }
        for (std::size_t t = 0; t < tparts.size(); ++t)
          if (parts.voxels[tparts[t]] >= (unsigned long long)min_part_voxels)
            for (int j = 0; j < 3; ++j) kept.triangles.push_back(index[mesh.triangles[t * 3 + j]]);
        mesh.positions.swap(kept.positions); mesh.normals.swap(kept.normals); mesh.rgba.swap(kept.rgba);
        mesh.triangles.swap(kept.triangles);
      }
      writePly(dump_mesh, mesh);
      std::cout << "mesh vertices " << mesh.positions.size() / 3 << " triangles " << mesh.triangles.size() / 3 << std::endl;
    }
    if (!dump_points.empty()) {
      PointCloud cloud;
      ReconPoints(calib_files, &cv, sc.bbox).extractPoints(cloud);
      writePly(dump_points, cloud);
      std::cout << "points " << cloud.pixels.size() << std::endl;
    }
    if (pick[0] >= 0) {
      std::vector<float> origin, direction, hit, normal, rgba;
      std::vector<uint32_t> step;
      pick_ray(mv, pr, VW, VH, pick[0], pick[1], origin, direction);
      recon.castRays(origin, direction, hit, normal, rgba, step);
      std::printf("pick origin %.9g %.9g %.9g direction %.9g %.9g %.9g hit %.9g %.9g %.9g normal %.9g %.9g %.9g rgba %.9g %.9g %.9g %.9g step %u\n",
                  origin[0], origin[1], origin[2], direction[0], direction[1], direction[2], hit[0], hit[1], hit[2],
                  normal[0], normal[1], normal[2], rgba[0], rgba[1], rgba[2], rgba[3], (unsigned)step[0]);
      std::fflush(stdout);
    }
    if (!recon_mode.empty()) {
      // the other reconstructions consume the maps of the last processTextures() (and, ReconCalibs, the fused volume)
      std::vector<float> const* rgba = nullptr; std::vector<float> const* depth = nullptr;
      ReconPoints points(calib_files, &cv, sc.bbox);
      ReconTrigrid trigrid(calib_files, &cv, sc.bbox);
      ReconCalibs calibs(calib_files, &cv, sc.bbox);
      if (recon_mode == "points") {
        points.setShadeMode(shade); points.resize(VW, VH); points.setViewMatrices(mv, pr); points.drawF();
        rgba = &points.colorImage(); depth = &points.depthImage();
      } else if (recon_mode == "trigrid") {
        if (min_length > 0.0f) trigrid.setMinLength(min_length);
        trigrid.setShadeMode(shade); trigrid.resize(VW, VH); trigrid.setViewMatrices(mv, pr); trigrid.drawF();
        rgba = &trigrid.colorImage(); depth = &trigrid.depthImage();
      } else if (recon_mode == "calibs") {
        calibs.setTsdfLimit(limit); calibs.resize(VW, VH); calibs.setViewMatrices(mv, pr); calibs.drawF();
        rgba = &calibs.colorImage(); depth = &calibs.depthImage();
      } else {
        throw std::runtime_error("--recon takes points, trigrid or calibs");
      }
      std::size_t covered = 0;
      for (float d : *depth) covered += d < 1.0f ? 1 : 0;
      std::cout << "recon " << recon_mode << " covered pixels " << covered << std::endl;
      if (!dump_recon.empty()) {
        std::ofstream o(dump_recon, std::ios::binary);
        o.write(reinterpret_cast<char const*>(rgba->data()), (std::streamsize)(rgba->size() * sizeof(float)));
        o.write(reinterpret_cast<char const*>(depth->data()), (std::streamsize)(depth->size() * sizeof(float)));
      }
    }
    if (!dump_image.empty()) {
      std::ofstream o(dump_image, std::ios::binary);
      o.write(reinterpret_cast<char const*>(recon.colorImage().data()), (std::streamsize)(recon.colorImage().size() * sizeof(float)));
      o.write(reinterpret_cast<char const*>(recon.depthImage().data()), (std::streamsize)(recon.depthImage().size() * sizeof(float)));
    }
  } catch (std::exception const& e) {
    std::cerr << "fusion_playback: " << e.what() << std::endl;
    return 1;
  }
  return 0;
}
