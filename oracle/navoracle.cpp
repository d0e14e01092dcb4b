// navoracle.cpp -- CPU restatement of the two hot paths (checker for the CUDA implementation).
//
// TEST INFRASTRUCTURE ONLY: used by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
// --impl reference legs.  Nothing under navigation_b200/ links or loads this file.
//
// Written from scratch as plain single-threaded C++ following the reference's algorithms; every function cites the
// reference file:line it follows.  It is pinned (tests/test_oracle_*.py) against
//   * the reference's own known-answer tests (costmap_2d/test/inflation_tests.cpp, obstacle_tests.cpp,
//     base_local_planner/test/{map_grid_test,utest,line_iterator_test,velocity_iterator_test}.cpp), and
//   * oracle/_ref/libnavref.so -- the reference's unmodified sources compiled in place -- on seeded random inputs
//     (bit-for-bit grids, costs and selections), with golden fixtures of those runs committed under tests/golden/.
//
// libstdc++'s std::priority_queue is kept for inflation on purpose: the reference's output depends on its heap tie
// order (SURVEY.md section 7), and the same container + push order reproduces it hash-for-hash.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <memory>
#include <queue>
#include <vector>

#include "oracle_api.h"
#include "scan_ingest_restated.h"
#include "plan_restated.h"

namespace {

enum : uint8_t { kFree = 0, kInscribed = 253, kLethal = 254, kNoInfo = 255 };  // cost_values.h:42-45

// ------------------------------------------------------------------ Costmap2D-shaped grid (costmap_2d.cpp)
struct Grid {
  unsigned sx = 0, sy = 0;
  double res = 0, ox = 0, oy = 0;
  uint8_t def = 0;
  std::vector<uint8_t> c;

  void resize(unsigned nx, unsigned ny, double r, double x, double y) {  // resizeMap :71-85
    sx = nx; sy = ny; res = r; ox = x; oy = y;
    c.assign(size_t(sx) * sy, def);
  }
  void reset_window(unsigned x0, unsigned y0, unsigned xn, unsigned yn) {  // resetMap :93-99
    unsigned len = xn - x0;
    for (unsigned y = y0 * sx + x0; y < yn * sx + x0; y += sx) memset(c.data() + y, def, len);
  }
  bool world_to_map(double wx, double wy, unsigned& mx, unsigned& my) const {  // worldToMap :208-220
    if (wx < ox || wy < oy) return false;
    mx = (int)((wx - ox) / res);
    my = (int)((wy - oy) / res);
    return mx < sx && my < sy;
  }
  void map_to_world(unsigned mx, unsigned my, double& wx, double& wy) const {  // mapToWorld :202-206
    wx = ox + (mx + 0.5) * res;
    wy = oy + (my + 0.5) * res;
  }
  void world_to_map_enforce(double wx, double wy, int& mx, int& my) const {  // worldToMapEnforceBounds :228-262
    if (wx < ox) mx = 0;
    else if (wx > res * (sx - 1) + ox) mx = sx - 1;
    else mx = (int)((wx - ox) / res);
    if (wy < oy) my = 0;
    else if (wy > res * (sy - 1) + oy) my = sy - 1;
    else my = (int)((wy - oy) / res);
  }
  unsigned cell_distance(double world_dist) const {  // cellDistance :181-185
    return (unsigned)std::max(0.0, ceil(world_dist / res));
  }
  double size_m_x() const { return (sx - 1 + 0.5) * res; }  // getSizeInMetersX :440-443
  double size_m_y() const { return (sy - 1 + 0.5) * res; }

  void update_origin(double nox, double noy) {  // updateOrigin :264-313
    int cell_ox = int((nox - ox) / res), cell_oy = int((noy - oy) / res);
    double new_grid_ox = ox + cell_ox * res, new_grid_oy = oy + cell_oy * res;
    int isx = sx, isy = sy;
    int llx = std::min(std::max(cell_ox, 0), isx), lly = std::min(std::max(cell_oy, 0), isy);
    int urx = std::min(std::max(cell_ox + isx, 0), isx), ury = std::min(std::max(cell_oy + isy, 0), isy);
    unsigned w = urx - llx, h = ury - lly;
    std::vector<uint8_t> keep(size_t(w) * h);
    for (unsigned r = 0; r < h; ++r) memcpy(keep.data() + size_t(r) * w, c.data() + size_t(lly + r) * sx + llx, w);
    std::fill(c.begin(), c.end(), def);
    ox = new_grid_ox;
    oy = new_grid_oy;
    int start_x = llx - cell_ox, start_y = lly - cell_oy;
    for (unsigned r = 0; r < h; ++r) memcpy(c.data() + size_t(start_y + r) * sx + start_x, keep.data() + size_t(r) * w, w);
  }
};

// Costmap2D::raytraceLine + bresenham2D (costmap_2d.h:359-412): calls at(offset) for each visited cell.
template <class F>
void raytrace_line(unsigned size_x, F at, unsigned x0, unsigned y0, unsigned x1, unsigned y1,
                   unsigned max_length = UINT32_MAX) {
  int dx = x1 - x0, dy = y1 - y0;
  unsigned adx = abs(dx), ady = abs(dy);
  int off_dx = dx > 0 ? 1 : -1;
  int off_dy = (dy > 0 ? 1 : -1) * int(size_x);
  unsigned offset = y0 * size_x + x0;
  double dist = hypot(dx, dy);
  double scale = (dist == 0.0) ? 1.0 : std::min(1.0, max_length / dist);
  unsigned abs_da, abs_db;
  int off_a, off_b;
  if (adx >= ady) { abs_da = adx; abs_db = ady; off_a = off_dx; off_b = off_dy; }
  else { abs_da = ady; abs_db = adx; off_a = off_dy; off_b = off_dx; }
  int err = abs_da / 2;
  unsigned end = std::min((unsigned)(scale * abs_da), abs_da);
  for (unsigned i = 0; i < end; ++i) {
    at(offset);
    offset += off_a;
    err += abs_db;
    if ((unsigned)err >= abs_da) {
      offset += off_b;
      err -= abs_da;
    }
  }
  at(offset);
}

struct Cell { unsigned x, y; };

// Costmap2D::convexFillCells + polygonOutlineCells (costmap_2d.cpp:344-428), quirks included.
void convex_fill_cells(unsigned size_x, const std::vector<Cell>& poly, std::vector<Cell>& cells) {
  if (poly.size() < 3) return;
  auto gather = [&](unsigned off) { cells.push_back(Cell{off % size_x, off / size_x}); };
  for (size_t i = 0; i + 1 < poly.size(); ++i) raytrace_line(size_x, gather, poly[i].x, poly[i].y, poly[i + 1].x, poly[i + 1].y);
  raytrace_line(size_x, gather, poly.back().x, poly.back().y, poly[0].x, poly[0].y);
  // the reference's "bubble sort by x" (stable, back-stepping)
  size_t i = 0;
  while (i < cells.size() - 1) {
    if (cells[i].x > cells[i + 1].x) {
      std::swap(cells[i], cells[i + 1]);
      if (i > 0) --i;
    } else {
      ++i;
    }
  }
  i = 0;
  Cell min_pt, max_pt;
  unsigned min_x = cells[0].x, max_x = cells[cells.size() - 1].x;
  for (unsigned x = min_x; x <= max_x; ++x) {
    if (i >= cells.size() - 1) break;
    if (cells[i].y < cells[i + 1].y) { min_pt = cells[i]; max_pt = cells[i + 1]; }
    else { min_pt = cells[i + 1]; max_pt = cells[i]; }
    i += 2;
    while (i < cells.size() && cells[i].x == x) {
      if (cells[i].y < min_pt.y) min_pt = cells[i];
      else if (cells[i].y > max_pt.y) max_pt = cells[i];
      ++i;
    }
    for (unsigned y = min_pt.y; y < max_pt.y; ++y) cells.push_back(Cell{x, y});
  }
}

// costmap_math.h distance / costmap_math.cpp:32-63 distanceToLine
double dist2d(double x0, double y0, double x1, double y1) { return hypot(x1 - x0, y1 - y0); }
double distance_to_line(double pX, double pY, double x0, double y0, double x1, double y1) {
  double A = pX - x0, B = pY - y0, C = x1 - x0, D = y1 - y0;
  double dot = A * C + B * D, len_sq = C * C + D * D, param = dot / len_sq;
  double xx, yy;
  if (param < 0) { xx = x0; yy = y0; }
  else if (param > 1) { xx = x1; yy = y1; }
  else { xx = x0 + param * C; yy = y0 + param * D; }
  return dist2d(pX, pY, xx, yy);
}
struct Pt { double x, y; };
void min_max_distances(const std::vector<Pt>& fp, double& mn, double& mx) {  // footprint.cpp:41-67
  mn = std::numeric_limits<double>::max();
  mx = 0.0;
  if (fp.size() <= 2) return;
  for (size_t i = 0; i < fp.size(); ++i) {
    const Pt& a = fp[i];
    const Pt& b = fp[(i + 1) % fp.size()];
    double vd = dist2d(0, 0, a.x, a.y), ed = distance_to_line(0, 0, a.x, a.y, b.x, b.y);
    mn = std::min(mn, std::min(vd, ed));
    mx = std::max(mx, std::max(vd, ed));
  }
}
void transform_footprint(double x, double y, double th, const std::vector<Pt>& spec, std::vector<Pt>& out) {  // :106-120
  out.clear();
  double c = cos(th), s = sin(th);
  for (const Pt& p : spec) out.push_back(Pt{x + (p.x * c - p.y * s), y + (p.x * s + p.y * c)});
}

// ------------------------------------------------------------------ layers
struct Bounds { double minx, miny, maxx, maxy; };
void touch(double x, double y, Bounds& b) {  // costmap_layer.cpp:8-14
  b.minx = std::min(x, b.minx); b.miny = std::min(y, b.miny);
  b.maxx = std::max(x, b.maxx); b.maxy = std::max(y, b.maxy);
}

// the four merge policies, costmap_layer.cpp:62-157
void merge(int policy, const Grid& layer, Grid& master, int min_i, int min_j, int max_i, int max_j) {
  unsigned span = master.sx;
  for (int j = min_j; j < max_j; j++) {
    unsigned it = j * span + min_i;
    for (int i = min_i; i < max_i; i++, it++) {
      uint8_t v = layer.c[it];
      uint8_t& m = master.c[it];
      switch (policy) {
        case NAVO_TRUE_OVERWRITE: m = v; break;
        case NAVO_OVERWRITE: if (v != kNoInfo) m = v; break;
        case NAVO_MAX:
          if (v == kNoInfo) break;
          if (m == kNoInfo || m < v) m = v;
          break;
        case NAVO_ADDITION:
          if (v == kNoInfo) break;
          if (m == kNoInfo) m = v;
          else {
            int sum = m + v;
            m = sum >= kInscribed ? kInscribed - 1 : sum;
          }
          break;
        default: break;
      }
    }
  }
}

struct Obs {
  double ox, oy, oz, obstacle_range, raytrace_range;
  std::vector<float> xyz;
  bool marking, clearing;
};

struct Costmap;

struct LayerBase {
  bool enabled = true;
  virtual ~LayerBase() {}
  virtual void match_size(Costmap&) {}
  virtual void update_bounds(Costmap&, double, double, double, Bounds&) {}
  virtual void update_costs(Costmap&, int, int, int, int) {}
  virtual void on_footprint_changed(Costmap&) {}
  virtual Grid* grid() { return nullptr; }
};

struct Costmap {
  Grid master;
  bool rolling = false, track_unknown = false;
  std::vector<std::unique_ptr<LayerBase>> layers;
  std::vector<Pt> footprint;
  double inscribed = 0, circumscribed = 0;
  int bx0 = 0, bxn = 0, by0 = 0, byn = 0;

  void update_map(double rx, double ry, double ryaw) {  // layered_costmap.cpp:79-150
    if (rolling) master.update_origin(rx - master.size_m_x() / 2, ry - master.size_m_y() / 2);
    if (layers.empty()) return;
    Bounds b{1e30, 1e30, -1e30, -1e30};
    for (auto& l : layers) l->update_bounds(*this, rx, ry, ryaw, b);
    int x0, xn, y0, yn;
    master.world_to_map_enforce(b.minx, b.miny, x0, y0);
    master.world_to_map_enforce(b.maxx, b.maxy, xn, yn);
    x0 = std::max(0, x0);
    xn = std::min(int(master.sx), xn + 1);
    y0 = std::max(0, y0);
    yn = std::min(int(master.sy), yn + 1);
    bx0 = x0; bxn = xn; by0 = y0; byn = yn;
    if (xn < x0 || yn < y0) return;
    master.reset_window(x0, y0, xn, yn);
    for (auto& l : layers) l->update_costs(*this, x0, y0, xn, yn);
  }
};

struct CostLayerBase : LayerBase {  // CostmapLayer (costmap_layer.h:48-151)
  Grid g;
  void match_size(Costmap& cm) override {
    g.def = cm.track_unknown ? kNoInfo : kFree;
    g.resize(cm.master.sx, cm.master.sy, cm.master.res, cm.master.ox, cm.master.oy);
  }
  Grid* grid() override { return &g; }
};

struct GridLayer : CostLayerBase {  // StaticLayer non-rolling branch, static_layer.cpp:263-299
  int policy;
  unsigned x = 0, y = 0, w = 0, h = 0;
  bool updated = false;
  explicit GridLayer(int p) : policy(p) {}
  void update_bounds(Costmap& cm, double, double, double, Bounds& b) override {
    if (!cm.rolling && !updated) return;
    double wx, wy;
    g.map_to_world(x, y, wx, wy);
    b.minx = std::min(wx, b.minx);
    b.miny = std::min(wy, b.miny);
    g.map_to_world(x + w, y + h, wx, wy);
    b.maxx = std::max(wx, b.maxx);
    b.maxy = std::max(wy, b.maxy);
    updated = false;
  }
  void update_costs(Costmap& cm, int a, int b_, int c_, int d) override {
    if (!enabled) return;
    merge(policy, g, cm.master, a, b_, c_, d);
  }
};

struct ObstacleLayer : CostLayerBase {  // obstacle_layer.cpp:340-448, 498-610
  int combination_method;
  bool footprint_clearing;
  double max_obstacle_height;
  std::vector<Obs> obs;
  std::vector<Pt> transformed_footprint;
  ObstacleLayer(int cmeth, bool fc, double mh) : combination_method(cmeth), footprint_clearing(fc), max_obstacle_height(mh) {}

  void raytrace_freespace(const Obs& o, Bounds& b) {  // :498-576
    double ox = o.ox, oy = o.oy;
    unsigned x0, y0;
    if (!g.world_to_map(ox, oy, x0, y0)) return;
    double origin_x = g.ox, origin_y = g.oy;
    double map_end_x = origin_x + g.sx * g.res, map_end_y = origin_y + g.sy * g.res;
    touch(ox, oy, b);
    for (size_t i = 0; i < o.xyz.size() / 3; ++i) {
      double wx = o.xyz[3 * i], wy = o.xyz[3 * i + 1];
      double a = wx - ox, bb = wy - oy;
      if (wx < origin_x) { double t = (origin_x - ox) / a; wx = origin_x; wy = oy + bb * t; }
      if (wy < origin_y) { double t = (origin_y - oy) / bb; wx = ox + a * t; wy = origin_y; }
      if (wx > map_end_x) { double t = (map_end_x - ox) / a; wx = map_end_x - .001; wy = oy + bb * t; }
      if (wy > map_end_y) { double t = (map_end_y - oy) / bb; wx = ox + a * t; wy = map_end_y - .001; }
      unsigned x1, y1;
      if (!g.world_to_map(wx, wy, x1, y1)) continue;
      unsigned cell_range = g.cell_distance(o.raytrace_range);
      uint8_t* cells = g.c.data();
      raytrace_line(g.sx, [cells](unsigned off) { cells[off] = kFree; }, x0, y0, x1, y1, cell_range);
      double dx = wx - ox, dy = wy - oy;  // updateRaytraceBounds :602-610
      double full = hypot(dx, dy);
      double scale = std::min(1.0, o.raytrace_range / full);
      touch(ox + dx * scale, oy + dy * scale, b);
    }
  }

  void update_bounds(Costmap& cm, double rx, double ry, double ryaw, Bounds& b) override {  // :340-413
    if (cm.rolling) g.update_origin(rx - g.size_m_x() / 2, ry - g.size_m_y() / 2);
    if (!enabled) return;
    for (const Obs& o : obs)
      if (o.clearing) raytrace_freespace(o, b);
    for (const Obs& o : obs) {
      if (!o.marking) continue;
      double sq_range = o.obstacle_range * o.obstacle_range;
      for (size_t i = 0; i < o.xyz.size() / 3; ++i) {
        double px = o.xyz[3 * i], py = o.xyz[3 * i + 1], pz = o.xyz[3 * i + 2];
        if (pz > max_obstacle_height) continue;
        double sq = (px - o.ox) * (px - o.ox) + (py - o.oy) * (py - o.oy) + (pz - o.oz) * (pz - o.oz);
        if (sq >= sq_range) continue;
        unsigned mx, my;
        if (!g.world_to_map(px, py, mx, my)) continue;
        g.c[size_t(my) * g.sx + mx] = kLethal;
        touch(px, py, b);
      }
    }
    if (!footprint_clearing) return;  // updateFootprint :415-425
    transform_footprint(rx, ry, ryaw, cm.footprint, transformed_footprint);
    for (const Pt& p : transformed_footprint) touch(p.x, p.y, b);
  }

  void update_costs(Costmap& cm, int a, int b_, int c_, int d) override {  // :427-448
    if (!enabled) return;
    if (footprint_clearing) {  // setConvexPolygonCost, costmap_2d.cpp:315-342
      std::vector<Cell> poly, cells;
      bool ok = true;
      for (const Pt& p : transformed_footprint) {
        Cell loc;
        if (!g.world_to_map(p.x, p.y, loc.x, loc.y)) { ok = false; break; }
        poly.push_back(loc);
      }
      if (ok) {
        convex_fill_cells(g.sx, poly, cells);
        for (const Cell& cc : cells) g.c[size_t(cc.y) * g.sx + cc.x] = kFree;
      }
    }
    if (combination_method == 0) merge(NAVO_OVERWRITE, g, cm.master, a, b_, c_, d);
    else if (combination_method == 1) merge(NAVO_MAX, g, cm.master, a, b_, c_, d);
  }
};


// ------------------------------------------------------------------ VoxelLayer + voxel_grid::VoxelGrid
// costmap_2d/plugins/voxel_layer.cpp:84-177, 262-438 and voxel_grid/include/voxel_grid/voxel_grid.h:95-118, 226-385.
// A column is one uint32: bit z = "unknown or marked", bit z + 16 = "marked" (known marked 11, unknown 01, free 00).
struct VoxelLayer : ObstacleLayer {
  double origin_z, z_resolution;
  unsigned size_z, unknown_threshold, mark_threshold;
  std::vector<uint32_t> vox;
  VoxelLayer(int cmeth, bool fc, double mh, double oz, double zres, int zv, int unknown_thr, int mark_thr)
      : ObstacleLayer(cmeth, fc, mh), origin_z(oz), z_resolution(zres), size_z(std::min(zv, 16)),
        unknown_threshold(unknown_thr + (16 - zv)),  // voxel_layer.cpp:92 (VOXEL_BITS = 16)
        mark_threshold(mark_thr) {}
  void match_size(Costmap& cm) override {  // :97-102: the voxel grid starts all-unknown
    ObstacleLayer::match_size(cm);
    vox.assign(size_t(g.sx) * g.sy, 0x0000ffffu);
  }
  static bool bits_below_threshold(unsigned n, unsigned thr) {  // voxel_grid.h:160-174
    unsigned count = 0;
    for (; n;) {
      ++count;
      if (count > thr) return false;
      n &= n - 1;
    }
    return true;
  }
  bool w2m3f(double wx, double wy, double wz, double& mx, double& my, double& mz) const {  // voxel_layer.h:103-115
    if (wx < g.ox || wy < g.oy || wz < origin_z) return false;
    mx = (wx - g.ox) / g.res;
    my = (wy - g.oy) / g.res;
    mz = (wz - origin_z) / z_resolution;
    return mx < g.sx && my < g.sy && mz < size_z;
  }
  bool w2m3(double wx, double wy, double wz, unsigned& mx, unsigned& my, unsigned& mz) const {  // :117-130
    if (wx < g.ox || wy < g.oy || wz < origin_z) return false;
    mx = (int)((wx - g.ox) / g.res);
    my = (int)((wy - g.oy) / g.res);
    mz = (int)((wz - origin_z) / z_resolution);
    return mx < g.sx && my < g.sy && mz < size_z;
  }
  // VoxelGrid::clearVoxelLineInMap = raytraceLine + bresenham3D + ClearVoxelInMap (voxel_grid.h:226-297, 335-372)
  void clear_line(double x0, double y0, double z0, double x1, double y1, double z1, unsigned max_length) {
    if (x0 >= g.sx || y0 >= g.sy || z0 >= size_z || x1 >= g.sx || y1 >= g.sy || z1 >= size_z) return;  // voxel_grid.cpp:147-152
    int dx = int(x1) - int(x0), dy = int(y1) - int(y0), dz = int(z1) - int(z0);
    unsigned adx = abs(dx), ady = abs(dy), adz = abs(dz);
    int off_dx = dx > 0 ? 1 : -1, off_dy = (dy > 0 ? 1 : -1) * int(g.sx), off_dz = dz > 0 ? 1 : -1;
    unsigned z_mask = ((1u << 16) | 1u) << (unsigned)z0;
    unsigned offset = (unsigned)y0 * g.sx + (unsigned)x0;
    double dist = sqrt((x0 - x1) * (x0 - x1) + (y0 - y1) * (y0 - y1) + (z0 - z1) * (z0 - z1));
    double scale = std::min(1.0, max_length / dist);
    auto at = [&]() {
      uint32_t& col = vox[offset];
      col &= ~z_mask;
      unsigned unknown_bits = uint16_t(col >> 16) ^ uint16_t(col);
      unsigned marked_bits = col >> 16;
      if (bits_below_threshold(marked_bits, mark_threshold)) {
        g.c[offset] = bits_below_threshold(unknown_bits, unknown_threshold) ? kFree : kNoInfo;
      }
    };
    // axis kinds: 0 = grid offset (x or y), 1 = z mask
    auto step = [&](int kind, int off) {
      if (kind == 0) offset += off;
      else if (off > 0) z_mask <<= 1;
      else z_mask >>= 1;
    };
    auto bres = [&](int ka, int kb, int kc, unsigned da, unsigned db, unsigned dc, int err_b, int err_c, int oa, int ob,
                    int oc, unsigned max_len) {
      unsigned end = std::min(max_len, da);
      for (unsigned i = 0; i < end; ++i) {
        at();
        step(ka, oa);
        err_b += db;
        err_c += dc;
        if ((unsigned)err_b >= da) { step(kb, ob); err_b -= da; }
        if ((unsigned)err_c >= da) { step(kc, oc); err_c -= da; }
      }
      at();
    };
    if (adx >= std::max(ady, adz)) bres(0, 0, 1, adx, ady, adz, adx / 2, adx / 2, off_dx, off_dy, off_dz, (unsigned)(scale * adx));
    else if (ady >= adz) bres(0, 0, 1, ady, adx, adz, ady / 2, ady / 2, off_dy, off_dx, off_dz, (unsigned)(scale * ady));
    else bres(1, 0, 0, adz, adx, ady, adz / 2, adz / 2, off_dz, off_dx, off_dy, (unsigned)(scale * adz));
  }
  void raytrace_freespace_voxel(const Obs& o, Bounds& b) {  // voxel_layer.cpp:262-350
    if (o.xyz.empty()) return;
    double sensor_x, sensor_y, sensor_z;
    const double ox = o.ox, oy = o.oy, oz = o.oz;
    if (!w2m3f(ox, oy, oz, sensor_x, sensor_y, sensor_z)) return;
    const double map_end_x = g.ox + g.size_m_x(), map_end_y = g.oy + g.size_m_y();
    for (size_t i = 0; i < o.xyz.size() / 3; ++i) {
      double wpx = o.xyz[3 * i], wpy = o.xyz[3 * i + 1], wpz = o.xyz[3 * i + 2];
      double distance = sqrt((wpx - ox) * (wpx - ox) + (wpy - oy) * (wpy - oy) + (wpz - oz) * (wpz - oz));
      double scaling_fact = 1.0;
      scaling_fact = std::max(std::min(scaling_fact, (distance - 2 * g.res) / distance), 0.0);
      wpx = scaling_fact * (wpx - ox) + ox;
      wpy = scaling_fact * (wpy - oy) + oy;
      wpz = scaling_fact * (wpz - oz) + oz;
      double a = wpx - ox, bb = wpy - oy, c = wpz - oz, t = 1.0;
      if (wpz > max_obstacle_height) t = std::max(0.0, std::min(t, (max_obstacle_height - 0.01 - oz) / c));
      else if (wpz < origin_z) t = std::min(t, (origin_z - oz) / c);
      if (wpx < g.ox) t = std::min(t, (g.ox - ox) / a);
      if (wpy < g.oy) t = std::min(t, (g.oy - oy) / bb);
      if (wpx > map_end_x) t = std::min(t, (map_end_x - ox) / a);
      if (wpy > map_end_y) t = std::min(t, (map_end_y - oy) / bb);
      wpx = ox + a * t;
      wpy = oy + bb * t;
      wpz = oz + c * t;
      double px, py, pz;
      if (w2m3f(wpx, wpy, wpz, px, py, pz)) {
        clear_line(sensor_x, sensor_y, sensor_z, px, py, pz, g.cell_distance(o.raytrace_range));
        double dx = wpx - ox, dy = wpy - oy;  // updateRaytraceBounds, obstacle_layer.cpp:602-610
        double full = hypot(dx, dy);
        double scale = std::min(1.0, o.raytrace_range / full);
        touch(ox + dx * scale, oy + dy * scale, b);
      }
    }
  }
  void update_origin_voxel(double nox, double noy) {  // voxel_layer.cpp:371-438
    int cell_ox = int((nox - g.ox) / g.res), cell_oy = int((noy - g.oy) / g.res);
    int isx = g.sx, isy = g.sy;
    int llx = std::min(std::max(cell_ox, 0), isx), lly = std::min(std::max(cell_oy, 0), isy);
    int urx = std::min(std::max(cell_ox + isx, 0), isx), ury = std::min(std::max(cell_oy + isy, 0), isy);
    unsigned w = urx - llx, h = ury - lly;
    std::vector<uint32_t> keep(size_t(w) * h);
    for (unsigned r = 0; r < h; ++r) memcpy(keep.data() + size_t(r) * w, vox.data() + size_t(lly + r) * g.sx + llx, w * 4);
    g.update_origin(nox, noy);  // the 2-D part (copy, reset to default, copy back, origin)
    std::fill(vox.begin(), vox.end(), 0x0000ffffu);
    int start_x = llx - cell_ox, start_y = lly - cell_oy;
    for (unsigned r = 0; r < h; ++r) memcpy(vox.data() + size_t(start_y + r) * g.sx + start_x, keep.data() + size_t(r) * w, w * 4);
  }
  void update_bounds(Costmap& cm, double rx, double ry, double ryaw, Bounds& b) override {  // voxel_layer.cpp:116-177
    if (cm.rolling) update_origin_voxel(rx - g.size_m_x() / 2, ry - g.size_m_y() / 2);
    if (!enabled) return;
    for (const Obs& o : obs)
      if (o.clearing) raytrace_freespace_voxel(o, b);
    for (const Obs& o : obs) {
      if (!o.marking) continue;
      double sq_range = o.obstacle_range * o.obstacle_range;
      for (size_t i = 0; i < o.xyz.size() / 3; ++i) {
        const float fx = o.xyz[3 * i], fy = o.xyz[3 * i + 1], fz = o.xyz[3 * i + 2];
        if (fz > max_obstacle_height) continue;
        double sq = (fx - o.ox) * (fx - o.ox) + (fy - o.oy) * (fy - o.oy) + (fz - o.oz) * (fz - o.oz);
        if (sq >= sq_range) continue;
        unsigned mx, my, mz;
        if (fz < origin_z) {
          if (!w2m3(fx, fy, origin_z, mx, my, mz)) continue;
        } else if (!w2m3(fx, fy, fz, mx, my, mz)) {
          continue;
        }
        uint32_t& col = vox[size_t(my) * g.sx + mx];  // markVoxelInMap, voxel_grid.h:98-118
        col |= ((uint32_t)1 << mz << 16) | (1u << mz);
        if (!bits_below_threshold(col >> 16, mark_threshold)) {
          g.c[size_t(my) * g.sx + mx] = kLethal;
          touch((double)fx, (double)fy, b);
        }
      }
    }
    if (!footprint_clearing) return;
    transform_footprint(rx, ry, ryaw, cm.footprint, transformed_footprint);
    for (const Pt& p : transformed_footprint) touch(p.x, p.y, b);
  }
};

struct QCell {  // CellData, inflation_layer.h:55-85
  double distance;
  unsigned index, x, y, sx, sy;
};
struct QLess {
  bool operator()(const QCell& a, const QCell& b) const { return a.distance > b.distance; }
};

struct InflationLayer : LayerBase {  // inflation_layer.cpp
  double radius = 0.55, weight = 10.0, inscribed = 0, res = 0;
  unsigned R = 0;
  bool need_reinflation = false;
  double lminx = -std::numeric_limits<float>::max(), lminy = -std::numeric_limits<float>::max();
  double lmaxx = std::numeric_limits<float>::max(), lmaxy = std::numeric_limits<float>::max();
  std::vector<uint8_t> costs;  // (R+2)^2
  std::vector<double> dists;
  std::vector<uint8_t> seen;

  uint8_t compute_cost(double d) const {  // inflation_layer.h:114-129
    if (d == 0) return kLethal;
    if (d * res <= inscribed) return kInscribed;
    double factor = exp(-1.0 * weight * (d * res - inscribed));
    return (uint8_t)((kInscribed - 1) * factor);
  }
  void compute_caches() {  // :295-328
    if (R == 0) return;
    unsigned n = R + 2;
    costs.assign(n * n, 0);
    dists.assign(n * n, 0);
    for (unsigned i = 0; i < n; ++i)
      for (unsigned j = 0; j < n; ++j) {
        dists[i * n + j] = hypot(i, j);
        costs[i * n + j] = compute_cost(dists[i * n + j]);
      }
  }
  void set_params(Costmap& cm, double r, double w) {  // :356-370
    if (weight != w || radius != r) {
      radius = r;
      R = cm.master.cell_distance(radius);
      weight = w;
      need_reinflation = true;
      compute_caches();
    }
  }
  void match_size(Costmap& cm) override {  // :110-123
    res = cm.master.res;
    R = cm.master.cell_distance(radius);
    compute_caches();
    seen.assign(size_t(cm.master.sx) * cm.master.sy, 0);
  }
  void on_footprint_changed(Costmap& cm) override {  // :160-170
    inscribed = cm.inscribed;
    R = cm.master.cell_distance(radius);
    compute_caches();
    need_reinflation = true;
  }
  void update_bounds(Costmap&, double, double, double, Bounds& b) override {  // :125-158
    if (need_reinflation) {
      lminx = b.minx; lminy = b.miny; lmaxx = b.maxx; lmaxy = b.maxy;
      b.minx = -std::numeric_limits<float>::max();
      b.miny = -std::numeric_limits<float>::max();
      b.maxx = std::numeric_limits<float>::max();
      b.maxy = std::numeric_limits<float>::max();
      need_reinflation = false;
    } else {
      double tx0 = lminx, ty0 = lminy, tx1 = lmaxx, ty1 = lmaxy;
      lminx = b.minx; lminy = b.miny; lmaxx = b.maxx; lmaxy = b.maxy;
      b.minx = std::min(tx0, b.minx) - radius;
      b.miny = std::min(ty0, b.miny) - radius;
      b.maxx = std::max(tx1, b.maxx) + radius;
      b.maxy = std::max(ty1, b.maxy) + radius;
    }
  }
  // Tie-policy variants (checker-only; see oracle_api.h navo_inflation_set_variant).  0 = the reference as written.
  int variant = 0;
  uint64_t variant_seed = 0;
  int last_rounds = 0;  // rounds of the level-synchronous variant's last update_costs

  void write_cell(Grid& m, unsigned index, uint8_t cost) const {  // :249-254
    uint8_t old = m.c[index];
    if (old == kNoInfo && cost >= kInscribed) m.c[index] = cost;
    else m.c[index] = std::max(old, cost);
  }

  void update_costs(Costmap& cm, int min_i, int min_j, int max_i, int max_j) override {  // :172-266
    if (!enabled) return;
    // R == 0: compute_caches left the tables empty, and the reference would index them (undefined behaviour); an
    // inflation radius below one cell inflates nothing instead, as the CUDA library does
    if (R == 0) return;
    Grid& m = cm.master;
    unsigned size_x = m.sx, size_y = m.sy;
    if (seen.size() != size_t(size_x) * size_y) seen.resize(size_t(size_x) * size_y);
    std::fill(seen.begin(), seen.end(), 0);
    min_i -= R; min_j -= R; max_i += R; max_j += R;
    min_i = std::max(0, min_i);
    min_j = std::max(0, min_j);
    max_i = std::min(int(size_x), max_i);
    max_j = std::min(int(size_y), max_j);
    if (variant == 4) return update_costs_exact(m, min_i, min_j, max_i, max_j);
    if (variant == 5) return update_costs_level_sync(m, min_i, min_j, max_i, max_j, nullptr);
    if (variant == 6) {
      // certificate that variant 5 is a legal execution: run it on a scratch copy to learn which source every cell
      // ended up with, then run the reference's SEQUENTIAL priority-queue loop, breaking equal-distance ties in favour
      // of the entry that carries that source (oldest first otherwise).  The result must equal variant 5's.
      Grid scratch = m;
      hint.clear();
      update_costs_level_sync(scratch, min_i, min_j, max_i, max_j, &hint);
      std::fill(seen.begin(), seen.end(), 0);
    }
    if (variant != 0) return update_costs_tie_variant(m, min_i, min_j, max_i, max_j);
    std::priority_queue<QCell, std::vector<QCell>, QLess> q;
    const unsigned n = R + 2;
    auto enqueue = [&](unsigned index, unsigned mx, unsigned my, unsigned sx, unsigned sy) {  // :277-293
      if (seen[index]) return;
      unsigned dx = abs(int(mx) - int(sx)), dy = abs(int(my) - int(sy));
      double d = dists[dx * n + dy];
      if (d > R) return;
      q.push(QCell{d, index, mx, my, sx, sy});
    };
    for (int j = min_j; j < max_j; j++)
      for (int i = min_i; i < max_i; i++) {
        unsigned index = j * size_x + i;
        if (m.c[index] == kLethal) enqueue(index, i, j, i, j);
      }
    while (!q.empty()) {
      QCell cur = q.top();
      q.pop();
      if (seen[cur.index]) continue;
      seen[cur.index] = 1;
      unsigned dx = abs(int(cur.x) - int(cur.sx)), dy = abs(int(cur.y) - int(cur.sy));
      write_cell(m, cur.index, costs[dx * n + dy]);
      if (cur.x > 0) enqueue(cur.index - 1, cur.x - 1, cur.y, cur.sx, cur.sy);
      if (cur.y > 0) enqueue(cur.index - size_x, cur.x, cur.y - 1, cur.sx, cur.sy);
      if (cur.x < size_x - 1) enqueue(cur.index + 1, cur.x + 1, cur.y, cur.sx, cur.sy);
      if (cur.y < size_y - 1) enqueue(cur.index + size_x, cur.x, cur.y + 1, cur.sx, cur.sy);
    }
  }

  // The same algorithm (:172-293) with the one thing the reference leaves to libstdc++'s heap history made explicit:
  // which of several queue entries with EQUAL distance is popped first.  variant 1 = oldest first (FIFO), 2 = newest
  // first (LIFO), 3 = a seeded pseudo-random order.  Every variant is a legal execution of the reference's loop under
  // some heap implementation; cells whose value differs between variants are the "tie-variant mask".
  struct TCell {
    double distance;
    uint64_t tie;
    unsigned index, x, y, sx, sy;
  };
  struct TLess {
    bool operator()(const TCell& a, const TCell& b) const {
      return a.distance > b.distance || (a.distance == b.distance && a.tie > b.tie);
    }
  };
  static uint64_t mix64(uint64_t z) {  // splitmix64 finaliser
    z += 0x9e3779b97f4a7c15ull;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
  }
  void update_costs_tie_variant(Grid& m, int min_i, int min_j, int max_i, int max_j) {
    unsigned size_x = m.sx, size_y = m.sy;
    std::priority_queue<TCell, std::vector<TCell>, TLess> q;
    const unsigned n = R + 2;
    uint64_t seq = 0;
    auto enqueue = [&](unsigned index, unsigned mx, unsigned my, unsigned sx, unsigned sy) {
      if (seen[index]) return;
      unsigned dx = abs(int(mx) - int(sx)), dy = abs(int(my) - int(sy));
      double d = dists[dx * n + dy];
      if (d > R) return;
      uint64_t s = seq++;
      uint64_t tie = variant == 1 ? s : variant == 2 ? ~s : mix64(s ^ (variant_seed * 0x2545f4914f6cdd1dull));
      if (variant == 6) tie = s | (hint[index] == int32_t(sy * size_x + sx) ? 0 : (1ull << 63));
      q.push(TCell{d, tie, index, mx, my, sx, sy});
    };
    for (int j = min_j; j < max_j; j++)
      for (int i = min_i; i < max_i; i++) {
        unsigned index = j * size_x + i;
        if (m.c[index] == kLethal) enqueue(index, i, j, i, j);
      }
    while (!q.empty()) {
      TCell cur = q.top();
      q.pop();
      if (seen[cur.index]) continue;
      seen[cur.index] = 1;
      unsigned dx = abs(int(cur.x) - int(cur.sx)), dy = abs(int(cur.y) - int(cur.sy));
      write_cell(m, cur.index, costs[dx * n + dy]);
      if (cur.x > 0) enqueue(cur.index - 1, cur.x - 1, cur.y, cur.sx, cur.sy);
      if (cur.y > 0) enqueue(cur.index - size_x, cur.x, cur.y - 1, cur.sx, cur.sy);
      if (cur.x < size_x - 1) enqueue(cur.index + 1, cur.x + 1, cur.y, cur.sx, cur.sy);
      if (cur.y < size_y - 1) enqueue(cur.index + size_x, cur.x, cur.y + 1, cur.sx, cur.sy);
    }
  }

  // variant 4: exact windowed nearest-seed inflation -- every cell within cached distance <= R of a LETHAL cell of
  // the seed region gets the cached cost of its NEAREST seed (what an unobstructed propagation would deliver).  This is
  // the specification of the CUDA library's inflation mode 0.  Brute force; checker sizes only.
  void update_costs_exact(Grid& m, int min_i, int min_j, int max_i, int max_j) {
    const int size_x = m.sx, size_y = m.sy, r = R;
    const unsigned n = R + 2;
    std::vector<std::pair<int, int>> offs;
    for (int dy = -r; dy <= r; ++dy)
      for (int dx = -r; dx <= r; ++dx)
        if (!(dists[unsigned(abs(dx)) * n + unsigned(abs(dy))] > R)) offs.emplace_back(dx, dy);
    std::vector<uint8_t> best(size_t(size_x) * size_y, 0), hit(size_t(size_x) * size_y, 0);
    std::vector<double> bd(size_t(size_x) * size_y, 1e300);
    for (int j = min_j; j < max_j; j++)
      for (int i = min_i; i < max_i; i++) {
        if (m.c[size_t(j) * size_x + i] != kLethal) continue;
        for (auto& o : offs) {
          int x = i + o.first, y = j + o.second;
          if (x < 0 || y < 0 || x >= size_x || y >= size_y) continue;
          unsigned dx = abs(o.first), dy = abs(o.second);
          double d = dists[dx * n + dy];
          size_t idx = size_t(y) * size_x + x;
          if (d < bd[idx]) { bd[idx] = d; best[idx] = costs[dx * n + dy]; hit[idx] = 1; }
        }
      }
    for (size_t idx = 0; idx < hit.size(); ++idx)
      if (hit[idx]) write_cell(m, unsigned(idx), best[idx]);
  }

  // variant 5: level-synchronous nearest-source propagation -- the specification of the CUDA library's inflation
  // mode 1.  The reference's loop (:226-265) with one particular, order-independent choice among equal-distance queue
  // entries: per round, every unseen cell's best pending entry is the minimum cached distance over the sources carried
  // by its already-popped 4-neighbours (first of -x, -y, +x, +y on equal distance; an entry exists iff the neighbour
  // was popped while this cell was unseen and the distance gate :286-287 passed); the round pops ALL cells whose best
  // entry has the globally smallest distance.  Entries pushed by a pop never have the popped entry's own distance
  // (dx^2+dy^2 changes parity between 4-neighbours), so a round is a legal sequence of reference pops.
  std::vector<int32_t> hint;
  void update_costs_level_sync(Grid& m, int min_i, int min_j, int max_i, int max_j, std::vector<int32_t>* owner_out) {
    const int size_x = m.sx, size_y = m.sy;
    const unsigned n = R + 2;
    const size_t cells = size_t(size_x) * size_y;
    std::vector<int32_t> owner(cells, -1);
    std::vector<unsigned> frontier, next;  // unseen cells with at least one popped neighbour
    std::vector<uint8_t> in_frontier(cells, 0);
    auto push_frontier = [&](int x, int y) {
      if (x < 0 || y < 0 || x >= size_x || y >= size_y) return;
      size_t idx = size_t(y) * size_x + x;
      if (owner[idx] >= 0 || in_frontier[idx]) return;
      in_frontier[idx] = 1;
      frontier.push_back(unsigned(idx));
    };
    last_rounds = 0;
    std::vector<unsigned> popped;
    for (int j = min_j; j < max_j; j++)
      for (int i = min_i; i < max_i; i++) {
        unsigned index = j * size_x + i;
        if (m.c[index] == kLethal) { owner[index] = int32_t(index); popped.push_back(index); }
      }
    if (popped.empty()) {
      if (owner_out) owner_out->swap(owner);
      return;
    }
    for (unsigned index : popped) write_cell(m, index, costs[0]);
    last_rounds = 1;  // the seeds pop in the first round (distance 0), as the CUDA library counts rounds
    struct Best { double d; int32_t src; };
    auto best_entry = [&](unsigned idx) {
      int x = idx % size_x, y = idx / size_x;
      Best b{1e300, -1};
      const int nx[4] = {x - 1, x, x + 1, x}, ny[4] = {y, y - 1, y, y + 1};
      for (int k = 0; k < 4; ++k) {
        if (nx[k] < 0 || ny[k] < 0 || nx[k] >= size_x || ny[k] >= size_y) continue;
        int32_t s = owner[size_t(ny[k]) * size_x + nx[k]];
        if (s < 0) continue;
        unsigned dx = abs(x - int(s % size_x)), dy = abs(y - int(s / size_x));
        if (dx > R + 1 || dy > R + 1) continue;  // cannot happen (the neighbour is within R of s); table guard
        double d = dists[dx * n + dy];
        if (d > R) continue;
        if (d < b.d) { b.d = d; b.src = s; }
      }
      return b;
    };
    for (;;) {
      for (unsigned index : popped) {
        int x = index % size_x, y = index / size_x;
        push_frontier(x - 1, y); push_frontier(x, y - 1); push_frontier(x + 1, y); push_frontier(x, y + 1);
      }
      popped.clear();
      double kmin = 1e300;
      for (unsigned idx : frontier) kmin = std::min(kmin, best_entry(idx).d);
      if (kmin == 1e300) break;
      ++last_rounds;
      next.clear();
      std::vector<std::pair<unsigned, int32_t>> fin;
      for (unsigned idx : frontier) {
        Best b = best_entry(idx);
        if (b.d == kmin) fin.emplace_back(idx, b.src);
        else next.push_back(idx);
      }
      for (auto& f : fin) {
        owner[f.first] = f.second;
        in_frontier[f.first] = 0;
        popped.push_back(f.first);
        unsigned dx = abs(int(f.first % size_x) - int(f.second % size_x));
        unsigned dy = abs(int(f.first / size_x) - int(f.second / size_x));
        write_cell(m, f.first, costs[dx * n + dy]);
      }
      frontier.swap(next);
    }
    if (owner_out) owner_out->swap(owner);
  }
};

// ------------------------------------------------------------------ Path B
struct V3f { float v[3]; float& operator[](int i) { return v[i]; } const float& operator[](int i) const { return v[i]; } };

std::vector<double> velocity_samples(double mn, double mx, int n) {  // velocity_iterator.h:49-74
  std::vector<double> s;
  if (mn == mx) { s.push_back(mn); return s; }
  n = std::max(2, n);
  double step = (mx - mn) / double(std::max(1, n - 1));
  double cur, next = mn;
  for (int j = 0; j < n - 1; ++j) {
    cur = next;
    next += step;
    s.push_back(cur);
    if (cur < 0 && next > 0) s.push_back(0.0);
  }
  s.push_back(mx);
  return s;
}

struct Traj {
  double xv = 0, yv = 0, thv = 0, cost = -1;
  std::vector<double> x, y, th;
};

struct LineIt {  // line_iterator.h:38-139
  int x, y, dx, dy, cur = 0, xinc1, xinc2, yinc1, yinc2, den, num, numadd, numpixels;
  LineIt(int x0, int y0, int x1, int y1) : x(x0), y(y0), dx(abs(x1 - x0)), dy(abs(y1 - y0)) {
    xinc1 = xinc2 = (x1 >= x0) ? 1 : -1;
    yinc1 = yinc2 = (y1 >= y0) ? 1 : -1;
    if (dx >= dy) { xinc1 = 0; yinc2 = 0; den = dx; num = dx / 2; numadd = dy; numpixels = dx; }
    else { xinc2 = 0; yinc1 = 0; den = dy; num = dy / 2; numadd = dx; numpixels = dy; }
  }
  bool valid() const { return cur <= numpixels; }
  void advance() {
    num += numadd;
    if (num >= den) { num -= den; x += xinc1; y += yinc1; }
    x += xinc2;
    y += yinc2;
    cur++;
  }
};

// MapGrid::computeTargetDistance (map_grid.cpp:258-310) over explicit seeds; dist pre-filled with "unreachable".
void mapgrid_bfs(const Grid& cm, bool allow_unknown, std::vector<double>& dist, std::vector<uint8_t>& mark,
                 std::queue<unsigned>& q, const std::vector<uint8_t>* within_robot = nullptr) {
  const unsigned sx = cm.sx, sy = cm.sy;
  const double obstacle = double(size_t(sx) * sy);
  auto visit = [&](unsigned cur, unsigned chk) {
    if (mark[chk]) return;
    mark[chk] = 1;
    uint8_t cost = cm.c[chk];  // updatePathCell :103-123
    if (!(within_robot && (*within_robot)[chk]) &&
        (cost == kLethal || cost == kInscribed || (cost == kNoInfo && !allow_unknown))) {
      dist[chk] = obstacle;
      return;
    }
    double nd = dist[cur] + 1;
    if (nd < dist[chk]) dist[chk] = nd;
    q.push(chk);
  };
  while (!q.empty()) {
    unsigned cur = q.front();
    q.pop();
    unsigned cx = cur % sx, cy = cur / sx;
    if (cx > 0) visit(cur, cur - 1);
    if (cx < sx - 1) visit(cur, cur + 1);
    if (cy > 0) visit(cur, cur - sx);
    if (cy < sy - 1) visit(cur, cur + sx);
  }
}

void adjust_plan_resolution(const std::vector<Pt>& in, std::vector<Pt>& out, double resolution) {  // map_grid.cpp:135-171
  if (in.empty()) return;
  double last_x = in[0].x, last_y = in[0].y;
  out.push_back(in[0]);
  double min_sq = resolution * resolution * 4;
  for (size_t i = 1; i < in.size(); ++i) {
    double lx = in[i].x, ly = in[i].y;
    double sq = (lx - last_x) * (lx - last_x) + (ly - last_y) * (ly - last_y);
    if (sq > min_sq) {
      int steps = ((sqrt(sq) - sqrt(min_sq)) / resolution) - 1;
      double ddx = (lx - last_x) / steps, ddy = (ly - last_y) / steps;
      for (int j = 1; j < steps; ++j) out.push_back(Pt{last_x + j * ddx, last_y + j * ddy});
    }
    out.push_back(in[i]);
    last_x = lx;
    last_y = ly;
  }
}

struct MapGridCritic {  // MapGridCostFunction + MapGrid
  bool local_goal = false, stop_on_failure = true;
  double xshift = 0, scale = 1;
  std::vector<Pt> target;
  std::vector<double> dist;

  void prepare(const Grid& cm, bool allow_unknown) {  // map_grid_cost_function.cpp:59-68, map_grid.cpp:127-254
    size_t n = size_t(cm.sx) * cm.sy;
    dist.assign(n, double(n + 1));
    std::vector<uint8_t> mark(n, 0);
    std::queue<unsigned> q;
    std::vector<Pt> adj;
    adjust_plan_resolution(target, adj, cm.res);
    bool started = false;
    int gx = -1, gy = -1;
    for (size_t i = 0; i < adj.size(); ++i) {
      unsigned mx, my;
      if (cm.world_to_map(adj[i].x, adj[i].y, mx, my) && cm.c[size_t(my) * cm.sx + mx] != kNoInfo) {
        if (local_goal) { gx = mx; gy = my; }
        else {
          unsigned id = my * cm.sx + mx;
          dist[id] = 0.0;
          mark[id] = 1;
          q.push(id);
        }
        started = true;
      } else if (started) {
        break;
      }
    }
    if (!started) return;
    if (local_goal && gx >= 0 && gy >= 0) {
      unsigned id = gy * cm.sx + gx;
      dist[id] = 0.0;
      mark[id] = 1;
      q.push(id);
    }
    mapgrid_bfs(cm, allow_unknown, dist, mark, q);
  }

  double score(const Grid& cm, const Traj& t) const {  // map_grid_cost_function.cpp:75-129 (aggregation Last)
    double cost = 0.0;
    const double n = double(dist.size());
    for (size_t i = 0; i < t.x.size(); ++i) {
      double px = t.x[i], py = t.y[i], pth = t.th[i];
      if (xshift != 0.0) {
        px = px + xshift * cos(pth);
        py = py + xshift * sin(pth);
      }
      unsigned cx, cy;
      if (!cm.world_to_map(px, py, cx, cy)) return -4.0;
      double d = dist[size_t(cy) * cm.sx + cx];
      if (stop_on_failure) {
        if (d == n) return -3.0;
        if (d == n + 1) return -2.0;
      }
      cost = d;
    }
    return cost;
  }
};

struct Dwa {
  navo_dwa_config cfg;
  Grid cm;
  std::vector<Pt> plan;
  MapGridCritic path, goal, goal_front, alignment;
  double obstacle_scale = 0;
  // oscillation state (oscillation_cost_function.h:78-83)
  bool strafe_pos_only = false, strafe_neg_only = false, strafing_pos = false, strafing_neg = false;
  bool rot_pos_only = false, rot_neg_only = false, rotating_pos = false, rotating_neg = false;
  bool forward_pos_only = false, forward_neg_only = false, forward_pos = false, forward_neg = false;
  V3f prev_stationary{{0, 0, 0}};
  std::vector<Pt> footprint;
  Traj result;

  void reconfigure() {  // dwa_planner.cpp:52-112, ctor :116-182
    double r = cm.res;
    path.scale = alignment.scale = r * cfg.path_distance_bias * 0.5;
    goal.scale = goal_front.scale = r * cfg.goal_distance_bias * 0.5;
    obstacle_scale = r * cfg.occdist_scale;
    goal.local_goal = goal_front.local_goal = true;
    goal_front.stop_on_failure = alignment.stop_on_failure = false;
    goal_front.xshift = alignment.xshift = cfg.forward_point_distance;
  }
  void reset_osc() {  // oscillation_cost_function.cpp:84-99
    strafe_pos_only = strafe_neg_only = strafing_pos = strafing_neg = false;
    rot_pos_only = rot_neg_only = rotating_pos = rotating_neg = false;
    forward_pos_only = forward_neg_only = forward_pos = forward_neg = false;
  }
  double osc_score(const Traj& t) const {  // :166-176
    if ((forward_pos_only && t.xv < 0.0) || (forward_neg_only && t.xv > 0.0) || (strafe_pos_only && t.yv < 0.0) ||
        (strafe_neg_only && t.yv > 0.0) || (rot_pos_only && t.thv < 0.0) || (rot_neg_only && t.thv > 0.0))
      return -5.0;
    return 0.0;
  }
  bool set_osc_flags(const Traj& t, double min_vel_trans) {  // :101-164
    bool flag_set = false;
    if (t.xv < 0.0) { if (forward_pos) { forward_neg_only = true; flag_set = true; } forward_pos = false; forward_neg = true; }
    if (t.xv > 0.0) { if (forward_neg) { forward_pos_only = true; flag_set = true; } forward_neg = false; forward_pos = true; }
    if (fabs(t.xv) <= min_vel_trans) {
      if (t.yv < 0) { if (strafing_pos) { strafe_neg_only = true; flag_set = true; } strafing_pos = false; strafing_neg = true; }
      if (t.yv > 0) { if (strafing_neg) { strafe_pos_only = true; flag_set = true; } strafing_neg = false; strafing_pos = true; }
      if (t.thv < 0) { if (rotating_pos) { rot_neg_only = true; flag_set = true; } rotating_pos = false; rotating_neg = true; }
      if (t.thv > 0) { if (rotating_neg) { rot_pos_only = true; flag_set = true; } rotating_neg = false; rotating_pos = true; }
    }
    return flag_set;
  }
  void update_osc_flags(const V3f& pos, const Traj& t, double min_vel_trans) {  // :56-82
    if (t.cost < 0) return;
    if (set_osc_flags(t, min_vel_trans)) prev_stationary = pos;
    if (forward_pos_only || forward_neg_only || strafe_pos_only || strafe_neg_only || rot_pos_only || rot_neg_only) {
      double xd = pos[0] - prev_stationary[0], yd = pos[1] - prev_stationary[1];
      double sq = xd * xd + yd * yd;
      double thd = pos[2] - prev_stationary[2];
      if (sq > cfg.oscillation_reset_dist * cfg.oscillation_reset_dist || fabs(thd) > cfg.oscillation_reset_angle) reset_osc();
    }
  }

  // SimpleTrajectoryGenerator::initialise, simple_trajectory_generator.cpp:60-135
  void enumerate_samples(const V3f& pos, const V3f& vel, const V3f& goal, std::vector<V3f>& out) const {
    double max_vel_th = cfg.max_rot_vel, min_vel_th = -1.0 * max_vel_th;
    V3f acc{{float(cfg.acc_lim_x), float(cfg.acc_lim_y), float(cfg.acc_lim_theta)}};
    double min_vel_x = cfg.min_vel_x, max_vel_x = cfg.max_vel_x, min_vel_y = cfg.min_vel_y, max_vel_y = cfg.max_vel_y;
    int nx = std::max(1, cfg.vx_samples), ny = std::max(1, cfg.vy_samples), nth = std::max(1, cfg.vth_samples);
    V3f mx{{0, 0, 0}}, mn{{0, 0, 0}};
    if (!cfg.use_dwa) {
      double dist = hypot(goal[0] - pos[0], goal[1] - pos[1]);
      max_vel_x = std::max(std::min(max_vel_x, dist / cfg.sim_time), min_vel_x);
      max_vel_y = std::max(std::min(max_vel_y, dist / cfg.sim_time), min_vel_y);
      mx[0] = std::min(max_vel_x, vel[0] + acc[0] * cfg.sim_time);
      mx[1] = std::min(max_vel_y, vel[1] + acc[1] * cfg.sim_time);
      mx[2] = std::min(max_vel_th, vel[2] + acc[2] * cfg.sim_time);
      mn[0] = std::max(min_vel_x, vel[0] - acc[0] * cfg.sim_time);
      mn[1] = std::max(min_vel_y, vel[1] - acc[1] * cfg.sim_time);
      mn[2] = std::max(min_vel_th, vel[2] - acc[2] * cfg.sim_time);
    } else {
      mx[0] = std::min(max_vel_x, vel[0] + acc[0] * cfg.sim_period);
      mx[1] = std::min(max_vel_y, vel[1] + acc[1] * cfg.sim_period);
      mx[2] = std::min(max_vel_th, vel[2] + acc[2] * cfg.sim_period);
      mn[0] = std::max(min_vel_x, vel[0] - acc[0] * cfg.sim_period);
      mn[1] = std::max(min_vel_y, vel[1] - acc[1] * cfg.sim_period);
      mn[2] = std::max(min_vel_th, vel[2] - acc[2] * cfg.sim_period);
    }
    std::vector<double> xs = velocity_samples(mn[0], mx[0], nx), ys = velocity_samples(mn[1], mx[1], ny),
                        ths = velocity_samples(mn[2], mx[2], nth);
    for (double a : xs)
      for (double b : ys)
        for (double c : ths) out.push_back(V3f{{float(a), float(b), float(c)}});
  }

  // generateTrajectory, simple_trajectory_generator.cpp:180-251 (+ computeNewPositions/Velocities :253-276)
  bool generate(V3f pos, const V3f& vel, const V3f& s, Traj& t) const {
    double vmag = hypot(s[0], s[1]);
    const double eps = 1e-4;
    t.cost = -1.0;
    t.x.clear(); t.y.clear(); t.th.clear();
    if ((cfg.min_trans_vel >= 0 && vmag + eps < cfg.min_trans_vel) && (cfg.min_rot_vel >= 0 && fabs(s[2]) + eps < cfg.min_rot_vel))
      return false;
    if (cfg.max_trans_vel >= 0 && vmag - eps > cfg.max_trans_vel) return false;
    double sim_time_distance = vmag * cfg.sim_time;
    double sim_time_angle = fabs(s[2]) * cfg.sim_time;
    int num_steps = ceil(std::max(sim_time_distance / cfg.sim_granularity, sim_time_angle / cfg.angular_sim_granularity));
    double dt = cfg.sim_time / num_steps;
    V3f acc{{float(cfg.acc_lim_x), float(cfg.acc_lim_y), float(cfg.acc_lim_theta)}};
    auto new_vel = [&](const V3f& v) {
      V3f nv{{0, 0, 0}};
      for (int i = 0; i < 3; ++i) {
        if (v[i] < s[i]) nv[i] = std::min(double(s[i]), v[i] + acc[i] * dt);
        else nv[i] = std::max(double(s[i]), v[i] - acc[i] * dt);
      }
      return nv;
    };
    V3f loop_vel;
    const bool continued = !cfg.use_dwa;
    if (continued) loop_vel = new_vel(vel);
    else loop_vel = s;
    t.xv = loop_vel[0]; t.yv = loop_vel[1]; t.thv = loop_vel[2];
    for (int i = 0; i < num_steps; ++i) {
      t.x.push_back(pos[0]); t.y.push_back(pos[1]); t.th.push_back(pos[2]);
      if (continued) loop_vel = new_vel(loop_vel);
      V3f np;
      np[0] = pos[0] + (loop_vel[0] * cos(double(pos[2])) + loop_vel[1] * cos(M_PI_2 + pos[2])) * dt;
      np[1] = pos[1] + (loop_vel[0] * sin(double(pos[2])) + loop_vel[1] * sin(M_PI_2 + pos[2])) * dt;
      np[2] = pos[2] + loop_vel[2] * dt;
      pos = np;
    }
    return num_steps > 0;
  }

  // CostmapModel::pointCost / lineCost / footprintCost (costmap_model.cpp:50-142) + WorldModel wrapper (world_model.h:65-86)
  double footprint_cost(double x, double y, double th) const {
    const bool allow_unknown = cfg.allow_unknown != 0;
    double c = cos(th), s = sin(th);
    unsigned cx, cy;
    if (!cm.world_to_map(x, y, cx, cy)) return -1.0;
    if (footprint.size() < 3) {
      uint8_t cost = cm.c[size_t(cy) * cm.sx + cx];
      if (cost == kLethal || cost == kInscribed || (cost == kNoInfo && !allow_unknown)) return -1.0;
      return cost;
    }
    double fcost = 0.0;
    const size_t n = footprint.size();
    for (size_t i = 0; i < n; ++i) {
      const Pt& a = footprint[i];
      const Pt& b = footprint[(i + 1) % n];
      double ax = x + (a.x * c - a.y * s), ay = y + (a.x * s + a.y * c);
      double bx = x + (b.x * c - b.y * s), by = y + (b.x * s + b.y * c);
      unsigned x0, y0, x1, y1;
      if (!cm.world_to_map(ax, ay, x0, y0)) return -1.0;
      if (!cm.world_to_map(bx, by, x1, y1)) return -1.0;
      double line_cost = 0.0;
      for (LineIt l(x0, y0, x1, y1); l.valid(); l.advance()) {
        uint8_t cost = cm.c[size_t(l.y) * cm.sx + l.x];
        if (cost == kLethal || (cost == kNoInfo && !allow_unknown)) return -1.0;
        if (line_cost < cost) line_cost = cost;
      }
      fcost = std::max(line_cost, fcost);
    }
    return fcost;
  }
  double obstacle_score(const Traj& t) const {  // obstacle_cost_function.cpp:74-142
    double cost = 0;
    if (footprint.empty()) return -9;
    for (size_t i = 0; i < t.x.size(); ++i) {
      double f = footprint_cost(t.x[i], t.y[i], t.th[i]);
      if (f < 0) return -6.0;
      unsigned cx, cy;
      if (!cm.world_to_map(t.x[i], t.y[i], cx, cy)) return -7.0;
      double occ = std::max(std::max(0.0, f), double(cm.c[size_t(cy) * cm.sx + cx]));
      if (cfg.sum_scores) cost += occ;
      else cost = occ;
    }
    return cost;
  }

  // SimpleScoredSamplingPlanner::scoreTrajectory, simple_scored_sampling_planner.cpp:50-79
  double score(const Traj& t, double best) const {
    double total = 0;
    for (int k = 0; k < 6; ++k) {
      double scale, cost;
      switch (k) {  // critic order dwa_planner.cpp:167-173
        case 0: scale = 1.0; break;  // OscillationCostFunction keeps TrajectoryCostFunction's default scale 1.0
        case 1: scale = obstacle_scale; break;
        case 2: scale = goal_front.scale; break;
        case 3: scale = alignment.scale; break;
        case 4: scale = path.scale; break;
        default: scale = goal.scale; break;
      }
      if (scale == 0) continue;
      switch (k) {
        case 0: cost = osc_score(t); break;
        case 1: cost = obstacle_score(t); break;
        case 2: cost = goal_front.score(cm, t); break;
        case 3: cost = alignment.score(cm, t); break;
        case 4: cost = path.score(cm, t); break;
        default: cost = goal.score(cm, t); break;
      }
      if (cost < 0) { total = cost; break; }
      if (cost != 0) cost *= scale;
      total += cost;
      if (best > 0 && total > best) break;
    }
    return total;
  }

  void prepare_all() {
    const bool au = cfg.allow_unknown != 0;
    goal_front.prepare(cm, au);
    alignment.prepare(cm, au);
    path.prepare(cm, au);
    goal.prepare(cm, au);
  }
};

std::vector<Pt> to_pts(const double* xy, int n) {
  std::vector<Pt> v(n);
  for (int i = 0; i < n; ++i) v[i] = Pt{xy[2 * i], xy[2 * i + 1]};
  return v;
}

// ---------------------------------------------------------------------------------------------------------------
// Legacy base_local_planner::TrajectoryPlanner (base_local_planner/src/trajectory_planner.cpp), restated.
struct Tp {
  navo_tp_config cfg;
  Grid cm;
  std::vector<Pt> footprint, plan;
  std::vector<double> path_dist, goal_dist;  // path_map_ / goal_map_ target_dist
  bool stuck_left = false, stuck_right = false, stuck_left_strafe = false, stuck_right_strafe = false;
  bool rotating_left = false, rotating_right = false, strafe_left = false, strafe_right = false;
  bool escaping = false, final_goal_valid = false;
  double prev_x = 0, prev_y = 0, escape_x = 0, escape_y = 0, escape_theta = 0, final_goal_x = 0, final_goal_y = 0;

  struct Result {
    double cost = -1.0, xv = 0, yv = 0, thetav = 0;
    std::vector<double> x, y, th;
  };

  // CostmapModel::footprintCost through WorldModel::footprintCost (world_model.h:65-86, costmap_model.cpp:50-142)
  double footprint_cost(double x, double y, double th) const {
    const bool allow_unknown = cfg.allow_unknown != 0;
    const double c = cos(th), s = sin(th);
    unsigned cx, cy;
    if (!cm.world_to_map(x, y, cx, cy)) return -1.0;
    if (footprint.size() < 3) {
      const uint8_t cost = cm.c[size_t(cy) * cm.sx + cx];
      if (cost == kLethal || cost == kInscribed || (cost == kNoInfo && !allow_unknown)) return -1.0;
      return cost;
    }
    double fcost = 0.0;
    const size_t n = footprint.size();
    for (size_t i = 0; i < n; ++i) {
      const Pt& a = footprint[i];
      const Pt& b = footprint[(i + 1) % n];
      unsigned x0, y0, x1, y1;
      if (!cm.world_to_map(x + (a.x * c - a.y * s), y + (a.x * s + a.y * c), x0, y0)) return -1.0;
      if (!cm.world_to_map(x + (b.x * c - b.y * s), y + (b.x * s + b.y * c), x1, y1)) return -1.0;
      double line_cost = 0.0;
      for (LineIt l(x0, y0, x1, y1); l.valid(); l.advance()) {
        const uint8_t cost = cm.c[size_t(l.y) * cm.sx + l.x];
        if (cost == kLethal || (cost == kNoInfo && !allow_unknown)) return -1.0;
        if (line_cost < cost) line_cost = cost;
      }
      fcost = std::max(line_cost, fcost);
    }
    return fcost;
  }

  // lineCost / pointCost (:389-475): true when no cell of the Bresenham line is LETHAL / INSCRIBED / disallowed unknown
  bool line_clear(int x0, int x1, int y0, int y1) const {
    const int dx = abs(x1 - x0), dy = abs(y1 - y0);
    const int xi = x1 >= x0 ? 1 : -1, yi = y1 >= y0 ? 1 : -1;
    const bool xmajor = dx >= dy;
    const int den = xmajor ? dx : dy, numadd = xmajor ? dy : dx;
    int num = den / 2, x = x0, y = y0;
    for (int k = 0; k <= den; ++k) {
      const uint8_t c = cm.c[size_t(y) * cm.sx + x];
      if (c == kLethal || c == kInscribed || (c == kNoInfo && !cfg.allow_unknown)) return false;
      num += numadd;
      if (num >= den) {
        num -= den;
        if (xmajor) y += yi; else x += xi;
      }
      if (xmajor) x += xi; else y += yi;
    }
    return true;
  }

  double heading_diff(int cell_x, int cell_y, double x, double y, double heading) const {  // :372-387
    for (int i = (int)plan.size() - 1; i >= 0; --i) {
      unsigned gx, gy;
      if (cm.world_to_map(plan[i].x, plan[i].y, gx, gy) && line_clear(cell_x, (int)gx, cell_y, (int)gy)) {
        double wx, wy;
        cm.map_to_world(gx, gy, wx, wy);
        double a = fmod(fmod(atan2(wy - y, wx - x) - heading, 2.0 * M_PI) + 2.0 * M_PI, 2.0 * M_PI);  // angles.h
        if (a > M_PI) a -= 2.0 * M_PI;
        return fabs(a);
      }
    }
    return DBL_MAX;
  }

  static double new_velocity(double vg, double vi, double a_max, double dt) {  // trajectory_planner.h:369-375
    if ((vg - vi) >= 0) return std::min(vg, vi + a_max * dt);
    return std::max(vg, vi - a_max * dt);
  }

  // generateTrajectory (:214-370)
  void generate(double x, double y, double theta, double vx, double vy, double vtheta, double vx_samp, double vy_samp,
                double vtheta_samp, double acc_x, double acc_y, double acc_theta, double impossible_cost, Result& t) const {
    double x_i = x, y_i = y, theta_i = theta, vx_i = vx, vy_i = vy, vtheta_i = vtheta;
    const double vmag = hypot(vx_samp, vy_samp);
    int num_steps;
    if (!cfg.heading_scoring)
      num_steps = int(std::max((vmag * cfg.sim_time) / cfg.sim_granularity, fabs(vtheta_samp) / cfg.angular_sim_granularity) + 0.5);
    else
      num_steps = int(cfg.sim_time / cfg.sim_granularity + 0.5);
    if (num_steps == 0) num_steps = 1;
    const double dt = cfg.sim_time / num_steps;
    double time = 0.0;
    t.x.clear(); t.y.clear(); t.th.clear();
    t.xv = vx_samp; t.yv = vy_samp; t.thetav = vtheta_samp;
    t.cost = -1.0;
    double path_d = 0.0, goal_d = 0.0, occ_cost = 0.0, hdiff = 0.0;
    for (int i = 0; i < num_steps; ++i) {
      unsigned cell_x, cell_y;
      if (!cm.world_to_map(x_i, y_i, cell_x, cell_y)) { t.cost = -1.0; return; }
      const double fc = footprint_cost(x_i, y_i, theta_i);
      if (fc < 0) { t.cost = -1.0; return; }
      occ_cost = std::max(std::max(occ_cost, fc), double(cm.c[size_t(cell_y) * cm.sx + cell_x]));
      if (cfg.simple_attractor) {
        goal_d = (x_i - plan.back().x) * (x_i - plan.back().x) + (y_i - plan.back().y) * (y_i - plan.back().y);
      } else {
        bool update = true;
        if (cfg.heading_scoring) {
          if (time >= cfg.heading_scoring_timestep && time < cfg.heading_scoring_timestep + dt)
            hdiff = heading_diff((int)cell_x, (int)cell_y, x_i, y_i, theta_i);
          else
            update = false;
        }
        if (update) {
          path_d = path_dist[size_t(cell_y) * cm.sx + cell_x];
          goal_d = goal_dist[size_t(cell_y) * cm.sx + cell_x];
          if (impossible_cost <= goal_d || impossible_cost <= path_d) { t.cost = -2.0; return; }
        }
      }
      t.x.push_back(x_i); t.y.push_back(y_i); t.th.push_back(theta_i);
      vx_i = new_velocity(vx_samp, vx_i, acc_x, dt);
      vy_i = new_velocity(vy_samp, vy_i, acc_y, dt);
      vtheta_i = new_velocity(vtheta_samp, vtheta_i, acc_theta, dt);
      const double nx = x_i + (vx_i * cos(theta_i) + vy_i * cos(M_PI_2 + theta_i)) * dt;  // trajectory_planner.h:332-358
      const double ny = y_i + (vx_i * sin(theta_i) + vy_i * sin(M_PI_2 + theta_i)) * dt;
      theta_i = theta_i + vtheta_i * dt;
      x_i = nx; y_i = ny;
      time += dt;
    }
    if (!cfg.heading_scoring) t.cost = cfg.pdist_scale * path_d + goal_d * cfg.gdist_scale + cfg.occdist_scale * occ_cost;
    else t.cost = cfg.occdist_scale * occ_cost + cfg.pdist_scale * path_d + 0.3 * hdiff + goal_d * cfg.gdist_scale;
  }

  // FootprintHelper::getFootprintCells(pos, spec, costmap, fill = true) (footprint_helper.cpp:51-246)
  std::vector<std::pair<long long, long long>> footprint_cells(double x_i, double y_i, double theta_i) const {
    std::vector<std::pair<long long, long long>> cells;
    if (footprint.size() <= 1) {
      unsigned mx, my;
      if (cm.world_to_map(x_i, y_i, mx, my)) cells.push_back({mx, my});
      return cells;
    }
    const double cos_th = cos(theta_i), sin_th = sin(theta_i);
    auto line = [&](int x0, int x1, int y0, int y1) {  // getLineCells :51-120
      const int dx = abs(x1 - x0), dy = abs(y1 - y0), xi = x1 >= x0 ? 1 : -1, yi = y1 >= y0 ? 1 : -1;
      const bool xmajor = dx >= dy;
      const int den = xmajor ? dx : dy, numadd = xmajor ? dy : dx;
      int num = den / 2, x = x0, y = y0;
      for (int k = 0; k <= den; ++k) {
        cells.push_back({x, y});
        num += numadd;
        if (num >= den) { num -= den; if (xmajor) y += yi; else x += xi; }
        if (xmajor) x += xi; else y += yi;
      }
    };
    const size_t n = footprint.size();
    for (size_t i = 0; i < n; ++i) {
      const Pt& p = footprint[i];
      const Pt& q = footprint[(i + 1) % n];
      unsigned x0, y0, x1, y1;
      if (!cm.world_to_map(x_i + (p.x * cos_th - p.y * sin_th), y_i + (p.x * sin_th + p.y * cos_th), x0, y0)) return cells;
      if (!cm.world_to_map(x_i + (q.x * cos_th - q.y * sin_th), y_i + (q.x * sin_th + q.y * cos_th), x1, y1)) return cells;
      line((int)x0, (int)x1, (int)y0, (int)y1);
    }
    // getFillCells :123-178: the swap-adjacent sort (stable by x), then the column walk over the growing vector
    size_t i = 0;
    while (i + 1 < cells.size()) {
      if (cells[i].first > cells[i + 1].first) {
        std::swap(cells[i], cells[i + 1]);
        if (i > 0) --i;
      } else {
        ++i;
      }
    }
    i = 0;
    const unsigned min_x = (unsigned)cells.front().first, max_x = (unsigned)cells.back().first;
    for (unsigned x = min_x; x <= max_x; ++x) {
      if (i >= cells.size() - 1) break;
      std::pair<long long, long long> lo, hi;
      if (cells[i].second < cells[i + 1].second) { lo = cells[i]; hi = cells[i + 1]; }
      else { lo = cells[i + 1]; hi = cells[i]; }
      i += 2;
      while (i < cells.size() && cells[i].first == (long long)x) {
        if (cells[i].second < lo.second) lo = cells[i];
        else if (cells[i].second > hi.second) hi = cells[i];
        ++i;
      }
      for (unsigned yy = (unsigned)lo.second; yy < (unsigned)hi.second; ++yy) cells.push_back({(long long)x, (long long)yy});
    }
    return cells;
  }

  // MapGrid::setTargetCells / setLocalGoal (map_grid.cpp:174-254) into `dist`
  void wavefront(bool local_goal, const std::vector<uint8_t>* within, std::vector<double>& dist) const {
    const size_t n = size_t(cm.sx) * cm.sy;
    dist.assign(n, double(n + 1));
    std::vector<uint8_t> mark(n, 0);
    std::queue<unsigned> q;
    std::vector<Pt> adj;
    adjust_plan_resolution(plan, adj, cm.res);
    bool started = false;
    int gx = -1, gy = -1;
    for (size_t i = 0; i < adj.size(); ++i) {
      unsigned mx, my;
      if (cm.world_to_map(adj[i].x, adj[i].y, mx, my) && cm.c[size_t(my) * cm.sx + mx] != kNoInfo) {
        if (local_goal) { gx = mx; gy = my; }
        else {
          const unsigned id = my * cm.sx + mx;
          dist[id] = 0.0;
          mark[id] = 1;
          q.push(id);
        }
        started = true;
      } else if (started) {
        break;
      }
    }
    if (!started) return;
    if (local_goal && gx >= 0 && gy >= 0) {
      const unsigned id = gy * cm.sx + gx;
      dist[id] = 0.0;
      mark[id] = 1;
      q.push(id);
    }
    mapgrid_bfs(cm, cfg.allow_unknown != 0, dist, mark, q, within);
  }

  // createTrajectories (:537-905)
  Result create(double x, double y, double theta, double vx, double vy, double vtheta) {
    const double acc_x = cfg.acc_lim_x, acc_y = cfg.acc_lim_y, acc_theta = cfg.acc_lim_theta;
    double max_vel_x = cfg.max_vel_x, max_vel_theta, min_vel_x, min_vel_theta;
    if (final_goal_valid) max_vel_x = std::min(max_vel_x, hypot(final_goal_x - x, final_goal_y - y) / cfg.sim_time);
    const double horizon = cfg.dwa ? cfg.sim_period : cfg.sim_time;
    max_vel_x = std::max(std::min(max_vel_x, vx + acc_x * horizon), cfg.min_vel_x);
    min_vel_x = std::max(cfg.min_vel_x, vx - acc_x * horizon);
    max_vel_theta = std::min(cfg.max_vel_th, vtheta + acc_theta * horizon);
    min_vel_theta = std::max(cfg.min_vel_th, vtheta - acc_theta * horizon);
    const double dvx = (max_vel_x - min_vel_x) / (cfg.vx_samples - 1);
    const double dvtheta = (max_vel_theta - min_vel_theta) / (cfg.vtheta_samples - 1);
    double vx_samp = min_vel_x, vtheta_samp = min_vel_theta, vy_samp = 0.0;
    Result one, two;
    Result* best = &one;
    Result* comp = &two;
    best->cost = -1.0;
    comp->cost = -1.0;
    const double impossible = double(size_t(cm.sx) * cm.sy);
    auto gen = [&](double a, double b, double c) { generate(x, y, theta, vx, vy, vtheta, a, b, c, acc_x, acc_y, acc_theta, impossible, *comp); };
    auto better = [&]() { return comp->cost >= 0 && (comp->cost < best->cost || best->cost < 0); };
    if (!escaping) {
      for (int i = 0; i < cfg.vx_samples; ++i) {
        vtheta_samp = 0;
        gen(vx_samp, vy_samp, vtheta_samp);
        if (better()) std::swap(best, comp);
        vtheta_samp = min_vel_theta;
        for (int j = 0; j < cfg.vtheta_samples - 1; ++j) {
          gen(vx_samp, vy_samp, vtheta_samp);
          if (better()) std::swap(best, comp);
          vtheta_samp += dvtheta;
        }
        vx_samp += dvx;
      }
      if (cfg.holonomic_robot) {
        gen(0.1, 0.1, 0.0);
        if (better()) std::swap(best, comp);
        gen(0.1, -0.1, 0.0);
        if (better()) std::swap(best, comp);
      }
    }
    vtheta_samp = min_vel_theta;
    vx_samp = 0.0;
    vy_samp = 0.0;
    double heading_dist = DBL_MAX;
    auto ahead = [&](const Result& t, double& out) {  // goal distance one heading_lookahead ahead of the end point
      const double th_r = t.th.back();
      unsigned cx, cy;
      if (!cm.world_to_map(t.x.back() + cfg.heading_lookahead * cos(th_r), t.y.back() + cfg.heading_lookahead * sin(th_r), cx, cy))
        return false;
      out = goal_dist[size_t(cy) * cm.sx + cx];
      return true;
    };
    for (int i = 0; i < cfg.vtheta_samples; ++i) {
      const double limited = vtheta_samp > 0 ? std::max(vtheta_samp, cfg.min_in_place_vel_th)
                                             : std::min(vtheta_samp, -1.0 * cfg.min_in_place_vel_th);
      gen(vx_samp, vy_samp, limited);
      if (comp->cost >= 0 && (comp->cost <= best->cost || best->cost < 0 || best->yv != 0.0) &&
          (vtheta_samp > dvtheta || vtheta_samp < -1 * dvtheta)) {
        double ag;
        if (ahead(*comp, ag) && ag < heading_dist) {
          if (vtheta_samp < 0 && !stuck_left) { std::swap(best, comp); heading_dist = ag; }
          else if (vtheta_samp > 0 && !stuck_right) { std::swap(best, comp); heading_dist = ag; }
        }
      }
      vtheta_samp += dvtheta;
    }
    auto reset_if_moved = [&]() {
      if (hypot(x - prev_x, y - prev_y) > cfg.oscillation_reset_dist)
        rotating_left = rotating_right = strafe_left = strafe_right = stuck_left = stuck_right = stuck_left_strafe =
            stuck_right_strafe = false;
    };
    auto leave_escape = [&]() {
      double a = fmod(fmod(theta - escape_theta, 2.0 * M_PI) + 2.0 * M_PI, 2.0 * M_PI);
      if (a > M_PI) a -= 2.0 * M_PI;
      if (hypot(x - escape_x, y - escape_y) > cfg.escape_reset_dist || fabs(a) > cfg.escape_reset_theta) escaping = false;
    };
    if (best->cost >= 0) {  // :700-749
      if (!(best->xv > 0)) {
        if (best->thetav < 0) { if (rotating_right) stuck_right = true; rotating_right = true; }
        else if (best->thetav > 0) { if (rotating_left) stuck_left = true; rotating_left = true; }
        else if (best->yv > 0) { if (strafe_right) stuck_right_strafe = true; strafe_right = true; }
        else if (best->yv < 0) { if (strafe_left) stuck_left_strafe = true; strafe_left = true; }
        prev_x = x;
        prev_y = y;
      }
      reset_if_moved();
      leave_escape();
      return *best;
    }
    if (cfg.holonomic_robot) {  // :752-797
      vtheta_samp = min_vel_theta;
      vx_samp = 0.0;
      for (int i = 0; i < cfg.n_y_vels; ++i) {
        vtheta_samp = 0;
        vy_samp = cfg.y_vels[i];
        gen(vx_samp, vy_samp, vtheta_samp);
        if (comp->cost >= 0 && (comp->cost <= best->cost || best->cost < 0)) {
          double ag;
          if (ahead(*comp, ag) && ag < heading_dist) {
            if (vy_samp > 0 && !stuck_left_strafe) { std::swap(best, comp); heading_dist = ag; }
            else if (vy_samp < 0 && !stuck_right_strafe) { std::swap(best, comp); heading_dist = ag; }
          }
        }
      }
    }
    if (best->cost >= 0) {  // :800-848
      if (!(best->xv > 0)) {
        if (best->thetav < 0) { if (rotating_right) stuck_right = true; rotating_left = true; }
        else if (best->thetav > 0) { if (rotating_left) stuck_left = true; rotating_right = true; }
        else if (best->yv > 0) { if (strafe_right) stuck_right_strafe = true; strafe_left = true; }
        else if (best->yv < 0) { if (strafe_left) stuck_left_strafe = true; strafe_right = true; }
        prev_x = x;
        prev_y = y;
      }
      reset_if_moved();
      leave_escape();
      return *best;
    }
    gen(cfg.backup_vel, 0.0, 0.0);  // :851-903
    std::swap(best, comp);
    reset_if_moved();
    if (!escaping && best->cost > -2.0) {
      escape_x = x;
      escape_y = y;
      escape_theta = theta;
      escaping = true;
    }
    leave_escape();
    if (best->cost == -1.0) best->cost = 1.0;
    return *best;
  }

  // findBestPath (:908-980)
  Result find_best_path(const double pose[3], const double vel[3]) {
    const double x = (float)pose[0], y = (float)pose[1], theta = (float)pose[2];  // Eigen::Vector3f pos / vel
    const double vx = (float)vel[0], vy = (float)vel[1], vtheta = (float)vel[2];
    std::vector<uint8_t> within(size_t(cm.sx) * cm.sy, 0);
    for (const auto& c : footprint_cells(x, y, theta)) within[size_t(c.second) * cm.sx + c.first] = 1;
    wavefront(false, &within, path_dist);
    wavefront(true, nullptr, goal_dist);
    return create(x, y, theta, vx, vy, vtheta);
  }
};

}  // namespace

extern "C" {

// ---- legacy TrajectoryPlanner (restated above)
void navo_tp_default_config(navo_tp_config* c) {  // trajectory_planner_ros.cpp:116-213
  memset(c, 0, sizeof(*c));
  c->acc_lim_x = 2.5; c->acc_lim_y = 2.5; c->acc_lim_theta = 3.2;
  c->sim_time = 1.0; c->sim_granularity = 0.025; c->angular_sim_granularity = 0.025; c->sim_period = 0.05;
  c->pdist_scale = 0.6; c->gdist_scale = 0.8; c->occdist_scale = 0.01;
  c->heading_lookahead = 0.325; c->oscillation_reset_dist = 0.05; c->escape_reset_dist = 0.10;
  c->escape_reset_theta = M_PI_4;
  c->max_vel_x = 0.5; c->min_vel_x = 0.1; c->max_vel_th = 1.0; c->min_vel_th = -1.0; c->min_in_place_vel_th = 0.4;
  c->backup_vel = -0.1; c->heading_scoring_timestep = 0.8; c->stop_time_buffer = 0.2;
  c->y_vels[0] = -0.3; c->y_vels[1] = -0.1; c->y_vels[2] = 0.1; c->y_vels[3] = 0.3; c->n_y_vels = 4;
  c->vx_samples = 3; c->vtheta_samples = 20;
  c->holonomic_robot = 1; c->dwa = 1; c->heading_scoring = 0; c->simple_attractor = 0; c->allow_unknown = 0;
}
void* navo_tp_create(const navo_tp_config* cfg, uint32_t size_x, uint32_t size_y, double resolution,
                     const double* footprint_xy, int n_footprint) {
  Tp* t = new Tp;
  t->cfg = *cfg;
  t->cm.resize(size_x, size_y, resolution, 0.0, 0.0);
  for (int i = 0; i < n_footprint; ++i) t->footprint.push_back(Pt{footprint_xy[2 * i], footprint_xy[2 * i + 1]});
  const size_t n = size_t(size_x) * size_y;
  t->path_dist.assign(n, double(n + 1));  // MapGrid ctor + resetPathDist: unreachable everywhere
  t->goal_dist.assign(n, double(n + 1));
  return t;
}
void navo_tp_destroy(void* h) { delete static_cast<Tp*>(h); }
void navo_tp_reconfigure(void* h, const navo_tp_config* cfg) {  // trajectory_planner.cpp:59-133
  Tp* t = static_cast<Tp*>(h);
  t->cfg = *cfg;
  if (t->cfg.vx_samples <= 0) t->cfg.vx_samples = 1;
  if (t->cfg.vtheta_samples <= 0) t->cfg.vtheta_samples = 1;
}
void navo_tp_set_footprint(void* h, const double* xy, int n) {  // trajectory_planner.h:195
  static_cast<Tp*>(h)->footprint = to_pts(xy, n);
}
void navo_tp_set_costmap(void* h, const uint8_t* grid, double origin_x, double origin_y) {
  Tp* t = static_cast<Tp*>(h);
  t->cm.ox = origin_x;
  t->cm.oy = origin_y;
  memcpy(t->cm.c.data(), grid, t->cm.c.size());
}
void navo_tp_update_plan(void* h, const double* plan_xy, int n) {  // updatePlan(plan, false) :477-502
  Tp* t = static_cast<Tp*>(h);
  t->plan.clear();
  for (int i = 0; i < n; ++i) t->plan.push_back(Pt{plan_xy[2 * i], plan_xy[2 * i + 1]});
  t->final_goal_valid = n > 0;
  if (n > 0) { t->final_goal_x = t->plan.back().x; t->final_goal_y = t->plan.back().y; }
}
int navo_tp_find_best_path(void* h, const double pose[3], const double vel[3], navo_tp_result* result, double* points,
                           int points_capacity) {
  Tp* t = static_cast<Tp*>(h);
  const Tp::Result r = t->find_best_path(pose, vel);
  result->cost = r.cost; result->xv = r.xv; result->yv = r.yv; result->thetav = r.thetav;
  result->n_points = (int)r.x.size();
  result->flags = (t->stuck_left ? 1 : 0) | (t->stuck_right ? 2 : 0) | (t->stuck_left_strafe ? 4 : 0) |
                  (t->stuck_right_strafe ? 8 : 0) | (t->rotating_left ? 16 : 0) | (t->rotating_right ? 32 : 0) |
                  (t->strafe_left ? 64 : 0) | (t->strafe_right ? 128 : 0) | (t->escaping ? 256 : 0);
  for (int i = 0; i < result->n_points && i < points_capacity; ++i) {
    points[3 * i] = r.x[i]; points[3 * i + 1] = r.y[i]; points[3 * i + 2] = r.th[i];
  }
  return 0;
}
double navo_tp_score_trajectory(void* h, const double pose[3], const double vel[3], const double vs[3]) {  // :520-535
  Tp* t = static_cast<Tp*>(h);
  Tp::Result r;
  t->generate(pose[0], pose[1], pose[2], vel[0], vel[1], vel[2], vs[0], vs[1], vs[2], t->cfg.acc_lim_x, t->cfg.acc_lim_y,
              t->cfg.acc_lim_theta, double(size_t(t->cm.sx) * t->cm.sy), r);
  return r.cost;
}
void navo_tp_get_grid(void* h, int which, double* out) {
  Tp* t = static_cast<Tp*>(h);
  const std::vector<double>& d = which == 0 ? t->path_dist : t->goal_dist;
  memcpy(out, d.data(), d.size() * sizeof(double));
}

const char* navo_impl_name(void) { return "port"; }

void* navo_costmap_create(uint32_t size_x, uint32_t size_y, double resolution, double origin_x, double origin_y,
                          int rolling_window, int track_unknown) {
  Costmap* cm = new Costmap;
  cm->rolling = rolling_window != 0;
  cm->track_unknown = track_unknown != 0;
  cm->master.def = track_unknown ? kNoInfo : kFree;
  cm->master.resize(size_x, size_y, resolution, origin_x, origin_y);
  return cm;
}
void navo_costmap_destroy(void* h) { delete static_cast<Costmap*>(h); }
static int add_layer(Costmap* cm, LayerBase* l) {
  cm->layers.emplace_back(l);
  l->match_size(*cm);
  return int(cm->layers.size()) - 1;
}
int navo_costmap_add_grid_layer(void* h, int policy) { return add_layer(static_cast<Costmap*>(h), new GridLayer(policy)); }
int navo_costmap_add_obstacle_layer(void* h, int combination_method, int footprint_clearing, double max_obstacle_height) {
  return add_layer(static_cast<Costmap*>(h), new ObstacleLayer(combination_method, footprint_clearing != 0, max_obstacle_height));
}
int navo_costmap_add_voxel_layer(void* h, int combination_method, int footprint_clearing, double max_obstacle_height,
                                 double origin_z, double z_resolution, int z_voxels, int unknown_threshold,
                                 int mark_threshold) {
  return add_layer(static_cast<Costmap*>(h), new VoxelLayer(combination_method, footprint_clearing != 0, max_obstacle_height,
                                                            origin_z, z_resolution, z_voxels, unknown_threshold, mark_threshold));
}
void navo_layer_get_voxels(void* h, int layer, uint32_t* out) {
  VoxelLayer* v = dynamic_cast<VoxelLayer*>(static_cast<Costmap*>(h)->layers[layer].get());
  if (v) memcpy(out, v->vox.data(), v->vox.size() * sizeof(uint32_t));
}
int navo_voxel_line_cells(uint32_t size_x, double x0, double y0, double z0, double x1, double y1, double z1,
                          uint32_t max_length, uint32_t* offsets_out, int32_t* z_out, int capacity) {
  // same walk as VoxelLayer::clear_line, collecting instead of clearing
  int dx = int(x1) - int(x0), dy = int(y1) - int(y0), dz = int(z1) - int(z0);
  unsigned adx = abs(dx), ady = abs(dy), adz = abs(dz);
  int off_dx = dx > 0 ? 1 : -1, off_dy = (dy > 0 ? 1 : -1) * int(size_x), off_dz = dz > 0 ? 1 : -1;
  unsigned z_mask = ((1u << 16) | 1u) << (unsigned)z0, offset = (unsigned)y0 * size_x + (unsigned)x0;
  double dist = sqrt((x0 - x1) * (x0 - x1) + (y0 - y1) * (y0 - y1) + (z0 - z1) * (z0 - z1));
  double scale = std::min(1.0, max_length / dist);
  int n = 0;
  auto at = [&]() {
    if (n < capacity) {
      offsets_out[n] = offset;
      z_out[n] = __builtin_ctz(z_mask & 0xffffu ? z_mask & 0xffffu : 0x10000u);
    }
    ++n;
  };
  auto step = [&](int kind, int off) {
    if (kind == 0) offset += off;
    else if (off > 0) z_mask <<= 1;
    else z_mask >>= 1;
  };
  auto bres = [&](int ka, int kb, int kc, unsigned da, unsigned db, unsigned dc, int oa, int ob, int oc, unsigned max_len) {
    int err_b = da / 2, err_c = da / 2;
    unsigned end = std::min(max_len, da);
    for (unsigned i = 0; i < end; ++i) {
      at();
      step(ka, oa);
      err_b += db;
      err_c += dc;
      if ((unsigned)err_b >= da) { step(kb, ob); err_b -= da; }
      if ((unsigned)err_c >= da) { step(kc, oc); err_c -= da; }
    }
    at();
  };
  if (adx >= std::max(ady, adz)) bres(0, 0, 1, adx, ady, adz, off_dx, off_dy, off_dz, (unsigned)(scale * adx));
  else if (ady >= adz) bres(0, 0, 1, ady, adx, adz, off_dy, off_dx, off_dz, (unsigned)(scale * ady));
  else bres(1, 0, 0, adz, adx, ady, off_dz, off_dx, off_dy, (unsigned)(scale * adz));
  return n;
}
int navo_costmap_add_inflation_layer(void* h, double inflation_radius, double cost_scaling_factor) {
  Costmap* cm = static_cast<Costmap*>(h);
  InflationLayer* il = new InflationLayer;
  // onInitialize: the dynamic_reconfigure server delivers the defaults (0.55, 10) first, then matchSize (:71-98)
  il->weight = 0; il->radius = 0;
  il->res = cm->master.res;
  il->set_params(*cm, 0.55, 10.0);
  il->need_reinflation = true;
  int id = add_layer(cm, il);
  il->set_params(*cm, inflation_radius, cost_scaling_factor);
  return id;
}
void navo_costmap_set_footprint(void* h, const double* xy, int n) {  // layered_costmap.cpp:163-173
  Costmap* cm = static_cast<Costmap*>(h);
  cm->footprint = to_pts(xy, n);
  min_max_distances(cm->footprint, cm->inscribed, cm->circumscribed);
  for (auto& l : cm->layers) l->on_footprint_changed(*cm);
}
void navo_grid_layer_set(void* h, int layer, const uint8_t* data) {
  GridLayer* g = static_cast<GridLayer*>(static_cast<Costmap*>(h)->layers[layer].get());
  memcpy(g->g.c.data(), data, g->g.c.size());
  g->x = g->y = 0; g->w = g->g.sx; g->h = g->g.sy;
  g->updated = true;
}
void navo_grid_layer_touch(void* h, int layer, uint32_t x, uint32_t y, uint32_t w, uint32_t hgt) {
  GridLayer* g = static_cast<GridLayer*>(static_cast<Costmap*>(h)->layers[layer].get());
  g->x = x; g->y = y; g->w = w; g->h = hgt;
  g->updated = true;
}
void navo_layer_set_enabled(void* h, int layer, int enabled) {
  LayerBase* l = static_cast<Costmap*>(h)->layers[layer].get();
  // InflationLayer::reconfigureCB (inflation_layer.cpp:104-107): switching the layer on or off reinflates the whole map
  if (InflationLayer* il = dynamic_cast<InflationLayer*>(l))
    if (il->enabled != (enabled != 0)) il->need_reinflation = true;
  l->enabled = enabled != 0;
}
void navo_obstacle_set_observations(void* h, int layer, const navo_observation* obs, int n_obs) {
  ObstacleLayer* ol = static_cast<ObstacleLayer*>(static_cast<Costmap*>(h)->layers[layer].get());
  ol->obs.clear();
  for (int i = 0; i < n_obs; ++i) {
    Obs o;
    o.ox = obs[i].origin_x; o.oy = obs[i].origin_y; o.oz = obs[i].origin_z;
    o.obstacle_range = obs[i].obstacle_range;
    o.raytrace_range = obs[i].raytrace_range;
    o.xyz.assign(obs[i].xyz, obs[i].xyz + 3 * size_t(obs[i].n_points));
    o.marking = obs[i].marking != 0;
    o.clearing = obs[i].clearing != 0;
    ol->obs.push_back(std::move(o));
  }
}
void navo_inflation_set_params(void* h, int layer, double inflation_radius, double cost_scaling_factor) {
  Costmap* cm = static_cast<Costmap*>(h);
  static_cast<InflationLayer*>(cm->layers[layer].get())->set_params(*cm, inflation_radius, cost_scaling_factor);
}
int navo_inflation_set_variant(void* h, int layer, int variant, uint64_t seed) {
  if (variant < 0 || variant > 6) return -1;
  InflationLayer* il = static_cast<InflationLayer*>(static_cast<Costmap*>(h)->layers[layer].get());
  il->variant = variant;
  il->variant_seed = seed;
  return 0;
}
int navo_inflation_last_rounds(void* h, int layer) {
  return static_cast<InflationLayer*>(static_cast<Costmap*>(h)->layers[layer].get())->last_rounds;
}
void navo_costmap_update_map(void* h, double rx, double ry, double ryaw, int32_t w[4]) {
  Costmap* cm = static_cast<Costmap*>(h);
  cm->update_map(rx, ry, ryaw);
  w[0] = cm->bx0; w[1] = cm->bxn; w[2] = cm->by0; w[3] = cm->byn;
}
void navo_costmap_get(void* h, uint8_t* out) {
  Costmap* cm = static_cast<Costmap*>(h);
  memcpy(out, cm->master.c.data(), cm->master.c.size());
}
void navo_costmap_set(void* h, const uint8_t* in) {
  Costmap* cm = static_cast<Costmap*>(h);
  memcpy(cm->master.c.data(), in, cm->master.c.size());
}
void navo_layer_get(void* h, int layer, uint8_t* out) {
  Grid* g = static_cast<Costmap*>(h)->layers[layer]->grid();
  if (g) memcpy(out, g->c.data(), g->c.size());
}
void navo_costmap_get_origin(void* h, double out[2]) {
  Costmap* cm = static_cast<Costmap*>(h);
  out[0] = cm->master.ox;
  out[1] = cm->master.oy;
}
int navo_inflation_tables(void* h, int layer, uint8_t* costs_out, double* dists_out, int capacity) {
  InflationLayer* il = static_cast<InflationLayer*>(static_cast<Costmap*>(h)->layers[layer].get());
  int n = il->R + 2;
  if (n * n > capacity || il->R == 0) return il->R;
  memcpy(costs_out, il->costs.data(), size_t(n) * n);
  memcpy(dists_out, il->dists.data(), size_t(n) * n * sizeof(double));
  return il->R;
}

void navo_interpret_values(const uint8_t* in, uint8_t* out, int64_t n, int track_unknown, uint8_t unknown_cost_value,
                           uint8_t lethal_threshold, int trinary) {  // static_layer.cpp:149-163
  for (int64_t i = 0; i < n; ++i) {
    uint8_t v = in[i];
    if (v == unknown_cost_value) out[i] = track_unknown ? kNoInfo : kFree;
    else if (v >= lethal_threshold) out[i] = kLethal;
    else if (trinary) out[i] = kFree;
    else out[i] = (uint8_t)(((double)v / lethal_threshold) * kLethal);
  }
}

int navo_raytrace_cells(uint32_t size_x, uint32_t x0, uint32_t y0, uint32_t x1, uint32_t y1, uint32_t max_length,
                        uint32_t* offsets_out, int capacity) {
  int n = 0;
  raytrace_line(size_x, [&](unsigned off) { if (n < capacity) offsets_out[n] = off; ++n; }, x0, y0, x1, y1, max_length);
  return n;
}
void navo_footprint_radii(const double* xy, int n, double* inscribed, double* circumscribed) {
  min_max_distances(to_pts(xy, n), *inscribed, *circumscribed);
}

// ---- Path B
void navo_dwa_default_config(navo_dwa_config* c) {
  // base_local_planner/src/local_planner_limits/__init__.py:15-45, dwa_local_planner/cfg/DWAPlanner.cfg:15-43
  c->max_trans_vel = 0.55; c->min_trans_vel = 0.1; c->max_vel_x = 0.55; c->min_vel_x = 0.0;
  c->max_vel_y = 0.1; c->min_vel_y = -0.1; c->max_rot_vel = 1.0; c->min_rot_vel = 0.4;
  c->acc_lim_x = 2.5; c->acc_lim_y = 2.5; c->acc_lim_theta = 3.2;
  c->sim_time = 1.7; c->sim_granularity = 0.025; c->angular_sim_granularity = 0.1; c->sim_period = 0.05;
  c->path_distance_bias = 32.0; c->goal_distance_bias = 24.0; c->occdist_scale = 0.01;
  c->forward_point_distance = 0.325; c->cheat_factor = 1.0;
  c->oscillation_reset_dist = 0.05; c->oscillation_reset_angle = 0.2;
  c->scaling_speed = 0.25; c->max_scaling_factor = 0.2;
  c->vx_samples = 3; c->vy_samples = 10; c->vth_samples = 20;
  c->use_dwa = 1; c->sum_scores = 0; c->allow_unknown = 0;
}
void* navo_dwa_create(const navo_dwa_config* cfg, uint32_t size_x, uint32_t size_y, double resolution) {
  Dwa* d = new Dwa;
  d->cfg = *cfg;
  d->cm.def = 0;
  d->cm.resize(size_x, size_y, resolution, 0.0, 0.0);
  d->reconfigure();
  return d;
}
void navo_dwa_destroy(void* h) { delete static_cast<Dwa*>(h); }
void navo_dwa_reconfigure(void* h, const navo_dwa_config* cfg) {  // dwa_planner.cpp:52-112
  Dwa* d = static_cast<Dwa*>(h);
  d->cfg = *cfg;
  d->reconfigure();
}
void navo_dwa_set_costmap(void* h, const uint8_t* grid, double origin_x, double origin_y) {
  Dwa* d = static_cast<Dwa*>(h);
  d->cm.ox = origin_x;
  d->cm.oy = origin_y;
  memcpy(d->cm.c.data(), grid, d->cm.c.size());
}
void navo_dwa_set_plan(void* h, const double pose[3], const double* plan_xy, int n) {  // dwa_planner.cpp:240-286
  Dwa* d = static_cast<Dwa*>(h);
  d->plan = to_pts(plan_xy, n);
  d->path.target = d->plan;
  d->goal.target = d->plan;
  Pt g = d->plan.back();
  V3f pos{{float(pose[0]), float(pose[1]), float(pose[2])}};
  double sq = (pos[0] - g.x) * (pos[0] - g.x) + (pos[1] - g.y) * (pos[1] - g.y);
  std::vector<Pt> front = d->plan;
  double ang = atan2(g.y - pos[1], g.x - pos[0]);
  front.back().x = front.back().x + d->cfg.forward_point_distance * cos(ang);
  front.back().y = front.back().y + d->cfg.forward_point_distance * sin(ang);
  d->goal_front.target = front;
  if (sq > d->cfg.forward_point_distance * d->cfg.forward_point_distance * d->cfg.cheat_factor) {
    d->alignment.scale = d->cm.res * d->cfg.path_distance_bias * 0.5;
    d->alignment.target = d->plan;
  } else {
    d->alignment.scale = 0.0;
  }
}
void navo_dwa_reset_oscillation(void* h) { static_cast<Dwa*>(h)->reset_osc(); }
int navo_dwa_get_oscillation_mask(void* h) {
  Dwa* d = static_cast<Dwa*>(h);
  return int(d->forward_pos_only) | int(d->forward_neg_only) << 1 | int(d->strafe_pos_only) << 2 |
         int(d->strafe_neg_only) << 3 | int(d->rot_pos_only) << 4 | int(d->rot_neg_only) << 5;
}

int navo_dwa_find_best_path(void* h, const double pose[3], const double velv[3], const double* footprint_xy,
                            int n_footprint, navo_dwa_result* result, double* all_costs, int all_capacity,
                            double* best_points, int points_capacity) {  // dwa_planner.cpp:292-371
  Dwa* d = static_cast<Dwa*>(h);
  d->footprint = to_pts(footprint_xy, n_footprint);
  V3f pos{{float(pose[0]), float(pose[1]), float(pose[2])}};
  V3f vel{{float(velv[0]), float(velv[1]), float(velv[2])}};
  V3f goal{{float(d->plan.back().x), float(d->plan.back().y), 0.f}};
  std::vector<V3f> samples;
  d->enumerate_samples(pos, vel, goal, samples);
  // findBestTrajectory, simple_scored_sampling_planner.cpp:81-142
  d->prepare_all();
  Traj loop, best;
  double best_cost = -1;
  int best_index = -1, n_scored = 0;
  for (size_t i = 0; i < samples.size(); ++i) {
    double reported = std::numeric_limits<double>::quiet_NaN();
    if (d->generate(pos, vel, samples[i], loop)) {
      double c = d->score(loop, best_cost);
      reported = c;
      ++n_scored;
      if (c >= 0 && (best_cost < 0 || c < best_cost)) {
        best_cost = c;
        best = loop;
        best_index = int(i);
      }
    }
    if (all_costs && int(i) < all_capacity) all_costs[i] = reported;
  }
  // result_traj_ persists across cycles: only cost_ is reset, velocities and points stay stale when nothing is
  // valid (dwa_planner.cpp:316, simple_scored_sampling_planner.cpp:123-134)
  Traj& res = d->result;
  res.cost = -7;
  if (best_cost >= 0) {
    res = best;
    res.cost = best_cost;
  }
  d->update_osc_flags(pos, res, d->cfg.min_trans_vel);
  result->cost = res.cost;
  result->xv = res.xv; result->yv = res.yv; result->thetav = res.thv;
  result->best_index = best_index;
  result->n_samples = int(samples.size());
  result->n_scored = n_scored;
  result->n_points = int(res.x.size());
  if (best_points)
    for (size_t i = 0; i < res.x.size() && int(i) < points_capacity; ++i) {
      best_points[3 * i] = res.x[i];
      best_points[3 * i + 1] = res.y[i];
      best_points[3 * i + 2] = res.th[i];
    }
  return best_cost >= 0 ? 1 : 0;
}
double navo_dwa_check_trajectory(void* h, const double pose[3], const double velv[3], const double vel_samples[3],
                                 const double* footprint_xy, int n_footprint) {  // dwa_planner.cpp:213-237
  Dwa* d = static_cast<Dwa*>(h);
  d->footprint = to_pts(footprint_xy, n_footprint);
  V3f pos{{float(pose[0]), float(pose[1]), float(pose[2])}};
  V3f vel{{float(velv[0]), float(velv[1]), float(velv[2])}};
  V3f samp{{float(vel_samples[0]), float(vel_samples[1]), float(vel_samples[2])}};
  d->reset_osc();
  Traj t;
  d->generate(pos, vel, samp, t);  // a rejected sample leaves an empty trajectory, which every critic scores as 0
  return d->score(t, -1);
}
void navo_dwa_get_grid(void* h, int which, double* out) {
  Dwa* d = static_cast<Dwa*>(h);
  MapGridCritic* g[4] = {&d->path, &d->goal, &d->goal_front, &d->alignment};
  memcpy(out, g[which]->dist.data(), g[which]->dist.size() * sizeof(double));
}
void navo_dwa_prepare_only(void* h) { static_cast<Dwa*>(h)->prepare_all(); }

int navo_velocity_samples(double vmin, double vmax, int num_samples, double* out, int capacity) {
  std::vector<double> s = velocity_samples(vmin, vmax, num_samples);
  for (size_t i = 0; i < s.size() && int(i) < capacity; ++i) out[i] = s[i];
  return int(s.size());
}
int navo_line_cells(int x0, int y0, int x1, int y1, int32_t* xy_out, int capacity) {
  int n = 0;
  for (LineIt l(x0, y0, x1, y1); l.valid(); l.advance()) {
    if (n < capacity) { xy_out[2 * n] = l.x; xy_out[2 * n + 1] = l.y; }
    ++n;
  }
  return n;
}
void navo_mapgrid_bfs(const uint8_t* costs, uint32_t size_x, uint32_t size_y, const int32_t* seeds_xy, int n_seeds,
                      int allow_unknown, double* dist_out) {
  Grid cm;
  cm.resize(size_x, size_y, 1.0, 0, 0);
  memcpy(cm.c.data(), costs, cm.c.size());
  size_t n = cm.c.size();
  std::vector<double> dist(n, double(n + 1));
  std::vector<uint8_t> mark(n, 0);
  std::queue<unsigned> q;
  for (int i = 0; i < n_seeds; ++i) {
    unsigned id = seeds_xy[2 * i + 1] * size_x + seeds_xy[2 * i];
    dist[id] = 0.0;
    mark[id] = 1;
    q.push(id);
  }
  mapgrid_bfs(cm, allow_unknown != 0, dist, mark, q);
  memcpy(dist_out, dist.data(), n * sizeof(double));
}

}  // extern "C"
