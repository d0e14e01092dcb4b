// fleet_costmap_kernels.cuh -- one LayeredCostmap::updateMap (src/layered_costmap.cpp:79-150) of a rolling local costmap
// [ObstacleLayer, InflationLayer] or [VoxelLayer, InflationLayer] for every robot of a sensing fleet, one CTA per robot,
// the grids (and the voxel columns) in shared memory.  Built from the single costmap's device helpers
// (costmap_kernels.cuh) so a robot's result is bit for bit what navgpu_costmap computes with the same two layers.
#pragma once

#include "costmap_kernels.cuh"
#include "fleet_costmap.cuh"

namespace navgpu {

// where a robot's sources are in the fleet-wide tables (navgpu_fleet_set_scans)
struct FleetScanRobot {
  int clear_first, n_clear, rays;  // clearing DevObs [clear_first, + n_clear) of the fleet's table; total rays
  int mark_first, n_mark, marks;   // marking DevObs, likewise; total marking points
  long long mark_base;             // the robot's first entry of the marking scratch
};

constexpr int kFleetCmThreads = 256;
constexpr int kFleetFootprint = 16;               // = kMaxFootprint of the planner side
constexpr int kFleetPolyCells = kPolySmallCells;  // footprint rasteriser scratch (entries of each of its two arrays)

struct FleetCostmapArgs {
  uint8_t* layer;   // n x sy x pitch: every robot's ObstacleLayer (or VoxelLayer) grid
  uint8_t* master;  // n x sy x pitch: every robot's master grid (what the planner side scores against)
  unsigned sx, sy, pitch;
  unsigned spitch;  // row pitch of the grids in shared memory
  double res;
  uint8_t def;      // default value of both grids (track_unknown ? NO_INFORMATION : FREE_SPACE)
  int policy;       // NAVGPU_OVERWRITE or NAVGPU_MAX (ObstacleLayer::combination_method_)
  int footprint_clearing;
  double max_obstacle_height;
  int nfp;
  double fpx[kFleetFootprint], fpy[kFleetFootprint];  // footprint, robot frame
  const FleetScanRobot* robots;
  const FleetCmStep* steps;
  const DevObs* clear;
  const DevObs* mark;
  const float* xyz;        // every robot's projected clouds (k_project_scans)
  long long* mark_cells;   // one entry per marking point
  DevBox* boxes;           // n x 2: the obstacle layer's touched box (the inflation entry is unused)
  InflationBoundsState* infl;  // n x 2: InflationLayer::last_* of every robot (entry 1)
  DevWindow* win;          // n: the cycle's window
  int reinflate;           // InflationLayer::need_reinflation_ (the first step)
  double inflation_radius;
  int R;                   // cell inflation radius; 0: the inflation layer does nothing
  const uint8_t* cost_d2;  // R * R + 1 entries: cost by squared cell distance
  uint32_t* vox;           // voxel fleets: n x sy x pitch, every robot's VoxelLayer columns
  VoxelGeom v;             // voxel fleets: the VoxelLayer's geometry and thresholds
};

// Dynamic shared memory of k_fleet_costmap: the rasteriser's two arrays, the seed bitmask (one word of 32 cells per
// row position plus an empty word on either side), the obstacle grid, the master grid, the horizontal seed distances,
// one "row has a seed" byte per row and the cost table.  A voxel fleet also holds the robot's columns (4 B per cell);
// they are written back before the inflation, so the seed bitmask and the horizontal distances reuse their space.
__host__ __device__ inline unsigned fleet_seed_words(unsigned sx) { return (sx + 31) / 32 + 2; }
__host__ __device__ inline size_t fleet_costmap_smem(unsigned sy, unsigned spitch, unsigned seed_words, int R,
                                                     bool voxel = false) {
  const size_t seed = size_t(sy) * seed_words * sizeof(uint32_t), hx = size_t(sy) * spitch;
  const size_t cols = voxel ? size_t(sy) * spitch * sizeof(uint32_t) : 0;
  const size_t shared = cols > seed + hx ? cols : seed + hx;
  return 2 * kFleetPolyCells * sizeof(uint32_t) + shared + 2 * size_t(sy) * spitch + sy + size_t(R) * R + 1;
}

// Per robot (CTA), in the order of the reference:
//   1. Costmap2D::updateOrigin of both grids: the previous grids shifted by the step's cell offset while they are
//      loaded, the default value in the new cells (costmap_2d.cpp:264-313); a voxel fleet's columns likewise, unknown
//      columns in the new cells (VoxelLayer::updateOrigin, voxel_layer.cpp:371-438)
//   2. ObstacleLayer::updateBounds (obstacle_layer.cpp:340-413): ray-trace clearing of every clearing source (one warp
//      per ray, raytrace_ray on the shared grid), a barrier, marking (mark_prepare), the touched bounds of the sensor
//      origins and the footprint.
//      Voxel (VoxelLayer::updateBounds, voxel_layer.cpp:118-180): every ray's 3-D clear on the shared columns
//      (voxel_clear_ray), a barrier, every ray's 2-D cells from the final columns (voxel_commit_ray), a barrier, then
//      marking (voxel_mark_cell + voxel_mark_commit); the sensor origins are not touched.  The columns are written back
//      here, their space goes to the inflation's scratch.
//   3. ObstacleLayer::updateCosts' footprint clearing (:427-435) on the obstacle grid
//   4. the bounds pass (finalize_bounds: InflationLayer::updateBounds with this robot's last_* state, the window)
//   5. resetMap of the window, the obstacle grid merged with Overwrite or Max, and InflationLayer::updateCosts as the
//      exact windowed nearest-seed inflation of k_update_costs over the whole robot map (its halo is the map itself)
//   6. both grids written back
template <bool kVoxel>
__device__ __forceinline__ void fleet_costmap_cta(const FleetCostmapArgs& a) {
  extern __shared__ __align__(16) uint8_t fsm[];
  __shared__ unsigned long long s_box[kFleetCmThreads / 32][4];
  __shared__ __align__(8) unsigned char s_ba_bytes[sizeof(BoundsArgs)];  // (BoundsArgs has member initialisers)
  BoundsArgs& s_ba = *reinterpret_cast<BoundsArgs*>(s_ba_bytes);
  __shared__ DevWindow s_win;
  __shared__ PolyArgs s_poly;
  __shared__ int s_do_poly;
  const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int nt = kFleetCmThreads, n_warps = kFleetCmThreads / 32;
  const int sx = (int)a.sx, sy = (int)a.sy, sp = (int)a.spitch, R = a.R;
  const int bw = (int)fleet_seed_words(a.sx);
  uint32_t* poly_cells = reinterpret_cast<uint32_t*>(fsm);
  uint32_t* poly_sorted = poly_cells + kFleetPolyCells;
  uint32_t* bits = poly_sorted + kFleetPolyCells;
  uint8_t *lay, *mas, *hx;
  uint32_t* cols = bits;  // voxel: the columns, over the seed bitmask and the horizontal distances
  if constexpr (kVoxel) {
    hx = reinterpret_cast<uint8_t*>(bits + sy * bw);
    lay = reinterpret_cast<uint8_t*>(bits) + max(sy * sp * (int)sizeof(uint32_t), sy * bw * (int)sizeof(uint32_t) + sy * sp);
    mas = lay + sy * sp;
  } else {
    lay = reinterpret_cast<uint8_t*>(bits + sy * bw);
    mas = lay + sy * sp;
    hx = mas + sy * sp;
  }
  uint8_t* rowany = (kVoxel ? mas : hx) + sy * sp;
  uint8_t* table = rowany + sy;

  const FleetCmStep st = a.steps[r];
  const FleetScanRobot rb = a.robots[r];
  const size_t gbase = (size_t)r * a.sy * a.pitch;
  const Geom g{a.sx, a.sy, a.spitch, a.res, st.ox, st.oy};

  // 1. both grids, shifted (k_shift_grid's rule)
  for (int i = tid; i < sy * sx; i += nt) {
    const int y = i / sx, x = i - y * sx;
    const long long ox = (long long)x + st.cell_dx, oy = (long long)y + st.cell_dy;
    uint8_t l = a.def, m = a.def;
    if (ox >= 0 && ox < sx && oy >= 0 && oy < sy) {
      const size_t o = gbase + (size_t)oy * a.pitch + (size_t)ox;
      l = a.layer[o];
      m = a.master[o];
    }
    lay[y * sp + x] = l;
    mas[y * sp + x] = m;
    if constexpr (kVoxel) {
      uint32_t c = 0x0000ffffu;  // k_shift_voxels' rule
      if (ox >= 0 && ox < sx && oy >= 0 && oy < sy) c = a.vox[gbase + (size_t)oy * a.pitch + (size_t)ox];
      cols[y * sp + x] = c;
    }
  }
  for (int i = tid; i <= R * R && R > 0; i += nt) table[i] = a.cost_d2[i];
  BoxAcc acc;
  if (tid == 0) {
    // raytraceFreespace touches the origin of every clearing source that lies on the map (:504-521); the VoxelLayer's
    // does not
    for (int k = 0; k < rb.n_clear && !kVoxel; ++k) {
      const DevObs& o = a.clear[rb.clear_first + k];
      unsigned mx, my;
      if (world_to_map(g, o.ox, o.oy, mx, my)) acc.touch(o.ox, o.oy);
    }
    // updateFootprint (:415-425, transformFootprint footprint.cpp:106-120) and the polygon's cells for updateCosts
    // (worldToMap of every vertex; one off the map: no clearing, costmap_2d.cpp:315-342)
    int n = 0;
    bool on_map = true;
    if (a.footprint_clearing) {
      for (int k = 0; k < a.nfp; ++k) {
        const double wx = st.rx + (a.fpx[k] * st.cos_th - a.fpy[k] * st.sin_th);
        const double wy = st.ry + (a.fpx[k] * st.sin_th + a.fpy[k] * st.cos_th);
        acc.touch(wx, wy);
        unsigned mx, my;
        if (on_map && world_to_map(g, wx, wy, mx, my)) {
          s_poly.vx[n] = (int)mx;
          s_poly.vy[n] = (int)my;
          ++n;
        } else {
          on_map = false;
        }
      }
    }
    s_poly.n = n;
    s_do_poly = on_map && n >= 3;
  }
  __syncthreads();

  // 2. every ray cleared before any point is marked (:362-368)
  const DevObs* ctab = a.clear + rb.clear_first;
  const DevObs* mtab = a.mark + rb.mark_first;
  if constexpr (kVoxel) {
    for (int ray = warp; ray < rb.rays; ray += n_warps)
      voxel_clear_ray(cols, g, a.v, ctab, rb.n_clear, a.xyz, a.max_obstacle_height, acc, ray, lane);
    __syncthreads();
    for (int ray = warp; ray < rb.rays; ray += n_warps)
      voxel_commit_ray(lay, cols, g, a.v, ctab, rb.n_clear, a.xyz, a.max_obstacle_height, ray, lane);
    __syncthreads();
    for (int t = tid; t < rb.marks; t += nt) {
      const long long c = voxel_mark_cell(g, a.v, mtab, rb.n_mark, a.xyz, a.max_obstacle_height, acc, t);
      if (c >= 0) voxel_mark_commit(lay, cols, a.v.mark_threshold, c);
    }
    __syncthreads();
    for (int i = tid; i < sy * sx; i += nt) {  // the columns are final
      const int y = i / sx, x = i - y * sx;
      a.vox[gbase + (size_t)y * a.pitch + x] = cols[y * sp + x];
    }
  } else {
    for (int ray = warp; ray < rb.rays; ray += n_warps) raytrace_ray(lay, g, ctab, rb.n_clear, a.xyz, rb.rays, acc, ray, lane);
    __syncthreads();
    long long* cells = a.mark_cells + rb.mark_base;
    for (int t = tid; t < rb.marks; t += nt) {
      mark_prepare(g, mtab, rb.n_mark, a.xyz, a.max_obstacle_height, acc, cells, t);
      const long long c = cells[t];
      if (c >= 0) lay[c] = kLethal;
    }
    __syncthreads();
  }

  // 3. the footprint polygon to FREE_SPACE, after the marks
  if (s_do_poly) polygon_clear_cta(lay, a.spitch, s_poly, kFree, poly_cells, poly_sorted, kFleetPolyCells);

  // 4. bounds -> window
  DevBox* box = a.boxes + 2 * (size_t)r;
  acc.flush_cta(box, s_box);
  __syncthreads();
  if (tid == 0) {
    s_ba.n_layers = 2;
    s_ba.layer[0] = BoundsLayer{0, 0, 0.0, 0.0, 0.0, 0.0};  // everything the obstacle layer touched is in its box
    s_ba.layer[1] = BoundsLayer{2, a.reinflate, a.inflation_radius, 0.0, 0.0, 0.0};
    s_ba.master = g;
    s_ba.mirror_dirty = nullptr;
    s_ba.mirror_pad = 0;
    finalize_bounds(s_ba, box, a.infl + 2 * (size_t)r, &s_win);
    a.win[r] = s_win;
  }
  __syncthreads();

  // 5. reset + merge inside the window, then inflation (k_update_costs' three phases over the whole map)
  const DevWindow w = s_win;
  if (w.valid) {
    const int ww = w.xn - w.x0;
    for (int i = tid; i < ww * (w.yn - w.y0); i += nt) {
      const int y = w.y0 + i / ww, x = w.x0 + i % ww;
      mas[y * sp + x] = apply_policy(a.def, lay[y * sp + x], a.policy);
    }
    __syncthreads();
    if (R > 0) {
      // seed region: window +- R clamped to the map (inflation_layer.cpp:203-211)
      const int sx0 = max(0, w.x0 - R), sxn = min(sx, w.xn + R);
      const int sy0 = max(0, w.y0 - R), syn = min(sy, w.yn + R);
      for (int i = tid; i < sy * bw; i += nt) {
        const int y = i / bw, wi = i - y * bw;
        uint32_t word = 0;
        if (wi > 0 && wi < bw - 1 && y >= sy0 && y < syn) {
          const int x0 = (wi - 1) * 32;
          for (int b = 0; b < 32; ++b) {
            const int x = x0 + b;
            if (x >= sx0 && x < sxn && mas[y * sp + x] == kLethal) word |= 1u << b;
          }
        }
        bits[i] = word;
      }
      __syncthreads();
      for (int y = tid; y < sy; y += nt) {
        uint32_t any = 0;
        for (int wi = 1; wi < bw - 1; ++wi) any |= bits[y * bw + wi];
        rowany[y] = any != 0;
      }
      // horizontal distance to the nearest seed of the same row, |dx| <= R (255 = none)
      for (int i = tid; i < sy * sx; i += nt) {
        const int y = i / sx, x = i - y * sx;
        const uint32_t* wrow = bits + y * bw;
        const int p = 32 + x;  // bit position of this cell in the row
        auto word = [&](int k) -> uint32_t { return (k < 0 || k >= bw) ? 0u : wrow[k]; };
        auto window32 = [&](int q) -> uint32_t {  // bits q .. q+31
          const int wi = q >> 5, sh = q & 31;
          return __funnelshift_r(word(wi), word(wi + 1), sh);
        };
        int best = 255;
        for (int base = 0; base <= R; base += 32) {
          const uint32_t right = window32(p + base);      // bit k  <-> distance base + k
          const uint32_t left = window32(p - base - 31);  // bit 31-k <-> distance base + k
          int d = 255;
          if (right) d = base + (__ffs(right) - 1);
          if (left) d = min(d, base + __clz(left));
          if (d != 255) { best = d; break; }
        }
        hx[y * sp + x] = (uint8_t)(best <= R ? best : 255);
      }
      __syncthreads();
      // d^2 = min over dy of dy^2 + hx(y + dy)^2, rows of the map only
      const int R2 = R * R;
      for (int i = tid; i < sy * sx; i += nt) {
        const int y = i / sx, x = i - y * sx;
        int best = 0x7fffffff;
        for (int yy = max(0, y - R); yy <= min(sy - 1, y + R); ++yy) {
          if (!rowany[yy]) continue;
          const int h = hx[yy * sp + x];
          if (h != 255) best = min(best, h * h + (yy - y) * (yy - y));
        }
        if (best <= R2) mas[y * sp + x] = inflate_combine(mas[y * sp + x], table[best]);
      }
    }
  }
  __syncthreads();

  // 6. write-back
  for (int i = tid; i < sy * sx; i += nt) {
    const int y = i / sx, x = i - y * sx;
    const size_t o = gbase + (size_t)y * a.pitch + x;
    a.layer[o] = lay[y * sp + x];
    a.master[o] = mas[y * sp + x];
  }
}

__global__ void __launch_bounds__(kFleetCmThreads) k_fleet_costmap(FleetCostmapArgs a) { fleet_costmap_cta<false>(a); }
// two CTAs per SM is what the shared memory of a 120 x 120 robot allows; this bound lets ptxas keep the voxel steps in
// registers (a single-argument bound settles on 64 registers and spills)
__global__ void __launch_bounds__(kFleetCmThreads, 2) k_fleet_costmap_voxel(FleetCostmapArgs a) { fleet_costmap_cta<true>(a); }

// ---------------------------------------------------------------------------------------------------------------
// Batched scan ingest (navgpu_fleet_set_scan_batch): every robot carries the same sources, source s of robot r is row r
// of the source's arrays.  The tables k_fleet_costmap reads are then regular, and what navgpu_fleet_set_scans lists
// robot by robot is one index computation away:
//   points     robot-major: point i of source s of robot r is r * points + point_first(s) + i
//   d_obs      n * n_clear clearing entries (robot-major, a robot's clearing sources in order, listed even without
//              points), then n * n_mark marking entries (sources with points only)
//   mark_base  r * marks
constexpr int kScanBatchSources = 32;  // sources per batch: they travel as kernel parameters
constexpr int kScanBatchThreads = 256;

struct ScanBatchSource {
  const float* data;      // [n][n_points] ranges or [n][n_points][3] sensor-frame points
  const double* stg;      // [n][7]: translation x, y, z, rotation x, y, z, w
  double angle_min, angle_increment;  // the float fields, widened exactly (ScanRec)
  double min_obstacle_height, max_obstacle_height, obstacle_range, raytrace_range;
  float range_min, range_max;
  int n_points, is_cloud, inf_is_valid, flags;  // flags: bit0 marking, bit1 clearing (DevObs)
  int point_first;             // the source's first point within its robot
  int clear_slot, mark_slot;   // its entry among the robot's clearing / marking entries; -1: not listed
  int clear_ray, mark_ray;     // DevObs::first_ray of those entries
};

struct ScanBatchArgs {
  ScanBatchSource src[kScanBatchSources];
  int n_sources, n;
  int points, n_clear, n_mark, rays, marks;  // per robot
  float* xyz;
  DevObs* obs;
  FleetScanRobot* robots;
};

// grid (x, max(1, n_sources)): blockIdx.y is the source; x covers max(n, n * n_points) threads.  Thread t < n of source
// s writes robot t's DevObs of s (and, on source 0, robot t's FleetScanRobot); thread t < n * n_points projects point
// t % n_points of robot t / n_points through project_point, the per-point body of k_project_scans.
__global__ void __launch_bounds__(kScanBatchThreads) k_fleet_scan_batch(const ScanBatchArgs a) {
  const int t = blockIdx.x * kScanBatchThreads + threadIdx.x, s = blockIdx.y;
  if (s == 0 && t < a.n) {
    FleetScanRobot rb;
    rb.clear_first = t * a.n_clear; rb.n_clear = a.n_clear; rb.rays = a.rays;
    rb.mark_first = a.n * a.n_clear + t * a.n_mark; rb.n_mark = a.n_mark; rb.marks = a.marks;
    rb.mark_base = (long long)t * a.marks;
    a.robots[t] = rb;
  }
  if (s >= a.n_sources) return;
  const ScanBatchSource& src = a.src[s];
  if (t < a.n && (src.clear_slot >= 0 || src.mark_slot >= 0)) {
    const double* tr = src.stg + 7 * (size_t)t;
    DevObs d;
    d.ox = tr[0]; d.oy = tr[1]; d.oz = tr[2];  // the sensor origin (observation_buffer.cpp:143-151)
    d.obstacle_range = src.obstacle_range;
    d.raytrace_range = src.raytrace_range;
    d.first_point = t * a.points + src.point_first;
    d.n_points = src.n_points;
    d.flags = src.flags;
    if (src.clear_slot >= 0) {
      d.first_ray = src.clear_ray;
      a.obs[t * a.n_clear + src.clear_slot] = d;
    }
    if (src.mark_slot >= 0) {
      d.first_ray = src.mark_ray;
      a.obs[a.n * a.n_clear + t * a.n_mark + src.mark_slot] = d;
    }
  }
  if (t >= a.n * src.n_points) return;
  const int r = t / src.n_points, i = t - r * src.n_points;
  const double* tr = src.stg + 7 * (size_t)r;
  ScanRec rec;  // the projection record of (robot r, source s); its transform is built after the sensor-frame point
  rec.angle_min = src.angle_min;
  rec.angle_increment = src.angle_increment;
  rec.range_min = src.range_min;
  rec.range_max = src.range_max;
  rec.min_obstacle_height = src.min_obstacle_height;
  rec.max_obstacle_height = src.max_obstacle_height;
  rec.inf_is_valid = src.inf_is_valid;
  rec.is_cloud = src.is_cloud;
  const float* row = src.data + (size_t)r * src.n_points * (src.is_cloud ? 3 : 1);
  project_point(rec, row, i, a.xyz + 3 * ((size_t)r * a.points + src.point_first + i),
                [&](float m[9], float t3[3]) { sensor_affine(tr + 3, tr, m, t3); });
}

}  // namespace navgpu
