// costmap_kernels.cuh -- Path A device code: layered costmap update on the GPU (sm_100a).
//
// Reference semantics (file:line under /root/reference/costmap_2d) are cited next to each kernel; the host side
// that sequences them per LayeredCostmap::updateMap is in costmap.cu.
#pragma once

#include "common.cuh"

namespace navgpu {

struct Geom {
  unsigned sx, sy, pitch;
  double res, ox, oy;
};

// Costmap2D::worldToMap, src/costmap_2d.cpp:208-220
__device__ __forceinline__ bool world_to_map(const Geom& g, double wx, double wy, unsigned& mx, unsigned& my) {
  if (wx < g.ox || wy < g.oy) return false;
  mx = (unsigned)(int)((wx - g.ox) / g.res);
  my = (unsigned)(int)((wy - g.oy) / g.res);
  return mx < g.sx && my < g.sy;
}

// CostmapLayer::touch (src/costmap_layer.cpp:8-14) accumulated per thread in registers, then reduced per warp with
// shuffles and folded into the layer's device box with one atomic per warp and coordinate
struct BoxAcc {
  unsigned long long minx = ~0ull, miny = ~0ull, maxx = 0ull, maxy = 0ull;
  __device__ __forceinline__ void touch(double x, double y) {
    const unsigned long long ex = enc_double(x), ey = enc_double(y);
    minx = min(minx, ex); maxx = max(maxx, ex);
    miny = min(miny, ey); maxy = max(maxy, ey);
  }
  __device__ __forceinline__ void merge(const BoxAcc& o) {
    minx = min(minx, o.minx); maxx = max(maxx, o.maxx);
    miny = min(miny, o.miny); maxy = max(maxy, o.maxy);
  }
  // every thread of the CTA must call; one atomic per coordinate and CTA (the box words are shared by every CTA of
  // the launch, so per-warp atomics serialise on four L2 addresses)
  __device__ __forceinline__ void flush_cta(DevBox* box, unsigned long long (*s_box)[4]) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      minx = min(minx, __shfl_xor_sync(0xffffffffu, minx, o));
      maxx = max(maxx, __shfl_xor_sync(0xffffffffu, maxx, o));
      miny = min(miny, __shfl_xor_sync(0xffffffffu, miny, o));
      maxy = max(maxy, __shfl_xor_sync(0xffffffffu, maxy, o));
    }
    const int warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    if ((threadIdx.x & 31) == 0) {
      s_box[warp][0] = minx; s_box[warp][1] = miny; s_box[warp][2] = maxx; s_box[warp][3] = maxy;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
      const bool is_min = threadIdx.x < 2;
      unsigned long long v = s_box[0][threadIdx.x];
      for (int w = 1; w < n_warps; ++w) v = is_min ? min(v, s_box[w][threadIdx.x]) : max(v, s_box[w][threadIdx.x]);
      unsigned long long any = s_box[0][2];
      for (int w = 1; w < n_warps; ++w) any = max(any, s_box[w][2]);
      if (any != 0ull) {
        unsigned long long* dst = threadIdx.x == 0 ? &box->minx : threadIdx.x == 1 ? &box->miny : threadIdx.x == 2 ? &box->maxx : &box->maxy;
        if (is_min) atomicMin(dst, v);
        else atomicMax(dst, v);
      }
    }
  }
  __device__ __forceinline__ void reduce_warp() {  // all 32 lanes must call; every lane ends up with the warp's box
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      minx = min(minx, __shfl_xor_sync(0xffffffffu, minx, o));
      maxx = max(maxx, __shfl_xor_sync(0xffffffffu, maxx, o));
      miny = min(miny, __shfl_xor_sync(0xffffffffu, miny, o));
      maxy = max(maxy, __shfl_xor_sync(0xffffffffu, maxy, o));
    }
  }
  // s_box holds one box per warp (written before the barrier in front of this call): threads 0..3 fold them into the
  // layer's device box, one atomic per coordinate and CTA
  static __device__ __forceinline__ void flush_rows(DevBox* box, unsigned long long (*s_box)[4], int n_rows) {
    if (threadIdx.x < 4) {
      const bool is_min = threadIdx.x < 2;
      unsigned long long v = s_box[0][threadIdx.x], any = s_box[0][2];
      for (int w = 1; w < n_rows; ++w) {
        v = is_min ? min(v, s_box[w][threadIdx.x]) : max(v, s_box[w][threadIdx.x]);
        any = max(any, s_box[w][2]);
      }
      if (any != 0ull) {
        unsigned long long* dst = threadIdx.x == 0 ? &box->minx : threadIdx.x == 1 ? &box->miny : threadIdx.x == 2 ? &box->maxx : &box->maxy;
        if (is_min) atomicMin(dst, v);
        else atomicMax(dst, v);
      }
    }
  }
  __device__ __forceinline__ void flush_warp(DevBox* box) {  // all 32 lanes must call
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      minx = min(minx, __shfl_xor_sync(0xffffffffu, minx, o));
      maxx = max(maxx, __shfl_xor_sync(0xffffffffu, maxx, o));
      miny = min(miny, __shfl_xor_sync(0xffffffffu, miny, o));
      maxy = max(maxy, __shfl_xor_sync(0xffffffffu, maxy, o));
    }
    if ((threadIdx.x & 31) == 0 && maxx != 0ull) {
      atomicMin(&box->minx, minx);
      atomicMax(&box->maxx, maxx);
      atomicMin(&box->miny, miny);
      atomicMax(&box->maxy, maxy);
    }
  }
};

// ---------------------------------------------------------------------------------------------------------------
// Rolling-window origin shift, Costmap2D::updateOrigin (src/costmap_2d.cpp:264-313): out of place,
// dst(x, y) = src(x + cell_ox, y + cell_oy) where that lies inside the old grid, default elsewhere.
__global__ void k_shift_grid(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, unsigned sx, unsigned sy,
                             unsigned pitch, int cell_ox, int cell_oy, uint8_t def) {
  unsigned x = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned y = blockIdx.y;
  if (x >= pitch || y >= sy) return;
  uint8_t v = def;
  long long ox = (long long)x + cell_ox, oy = (long long)y + cell_oy;
  if (x < sx && ox >= 0 && ox < (long long)sx && oy >= 0 && oy < (long long)sy) v = src[(size_t)oy * pitch + ox];
  dst[(size_t)y * pitch + x] = v;
}

// ---------------------------------------------------------------------------------------------------------------
// StaticLayer::interpretValue over an OccupancyGrid (plugins/static_layer.cpp:149-163, applied as in :196-207)
__global__ void k_interpret_occupancy(const int8_t* __restrict__ occ, uint8_t* __restrict__ grid, unsigned sx,
                                      unsigned sy, unsigned pitch, int track_unknown, uint8_t unknown_cost_value,
                                      uint8_t lethal_threshold, int trinary) {
  unsigned x = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned y = blockIdx.y;
  if (x >= sx || y >= sy) return;
  uint8_t value = (uint8_t)occ[(size_t)y * sx + x];
  uint8_t r;
  if (value == unknown_cost_value) r = track_unknown ? kNoInfo : kFree;
  else if (value >= lethal_threshold) r = kLethal;
  else if (trinary) r = kFree;
  else {
    double scale = (double)value / lethal_threshold;
    r = (uint8_t)(scale * kLethal);
  }
  grid[(size_t)y * pitch + x] = r;
}

// ---------------------------------------------------------------------------------------------------------------
// Observations as laid out on the device
struct DevObs {
  double ox, oy, oz, obstacle_range, raytrace_range;
  int first_point, n_points;
  int first_ray;  // prefix over clearing observations (rays) / marking observations (points), per kernel
  int flags;      // bit0 marking, bit1 clearing
};

// ---------------------------------------------------------------------------------------------------------------
// Observation ingest (SURVEY.md 8f-3): sensor_msgs/LaserScan ranges -> world-frame cloud of an Observation, i.e. what
// ObstacleLayer::laserScanCallback (plugins/obstacle_layer.cpp:252-275; laserScanValidInfCallback :277-311) and
// ObservationBuffer::bufferCloud (src/observation_buffer.cpp:129-195) produce on the host:
//   1. laser_geometry::LaserProjection::projectLaser (laser_geometry 1.6.x, not part of the reference tree): a ray is
//      kept when range < range_max && range >= range_min; x = float(double(range) * cos(angle_min + double(i) *
//      angle_increment)), y likewise with sin, z = 0.  (transformLaserScanToPointCloud is called with the scan's own
//      frame as the target, obstacle_layer.cpp:262, so its per-ray transform is the identity.)
//   2. pcl_ros::transformPointCloud into the global frame (pcl_ros 1.4.x transforms.hpp + PCL 1.7): the tf rotation
//      becomes an Eigen::Quaternionf, its float rotation matrix and the float translation form an Affine3f, every
//      point is ((m0 * x + m1 * y) + m2 * z) + t per row in float.
//   3. points with z outside [min_obstacle_height, max_obstacle_height] are dropped (observation_buffer.cpp:170-177).
// Every ray keeps its slot in the observation's cloud; a dropped ray is stored as NaN, which raytrace_ray and
// mark_prepare skip -- clearing and marking are order independent, so this equals the compacted cloud.
struct ScanRec {
  double angle_min, angle_increment;  // float fields of the message, widened exactly
  float range_min, range_max;
  float m[9], t[3];  // Affine3f: rotation (row-major) and translation
  double min_obstacle_height, max_obstacle_height;
  int inf_is_valid;  // laserScanValidInfCallback: +inf becomes range_max - 0.0001f
  int first_point, n_points;
  int first_range;  // offset (in floats) into the uploaded ranges / sensor-frame points
  int is_cloud;     // 0: LaserScan ranges; 1: a PointCloud / PointCloud2 source, n_points x (x, y, z) in the sensor frame
};

// pcl_ros::transformPointCloud's Affine3f of a tf transform: Eigen::Quaternionf(w, x, y, z) -> float rotation matrix
// (Eigen's QuaternionBase::toRotationMatrix, row-major into m), Eigen::Vector3f translation into t; all arithmetic in
// float.  Shared by the host's record builder and k_fleet_scan_batch: x86-64 g++ does not contract and the device
// build has -fmad=false, so both round every operation alike.
__host__ __device__ inline void sensor_affine(const double q[4], const double tr[3], float m[9], float t[3]) {
  const float qx = (float)q[0], qy = (float)q[1], qz = (float)q[2], qw = (float)q[3];
  const float tx = 2.0f * qx, ty = 2.0f * qy, tz = 2.0f * qz;
  const float twx = tx * qw, twy = ty * qw, twz = tz * qw, txx = tx * qx, txy = ty * qx, txz = tz * qx, tyy = ty * qy,
              tyz = tz * qy, tzz = tz * qz;
  m[0] = 1.0f - (tyy + tzz); m[1] = txy - twz; m[2] = txz + twy;
  m[3] = txy + twz; m[4] = 1.0f - (txx + tzz); m[5] = tyz - twx;
  m[6] = txz - twy; m[7] = tyz + twx; m[8] = 1.0f - (txx + tyy);
  for (int k = 0; k < 3; ++k) t[k] = (float)tr[k];
}

// Point i of the scan described by r (first_point / first_range are not read): its world-frame (x, y, z) into out, or
// NaN when the ray is dropped.  src: the scan's ranges, or its sensor-frame points for a cloud.  affine(m, t) yields
// the record's rotation and translation (r.m / r.t are not read); it is called after the sensor-frame point exists, so
// a caller that computes them does not hold them across sincos.
template <class Affine>
__device__ __forceinline__ void project_point(const ScanRec& r, const float* __restrict__ src, int i,
                                              float* __restrict__ out, Affine affine) {
  const float nanf_ = __int_as_float(0x7fc00000);
  float ox = nanf_, oy = nanf_, oz = nanf_;
  float x = 0.0f, y = 0.0f, z = 0.0f;
  bool keep;
  if (r.is_cloud) {  // pointCloudCallback / pointCloud2Callback (obstacle_layer.cpp:313-339): the points as they are
    x = src[3 * i];
    y = src[3 * i + 1];
    z = src[3 * i + 2];
    keep = true;
  } else {
    float range = src[i];
    if (r.inf_is_valid && !isfinite(range) && range > 0) range = r.range_max - 0.0001f;
    keep = range < r.range_max && range >= r.range_min;
    if (keep) {
      const double ang = r.angle_min + (double)i * r.angle_increment;
      double sn, cs;
      sincos(ang, &sn, &cs);
      x = (float)((double)range * cs);
      y = (float)((double)range * sn);
    }
  }
  if (keep) {
    float m[9], t[3];
    affine(m, t);
    const float gx = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], x), __fmul_rn(m[1], y)), __fmul_rn(m[2], z)), t[0]);
    const float gy = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[3], x), __fmul_rn(m[4], y)), __fmul_rn(m[5], z)), t[1]);
    const float gz = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[6], x), __fmul_rn(m[7], y)), __fmul_rn(m[8], z)), t[2]);
    if ((double)gz <= r.max_obstacle_height && (double)gz >= r.min_obstacle_height) {
      ox = gx; oy = gy; oz = gz;
    }
  }
  out[0] = ox; out[1] = oy; out[2] = oz;
}

__global__ void k_project_scans(const ScanRec* __restrict__ recs, int n_scans, const float* __restrict__ ranges,
                                float* __restrict__ xyz, int total) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  // the last record that starts at or before point t (binary search: a fleet projects thousands of records at once)
  int k = 0, hi = n_scans - 1;
  while (k < hi) {
    const int mid = (k + hi + 1) >> 1;
    if (recs[mid].first_point - recs[0].first_point <= t) k = mid;
    else hi = mid - 1;
  }
  const ScanRec& r = recs[k];
  const int i = t - (r.first_point - recs[0].first_point);
  project_point(r, ranges + r.first_range, i, xyz + 3 * (size_t)(r.first_point + i), [&](float m[9], float tr[3]) {
    for (int k = 0; k < 9; ++k) m[k] = r.m[k];
    for (int k = 0; k < 3; ++k) tr[k] = r.t[k];
  });
}

// ObstacleLayer::raytraceFreespace (plugins/obstacle_layer.cpp:498-576) + Costmap2D::raytraceLine / bresenham2D
// (include/costmap_2d/costmap_2d.h:359-412) + updateRaytraceBounds (:602-610).
// One warp per ray.  All lanes evaluate the fp64 clip (identical operation order to the reference, no FMA
// contraction); the Bresenham walk is evaluated in closed form so the lanes write cells i, i+32, ... in parallel:
// after i major steps the reference's error accumulator has taken floor((abs_da/2 + i*abs_db)/abs_da) minor steps.
// All writers store FREE_SPACE, so write order between rays does not matter.
__device__ __forceinline__ void raytrace_ray(uint8_t* __restrict__ grid, const Geom& g, const DevObs* __restrict__ obs,
                                             int n_obs, const float* __restrict__ xyz, int total_rays, BoxAcc& acc,
                                             int warp, int lane) {
  bool touch1 = false;
  double t1x = 0, t1y = 0;
  if (warp < total_rays) {
    int k = 0;
    while (k + 1 < n_obs && obs[k + 1].first_ray <= warp) ++k;
    const DevObs o = obs[k];
    const int pi = o.first_point + (warp - o.first_ray);
    const double ox = o.ox, oy = o.oy;
    unsigned x0, y0;
    // a NaN point is a ray the on-device scan ingest dropped (k_project_scans): it is not part of the cloud
    const float px_raw = xyz[3 * (size_t)pi];
    if (px_raw == px_raw && world_to_map(g, ox, oy, x0, y0)) {  // origin off the map: the whole observation is skipped (:507-513)
      const double origin_x = g.ox, origin_y = g.oy;
      const double map_end_x = origin_x + g.sx * g.res;
      const double map_end_y = origin_y + g.sy * g.res;
      double wx = xyz[3 * (size_t)pi], wy = xyz[3 * (size_t)pi + 1];
      const double a = wx - ox, b = wy - oy;
      if (wx < origin_x) {
        double t = (origin_x - ox) / a;
        wx = origin_x;
        wy = oy + b * t;
      }
      if (wy < origin_y) {
        double t = (origin_y - oy) / b;
        wx = ox + a * t;
        wy = origin_y;
      }
      if (wx > map_end_x) {
        double t = (map_end_x - ox) / a;
        wx = map_end_x - .001;
        wy = oy + b * t;
      }
      if (wy > map_end_y) {
        double t = (map_end_y - oy) / b;
        wx = ox + a * t;
        wy = map_end_y - .001;
      }
      unsigned x1, y1;
      if (world_to_map(g, wx, wy, x1, y1)) {
        const unsigned cell_range = (unsigned)fmax(0.0, ceil(o.raytrace_range / g.res));  // cellDistance :181-185
        const int dx = (int)x1 - (int)x0, dy = (int)y1 - (int)y0;
        const unsigned adx = abs(dx), ady = abs(dy);
        const int off_dx = dx > 0 ? 1 : -1;
        const int off_dy = (dy > 0 ? 1 : -1) * (int)g.pitch;
        const double dist = hypot((double)dx, (double)dy);
        const double scale = (dist == 0.0) ? 1.0 : fmin(1.0, cell_range / dist);
        unsigned da, db;
        int off_a, off_b;
        if (adx >= ady) { da = adx; db = ady; off_a = off_dx; off_b = off_dy; }
        else { da = ady; db = adx; off_a = off_dy; off_b = off_dx; }
        const unsigned end = min((unsigned)(scale * da), da);
        const long long start = (long long)y0 * g.pitch + x0;
        const unsigned half = da / 2;
        if (da < 32768u) {  // i * db < 2^30: the closed form fits 32-bit arithmetic
          for (unsigned i = lane; i <= end; i += 32) {  // cells 0..end-1 of the loop plus the final at(offset)
            const unsigned m = da ? (half + i * db) / da : 0u;
            grid[start + (long long)((int)i * off_a + (int)m * off_b)] = kFree;
          }
        } else {
          for (unsigned i = lane; i <= end; i += 32) {
            const unsigned m = (unsigned)((half + (unsigned long long)i * db) / da);
            grid[start + (long long)i * off_a + (long long)m * off_b] = kFree;
          }
        }
        // updateRaytraceBounds
        const double ddx = wx - ox, ddy = wy - oy;
        const double full = hypot(ddx, ddy);
        const double s2 = fmin(1.0, o.raytrace_range / full);
        touch1 = true;
        t1x = ox + ddx * s2;
        t1y = oy + ddy * s2;
      }
    }
  }
  // every lane of the warp holds the same end point
  if (touch1 && lane == 0) acc.touch(t1x, t1y);
}

// ObstacleLayer::updateBounds marking loop (plugins/obstacle_layer.cpp:368-410), split in two so that the fp64 tests
// run on every CTA while the stores wait for all ray-trace clearing to finish:
//   mark_prepare  one thread per point: height / range tests, worldToMap, touch; leaves the cell offset (or -1) in
//                 `cells`
//   mark_commit   the threads of ONE CTA store LETHAL_OBSTACLE to the prepared offsets
__device__ __forceinline__ void mark_prepare(const Geom& g, const DevObs* __restrict__ obs, int n_obs,
                                             const float* __restrict__ xyz, double max_obstacle_height, BoxAcc& acc,
                                             long long* __restrict__ cells, int t) {
  int k = 0;
  while (k + 1 < n_obs && obs[k + 1].first_ray <= t) ++k;
  const DevObs o = obs[k];
  const size_t pi = (size_t)(o.first_point + (t - o.first_ray));
  const double px = xyz[3 * pi], py = xyz[3 * pi + 1], pz = xyz[3 * pi + 2];
  long long cell = -1;
  if (px == px && !(pz > max_obstacle_height)) {  // NaN: a ray dropped by the on-device scan ingest
    const double sq_dist = (px - o.ox) * (px - o.ox) + (py - o.oy) * (py - o.oy) + (pz - o.oz) * (pz - o.oz);
    if (!(sq_dist >= o.obstacle_range * o.obstacle_range)) {
      unsigned mx, my;
      if (world_to_map(g, px, py, mx, my)) {
        cell = (long long)my * g.pitch + mx;
        acc.touch(px, py);
      }
    }
  }
  cells[t] = cell;
}

constexpr unsigned kMarkTileW = 256, kMarkTileH = 32;  // = k_merge_seed's tile (static_assert next to that kernel)
// (called by the first `nt` threads of the CTA; nt = 0: all of them)
__device__ __forceinline__ void mark_commit_cta(uint8_t* __restrict__ grid, const long long* cells, int total_points,
                                                uint8_t* __restrict__ tile_used = nullptr, unsigned pitch = 1, int nt = 0) {
  if (nt == 0) nt = blockDim.x;
  constexpr int kU = 13;  // loads in flight per thread: a few thousand marks are one round trip for 224 threads
  for (int base = threadIdx.x; base < total_points; base += kU * nt) {
    long long cell[kU];
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      const int t = base + u * nt;
      cell[u] = t < total_points ? __ldcg(cells + t) : -1;  // written by other CTAs of this launch: read past L1
    }
#pragma unroll
    for (int u = 0; u < kU; ++u)
      if (cell[u] >= 0) {
        grid[cell[u]] = kLethal;
        if (tile_used) {  // MergeLayers::used: this tile no longer is all FREE_SPACE
          const unsigned y = (unsigned)(cell[u] / pitch), x = (unsigned)(cell[u] - (long long)y * pitch);
          tile_used[(y / (kMarkTileH)) * ((pitch + kMarkTileW - 1) / kMarkTileW) + x / kMarkTileW] = 1;
        }
      }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Costmap2D::setConvexPolygonCost -> convexFillCells -> polygonOutlineCells (src/costmap_2d.cpp:315-428).
// One CTA.  Outline cells come from the closed-form Bresenham (parallel), the reference's back-stepping bubble sort
// is a stable sort by x (parallel rank), and the column walk -- which in the reference iterates over the very
// vector it appends to -- is replayed verbatim by one thread so that degenerate footprints fill identically.
constexpr int kPolyMaxCells = 12288;   // stand-alone kernel (dynamic shared memory)
constexpr int kPolySmallCells = 2048;  // inside k_obstacle_update (static shared memory)
struct PolyArgs {
  int n;
  int vx[32], vy[32];
};
// cells / sorted: `capacity` packed (x | y << 16) entries each: the outline in order, and the vector convexFillCells
// works on.  Called by every thread of one CTA.
// First stage, by one warp (kWarp: lanes of the calling warp, warp-level barriers) or by the whole CTA: the outline
// cells, and for regular outlines -- every column between the extreme vertices holds at least two outline cells, which
// is what a closed outline gives -- per-column [min_y, max_y) in `sorted` (colmin | colmax | colcnt, W entries each):
// the reference's column walk (costmap_2d.cpp:391-427) is then a per-column fill, the first two sorted entries of a
// column seed min / max and the rest extend them.  Returns whether the outline is regular (uniform over the callers).
template <bool kWarp>
__device__ __forceinline__ bool polygon_prepare(const PolyArgs& poly, uint32_t* cells, uint32_t* sorted, int capacity) {
  __shared__ int edge_first[33];
  __shared__ int s_irregular;
  const int tid = kWarp ? (int)(threadIdx.x & 31) : (int)threadIdx.x, nt = kWarp ? 32 : (int)blockDim.x;
  auto sync = [] { if (kWarp) __syncwarp(); else __syncthreads(); };
  if (tid == 0) {
    int acc = 0;
    for (int k = 0; k < poly.n; ++k) {
      const int k1 = (k + 1) % poly.n;
      edge_first[k] = acc;
      acc += max(abs(poly.vx[k1] - poly.vx[k]), abs(poly.vy[k1] - poly.vy[k])) + 1;
    }
    edge_first[poly.n] = acc;
    s_irregular = 1;
  }
  sync();
  const int n_outline = edge_first[poly.n];
  for (int j = tid; j < n_outline; j += nt) {
    int k = 0;
    while (edge_first[k + 1] <= j) ++k;
    const int i = j - edge_first[k];
    const int k1 = (k + 1) % poly.n;
    const int dx = poly.vx[k1] - poly.vx[k], dy = poly.vy[k1] - poly.vy[k];
    const int adx = abs(dx), ady = abs(dy);
    const int sxn = dx > 0 ? 1 : -1, syn = dy > 0 ? 1 : -1;
    int x = poly.vx[k], y = poly.vy[k];
    if (adx >= ady) {
      const int m = adx ? (adx / 2 + i * ady) / adx : 0;
      x += i * sxn;
      y += m * syn;
    } else {
      const int m = (ady / 2 + i * adx) / ady;
      y += i * syn;
      x += m * sxn;
    }
    cells[j] = (uint32_t)x | ((uint32_t)y << 16);
  }
  sync();
  int min_x = poly.vx[0], max_x = poly.vx[0];
  for (int k = 1; k < poly.n; ++k) { min_x = min(min_x, poly.vx[k]); max_x = max(max_x, poly.vx[k]); }
  const int W = max_x - min_x + 1;
  if (W >= 2 && 3 * W <= capacity) {  // uniform
    int* colmin = reinterpret_cast<int*>(sorted);
    int* colmax = colmin + W;
    int* colcnt = colmax + W;
    for (int c = tid; c < W; c += nt) { colmin[c] = 0x7fffffff; colmax[c] = -1; colcnt[c] = 0; }
    if (tid == 0) s_irregular = 0;
    sync();
    for (int j = tid; j < n_outline; j += nt) {
      const int c = (int)(cells[j] & 0xffffu) - min_x, y = (int)(cells[j] >> 16);
      atomicMin(&colmin[c], y);
      atomicMax(&colmax[c], y);
      atomicAdd(&colcnt[c], 1);
    }
    sync();
    for (int c = tid; c < W; c += nt)
      if (colcnt[c] < 2) s_irregular = 1;
    sync();
  }
  return s_irregular == 0;
}

// Second stage for regular outlines, by every thread of the CTA (behind a barrier after polygon_prepare)
// (tid of nt threads call; nt < 0: every thread of the CTA)
__device__ __forceinline__ void polygon_fill_regular(uint8_t* __restrict__ grid, unsigned pitch, const PolyArgs& poly,
                                                     uint8_t value, const uint32_t* cells, const uint32_t* sorted,
                                                     int tid = -1, int nt = -1) {
  if (nt < 0) { tid = threadIdx.x; nt = blockDim.x; }
  int min_x = poly.vx[0], max_x = poly.vx[0], min_y = poly.vy[0], max_y = poly.vy[0], n_outline = 0;
  for (int k = 0; k < poly.n; ++k) {
    const int k1 = (k + 1) % poly.n;
    min_x = min(min_x, poly.vx[k]); max_x = max(max_x, poly.vx[k]);
    min_y = min(min_y, poly.vy[k]); max_y = max(max_y, poly.vy[k]);
    n_outline += max(abs(poly.vx[k1] - poly.vx[k]), abs(poly.vy[k1] - poly.vy[k])) + 1;
  }
  const int W = max_x - min_x + 1, H = max_y - min_y + 1;
  const int* colmin = reinterpret_cast<const int*>(sorted);
  const int* colmax = colmin + W;
  for (int j = tid; j < n_outline; j += nt) grid[(size_t)(cells[j] >> 16) * pitch + (cells[j] & 0xffffu)] = value;
  for (int j = tid; j < W * H; j += nt) {
    const int c = j % W, y = min_y + j / W;
    if (y >= colmin[c] && y < colmax[c]) grid[(size_t)y * pitch + (min_x + c)] = value;
  }
}

// What is left for outlines that are not regular (degenerate footprints): the reference's walk replayed verbatim.
// `cells` holds the outline (polygon_prepare); every thread of the CTA calls.
// (tid of nt threads call, synchronising on named barrier 1 with nt participants; nt < 0: every thread of the CTA)
__device__ __forceinline__ void polygon_fill_irregular(uint8_t* __restrict__ grid, unsigned pitch, const PolyArgs& poly,
                                                       uint8_t value, uint32_t* cells, uint32_t* sorted, int capacity,
                                                       int tid = -1, int nt = -1) {
  __shared__ int n_total;
  const bool named = nt >= 0;
  if (nt < 0) { tid = threadIdx.x; nt = blockDim.x; }
  auto sync = [&] {
    if (named) asm volatile("bar.sync 1, %0;" ::"r"(nt) : "memory");
    else __syncthreads();
  };
  int n_outline = 0;
  for (int k = 0; k < poly.n; ++k) {
    const int k1 = (k + 1) % poly.n;
    n_outline += max(abs(poly.vx[k1] - poly.vx[k]), abs(poly.vy[k1] - poly.vy[k])) + 1;
  }
  for (int j = tid; j < n_outline; j += nt) {  // stable rank by x
    const uint32_t xj = cells[j] & 0xffffu;
    int rank = 0;
    for (int i = 0; i < n_outline; ++i) {
      const uint32_t xi = cells[i] & 0xffffu;
      rank += (xi < xj) || (xi == xj && i < j);
    }
    sorted[rank] = cells[j];
  }
  sync();
  if (tid == 0) {
    int size = n_outline;
    auto X = [&](int i) { return (int)(sorted[i] & 0xffffu); };
    auto Y = [&](int i) { return (int)(sorted[i] >> 16); };
    int i = 0;
    const int min_x = X(0), max_x = X(size - 1);
    for (int x = min_x; x <= max_x; ++x) {
      if (i >= size - 1) break;
      int min_y, max_y;
      if (Y(i) < Y(i + 1)) { min_y = Y(i); max_y = Y(i + 1); }
      else { min_y = Y(i + 1); max_y = Y(i); }
      i += 2;
      while (i < size && X(i) == x) {
        if (Y(i) < min_y) min_y = Y(i);
        else if (Y(i) > max_y) max_y = Y(i);
        ++i;
      }
      for (int y = min_y; y < max_y && size < capacity; ++y) sorted[size++] = (uint32_t)x | ((uint32_t)y << 16);
    }
    n_total = size;
  }
  sync();
  for (int j = tid; j < n_total; j += nt) {
    const uint32_t c = sorted[j];
    grid[(size_t)(c >> 16) * pitch + (c & 0xffffu)] = value;
  }
}

// The whole thing by one CTA (cells / sorted: `capacity` entries each)
__device__ __forceinline__ void polygon_clear_cta(uint8_t* __restrict__ grid, unsigned pitch, const PolyArgs& poly,
                                                  uint8_t value, uint32_t* cells, uint32_t* sorted, int capacity) {
  if (polygon_prepare<false>(poly, cells, sorted, capacity)) {
    polygon_fill_regular(grid, pitch, poly, value, cells, sorted);
    return;
  }
  __syncthreads();  // the scratch is reused by the walk
  polygon_fill_irregular(grid, pitch, poly, value, cells, sorted, capacity);
}

// ---------------------------------------------------------------------------------------------------------------
// Bounds pass of LayeredCostmap::updateMap (src/layered_costmap.cpp:96-135): walks the layers in plugin order,
// unions what each contributed (host-known boxes for grid layers / footprints, device-accumulated boxes for the
// observation kernels), applies InflationLayer::updateBounds (plugins/inflation_layer.cpp:125-158) with its
// device-resident last_* state, and converts to the cell window with worldToMapEnforceBounds (:228-262).
constexpr int kMaxLayers = 8;
struct BoundsLayer {
  int kind;  // 0 union-box layer (grid / obstacle), 2 inflation
  int flag;  // kind 0: host box present; kind 2: need_reinflation_
  double hx0, hy0, hx1, hy1;  // host-known box contribution (kind 0), inflation_radius_ in hx0 (kind 2)
};
struct BoundsArgs {
  int n_layers;
  BoundsLayer layer[kMaxLayers];
  Geom master;
  // host mirror (mirror_kernels.cuh): every cycle adds its window, grown by what inflation can write beyond it, to the
  // box of cells the master grid may have changed in since the mirror was last brought up to date
  DevWindow* mirror_dirty = nullptr;
  int mirror_pad = 0;  // cells: 2 x the largest cell inflation radius of the stack (writes reach window +- 2R)
};
struct InflationBoundsState {
  double last_min_x, last_min_y, last_max_x, last_max_y;
};
__device__ __forceinline__ void finalize_bounds(const BoundsArgs& a, DevBox* boxes, InflationBoundsState* infl,
                                                DevWindow* win) {  // one thread
  double minx = 1e30, miny = 1e30, maxx = -1e30, maxy = -1e30;
  for (int l = 0; l < a.n_layers; ++l) {
    const BoundsLayer& L = a.layer[l];
    if (L.kind == 0) {
      if (L.flag) {
        minx = fmin(minx, L.hx0); miny = fmin(miny, L.hy0);
        maxx = fmax(maxx, L.hx1); maxy = fmax(maxy, L.hy1);
      }
      // accumulated with atomics by other CTAs: read past L1
      DevBox b;
      b.minx = __ldcg(&boxes[l].minx); b.miny = __ldcg(&boxes[l].miny);
      b.maxx = __ldcg(&boxes[l].maxx); b.maxy = __ldcg(&boxes[l].maxy);
      if (b.maxx != 0ull) {  // something was touched on the device this cycle
        minx = fmin(minx, dec_double(b.minx)); miny = fmin(miny, dec_double(b.miny));
        maxx = fmax(maxx, dec_double(b.maxx)); maxy = fmax(maxy, dec_double(b.maxy));
      }
      boxes[l] = DevBox{~0ull, ~0ull, 0ull, 0ull};  // re-armed for the next cycle
    } else if (L.kind == 2) {
      InflationBoundsState& s = infl[l];
      const double fmaxf_ = 3.40282346638528859811704183484516925e+38;  // std::numeric_limits<float>::max()
      if (L.flag) {
        s.last_min_x = minx; s.last_min_y = miny; s.last_max_x = maxx; s.last_max_y = maxy;
        minx = -fmaxf_; miny = -fmaxf_; maxx = fmaxf_; maxy = fmaxf_;
      } else {
        const double tx0 = s.last_min_x, ty0 = s.last_min_y, tx1 = s.last_max_x, ty1 = s.last_max_y;
        s.last_min_x = minx; s.last_min_y = miny; s.last_max_x = maxx; s.last_max_y = maxy;
        minx = fmin(tx0, minx) - L.hx0;
        miny = fmin(ty0, miny) - L.hx0;
        maxx = fmax(tx1, maxx) + L.hx0;
        maxy = fmax(ty1, maxy) + L.hx0;
      }
    }
  }
  const Geom& g = a.master;
  auto enforce = [&](double w, double origin, unsigned size) -> int {
    if (w < origin) return 0;
    if (w > g.res * (size - 1) + origin) return (int)(size - 1);
    return (int)((w - origin) / g.res);
  };
  int x0 = enforce(minx, g.ox, g.sx), y0 = enforce(miny, g.oy, g.sy);
  int xn = enforce(maxx, g.ox, g.sx), yn = enforce(maxy, g.oy, g.sy);
  x0 = max(0, x0);
  xn = min((int)g.sx, xn + 1);
  y0 = max(0, y0);
  yn = min((int)g.sy, yn + 1);
  win->x0 = x0; win->xn = xn; win->y0 = y0; win->yn = yn;
  win->valid = !(xn < x0 || yn < y0);
  if (a.mirror_dirty && win->valid) {
    DevWindow& d = *a.mirror_dirty;
    const int p = a.mirror_pad;
    const int dx0 = max(0, x0 - p), dxn = min((int)g.sx, xn + p), dy0 = max(0, y0 - p), dyn = min((int)g.sy, yn + p);
    if (d.valid) {
      d.x0 = min(d.x0, dx0); d.xn = max(d.xn, dxn); d.y0 = min(d.y0, dy0); d.yn = max(d.yn, dyn);
    } else {
      d.x0 = dx0; d.xn = dxn; d.y0 = dy0; d.yn = dyn;
      d.valid = 1;
    }
  }
}

__global__ void k_finalize_bounds(BoundsArgs a, DevBox* boxes, InflationBoundsState* infl, DevWindow* win) {
  if (threadIdx.x == 0 && blockIdx.x == 0) finalize_bounds(a, boxes, infl, win);
}

// stand-alone polygon rasteriser for footprints too large for k_obstacle_update's static scratch
__global__ void k_polygon_clear(uint8_t* __restrict__ grid, unsigned pitch, PolyArgs poly, uint8_t value) {
  extern __shared__ uint32_t poly_smem[];
  polygon_clear_cta(grid, pitch, poly, value, poly_smem, poly_smem + kPolyMaxCells, kPolyMaxCells);
}

// ---------------------------------------------------------------------------------------------------------------
// One launch per obstacle layer and cycle: ObstacleLayer::updateBounds + the footprint part of updateCosts
// (plugins/obstacle_layer.cpp:340-448).  Every CTA ray-traces 8 rays (one warp each).  The reference clears ALL rays
// before it marks ANY point (:362-365 then :368), so the CTA that finishes last (ticket + __threadfence, no
// spinning) marks the points, clears the footprint polygon (what updateCosts does first, on the same grid) and, for
// the last observation-driven layer of the stack, runs the bounds pass that needs every layer's accumulated box.
constexpr int kInlineObs = 16;
struct ObstacleArgs {
  uint8_t* grid;
  Geom g;
  const DevObs* clear;
  const DevObs* mark;
  DevObs clear_inline[kInlineObs], mark_inline[kInlineObs];  // used when n_clear / n_mark <= kInlineObs
  const float* xyz;
  int n_clear, total_rays, n_mark, total_marks;
  double max_obstacle_height;
  DevBox* box;  // this layer's box
  long long* mark_cells;  // total_marks entries of scratch
  unsigned* ticket;
  int do_poly;
  PolyArgs poly;
  int do_finalize;
  BoundsArgs ba;
  DevBox* boxes;
  InflationBoundsState* infl;
  DevWindow* win;
  uint8_t* tile_used = nullptr;  // MergeLayers::used of this layer (nullable)
  // set to done_epoch (release, gpu scope) by the last CTA as soon as the layer grid is complete (rays cleared, marks
  // stored, footprint cleared), before the bounds pass: early-mode k_merge_seed tiles in the rays' box wait for this
  // word instead of for the end of the kernel
  unsigned* done_flag = nullptr;
  unsigned done_epoch = 0;
};
constexpr int kObstacleThreads = 256;
// k_obstacle_update: eight ray warps and one more warp that runs this CTA's share of the marking tests next to them
// (two cold instruction streams side by side instead of one after the other)
constexpr int kObstacleRayWarps = 8, kObstacleUpdateThreads = 32 * (kObstacleRayWarps + 1);

__global__ void __maxnreg__(48) k_obstacle_update(ObstacleArgs a) {
  __shared__ uint32_t poly_cells[kPolySmallCells], poly_sorted[kPolySmallCells];
  __shared__ unsigned long long s_box[kObstacleRayWarps + 1][4];
  __shared__ bool s_last;
  const int lane = threadIdx.x & 31, cta_warp = threadIdx.x >> 5;
  cudaTriggerProgrammaticLaunchCompletion();  // k_merge_seed may be scheduled behind us; it waits for our completion
  // the observation tables travel in the kernel parameters when they fit (no dependent global loads to find a ray's
  // observation), else they are read from device memory
  const DevObs* clear_tab = a.n_clear <= kInlineObs ? a.clear_inline : a.clear;
  const DevObs* mark_tab = a.n_mark <= kInlineObs ? a.mark_inline : a.mark;
  BoxAcc acc;
  if (cta_warp < kObstacleRayWarps) {
    raytrace_ray(a.grid, a.g, clear_tab, a.n_clear, a.xyz, a.total_rays, acc, blockIdx.x * kObstacleRayWarps + cta_warp, lane);
    // (a ray touches its end point from lane 0 only: nothing to reduce within the warp)
    if (lane == 0) { s_box[cta_warp][0] = acc.minx; s_box[cta_warp][1] = acc.miny; s_box[cta_warp][2] = acc.maxx; s_box[cta_warp][3] = acc.maxy; }
  } else {  // this CTA's share of the marking tests
    const int per_cta = (a.total_marks + gridDim.x - 1) / gridDim.x;
    for (int i = lane; i < per_cta; i += 32) {
      const int t = blockIdx.x * per_cta + i;
      if (t < a.total_marks)
        mark_prepare(a.g, mark_tab, a.n_mark, a.xyz, a.max_obstacle_height, acc, a.mark_cells, t);
    }
    acc.reduce_warp();
    if (lane == 0) { s_box[cta_warp][0] = acc.minx; s_box[cta_warp][1] = acc.miny; s_box[cta_warp][2] = acc.maxx; s_box[cta_warp][3] = acc.maxy; }
  }
  __syncthreads();
  BoxAcc::flush_rows(a.box, s_box, kObstacleRayWarps + 1);
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = atomicAdd(a.ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  // The last CTA: ray warps 0..6 store the marks, the ninth warp prepares the footprint polygon meanwhile, both then
  // store the polygon (behind the marks: named barrier 1 over those eight warps) and release the "layer grids complete"
  // word; ray warp 7 runs the bounds pass next to all that (it only reads the layers' boxes, complete since the last
  // ticket) -- a single thread's ~1500 dependent instructions that would otherwise end the kernel 9 us later.
  constexpr int kTailThreads = 32 * kObstacleRayWarps;  // warps 0..6 and 8
  __shared__ bool s_regular;
  if (cta_warp == kObstacleRayWarps - 1) {
    if (lane == 0 && a.do_finalize) finalize_bounds(a.ba, a.boxes, a.infl, a.win);
    return;
  }
  const int ttid = cta_warp < kObstacleRayWarps ? (int)threadIdx.x : (int)threadIdx.x - 32;  // 0 .. kTailThreads - 1
  if (cta_warp < kObstacleRayWarps) {
    mark_commit_cta(a.grid, a.mark_cells, a.total_marks, a.tile_used, a.g.pitch, 32 * (kObstacleRayWarps - 1));
  } else if (a.do_poly) {
    const bool regular = polygon_prepare<true>(a.poly, poly_cells, poly_sorted, kPolySmallCells);
    if (lane == 0) s_regular = regular;
  }
  asm volatile("bar.sync 1, %0;" ::"n"(kTailThreads) : "memory");
  if (a.do_poly) {
    if (s_regular) polygon_fill_regular(a.grid, a.g.pitch, a.poly, kFree, poly_cells, poly_sorted, ttid, kTailThreads);
    else polygon_fill_irregular(a.grid, a.g.pitch, a.poly, kFree, poly_cells, poly_sorted, kPolySmallCells, ttid, kTailThreads);
  }
  if (a.done_flag) {
    asm volatile("bar.sync 1, %0;" ::"n"(kTailThreads) : "memory");  // every mark / polygon store before the release
    if (threadIdx.x == 0) {
      __threadfence();
      asm volatile("st.release.gpu.u32 [%0], %1;" ::"l"(a.done_flag), "r"(a.done_epoch) : "memory");
    }
  }
  if (threadIdx.x == 0) *a.ticket = 0;  // re-armed for the next cycle
}

// Costmap2DPublisher's cost -> occupancy translation (src/costmap_2d_publisher.cpp:56-71, applied per cell in
// prepareGrid :95-113 and publishCostmap :139-152), fused with the packing of a window for the download:
// 0 -> 0, 253 -> 99, 254 -> 100, 255 -> -1, 1..252 -> 1 + 97 * (v - 1) / 251.
// Sixteen cells per thread: one aligned 16-byte load of the master row, a 256-entry table in shared memory, one
// 16-byte store when the packed output is aligned there (always for whole-row windows of maps whose width is a multiple
// of 16), byte stores at the window's edges otherwise.
__global__ void __launch_bounds__(256) k_translate_window(const uint8_t* __restrict__ master, unsigned pitch, int x0, int y0,
                                                           int w, int h, int8_t* __restrict__ out) {
  __shared__ uint8_t lut[256];
  {
    const int v = threadIdx.x;
    int o;
    if (v == 0) o = 0;
    else if (v == kInscribed) o = 99;
    else if (v == kLethal) o = 100;
    else if (v == kNoInfo) o = -1;
    else o = 1 + (97 * (v - 1)) / 251;
    lut[v] = (uint8_t)(int8_t)o;
  }
  __syncthreads();
  const int y = blockIdx.y;
  const int gx = ((x0 >> 4) + blockIdx.x * blockDim.x + threadIdx.x) << 4;  // first cell of my 16-cell group of the row
  if (y >= h || gx >= x0 + w) return;
  const uint4 v = *reinterpret_cast<const uint4*>(master + (size_t)(y0 + y) * pitch + gx);
  const uint32_t in[4] = {v.x, v.y, v.z, v.w};
  uint32_t o[4];
#pragma unroll
  for (int k = 0; k < 4; ++k)
    o[k] = (uint32_t)lut[in[k] & 0xffu] | ((uint32_t)lut[(in[k] >> 8) & 0xffu] << 8) |
           ((uint32_t)lut[(in[k] >> 16) & 0xffu] << 16) | ((uint32_t)lut[in[k] >> 24] << 24);
  int8_t* dst = out + (size_t)y * w + (gx - x0);  // (may point before `out` for the first group: guarded below)
  if (gx >= x0 && gx + 16 <= x0 + w && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
    *reinterpret_cast<uint4*>(dst) = make_uint4(o[0], o[1], o[2], o[3]);
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int cx = gx + i;
      if (cx >= x0 && cx < x0 + w) out[(size_t)y * w + (cx - x0)] = (int8_t)(o[i >> 2] >> (8 * (i & 3)));
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// VoxelLayer (plugins/voxel_layer.cpp) on voxel_grid::VoxelGrid columns (voxel_grid/include/voxel_grid/voxel_grid.h):
// one uint32 per cell, bit z = "unknown or marked", bit z + 16 = "marked".  The column array shares the 2-D layer
// grid's indexing (offset = y * pitch + x).
//
// The reference clears ray by ray and re-derives the 2-D cell after every cleared voxel (ClearVoxelInMap,
// voxel_grid.h:335-372).  Clearing only ever removes bits and both threshold tests are monotone in the bits, so the
// value a cell ends with is the rule applied to the column AFTER ALL clears (untouched when the marked count is still
// above its threshold).  Hence two launches: k_voxel_clear does every ray's atomicAnd (and the marking tests, into a
// scratch list); k_voxel_commit walks the rays again and writes the 2-D cells from the final columns, then its last
// CTA commits the marks (markVoxelInMap :98-118: all marking comes after all clearing, voxel_layer.cpp:136-177),
// clears the footprint polygon and finalises the bounds exactly like k_obstacle_update.
struct VoxelGeom {
  double origin_z, z_resolution;
  unsigned size_z, unknown_threshold, mark_threshold;
};

__device__ __forceinline__ bool bits_below_threshold(unsigned n, unsigned thr) { return (unsigned)__popc(n) <= thr; }

// VoxelLayer::worldToMap3DFloat (voxel_layer.h:103-115)
__device__ __forceinline__ bool world_to_map_3d_float(const Geom& g, const VoxelGeom& v, double wx, double wy, double wz,
                                                      double& mx, double& my, double& mz) {
  if (wx < g.ox || wy < g.oy || wz < v.origin_z) return false;
  mx = (wx - g.ox) / g.res;
  my = (wy - g.oy) / g.res;
  mz = (wz - v.origin_z) / v.z_resolution;
  return mx < g.sx && my < g.sy && mz < v.size_z;
}

// One ray of VoxelLayer::raytraceFreespace (voxel_layer.cpp:262-350) reduced to what VoxelGrid::raytraceLine /
// bresenham3D (voxel_grid.h:226-297) walks: start cell, dominant-axis length and the closed-form minor-axis steps.
struct VoxelRay {
  bool valid;
  long long start;  // y0 * pitch + x0
  int z0;
  unsigned da, db, dc, end;  // dominant / minor extents, number of bresenham iterations (cells 0 .. end are visited)
  int off_a, off_b, off_c;   // grid offsets per step; 0 for the axis that moves the z mask
  int dz_a, dz_b, dz_c;      // z steps per step of that axis (+-1 on the z axis, else 0)
  double ex, ey;             // updateRaytraceBounds end point
};

__device__ VoxelRay voxel_ray_setup(const Geom& g, const VoxelGeom& v, const DevObs& o, const float* __restrict__ xyz,
                                    int point, double max_obstacle_height) {
  VoxelRay r;
  r.valid = false;
  double sensor_x, sensor_y, sensor_z;
  const double ox = o.ox, oy = o.oy, oz = o.oz;
  if (!world_to_map_3d_float(g, v, ox, oy, oz, sensor_x, sensor_y, sensor_z)) return r;  // whole observation skipped
  const double map_end_x = g.ox + (g.sx - 1 + 0.5) * g.res, map_end_y = g.oy + (g.sy - 1 + 0.5) * g.res;  // getSizeInMeters
  double wpx = xyz[3 * (size_t)point], wpy = xyz[3 * (size_t)point + 1], wpz = xyz[3 * (size_t)point + 2];
  if (wpx != wpx) return r;  // NaN: a ray dropped by the on-device scan ingest (k_project_scans)
  const double distance = sqrt((wpx - ox) * (wpx - ox) + (wpy - oy) * (wpy - oy) + (wpz - oz) * (wpz - oz));
  double scaling_fact = 1.0;
  scaling_fact = fmax(fmin(scaling_fact, (distance - 2 * g.res) / distance), 0.0);
  wpx = scaling_fact * (wpx - ox) + ox;
  wpy = scaling_fact * (wpy - oy) + oy;
  wpz = scaling_fact * (wpz - oz) + oz;
  const double a = wpx - ox, b = wpy - oy, c = wpz - oz;
  double t = 1.0;
  if (wpz > max_obstacle_height) t = fmax(0.0, fmin(t, (max_obstacle_height - 0.01 - oz) / c));
  else if (wpz < v.origin_z) t = fmin(t, (v.origin_z - oz) / c);
  if (wpx < g.ox) t = fmin(t, (g.ox - ox) / a);
  if (wpy < g.oy) t = fmin(t, (g.oy - oy) / b);
  if (wpx > map_end_x) t = fmin(t, (map_end_x - ox) / a);
  if (wpy > map_end_y) t = fmin(t, (map_end_y - oy) / b);
  wpx = ox + a * t;
  wpy = oy + b * t;
  wpz = oz + c * t;
  double px, py, pz;
  if (!world_to_map_3d_float(g, v, wpx, wpy, wpz, px, py, pz)) return r;
  // clearVoxelLineInMap's own end-point test (voxel_grid.cpp:133-137) holds by construction of both points
  const unsigned cell_range = (unsigned)fmax(0.0, ceil(o.raytrace_range / g.res));  // cellDistance
  const int dx = (int)px - (int)sensor_x, dy = (int)py - (int)sensor_y, dz = (int)pz - (int)sensor_z;
  const unsigned adx = abs(dx), ady = abs(dy), adz = abs(dz);
  const int off_dx = dx > 0 ? 1 : -1, off_dy = (dy > 0 ? 1 : -1) * (int)g.pitch, sgn_dz = dz > 0 ? 1 : -1;
  const double dist = sqrt((sensor_x - px) * (sensor_x - px) + (sensor_y - py) * (sensor_y - py) +
                           (sensor_z - pz) * (sensor_z - pz));
  const double scale = fmin(1.0, cell_range / dist);
  r.start = (long long)(unsigned)sensor_y * g.pitch + (unsigned)sensor_x;
  r.z0 = (int)(unsigned)sensor_z;
  r.dz_a = r.dz_b = r.dz_c = 0;
  if (adx >= max(ady, adz)) {
    r.da = adx; r.db = ady; r.dc = adz;
    r.off_a = off_dx; r.off_b = off_dy; r.off_c = 0; r.dz_c = sgn_dz;
  } else if (ady >= adz) {
    r.da = ady; r.db = adx; r.dc = adz;
    r.off_a = off_dy; r.off_b = off_dx; r.off_c = 0; r.dz_c = sgn_dz;
  } else {
    r.da = adz; r.db = adx; r.dc = ady;
    r.off_a = 0; r.dz_a = sgn_dz; r.off_b = off_dx; r.off_c = off_dy;
  }
  r.end = min((unsigned)(scale * r.da), r.da);
  const double ddx = wpx - ox, ddy = wpy - oy;  // updateRaytraceBounds (obstacle_layer.cpp:602-610)
  const double s2 = fmin(1.0, o.raytrace_range / hypot(ddx, ddy));
  r.ex = ox + ddx * s2;
  r.ey = oy + ddy * s2;
  r.valid = true;
  return r;
}

// voxel i of the ray (0 <= i <= end): after i iterations the error accumulators of bresenham3D have produced
// floor((da/2 + i*db) / da) steps on axis b and likewise on c
__device__ __forceinline__ void voxel_ray_cell(const VoxelRay& r, unsigned i, long long& offset, int& z) {
  const unsigned half = r.da / 2;
  const unsigned nb = r.da ? (unsigned)((half + (unsigned long long)i * r.db) / r.da) : 0u;
  const unsigned nc = r.da ? (unsigned)((half + (unsigned long long)i * r.dc) / r.da) : 0u;
  offset = r.start + (long long)i * r.off_a + (long long)nb * r.off_b + (long long)nc * r.off_c;
  z = r.z0 + (int)i * r.dz_a + (int)nb * r.dz_b + (int)nc * r.dz_c;
}

struct VoxelArgs {
  uint8_t* grid;   // the layer's 2-D grid
  uint32_t* vox;   // the columns, same indexing
  Geom g;
  VoxelGeom v;
  const DevObs* clear;
  const DevObs* mark;
  const float* xyz;
  int n_clear, total_rays, n_mark, total_marks;
  double max_obstacle_height;
  DevBox* box;
  long long* mark_cells;  // total_marks entries: (offset << 5) | z, or -1
  unsigned* ticket;
  int do_poly;
  PolyArgs poly;
  int do_finalize;
  BoundsArgs ba;
  DevBox* boxes;
  InflationBoundsState* infl;
  DevWindow* win;
};

__device__ __forceinline__ const DevObs& obs_of(const DevObs* tab, int n, int index, int& local) {
  int k = 0;
  while (k + 1 < n && tab[k + 1].first_ray <= index) ++k;
  local = tab[k].first_point + (index - tab[k].first_ray);
  return tab[k];
}

// The per-ray, per-point steps of the VoxelLayer, shared by the single costmap (k_voxel_clear, k_voxel_commit: columns
// in global memory, g.pitch = the grid's pitch) and the sensing fleet (k_fleet_costmap_voxel: columns and 2-D grid in
// shared memory, g.pitch = their shared row pitch).  `ray` / `t` index the clearing / marking table `obs`.
//
// clearing: ray `ray`'s atomicAnd on the columns, one warp; lane 0 touches its updateRaytraceBounds end point
__device__ __forceinline__ void voxel_clear_ray(uint32_t* vox, const Geom& g, const VoxelGeom& v, const DevObs* obs,
                                                int n_obs, const float* __restrict__ xyz, double max_obstacle_height,
                                                BoxAcc& acc, int ray, int lane) {
  int point;
  const DevObs& o = obs_of(obs, n_obs, ray, point);
  const VoxelRay r = voxel_ray_setup(g, v, o, xyz, point, max_obstacle_height);
  if (r.valid) {
    for (unsigned i = lane; i <= r.end; i += 32) {
      long long off;
      int z;
      voxel_ray_cell(r, i, off, z);
      atomicAnd(&vox[off], ~(0x00010001u << z));  // clear unknown and clear cell
    }
    if (lane == 0) acc.touch(r.ex, r.ey);
  }
}

// commit: the 2-D cells of ray `ray` from the final columns (every clear of the cycle done), one warp
__device__ __forceinline__ void voxel_commit_ray(uint8_t* grid, const uint32_t* vox, const Geom& g, const VoxelGeom& v,
                                                 const DevObs* obs, int n_obs, const float* __restrict__ xyz,
                                                 double max_obstacle_height, int ray, int lane) {
  int point;
  const DevObs& o = obs_of(obs, n_obs, ray, point);
  const VoxelRay r = voxel_ray_setup(g, v, o, xyz, point, max_obstacle_height);
  if (r.valid) {
    for (unsigned i = lane; i <= r.end; i += 32) {
      long long off;
      int z;
      voxel_ray_cell(r, i, off, z);
      const uint32_t col = vox[off];
      const unsigned unknown_bits = (uint16_t)(col >> 16) ^ (uint16_t)col, marked_bits = col >> 16;
      if (bits_below_threshold(marked_bits, v.mark_threshold))
        grid[off] = bits_below_threshold(unknown_bits, v.unknown_threshold) ? kFree : kNoInfo;
    }
  }
}

// marking test of point t (voxel_layer.cpp:136-177): (offset << 5) | z of its voxel, or -1; touches the point
__device__ __forceinline__ long long voxel_mark_cell(const Geom& g, const VoxelGeom& v, const DevObs* obs, int n_obs,
                                                     const float* __restrict__ xyz, double max_obstacle_height,
                                                     BoxAcc& acc, int t) {
  int point;
  const DevObs& o = obs_of(obs, n_obs, t, point);
  const float fx = xyz[3 * (size_t)point], fy = xyz[3 * (size_t)point + 1], fz = xyz[3 * (size_t)point + 2];
  long long cell = -1;
  if (fx == fx && !(fz > max_obstacle_height)) {  // NaN: dropped by the scan ingest
    const double sq_dist = (fx - o.ox) * (fx - o.ox) + (fy - o.oy) * (fy - o.oy) + (fz - o.oz) * (fz - o.oz);
    if (!(sq_dist >= o.obstacle_range * o.obstacle_range)) {
      const double wz = fz < v.origin_z ? v.origin_z : (double)fz;
      const double wx = fx, wy = fy;
      if (!(wx < g.ox || wy < g.oy || wz < v.origin_z)) {  // worldToMap3D, voxel_layer.h:117-130
        const unsigned mx = (unsigned)(int)((wx - g.ox) / g.res), my = (unsigned)(int)((wy - g.oy) / g.res),
                       mz = (unsigned)(int)((wz - v.origin_z) / v.z_resolution);
        if (mx < g.sx && my < g.sy && mz < v.size_z) {
          cell = (((long long)my * g.pitch + mx) << 5) | mz;
          acc.touch((double)fx, (double)fy);  // every marked voxel touches, whatever mark_threshold
        }
      }
    }
  }
  return cell;
}

// markVoxelInMap + LETHAL_OBSTACLE of one voxel_mark_cell result (>= 0), after every clear and commit of the cycle
__device__ __forceinline__ void voxel_mark_commit(uint8_t* grid, uint32_t* vox, unsigned mark_threshold, long long cell) {
  const long long off = cell >> 5;
  const unsigned z = (unsigned)(cell & 31);
  if (mark_threshold == 0) {  // one marked voxel already exceeds the threshold: no need to wait for the old column
    atomicOr(&vox[off], 0x00010001u << z);
    grid[off] = kLethal;
  } else {
    const uint32_t col = atomicOr(&vox[off], 0x00010001u << z) | (0x00010001u << z);
    if (!bits_below_threshold(col >> 16, mark_threshold)) grid[off] = kLethal;
  }
}

__global__ void __launch_bounds__(kObstacleThreads) k_voxel_clear(VoxelArgs a) {
  __shared__ unsigned long long s_box[kObstacleThreads / 32][4];
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * kObstacleThreads + threadIdx.x) >> 5;
  BoxAcc acc;
  if (warp < a.total_rays)
    voxel_clear_ray(a.vox, a.g, a.v, a.clear, a.n_clear, a.xyz, a.max_obstacle_height, acc, warp, lane);
  {  // this CTA's share of the marking tests
    const int per_cta = (a.total_marks + gridDim.x - 1) / gridDim.x;
    for (int i = threadIdx.x; i < per_cta; i += kObstacleThreads) {
      const int t = blockIdx.x * per_cta + i;
      if (t >= a.total_marks) continue;
      a.mark_cells[t] = voxel_mark_cell(a.g, a.v, a.mark, a.n_mark, a.xyz, a.max_obstacle_height, acc, t);
    }
  }
  acc.flush_cta(a.box, s_box);
}

__global__ void __launch_bounds__(kObstacleThreads) k_voxel_commit(VoxelArgs a) {
  __shared__ uint32_t poly_cells[kPolySmallCells], poly_sorted[kPolySmallCells];
  __shared__ bool s_last;
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * kObstacleThreads + threadIdx.x) >> 5;
  cudaTriggerProgrammaticLaunchCompletion();
  // final columns: every clear of this cycle happened in k_voxel_clear
  if (warp < a.total_rays)
    voxel_commit_ray(a.grid, a.vox, a.g, a.v, a.clear, a.n_clear, a.xyz, a.max_obstacle_height, warp, lane);
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = atomicAdd(a.ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  for (int t = threadIdx.x; t < a.total_marks; t += kObstacleThreads) {  // markVoxelInMap + LETHAL_OBSTACLE
    const long long cell = a.mark_cells[t];
    if (cell >= 0) voxel_mark_commit(a.grid, a.vox, a.v.mark_threshold, cell);
  }
  __syncthreads();
  if (a.do_poly) polygon_clear_cta(a.grid, a.g.pitch, a.poly, kFree, poly_cells, poly_sorted, kPolySmallCells);
  if (threadIdx.x == 0) {
    *a.ticket = 0;
    if (a.do_finalize) {
      __threadfence();
      finalize_bounds(a.ba, a.boxes, a.infl, a.win);
    }
  }
}

// VoxelLayer::updateOrigin's column part (voxel_layer.cpp:371-438): same shift as k_shift_grid, unknown columns elsewhere
__global__ void k_shift_voxels(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, unsigned sx, unsigned sy,
                               unsigned pitch, int cell_ox, int cell_oy) {
  unsigned x = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned y = blockIdx.y;
  if (x >= pitch || y >= sy) return;
  uint32_t v = 0x0000ffffu;
  long long ox = (long long)x + cell_ox, oy = (long long)y + cell_oy;
  if (x < sx && ox >= 0 && ox < (long long)sx && oy >= 0 && oy < (long long)sy) v = src[(size_t)oy * pitch + ox];
  dst[(size_t)y * pitch + x] = v;
}

__global__ void k_set_window(DevWindow* win, int x0, int xn, int y0, int yn) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    win->x0 = x0; win->xn = xn; win->y0 = y0; win->yn = yn;
    win->valid = !(xn < x0 || yn < y0);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// The cost sweep of a cycle: Costmap2D::resetMap (src/costmap_2d.cpp:93-99), the CostmapLayer merge policies
// (src/costmap_layer.cpp:62-157) of every enabled cost layer in plugin order, and InflationLayer::updateCosts
// (plugins/inflation_layer.cpp:172-266), fused into ONE pass over the master grid.
//
// Inside the window a cell's pre-inflation value is a pure function of the layer grids (reset -> merges), so a tile
// recomputes it for its halo instead of reading what a neighbouring CTA writes; outside the window it is the
// previous master value, whose "== LETHAL" predicate inflation can never change.  Inflation is evaluated as the
// exact windowed nearest-seed distance: seeds are the LETHAL cells of (window +- R, clamped), a cell within
// hypot <= R of a seed gets max(old, table[d]) (NO_INFORMATION is replaced only by costs >= INSCRIBED), cells may be
// written up to window +- 2R exactly like the reference's unclamped propagation.  d^2 = dy^2 + hx^2 with hx the
// per-row distance to the nearest seed, taken from per-row seed bitmasks with clz/ffs.
struct MergeLayers {
  int n;
  const uint8_t* grid[kMaxLayers];
  int policy[kMaxLayers];
  // Per layer, nullable: one byte per k_merge_seed sub-tile (256 x 32 cells, row-major over ceil(pitch / 256) columns), 0 as
  // long as every cell of the tile still holds FREE_SPACE.  An obstacle layer is FREE_SPACE almost everywhere (marks
  // exist where scans ever ended): the merge takes zeros for such a tile instead of reading 8 KB of them from HBM.
  const uint8_t* used[kMaxLayers] = {};
};
struct UpdateArgs {
  uint8_t* master;
  unsigned sx, sy, pitch;
  uint8_t def;
  int do_reset;
  const DevWindow* win;
  MergeLayers ml;
  int R;                   // 0: no inflation in this pass
  const uint8_t* cost_d2;  // R*R+1 entries: cost by squared cell distance
  int reach2;              // largest squared distance whose cost is not 0 (a cost of 0 never changes a cell)
  // early != 0: the host knows this cycle's window is the whole map and that the kernel launched just before the sweep
  // (k_obstacle_update) writes layer cells only inside [ex0, exn) x [ey0, eyn): see k_merge_seed
  int early = 0, ex0 = 0, exn = 0, ey0 = 0, eyn = 0;
  // early mode: the word the last k_obstacle_update sets to obst_epoch once the layer grids hold everything this cycle
  // writes to them (marks and footprint included) -- before it finalises the bounds; null: wait for the whole kernel
  const unsigned* obst_flag = nullptr;
  unsigned obst_epoch = 0;
};

__device__ __forceinline__ uint8_t apply_policy(uint8_t m, uint8_t v, int policy) {
  switch (policy) {
    case NAVGPU_TRUE_OVERWRITE: return v;
    case NAVGPU_OVERWRITE: return v != kNoInfo ? v : m;
    case NAVGPU_MAX: return (v == kNoInfo) ? m : ((m == kNoInfo || m < v) ? v : m);
    case NAVGPU_ADDITION: {
      if (v == kNoInfo) return m;
      if (m == kNoInfo) return v;
      const int sum = (int)m + (int)v;
      return sum >= kInscribed ? (uint8_t)(kInscribed - 1) : (uint8_t)sum;
    }
    default: return m;
  }
}

__device__ __forceinline__ uint8_t inflate_combine(uint8_t old, uint8_t cost) {  // inflation_layer.cpp:249-254
  if (old == kNoInfo && cost >= kInscribed) return cost;
  return old > cost ? old : cost;
}

constexpr int kTX = 128, kTY = 32, kUpdateThreads = 256;

// generic kernel: any R <= 254
__global__ void __launch_bounds__(kUpdateThreads) k_update_costs(UpdateArgs a) {
  extern __shared__ __align__(16) uint8_t smem[];
  const DevWindow w = *a.win;
  if (!w.valid) return;
  const int R = a.R;
  const int tx0 = blockIdx.x * kTX, ty0 = blockIdx.y * kTY;
  // affected region: the window itself, plus 2R around it when inflating
  if (tx0 >= w.xn + 2 * R || tx0 + kTX <= w.x0 - 2 * R || ty0 >= w.yn + 2 * R || ty0 + kTY <= w.y0 - 2 * R) return;

  const int HX = (R + 7) & ~7;            // x halo rounded to the 8-cell load granularity
  const int groups = (kTX + 2 * HX) / 8;  // 8-cell groups per region row
  const int rows = kTY + 2 * R;
  const int bits_pitch = (groups + 3) & ~3;  // bytes per row of the seed bitmask, whole 32-bit words
  uint8_t* tile = smem;                                   // kTY x kTX pre-inflation values, then results
  uint8_t* bits = tile + kTX * kTY;                       // rows x bits_pitch
  uint8_t* hx = bits + ((rows * bits_pitch + 15) & ~15);  // rows x kTX horizontal distances
  uint8_t* table = hx + rows * kTX;                       // R*R+1
  const int tid = threadIdx.x;

  if (R > 0)
    for (int i = tid; i <= R * R; i += kUpdateThreads) table[i] = a.cost_d2[i];
  // seed region: window +- R clamped to the map (inflation_layer.cpp:203-211)
  const int sx0 = max(0, w.x0 - R), sxn = min((int)a.sx, w.xn + R);
  const int sy0 = max(0, w.y0 - R), syn = min((int)a.sy, w.yn + R);
  const int rx0 = tx0 - HX, ry0 = ty0 - R;

  // phase 1: pre-inflation values of the region, 8 cells per item
  for (int item = tid; item < rows * groups; item += kUpdateThreads) {
    const int row = item / groups, grp = item - row * groups;
    const int y = ry0 + row, x = rx0 + grp * 8;
    uint32_t seedbits = 0;
    const bool own_row = row >= R && row < R + kTY;
    if (y >= 0 && y < (int)a.sy && x >= 0 && x < (int)a.sx) {
      const size_t off = (size_t)y * a.pitch + x;
      const bool row_in = y >= w.y0 && y < w.yn;
      const bool any_in = row_in && x + 8 > w.x0 && x < w.xn;
      const bool all_in = row_in && x >= w.x0 && x + 8 <= w.xn;
      uint2 mv = make_uint2(0, 0);
      if (!(all_in && a.do_reset)) mv = *reinterpret_cast<const uint2*>(a.master + off);
      uint2 lv[kMaxLayers];
      if (any_in)
        for (int l = 0; l < a.ml.n; ++l) lv[l] = *reinterpret_cast<const uint2*>(a.ml.grid[l] + off);
      uint2 outv = make_uint2(0, 0);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int cx = x + i;
        const uint32_t mword = i < 4 ? mv.x : mv.y;
        uint8_t v = (uint8_t)(mword >> (8 * (i & 3)));
        const bool inwin = row_in && cx >= w.x0 && cx < w.xn;
        if (inwin) {
          if (a.do_reset) v = a.def;
          for (int l = 0; l < a.ml.n; ++l) {
            const uint32_t lword = i < 4 ? lv[l].x : lv[l].y;
            v = apply_policy(v, (uint8_t)(lword >> (8 * (i & 3))), a.ml.policy[l]);
          }
        }
        if (cx >= (int)a.sx) v = 0;
        if (v == kLethal && cx >= sx0 && cx < sxn && y >= sy0 && y < syn) seedbits |= 1u << i;
        if (i < 4) outv.x |= (uint32_t)v << (8 * i);
        else outv.y |= (uint32_t)v << (8 * (i - 4));
      }
      if (own_row && x >= tx0 && x < tx0 + kTX)
        *reinterpret_cast<uint2*>(tile + (row - R) * kTX + (x - tx0)) = outv;
    } else if (own_row && x >= tx0 && x < tx0 + kTX) {
      *reinterpret_cast<uint2*>(tile + (row - R) * kTX + (x - tx0)) = make_uint2(0, 0);
    }
    bits[row * bits_pitch + grp] = (uint8_t)seedbits;
  }
  // zero the pad bytes of each bitmask row so whole-word reads are clean
  for (int i = tid; i < rows * (bits_pitch - groups); i += kUpdateThreads) {
    const int row = i / (bits_pitch - groups), k = i - row * (bits_pitch - groups);
    bits[row * bits_pitch + groups + k] = 0;
  }
  __syncthreads();

  if (R > 0) {
    // phase 2: horizontal distance to the nearest seed of the same row, |dx| <= R (255 = none)
    const int nwords = bits_pitch / 4;
    for (int item = tid; item < rows * kTX; item += kUpdateThreads) {
      const int row = item / kTX, tx = item - row * kTX;
      const uint32_t* wrow = reinterpret_cast<const uint32_t*>(bits + row * bits_pitch);
      const int p = HX + tx;  // bit position of this cell in the row
      auto word = [&](int i) -> uint32_t { return (i < 0 || i >= nwords) ? 0u : wrow[i]; };
      auto window32 = [&](int q) -> uint32_t {  // bits q .. q+31
        const int wi = q >> 5, sh = q & 31;
        return __funnelshift_r(word(wi), word(wi + 1), sh);
      };
      int best = 255;
      for (int base = 0; base <= R; base += 32) {
        const uint32_t right = window32(p + base);       // bit k  <-> distance base + k
        const uint32_t left = window32(p - base - 31);   // bit 31-k <-> distance base + k
        int d = 255;
        if (right) d = base + (__ffs(right) - 1);
        if (left) d = min(d, base + __clz(left));
        if (d != 255) { best = d; break; }
      }
      hx[item] = (uint8_t)(best <= R ? best : 255);
    }
    __syncthreads();

    // phase 3: d^2 = min over dy of dy^2 + hx(y+dy)^2 ; one thread per column, 16 rows each
    const int tx = tid & (kTX - 1), half = tid / kTX;
    const int R2 = R * R;
    for (int r = half * (kTY / 2); r < (half + 1) * (kTY / 2); ++r) {
      int best = 0x7fffffff;
      const uint8_t* col = hx + (r + R) * kTX + tx;  // row of this cell inside the region
      for (int dy = -R; dy <= R; ++dy) {
        const int h = col[dy * kTX];
        const int d2 = (h == 255) ? 0x7fffffff : h * h + dy * dy;
        best = min(best, d2);
      }
      if (best <= R2) {
        uint8_t* cell = tile + r * kTX + tx;
        *cell = inflate_combine(*cell, table[best]);
      }
    }
    __syncthreads();
  }

  // write-back: the whole tile, 16 cells per thread (unchanged cells are rewritten with their own value)
  for (int item = tid; item < kTX * kTY / 16; item += kUpdateThreads) {
    const int r = item / (kTX / 16), c = (item - r * (kTX / 16)) * 16;
    const int y = ty0 + r, x = tx0 + c;
    if (y < (int)a.sy && x < (int)a.pitch)
      *reinterpret_cast<uint4*>(a.master + (size_t)y * a.pitch + x) = *reinterpret_cast<const uint4*>(tile + r * kTX + c);
  }
}


// ---------------------------------------------------------------------------------------------------------------
// Fast path of the same sweep for R <= 31 cells (every configuration the reference's defaults produce), split in two
// kernels so that the layer merge is a pure streaming pass and only ONE BIT per cell crosses tile borders:
//
//   k_merge_seed   16 cells per thread: uint4 loads of every layer, merge policies on 4 packed bytes per 32-bit op,
//                  uint4 store of the pre-inflation master value, and the "== LETHAL and inside the seed region"
//                  predicate as a uint16 into a device-wide seed bitmask (1 bit per cell, 2 MB at 4000^2).
//   k_inflate      tile 128 x 64 cells per CTA: seed words of the tile + halo (R rows, 32 columns) come from the
//                  bitmask; phase 2 turns every row that has seeds into squared horizontal distances (clz/ffs on
//                  funnel-shifted windows, packed u16x2); phase 3 gives each thread 4 columns x 4 rows of
//                  accumulators and walks only the non-empty rows of its (4 + 2R)-row window with ONE
//                  VIADDMNMX.U16x2 per row and cell pair; the epilogue looks the cost up by d^2 and applies
//                  InflationLayer's max / NO_INFORMATION rule directly on the master grid, four cells of a row per
//                  32-bit access, touching only rows that inflation reaches.  A tile whose seed words are all zero
//                  exits after the load.
// k_merge_seed: a CTA walks kMSSubTiles sub-tiles of 256 columns x 32 rows (what MergeLayers::used summarises) top to
// bottom: 256 x 128 cells per CTA.  (CTAs of one sub-tile live ~1.7 us and a freed slot stays empty for about a
// microsecond before its next CTA runs -- DESIGN.md "Known limits" --; four times the work per CTA makes the 4000^2 pass
// a single wave of 500 CTAs.)
constexpr int kMSGroupsX = 16, kMSRowsY = 16, kMSRowIters = 2, kMSSubTiles = 2;
constexpr int kMSTileH = kMSRowsY * kMSRowIters * kMSSubTiles;
static_assert(kMSGroupsX * 16 == (int)kMarkTileW && kMSRowsY * kMSRowIters == (int)kMarkTileH, "MergeLayers::used tile");
// k_inflate: a region row is 6 seed words (the 128 tile columns and one word of halo on either side)
constexpr int kITX = 128, kITY = 64, kIThreads = 256, kIMaxRows = kITY + 2 * 31, kISeedWords = kITX / 32 + 2;
static_assert(kIMaxRows <= kIThreads, "k_inflate: one thread per region row");
constexpr int kIMaskWords = (kIMaxRows + 32 + (4 + 2 * 31) + 31) / 32 + 1;
constexpr int kISparseRows = 14;  // k_inflate phase 3: up to this many seeded rows per window take the set-bit walk
constexpr uint32_t kH2Inf = 0x3000;  // "no seed within R on this row" (as a squared distance, per 16-bit half)

// layout of the seed bitmask: one row per grid row, 2 zero pad groups (32 cells) on either side of the row
__host__ __device__ inline unsigned seed_pitch16(unsigned pitch) { return pitch / 16 + 4; }

struct MergeSeedArgs {
  uint8_t* master;
  unsigned sx, sy, pitch;
  uint8_t def;
  int do_reset;
  const DevWindow* win;
  MergeLayers ml;
  int R;            // 0: merge only (seeds may be null)
  uint16_t* seeds;  // sy x seed_pitch16(pitch)
  int early = 0, ex0 = 0, exn = 0, ey0 = 0, eyn = 0;  // see UpdateArgs
  const unsigned* obst_flag = nullptr;                // see UpdateArgs
  unsigned obst_epoch = 0;
  // early mode with k_inflate behind us: every CTA publishes `epoch` in ready[blockIdx.y * gridDim.x + blockIdx.x] once
  // its tile (master cells and seed bits) is written, and k_inflate's tiles wait for just the tiles they read
  unsigned* ready = nullptr;
  unsigned epoch = 0;
  int lean = 0;  // the stack is "TrueOverwrite, then at most one Max / Overwrite layer": interior tiles take merge_seed_lean
};

__device__ __forceinline__ uint32_t inc4(uint32_t x) {  // per-byte x + 1 (mod 256), no carry between bytes
  return ((x & 0x7f7f7f7fu) + 0x01010101u) ^ (x & 0x80808080u);
}

__device__ __forceinline__ uint32_t merge4(uint32_t m, uint32_t v, int policy) {
  switch (policy) {
    case NAVGPU_TRUE_OVERWRITE: return v;
    case NAVGPU_OVERWRITE: {
      const uint32_t vn = __vcmpeq4(v, 0xffffffffu);
      return (m & vn) | (v & ~vn);
    }
    case NAVGPU_MAX: {
      // "skip layer == 255; write if master == 255 or master < layer" is an unsigned maximum once NO_INFORMATION is
      // rotated to the bottom of the order: x -> x + 1 (mod 256) per byte sends 255 to 0 and keeps every other order
      const uint32_t take = __vcmpltu4(inc4(m), inc4(v));
      return (v & take) | (m & ~take);
    }
    case NAVGPU_ADDITION: {
      const uint32_t vn = __vcmpeq4(v, 0xffffffffu), mn = __vcmpeq4(m, 0xffffffffu);
      uint32_t s = __vaddus4(m, v);
      const uint32_t ge = __vcmpgeu4(s, 0xfdfdfdfdu);
      s = (ge & 0xfcfcfcfcu) | (s & ~ge);
      const uint32_t r = (mn & v) | (~mn & s);
      return (vn & m) | (~vn & r);
    }
    default: return m;
  }
}

__device__ __forceinline__ uint4 merge16(uint4 m, uint4 v, int policy) {
  // the switch sits outside the four word-merges so it is resolved once per 16 cells
  switch (policy) {
    case NAVGPU_TRUE_OVERWRITE: return v;
    case NAVGPU_OVERWRITE:
      return make_uint4(merge4(m.x, v.x, NAVGPU_OVERWRITE), merge4(m.y, v.y, NAVGPU_OVERWRITE),
                        merge4(m.z, v.z, NAVGPU_OVERWRITE), merge4(m.w, v.w, NAVGPU_OVERWRITE));
    case NAVGPU_MAX:
      if ((v.x | v.y | v.z | v.w) == 0) {  // an all-FREE_SPACE group of the layer only turns NO_INFORMATION into 0
        return make_uint4(m.x & ~__vcmpeq4(m.x, 0xffffffffu), m.y & ~__vcmpeq4(m.y, 0xffffffffu),
                          m.z & ~__vcmpeq4(m.z, 0xffffffffu), m.w & ~__vcmpeq4(m.w, 0xffffffffu));
      }
      if ((v.x & v.y & v.z & v.w) == 0xffffffffu) return m;  // an all-NO_INFORMATION group changes nothing
      return make_uint4(merge4(m.x, v.x, NAVGPU_MAX), merge4(m.y, v.y, NAVGPU_MAX), merge4(m.z, v.z, NAVGPU_MAX),
                        merge4(m.w, v.w, NAVGPU_MAX));
    case NAVGPU_ADDITION:
      return make_uint4(merge4(m.x, v.x, NAVGPU_ADDITION), merge4(m.y, v.y, NAVGPU_ADDITION),
                        merge4(m.z, v.z, NAVGPU_ADDITION), merge4(m.w, v.w, NAVGPU_ADDITION));
    default: return m;
  }
}

// bit 7 of every byte of x that equals 255 (the low seven bits carry into bit 7 exactly when they are all set)
__device__ __forceinline__ uint32_t is255_4(uint32_t x) { return ((x & 0x7f7f7f7fu) + 0x01010101u) & x & 0x80808080u; }

__device__ __forceinline__ uint32_t lethal_bits4(uint32_t v) {  // one bit per byte that equals LETHAL_OBSTACLE
  const uint32_t e = is255_4(v ^ 0x01010101u) >> 7;
  return (e * 0x01020408u) >> 24;
}

// k_merge_seed on an interior tile of the usual stack: layer 0 merged with TrueOverwrite (StaticLayer on a non-rolling
// map, plugins/static_layer.cpp:318-326 -- whatever resetMap left is overwritten), optionally one more layer merged
// with Max or Overwrite (ObstacleLayer, plugins/obstacle_layer.cpp:431-443).  Same results as merge_seed_items<true>;
// what differs is the instruction count: 16-cell groups without a byte >= 128 (free space and low costs: almost all of
// a map) hold neither NO_INFORMATION nor LETHAL_OBSTACLE, so merging an all-FREE_SPACE group into them changes
// nothing and they seed nothing, and the tile summary byte of the second layer is fetched behind the first layer's
// loads instead of in front of them.
template <bool kEdge>
__device__ __forceinline__ void merge_seed_lean(const MergeSeedArgs& a, int x, int by0) {
  // kEdge: the tile reaches beyond the map's last row or column (the window being the whole map there): rows past the
  // map are skipped, the row padding behind the last column is written like cells (nothing reads it) and seeds nothing
  if (kEdge && x >= (int)a.pitch) return;
  const int y0 = by0 + threadIdx.y;
  const size_t off = (size_t)y0 * a.pitch + x, rs = (size_t)kMSRowsY * a.pitch;  // this thread's rows: y0 + 16 i
  const bool two = a.ml.n > 1;
  const int pol1 = a.ml.policy[1];
  const unsigned sp16 = seed_pitch16(a.pitch);
  uint16_t* srow = a.seeds + (size_t)y0 * sp16 + 2 + (x >> 4);
  uint32_t colmask = 0xffffu;
  if (kEdge && x + 16 > (int)a.sx) colmask = x >= (int)a.sx ? 0u : (1u << ((int)a.sx - x)) - 1u;
  auto load = [&](int sub, uint4* dst) {  // first layer, the two rows of sub-tile `sub`
#pragma unroll
    for (int it = 0; it < kMSRowIters; ++it) {
      const int row = kMSRowIters * sub + it;
      dst[it] = make_uint4(0, 0, 0, 0);
      if (!kEdge || y0 + row * kMSRowsY < (int)a.sy) dst[it] = *reinterpret_cast<const uint4*>(a.ml.grid[0] + off + row * rs);
    }
  };
  uint4 v[kMSSubTiles][kMSRowIters];  // every row of the thread in flight before the first is used
#pragma unroll
  for (int sub = 0; sub < kMSSubTiles; ++sub) load(sub, v[sub]);
  // the second layer's summary bytes of the sub-tiles, behind the first loads
  uint32_t use1 = two ? (1u << kMSSubTiles) - 1u : 0u;
  if (two && a.ml.used[1]) {
    use1 = 0;
#pragma unroll
    for (int sub = 0; sub < kMSSubTiles; ++sub)
      if (!kEdge || by0 + sub * (kMSRowsY * kMSRowIters) < (int)a.sy)
        use1 |= (a.ml.used[1][(blockIdx.y * kMSSubTiles + sub) * gridDim.x + blockIdx.x] != 0 ? 1u : 0u) << sub;
  }
#pragma unroll
  for (int sub = 0; sub < kMSSubTiles; ++sub) {
#pragma unroll
    for (int it = 0; it < kMSRowIters; ++it) {
      const int row = kMSRowIters * sub + it;
      if (kEdge && y0 + row * kMSRowsY >= (int)a.sy) continue;
      uint4 m = v[sub][it];
      uint32_t hi = (m.x | m.y | m.z | m.w) & 0x80808080u;  // some byte >= 128: the group may hold 254 / 255
      if (two) {
        uint4 o = make_uint4(0, 0, 0, 0);
        if ((use1 >> sub) & 1u) o = *reinterpret_cast<const uint4*>(a.ml.grid[1] + off + row * rs);
        if ((o.x | o.y | o.z | o.w) != 0 || pol1 != NAVGPU_MAX) {
          m = merge16(m, o, pol1);
          hi = (m.x | m.y | m.z | m.w) & 0x80808080u;
        } else if (hi) {  // Max with an all-FREE_SPACE group only turns NO_INFORMATION into 0
          m.x &= ~((is255_4(m.x) >> 7) * 0xffu); m.y &= ~((is255_4(m.y) >> 7) * 0xffu);
          m.z &= ~((is255_4(m.z) >> 7) * 0xffu); m.w &= ~((is255_4(m.w) >> 7) * 0xffu);
        }
      }
      *reinterpret_cast<uint4*>(a.master + off + row * rs) = m;
      if (a.R > 0) {
        uint32_t seed16 = 0;
        if (hi) seed16 = lethal_bits4(m.x) | (lethal_bits4(m.y) << 4) | (lethal_bits4(m.z) << 8) | (lethal_bits4(m.w) << 12);
        srow[(size_t)row * kMSRowsY * sp16] = (uint16_t)(seed16 & colmask);
      }
    }
  }
}

// body of k_merge_seed for one thread: kMSRowIters groups of 16 cells in one column of groups.  kInterior: the whole
// CTA tile lies inside the window, the seed region and the map, so every per-group edge test folds away.
template <bool kInterior>
__device__ __forceinline__ void merge_seed_items(const MergeSeedArgs& a, const DevWindow& w, int x, int by0, int sx0,
                                                 int sxn, int sy0, int syn, unsigned used_mask) {
  const int R = a.R;
  const unsigned sp16 = seed_pitch16(a.pitch);
  // A window that reaches the map's right edge owns the row padding behind it as well (nothing reads those bytes, and
  // their seed bits are masked off below), so a group that straddles only that edge keeps the packed 16-cell path
  // instead of the per-cell one -- every row of a map whose width is not a multiple of 16 has such a group.
  const int xn_all = w.xn == (int)a.sx ? (int)a.pitch : w.xn;
  const bool col_any = kInterior || (x + 16 > w.x0 && x < w.xn), col_all = kInterior || (x >= w.x0 && x + 16 <= xn_all);
  const bool col_seed = kInterior ? R > 0 : (R > 0 && x + 16 > sx0 && x < sxn);

  // loads of all row iterations first (memory-level parallelism), then the merges
  uint4 mv[kMSRowIters];
  uint4 lv[kMSRowIters][2];
#pragma unroll
  for (int it = 0; it < kMSRowIters; ++it) {
    const int y = by0 + threadIdx.y + it * kMSRowsY;
    mv[it] = make_uint4(0, 0, 0, 0);
    lv[it][0] = lv[it][1] = make_uint4(0, 0, 0, 0);
    if (!kInterior && y >= (int)a.sy) continue;
    const size_t off = (size_t)y * a.pitch + x;
    const bool row_in = kInterior || (y >= w.y0 && y < w.yn);
    const bool any_in = row_in && col_any, all_in = row_in && col_all;
    const bool need_master = any_in ? !(all_in && a.do_reset) : (col_seed && y >= sy0 && y < syn);
    if (need_master) mv[it] = *reinterpret_cast<const uint4*>(a.master + off);
    if (any_in) {
      if (a.ml.n > 0 && (used_mask & 1u)) lv[it][0] = *reinterpret_cast<const uint4*>(a.ml.grid[0] + off);
      if (a.ml.n > 1 && (used_mask & 2u)) lv[it][1] = *reinterpret_cast<const uint4*>(a.ml.grid[1] + off);
    }
  }
#pragma unroll
  for (int it = 0; it < kMSRowIters; ++it) {
    const int y = by0 + threadIdx.y + it * kMSRowsY;
    if (!kInterior && y >= (int)a.sy) continue;
    const size_t off = (size_t)y * a.pitch + x;
    const bool row_in = kInterior || (y >= w.y0 && y < w.yn);
    const bool any_in = row_in && col_any, all_in = row_in && col_all;
    uint4 v = mv[it];
    if (all_in) {
      if (a.do_reset) {
        const uint32_t d4 = a.def * 0x01010101u;
        v = make_uint4(d4, d4, d4, d4);
      }
      if (a.ml.n > 0) v = merge16(v, lv[it][0], a.ml.policy[0]);
      if (a.ml.n > 1) v = merge16(v, lv[it][1], a.ml.policy[1]);
      for (int l = 2; l < a.ml.n; ++l)
        v = merge16(v, (used_mask >> l) & 1u ? *reinterpret_cast<const uint4*>(a.ml.grid[l] + off) : make_uint4(0, 0, 0, 0),
                    a.ml.policy[l]);
    } else if (any_in) {  // group straddles the window edge: per-cell path
      uint32_t vv[4] = {v.x, v.y, v.z, v.w};
      for (int l = -1; l < a.ml.n; ++l) {
        uint4 lv4 = make_uint4(0, 0, 0, 0);
        if (l == 0) lv4 = lv[it][0];
        else if (l == 1) lv4 = lv[it][1];
        else if (l >= 2 && ((used_mask >> l) & 1u)) lv4 = *reinterpret_cast<const uint4*>(a.ml.grid[l] + off);
        const uint32_t lw[4] = {lv4.x, lv4.y, lv4.z, lv4.w};
        for (int i = 0; i < 16; ++i) {
          const int cx = x + i;
          if (cx < w.x0 || cx >= w.xn) continue;
          const int sh = 8 * (i & 3);
          uint8_t m = (uint8_t)(vv[i >> 2] >> sh);
          if (l < 0) { if (a.do_reset) m = a.def; }
          else m = apply_policy(m, (uint8_t)(lw[i >> 2] >> sh), a.ml.policy[l]);
          vv[i >> 2] = (vv[i >> 2] & ~(0xffu << sh)) | ((uint32_t)m << sh);
        }
      }
      v = make_uint4(vv[0], vv[1], vv[2], vv[3]);
    }
    if (any_in) *reinterpret_cast<uint4*>(a.master + off) = v;
    if (R > 0) {
      uint32_t seed16 = 0;
      if ((kInterior || (col_seed && y >= sy0 && y < syn)) && (v.x | v.y | v.z | v.w) != 0) {
        seed16 = lethal_bits4(v.x) | (lethal_bits4(v.y) << 4) | (lethal_bits4(v.z) << 8) | (lethal_bits4(v.w) << 12);
        if (!kInterior) {
          const int lo = min(16, max(0, sx0 - x)), hi = min(16, max(0, sxn - x));
          seed16 &= ((1u << hi) - 1u) & ~((1u << lo) - 1u);
        }
      }
      a.seeds[(size_t)y * sp16 + 2 + (x >> 4)] = (uint16_t)seed16;
    }
  }
}

__global__ void __launch_bounds__(kMSGroupsX * kMSRowsY, 5) k_merge_seed(MergeSeedArgs a) {
  // launched with programmatic stream serialization: let k_inflate be scheduled as soon as every CTA of this grid
  // is resident, and wait for the kernel before us (window, obstacle grid) before reading anything
  cudaTriggerProgrammaticLaunchCompletion();
  constexpr int kW = kMSGroupsX * 16, kH = kMSTileH;
  const int bx0 = blockIdx.x * kW, by0 = blockIdx.y * kH;
  DevWindow w;
  if (a.early) {
    // The window is the whole map whatever the obstacle kernel ahead of us adds to the bounds (they only grow), and that
    // kernel -- a latency chain of a few thousand rays on a fraction of the SMs -- writes layer cells only inside the
    // box of its rays, marks and footprint.  Tiles outside that box do not wait for it: the streaming merge of ~95 % of
    // the map overlaps the ray tracing.  CTA (0, 0) always waits for all of that kernel at its END, so that this grid
    // completes after it and a k_inflate that waits for this grid sees everything that kernel wrote (the window record
    // included) -- not in front of its own tile, which five inflation tiles need.
    w.x0 = 0; w.xn = (int)a.sx; w.y0 = 0; w.yn = (int)a.sy; w.valid = 1;
    const bool touched = bx0 < a.exn && bx0 + kW > a.ex0 && by0 < a.eyn && by0 + kH > a.ey0;
    // (CTA (0, 0) waits for the END of the obstacle kernel -- but behind its own work, see below)
    if (touched && !a.obst_flag) cudaGridDependencySynchronize();
    if (touched && a.obst_flag) {
      // (every CTA of the obstacle kernel is resident or done before this grid is scheduled: it triggers the programmatic
      // launch at its first instruction, so waiting for its last CTA cannot deadlock)
      if ((threadIdx.x | threadIdx.y) == 0) {
        unsigned seen;
        for (;;) {
          asm volatile("ld.acquire.gpu.u32 %0, [%1];" : "=r"(seen) : "l"(a.obst_flag) : "memory");
          if (seen == a.obst_epoch) break;
          __nanosleep(64);
        }
      }
      __syncthreads();
    }
    if (a.lean) {  // every tile: the window is the whole map
      if (bx0 + kW <= (int)a.sx && by0 + kH <= (int)a.sy) merge_seed_lean<false>(a, bx0 + threadIdx.x * 16, by0);
      else merge_seed_lean<true>(a, bx0 + threadIdx.x * 16, by0);
      if (a.ready) {
        __syncthreads();
        if ((threadIdx.x | threadIdx.y) == 0)
          asm volatile("st.release.gpu.u32 [%0], %1;" ::"l"(a.ready + blockIdx.y * gridDim.x + blockIdx.x), "r"(a.epoch) : "memory");
      }
      if ((blockIdx.x | blockIdx.y) == 0) cudaGridDependencySynchronize();  // this grid completes after the obstacle kernel
      return;
    }
  } else {
    cudaGridDependencySynchronize();
    w = *a.win;
  }
  if (!w.valid) return;
  const int R = a.R;
  // everything k_inflate can read: its tiles intersect window +- 2R, extend up to a tile further, and look R rows /
  // 32 columns beyond their own extent
  const int my = R > 0 ? 3 * R + kITY : 0, mx = R > 0 ? 2 * R + kITX + 32 : 0;
  if (bx0 >= w.xn + mx || bx0 + kW <= w.x0 - mx || by0 >= w.yn + my || by0 + kH <= w.y0 - my) return;
  const int sx0 = max(0, w.x0 - R), sxn = min((int)a.sx, w.xn + R);  // seed region (inflation_layer.cpp:203-211)
  const int sy0 = max(0, w.y0 - R), syn = min((int)a.sy, w.yn + R);
  const int x = bx0 + threadIdx.x * 16;
  // the window lies inside the map, the seed region contains the window: a tile inside the window is interior
  if (a.lean && bx0 >= w.x0 && bx0 + kW <= w.xn && by0 >= w.y0 && by0 + kH <= w.yn) {
    merge_seed_lean<false>(a, x, by0);
  } else {
    for (int sub = 0; sub < kMSSubTiles; ++sub) {  // sub-tile by sub-tile
      constexpr int kSH = kMSRowsY * kMSRowIters;
      const int sy_0 = by0 + sub * kSH;
      if (sy_0 >= (int)a.sy || sy_0 >= w.yn + my || sy_0 + kSH <= w.y0 - my) continue;
      const bool interior = bx0 >= w.x0 && bx0 + kW <= w.xn && sy_0 >= w.y0 && sy_0 + kSH <= w.yn;
      // layers whose tile summary says "all FREE_SPACE here" are not read (after the wait above: the obstacle kernel
      // sets the bytes of the tiles it marks)
      unsigned used_mask = 0xffffffffu;
      for (int l = 0; l < a.ml.n; ++l)
        if (a.ml.used[l] && a.ml.used[l][(blockIdx.y * kMSSubTiles + sub) * gridDim.x + blockIdx.x] == 0) used_mask &= ~(1u << l);
      if (interior) {
        merge_seed_items<true>(a, w, x, sy_0, sx0, sxn, sy0, syn, used_mask);
      } else if (x < (int)a.pitch) {
        merge_seed_items<false>(a, w, x, sy_0, sx0, sxn, sy0, syn, used_mask);
      }
    }
  }
  if (a.ready) {  // (early mode: the window is the whole map, no CTA left above)
    __syncthreads();
    if ((threadIdx.x | threadIdx.y) == 0)  // (release at gpu scope: cumulative over what the barrier made visible here)
      asm volatile("st.release.gpu.u32 [%0], %1;" ::"l"(a.ready + blockIdx.y * gridDim.x + blockIdx.x), "r"(a.epoch) : "memory");
  }
  if (a.early && (blockIdx.x | blockIdx.y) == 0) cudaGridDependencySynchronize();  // (see the early-mode comment above)
}

// k_inflate phase 3: dy^2 of window row j against the four output rows k of a group, (j - k)^2 in both 16-bit halves:
// c_dy2.v[j + 31][k] for j in [-31, 34] -- one broadcast 16-byte constant load per seeded row instead of an add chain
struct Dy2Table {
  uint32_t v[4 + 2 * 31][4];
  constexpr Dy2Table() : v() {
    for (int p = 0; p < 4 + 2 * 31; ++p)
      for (int k = 0; k < 4; ++k) v[p][k] = (uint32_t)((p - 31 - k) * (p - 31 - k)) * 0x10001u;
  }
};
__constant__ Dy2Table c_dy2 = Dy2Table();

// (lane 0 of a warp takes a number: a plain shared-memory atomic, without the warp-aggregation code the compiler wraps
// around atomicAdd)
__device__ __forceinline__ int smem_fetch_add(int* p, int v) {
  int old;
  asm volatile("atom.shared.add.s32 %0, [%1], %2;" : "=r"(old) : "r"((unsigned)__cvta_generic_to_shared(p)), "r"(v) : "memory");
  return old;
}

// global accesses through an address held in one 64-bit register pair (k_inflate's epilogue)
__device__ __forceinline__ uint32_t ldg_u32(unsigned long long addr) {
  uint32_t v;
  asm volatile("ld.global.u32 %0, [%1];" : "=r"(v) : "l"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void stg_u32(unsigned long long addr, uint32_t v) {
  asm volatile("st.global.u32 [%0], %1;" ::"l"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void stg_u8(unsigned long long addr, uint32_t v) {
  asm volatile("st.global.u8 [%0], %1;" ::"l"(addr), "r"(v) : "memory");
}

struct InflateArgs {
  uint8_t* master;
  unsigned sx, sy, pitch;
  const DevWindow* win;
  int R;
  int reach2;              // largest squared distance whose cost is not 0: nothing beyond it can change a cell
  int reach;               // floor(sqrt(reach2)): the effective radius in cells
  const uint8_t* cost_d2;  // R*R+1 entries: cost by squared cell distance
  const uint32_t* seeds;   // the bitmask written by k_merge_seed, viewed as 32-bit words
  // early mode (see MergeSeedArgs): the window is the whole map and a tile starts as soon as the k_merge_seed tiles it
  // reads have published `epoch`, instead of waiting for that whole grid (and, through it, for the obstacle kernel)
  const unsigned* ready = nullptr;
  unsigned epoch = 0;
  int ready_pitch = 0;  // k_merge_seed's gridDim.x
  unsigned* done = nullptr;  // nullable: one word per tile of this grid, set to `epoch` when the tile's cells are final
};

// RMAX bounds the effective reach (in cells) this instantiation can handle: the phase-3 walk is unrolled over
// 4 + 2 * RMAX region rows, so a small RMAX keeps the kernel's code (and its instruction-cache footprint) small.
template <int RMAX>
__device__ __forceinline__ void inflate_tile(const InflateArgs& a) {
  constexpr int kRows = kITY + 2 * RMAX;  // region rows this instantiation can hold
  constexpr int kH2W = kITX / 2;          // words per row of h2
  constexpr int kSW = kISeedWords;
  // packed u16x2 squared horizontal distances; lane l of phase 3 reads columns 4l .. 4l + 3 as words 2l, 2l + 1.
  // Before phase 2 fills a row, it holds other things no later step reads: the unpruned seed words of the region
  // (sbits, from the start of the array, until the pruning pass has read them), then the pruned words W0..W5 of row r
  // (columns tx0-32 .. tx0+159) at pbits_at(r) inside row r itself, which only the warp that computes row r reads
  __shared__ __align__(16) uint32_t h2[kRows * kH2W];
  uint32_t* const sbits = h2;
  // (staggered by 8 words from row to row: the pruning pass stores one row per thread without every thread of a warp
  // hitting the same banks)
  auto pbits_at = [&](int r) { return h2 + r * kH2W + 8 * (r & 7); };
  __shared__ uint32_t rowmask[kIMaskWords];  // bit (r + 32) <-> region row r has seeds
  // bit (r + 32) <-> region row r repeats row r - 1: same (non-zero) pruned seed words, hence the same horizontal
  // distances in every column of the tile.  Of a run of repeated rows only the row nearest to an output row can win
  // there (same hx^2, smaller dy^2): phase 2 computes the first row of a run only (canon[r] names it), phase 3 skips
  // the repeats further from its four output rows.  A vertical wall costs one row instead of one per map row.
  __shared__ uint32_t dupmask[kIMaskWords];
  __shared__ __align__(4) uint8_t canon[(kRows + 3) & ~3];
  __shared__ uint8_t rowlist[kRows];         // the same rows as a list (any order), n_seeded of them
  __shared__ int n_seeded;
  __shared__ int next_group;                 // phase 3: the next 4-row group nobody has taken yet
  // cost by d^2, table[reach2 + 1] = 0 ("out of reach"); reach <= RMAX bounds reach2 by (RMAX + 1)^2 - 1
  __shared__ __align__(16) uint8_t table[((RMAX + 1) * (RMAX + 1) + 1 + 15) & ~15];
  const int tx0 = blockIdx.x * kITX, ty0 = blockIdx.y * kITY;
  // early mode: the flags of the k_merge_seed tiles this tile reads (seeds: columns tx0 - 32 .. tx0 + kITX + 31, rows
  // ty0 - R .. ty0 + kITY + R - 1; master cells: the tile itself), one per thread, requested before anything else
  const unsigned* my_flag = nullptr;
  unsigned flag_seen = 0;
  cudaTriggerProgrammaticLaunchCompletion();  // (a k_mirror_diff behind us may become resident; it waits for our end)
  if (a.ready) {
    constexpr int kMW = kMSGroupsX * 16, kMH = kMSTileH;
    const int mx0 = max(0, tx0 - 32) / kMW, mx1 = min((int)a.pitch - 1, tx0 + kITX + 31) / kMW;
    const int my0 = max(0, ty0 - a.R) / kMH, my1 = min((int)a.sy - 1, ty0 + kITY + a.R - 1) / kMH;
    const int nx = mx1 - mx0 + 1, n = nx * (my1 - my0 + 1);  // <= 2 x 3 for R <= 31
    if ((int)threadIdx.x < n) {
      my_flag = a.ready + (my0 + (int)threadIdx.x / nx) * a.ready_pitch + mx0 + (int)threadIdx.x % nx;
      asm volatile("ld.acquire.gpu.u32 %0, [%1];" : "=r"(flag_seen) : "l"(my_flag) : "memory");
    }
  }
  // the cost table was uploaded long before this cycle: stage it while k_merge_seed is still draining, then wait
  {  // (by 32-bit words; the word that holds entry reach2 + 1 gets its zero on the way)
    const int zw = (a.reach2 + 1) >> 2;
    for (int i = threadIdx.x; i <= zw; i += kIThreads) {
      uint32_t v = reinterpret_cast<const uint32_t*>(a.cost_d2)[i];
      if (i == zw) v &= ~(0xffu << (8 * ((a.reach2 + 1) & 3)));
      reinterpret_cast<uint32_t*>(table)[i] = v;
    }
  }
  if (a.ready) {
    // Every k_merge_seed CTA is resident or done by the time this grid is scheduled (it triggers the programmatic launch
    // at its first instruction), so waiting for some of them cannot deadlock.
    if (my_flag) {
      while (flag_seen != a.epoch) {
        __nanosleep(32);
        asm volatile("ld.acquire.gpu.u32 %0, [%1];" : "=r"(flag_seen) : "l"(my_flag) : "memory");
      }
    }
    __syncthreads();  // (the window is the whole map: every tile of the grid is in it)
  } else {
    cudaGridDependencySynchronize();
    const DevWindow w = *a.win;
    if (!w.valid) return;
    const int R = a.R;
    if (tx0 >= w.xn + 2 * R || tx0 + kITX <= w.x0 - 2 * R || ty0 >= w.yn + 2 * R || ty0 + kITY <= w.y0 - 2 * R) return;
  }
  // from here on R is the effective reach: seeds further than sqrt(reach2) cells away only ever contribute cost 0,
  // and max(old, 0) / the NO_INFORMATION rule leave the cell as it is
  const int R = a.reach;
  const int rows = kITY + 2 * R;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned sp32 = seed_pitch16(a.pitch) / 2;

  // ---- seed words of the region (every load in flight before the first use); leave when there is nothing to inflate from
  int any = 0;
  {
    constexpr int NI = (kRows * kSW + kIThreads - 1) / kIThreads;
    uint32_t v[NI];
#pragma unroll
    for (int k = 0; k < NI; ++k) {
      const int i = tid + k * kIThreads, gy = ty0 - R + i / kSW;
      v[k] = 0;
      // (read past L1: in early mode a line of the bitmask can hold words of a k_merge_seed tile that is still running)
      if (i < rows * kSW && gy >= 0 && gy < (int)a.sy) v[k] = __ldcg(&a.seeds[(size_t)gy * sp32 + (tx0 >> 5) + i % kSW]);
    }
    if (tid < kIMaskWords) rowmask[tid] = dupmask[tid] = 0;
    if (tid == 0) n_seeded = next_group = 0;
#pragma unroll
    for (int k = 0; k < NI; ++k) {
      const int i = tid + k * kIThreads;
      if (i < rows * kSW) sbits[i] = v[k];
      any |= v[k] != 0;
    }
  }
  if (!__syncthreads_or(any)) return;

  // ---- interior seeds cannot be the nearest seed of any other cell: a seed whose four neighbours are seeds too has,
  // for every non-seed cell p, a neighbouring seed strictly closer to p (step along the larger coordinate difference),
  // so the minimum over all seeds is attained on the boundary seeds; the interior cell itself already holds LETHAL,
  // which max() keeps.  Dropping them empties most rows of thick structures for phases 2 and 3.  Seeds on the rim
  // of the loaded region (unknown neighbours) are kept.
  // Only seeds within R columns of the tile can matter (the top R bits of W0, the low R bits of W5): the pruned words
  // are masked that way.  One thread per region row: it also finds out whether its row repeats the row above (whose
  // pruned words it recomputes rather than wait for), and the warp's ballots become the row masks and the list of rows
  // phase 2 has to compute.
  uint32_t k[kSW];
  {
    auto pruned = [&](int r, uint32_t (&o)[kSW]) {
      const uint2* s2 = reinterpret_cast<const uint2*>(sbits + r * kSW);
      uint32_t c[kSW];
#pragma unroll
      for (int i = 0; i < kSW / 2; ++i) { const uint2 t = s2[i]; c[2 * i] = t.x; c[2 * i + 1] = t.y; }
      uint32_t nz = 0;
#pragma unroll
      for (int i = 0; i < kSW; ++i) { o[i] = c[i]; nz |= c[i]; }
      if (nz != 0 && r > 0 && r + 1 < rows) {
#pragma unroll
        for (int i = 0; i < kSW; ++i) {
          const uint32_t lo = (c[i] << 1) | (i > 0 ? c[i - 1] >> 31 : 0u);        // left neighbour is a seed
          const uint32_t hi = (c[i] >> 1) | (i + 1 < kSW ? c[i + 1] << 31 : 0u);  // right neighbour is a seed
          o[i] &= ~(lo & hi & sbits[(r - 1) * kSW + i] & sbits[(r + 1) * kSW + i]);
        }
      }
      o[0] &= ~(0xffffffffu >> R);
      o[kSW - 1] &= (1u << R) - 1u;
    };
    const int r = tid;  // (kRows <= kIMaxRows <= kIThreads)
    bool seeded = false, dup = false;
#pragma unroll
    for (int i = 0; i < kSW; ++i) k[i] = 0;
    if (r < rows) {
      pruned(r, k);
      uint32_t nz = 0;
#pragma unroll
      for (int i = 0; i < kSW; ++i) nz |= k[i];
      seeded = nz != 0;
      if (seeded && r > 0) {
        uint32_t p[kSW];
        pruned(r - 1, p);
        uint32_t ne = 0;
#pragma unroll
        for (int i = 0; i < kSW; ++i) ne |= k[i] ^ p[i];
        dup = ne == 0;
      }
    }
    const uint32_t sm = __ballot_sync(0xffffffffu, seeded), dm = __ballot_sync(0xffffffffu, dup);
    const uint32_t lm = sm & ~dm;  // rows whose distances phase 2 computes
    int base = 0;
    if (lane == 0 && sm) {
      rowmask[warp + 1] = sm;
      dupmask[warp + 1] = dm;
      if (lm) base = smem_fetch_add(&n_seeded, __popc(lm));
    }
    base = __shfl_sync(0xffffffffu, base, 0);
    if (seeded && !dup) rowlist[base + __popc(lm & ((1u << lane) - 1u))] = (uint8_t)r;
  }
  __syncthreads();

  // ---- phase 2: squared horizontal distances for the listed rows (one warp per row); before that the pruned words of
  // the listed rows go to their place (sbits is no longer read) and every row learns canon[r], the nearest row at or
  // above it that does not repeat its predecessor
  {
    if (tid < rows) {
      if (k[0] | k[1] | k[2] | k[3] | k[4] | k[5]) {
        uint32_t* pb = pbits_at(tid);
        *reinterpret_cast<uint4*>(pb) = make_uint4(k[0], k[1], k[2], k[3]);
        *reinterpret_cast<uint2*>(pb + 4) = make_uint2(k[4], k[5]);
      }
      int qq = warp;
      uint32_t z = ~dupmask[warp + 1] & (0xffffffffu >> (31 - lane));
      while (z == 0) z = ~dupmask[--qq + 1];  // (row 0 never repeats anything: the walk ends there at the latest)
      canon[tid] = (uint8_t)(32 * qq + 31 - __clz(z));
    }
    __syncthreads();
    const int n_rows_listed = n_seeded;
    for (int li = warp; li < n_rows_listed; li += kIThreads / 32) {
      const int r = rowlist[li];
      // lane l computes columns 4l .. 4l + 3, which lie in word 1 + l / 8 of the row
      const uint32_t* pw = pbits_at(r) + (lane >> 3);
      const uint32_t A = pw[0], B = pw[1], C = pw[2];
      __syncwarp();  // (every lane has read the pruned words before any lane overwrites them with distances)
      uint32_t packed[2] = {0u, 0u};
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int sh = (4 * lane + c) & 31;
        const uint32_t right = __funnelshift_r(B, C, sh);      // bit k    <-> dx = +k
        const uint32_t left = __funnelshift_rc(A, B, sh + 1);  // bit 31-k <-> dx = -k
        int d = 64;
        if (right) d = __ffs(right) - 1;
        if (left) d = min(d, __clz(left));
        const uint32_t hh = d <= R ? (uint32_t)(d * d) : kH2Inf;
        packed[c >> 1] |= hh << (16 * (c & 1));
      }
      *reinterpret_cast<uint2*>(h2 + r * kH2W + 2 * lane) = make_uint2(packed[0], packed[1]);
    }
  }
  __syncthreads();

  // ---- phase 3 + epilogue: a warp takes 128 columns x 4 rows at a time; lane l owns columns 4l .. 4l + 3, as the
  // accumulators acc[2k] (columns 4l, 4l + 1) and acc[2k + 1] (columns 4l + 2, 4l + 3) of output row k
  const uint32_t R2x2 = (uint32_t)a.reach2 * 0x10001u;
  const int x = tx0 + 4 * lane;
  const bool xok = x < (int)a.sx;
  // bytes of the lane's word that lie right of the map (inside the row padding): never computed, never written
  const int nvalid = (int)a.sx - x;
  const uint32_t keep_hi = nvalid >= 4 ? 0u : (nvalid <= 0 ? 0xffffffffu : 0xffffffffu << (8 * nvalid));
  const bool edge_tile = tx0 + kITX > (int)a.sx || ty0 + kITY > (int)a.sy;
  // (the groups are handed out as warps become free: a group far from every seed costs a few instructions, one next to a
  // shelf several hundred -- a fixed assignment leaves warps idle at the end of the tile)
  for (;;) {
    int g = 0;
    if (lane == 0) g = smem_fetch_add(&next_group, 1);
    g = __shfl_sync(0xffffffffu, g, 0);
    if (g >= kITY / 4) break;
    const int yr0 = g * 4;  // first tile row of this group; region rows yr0 .. yr0 + 3 + 2R
    uint32_t acc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[q] = 0x7fff7fffu;
    // Region rows that can matter for tile rows yr0 .. yr0 + 3 are r = yr0 + R + j with j in [-R, 3 + R]; rows beyond
    // +-R only ever add candidates above the reach, which changes nothing.  Two walks over the row mask of
    // j in [-RMAX, 3 + RMAX] (warp-uniform either way):
    //  * few seeded rows (the usual case: walls, shelves): visit the set bits only; dy^2 = (j - k)^2 for k = 0..3
    //    comes from a small constant table, one broadcast 16-byte load per row;
    //  * many seeded rows: the walk unrolled over j, so that dy^2 is an immediate operand of VIADDMNMX; rows without
    //    seeds cost one bit test, eight such rows one byte test.
    // Either way a visited row costs one 8-byte shared load of the lane's four hx^2 and eight VIADDMNMX.
    {
      constexpr int NJ = 4 + 2 * RMAX, NW = (NJ + 31) / 32, NB = (NJ + 7) / 8;
      const uint32_t* hb = h2 + 2 * lane;
      const uint8_t* cn = canon + yr0 + R;  // cn[j]: the row whose distances row j shares
      const int p0 = yr0 + R - RMAX + 32;  // position of j = -RMAX in rowmask (which is stored with a 32-row offset)
      const int wi = p0 >> 5, sh = p0 & 31;
      uint32_t mw[NW];
      uint32_t anyrow = 0;
      int nrows = 0;
#pragma unroll
      for (int q = 0; q < NW; ++q) {
        mw[q] = __funnelshift_r(rowmask[wi + q], rowmask[wi + q + 1], sh);
        if (q == NW - 1 && (NJ & 31) != 0) mw[q] &= (1u << (NJ & 31)) - 1u;
        // repeats: above the four output rows (j < 0) a row whose successor repeats it loses to that successor,
        // below them (j > 3) a row that repeats its predecessor loses to that predecessor; window position p = j + RMAX
        const uint32_t dw = __funnelshift_r(dupmask[wi + q], dupmask[wi + q + 1], sh);
        constexpr int kBelow = RMAX + 4;  // first window position below the output rows
        const uint32_t below = 32 * q >= kBelow ? 0xffffffffu : (32 * q + 32 <= kBelow ? 0u : 0xffffffffu << (kBelow & 31));
        uint32_t drop = below & dw;
        if (q == 0) drop |= ((1u << RMAX) - 1u) & (dw >> 1);
        mw[q] &= ~drop;
        anyrow |= mw[q];
        nrows += __popc(mw[q]);
      }
      if (anyrow == 0) continue;  // no seeded row anywhere near these four rows: nothing to inflate
      if (nrows <= kISparseRows) {
#pragma unroll
        for (int q = 0; q < NW; ++q) {
          uint32_t m = mw[q];
          while (m) {
            const int j = __ffs(m) - 1 + 32 * q - RMAX;
            m &= m - 1;
            const uint2 hh = *reinterpret_cast<const uint2*>(hb + cn[j] * kH2W);
            const uint4 dq = *reinterpret_cast<const uint4*>(c_dy2.v[j + 31]);
            acc[0] = __viaddmin_u16x2(hh.x, dq.x, acc[0]);
            acc[1] = __viaddmin_u16x2(hh.y, dq.x, acc[1]);
            acc[2] = __viaddmin_u16x2(hh.x, dq.y, acc[2]);
            acc[3] = __viaddmin_u16x2(hh.y, dq.y, acc[3]);
            acc[4] = __viaddmin_u16x2(hh.x, dq.z, acc[4]);
            acc[5] = __viaddmin_u16x2(hh.y, dq.z, acc[5]);
            acc[6] = __viaddmin_u16x2(hh.x, dq.w, acc[6]);
            acc[7] = __viaddmin_u16x2(hh.y, dq.w, acc[7]);
          }
        }
      } else {
#pragma unroll
        for (int c = 0; c < NB; ++c) {
          const uint32_t bits8 = (mw[c >> 2] >> ((c & 3) * 8)) & 0xffu;
          if (bits8 == 0) continue;
#pragma unroll
          for (int b = 0; b < 8; ++b) {
            const int j = 8 * c + b - RMAX;
            if (j > 3 + RMAX) continue;
            if (bits8 & (1u << b)) {
              const uint2 hh = *reinterpret_cast<const uint2*>(hb + cn[j] * kH2W);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const int dy = j - q;
                if (dy >= -RMAX && dy <= RMAX) {
                  acc[2 * q] = __viaddmin_u16x2(hh.x, (uint32_t)(dy * dy) * 0x10001u, acc[2 * q]);
                  acc[2 * q + 1] = __viaddmin_u16x2(hh.y, (uint32_t)(dy * dy) * 0x10001u, acc[2 * q + 1]);
                }
              }
            }
          }
        }
      }
    }
    // rows that inflation reaches somewhere in these 128 columns: read, combine (inflation_layer.cpp:249-254), write.
    // The lane's four cells of a row travel in one 32-bit word, so the byte maximum, the NO_INFORMATION test and the
    // "did anything change" test are paid once per four cells.  A cell out of reach looks up table[reach2 + 1] = 0 and
    // a row that is not read counts as 0: max(0, 0) stores nothing.
    const uint32_t out_of_reach = R2x2 + 0x10001u;
    if (edge_tile) {  // (block-uniform) rows below the map and lanes right of it: out of reach, nothing is read or written
      const int kmax = xok ? min(4, (int)a.sy - (ty0 + yr0)) : 0;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (q >= kmax) acc[2 * q] = acc[2 * q + 1] = 0x7fff7fffu;
    }
    // (the group's first cell as one 64-bit register pair: a row's address is then a single 32 x 32 + 64 multiply-add)
    unsigned long long prow = (unsigned long long)__cvta_generic_to_global(a.master + ((size_t)(ty0 + yr0) * a.pitch + x));
    asm volatile("" : "+l"(prow));
    uint32_t cur[4];
    bool reached = false;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      acc[2 * q] = __vminu2(acc[2 * q], out_of_reach);
      acc[2 * q + 1] = __vminu2(acc[2 * q + 1], out_of_reach);
      cur[q] = 0;
      // (both words are <= out_of_reach per half: their AND equals it exactly when both do)
      if ((acc[2 * q] & acc[2 * q + 1]) != out_of_reach) {
        cur[q] = ldg_u32(prow + (unsigned long long)((uint32_t)q * a.pitch));
        reached = true;
      }
    }
    if (!reached) continue;
    uint32_t out[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t da = acc[2 * q], db = acc[2 * q + 1];
      const uint32_t c = ((uint32_t)table[da & 0xffffu] | ((uint32_t)table[da >> 16] << 8) |
                          ((uint32_t)table[db & 0xffffu] << 16) | ((uint32_t)table[db >> 16] << 24)) & ~keep_hi;
      out[q] = __vmaxu4(cur[q], c);  // no cell NO_INFORMATION (the usual case): a plain maximum (:253-254)
      acc[2 * q] = c;                // (kept for the NO_INFORMATION rule below)
    }
    // NO_INFORMATION is replaced only by costs >= INSCRIBED_INFLATED_OBSTACLE, and then by the cost (:249-252): where
    // old == 255 the maximum is 255, and 255 - (255 - c) = c
    if ((__vcmpeq4(cur[0], 0xffffffffu) | __vcmpeq4(cur[1], 0xffffffffu) | __vcmpeq4(cur[2], 0xffffffffu) |
         __vcmpeq4(cur[3], 0xffffffffu)) != 0) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint32_t c = acc[2 * q];
        out[q] -= __vcmpeq4(cur[q], 0xffffffffu) & __vcmpgeu4(c, 0xfdfdfdfdu) & ~c;
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t diff = out[q] ^ cur[q];
      if (diff == 0) continue;
      const unsigned long long addr = prow + (unsigned long long)((uint32_t)q * a.pitch);
      if (keep_hi == 0) {
        stg_u32(addr, out[q]);
      } else {  // the lane's word reaches past the map: only its changed bytes, all of them left of sx, are stored
#pragma unroll
        for (int b = 0; b < 3; ++b)
          if ((diff >> (8 * b)) & 0xffu) stg_u8(addr + b, out[q] >> (8 * b));
      }
    }
  }
}

template <int RMAX>
__global__ void __launch_bounds__(kIThreads, 8) k_inflate(InflateArgs a) {
  inflate_tile<RMAX>(a);
  // tile (0, 0) of a sweep that runs on per-tile flags: behind the whole k_merge_seed grid, which completes behind the
  // obstacle kernel -- done[0] tells k_mirror_diff that the cycle's window record and dirty box are final
  if (a.ready && (blockIdx.x | blockIdx.y) == 0) cudaGridDependencySynchronize();
  // whichever way the tile ended: its master cells are final.  k_mirror_diff (the host mirror) starts on the tiles it
  // compares as soon as the inflate tiles that write them say so, instead of after the whole grid
  if (a.done) {
    __syncthreads();
    if (threadIdx.x == 0)
      asm volatile("st.release.gpu.u32 [%0], %1;" ::"l"(a.done + blockIdx.y * gridDim.x + blockIdx.x), "r"(a.epoch) : "memory");
  }
}

inline size_t update_costs_smem(int R) {
  const int HX = (R + 7) & ~7;
  const int groups = (kTX + 2 * HX) / 8;
  const int rows = kTY + 2 * R;
  const int bits_pitch = (groups + 3) & ~3;
  return (size_t)kTX * kTY + ((rows * bits_pitch + 15) & ~15) + (size_t)rows * kTX + (size_t)R * R + 1 + 16;
}

}  // namespace navgpu
