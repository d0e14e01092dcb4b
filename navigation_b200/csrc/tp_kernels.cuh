// tp_kernels.cuh -- the legacy base_local_planner::TrajectoryPlanner's rollout scoring on the device
// (base_local_planner/src/trajectory_planner.cpp:214-370 generateTrajectory), the second consumer of the footprint /
// MapGrid machinery of dwa_kernels.cuh (SURVEY.md 8f-4).
//
// One warp per velocity sample.  The trajectory is a sequential fp64 recurrence (acceleration-limited velocities,
// then x / y / theta), replayed by every lane in rounds of 32 steps; lane l keeps step l of the round, evaluates its
// trig, and the position prefix is accumulated in the reference's order through shuffles.  The per-step checks
// (worldToMap, footprint, path / goal distance) then run one step per lane, the footprint's (step, edge) walks
// spread over all 32 lanes.  The reference returns at the FIRST failing step; here every step of a round is
// evaluated and the lowest failing step decides, which is the same value.
#pragma once

#include "dwa_kernels.cuh"

namespace navgpu {

struct TpSampleResult {
  double cost;         // traj.cost_: >= 0 legal, -1 footprint / off the map, -2 no path to the goal
  double ahead_gdist;  // goal_map_ at the end point pushed heading_lookahead ahead (:672-681), -1 when off the map
  int n_points;        // points the trajectory holds (steps before the failing one)
  int pad_;
};

struct TpScoreArgs {
  DwaGeom g;
  const uint32_t* path_dist;  // path_map_ target_dist, sx*sy
  const uint32_t* goal_dist;  // goal_map_
  const double* samples;      // n x (vx_samp, vy_samp, vtheta_samp)
  int n;
  double x, y, theta, vx, vy, vtheta;  // robot state (already rounded through Eigen::Vector3f, :911-912)
  double acc_x, acc_y, acc_theta;
  double sim_time, sim_granularity, angular_sim_granularity;
  int simple_attractor;
  double goal_x, goal_y;  // last pose of the global plan (simple_attractor_)
  int heading_scoring;    // heading_scoring_: path / goal distance and the heading difference of ONE step only
  double heading_scoring_timestep;
  const double* plan_xy;  // the global plan as received (not resolution-adjusted), n_plan (x, y) pairs
  int n_plan;
  double pdist_scale, gdist_scale, occdist_scale;
  double heading_lookahead;
  int allow_unknown;
  int nfp;
  double fpx[kMaxFootprint], fpy[kMaxFootprint];
  TpSampleResult* out;
  double* points;     // nullable: n x points_stride x 3
  int points_stride;  // points kept per sample
};

// TrajectoryPlanner::computeNewVelocity, trajectory_planner.h:369-375
__device__ __forceinline__ double tp_new_velocity(double vg, double vi, double a_max, double dt) {
  if ((vg - vi) >= 0) return fmin(vg, vi + a_max * dt);
  return fmax(vg, vi - a_max * dt);
}

// TrajectoryPlanner::lineCost + pointCost (trajectory_planner.cpp:389-475): Bresenham from (x0, y0) to (x1, y1), both
// ends included; false as soon as a cell is LETHAL, INSCRIBED or (NO_INFORMATION and unknown is not allowed)
__device__ bool tp_line_is_clear(const TpScoreArgs& a, int x0, int x1, int y0, int y1) {
  const int dx = abs(x1 - x0), dy = abs(y1 - y0);
  const int xinc = x1 >= x0 ? 1 : -1, yinc = y1 >= y0 ? 1 : -1;
  const bool xmajor = dx >= dy;
  const int den = xmajor ? dx : dy, numadd = xmajor ? dy : dx;
  int num = den / 2, x = x0, y = y0;
  for (int k = 0; k <= den; ++k) {
    const int c = a.g.cost[y * (int)a.g.pitch + x];
    if (c == kLethal || c == kInscribed || (c == kNoInfo && !a.allow_unknown)) return false;
    num += numadd;
    if (num >= den) {
      num -= den;
      if (xmajor) y += yinc; else x += xinc;
    }
    if (xmajor) x += xinc; else y += yinc;
  }
  return true;
}

// TrajectoryPlanner::headingDiff (:372-387) with the whole warp: the farthest pose of the global plan that is on the
// map and in clear line of sight of the robot's cell; lanes test 32 candidates at a time, from the end of the plan.
// All lanes pass the same arguments and get the same result.
__device__ double tp_heading_diff(const TpScoreArgs& a, int cell_x, int cell_y, double x, double y, double heading, int lane) {
  for (int top = a.n_plan - 1; top >= 0; top -= 32) {
    const int i = top - lane;
    bool clear = false;
    int gx_c = 0, gy_c = 0;
    if (i >= 0 && dwa_world_to_map(a.g, a.plan_xy[2 * i], a.plan_xy[2 * i + 1], gx_c, gy_c))
      clear = tp_line_is_clear(a, cell_x, gx_c, cell_y, gy_c);
    const unsigned found = __ballot_sync(0xffffffffu, clear);
    if (found) {
      const int src = __ffs(found) - 1;  // the lowest lane holds the highest plan index
      gx_c = __shfl_sync(0xffffffffu, gx_c, src);
      gy_c = __shfl_sync(0xffffffffu, gy_c, src);
      const double gx = a.g.ox + (gx_c + 0.5) * a.g.res, gy = a.g.oy + (gy_c + 0.5) * a.g.res;  // Costmap2D::mapToWorld
      // angles::shortest_angular_distance(heading, atan2(...)) = normalize_angle(to - from)
      double d = fmod(fmod(atan2(gy - y, gx - x) - heading, 2.0 * M_PI) + 2.0 * M_PI, 2.0 * M_PI);
      if (d > M_PI) d -= 2.0 * M_PI;
      return fabs(d);
    }
  }
  return 1.7976931348623157e308;  // DBL_MAX
}

__device__ void tp_score_sample(const TpScoreArgs& a, int sample, int lane, double* warp_scratch) {
  const double vx_samp = a.samples[3 * sample], vy_samp = a.samples[3 * sample + 1], vth_samp = a.samples[3 * sample + 2];
  const double vmag = hypot(vx_samp, vy_samp);
  int num_steps = a.heading_scoring ? (int)(a.sim_time / a.sim_granularity + 0.5)
                                    : (int)(fmax((vmag * a.sim_time) / a.sim_granularity, fabs(vth_samp) / a.angular_sim_granularity) + 0.5);
  if (num_steps == 0) num_steps = 1;
  const double dt = a.sim_time / num_steps;
  const uint32_t n_cells = a.g.sx * a.g.sy;  // path_map_.obstacleCosts(): the "impossible" cost (:535, :591)

  double sx = a.x, sy = a.y, sth = a.theta;  // state at the first step of the current round
  double vxi = a.vx, vyi = a.vy, vthi = a.vtheta;
  double occ_cost = 0.0, path_dist = 0.0, goal_dist = 0.0, ahead = -1.0, heading_diff = 0.0, time = 0.0;
  double fail_code = 0.0;
  int n_points = num_steps;
  double* out_pts = a.points ? a.points + (size_t)sample * a.points_stride * 3 : nullptr;

  for (int base = 0; base < num_steps; base += 32) {
    const int cnt = min(32, num_steps - base);
    // velocity / heading recurrence (:352-361): the point of step l uses theta_l; the move to step l + 1 uses the
    // velocities already advanced to l + 1 and, for x / y, still theta_l
    double th = sth, my_th = sth, my_vx = 0.0, my_vy = 0.0, my_time = 0.0;
    for (int l = 0; l < cnt; ++l) {
      if (lane == l) { my_th = th; my_time = time; }
      time += dt;  // `time += dt` once per step, as the reference accumulates it (:369)
      vxi = tp_new_velocity(vx_samp, vxi, a.acc_x, dt);
      vyi = tp_new_velocity(vy_samp, vyi, a.acc_y, dt);
      vthi = tp_new_velocity(vth_samp, vthi, a.acc_theta, dt);
      if (lane == l) { my_vx = vxi; my_vy = vyi; }
      th = th + vthi * dt;
    }
    double c, s;
    sincos(my_th, &s, &c);
    // computeNewXPosition / computeNewYPosition, trajectory_planner.h:332-347
    double ddx, ddy;
    if (my_vy != 0.0) {
      double c2, s2;
      sincos(M_PI_2 + my_th, &s2, &c2);
      ddx = (my_vx * c + my_vy * c2) * dt;
      ddy = (my_vx * s + my_vy * s2) * dt;
    } else {
      ddx = (my_vx * c + 0.0) * dt;
      ddy = (my_vx * s + 0.0) * dt;
    }
    double x = sx, y = sy, px = sx, py = sy;
    for (int l = 0; l < cnt; ++l) {
      if (lane == l) { px = x; py = y; }
      x = x + __shfl_sync(0xffffffffu, ddx, l);
      y = y + __shfl_sync(0xffffffffu, ddy, l);
    }
    sx = x;
    sy = y;
    sth = th;
    const bool active = lane < cnt;

    // ---- footprint of every step of the round: (step, vertex) cells, then (step, edge) walks, over all lanes
    double* pose_s = warp_scratch;
    unsigned* edge_max = reinterpret_cast<unsigned*>(warp_scratch + 128);
    pose_s[lane] = px;
    pose_s[32 + lane] = py;
    pose_s[64 + lane] = c;
    pose_s[96 + lane] = s;
    edge_max[lane] = 0;
    __syncwarp();
    if (a.nfp >= 3) {
      int* vcell = reinterpret_cast<int*>(warp_scratch + 128 + 16);
      const int items = cnt * a.nfp;
      const unsigned inv_nfp = (65536u + (unsigned)a.nfp - 1u) / (unsigned)a.nfp;  // exact for it < 512, nfp <= 16
      for (int it = lane; it < items; it += 32) {
        const int p = (int)(((unsigned)it * inv_nfp) >> 16), v = it - p * a.nfp;
        vcell[it] = footprint_vertex_cell(a, pose_s[p], pose_s[32 + p], pose_s[64 + p], pose_s[96 + p], v);
      }
      __syncwarp();
      for (int it = lane; it < items; it += 32) {
        const int p = (int)(((unsigned)it * inv_nfp) >> 16), e = it - p * a.nfp;
        const int next = e + 1 < a.nfp ? it + 1 : it - e;  // packed [point][vertex] rows of nfp words
        const int ec = footprint_edge_cost(a, vcell[it], vcell[next]);
        atomicMax(&edge_max[p], ec < 0 ? 0x80000000u : (unsigned)ec);
      }
      __syncwarp();
    }
    // ---- my step
    double code = 0.0, occ = 0.0, pd = 0.0, gd = 0.0;
    bool heading_step = false;
    int my_cx = 0, my_cy = 0;
    if (active) {
      int cx, cy;
      if (!dwa_world_to_map(a.g, px, py, cx, cy)) code = -1.0;  // off the known map (:274-277)
      else {
        const int centre = a.g.cost[cy * (int)a.g.pitch + cx];
        int f = (int)edge_max[lane];
        if (a.nfp < 3)  // CostmapModel::footprintCost without a polygon: the centre cell alone (costmap_model.cpp:61-67)
          f = (centre == kLethal || centre == kInscribed || (centre == kNoInfo && !a.allow_unknown)) ? -1 : centre;
        if (f < 0) code = -1.0;  // the footprint hits an obstacle (:283-285)
        else {
          occ = fmax((double)f, (double)centre);
          if (a.simple_attractor) {
            gd = (px - a.goal_x) * (px - a.goal_x) + (py - a.goal_y) * (py - a.goal_y);
          } else {
            // with heading scoring only the step inside [timestep, timestep + dt) looks at the distance maps (:318-331)
            heading_step = a.heading_scoring && my_time >= a.heading_scoring_timestep && my_time < a.heading_scoring_timestep + dt;
            if (!a.heading_scoring || heading_step) {
              const uint32_t pdi = a.path_dist[cy * (int)a.g.sx + cx], gdi = a.goal_dist[cy * (int)a.g.sx + cx];
              pd = (double)pdi;
              gd = (double)gdi;
              if (n_cells <= gdi || n_cells <= pdi) code = -2.0;  // no clear path to the goal (:337-342)
            }
            my_cx = cx;
            my_cy = cy;
          }
        }
      }
    }
    __syncwarp();
    const unsigned failing = __ballot_sync(0xffffffffu, code != 0.0);
    if (out_pts && active && (!failing || lane < __ffs(failing) - 1) && base + lane < a.points_stride) {
      out_pts[3 * (base + lane)] = px;
      out_pts[3 * (base + lane) + 1] = py;
      out_pts[3 * (base + lane) + 2] = my_th;
    }
    if (failing) {
      const int first = __ffs(failing) - 1;
      fail_code = __shfl_sync(0xffffffffu, code, first);
      n_points = base + first;
      break;
    }
    double m = active ? occ : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    occ_cost = fmax(occ_cost, m);
    if (!a.heading_scoring || a.simple_attractor) {
      path_dist = __shfl_sync(0xffffffffu, pd, cnt - 1);
      goal_dist = __shfl_sync(0xffffffffu, gd, cnt - 1);
    } else {
      const unsigned hs = __ballot_sync(0xffffffffu, heading_step);
      if (hs) {  // at most one step of a trajectory qualifies
        const int src = __ffs(hs) - 1;
        path_dist = __shfl_sync(0xffffffffu, pd, src);
        goal_dist = __shfl_sync(0xffffffffu, gd, src);
        heading_diff = tp_heading_diff(a, __shfl_sync(0xffffffffu, my_cx, src), __shfl_sync(0xffffffffu, my_cy, src),
                                       __shfl_sync(0xffffffffu, px, src), __shfl_sync(0xffffffffu, py, src),
                                       __shfl_sync(0xffffffffu, my_th, src), lane);
      }
    }
    if (base + cnt >= num_steps) {  // the end point, pushed heading_lookahead ahead (:672-681 / :760-769)
      double ag = -1.0;
      if (lane == cnt - 1) {
        int cx, cy;
        if (dwa_world_to_map(a.g, px + a.heading_lookahead * c, py + a.heading_lookahead * s, cx, cy))
          ag = (double)a.goal_dist[cy * (int)a.g.sx + cx];
      }
      ahead = __shfl_sync(0xffffffffu, ag, cnt - 1);
    }
  }
  if (lane == 0) {
    TpSampleResult r;
    const double legal = a.heading_scoring
                             ? a.occdist_scale * occ_cost + a.pdist_scale * path_dist + 0.3 * heading_diff + goal_dist * a.gdist_scale
                             : a.pdist_scale * path_dist + goal_dist * a.gdist_scale + a.occdist_scale * occ_cost;  // :362-367
    r.cost = fail_code != 0.0 ? fail_code : legal;
    r.ahead_gdist = fail_code != 0.0 ? -1.0 : ahead;
    r.n_points = n_points;
    r.pad_ = 0;
    a.out[sample] = r;
  }
}

__global__ void __launch_bounds__(kDwaWarpsPerBlock * 32) k_tp_score(TpScoreArgs a) {
  __shared__ double scratch[kDwaWarpsPerBlock][kWarpScratchDoubles];
  cudaGridDependencySynchronize();  // launched behind the two MapGrid wavefronts
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sample = blockIdx.x * kDwaWarpsPerBlock + warp;
  if (sample >= a.n) return;
  tp_score_sample(a, sample, lane, scratch[warp]);
}

// ---------------------------------------------------------------------------------------------------------------
// FootprintHelper::getFootprintCells(pos, footprint_spec_, costmap_, fill = true), footprint_helper.cpp:180-246, for
// the host (the single planner) and the device (fleets) alike.  Cells are packed y << 16 | x (maps are at most 32767
// cells a side) into a caller-provided buffer of `cap` cells; cos / sin of the heading come from the caller, so both
// sides see the host's libm values.  Returns the number of cells, or -1 when they would not fit (tp_footprint_capacity
// bounds them).  Multiplications are rounded one by one, as the reference's x86-64 code rounds them.
__host__ __device__ __forceinline__ double tp_mul(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}

struct TpCellBuffer {
  uint32_t* cell;
  int n, cap;
  __host__ __device__ bool push(unsigned x, unsigned y) {
    if (n >= cap) return false;
    cell[n++] = (y << 16) | x;
    return true;
  }
};

// Costmap2D::worldToMap (costmap_2d.cpp:208-220)
__host__ __device__ __forceinline__ bool tp_world_to_map(double wx, double wy, double ox, double oy, double res,
                                                         unsigned sx, unsigned sy, unsigned& mx, unsigned& my) {
  if (wx < ox || wy < oy) return false;
  mx = (int)((wx - ox) / res);
  my = (int)((wy - oy) / res);
  return mx < sx && my < sy;
}

// FootprintHelper::getLineCells, footprint_helper.cpp:51-120
__host__ __device__ inline bool tp_line_cells(int x0, int x1, int y0, int y1, TpCellBuffer& out) {
  const int dx = abs(x1 - x0), dy = abs(y1 - y0);
  const int sxi = x1 >= x0 ? 1 : -1, syi = y1 >= y0 ? 1 : -1;
  const bool xmajor = dx >= dy;
  const int den = xmajor ? dx : dy, numadd = xmajor ? dy : dx;
  int num = den / 2, x = x0, y = y0;
  for (int k = 0; k <= den; ++k) {
    if (!out.push((unsigned)x, (unsigned)y)) return false;
    num += numadd;
    if (num >= den) {
      num -= den;
      if (xmajor) y += syi; else x += sxi;
    }
    if (xmajor) x += sxi; else y += syi;
  }
  return true;
}

// FootprintHelper::getFillCells, footprint_helper.cpp:123-178: the outline sorted by x (stable for equal x, as the
// adjacent-swap sort is), then one [min_y, max_y) run per column, appended to the list the walk itself is reading
__host__ __device__ inline bool tp_fill_cells(TpCellBuffer& fp) {
  uint32_t* c = fp.cell;
  for (int k = 1; k < fp.n; ++k) {  // insertion sort by x: stable
    const uint32_t key = c[k];
    int j = k - 1;
    while (j >= 0 && (c[j] & 0xffffu) > (key & 0xffffu)) {
      c[j + 1] = c[j];
      --j;
    }
    c[j + 1] = key;
  }
  int i = 0;
  const unsigned min_x = c[0] & 0xffffu, max_x = c[fp.n - 1] & 0xffffu;
  for (unsigned x = min_x; x <= max_x; ++x) {
    if (i >= fp.n - 1) break;
    uint32_t lo, hi;
    if ((c[i] >> 16) < (c[i + 1] >> 16)) { lo = c[i]; hi = c[i + 1]; }
    else { lo = c[i + 1]; hi = c[i]; }
    i += 2;
    while (i < fp.n && (c[i] & 0xffffu) == x) {
      if ((c[i] >> 16) < (lo >> 16)) lo = c[i];
      else if ((c[i] >> 16) > (hi >> 16)) hi = c[i];
      ++i;
    }
    for (unsigned y = lo >> 16; y < (hi >> 16); ++y)
      if (!fp.push(x, y)) return false;
  }
  return true;
}

__host__ __device__ inline int tp_footprint_cells(const double* fpx, const double* fpy, int nfp, double x_i, double y_i,
                                                  double cos_th, double sin_th, double ox, double oy, double res,
                                                  unsigned sx, unsigned sy, uint32_t* cells, int cap) {
  TpCellBuffer b{cells, 0, cap};
  if (nfp <= 1) {
    unsigned mx, my;
    if (tp_world_to_map(x_i, y_i, ox, oy, res, sx, sy, mx, my) && !b.push(mx, my)) return -1;
    return b.n;
  }
  for (int i = 0; i < nfp; ++i) {  // edges (i, i + 1), the closing edge last
    const int j = i + 1 < nfp ? i + 1 : 0;
    unsigned x0, y0, x1, y1;
    // a vertex off the map: the outline cells gathered so far, unfilled
    if (!tp_world_to_map(x_i + (tp_mul(fpx[i], cos_th) - tp_mul(fpy[i], sin_th)),
                         y_i + (tp_mul(fpx[i], sin_th) + tp_mul(fpy[i], cos_th)), ox, oy, res, sx, sy, x0, y0))
      return b.n;
    if (!tp_world_to_map(x_i + (tp_mul(fpx[j], cos_th) - tp_mul(fpy[j], sin_th)),
                         y_i + (tp_mul(fpx[j], sin_th) + tp_mul(fpy[j], cos_th)), ox, oy, res, sx, sy, x1, y1))
      return b.n;
    if (!tp_line_cells((int)x0, (int)x1, (int)y0, (int)y1, b)) return -1;
  }
  if (!tp_fill_cells(b)) return -1;
  return b.n;
}

// An upper bound of tp_footprint_cells' count for a footprint at any pose and resolution: every edge's line (at most
// its length in cells + 2), plus one run per column of the outline's bounding box, both at most the circumscribed
// diameter + 2 cells long
inline long long tp_footprint_capacity(const double* fpx, const double* fpy, int nfp, double res) {
  if (nfp <= 1) return 1;
  double r = 0.0;
  long long outline = 0;
  for (int i = 0; i < nfp; ++i) {
    const int j = i + 1 < nfp ? i + 1 : 0;
    r = fmax(r, hypot(fpx[i], fpy[i]));
    outline += (long long)(hypot(fpx[j] - fpx[i], fpy[j] - fpy[i]) / res) + 3;
  }
  const long long side = (long long)(2.0 * r / res) + 3;
  return outline + side * side;
}

// ---------------------------------------------------------------------------------------------------------------
// Fleets of legacy TrajectoryPlanners (navgpu_fleet_use_trajectory_planner): what changes per robot and step
struct TpFleetRobot {
  double x, y, theta, vx, vy, vtheta;  // through (float), as navgpu_tp_find_best_path rounds them
  double cos_th, sin_th;               // the host's cos / sin of theta, for the footprint cells
  double ox, oy;                       // the robot's map origin
  double goal_x, goal_y;               // last pose of its plan (0, 0 without one)
  int plan_offset, n_plan;             // its raw plan in the fleet's plan array (n_plan is 0 without heading scoring)
  int sample_offset, n_samples;        // its slice of the step's samples and results
};

struct TpFleetLayout {
  const uint8_t* cost;       // robot r's local costmap at cost + r * cost_stride, row pitch g.pitch
  size_t cost_stride;
  uint32_t* dist;            // robot r: path_map_ at dist + 2r * sx*sy, goal_map_ right after it
  uint32_t* within;          // robot r: MapCell::within_robot bits at within + r * within_words
  int within_words;
  const double* plans_raw;   // every robot's raw plan, (x, y) pairs
  const double* samples;     // n_total x 3
  TpSampleResult* out;       // n_total
  const double* fpx;         // the footprint (device copy), nfp vertices
  const double* fpy;
  int cells_cap;             // tp_footprint_capacity of the footprint
};

// TrajectoryPlanner::findBestPath's path_map_ cells under the robot (trajectory_planner.cpp:918-930) for every robot:
// one warp per robot clears its bit mask while lane 0 gathers the cells in shared memory; the warp then sets them.
// A robot without samples is left out of the step (navgpu_fleet_set_active; an active robot always has the backup
// sample): its bits stay as they are.
__global__ void __launch_bounds__(32) k_tp_fleet_footprint(TpFleetLayout L, const TpFleetRobot* robots, unsigned sx,
                                                           unsigned sy, double res, int nfp) {
  extern __shared__ uint32_t s_cells[];
  __shared__ int s_n;
  const int robot = blockIdx.x, lane = threadIdx.x;
  if (robots[robot].n_samples == 0) return;
  uint32_t* within = L.within + (size_t)robot * L.within_words;
  for (int w = lane; w < L.within_words; w += 32) within[w] = 0u;
  if (lane == 0) {
    const TpFleetRobot& r = robots[robot];
    s_n = tp_footprint_cells(L.fpx, L.fpy, nfp, r.x, r.y, r.cos_th, r.sin_th, r.ox, r.oy, res, sx, sy, s_cells, L.cells_cap);
  }
  __syncwarp();
  const int W = (int)(sx + 31) / 32;
  for (int k = lane; k < s_n; k += 32) {
    const unsigned x = s_cells[k] & 0xffffu, y = s_cells[k] >> 16;
    if (x < sx && y < sy) atomicOr(&within[y * W + (x >> 5)], 1u << (x & 31));
  }
}

// generateTrajectory of every robot's velocity samples in one launch: robot-major CTAs, blocks_per_robot per robot, one
// warp per sample, each CTA scoring against its robot's view of the arguments (no points are stored)
__global__ void __launch_bounds__(kDwaWarpsPerBlock * 32) k_tp_fleet_score(TpScoreArgs base, TpFleetLayout L,
                                                                         const TpFleetRobot* robots, int blocks_per_robot) {
  __shared__ TpScoreArgs s_a;
  __shared__ double scratch[kDwaWarpsPerBlock][kWarpScratchDoubles];
  const int robot = blockIdx.x / blocks_per_robot, local = blockIdx.x % blocks_per_robot;
  const TpFleetRobot& r = robots[robot];
  const int n = r.n_samples;
  if (local * kDwaWarpsPerBlock >= n) return;  // no samples for this CTA
  const uint32_t* src = reinterpret_cast<const uint32_t*>(&base);
  uint32_t* dst = reinterpret_cast<uint32_t*>(&s_a);
  for (int i = threadIdx.x; i < (int)(sizeof(TpScoreArgs) / 4); i += blockDim.x) dst[i] = src[i];
  __syncthreads();
  if (threadIdx.x == 0) {
    const size_t cells = (size_t)base.g.sx * base.g.sy;
    s_a.g.cost = L.cost + (size_t)robot * L.cost_stride;
    s_a.g.ox = r.ox;
    s_a.g.oy = r.oy;
    s_a.path_dist = L.dist + 2 * (size_t)robot * cells;
    s_a.goal_dist = s_a.path_dist + cells;
    s_a.samples = L.samples + 3 * (size_t)r.sample_offset;
    s_a.n = n;
    s_a.x = r.x; s_a.y = r.y; s_a.theta = r.theta;
    s_a.vx = r.vx; s_a.vy = r.vy; s_a.vtheta = r.vtheta;
    s_a.goal_x = r.goal_x;
    s_a.goal_y = r.goal_y;
    s_a.plan_xy = L.plans_raw + 2 * (size_t)r.plan_offset;
    s_a.n_plan = r.n_plan;
    s_a.out = L.out + r.sample_offset;
    s_a.points = nullptr;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sample = local * kDwaWarpsPerBlock + warp;
  if (sample >= n) return;
  tp_score_sample(s_a, sample, lane, scratch[warp]);
}

}  // namespace navgpu
