// dwa.cu -- Path B host side: the DWA rollout scorer behind the navgpu_dwa_* C ABI.
//
// Mirrors dwa_local_planner::DWAPlanner's wiring of base_local_planner's generator, critics and search
// (dwa_local_planner/src/dwa_planner.cpp:52-182, 240-371).  Grid work (4x MapGrid wavefront), rollouts, critics and
// the argmin run in dwa_kernels.cuh; the host keeps the planner's scalar state: configuration, plan geometry,
// the per-axis velocity samples (VelocityIterator is a 20-entry fp64 accumulation) and the oscillation flags.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <limits>
#include <memory>
#include <vector>

#include "dwa_kernels.cuh"
#include "fleet_costmap.cuh"
#include "tp_kernels.cuh"

using namespace navgpu;

namespace {

struct P2 {
  double x, y;
};

// MapGrid::adjustPlanResolution, base_local_planner/src/map_grid.cpp:135-171 (plan geometry only)
void adjust_plan_resolution(const std::vector<P2>& in, std::vector<P2>& out, double resolution) {
  out.clear();
  if (in.empty()) return;
  double last_x = in[0].x, last_y = in[0].y;
  out.push_back(in[0]);
  const double min_sq_resolution = resolution * resolution * 4;
  for (size_t i = 1; i < in.size(); ++i) {
    const double loop_x = in[i].x, loop_y = in[i].y;
    const double sqdist = (loop_x - last_x) * (loop_x - last_x) + (loop_y - last_y) * (loop_y - last_y);
    if (sqdist > min_sq_resolution) {
      const int steps = ((sqrt(sqdist) - sqrt(min_sq_resolution)) / resolution) - 1;
      const double deltax = (loop_x - last_x) / steps, deltay = (loop_y - last_y) / steps;
      for (int j = 1; j < steps; ++j) out.push_back(P2{last_x + j * deltax, last_y + j * deltay});
    }
    out.push_back(in[i]);
    last_x = loop_x;
    last_y = loop_y;
  }
}

// two resolution-adjusted plans with the same points seed the same MapGrid
bool same_plan(const std::vector<P2>& a, const std::vector<P2>& b) {
  return a.size() == b.size() && (a.empty() || memcmp(a.data(), b.data(), a.size() * sizeof(P2)) == 0);
}

// the critic scales of DWAPlanner::reconfigure (dwa_planner.cpp:52-112)
struct DwaScales {
  double path, goal, obstacle, alignment;
};
DwaScales dwa_scales(const navgpu_dwa_config& c, double res) {
  return DwaScales{res * c.path_distance_bias * 0.5, res * c.goal_distance_bias * 0.5, res * c.occdist_scale,
                   res * c.path_distance_bias * 0.5};
}

// DWAPlanner's plan state: one per planner handle, one per fleet robot
struct DwaPlans {
  std::vector<P2> plan;  // as received
  // resolution-adjusted: 0 global plan, 1 front plan, 2 what the alignment critic last received
  std::vector<P2> adjusted[3];
  double alignment_scale = 0;
  bool align_is_path = false;   // adjusted[2] == adjusted[0]: the alignment grid is the path grid, computed once
};

// DWAPlanner::updatePlanAndLocalCosts (dwa_planner.cpp:240-286) for a plan of n > 0 (x, y) points; returns whether the
// alignment critic received new target poses (adjusted[2])
bool update_plan_and_local_costs(DwaPlans& p, const navgpu_dwa_config& c, double res, const double pose[3],
                                 const double* plan_xy, int n) {
  p.plan.resize(n);
  for (int i = 0; i < n; ++i) p.plan[i] = P2{plan_xy[2 * i], plan_xy[2 * i + 1]};
  adjust_plan_resolution(p.plan, p.adjusted[0], res);
  const P2 goal = p.plan.back();
  const float pos[3] = {(float)pose[0], (float)pose[1], (float)pose[2]};
  const double sq_dist = (pos[0] - goal.x) * (pos[0] - goal.x) + (pos[1] - goal.y) * (pos[1] - goal.y);
  std::vector<P2> front = p.plan;
  const double angle_to_goal = atan2(goal.y - pos[1], goal.x - pos[0]);
  front.back().x = front.back().x + c.forward_point_distance * cos(angle_to_goal);
  front.back().y = front.back().y + c.forward_point_distance * sin(angle_to_goal);
  adjust_plan_resolution(front, p.adjusted[1], res);
  const bool align_replaced = sq_dist > c.forward_point_distance * c.forward_point_distance * c.cheat_factor;
  if (align_replaced) {
    p.alignment_scale = dwa_scales(c, res).alignment;
    p.adjusted[2] = p.adjusted[0];
  } else {
    p.alignment_scale = 0.0;  // the alignment critic keeps the target poses it had (:282-285)
  }
  p.align_is_path = same_plan(p.adjusted[2], p.adjusted[0]);
  return align_replaced;
}

// the scoring arguments that come from the configuration, the critic scales and the footprint
void dwa_config_args(const navgpu_dwa_config& c, const DwaScales& s, const double* footprint_xy, int n_footprint,
                     DwaScoreArgs& a) {
  a.acc[0] = (float)c.acc_lim_x; a.acc[1] = (float)c.acc_lim_y; a.acc[2] = (float)c.acc_lim_theta;
  a.min_trans_vel = c.min_trans_vel; a.max_trans_vel = c.max_trans_vel; a.min_rot_vel = c.min_rot_vel;
  a.sim_time = c.sim_time; a.sim_granularity = c.sim_granularity; a.angular_sim_granularity = c.angular_sim_granularity;
  a.use_dwa = c.use_dwa; a.sum_scores = c.sum_scores; a.allow_unknown = c.allow_unknown;
  a.scale_obstacle = s.obstacle;
  a.scale_goal_front = s.goal;
  a.scale_alignment = s.alignment;
  a.scale_path = s.path;
  a.scale_goal = s.goal;
  a.xshift = c.forward_point_distance;
  a.nfp = n_footprint;
  for (int k = 0; k < n_footprint; ++k) { a.fpx[k] = footprint_xy[2 * k]; a.fpy[k] = footprint_xy[2 * k + 1]; }
}

constexpr int kPointsCapacity = 4096;

struct Cycle {
  DwaScoreArgs args;
  long long n_samples = 0;
};

}  // namespace

namespace {
// Upload of a small host grid (the local costmap a planner scores against) without waiting for the stream: the rows
// are copied into a pinned staging buffer owned by the handle and go to the device asynchronously; the buffer is
// reused once the previous upload from it has completed (event).
int stage_grid_upload(uint8_t** stage, cudaEvent_t* ev, uint8_t* dev, unsigned pitch, const uint8_t* host_grid, unsigned sx,
                      unsigned sy, cudaStream_t stream) {
  const size_t bytes = size_t(sx) * sy;
  if (!*stage) {
    NAVGPU_CUDA(cudaMallocHost(stage, bytes));
    NAVGPU_CUDA(cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
  } else {
    NAVGPU_CUDA(cudaEventSynchronize(*ev));
  }
  memcpy(*stage, host_grid, bytes);
  NAVGPU_CUDA(cudaMemcpy2DAsync(dev, pitch, *stage, sx, sx, sy, cudaMemcpyHostToDevice, stream));
  NAVGPU_CUDA(cudaEventRecord(*ev, stream));
  return NAVGPU_OK;
}
}  // namespace

struct navgpu_dwa {
  int device = 0;
  cudaStream_t stream = nullptr;
  navgpu_dwa_config cfg;
  unsigned sx = 0, sy = 0;
  double res = 0;
  // local costmap: own copy (set_costmap) or a borrowed device grid (set_costmap_device)
  uint8_t* d_cost_own = nullptr;
  const uint8_t* d_cost = nullptr;
  uint8_t* h_cost_stage = nullptr;  // pinned staging of set_costmap
  cudaEvent_t ev_cost_stage = nullptr;
  unsigned pitch = 0;
  double ox = 0, oy = 0;
  DwaPlans plans;
  double* d_plan[3] = {nullptr, nullptr, nullptr};  // device copies of plans.adjusted
  size_t plan_capacity[3] = {0, 0, 0};
  bool plan_dirty[3] = {false, false, false};
  bool align_aliased = false;  // the grids of the last prepare() were laid out with plans.align_is_path
  DwaScales scales = {};
  uint32_t* d_dist[4] = {nullptr, nullptr, nullptr, nullptr};
  float* d_samples = nullptr;
  size_t samples_capacity = 0;
  float* h_samples_stage = nullptr;  // pinned staging of the per-axis samples
  size_t samples_stage_capacity = 0;
  cudaEvent_t ev_samples_stage = nullptr;
  bool samples_on_device = false;  // d_samples holds last_samples
  double* d_block_cost = nullptr;
  long long* d_block_index = nullptr;
  size_t block_capacity = 0;
  unsigned int* d_counters = nullptr;
  double* d_best_cost = nullptr;
  long long* d_best_index = nullptr;
  DwaDeviceResult* h_result = nullptr;  // pinned + mapped: written by the finishing step on the device
  double* h_points = nullptr;           // pinned + mapped
  double* h_best = nullptr;             // pinned: cost, index (as long long bits)
  double* d_terms = nullptr;
  double* d_reported = nullptr;
  size_t terms_capacity = 0;
  Oscillation osc;
  // result_traj_ persists across cycles (dwa_planner.cpp:316, simple_scored_sampling_planner.cpp:123-134)
  double res_v[3] = {0, 0, 0};
  std::vector<double> res_points;
  long long n_samples_last = 0;
  bool have_last = false;
  Cycle last;  // arguments of the last score_range launch (for finish_sharded)
  // sharded sweeps with the device-side exchange (navgpu_dwa_shard_*)
  ShardExchange* d_shard = nullptr;                 // this rank's exchange buffer
  ShardExchange* shard_peer[kShardMaxWorld] = {};   // every rank's buffer as mapped here
  bool shard_ipc[kShardMaxWorld] = {};              // opened with cudaIpcOpenMemHandle (to be closed)
  int shard_rank = 0, shard_world = 0;
  unsigned long long shard_seq = 0;
  Cycle shard_cycle;
  bool shard_pending = false;
  // TrajectoryCostFunction backend (navgpu_dwa_score_trajectories): device copies of the caller's trajectories
  char* d_traj = nullptr;
  size_t traj_capacity = 0;
  std::vector<float> last_samples;  // per-axis samples of the last search (xs | ys | ths), see navgpu_dwa_get_samples
  int last_nx = 0, last_ny = 0, last_nth = 0;
};

namespace {

int use_device(navgpu_dwa* h) {
  NAVGPU_CUDA(cudaSetDevice(h->device));
  return NAVGPU_OK;
}

void apply_config(navgpu_dwa* h) {  // DWAPlanner::reconfigure, dwa_planner.cpp:52-112
  h->scales = dwa_scales(h->cfg, h->res);
  h->plans.alignment_scale = h->scales.alignment;
}

int upload_plan(navgpu_dwa* h, int k) {
  if (!h->plan_dirty[k]) return NAVGPU_OK;
  const std::vector<P2>& v = h->plans.adjusted[k];
  if (v.size() > h->plan_capacity[k]) {
    if (h->d_plan[k]) cudaFree(h->d_plan[k]);
    h->d_plan[k] = nullptr;
    const size_t cap = std::max<size_t>(256, v.size() * 2);
    NAVGPU_CUDA(cudaMalloc(&h->d_plan[k], cap * sizeof(P2)));
    h->plan_capacity[k] = cap;
  }
  if (!v.empty()) {
    NAVGPU_CUDA(cudaMemcpyAsync(h->d_plan[k], v.data(), v.size() * sizeof(P2), cudaMemcpyHostToDevice, h->stream));
    NAVGPU_CUDA(cudaStreamSynchronize(h->stream));  // pageable source owned by the handle
  }
  h->plan_dirty[k] = false;
  return NAVGPU_OK;
}

// SimpleTrajectoryGenerator::initialise, simple_trajectory_generator.cpp:60-135: the per-axis samples
struct Samples {
  std::vector<float> v;  // xs | ys | ths
  int nx = 0, ny = 0, nth = 0;
};
Samples enumerate_samples(const navgpu_dwa_config& cfg, const float pos[3], const float vel[3], const float goal[2]) {
  Samples s;
  int n[3], c[3];
  dwa_axis_samples(cfg, n);
  s.v.resize(size_t(dwa_axis_bound(n[0])) + dwa_axis_bound(n[1]) + dwa_axis_bound(n[2]));
  navgpu::enumerate_samples(cfg, pos, vel, goal, s.v.data(), c);
  s.nx = c[0]; s.ny = c[1]; s.nth = c[2];
  s.v.resize(size_t(c[0]) + c[1] + c[2]);
  return s;
}

// MapGridCostFunction::prepare for `n_ctas` grids of sx x sy cells (jobs_per_robot per robot): the register-resident
// bit-sliced kernel when the map's bit words fit 4 per thread, else the general shared-memory kernel
int launch_mapgrid(unsigned sx, unsigned sy, cudaStream_t stream, const MapGridArgs& ma, int n_ctas, int jobs_per_robot) {
  const int W = (sx + 31) / 32, NW = W * (int)sy;
  int planes = 1;
  while ((1ull << planes) <= (unsigned long long)sx * sy + 1) ++planes;  // levels go up to n_cells
  const size_t sliced_smem = (size_t(3 + planes) * NW + 2) * sizeof(uint32_t);
  const int wpt = (NW + kMapGridThreads - 1) / kMapGridThreads;
  // maps of at most 128 x 128 cells: the row kernel (registers + warp shuffles, a barrier per 16 levels).  A
  // planner's few grids run with 512 threads per CTA -- the warps beyond the search warps help with the passable bits,
  // the seeds and the epilogue; a fleet's thousands of grids run the search warps only.
  // NAVGPU_MAPGRID=sliced | rows and NAVGPU_MAPGRID_HELPERS=0 | 1 force a variant (tests, measurements).
  const char* force = getenv("NAVGPU_MAPGRID");
  const char* force_helpers = getenv("NAVGPU_MAPGRID_HELPERS");
  const bool rows_fit = sx <= 128 && sy <= 128;
  if (rows_fit && !(force && !strcmp(force, "sliced"))) {
    const bool helpers = force_helpers ? atoi(force_helpers) != 0 : n_ctas < 1024;
    const size_t smem = size_t(15) * NW * sizeof(uint32_t);
    k_mapgrid_prepare_rows<4, 2, 8><<<n_ctas, helpers ? 512 : 128, smem, stream>>>(ma, jobs_per_robot);
  } else if (wpt <= 4 && planes <= kMapGridMaxPlanes && sliced_smem <= 200 * 1024) {
    auto launch = [&](auto kernel) -> int {
      if (sliced_smem > 48 * 1024)
        NAVGPU_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sliced_smem));
      kernel<<<n_ctas, kMapGridThreads, sliced_smem, stream>>>(ma, jobs_per_robot, planes);
      return NAVGPU_OK;
    };
    switch (wpt) {
      case 1: NAVGPU_TRY(launch(k_mapgrid_prepare_sliced<1>)); break;
      case 2: NAVGPU_TRY(launch(k_mapgrid_prepare_sliced<2>)); break;
      case 3: NAVGPU_TRY(launch(k_mapgrid_prepare_sliced<3>)); break;
      default: NAVGPU_TRY(launch(k_mapgrid_prepare_sliced<4>)); break;
    }
  } else {
    const size_t mg_smem = size_t(4) * NW * sizeof(uint32_t);
    if (mg_smem > 200 * 1024) return fail(NAVGPU_ERR_UNSUPPORTED, "local costmap %ux%u too large for the MapGrid kernel", sx, sy);
    if (mg_smem > 48 * 1024)
      NAVGPU_CUDA(cudaFuncSetAttribute(k_mapgrid_prepare, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mg_smem));
    k_mapgrid_prepare<<<n_ctas, kMapGridThreads, mg_smem, stream>>>(ma, jobs_per_robot);
  }
  NAVGPU_LAUNCHED(1);
  return NAVGPU_OK;
}

// prepare() of the critics (simple_scored_sampling_planner.cpp:87-93): the plans reach the device, then four MapGrid
// wavefronts, one CTA each
int prepare_grids(navgpu_dwa* h, const DwaGeom& g) {
  for (int k = 0; k < 3; ++k) NAVGPU_TRY(upload_plan(h, k));
  MapGridArgs ma;
  ma.g = g;
  ma.allow_unknown = h->cfg.allow_unknown;
  const std::vector<P2>* adjusted = h->plans.adjusted;
  ma.job[0] = MapGridJob{h->d_plan[0], (int)adjusted[0].size(), 0, h->d_dist[0]};  // path: setTargetCells
  ma.job[1] = MapGridJob{h->d_plan[0], (int)adjusted[0].size(), 1, h->d_dist[1]};  // goal: setLocalGoal
  ma.job[2] = MapGridJob{h->d_plan[1], (int)adjusted[1].size(), 1, h->d_dist[2]};  // goal_front
  ma.job[3] = MapGridJob{h->d_plan[2], (int)adjusted[2].size(), 0, h->d_dist[3]};  // alignment
  if (h->plans.align_is_path) {  // same poses, same mode as the path grid: one wavefront serves both critics
    ma.job[3].dist = h->d_dist[0];
    ma.job[3].skip = 1;
  }
  ma.fleet = nullptr;
  NAVGPU_TRY(launch_mapgrid(h->sx, h->sy, h->stream, ma, 4, 4));
  h->align_aliased = h->plans.align_is_path;
  return NAVGPU_OK;
}

// the critics' part of the scoring arguments: geometry, distance grids, scales, footprint, flags
int critic_args(navgpu_dwa* h, const DwaGeom& g, const double* footprint_xy, int n_footprint, DwaScoreArgs& a) {
  if (n_footprint < 0 || n_footprint > kMaxFootprint) return fail(NAVGPU_ERR_UNSUPPORTED, "footprint with more than %d vertices", kMaxFootprint);
  dwa_config_args(h->cfg, h->scales, footprint_xy, n_footprint, a);
  a.scale_alignment = h->plans.alignment_scale;  // 0 near the goal (set_plan)
  a.g = g;
  for (int k = 0; k < 4; ++k) a.dist[k] = h->d_dist[k];
  if (h->align_aliased) a.dist[3] = h->d_dist[0];
  a.osc_mask = h->osc.mask();
  return NAVGPU_OK;
}

// uploads the per-cycle inputs and launches the 4 MapGrid wavefronts; fills the scoring arguments
int begin_cycle(navgpu_dwa* h, const double pose[3], const double velv[3], const double* footprint_xy, int n_footprint,
                Cycle& cy, bool prepare = true) {
  NAVGPU_TRY(use_device(h));
  if (!h->d_cost) return fail(NAVGPU_ERR_INVALID, "no costmap set");
  if (h->plans.plan.empty()) return fail(NAVGPU_ERR_INVALID, "no plan set");
  if (n_footprint < 0 || n_footprint > kMaxFootprint) return fail(NAVGPU_ERR_UNSUPPORTED, "footprint with more than %d vertices", kMaxFootprint);
  const float pos[3] = {(float)pose[0], (float)pose[1], (float)pose[2]};  // Eigen::Vector3f, dwa_planner.cpp:303-306
  const float vel[3] = {(float)velv[0], (float)velv[1], (float)velv[2]};
  const float goal[2] = {(float)h->plans.plan.back().x, (float)h->plans.plan.back().y};
  Samples s = enumerate_samples(h->cfg, pos, vel, goal);
  const bool inline_samples = s.v.size() <= (size_t)kInlineSamples;  // they then travel in the kernel parameters
  if (!inline_samples) {
    if (s.v.size() > h->samples_capacity) {
      if (h->d_samples) cudaFree(h->d_samples);
      h->d_samples = nullptr;
      NAVGPU_CUDA(cudaMalloc(&h->d_samples, s.v.size() * 2 * sizeof(float)));
      h->samples_capacity = s.v.size() * 2;
      h->samples_on_device = false;
    }
    // the samples only change with the robot's velocity and the limits: an identical set is already on the device; a new
    // one goes through a pinned staging buffer (no wait for the stream)
    if (!h->samples_on_device || s.v != h->last_samples) {
      const size_t bytes = s.v.size() * sizeof(float);
      if (bytes > h->samples_stage_capacity) {
        if (h->h_samples_stage) cudaFreeHost(h->h_samples_stage);
        h->h_samples_stage = nullptr;
        NAVGPU_CUDA(cudaMallocHost(&h->h_samples_stage, 2 * bytes));
        h->samples_stage_capacity = 2 * bytes;
      }
      if (!h->ev_samples_stage) NAVGPU_CUDA(cudaEventCreateWithFlags(&h->ev_samples_stage, cudaEventDisableTiming));
      else NAVGPU_CUDA(cudaEventSynchronize(h->ev_samples_stage));
      memcpy(h->h_samples_stage, s.v.data(), bytes);
      NAVGPU_CUDA(cudaMemcpyAsync(h->d_samples, h->h_samples_stage, bytes, cudaMemcpyHostToDevice, h->stream));
      NAVGPU_CUDA(cudaEventRecord(h->ev_samples_stage, h->stream));
      h->samples_on_device = true;
    }
  } else {
    h->samples_on_device = false;
  }
  h->last_samples = s.v;
  h->last_nx = s.nx; h->last_ny = s.ny; h->last_nth = s.nth;

  DwaGeom g{h->d_cost, h->sx, h->sy, h->pitch, h->res, h->ox, h->oy, 1.0 / h->res};
  if (prepare) NAVGPU_TRY(prepare_grids(h, g));

  DwaScoreArgs& a = cy.args;
  NAVGPU_TRY(critic_args(h, g, footprint_xy, n_footprint, a));
  a.vxs = h->d_samples;
  a.vys = h->d_samples + s.nx;
  a.vths = h->d_samples + s.nx + s.ny;
  a.nx = s.nx; a.ny = s.ny; a.nth = s.nth;
  a.inline_samples = inline_samples ? 1 : 0;
  if (inline_samples) memcpy(a.samples_inline, s.v.data(), s.v.size() * sizeof(float));
  cy.n_samples = (long long)s.nx * s.ny * s.nth;
  a.begin = 0;
  a.end = cy.n_samples;
  a.stride_rank = 0;
  a.stride_world = 1;
  for (int k = 0; k < kShardMaxWorld; ++k) a.shard_peer[k] = nullptr;
  a.shard_seq = 0;
  for (int k = 0; k < 3; ++k) { a.pos[k] = pos[k]; a.vel[k] = vel[k]; }
  a.all_terms = nullptr;
  a.counters = h->d_counters;
  a.best_cost = h->d_best_cost;
  a.best_index = h->d_best_index;
  a.finish_out = nullptr;
  a.finish_points = nullptr;
  a.finish_capacity = 0;
  h->n_samples_last = cy.n_samples;
  return NAVGPU_OK;
}

int launch_score(navgpu_dwa* h, Cycle& cy, bool finish) {
  DwaScoreArgs& a = cy.args;
  const long long n = a.end - a.begin;
  if (n <= 0) return fail(NAVGPU_ERR_INVALID, "empty sample range");
  const long long all_blocks = (n + kDwaWarpsPerBlock - 1) / kDwaWarpsPerBlock;
  // block-cyclic share of this rank (every rank launches at least one CTA so that its exchange step runs)
  const long long blocks = std::max<long long>(1, (all_blocks - a.stride_rank + a.stride_world - 1) / a.stride_world);
  if (blocks > 0x7fffffffLL) return fail(NAVGPU_ERR_UNSUPPORTED, "too many samples in one launch");
  if ((size_t)blocks > h->block_capacity) {
    if (h->d_block_cost) cudaFree(h->d_block_cost);
    if (h->d_block_index) cudaFree(h->d_block_index);
    h->d_block_cost = nullptr;
    h->d_block_index = nullptr;
    NAVGPU_CUDA(cudaMalloc(&h->d_block_cost, blocks * sizeof(double)));
    NAVGPU_CUDA(cudaMalloc(&h->d_block_index, blocks * sizeof(long long)));
    h->block_capacity = blocks;
  }
  a.block_cost = h->d_block_cost;
  a.block_index = h->d_block_index;
  if (finish) {  // the last CTA regenerates the winner into mapped host memory and re-arms both counters
    a.finish_out = h->h_result;
    a.finish_points = h->h_points;
    a.finish_capacity = kPointsCapacity;
  } else {
    NAVGPU_CUDA(cudaMemsetAsync(h->d_counters, 0, 2 * sizeof(unsigned int), h->stream));
  }
  NAVGPU_CUDA(launch_pdl(k_dwa_score, dim3((unsigned)blocks), dim3(kDwaWarpsPerBlock * 32), 0, h->stream, a));
  NAVGPU_LAUNCHED(1);
  return NAVGPU_OK;
}

}  // namespace

extern "C" {

void navgpu_dwa_default_config(navgpu_dwa_config* c) {
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

int navgpu_dwa_create(navgpu_dwa** out, const navgpu_dwa_config* cfg, uint32_t size_x, uint32_t size_y,
                      double resolution, int device) {
  if (!out || !cfg || size_x == 0 || size_y == 0 || !(resolution > 0)) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (navgpu_device_count() <= device) return fail(NAVGPU_ERR_CUDA, "no CUDA device %d (libnavgpu has no CPU fallback)", device);
  if ((unsigned long long)size_x * size_y + 1 >= 0xffffffffull || size_x > 32767 || size_y > 32767)
    return fail(NAVGPU_ERR_UNSUPPORTED, "local costmap too large");
  std::unique_ptr<navgpu_dwa> h(new navgpu_dwa);
  h->device = device;
  h->cfg = *cfg;
  h->sx = size_x; h->sy = size_y; h->res = resolution;
  NAVGPU_CUDA(cudaSetDevice(device));
  NAVGPU_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  for (int k = 0; k < 4; ++k) NAVGPU_CUDA(cudaMalloc(&h->d_dist[k], size_t(size_x) * size_y * sizeof(uint32_t)));
  NAVGPU_CUDA(cudaMalloc(&h->d_counters, 2 * sizeof(unsigned int)));
  NAVGPU_CUDA(cudaMemset(h->d_counters, 0, 2 * sizeof(unsigned int)));
  NAVGPU_CUDA(cudaMalloc(&h->d_best_cost, sizeof(double)));
  NAVGPU_CUDA(cudaMalloc(&h->d_best_index, sizeof(long long)));
  // result record and winner points are written by the kernels straight into mapped pinned host memory (unified
  // addressing: the same pointer is valid on the device)
  NAVGPU_CUDA(cudaHostAlloc(&h->h_result, sizeof(DwaDeviceResult), cudaHostAllocMapped));
  NAVGPU_CUDA(cudaHostAlloc(&h->h_points, size_t(kPointsCapacity) * 3 * sizeof(double), cudaHostAllocMapped));
  NAVGPU_CUDA(cudaMallocHost(&h->h_best, 2 * sizeof(double)));
  apply_config(h.get());
  *out = h.release();
  return NAVGPU_OK;
}

int navgpu_dwa_destroy(navgpu_dwa* h) {
  if (!h) return NAVGPU_OK;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  cudaFree(h->d_cost_own);
  if (h->h_cost_stage) cudaFreeHost(h->h_cost_stage);
  if (h->h_samples_stage) cudaFreeHost(h->h_samples_stage);
  if (h->ev_samples_stage) cudaEventDestroy(h->ev_samples_stage);
  if (h->ev_cost_stage) cudaEventDestroy(h->ev_cost_stage);
  for (int k = 0; k < 3; ++k) cudaFree(h->d_plan[k]);
  for (int k = 0; k < 4; ++k) cudaFree(h->d_dist[k]);
  cudaFree(h->d_samples); cudaFree(h->d_block_cost); cudaFree(h->d_block_index); cudaFree(h->d_counters);
  cudaFree(h->d_best_cost); cudaFree(h->d_best_index);
  cudaFree(h->d_terms); cudaFree(h->d_reported);
  for (int r = 0; r < kShardMaxWorld; ++r)
    if (h->shard_ipc[r] && h->shard_peer[r]) cudaIpcCloseMemHandle(h->shard_peer[r]);
  cudaFree(h->d_shard);
  cudaFree(h->d_traj);
  cudaFreeHost(h->h_result); cudaFreeHost(h->h_points); cudaFreeHost(h->h_best);
  cudaStreamDestroy(h->stream);
  delete h;
  return NAVGPU_OK;
}

int navgpu_dwa_reconfigure(navgpu_dwa* h, const navgpu_dwa_config* cfg) {
  if (!h || !cfg) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  h->cfg = *cfg;
  apply_config(h);
  return NAVGPU_OK;
}

int navgpu_dwa_set_costmap(navgpu_dwa* h, const uint8_t* host_grid, double origin_x, double origin_y) {
  if (!h || !host_grid) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  NAVGPU_TRY(use_device(h));
  const unsigned pitch = grid_pitch(h->sx);
  if (!h->d_cost_own) NAVGPU_CUDA(cudaMalloc(&h->d_cost_own, size_t(pitch) * h->sy));
  NAVGPU_TRY(stage_grid_upload(&h->h_cost_stage, &h->ev_cost_stage, h->d_cost_own, pitch, host_grid, h->sx, h->sy, h->stream));
  h->d_cost = h->d_cost_own;
  h->pitch = pitch;
  h->ox = origin_x;
  h->oy = origin_y;
  return NAVGPU_OK;
}

int navgpu_dwa_set_costmap_device(navgpu_dwa* h, const uint8_t* dev_grid, uint32_t pitch, double origin_x, double origin_y) {
  if (!h || !dev_grid || pitch < h->sx) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  h->d_cost = dev_grid;
  h->pitch = pitch;
  h->ox = origin_x;
  h->oy = origin_y;
  return NAVGPU_OK;
}

int navgpu_dwa_set_plan(navgpu_dwa* h, const double pose[3], const double* plan_xy, int n) {
  if (!h || !pose || !plan_xy || n <= 0) return fail(NAVGPU_ERR_INVALID, "bad plan");
  if (update_plan_and_local_costs(h->plans, h->cfg, h->res, pose, plan_xy, n)) h->plan_dirty[2] = true;
  h->plan_dirty[0] = h->plan_dirty[1] = true;
  return NAVGPU_OK;
}

int navgpu_dwa_reset_oscillation(navgpu_dwa* h) {
  if (!h) return fail(NAVGPU_ERR_INVALID, "null handle");
  h->osc.reset();
  return NAVGPU_OK;
}

int navgpu_dwa_get_oscillation_mask(navgpu_dwa* h, int* mask_out) {
  if (!h || !mask_out) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  *mask_out = h->osc.mask();
  return NAVGPU_OK;
}

// waits for the finishing step, then applies what findBestPath does with the winner on the host
static int collect(navgpu_dwa* h, Cycle& cy, const double pose[3], navgpu_dwa_result* result, double* best_points,
                   int points_capacity) {
  NAVGPU_CUDA(cudaGetLastError());
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  const DwaDeviceResult& r = *h->h_result;
  if (r.cost >= 0) h->res_points.assign(h->h_points, h->h_points + size_t(3) * r.n_points);
  apply_dwa_result(r, h->cfg, pose, (int32_t)cy.n_samples, h->res_v, h->osc, result);
  if (result) result->n_points = (int32_t)(h->res_points.size() / 3);
  if (best_points) {
    const size_t n = std::min<size_t>(h->res_points.size() / 3, (size_t)std::max(0, points_capacity));
    memcpy(best_points, h->res_points.data(), n * 3 * sizeof(double));
  }
  return NAVGPU_OK;
}

int navgpu_dwa_find_best_path(navgpu_dwa* h, const double pose[3], const double vel[3], const double* footprint_xy,
                              int n_footprint, navgpu_dwa_result* result, double* all_costs, int all_capacity,
                              double* best_points, int points_capacity) {
  if (!h || !pose || !vel || (n_footprint > 0 && !footprint_xy)) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  Cycle cy;
  NAVGPU_TRY(begin_cycle(h, pose, vel, footprint_xy, n_footprint, cy));
  if (all_costs) {
    const size_t need = size_t(cy.n_samples);
    if (need > h->terms_capacity) {
      if (h->d_terms) cudaFree(h->d_terms);
      if (h->d_reported) cudaFree(h->d_reported);
      h->d_terms = h->d_reported = nullptr;
      NAVGPU_CUDA(cudaMalloc(&h->d_terms, need * 6 * sizeof(double)));
      NAVGPU_CUDA(cudaMalloc(&h->d_reported, need * sizeof(double)));
      h->terms_capacity = need;
    }
    cy.args.all_terms = h->d_terms;
  }
  NAVGPU_TRY(launch_score(h, cy, true));
  if (all_costs) {
    k_dwa_report<<<1, 1024, 0, h->stream>>>(h->d_terms, h->d_reported, cy.n_samples);
    NAVGPU_LAUNCHED(1);
  }
  NAVGPU_TRY(collect(h, cy, pose, result, best_points, points_capacity));
  if (all_costs) {
    const size_t n = std::min<size_t>((size_t)cy.n_samples, (size_t)std::max(0, all_capacity));
    NAVGPU_CUDA(cudaMemcpy(all_costs, h->d_reported, n * sizeof(double), cudaMemcpyDeviceToHost));
  }
  return NAVGPU_OK;
}

int navgpu_dwa_find_best_path_async(navgpu_dwa* h, const double pose[3], const double vel[3], const double* footprint_xy,
                                    int n_footprint) {
  if (!h || !pose || !vel) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  Cycle cy;
  NAVGPU_TRY(begin_cycle(h, pose, vel, footprint_xy, n_footprint, cy));
  NAVGPU_TRY(launch_score(h, cy, true));
  NAVGPU_CUDA(cudaGetLastError());
  return NAVGPU_OK;
}

int navgpu_dwa_check_trajectory(navgpu_dwa* h, const double pose[3], const double vel[3], const double vel_samples[3],
                                const double* footprint_xy, int n_footprint, double* cost_out) {
  if (!h || !pose || !vel || !vel_samples || !cost_out || (n_footprint > 0 && !footprint_xy))
    return fail(NAVGPU_ERR_INVALID, "bad arguments");
  h->osc.reset();  // dwa_planner.cpp:217
  Cycle cy;
  NAVGPU_TRY(begin_cycle(h, pose, vel, footprint_xy, n_footprint, cy, false));  // critics keep their last prepare()
  DwaScoreArgs& a = cy.args;
  a.nx = a.ny = a.nth = 1;
  a.inline_samples = 1;
  for (int k = 0; k < 3; ++k) a.samples_inline[k] = (float)vel_samples[k];  // Eigen::Vector3f vel_samples
  a.begin = 0;
  a.end = 1;
  a.osc_mask = 0;
  double* out = reinterpret_cast<double*>(h->h_points);  // mapped pinned scratch
  k_dwa_check<<<1, 32, 0, h->stream>>>(a, out);
  NAVGPU_LAUNCHED(1);
  NAVGPU_CUDA(cudaGetLastError());
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  *cost_out = *out;
  return NAVGPU_OK;
}

// ---- the batched TrajectoryCostFunction backend ---------------------------------------------------------------------
int navgpu_dwa_prepare(navgpu_dwa* h) {
  if (!h) return fail(NAVGPU_ERR_INVALID, "null handle");
  NAVGPU_TRY(use_device(h));
  if (!h->d_cost) return fail(NAVGPU_ERR_INVALID, "no costmap set");
  if (h->plans.plan.empty()) return fail(NAVGPU_ERR_INVALID, "no plan set");
  const DwaGeom g{h->d_cost, h->sx, h->sy, h->pitch, h->res, h->ox, h->oy, 1.0 / h->res};
  NAVGPU_TRY(prepare_grids(h, g));
  NAVGPU_CUDA(cudaGetLastError());
  return NAVGPU_OK;
}

int navgpu_dwa_score_trajectories(navgpu_dwa* h, int n_traj, const int32_t* offsets, const double* points_xyth,
                                  const double* vels, const double* footprint_xy, int n_footprint, double* costs_out,
                                  double* terms_out) {
  if (!h || n_traj < 0 || (n_traj > 0 && (!offsets || !vels || !costs_out)) || (n_footprint > 0 && !footprint_xy))
    return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (n_traj == 0) return NAVGPU_OK;
  NAVGPU_TRY(use_device(h));
  if (!h->d_cost) return fail(NAVGPU_ERR_INVALID, "no costmap set");
  const long long n_points = offsets[n_traj];
  if (offsets[0] != 0 || n_points < 0 || (n_points > 0 && !points_xyth)) return fail(NAVGPU_ERR_INVALID, "bad trajectory offsets");
  for (int t = 0; t < n_traj; ++t)
    if (offsets[t + 1] < offsets[t]) return fail(NAVGPU_ERR_INVALID, "trajectory offsets must not decrease");
  // device copies: [points | vels | costs | terms | offsets]
  const size_t b_points = size_t(n_points) * 3 * sizeof(double), b_vels = size_t(n_traj) * 3 * sizeof(double),
               b_costs = size_t(n_traj) * sizeof(double), b_terms = terms_out ? size_t(n_traj) * 6 * sizeof(double) : 0,
               b_off = size_t(n_traj + 1) * sizeof(int32_t);
  const size_t need = b_points + b_vels + b_costs + b_terms + b_off;
  if (need > h->traj_capacity) {
    if (h->d_traj) cudaFree(h->d_traj);
    h->d_traj = nullptr;
    NAVGPU_CUDA(cudaMalloc(&h->d_traj, 2 * need));
    h->traj_capacity = 2 * need;
  }
  double* d_points = reinterpret_cast<double*>(h->d_traj);
  double* d_vels = reinterpret_cast<double*>(h->d_traj + b_points);
  double* d_costs = reinterpret_cast<double*>(h->d_traj + b_points + b_vels);
  double* d_terms = terms_out ? reinterpret_cast<double*>(h->d_traj + b_points + b_vels + b_costs) : nullptr;
  int* d_off = reinterpret_cast<int*>(h->d_traj + b_points + b_vels + b_costs + b_terms);
  if (b_points) NAVGPU_CUDA(cudaMemcpyAsync(d_points, points_xyth, b_points, cudaMemcpyHostToDevice, h->stream));
  NAVGPU_CUDA(cudaMemcpyAsync(d_vels, vels, b_vels, cudaMemcpyHostToDevice, h->stream));
  NAVGPU_CUDA(cudaMemcpyAsync(d_off, offsets, b_off, cudaMemcpyHostToDevice, h->stream));
  DwaScoreArgs a;
  memset(&a, 0, sizeof(a));
  const DwaGeom g{h->d_cost, h->sx, h->sy, h->pitch, h->res, h->ox, h->oy, 1.0 / h->res};
  NAVGPU_TRY(critic_args(h, g, footprint_xy, n_footprint, a));
  const int blocks = (n_traj + kDwaWarpsPerBlock - 1) / kDwaWarpsPerBlock;
  k_dwa_score_points<<<blocks, kDwaWarpsPerBlock * 32, 0, h->stream>>>(a, d_off, d_points, d_vels, n_traj, d_costs, d_terms);
  NAVGPU_LAUNCHED(1);
  NAVGPU_CUDA(cudaGetLastError());
  NAVGPU_CUDA(cudaMemcpyAsync(costs_out, d_costs, b_costs, cudaMemcpyDeviceToHost, h->stream));
  if (terms_out) NAVGPU_CUDA(cudaMemcpyAsync(terms_out, d_terms, b_terms, cudaMemcpyDeviceToHost, h->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  return NAVGPU_OK;
}

int navgpu_dwa_update_oscillation(navgpu_dwa* h, const double pose[3], double cost, double xv, double yv, double thetav) {
  if (!h || !pose) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  const float pos[3] = {(float)pose[0], (float)pose[1], (float)pose[2]};
  h->osc.update(pos, cost, xv, yv, thetav, h->cfg.min_trans_vel, h->cfg.oscillation_reset_dist, h->cfg.oscillation_reset_angle);
  return NAVGPU_OK;
}

int navgpu_dwa_get_samples(navgpu_dwa* h, int32_t counts_out[3], float* samples_out, int capacity) {
  if (!h || !counts_out || capacity < 0 || (capacity > 0 && !samples_out)) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  counts_out[0] = h->last_nx; counts_out[1] = h->last_ny; counts_out[2] = h->last_nth;
  const size_t n = std::min<size_t>(h->last_samples.size(), (size_t)capacity);
  if (n) memcpy(samples_out, h->last_samples.data(), n * sizeof(float));
  return h->last_samples.size() > (size_t)capacity ? fail(NAVGPU_ERR_CAPACITY, "samples_out too small") : NAVGPU_OK;
}

int navgpu_dwa_score_range(navgpu_dwa* h, const double pose[3], const double vel[3], const double* footprint_xy,
                           int n_footprint, int64_t begin, int64_t end, double* best_cost, int64_t* best_index,
                           int64_t* n_samples_total) {
  if (!h || !pose || !vel || !best_cost || !best_index) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  Cycle cy;
  NAVGPU_TRY(begin_cycle(h, pose, vel, footprint_xy, n_footprint, cy));
  if (n_samples_total) *n_samples_total = cy.n_samples;
  begin = std::max<int64_t>(0, begin);
  end = std::min<int64_t>(cy.n_samples, end);
  if (end <= begin) {
    h->last = cy;
    h->have_last = true;
    *best_cost = std::numeric_limits<double>::infinity();
    *best_index = -1;
    NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
    return NAVGPU_OK;
  }
  cy.args.begin = begin;
  cy.args.end = end;
  NAVGPU_TRY(launch_score(h, cy, false));
  NAVGPU_CUDA(cudaGetLastError());
  h->last = cy;
  h->have_last = true;
  NAVGPU_CUDA(cudaMemcpyAsync(&h->h_best[0], h->d_best_cost, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  NAVGPU_CUDA(cudaMemcpyAsync(&h->h_best[1], h->d_best_index, sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  *best_cost = h->h_best[0];
  long long idx;
  memcpy(&idx, &h->h_best[1], sizeof(idx));
  *best_index = idx;
  return NAVGPU_OK;
}

int navgpu_dwa_finish_sharded(navgpu_dwa* h, const double pose[3], const double* costs, const int64_t* indices,
                              int n_ranks, navgpu_dwa_result* result, double* best_points, int points_capacity) {
  if (!h || !pose || !costs || !indices || n_ranks <= 0) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (!h->have_last) return fail(NAVGPU_ERR_INVALID, "navgpu_dwa_score_range must run first");
  NAVGPU_TRY(use_device(h));
  // every rank applies the same rule: smallest cost, lowest sample index on ties == "first strictly smaller"
  // (simple_scored_sampling_planner.cpp:111-116)
  double bc = std::numeric_limits<double>::infinity();
  long long bi = -1;
  for (int r = 0; r < n_ranks; ++r)
    if (indices[r] >= 0 && (bi < 0 || costs[r] < bc || (costs[r] == bc && indices[r] < bi))) {
      bc = costs[r];
      bi = indices[r];
    }
  Cycle cy = h->last;
  if (bi < 0) {  // nothing valid anywhere: result_traj_.cost_ = -7, flags untouched
    // the generated-samples counter is normally read and cleared by the finishing kernel, which does not run here
    NAVGPU_CUDA(cudaMemsetAsync(h->d_counters, 0, 2 * sizeof(unsigned int), h->stream));
    if (result) {
      result->cost = -7.0;
      result->xv = h->res_v[0]; result->yv = h->res_v[1]; result->thetav = h->res_v[2];
      result->best_index = -1;
      result->n_samples = (int32_t)cy.n_samples;
      result->n_scored = 0;
      result->n_points = (int32_t)(h->res_points.size() / 3);
    }
    return NAVGPU_OK;
  }
  k_dwa_finish<<<1, 32, 0, h->stream>>>(cy.args, bi, bc, h->h_result, h->h_points, kPointsCapacity);
  NAVGPU_LAUNCHED(1);
  return collect(h, cy, pose, result, best_points, points_capacity);
}

int navgpu_dwa_score_strided(navgpu_dwa* h, const double pose[3], const double vel[3], const double* footprint_xy,
                             int n_footprint, int rank, int world, double* best_cost, int64_t* best_index,
                             int64_t* n_samples_total) {
  if (!h || !pose || !vel || !best_cost || !best_index || world < 1 || rank < 0 || rank >= world)
    return fail(NAVGPU_ERR_INVALID, "bad arguments");
  Cycle cy;
  NAVGPU_TRY(begin_cycle(h, pose, vel, footprint_xy, n_footprint, cy));
  if (n_samples_total) *n_samples_total = cy.n_samples;
  cy.args.stride_rank = rank;
  cy.args.stride_world = world;
  NAVGPU_TRY(launch_score(h, cy, false));
  NAVGPU_CUDA(cudaGetLastError());
  h->last = cy;
  h->have_last = true;
  NAVGPU_CUDA(cudaMemcpyAsync(&h->h_best[0], h->d_best_cost, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  NAVGPU_CUDA(cudaMemcpyAsync(&h->h_best[1], h->d_best_index, sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  *best_cost = h->h_best[0];
  long long idx;
  memcpy(&idx, &h->h_best[1], sizeof(idx));
  *best_index = idx;
  return NAVGPU_OK;
}

// ---- sharded sweep with the device-side exchange ------------------------------------------------------------------
static int shard_alloc(navgpu_dwa* h) {
  if (h->d_shard) return NAVGPU_OK;
  NAVGPU_TRY(use_device(h));
  NAVGPU_CUDA(cudaMalloc(&h->d_shard, sizeof(ShardExchange)));
  NAVGPU_CUDA(cudaMemset(h->d_shard, 0, sizeof(ShardExchange)));  // seq 0 = "no sweep yet"
  return NAVGPU_OK;
}

static void shard_disconnect(navgpu_dwa* h) {
  for (int r = 0; r < kShardMaxWorld; ++r) {
    if (h->shard_ipc[r] && h->shard_peer[r]) cudaIpcCloseMemHandle(h->shard_peer[r]);
    h->shard_peer[r] = nullptr;
    h->shard_ipc[r] = false;
  }
  h->shard_world = 0;
}

int navgpu_dwa_shard_export(navgpu_dwa* h, void* ipc_handle_out) {
  if (!h || !ipc_handle_out) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  static_assert(sizeof(cudaIpcMemHandle_t) == NAVGPU_IPC_HANDLE_BYTES, "IPC handle size");
  NAVGPU_TRY(shard_alloc(h));
  cudaIpcMemHandle_t mh;
  NAVGPU_CUDA(cudaIpcGetMemHandle(&mh, h->d_shard));
  memcpy(ipc_handle_out, &mh, sizeof(mh));
  return NAVGPU_OK;
}

int navgpu_dwa_shard_connect(navgpu_dwa* h, int rank, int world, const void* ipc_handles) {
  if (!h || !ipc_handles || world < 1 || world > kShardMaxWorld || rank < 0 || rank >= world)
    return fail(NAVGPU_ERR_INVALID, "bad arguments (world <= %d)", kShardMaxWorld);
  NAVGPU_TRY(shard_alloc(h));
  shard_disconnect(h);
  const char* base = static_cast<const char*>(ipc_handles);
  for (int r = 0; r < world; ++r) {
    if (r == rank) {
      h->shard_peer[r] = h->d_shard;
      continue;
    }
    cudaIpcMemHandle_t mh;
    memcpy(&mh, base + size_t(r) * NAVGPU_IPC_HANDLE_BYTES, sizeof(mh));
    void* p = nullptr;
    NAVGPU_CUDA(cudaIpcOpenMemHandle(&p, mh, cudaIpcMemLazyEnablePeerAccess));
    h->shard_peer[r] = static_cast<ShardExchange*>(p);
    h->shard_ipc[r] = true;
  }
  h->shard_rank = rank;
  h->shard_world = world;
  h->shard_seq = 0;
  return NAVGPU_OK;
}

int navgpu_dwa_shard_connect_local(navgpu_dwa* const* handles, int world) {
  if (!handles || world < 1 || world > kShardMaxWorld) return fail(NAVGPU_ERR_INVALID, "bad arguments (world <= %d)", kShardMaxWorld);
  for (int r = 0; r < world; ++r) {
    if (!handles[r]) return fail(NAVGPU_ERR_INVALID, "null handle");
    NAVGPU_TRY(shard_alloc(handles[r]));
  }
  for (int r = 0; r < world; ++r) {
    navgpu_dwa* h = handles[r];
    NAVGPU_TRY(use_device(h));
    shard_disconnect(h);
    for (int q = 0; q < world; ++q) {
      if (handles[q]->device != h->device) {
        int can = 0;
        NAVGPU_CUDA(cudaDeviceCanAccessPeer(&can, h->device, handles[q]->device));
        if (!can) return fail(NAVGPU_ERR_UNSUPPORTED, "device %d cannot access device %d", h->device, handles[q]->device);
        cudaError_t e = cudaDeviceEnablePeerAccess(handles[q]->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) NAVGPU_CUDA(e);
        (void)cudaGetLastError();
      }
      h->shard_peer[q] = handles[q]->d_shard;
    }
    h->shard_rank = r;
    h->shard_world = world;
    h->shard_seq = 0;
  }
  return NAVGPU_OK;
}

int navgpu_dwa_find_best_path_sharded_async(navgpu_dwa* h, const double pose[3], const double vel[3],
                                            const double* footprint_xy, int n_footprint) {
  if (!h || !pose || !vel || (n_footprint > 0 && !footprint_xy)) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (h->shard_world < 1) return fail(NAVGPU_ERR_INVALID, "navgpu_dwa_shard_connect must run first");
  Cycle cy;
  NAVGPU_TRY(begin_cycle(h, pose, vel, footprint_xy, n_footprint, cy));
  cy.args.stride_rank = h->shard_rank;
  cy.args.stride_world = h->shard_world;
  for (int r = 0; r < h->shard_world; ++r) cy.args.shard_peer[r] = h->shard_peer[r];
  cy.args.shard_seq = ++h->shard_seq;
  NAVGPU_TRY(launch_score(h, cy, true));
  NAVGPU_CUDA(cudaGetLastError());
  h->shard_cycle = cy;
  h->shard_pending = true;
  return NAVGPU_OK;
}

int navgpu_dwa_sharded_collect(navgpu_dwa* h, const double pose[3], navgpu_dwa_result* result, double* best_points,
                               int points_capacity) {
  if (!h || !pose) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (!h->shard_pending) return fail(NAVGPU_ERR_INVALID, "no sharded sweep in flight");
  NAVGPU_TRY(use_device(h));
  h->shard_pending = false;
  return collect(h, h->shard_cycle, pose, result, best_points, points_capacity);
}

int navgpu_dwa_find_best_path_sharded(navgpu_dwa* h, const double pose[3], const double vel[3], const double* footprint_xy,
                                      int n_footprint, navgpu_dwa_result* result, double* best_points, int points_capacity) {
  NAVGPU_TRY(navgpu_dwa_find_best_path_sharded_async(h, pose, vel, footprint_xy, n_footprint));
  return navgpu_dwa_sharded_collect(h, pose, result, best_points, points_capacity);
}

int navgpu_dwa_get_grid(navgpu_dwa* h, int which, double* host_out) {
  if (!h || which < 0 || which > 3 || !host_out) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  NAVGPU_TRY(use_device(h));
  const size_t n = size_t(h->sx) * h->sy;
  std::vector<uint32_t> tmp(n);
  const uint32_t* src = (which == 3 && h->align_aliased) ? h->d_dist[0] : h->d_dist[which];
  NAVGPU_CUDA(cudaMemcpyAsync(tmp.data(), src, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  for (size_t i = 0; i < n; ++i) host_out[i] = (double)tmp[i];
  return NAVGPU_OK;
}

int navgpu_dwa_synchronize(navgpu_dwa* h) {
  if (!h) return fail(NAVGPU_ERR_INVALID, "null handle");
  NAVGPU_TRY(use_device(h));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  return NAVGPU_OK;
}

void* navgpu_dwa_stream(navgpu_dwa* h) { return h ? (void*)h->stream : nullptr; }

}  // extern "C"

// ==================================================================================================================
// Fleet mode (config C5): N independent robots per control cycle -- inflation of every robot's local costmap, four
// MapGrid wavefronts per robot, rollout scoring of every robot's velocity samples -- as a handful of launches.
// The N local maps are stacked along y in ONE device-resident layered costmap (static-style layer + inflation
// layer) with kFleetPadRows rows of free space between robots so inflation cannot leak from one robot into the next;
// the planner side reuses the single-planner kernels with per-robot arguments (FleetRobot).
// ==================================================================================================================
namespace {
constexpr unsigned kFleetPadRows = 64;  // >= 2 * the largest cell inflation radius the fast sweep supports (31)
}

// the planner side of fleets of legacy TrajectoryPlanners (navgpu_fleet_use_trajectory_planner, tp_host.inc)
struct FleetTp;
static void fleet_tp_free(FleetTp* t);
static int fleet_tp_set_plans(navgpu_fleet* f, const double* plan_xy, const int32_t* plan_offsets);
static int fleet_tp_check(navgpu_fleet* f, const double* poses, const double* vels, const int32_t* offsets,
                          const double* vel_samples, double* costs_out);

struct navgpu_fleet {
  int device = 0;
  int n = 0;
  unsigned sx = 0, sy = 0, stride = 0;  // rows per robot in the stacked grid
  double res = 0;
  navgpu_dwa_config cfg;
  navgpu_costmap* costmap = nullptr;  // raw-map fleets: the stacked costmap
  FleetCostmap* sensing = nullptr;    // sensing fleets (navgpu_fleet_create_sensing): the robots' rolling costmaps
  int static_layer = -1;
  cudaStream_t stream = nullptr;  // the costmap's stream
  uint8_t* d_raw = nullptr;       // n x sy x sx: the raw maps as they arrive from the host
  uint8_t* d_stage = nullptr;     // n x stride x pitch staging of the raw maps (pad rows stay zero)
  unsigned pitch = 0;
  const uint8_t* d_master = nullptr;
  std::vector<double> origins;  // n x 2
  std::vector<DwaPlans> plans;   // per robot
  std::vector<float> h_samples;  // per-step staging of every robot's velocity samples
  bool grids_dirty = true;       // geometry / plans changed: the robots' MapGrid jobs must reach the device before the wavefronts
  std::vector<double> footprint;
  DwaScales scales = {};
  // device side
  FleetRobot* d_robots = nullptr;
  double* d_plans = nullptr;
  size_t plans_capacity = 0;
  float* d_samples = nullptr;
  size_t samples_capacity = 0;
  uint32_t* d_dist = nullptr;  // n x 4 x sx*sy
  double* d_block_cost = nullptr;
  long long* d_block_index = nullptr;
  size_t blocks_capacity = 0;
  unsigned* d_generated = nullptr;
  DwaDeviceResult* d_results = nullptr;
  DwaDeviceResult* h_results = nullptr;  // pinned
  bool plans_dirty = true;
  std::vector<FleetRobot> h_robots;
  std::vector<size_t> plan_off;  // per robot x 3 plans: offset (in points) into d_plans
  bool started = false;          // set_plans or a step has run
  FleetTp* tp = nullptr;         // non-null: the robots run base_local_planner::TrajectoryPlanner instead of DWAPlanner
  // per robot: 1 = planned by the steps (navgpu_fleet_set_active)
  std::vector<uint8_t> active;
  // per robot: oscillation flags, result velocities, planned / aliased, a sensing fleet's origin (FleetDwaState).  The
  // host copy (pinned) is current unless state_on_device: a device step ran since the host last brought it back
  // (fleet_state_to_host); the next device step uploads it when the host copy is the current one
  FleetDwaState* h_state = nullptr;
  FleetDwaState* d_state = nullptr;
  bool state_on_device = false;
  // device steps (navgpu_fleet_step_device), sized at the first one: every robot's samples at a fixed slot, its flags
  // (kFleetActive, kFleetAligned), and a pinned staging of the MapGrid records and flags, uploaded after
  // set_plans / set_active / set_maps (records_dirty)
  float* d_slot_samples = nullptr;
  uint8_t* d_flags = nullptr;
  char* h_records_stage = nullptr;
  cudaEvent_t ev_records_stage = nullptr;
  bool records_dirty = true;
  // navgpu_fleet_check_trajectories (DWAPlanner): per robot a one-sample record, per candidate its robot, velocity, cost
  std::vector<FleetRobot> h_check;
  char* d_check = nullptr;
  size_t check_capacity = 0;
};

// what every fleet holds for its planner side: the DWAPlanner parameters and critic scales ...
static void init_planner_scalars(navgpu_fleet* f, int n_robots, const navgpu_dwa_config* cfg, uint32_t size_x,
                                 uint32_t size_y, double resolution, const double* footprint_xy, int n_footprint,
                                 int device) {
  f->device = device;
  f->n = n_robots;
  f->sx = size_x; f->sy = size_y;
  f->res = resolution;
  f->cfg = *cfg;
  f->footprint.assign(footprint_xy, footprint_xy + 2 * n_footprint);
  f->scales = dwa_scales(*cfg, resolution);
}

// ... and its per-robot buffers (device and host)
static int alloc_planner_side(navgpu_fleet* f) {
  const int n_robots = f->n;
  NAVGPU_CUDA(cudaSetDevice(f->device));
  NAVGPU_CUDA(cudaMalloc(&f->d_robots, sizeof(FleetRobot) * n_robots));
  NAVGPU_CUDA(cudaMalloc(&f->d_dist, size_t(n_robots) * 4 * f->sx * f->sy * sizeof(uint32_t)));
  NAVGPU_CUDA(cudaMalloc(&f->d_generated, sizeof(unsigned) * n_robots));
  NAVGPU_CUDA(cudaMemset(f->d_generated, 0, sizeof(unsigned) * n_robots));
  NAVGPU_CUDA(cudaMalloc(&f->d_results, sizeof(DwaDeviceResult) * n_robots));
  NAVGPU_CUDA(cudaMallocHost(&f->h_results, sizeof(DwaDeviceResult) * n_robots));
  NAVGPU_CUDA(cudaMallocHost(&f->h_state, sizeof(FleetDwaState) * n_robots));
  for (int r = 0; r < n_robots; ++r) f->h_state[r] = FleetDwaState{};
  f->origins.assign(size_t(2) * n_robots, 0.0);
  f->plans.resize(n_robots);
  f->h_robots.resize(n_robots);
  f->active.assign(n_robots, 1);
  return NAVGPU_OK;
}

// the argument checks of every kind of fleet
static int check_fleet_args(navgpu_fleet** out, int n_robots, const navgpu_dwa_config* cfg, uint32_t size_x,
                            uint32_t size_y, double resolution, const double* footprint_xy, int n_footprint, int device) {
  if (!out || !cfg || n_robots <= 0 || size_x == 0 || size_y == 0 || !(resolution > 0) || n_footprint < 0 ||
      n_footprint > kMaxFootprint || (n_footprint > 0 && !footprint_xy))
    return fail(NAVGPU_ERR_INVALID, "bad fleet arguments");
  if (navgpu_device_count() <= device) return fail(NAVGPU_ERR_CUDA, "no CUDA device %d (libnavgpu has no CPU fallback)", device);
  if (size_x > 32767 || size_y > 32767) return fail(NAVGPU_ERR_UNSUPPORTED, "local costmap too large");
  return NAVGPU_OK;
}

// The start of every fleet step, before the robots' MapGrid records go up: a sensing fleet rolls every robot's origin
// (host scalars; its costmap kernel follows later, fleet_costmap_enqueue), a raw-map fleet enqueues one full-window
// update of the stacked costmap (Path A for all robots)
static int fleet_costmap_front(navgpu_fleet* f, const double* poses) {
  if (f->sensing) {
    NAVGPU_TRY(fleet_costmap_roll(f->sensing, poses, f->origins.data()));
    f->grids_dirty = true;
    return NAVGPU_OK;
  }
  NAVGPU_TRY(navgpu_grid_layer_touch(f->costmap, f->static_layer, 0, 0, f->sx, f->stride * f->n));
  return navgpu_costmap_update_map_async(f->costmap, 0.0, 0.0, 0.0);
}

// n_plans plans (plan_at(i) is plan i) concatenated into a device buffer that grows as needed, off[i] = where plan i
// starts in it, in points (pageable source: the copy completes before returning)
template <class PlanAt>
static int fleet_upload_plans(size_t n_plans, PlanAt plan_at, std::vector<size_t>& off, double** d, size_t* cap,
                              cudaStream_t stream) {
  off.assign(n_plans, 0);
  size_t total = 0;
  for (size_t i = 0; i < n_plans; ++i) { off[i] = total; total += plan_at(i).size(); }
  if (total == 0) return NAVGPU_OK;
  std::vector<P2> flat;
  flat.reserve(total);
  for (size_t i = 0; i < n_plans; ++i) flat.insert(flat.end(), plan_at(i).begin(), plan_at(i).end());
  if (total > *cap) {
    cudaFree(*d);
    *d = nullptr;
    *cap = 0;
    NAVGPU_CUDA(cudaMalloc(d, total * 2 * sizeof(P2)));
    *cap = total * 2;
  }
  NAVGPU_CUDA(cudaMemcpyAsync(*d, flat.data(), total * sizeof(P2), cudaMemcpyHostToDevice, stream));
  NAVGPU_CUDA(cudaStreamSynchronize(stream));
  return NAVGPU_OK;
}

// every robot's MapGrid record, when geometry or plans changed: its master grid and map origin, then the planner's
// jobs (set_jobs(r, job)); the records reach the device before the wavefronts
template <class SetJobs>
static int fleet_upload_grids(navgpu_fleet* f, SetJobs set_jobs) {
  if (!f->grids_dirty) return NAVGPU_OK;
  for (int r = 0; r < f->n; ++r) {
    MapGridRobot& G = f->h_robots[r].grids;
    G.g = DwaGeom{f->d_master + size_t(r) * f->stride * f->pitch, f->sx, f->sy, f->pitch, f->res, f->origins[2 * r],
                  f->origins[2 * r + 1], 1.0 / f->res};
    set_jobs(r, G.job);
  }
  NAVGPU_CUDA(cudaMemcpyAsync(f->d_robots, f->h_robots.data(), sizeof(FleetRobot) * f->n, cudaMemcpyHostToDevice, f->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(f->stream));  // pageable source, rewritten by the step
  f->grids_dirty = false;
  return NAVGPU_OK;
}

// the scoring arguments every robot of a DWAPlanner fleet shares (fleet_patch_args adds each robot's own)
static void fleet_dwa_base_args(const navgpu_fleet* f, DwaScoreArgs& base) {
  memset(&base, 0, sizeof(base));
  base.g = DwaGeom{nullptr, f->sx, f->sy, f->pitch, f->res, 0.0, 0.0, 1.0 / f->res};
  dwa_config_args(f->cfg, f->scales, f->footprint.data(), (int)(f->footprint.size() / 2), base);  // (scale_alignment: per robot)
}

// the MapGrid wavefronts of every robot, jobs_per_robot each, in one launch (each CTA reads its robot's record)
static int fleet_launch_mapgrid(navgpu_fleet* f, int allow_unknown, int jobs_per_robot) {
  MapGridArgs ma;
  memset(&ma, 0, sizeof(ma));
  ma.g = DwaGeom{nullptr, f->sx, f->sy, f->pitch, f->res, 0.0, 0.0, 1.0 / f->res};
  ma.allow_unknown = allow_unknown;
  ma.fleet = f->d_robots;
  return launch_mapgrid(f->sx, f->sy, f->stream, ma, jobs_per_robot * f->n, jobs_per_robot);
}

// Brings the host copy of the per-robot state up to date after device steps (one copy and a wait); every host call that
// reads or changes that state calls this first, so that host and device steps can be mixed on one fleet
static int fleet_state_to_host(navgpu_fleet* f) {
  if (!f->state_on_device) return NAVGPU_OK;
  NAVGPU_CUDA(cudaSetDevice(f->device));
  NAVGPU_CUDA(cudaMemcpyAsync(f->h_state, f->d_state, sizeof(FleetDwaState) * f->n, cudaMemcpyDeviceToHost, f->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(f->stream));
  f->state_on_device = false;
  if (f->sensing) {  // the device rolled the origins
    for (int r = 0; r < f->n; ++r) {
      f->origins[2 * r] = f->h_state[r].origin[0];
      f->origins[2 * r + 1] = f->h_state[r].origin[1];
    }
    fleet_costmap_set_origins(f->sensing, f->origins.data());
  }
  return NAVGPU_OK;
}

// robot r's four MapGrid jobs of a DWAPlanner fleet step (path, goal, goal_front, alignment)
static void fleet_dwa_jobs(const navgpu_fleet* f, int r, MapGridJob* job) {
  const size_t cells = size_t(f->sx) * f->sy;
  const DwaPlans& p = f->plans[r];
  const double* plan[3];
  for (int k = 0; k < 3; ++k) plan[k] = f->d_plans + 2 * f->plan_off[3 * r + k];
  uint32_t* dist = f->d_dist + size_t(r) * 4 * cells;
  job[0] = MapGridJob{plan[0], (int)p.adjusted[0].size(), 0, dist};
  job[1] = MapGridJob{plan[0], (int)p.adjusted[0].size(), 1, dist + cells};
  job[2] = MapGridJob{plan[1], (int)p.adjusted[1].size(), 1, dist + 2 * cells};
  job[3] = MapGridJob{plan[2], (int)p.adjusted[2].size(), 0, dist + 3 * cells};
  if (p.align_is_path) {  // the alignment critic holds the path critic's poses: one wavefront serves both
    job[3].dist = dist;
    job[3].skip = 1;
  }
  if (!f->active[r])  // left out of the search: its grids stay as its last planning step left them
    for (int k = 0; k < 4; ++k) job[k].skip = 1;
}

// every robot's path, front and alignment plans, robot after robot, when set_plans changed them
static int fleet_dwa_upload_plans(navgpu_fleet* f) {
  if (!f->plans_dirty) return NAVGPU_OK;
  auto plan_at = [&](size_t i) -> const std::vector<P2>& { return f->plans[i / 3].adjusted[i % 3]; };
  NAVGPU_TRY(fleet_upload_plans(size_t(3) * f->n, plan_at, f->plan_off, &f->d_plans, &f->plans_capacity, f->stream));
  f->plans_dirty = false;
  return NAVGPU_OK;
}

extern "C" {

int navgpu_fleet_create(navgpu_fleet** out, int n_robots, const navgpu_dwa_config* cfg, uint32_t size_x, uint32_t size_y,
                        double resolution, double inflation_radius, double cost_scaling_factor,
                        const double* footprint_xy, int n_footprint, int device) {
  NAVGPU_TRY(check_fleet_args(out, n_robots, cfg, size_x, size_y, resolution, footprint_xy, n_footprint, device));
  // the robots' maps are stacked with kFleetPadRows free rows between them: a larger cell inflation radius
  // (Costmap2D::cellDistance, costmap_2d.cpp:181-185) would inflate one robot's obstacles into its neighbour's map
  if (inflation_radius > 0 && std::ceil(inflation_radius / resolution) > (double)kFleetPadRows)
    return fail(NAVGPU_ERR_UNSUPPORTED, "fleet inflation radius of %.0f cells exceeds the %u rows between stacked maps",
                std::ceil(inflation_radius / resolution), kFleetPadRows);
  std::unique_ptr<navgpu_fleet> f(new navgpu_fleet);
  init_planner_scalars(f.get(), n_robots, cfg, size_x, size_y, resolution, footprint_xy, n_footprint, device);
  f->stride = size_y + kFleetPadRows;
  if ((unsigned long long)f->stride * n_robots > 0x7fffffffull) return fail(NAVGPU_ERR_UNSUPPORTED, "fleet too large");
  // the stacked costmap: every robot's window is "the whole map" each cycle, like a rolling local costmap
  NAVGPU_TRY(navgpu_costmap_create(&f->costmap, size_x, f->stride * n_robots, resolution, 0.0, 0.0, 0, 0, device));
  NAVGPU_TRY(navgpu_costmap_add_grid_layer(f->costmap, NAVGPU_TRUE_OVERWRITE, &f->static_layer));
  int il;
  NAVGPU_TRY(navgpu_costmap_add_inflation_layer(f->costmap, inflation_radius, cost_scaling_factor, &il));
  NAVGPU_TRY(navgpu_costmap_set_footprint(f->costmap, footprint_xy, n_footprint));
  f->stream = (cudaStream_t)navgpu_costmap_stream(f->costmap);
  uint32_t pitch;
  NAVGPU_TRY(navgpu_costmap_device_grid(f->costmap, &f->d_master, &pitch));
  f->pitch = pitch;
  NAVGPU_CUDA(cudaSetDevice(device));
  const size_t stage_bytes = size_t(pitch) * f->stride * n_robots;
  NAVGPU_CUDA(cudaMalloc(&f->d_stage, stage_bytes));
  NAVGPU_CUDA(cudaMemset(f->d_stage, 0, stage_bytes));
  NAVGPU_CUDA(cudaMalloc(&f->d_raw, size_t(n_robots) * size_y * size_x));
  NAVGPU_TRY(alloc_planner_side(f.get()));
  *out = f.release();
  return NAVGPU_OK;
}

// navgpu_fleet_create_sensing and navgpu_fleet_create_sensing_voxel (voxel non-null)
static int create_sensing(navgpu_fleet** out, int n_robots, const navgpu_dwa_config* cfg, uint32_t size_x,
                          uint32_t size_y, double resolution, const navgpu_fleet_costmap_config* cm,
                          const navgpu_fleet_voxel_config* voxel, const double* footprint_xy, int n_footprint,
                          int device) {
  if (!cm) return fail(NAVGPU_ERR_INVALID, "bad fleet arguments");
  NAVGPU_TRY(check_fleet_args(out, n_robots, cfg, size_x, size_y, resolution, footprint_xy, n_footprint, device));
  std::unique_ptr<navgpu_fleet> f(new navgpu_fleet);
  init_planner_scalars(f.get(), n_robots, cfg, size_x, size_y, resolution, footprint_xy, n_footprint, device);
  f->stride = size_y;  // robot r's master grid starts at row r * size_y
  int rc = fleet_costmap_create(&f->sensing, n_robots, size_x, size_y, resolution, *cm, voxel, footprint_xy, n_footprint,
                                device);
  if (rc == NAVGPU_OK) {
    f->stream = fleet_costmap_stream(f->sensing);
    f->d_master = fleet_costmap_master(f->sensing, &f->pitch);
    rc = alloc_planner_side(f.get());
  }
  if (rc != NAVGPU_OK) {  // free what was allocated (the message of the failure stays)
    navgpu_fleet_destroy(f.release());
    return rc;
  }
  *out = f.release();
  return NAVGPU_OK;
}

int navgpu_fleet_create_sensing(navgpu_fleet** out, int n_robots, const navgpu_dwa_config* cfg, uint32_t size_x,
                                uint32_t size_y, double resolution, const navgpu_fleet_costmap_config* cm,
                                const double* footprint_xy, int n_footprint, int device) {
  return create_sensing(out, n_robots, cfg, size_x, size_y, resolution, cm, nullptr, footprint_xy, n_footprint, device);
}

int navgpu_fleet_create_sensing_voxel(navgpu_fleet** out, int n_robots, const navgpu_dwa_config* cfg, uint32_t size_x,
                                      uint32_t size_y, double resolution, const navgpu_fleet_costmap_config* cm,
                                      const navgpu_fleet_voxel_config* voxel, const double* footprint_xy,
                                      int n_footprint, int device) {
  if (!voxel) return fail(NAVGPU_ERR_INVALID, "null voxel config");
  return create_sensing(out, n_robots, cfg, size_x, size_y, resolution, cm, voxel, footprint_xy, n_footprint, device);
}


int navgpu_fleet_destroy(navgpu_fleet* f) {
  if (!f) return NAVGPU_OK;
  cudaSetDevice(f->device);
  if (f->stream) cudaStreamSynchronize(f->stream);
  cudaFree(f->d_stage); cudaFree(f->d_raw); cudaFree(f->d_robots); cudaFree(f->d_plans); cudaFree(f->d_samples); cudaFree(f->d_dist);
  cudaFree(f->d_block_cost); cudaFree(f->d_block_index); cudaFree(f->d_generated); cudaFree(f->d_results);
  cudaFree(f->d_check);
  cudaFreeHost(f->h_results);
  cudaFree(f->d_state); cudaFree(f->d_slot_samples); cudaFree(f->d_flags);
  if (f->h_state) cudaFreeHost(f->h_state);
  if (f->h_records_stage) cudaFreeHost(f->h_records_stage);
  if (f->ev_records_stage) cudaEventDestroy(f->ev_records_stage);
  fleet_tp_free(f->tp);
  navgpu_costmap_destroy(f->costmap);
  fleet_costmap_destroy(f->sensing);  // (owns the stream of a sensing fleet)
  delete f;
  return NAVGPU_OK;
}

// raw (un-inflated) local maps of all robots, [n][size_y][size_x] in HOST memory, and their world origins [n][2]
int navgpu_fleet_set_maps(navgpu_fleet* f, const uint8_t* raw_maps, const double* origins_xy) {
  if (!f || !raw_maps || !origins_xy) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (f->sensing) return fail(NAVGPU_ERR_INVALID, "a sensing fleet builds its maps from scans (navgpu_fleet_set_scans)");
  NAVGPU_CUDA(cudaSetDevice(f->device));
  f->origins.assign(origins_xy, origins_xy + size_t(2) * f->n);
  f->grids_dirty = true;  // the robots' map origins changed
  f->records_dirty = true;
  // one contiguous H2D copy, then a device-side scatter into the padded stack
  const size_t raw_bytes = size_t(f->n) * f->sy * f->sx;
  NAVGPU_CUDA(cudaMemcpyAsync(f->d_raw, raw_maps, raw_bytes, cudaMemcpyHostToDevice, f->stream));
  {
    dim3 block(32, 8);
    const size_t rows = size_t(f->n) * f->sy;
    k_fleet_scatter_maps<<<(unsigned)((rows + 7) / 8), block, 0, f->stream>>>(f->d_raw, f->d_stage, f->sx, f->sy, f->stride,
                                                                             f->pitch, (unsigned)f->n);
    NAVGPU_LAUNCHED(1);
  }
  NAVGPU_TRY(navgpu_grid_layer_set_device(f->costmap, f->static_layer, f->d_stage, f->pitch));
  NAVGPU_CUDA(cudaStreamSynchronize(f->stream));  // raw_maps may be pageable
  return NAVGPU_OK;
}

// DWAPlanner::updatePlanAndLocalCosts for every robot: plan_xy = concatenated (x, y) points, plan_offsets[n + 1] in
// points, poses [n][3]
int navgpu_fleet_set_plans(navgpu_fleet* f, const double* poses, const double* plan_xy, const int32_t* plan_offsets) {
  if (!f || !poses || !plan_xy || !plan_offsets) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  f->started = true;
  if (f->tp) return fleet_tp_set_plans(f, plan_xy, plan_offsets);
  for (int r = 0; r < f->n; ++r) {
    const int b = plan_offsets[r], e = plan_offsets[r + 1];
    if (e <= b) return fail(NAVGPU_ERR_INVALID, "robot %d has an empty plan", r);
    DwaPlans& p = f->plans[r];
    update_plan_and_local_costs(p, f->cfg, f->res, poses + 3 * r, plan_xy + 2 * b, e - b);
    if (p.adjusted[2].empty()) {  // never set before: scale 0 or the path itself, whose grid it then shares
      p.adjusted[2] = p.adjusted[0];
      p.align_is_path = true;
    }
  }
  f->plans_dirty = true;
  f->grids_dirty = true;
  f->records_dirty = true;
  return NAVGPU_OK;
}

int navgpu_fleet_reset_oscillation(navgpu_fleet* f) {
  if (!f) return fail(NAVGPU_ERR_INVALID, "null handle");
  if (f->tp) return fail(NAVGPU_ERR_INVALID, "a TrajectoryPlanner fleet has no DWA oscillation flags (see navgpu_fleet_step_tp's flags)");
  NAVGPU_TRY(fleet_state_to_host(f));
  for (int r = 0; r < f->n; ++r) f->h_state[r].osc.reset();
  return NAVGPU_OK;
}

// One control cycle of the whole fleet: inflate every local map, then DWAPlanner::findBestPath for every robot.
// poses, vels: [n][3]; results: n entries (n_points is always 0: the winners' points are not materialised).
int navgpu_fleet_step(navgpu_fleet* f, const double* poses, const double* vels, navgpu_dwa_result* results) {
  if (!f || !poses || !vels || !results) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (f->tp) return fail(NAVGPU_ERR_INVALID, "a TrajectoryPlanner fleet steps with navgpu_fleet_step_tp");
  f->started = true;
  NAVGPU_TRY(fleet_state_to_host(f));
  NAVGPU_CUDA(cudaSetDevice(f->device));
  const navgpu_dwa_config& c = f->cfg;
  const int n = f->n;
  NAVGPU_TRY(fleet_costmap_front(f, poses));
  NAVGPU_TRY(fleet_dwa_upload_plans(f));

  // ---- the MapGrid wavefronts only need each robot's geometry and plans, which change with set_maps / set_plans, not
  // per step: they are launched first, and the per-step host work below (sample enumeration for every robot) runs
  // while the GPU is busy with the costmap update and the wavefronts
  NAVGPU_TRY(fleet_upload_grids(f, [f](int r, MapGridJob* job) { fleet_dwa_jobs(f, r, job); }));
  // sensing fleet: LayeredCostmap::updateMap of every robot, before the wavefronts read the master grids
  if (f->sensing) NAVGPU_TRY(fleet_costmap_enqueue(f->sensing));
  NAVGPU_TRY(fleet_launch_mapgrid(f, c.allow_unknown, 4));

  // ---- per-robot scalars: samples (SimpleTrajectoryGenerator::initialise), pose, velocity, oscillation mask
  std::vector<float>& samples = f->h_samples;
  samples.clear();
  int max_samples = 0;
  for (int r = 0; r < n; ++r) {
    FleetRobot& R = f->h_robots[r];
    if (!f->active[r]) {  // no samples: its scoring CTAs exit at once
      R.nx = R.ny = R.nth = 0;
      R.samples_offset = (int)samples.size();
      continue;
    }
    const float pos[3] = {(float)poses[3 * r], (float)poses[3 * r + 1], (float)poses[3 * r + 2]};
    const float vel[3] = {(float)vels[3 * r], (float)vels[3 * r + 1], (float)vels[3 * r + 2]};
    const float goal[2] = {(float)f->plans[r].plan.back().x, (float)f->plans[r].plan.back().y};
    const Samples s = enumerate_samples(c, pos, vel, goal);
    if (s.v.size() > (size_t)kInlineSamples) {
      cudaStreamSynchronize(f->stream);
      return fail(NAVGPU_ERR_UNSUPPORTED, "more than %d per-axis samples per robot", kInlineSamples);
    }
    for (int k = 0; k < 3; ++k) { R.pos[k] = pos[k]; R.vel[k] = vel[k]; }
    R.osc_mask = f->h_state[r].osc.mask();
    R.scale_alignment = f->plans[r].alignment_scale;
    R.nx = s.nx; R.ny = s.ny; R.nth = s.nth;
    R.samples_offset = (int)samples.size();
    samples.insert(samples.end(), s.v.begin(), s.v.end());
    max_samples = std::max(max_samples, s.nx * s.ny * s.nth);
  }
  if (samples.size() > f->samples_capacity) {
    if (f->d_samples) cudaFree(f->d_samples);
    f->d_samples = nullptr;
    NAVGPU_CUDA(cudaMalloc(&f->d_samples, samples.size() * 2 * sizeof(float)));
    f->samples_capacity = samples.size() * 2;
  }
  if (!samples.empty())
    NAVGPU_CUDA(cudaMemcpyAsync(f->d_samples, samples.data(), samples.size() * sizeof(float), cudaMemcpyHostToDevice, f->stream));
  NAVGPU_CUDA(cudaMemcpyAsync(f->d_robots, f->h_robots.data(), sizeof(FleetRobot) * n, cudaMemcpyHostToDevice, f->stream));
  const int bpr = (max_samples + kDwaWarpsPerBlock - 1) / kDwaWarpsPerBlock;  // (0: no robot is active)
  const size_t blocks = size_t(bpr) * n;
  if (blocks > f->blocks_capacity) {
    if (f->d_block_cost) cudaFree(f->d_block_cost);
    if (f->d_block_index) cudaFree(f->d_block_index);
    f->d_block_cost = nullptr; f->d_block_index = nullptr;
    NAVGPU_CUDA(cudaMalloc(&f->d_block_cost, blocks * sizeof(double)));
    NAVGPU_CUDA(cudaMalloc(&f->d_block_index, blocks * sizeof(long long)));
    f->blocks_capacity = blocks;
  }
  if (blocks > 0x7fffffffull) return fail(NAVGPU_ERR_UNSUPPORTED, "too many samples in one fleet launch");

  // ---- rollouts + critics + per-robot argmin
  DwaScoreArgs base;
  fleet_dwa_base_args(f, base);
  if (bpr > 0) {
    k_fleet_score<<<(unsigned)blocks, kDwaWarpsPerBlock * 32, 0, f->stream>>>(base, f->d_robots, f->d_samples, bpr,
                                                                            f->d_block_cost, f->d_block_index, f->d_generated);
    k_fleet_finish<<<n, 32, 0, f->stream>>>(base, f->d_robots, f->d_samples, bpr, f->d_block_cost, f->d_block_index,
                                            f->d_generated, f->d_results);
    NAVGPU_LAUNCHED(2);
    NAVGPU_CUDA(cudaGetLastError());
    NAVGPU_CUDA(cudaMemcpyAsync(f->h_results, f->d_results, sizeof(DwaDeviceResult) * n, cudaMemcpyDeviceToHost, f->stream));
  }
  NAVGPU_CUDA(cudaStreamSynchronize(f->stream));

  // ---- host epilogue per active robot: result_traj_ bookkeeping + oscillation flags
  for (int r = 0; r < n; ++r) {
    if (!f->active[r]) continue;
    const FleetRobot& R = f->h_robots[r];
    FleetDwaState& S = f->h_state[r];
    apply_dwa_result(f->h_results[r], c, poses + 3 * r, R.nx * R.ny * R.nth, S.res_v, S.osc, &results[r]);
    results[r].n_points = 0;
    S.planned = 1;
    S.aliased = f->plans[r].align_is_path;
  }
  return NAVGPU_OK;
}

// navgpu_fleet_step with device memory: the same work as launches on the fleet's stream, no host wait (see navgpu.h)
int navgpu_fleet_step_device(navgpu_fleet* f, const double* poses, const double* vels, navgpu_dwa_result* results) {
  // every check before anything changes: a refused call leaves the fleet as it was
  if (!f || !poses || !vels || !results) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (f->tp) return fail(NAVGPU_ERR_UNSUPPORTED, "a TrajectoryPlanner fleet steps on the host (navgpu_fleet_step_tp)");
  const navgpu_dwa_config& c = f->cfg;
  if (!c.use_dwa) return fail(NAVGPU_ERR_UNSUPPORTED, "use_dwa = 0: its velocity window takes glibc's hypot, which the device does not reproduce");
  if (!on_device(poses, f->device) || !on_device(vels, f->device) || !on_device(results, f->device))
    return fail(NAVGPU_ERR_INVALID, "poses, vels and results must be device memory of device %d", f->device);
  // the scoring grid comes from the configuration, not from the robots' sample counts (those exist on the device only)
  int axes[3];
  dwa_axis_samples(c, axes);
  const long long bx = dwa_axis_bound(axes[0]), by = dwa_axis_bound(axes[1]), bth = dwa_axis_bound(axes[2]);
  const long long slot = bx + by + bth, bpr = (bx * by * bth + kDwaWarpsPerBlock - 1) / kDwaWarpsPerBlock;
  const int n = f->n;
  if (slot > kInlineSamples)
    return fail(NAVGPU_ERR_UNSUPPORTED, "up to %lld per-axis samples per robot; a device step holds %d", slot, kInlineSamples);
  if (slot * n > 0x7fffffffLL || bpr * n > 0x7fffffffLL) return fail(NAVGPU_ERR_UNSUPPORTED, "too many samples in one fleet launch");
  if (f->records_dirty)
    for (int r = 0; r < n; ++r)
      if (f->plans[r].plan.empty()) return fail(NAVGPU_ERR_INVALID, "robot %d has no plan (navgpu_fleet_set_plans)", r);
  NAVGPU_CUDA(cudaSetDevice(f->device));

  // buffers of device steps: sized at the first one, so later ones do not allocate
  if (!f->d_state) {
    NAVGPU_CUDA(cudaMalloc(&f->d_state, sizeof(FleetDwaState) * n));
    NAVGPU_CUDA(cudaMalloc(&f->d_slot_samples, sizeof(float) * slot * n));
    NAVGPU_CUDA(cudaMalloc(&f->d_flags, n));
    NAVGPU_CUDA(cudaMallocHost(&f->h_records_stage, (sizeof(FleetRobot) + 1) * n));
    NAVGPU_CUDA(cudaEventCreateWithFlags(&f->ev_records_stage, cudaEventDisableTiming));
  }
  const size_t blocks = size_t(bpr) * n;
  if (blocks > f->blocks_capacity) {
    cudaFree(f->d_block_cost);
    cudaFree(f->d_block_index);
    f->d_block_cost = nullptr; f->d_block_index = nullptr; f->blocks_capacity = 0;
    NAVGPU_CUDA(cudaMalloc(&f->d_block_cost, blocks * sizeof(double)));
    NAVGPU_CUDA(cudaMalloc(&f->d_block_index, blocks * sizeof(long long)));
    f->blocks_capacity = blocks;
  }
  f->started = true;
  if (!f->sensing) {  // Path A for all robots (a sensing fleet's update follows the roll in k_fleet_prepare)
    NAVGPU_TRY(navgpu_grid_layer_touch(f->costmap, f->static_layer, 0, 0, f->sx, f->stride * f->n));
    NAVGPU_TRY(navgpu_costmap_update_map_async(f->costmap, 0.0, 0.0, 0.0));
  }
  NAVGPU_TRY(fleet_dwa_upload_plans(f));
  if (!f->state_on_device) {  // host calls changed the state since the last device step (the host copy is pinned)
    if (f->sensing)
      for (int r = 0; r < n; ++r) {
        f->h_state[r].origin[0] = f->origins[2 * r];
        f->h_state[r].origin[1] = f->origins[2 * r + 1];
      }
    NAVGPU_CUDA(cudaMemcpyAsync(f->d_state, f->h_state, sizeof(FleetDwaState) * n, cudaMemcpyHostToDevice, f->stream));
    f->state_on_device = true;
  }
  if (f->records_dirty || f->grids_dirty) {  // set_plans, set_active or set_maps ran: the MapGrid records and flags
    FleetRobot* stage = reinterpret_cast<FleetRobot*>(f->h_records_stage);
    uint8_t* flags = reinterpret_cast<uint8_t*>(stage + n);
    NAVGPU_CUDA(cudaEventSynchronize(f->ev_records_stage));  // the previous upload from the staging has been read
    for (int r = 0; r < n; ++r) {
      FleetRobot& R = f->h_robots[r];
      R.grids.g = DwaGeom{f->d_master + size_t(r) * f->stride * f->pitch, f->sx, f->sy, f->pitch, f->res, f->origins[2 * r],
                          f->origins[2 * r + 1], 1.0 / f->res};
      fleet_dwa_jobs(f, r, R.grids.job);
      R.scale_alignment = f->plans[r].alignment_scale;
      stage[r] = R;
      flags[r] = (f->active[r] ? kFleetActive : 0) | (f->plans[r].align_is_path ? kFleetAligned : 0);
    }
    NAVGPU_CUDA(cudaMemcpyAsync(f->d_robots, stage, sizeof(FleetRobot) * n, cudaMemcpyHostToDevice, f->stream));
    NAVGPU_CUDA(cudaMemcpyAsync(f->d_flags, flags, n, cudaMemcpyHostToDevice, f->stream));
    NAVGPU_CUDA(cudaEventRecord(f->ev_records_stage, f->stream));
    f->records_dirty = f->grids_dirty = false;
  }

  const unsigned robot_ctas = (unsigned)((n + kFleetRobotThreads - 1) / kFleetRobotThreads);
  FleetPrepareArgs pa;
  pa.poses = poses; pa.vels = vels;
  pa.robots = f->d_robots; pa.state = f->d_state; pa.flags = f->d_flags;
  pa.samples = f->d_slot_samples; pa.slot = (int)slot; pa.n = n;
  pa.cfg = c;
  pa.steps = f->sensing ? fleet_costmap_device_steps(f->sensing) : nullptr;
  pa.sx = f->sx; pa.sy = f->sy; pa.res = f->res;
  k_fleet_prepare<<<robot_ctas, kFleetRobotThreads, 0, f->stream>>>(pa);
  NAVGPU_LAUNCHED(1);
  if (f->sensing) NAVGPU_TRY(fleet_costmap_enqueue(f->sensing, true));
  NAVGPU_TRY(fleet_launch_mapgrid(f, c.allow_unknown, 4));
  DwaScoreArgs base;
  fleet_dwa_base_args(f, base);
  k_fleet_score<<<(unsigned)blocks, kDwaWarpsPerBlock * 32, 0, f->stream>>>(base, f->d_robots, f->d_slot_samples, (int)bpr,
                                                                          f->d_block_cost, f->d_block_index, f->d_generated);
  k_fleet_finish<<<n, 32, 0, f->stream>>>(base, f->d_robots, f->d_slot_samples, (int)bpr, f->d_block_cost,
                                          f->d_block_index, f->d_generated, f->d_results);
  k_fleet_apply<<<robot_ctas, kFleetRobotThreads, 0, f->stream>>>(c, poses, f->d_robots, f->d_flags, f->d_results,
                                                                  f->d_state, results, n);
  NAVGPU_LAUNCHED(3);
  NAVGPU_CUDA(cudaGetLastError());
  return NAVGPU_OK;
}

// inflated local costmap of one robot (HOST, size_y x size_x), for parity checks
int navgpu_fleet_get_costmap(navgpu_fleet* f, int robot, uint8_t* host_out) {
  if (!f || robot < 0 || robot >= f->n || !host_out) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (f->sensing) return fleet_costmap_get(f->sensing, robot, true, host_out);
  return navgpu_costmap_get_window(f->costmap, 0, (int)(robot * f->stride), (int)f->sx, (int)(robot * f->stride + f->sy), host_out);
}

int navgpu_fleet_get_oscillation_mask(navgpu_fleet* f, int robot, int* mask_out) {
  if (!f || robot < 0 || robot >= f->n || !mask_out) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (f->tp) return fail(NAVGPU_ERR_INVALID, "a TrajectoryPlanner fleet has no DWA oscillation flags (see navgpu_fleet_step_tp's flags)");
  NAVGPU_TRY(fleet_state_to_host(f));
  *mask_out = f->h_state[robot].osc.mask();
  return NAVGPU_OK;
}

int navgpu_fleet_set_active(navgpu_fleet* f, const uint8_t* active) {
  if (!f) return fail(NAVGPU_ERR_INVALID, "null handle");
  if (active)
    for (int r = 0; r < f->n; ++r)
      if (active[r] > 1) return fail(NAVGPU_ERR_INVALID, "active[%d] is %d, not 0 or 1", r, (int)active[r]);
  for (int r = 0; r < f->n; ++r) {
    const uint8_t a = active ? active[r] : 1;
    if (a != f->active[r]) f->grids_dirty = f->records_dirty = true;  // the robot's MapGrid jobs change (skip)
    f->active[r] = a;
  }
  return NAVGPU_OK;
}

// DWAPlanner::checkTrajectory (dwa_planner.cpp:213-237) of every candidate, as navgpu_dwa_check_trajectory computes it
// on a handle holding the robot's current costmap and plans and the distance grids of its last planning step
int navgpu_fleet_check_trajectories(navgpu_fleet* f, const double* poses, const double* vels, const int32_t* offsets,
                                    const double* vel_samples, double* costs_out) {
  if (!f || !poses || !vels || !offsets || !vel_samples || !costs_out) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (offsets[0] != 0) return fail(NAVGPU_ERR_INVALID, "candidate offsets must start at 0");
  for (int r = 0; r < f->n; ++r)
    if (offsets[r + 1] < offsets[r]) return fail(NAVGPU_ERR_INVALID, "candidate offsets decrease at robot %d", r);
  NAVGPU_TRY(fleet_state_to_host(f));
  for (int r = 0; r < f->n; ++r)
    if (offsets[r + 1] > offsets[r] && !f->h_state[r].planned)
      return fail(NAVGPU_ERR_INVALID, "robot %d has candidates but was never active in a step", r);
  NAVGPU_CUDA(cudaSetDevice(f->device));
  if (f->tp) return fleet_tp_check(f, poses, vels, offsets, vel_samples, costs_out);
  const int n = f->n, total = offsets[n];
  if (total == 0) return NAVGPU_OK;
  const size_t cells = size_t(f->sx) * f->sy;
  // device copies: [one record per robot | robot of each candidate | candidates (float) | costs]
  auto up16 = [](size_t b) { return (b + 15) & ~size_t(15); };
  const size_t b_rob = up16(sizeof(FleetRobot) * n), b_of = up16(sizeof(int32_t) * total),
               b_vel = up16(sizeof(float) * 3 * total), b_cost = sizeof(double) * total;
  const size_t need = b_rob + b_of + b_vel + b_cost;
  if (need > f->check_capacity) {
    cudaFree(f->d_check);
    f->d_check = nullptr;
    f->check_capacity = 0;
    NAVGPU_CUDA(cudaMalloc(&f->d_check, 2 * need));
    f->check_capacity = 2 * need;
  }
  FleetRobot* d_rob = reinterpret_cast<FleetRobot*>(f->d_check);
  int32_t* d_of = reinterpret_cast<int32_t*>(f->d_check + b_rob);
  float* d_vel = reinterpret_cast<float*>(f->d_check + b_rob + b_of);
  double* d_cost = reinterpret_cast<double*>(f->d_check + b_rob + b_of + b_vel);
  std::vector<int32_t> robot_of(total);
  std::vector<float> vel_f(size_t(3) * total);
  f->h_check.resize(n);
  for (int r = 0; r < n; ++r) {
    const int b = offsets[r], e = offsets[r + 1];
    if (e == b) continue;
    f->h_state[r].osc.reset();  // dwa_planner.cpp:217
    FleetRobot& R = f->h_check[r];
    R.grids.g = DwaGeom{f->d_master + size_t(r) * f->stride * f->pitch, f->sx, f->sy, f->pitch, f->res, f->origins[2 * r],
                        f->origins[2 * r + 1], 1.0 / f->res};
    uint32_t* dist = f->d_dist + size_t(r) * 4 * cells;
    for (int k = 0; k < 4; ++k) R.grids.job[k].dist = dist + k * cells;
    if (f->h_state[r].aliased) R.grids.job[3].dist = dist;
    for (int k = 0; k < 3; ++k) { R.pos[k] = (float)poses[3 * r + k]; R.vel[k] = (float)vels[3 * r + k]; }
    R.osc_mask = 0;
    R.scale_alignment = f->plans[r].alignment_scale;
    R.nx = R.ny = R.nth = 1;
    R.samples_offset = 0;  // k_fleet_check hands each CTA its own candidate as the sample array
    for (int i = b; i < e; ++i) {
      robot_of[i] = r;
      for (int k = 0; k < 3; ++k) vel_f[3 * size_t(i) + k] = (float)vel_samples[3 * size_t(i) + k];  // Eigen::Vector3f
    }
  }
  NAVGPU_CUDA(cudaMemcpyAsync(d_rob, f->h_check.data(), sizeof(FleetRobot) * n, cudaMemcpyHostToDevice, f->stream));
  NAVGPU_CUDA(cudaMemcpyAsync(d_of, robot_of.data(), sizeof(int32_t) * total, cudaMemcpyHostToDevice, f->stream));
  NAVGPU_CUDA(cudaMemcpyAsync(d_vel, vel_f.data(), sizeof(float) * 3 * total, cudaMemcpyHostToDevice, f->stream));
  DwaScoreArgs base;
  fleet_dwa_base_args(f, base);
  k_fleet_check<<<(unsigned)total, 32, 0, f->stream>>>(base, d_rob, d_of, d_vel, d_cost);
  NAVGPU_LAUNCHED(1);
  NAVGPU_CUDA(cudaGetLastError());
  NAVGPU_CUDA(cudaMemcpyAsync(costs_out, d_cost, b_cost, cudaMemcpyDeviceToHost, f->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(f->stream));
  return NAVGPU_OK;
}

int navgpu_fleet_set_scans(navgpu_fleet* f, const navgpu_laser_scan* scans, const int32_t* offsets) {
  if (!f) return fail(NAVGPU_ERR_INVALID, "null handle");
  if (!f->sensing) return fail(NAVGPU_ERR_INVALID, "not a sensing fleet (navgpu_fleet_create_sensing)");
  return fleet_costmap_set_scans(f->sensing, scans, offsets);
}

int navgpu_fleet_set_scan_batch(navgpu_fleet* f, const navgpu_fleet_scan_source* sources, int n_sources) {
  if (!f) return fail(NAVGPU_ERR_INVALID, "null handle");
  if (!f->sensing) return fail(NAVGPU_ERR_INVALID, "not a sensing fleet (navgpu_fleet_create_sensing)");
  return fleet_costmap_set_scan_batch(f->sensing, sources, n_sources, false);
}

int navgpu_fleet_set_scan_batch_device(navgpu_fleet* f, const navgpu_fleet_scan_source* sources, int n_sources) {
  if (!f) return fail(NAVGPU_ERR_INVALID, "null handle");
  if (!f->sensing) return fail(NAVGPU_ERR_INVALID, "not a sensing fleet (navgpu_fleet_create_sensing)");
  return fleet_costmap_set_scan_batch(f->sensing, sources, n_sources, true);
}

void* navgpu_fleet_stream(navgpu_fleet* f) { return f ? (void*)f->stream : nullptr; }

int navgpu_fleet_get_layer(navgpu_fleet* f, int robot, uint8_t* host_out) {
  if (!f || robot < 0 || robot >= f->n || !host_out) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (!f->sensing) return fail(NAVGPU_ERR_INVALID, "not a sensing fleet (navgpu_fleet_create_sensing)");
  return fleet_costmap_get(f->sensing, robot, false, host_out);
}

int navgpu_fleet_get_voxels(navgpu_fleet* f, int robot, uint32_t* host_out) {
  if (!f || robot < 0 || robot >= f->n || !host_out) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (!f->sensing) return fail(NAVGPU_ERR_INVALID, "not a sensing fleet (navgpu_fleet_create_sensing_voxel)");
  return fleet_costmap_get_voxels(f->sensing, robot, host_out);
}

int navgpu_fleet_get_geometry(navgpu_fleet* f, int robot, double origin_out[2], int32_t window_out[4]) {
  if (!f || robot < 0 || robot >= f->n || !origin_out || !window_out) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (!f->sensing) return fail(NAVGPU_ERR_INVALID, "not a sensing fleet (navgpu_fleet_create_sensing)");
  NAVGPU_TRY(fleet_state_to_host(f));
  return fleet_costmap_geometry(f->sensing, robot, origin_out, window_out);
}

int navgpu_fleet_last_timing(navgpu_fleet* f, float* project_ms, float* costmap_ms) {
  if (!f) return fail(NAVGPU_ERR_INVALID, "null handle");
  if (!f->sensing) return fail(NAVGPU_ERR_INVALID, "not a sensing fleet (navgpu_fleet_create_sensing)");
  return fleet_costmap_last_timing(f->sensing, project_ms, costmap_ms);
}

}  // extern "C"

// the legacy TrajectoryPlanner shares this translation unit's kernels (MapGrid wavefront, footprint walks)
#include "tp_host.inc"
