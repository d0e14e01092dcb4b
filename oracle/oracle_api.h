/*
 * oracle_api.h -- C ABI shared by the two CPU checkers of this repository.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under navigation_b200/ may include, link or load anything
 * from oracle/.  Only tests/, __graft_entry__.smoke() and bench.py (cpu_baseline / --impl reference)
 * use it, and only as the checker or the timed CPU baseline.
 *
 * Two shared libraries export exactly these symbols:
 *   oracle/_ref/libnavref.so   the reference's own, unmodified hot-path sources compiled from
 *                              /root/reference against oracle/shim (built by oracle/Makefile,
 *                              git-ignored); glue in oracle/ref_harness.cpp.
 *   oracle/libnavoracle.so     a from-scratch CPU restatement (oracle/navoracle.cpp) that is
 *                              pinned against libnavref.so and the reference's golden vectors.
 *
 * Path A mirrors costmap_2d::LayeredCostmap + Layer plugins (costmap_2d/src/layered_costmap.cpp:79-150).
 * Path B mirrors dwa_local_planner::DWAPlanner::findBestPath (dwa_local_planner/src/dwa_planner.cpp:292-371).
 */
#ifndef NAV_ORACLE_API_H_
#define NAV_ORACLE_API_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* merge policies of CostmapLayer (costmap_2d/src/costmap_layer.cpp:62-157) */
enum { NAVO_TRUE_OVERWRITE = 0, NAVO_OVERWRITE = 1, NAVO_MAX = 2, NAVO_ADDITION = 3, NAVO_NOTHING = 4 };

/* one costmap_2d::Observation (costmap_2d/include/costmap_2d/observation.h:47-100) */
typedef struct {
  double origin_x, origin_y, origin_z;
  double obstacle_range, raytrace_range;
  const float* xyz; /* n_points * 3 float32, world frame (pcl::PointXYZ payload) */
  int32_t n_points;
  int32_t marking;  /* used by the marking loop  (obstacle_layer.cpp:368-410) */
  int32_t clearing; /* used by raytraceFreespace (obstacle_layer.cpp:498-576) */
  int32_t pad_;
} navo_observation;

/* ---- Path A ---- */
void* navo_costmap_create(uint32_t size_x, uint32_t size_y, double resolution, double origin_x, double origin_y,
                          int rolling_window, int track_unknown);
void navo_costmap_destroy(void* h);
/* layers are appended in plugin order; each call returns the layer index */
int navo_costmap_add_grid_layer(void* h, int policy);
int navo_costmap_add_obstacle_layer(void* h, int combination_method, int footprint_clearing,
                                    double max_obstacle_height);
/* VoxelLayer (costmap_2d/plugins/voxel_layer.cpp, cfg/VoxelPlugin.cfg): a 3-D obstacle layer; observations, enable and
 * grid read-back work through the obstacle-layer calls.  navo_layer_get_voxels: size_x*size_y uint32 columns. */
int navo_costmap_add_voxel_layer(void* h, int combination_method, int footprint_clearing, double max_obstacle_height,
                                 double origin_z, double z_resolution, int z_voxels, int unknown_threshold,
                                 int mark_threshold);
void navo_layer_get_voxels(void* h, int layer, uint32_t* out);
/* voxel_grid::VoxelGrid::raytraceLine (voxel_grid.h:226-297): the visited voxels as (grid offset, z) pairs; returns count */
int navo_voxel_line_cells(uint32_t size_x, double x0, double y0, double z0, double x1, double y1, double z1,
                          uint32_t max_length, uint32_t* offsets_out, int32_t* z_out, int capacity);
int navo_costmap_add_inflation_layer(void* h, double inflation_radius, double cost_scaling_factor);
/* LayeredCostmap::setFootprint (layered_costmap.cpp:163-173); xy = n (x,y) pairs in the robot frame */
void navo_costmap_set_footprint(void* h, const double* xy, int n);
/* overwrite the whole grid of a grid layer and flag it as updated (StaticLayer::incomingMap semantics) */
void navo_grid_layer_set(void* h, int layer, const uint8_t* data);
/* flag a grid layer region dirty without changing data: static_layer.cpp:263-285 bounds = map corners of (x,y,w,h) */
void navo_grid_layer_touch(void* h, int layer, uint32_t x, uint32_t y, uint32_t w, uint32_t hgt);
void navo_layer_set_enabled(void* h, int layer, int enabled);
/* observations persist until replaced (ObstacleLayer::addStaticObservation, obstacle_layer.cpp:450-464) */
void navo_obstacle_set_observations(void* h, int layer, const navo_observation* obs, int n_obs);
void navo_inflation_set_params(void* h, int layer, double inflation_radius, double cost_scaling_factor);
/* Checker-only: which legal execution of InflationLayer::updateCosts (inflation_layer.cpp:226-265) the checker runs.
 * The reference pops equal-distance queue entries in whatever order libstdc++'s heap history produces; on diagonal or
 * point-like obstacle boundaries the result depends on that order.  variant: 0 = the reference as written
 * (std::priority_queue, same push order: reproduces the compiled reference bit for bit), 1 = oldest entry first
 * (FIFO), 2 = newest first (LIFO), 3 = seeded pseudo-random order, 4 = exact windowed nearest-seed inflation (the
 * specification of libnavgpu's inflation mode 0; not a propagation), 5 = level-synchronous propagation (the
 * specification of libnavgpu's inflation mode 1; a legal execution), 6 = the certificate of that: the reference's
 * sequential priority-queue loop with equal-distance ties resolved towards variant 5's sources, which must reproduce
 * variant 5 bit for bit.  Cells that differ between variants 0-3 form the
 * "tie-variant mask" of a scenario.  Returns 0, or -1 when the library cannot run the variant (libnavref.so: only 0). */
int navo_inflation_set_variant(void* h, int layer, int variant, uint64_t seed);
/* rounds (distinct pop levels -- the seeds' level 0 included -- and repeats after a shorter entry appears) of
 * variant 5's last updateCosts: what navgpu_inflation_last_rounds reports for mode 1 */
int navo_inflation_last_rounds(void* h, int layer);
/* LayeredCostmap::updateMap; window_out = {x0, xn, y0, yn} (bx0_, bxn_, by0_, byn_) */
void navo_costmap_update_map(void* h, double robot_x, double robot_y, double robot_yaw, int32_t window_out[4]);
void navo_costmap_get(void* h, uint8_t* out);
void navo_costmap_set(void* h, const uint8_t* in); /* poke the master grid (tests of stateful windowing) */
void navo_layer_get(void* h, int layer, uint8_t* out);
void navo_costmap_get_origin(void* h, double out[2]);
/* InflationLayer cached tables: (R+2)*(R+2) entries each, row-major [i][j]; returns R = cell_inflation_radius_ */
int navo_inflation_tables(void* h, int layer, uint8_t* costs_out, double* dists_out, int capacity);

/* stand-alone helpers */
/* StaticLayer::interpretValue (static_layer.cpp:149-163) over n values */
void navo_interpret_values(const uint8_t* in, uint8_t* out, int64_t n, int track_unknown, uint8_t unknown_cost_value,
                           uint8_t lethal_threshold, int trinary);
/* Costmap2D::raytraceLine<MarkCell> cells, in visiting order (costmap_2d.h:359-412); returns count */
int navo_raytrace_cells(uint32_t size_x, uint32_t x0, uint32_t y0, uint32_t x1, uint32_t y1, uint32_t max_length,
                        uint32_t* offsets_out, int capacity);
/* calculateMinAndMaxDistances (footprint.cpp:41-67) */
void navo_footprint_radii(const double* xy, int n, double* inscribed, double* circumscribed);

/* observation ingest (SURVEY.md 8f-3), restated in oracle/scan_ingest_restated.h (see its header: the third-party
 * part of this path is PARITY UNPINNED).  Returns the number of points of the resulting world-frame cloud. */
typedef struct {
  const float* ranges;
  int32_t n_ranges;
  int32_t inf_is_valid;
  float angle_min, angle_increment, range_min, range_max;
  double translation[3];   /* tf: global frame <- sensor frame */
  double rotation_xyzw[4];
  double min_obstacle_height, max_obstacle_height;
  int32_t is_cloud; /* 1: `ranges` holds n_ranges sensor-frame points (x, y, z): a PointCloud(2) source, no projection */
  int32_t pad_;
} navo_laser_scan;
int navo_project_scan(const navo_laser_scan* scan, float* xyz_out, int capacity, double origin_out[3]);

/* ---- Path B ---- */
typedef struct {
  /* base_local_planner::LocalPlannerLimits (local_planner_limits.h:43-124) */
  double max_trans_vel, min_trans_vel, max_vel_x, min_vel_x, max_vel_y, min_vel_y, max_rot_vel, min_rot_vel;
  double acc_lim_x, acc_lim_y, acc_lim_theta;
  /* DWAPlannerConfig (dwa_local_planner/cfg/DWAPlanner.cfg) */
  double sim_time, sim_granularity, angular_sim_granularity, sim_period;
  double path_distance_bias, goal_distance_bias, occdist_scale;
  double forward_point_distance, cheat_factor;
  double oscillation_reset_dist, oscillation_reset_angle;
  double scaling_speed, max_scaling_factor;
  int32_t vx_samples, vy_samples, vth_samples;
  int32_t use_dwa, sum_scores, allow_unknown; /* allow_unknown: honoured by the restatement only (see DESIGN.md) */
} navo_dwa_config;

typedef struct {
  double cost;       /* result_traj_.cost_ (-7 when nothing valid; dwa_planner.cpp:316) */
  double xv, yv, thetav;
  int32_t best_index; /* index into the enumerated sample list (x outer, y, theta inner), -1 if none */
  int32_t n_samples;  /* number of enumerated samples */
  int32_t n_scored;   /* samples for which generateTrajectory returned true */
  int32_t n_points;   /* points of the winning trajectory */
} navo_dwa_result;

void navo_dwa_default_config(navo_dwa_config* cfg);
void* navo_dwa_create(const navo_dwa_config* cfg, uint32_t size_x, uint32_t size_y, double resolution);
void navo_dwa_destroy(void* h);
/* DWAPlanner::reconfigure (dwa_planner.cpp:52-112) of a live handle: plans, oscillation flags and result_traj_ are
 * kept.  cheat_factor and sum_scores, which the reference reads only at construction, are taken from cfg as well,
 * as navgpu_dwa_reconfigure takes them. */
void navo_dwa_reconfigure(void* h, const navo_dwa_config* cfg);
void navo_dwa_set_costmap(void* h, const uint8_t* grid, double origin_x, double origin_y);
/* DWAPlanner::updatePlanAndLocalCosts (dwa_planner.cpp:240-286); plan_xy = n (x,y) pairs */
void navo_dwa_set_plan(void* h, const double pose[3], const double* plan_xy, int n);
void navo_dwa_reset_oscillation(void* h);
int navo_dwa_get_oscillation_mask(void* h); /* bit0 fwd_pos_only,1 fwd_neg_only,2 strafe_pos_only,3 strafe_neg_only,4 rot_pos_only,5 rot_neg_only */
/* DWAPlanner::findBestPath.  all_costs (nullable, capacity >= n_samples): cost reported in all_explored for each
 * enumerated sample, NaN for samples the generator rejected.  best_points (nullable): 3*capacity doubles. */
int navo_dwa_find_best_path(void* h, const double pose[3], const double vel[3], const double* footprint_xy,
                            int n_footprint, navo_dwa_result* result, double* all_costs, int all_capacity,
                            double* best_points, int points_capacity);
/* DWAPlanner::checkTrajectory (dwa_planner.cpp:213-237): resets the oscillation flags, generates ONE trajectory for
 * vel_samples and scores it with the critics' current state (no prepare()); returns the cost (>= 0: legal) */
double navo_dwa_check_trajectory(void* h, const double pose[3], const double vel[3], const double vel_samples[3],
                                 const double* footprint_xy, int n_footprint);
/* the four MapGrid distance fields after prepare(): which = 0 path, 1 goal, 2 goal_front, 3 alignment */
void navo_dwa_get_grid(void* h, int which, double* out);
/* only the 4 prepare() calls (MapGrid BFS), for timing them separately */
void navo_dwa_prepare_only(void* h);

/* stand-alone Path-B helpers for the reference's golden vectors */
/* VelocityIterator samples (velocity_iterator.h:47-96); returns count */
int navo_velocity_samples(double vmin, double vmax, int num_samples, double* out, int capacity);
/* LineIterator cells (line_iterator.h:38-139); xy_out = pairs; returns count */
int navo_line_cells(int x0, int y0, int x1, int y1, int32_t* xy_out, int capacity);
/* MapGrid BFS from explicit seed cells over a cost grid (map_grid.cpp:258-310) */
void navo_mapgrid_bfs(const uint8_t* costs, uint32_t size_x, uint32_t size_y, const int32_t* seeds_xy, int n_seeds,
                      int allow_unknown, double* dist_out);

/* ---- legacy base_local_planner::TrajectoryPlanner (base_local_planner/src/trajectory_planner.cpp), SURVEY 8f-4:
 * the second consumer of the rollout scorer.  libnavref.so drives the reference's own class; libnavoracle.so restates
 * it (struct Tp in navoracle.cpp) and is pinned bit-for-bit against libnavref.so, the reference's utest.cpp known
 * answer and the golden fixtures generated from the reference (tests/golden/tp_*.npz). */
typedef struct {
  double acc_lim_x, acc_lim_y, acc_lim_theta;
  double sim_time, sim_granularity, angular_sim_granularity, sim_period;
  double pdist_scale, gdist_scale, occdist_scale;
  double heading_lookahead, oscillation_reset_dist, escape_reset_dist, escape_reset_theta;
  double max_vel_x, min_vel_x, max_vel_th, min_vel_th, min_in_place_vel_th, backup_vel;
  double heading_scoring_timestep, stop_time_buffer;
  double y_vels[8];
  int32_t n_y_vels, vx_samples, vtheta_samples;
  int32_t holonomic_robot, dwa, heading_scoring, simple_attractor;
  int32_t allow_unknown; /* indeterminate in the reference (uninitialised Costmap2D copy); honoured by the CUDA path */
} navo_tp_config;
typedef struct {
  double cost, xv, yv, thetav;
  int32_t n_points;
  /* bit0 stuck_left, 1 stuck_right, 2 stuck_left_strafe, 3 stuck_right_strafe, 4 rotating_left, 5 rotating_right,
   * 6 strafe_left, 7 strafe_right, 8 escaping_ */
  int32_t flags;
} navo_tp_result;
void navo_tp_default_config(navo_tp_config* cfg); /* trajectory_planner_ros.cpp:116-213 defaults */
void* navo_tp_create(const navo_tp_config* cfg, uint32_t size_x, uint32_t size_y, double resolution,
                     const double* footprint_xy, int n_footprint);
void navo_tp_destroy(void* h);
/* TrajectoryPlanner::reconfigure (trajectory_planner.cpp:59-133) of a live handle, which clamps vx_samples and
 * vtheta_samples to at least 1; the oscillation and escape state, the plan and the distance maps are kept.  sim_period,
 * which the reference reads only at construction, is taken from cfg as well, as navgpu_tp_reconfigure takes it
 * (stop_time_buffer, the other such parameter, is read by neither findBestPath nor scoreTrajectory). */
void navo_tp_reconfigure(void* h, const navo_tp_config* cfg);
/* TrajectoryPlanner::setFootprint (trajectory_planner.h:195): xy = n (x,y) pairs in the robot frame */
void navo_tp_set_footprint(void* h, const double* xy, int n);
void navo_tp_set_costmap(void* h, const uint8_t* grid, double origin_x, double origin_y);
/* TrajectoryPlanner::updatePlan(plan, compute_dists = false), trajectory_planner.cpp:477-502 */
void navo_tp_update_plan(void* h, const double* plan_xy, int n);
/* TrajectoryPlanner::findBestPath :908-980; points = 3 doubles per point of the returned trajectory; returns 0 */
int navo_tp_find_best_path(void* h, const double pose[3], const double vel[3], navo_tp_result* result, double* points,
                           int points_capacity);
/* TrajectoryPlanner::scoreTrajectory :520-535 on the distance maps of the last findBestPath */
double navo_tp_score_trajectory(void* h, const double pose[3], const double vel[3], const double vel_samples[3]);
/* path_map_ (0) / goal_map_ (1) target_dist after the last findBestPath */
void navo_tp_get_grid(void* h, int which, double* out);

/* plan preprocessing (SURVEY.md 8f-4), restated in oracle/plan_restated.h (see its header: tf is not in the tree) */
int navo_plan_transform(const double* plan_xyz, int n, const double robot_xy[2], const double m[9], const double t[3],
                        double dist_threshold, int* first_out, double* out_xyz);
int navo_plan_prune(const double* plan_xyz, int n, const double robot_xy[2]);

const char* navo_impl_name(void);

#ifdef __cplusplus
}
#endif
#endif
