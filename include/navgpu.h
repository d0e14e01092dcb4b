/*
 * navgpu.h -- C ABI of libnavgpu.so: B200-native (sm_100a) implementation of the ROS navigation stack's two
 * data-parallel hot paths.  Plain pointers and sizes only; every entry point returns a status code (0 = ok) and
 * never throws.  There is NO CPU fallback: every entry point that computes fails with NAVGPU_ERR_CUDA when no
 * CUDA device is usable.
 *
 * Path A -- costmap layering + inflation.  A device-resident layered costmap replacing, per update cycle,
 *   costmap_2d::LayeredCostmap::updateMap            costmap_2d/src/layered_costmap.cpp:79-150
 *   Costmap2D::resetMap / updateOrigin                costmap_2d/src/costmap_2d.cpp:93-99, 264-313
 *   CostmapLayer::updateWith{TrueOverwrite,Overwrite,Max,Addition}   costmap_2d/src/costmap_layer.cpp:62-157
 *   StaticLayer::updateBounds/updateCosts (non-rolling) + interpretValue   plugins/static_layer.cpp:149-163,263-299
 *   ObstacleLayer::updateBounds (raytraceFreespace + marking + footprint)  plugins/obstacle_layer.cpp:340-425,498-610
 *   ObstacleLayer::updateCosts (setConvexPolygonCost + merge)               plugins/obstacle_layer.cpp:427-448
 *   InflationLayer::updateBounds/updateCosts/computeCaches                  plugins/inflation_layer.cpp:125-328
 * plus stateless "plugin seam" calls on a HOST master grid for use from inside a costmap_2d::Layer subclass
 * (layer.h:65-72): navgpu_inflate_host, navgpu_merge_host.
 *
 * Path B -- DWA rollout scoring: see the navgpu_dwa_* block below (dwa_local_planner/src/dwa_planner.cpp:292-371).
 *
 * Threading: one CUDA stream per handle; the caller provides mutual exclusion per handle, exactly like the
 * reference's Costmap2D::mutex_t (layered_costmap.cpp:83) and DWAPlanner::configuration_mutex_ (dwa_planner.cpp:301).
 */
#ifndef NAVGPU_H_
#define NAVGPU_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
  NAVGPU_OK = 0,
  NAVGPU_ERR_CUDA = 1,        /* no device / CUDA runtime error (message via navgpu_last_error) */
  NAVGPU_ERR_INVALID = 2,     /* bad argument */
  NAVGPU_ERR_UNSUPPORTED = 3, /* configuration outside what the kernels implement */
  NAVGPU_ERR_CAPACITY = 4     /* caller-provided buffer too small */
};

/* merge policies (costmap_layer.cpp:62-157) */
enum { NAVGPU_TRUE_OVERWRITE = 0, NAVGPU_OVERWRITE = 1, NAVGPU_MAX = 2, NAVGPU_ADDITION = 3, NAVGPU_NOTHING = 4 };

/* cost_values.h:42-45 */
enum { NAVGPU_FREE_SPACE = 0, NAVGPU_INSCRIBED = 253, NAVGPU_LETHAL = 254, NAVGPU_NO_INFORMATION = 255 };

const char* navgpu_last_error(void);
/* number of usable CUDA devices (0 when none) */
int navgpu_device_count(void);
/* total number of kernels launched by this library in this process (for bench.py's gpu_launches) */
uint64_t navgpu_launch_count(void);

/* one costmap_2d::Observation (observation.h:47-100); xyz = n_points * 3 float32 in the world frame */
typedef struct {
  double origin_x, origin_y, origin_z;
  double obstacle_range, raytrace_range;
  const float* xyz;
  int32_t n_points;
  int32_t marking;
  int32_t clearing;
  int32_t pad_;
} navgpu_observation;

typedef struct navgpu_costmap navgpu_costmap;

/* ---- Path A: device-resident LayeredCostmap -------------------------------------------------------------- */
/* LayeredCostmap ctor + resizeMap (layered_costmap.cpp:50-77). device = CUDA ordinal. */
int navgpu_costmap_create(navgpu_costmap** out, uint32_t size_x, uint32_t size_y, double resolution, double origin_x,
                          double origin_y, int rolling_window, int track_unknown, int device);
int navgpu_costmap_destroy(navgpu_costmap* h);
/* layers are appended in plugin order (costmap_2d_ros.cpp:115-128); *layer_out receives the index */
int navgpu_costmap_add_grid_layer(navgpu_costmap* h, int policy, int* layer_out);
int navgpu_costmap_add_obstacle_layer(navgpu_costmap* h, int combination_method, int footprint_clearing,
                                      double max_obstacle_height, int* layer_out);
/* VoxelLayer (costmap_2d/plugins/voxel_layer.cpp, cfg/VoxelPlugin.cfg): the 3-D obstacle layer -- columns of up to 16
 * voxels (voxel_grid/include/voxel_grid/voxel_grid.h), 3-D Bresenham clearing, marking, rolling origin.  It takes
 * observations, enable and grid read-back through the obstacle-layer calls.  mark_threshold must be 0 (the default). */
int navgpu_costmap_add_voxel_layer(navgpu_costmap* h, int combination_method, int footprint_clearing,
                                   double max_obstacle_height, double origin_z, double z_resolution, int z_voxels,
                                   int unknown_threshold, int mark_threshold, int* layer_out);
/* the voxel columns (size_y x size_x uint32: bit z = unknown-or-marked, bit z + 16 = marked) to HOST */
int navgpu_layer_get_voxels(navgpu_costmap* h, int layer, uint32_t* host_out);
int navgpu_costmap_add_inflation_layer(navgpu_costmap* h, double inflation_radius, double cost_scaling_factor,
                                       int* layer_out);
/* LayeredCostmap::setFootprint (layered_costmap.cpp:163-173): n (x,y) pairs, robot frame */
int navgpu_costmap_set_footprint(navgpu_costmap* h, const double* xy, int n);
/* whole-grid upload of a grid layer from HOST memory, marks it updated (StaticLayer::incomingMap :165-223) */
int navgpu_grid_layer_set(navgpu_costmap* h, int layer, const uint8_t* host_data);
/* same, from DEVICE memory (row pitch in bytes) */
int navgpu_grid_layer_set_device(navgpu_costmap* h, int layer, const uint8_t* dev_data, uint32_t pitch);
/* OccupancyGrid ingest on the device: interpretValue over int8 occupancy from HOST memory (static_layer.cpp:149-207) */
int navgpu_grid_layer_set_occupancy(navgpu_costmap* h, int layer, const int8_t* host_occupancy, int track_unknown,
                                    uint8_t unknown_cost_value, uint8_t lethal_threshold, int trinary);
int navgpu_grid_layer_touch(navgpu_costmap* h, int layer, uint32_t x, uint32_t y, uint32_t w, uint32_t hgt);
int navgpu_layer_set_enabled(navgpu_costmap* h, int layer, int enabled);
/* observations persist until replaced (ObstacleLayer::addStaticObservation :450-464); copied H2D here */
int navgpu_obstacle_set_observations(navgpu_costmap* h, int layer, const navgpu_observation* obs, int n_obs);
/* Observation ingest on the device (SURVEY.md 8f-3): one sensor_msgs/LaserScan per observation instead of a
 * world-frame cloud.  Replaces, per scan, laser_geometry's projection in ObstacleLayer::laserScanCallback /
 * laserScanValidInfCallback (plugins/obstacle_layer.cpp:252-311) and ObservationBuffer::bufferCloud
 * (src/observation_buffer.cpp:129-195: sensor origin, pcl_ros::transformPointCloud into the global frame, height
 * filter).  sensor_to_global_* is the tf transform bufferCloud looks up (global_frame <- sensor frame). */
typedef struct {
  const float* ranges; /* LaserScan.ranges, n_ranges float32 (NaN / inf allowed, as on the wire) */
  int32_t n_ranges;
  int32_t inf_is_valid; /* inf_is_valid source parameter: +inf counts as range_max - 0.0001 (:277-292) */
  float angle_min, angle_increment, range_min, range_max;
  double sensor_to_global_translation[3];
  double sensor_to_global_rotation_xyzw[4]; /* unit quaternion, tf order */
  double min_obstacle_height, max_obstacle_height; /* of the ObservationBuffer */
  double obstacle_range, raytrace_range;
  int32_t marking, clearing;
  int32_t is_cloud; /* 0: LaserScan ranges; 1: `ranges` holds n_ranges sensor-frame points (3 floats each) */
  int32_t pad_;
} navgpu_laser_scan;
/* A PointCloud / PointCloud2 source is the same path without the projection (pointCloudCallback /
 * pointCloud2Callback, obstacle_layer.cpp:313-339): set `ranges` to the cloud's n_ranges x (x, y, z) float32 in the
 * SENSOR frame and is_cloud = 1 below; angle_* / range_* / inf_is_valid are then ignored. */
/* replaces the layer's observations by the n_scans scans (like navgpu_obstacle_set_observations, they persist) */
int navgpu_obstacle_set_scans(navgpu_costmap* h, int layer, const navgpu_laser_scan* scans, int n_scans);
/* the cloud of observation `index` as the layer holds it on the device, dropped rays removed (tests, debugging);
 * returns the point count in *n_out, copies min(count, capacity) points of 3 floats */
int navgpu_obstacle_get_cloud(navgpu_costmap* h, int layer, int index, float* xyz_out, int capacity, int* n_out);
/* InflationLayer::setInflationParameters (:356-370) */
int navgpu_inflation_set_params(navgpu_costmap* h, int layer, double inflation_radius, double cost_scaling_factor);
/* Which implementation of InflationLayer::updateCosts (inflation_layer.cpp:172-293) the layer runs.  Both write
 * max(old, cached cost) with the NO_INFORMATION rule (:249-254), both are tested bit for bit against a CPU
 * specification (oracle variants 4 / 5), and both equal the reference itself wherever the order in which its priority
 * queue pops equal-distance entries cannot matter (thick axis-aligned structures).
 *   0 (default)  exact windowed nearest-seed inflation: every cell within the cached distance R of a LETHAL cell of
 *                window +- R gets the cost of its NEAREST such cell.  Never lower than the reference; higher on the
 *                rare cells the reference's propagation reaches only with a farther source.
 *   1            level-synchronous nearest-source propagation: the reference's loop itself (sources carried through
 *                4-neighbours, `seen` at pop, distance gate at enqueue), equal distances resolved by a fixed rule
 *                instead of libstdc++'s heap history -- a legal execution of the reference's code; equals the reference
 *                on every cell whose value does not depend on that history.  R <= 127.  One persistent kernel with a
 *                grid barrier per distance level: about 1 ms at 4000 x 4000, R = 20 instead of 0.04 ms for mode 0. */
int navgpu_inflation_set_mode(navgpu_costmap* h, int layer, int mode);
/* number of pop rounds (distance levels) of the last mode-1 update of this costmap; synchronises the stream */
int navgpu_inflation_last_rounds(navgpu_costmap* h, int* rounds_out);
/* LayeredCostmap::updateMap.  Synchronous: returns after the cycle's kernels finished.
 * window_out = {x0, xn, y0, yn} (LayeredCostmap::getBounds). */
int navgpu_costmap_update_map(navgpu_costmap* h, double robot_x, double robot_y, double robot_yaw,
                              int32_t window_out[4]);
/* enqueue-only variant (no host synchronisation, no window read-back): for timing and pipelining */
int navgpu_costmap_update_map_async(navgpu_costmap* h, double robot_x, double robot_y, double robot_yaw);
int navgpu_costmap_synchronize(navgpu_costmap* h);
/* measurement hooks: when enabled, navgpu_costmap_update_map_async brackets the whole cycle and the fused
 * reset+merge+inflation sweep with CUDA events on the handle's stream; last_timing returns both (ms).  The events
 * themselves cost a few microseconds per cycle, so throughput is measured with profiling off. */
int navgpu_costmap_set_profiling(navgpu_costmap* h, int enabled);
/* test hook: use the generic (any-R) fused sweep kernel even where the R <= 31 two-kernel fast path applies */
int navgpu_costmap_force_generic_sweep(navgpu_costmap* h, int enabled);
int navgpu_costmap_last_timing(navgpu_costmap* h, float* cycle_ms, float* sweep_ms);
/* the sweep's two kernels separately: streaming merge + seed bitmask (k_merge_seed), inflation (k_inflate) */
int navgpu_costmap_last_timing_split(navgpu_costmap* h, float* merge_ms, float* inflate_ms);
/* the CUDA stream of this handle (cudaStream_t) so callers can record events on it */
void* navgpu_costmap_stream(navgpu_costmap* h);
/* master grid read-back to HOST: whole grid, or a window [x0,xn) x [y0,yn) packed row-major into out */
int navgpu_costmap_get(navgpu_costmap* h, uint8_t* host_out);
int navgpu_costmap_get_window(navgpu_costmap* h, int x0, int y0, int xn, int yn, uint8_t* host_out);
/* the same, written straight into a host grid whose rows are host_pitch bytes apart -- e.g. the buffer of the host
 * Costmap2D the adapter keeps in sync (host_grid points at cell (0, 0); the window lands at its own place in it) */
int navgpu_costmap_get_window_into(navgpu_costmap* h, int x0, int y0, int xn, int yn, uint8_t* host_grid,
                                   uint32_t host_pitch);
/* Keeps a HOST mirror of the master grid (the Costmap2D the rest of the stack reads after
 * LayeredCostmap::updateMap, layered_costmap.cpp:79-150) byte-identical to the device grid while moving only what
 * changed.  The device holds a shadow of what `host_grid` contains; one kernel compares the master grid with it in
 * tiles of 128 x 16 cells, writes the tiles that differ -- compacted, through mapped pinned memory -- and the call
 * scatters them into host_grid (rows host_pitch bytes apart, cell (0, 0) first).  The first call for a given host_grid,
 * a call after navgpu_costmap_mirror_invalidate, and a cycle that changed more than a quarter of the grid copy the whole
 * grid instead.  The call synchronises the handle's stream, so `navgpu_costmap_update_map_async` + this is one
 * complete cycle with a single host wait; the cycle's window is then available from navgpu_costmap_last_window.
 * rects_out (nullable): x0, y0, xn, yn of every changed tile, up to rects_capacity of them; *n_rects_out: how many
 * tiles changed (when it exceeds rects_capacity treat the whole grid as changed); *d2h_bytes_out: bytes that crossed
 * PCIe for this call.  The host must not write host_grid between calls (or must call navgpu_costmap_mirror_invalidate). */
int navgpu_costmap_get_changed(navgpu_costmap* h, uint8_t* host_grid, uint32_t host_pitch, int32_t* rects_out,
                               int rects_capacity, int32_t* n_rects_out, uint64_t* d2h_bytes_out);
int navgpu_costmap_mirror_invalidate(navgpu_costmap* h);
/* {x0, xn, y0, yn} of the last cycle whose window reached the host (navgpu_costmap_update_map, navgpu_costmap_get_changed) */
int navgpu_costmap_last_window(navgpu_costmap* h, int32_t window_out[4]);
/* page-lock / release a host buffer the caller owns, so that copies from and to it run at full PCIe speed (a pageable
 * 16 MB download takes about 4x as long); purely an optimisation, every entry point also accepts pageable memory */
int navgpu_host_register(void* ptr, size_t bytes);
int navgpu_host_unregister(void* ptr);
/* the same window as nav_msgs/OccupancyGrid data: Costmap2DPublisher's cost translation table
 * (costmap_2d/src/costmap_2d_publisher.cpp:56-71, 139-152) applied on the device while the window is packed */
int navgpu_costmap_get_window_occupancy(navgpu_costmap* h, int x0, int y0, int xn, int yn, int8_t* host_out);
int navgpu_costmap_set(navgpu_costmap* h, const uint8_t* host_in);
int navgpu_layer_get(navgpu_costmap* h, int layer, uint8_t* host_out);
int navgpu_costmap_get_origin(navgpu_costmap* h, double out[2]);
/* device pointer + pitch of the master grid (for zero-copy consumers such as the Path-B scorer) */
int navgpu_costmap_device_grid(navgpu_costmap* h, const uint8_t** dev_ptr, uint32_t* pitch);
/* InflationLayer cached tables (computeCaches :295-328), (R+2)*(R+2) each; *radius_out = cell_inflation_radius_ */
int navgpu_inflation_tables(navgpu_costmap* h, int layer, uint8_t* costs_out, double* dists_out, int capacity,
                            int* radius_out);

/* ---- Path A: stateless plugin-seam calls on a HOST master grid -------------------------------------------- */
/* Drop-in body for InflationLayer::updateCosts(master, min_i, min_j, max_i, max_j) (inflation_layer.cpp:172-266):
 * uploads the affected window, inflates on the device, writes the result back into master.  cost_table is the
 * (R+2)*(R+2) cached_costs_ array (row-major [dx][dy]) built with the reference formula. */
int navgpu_inflate_host(uint8_t* master, uint32_t size_x, uint32_t size_y, int min_i, int min_j, int max_i, int max_j,
                        const uint8_t* cost_table, uint32_t cell_inflation_radius, int device);
/* Drop-in body for CostmapLayer::updateWith* (costmap_layer.cpp:62-157) */
int navgpu_merge_host(uint8_t* master, const uint8_t* layer, uint32_t size_x, uint32_t size_y, int min_i, int min_j,
                      int max_i, int max_j, int policy, int device);
/* InflationLayer::computeCost table builder (inflation_layer.h:114-129, .cpp:295-328) -- host-side, exact formula */
int navgpu_build_cost_table(double resolution, double inscribed_radius, double inflation_radius,
                            double cost_scaling_factor, uint8_t* costs_out, double* dists_out, int capacity,
                            int* radius_out);

/* ---- Path B: DWA rollout scoring ------------------------------------------------------------------------- */
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
  int32_t use_dwa, sum_scores, allow_unknown;
} navgpu_dwa_config;

typedef struct {
  double cost; /* result_traj_.cost_; -7 when nothing valid (dwa_planner.cpp:316) */
  double xv, yv, thetav;
  int32_t best_index; /* index into the enumerated samples (x outer, y, theta inner); -1 if none */
  int32_t n_samples;
  int32_t n_scored;
  int32_t n_points;
} navgpu_dwa_result;

typedef struct navgpu_dwa navgpu_dwa;

void navgpu_dwa_default_config(navgpu_dwa_config* cfg);
/* DWAPlanner ctor + reconfigure (dwa_planner.cpp:52-182) for a local costmap of size_x x size_y cells */
int navgpu_dwa_create(navgpu_dwa** out, const navgpu_dwa_config* cfg, uint32_t size_x, uint32_t size_y,
                      double resolution, int device);
int navgpu_dwa_destroy(navgpu_dwa* h);
int navgpu_dwa_reconfigure(navgpu_dwa* h, const navgpu_dwa_config* cfg);
/* local costmap contents from HOST memory (what the critics read through Costmap2D*, dwa_planner.cpp:118-122) */
int navgpu_dwa_set_costmap(navgpu_dwa* h, const uint8_t* host_grid, double origin_x, double origin_y);
/* zero-copy: score against a device-resident grid (e.g. navgpu_costmap_device_grid of the local costmap) */
int navgpu_dwa_set_costmap_device(navgpu_dwa* h, const uint8_t* dev_grid, uint32_t pitch, double origin_x,
                                  double origin_y);
/* DWAPlanner::updatePlanAndLocalCosts (dwa_planner.cpp:240-286) */
int navgpu_dwa_set_plan(navgpu_dwa* h, const double pose[3], const double* plan_xy, int n);
/* DWAPlanner::setPlan's oscillation reset (dwa_planner.cpp:204-207) */
int navgpu_dwa_reset_oscillation(navgpu_dwa* h);
int navgpu_dwa_get_oscillation_mask(navgpu_dwa* h, int* mask_out);
/* DWAPlanner::findBestPath (dwa_planner.cpp:292-371): 4x MapGrid prepare, sample enumeration, rollout, 6 critics,
 * argmin, oscillation-flag update.  all_costs (nullable): per enumerated sample the cost the reference reports in
 * all_explored (NaN for samples its generator rejects).  best_points (nullable): 3*points_capacity doubles.
 * Returns NAVGPU_OK also when no valid trajectory exists (result->cost < 0, like the reference). */
int navgpu_dwa_find_best_path(navgpu_dwa* h, const double pose[3], const double vel[3], const double* footprint_xy,
                              int n_footprint, navgpu_dwa_result* result, double* all_costs, int all_capacity,
                              double* best_points, int points_capacity);
/* DWAPlanner::checkTrajectory (dwa_planner.cpp:213-237): resets the oscillation flags, generates the ONE trajectory
 * of vel_samples and scores it with the critics' state of the last findBestPath (no prepare()); *cost_out >= 0
 * means the trajectory is legal.  A sample the generator rejects scores 0, exactly like the reference. */
int navgpu_dwa_check_trajectory(navgpu_dwa* h, const double pose[3], const double vel[3], const double vel_samples[3],
                                const double* footprint_xy, int n_footprint, double* cost_out);
/* ---- the batched base_local_planner::TrajectoryCostFunction backend (trajectory_cost_function.h:52-82) -----------
 * For callers that keep the reference's own search (SimpleScoredSamplingPlanner, simple_scored_sampling_planner.cpp
 * :81-142) and / or their own TrajectorySampleGenerator: the six critics DWAPlanner wires up (dwa_planner.cpp:116-182),
 * as ONE cost function over trajectories the caller generated.
 *   navgpu_dwa_prepare             = prepare() of the critics: the four MapGridCostFunction wavefronts on the costmap
 *                                    and plan the handle holds (map_grid_cost_function.cpp:59-68); no host wait
 *   navgpu_dwa_score_trajectories  = scoreTrajectory for n_traj trajectories in one launch.  Trajectory t has points
 *                                    offsets[t] .. offsets[t + 1] - 1 of points_xyth (x, y, theta doubles, what
 *                                    Trajectory::getPoint returns) and velocities vels[3 t ..] = xv_, yv_, thetav_.
 *                                    costs_out[t] = what SimpleScoredSamplingPlanner::scoreTrajectory (:50-79) returns
 *                                    for it with best_traj_cost = -1: the critics' scaled costs summed in DWAPlanner's
 *                                    order, or the first negative code (-5 oscillation, -6 footprint / off the map,
 *                                    -9 empty footprint, -4 / -3 / -2 map grid).  terms_out (nullable): the six
 *                                    per-critic terms of every trajectory.
 *   navgpu_dwa_update_oscillation  = OscillationCostFunction::updateOscillationFlags (oscillation_cost_function.cpp
 *                                    :56-68) with the trajectory the caller's search selected. */
int navgpu_dwa_prepare(navgpu_dwa* h);
int navgpu_dwa_score_trajectories(navgpu_dwa* h, int n_traj, const int32_t* offsets, const double* points_xyth,
                                  const double* vels, const double* footprint_xy, int n_footprint, double* costs_out,
                                  double* terms_out);
int navgpu_dwa_update_oscillation(navgpu_dwa* h, const double pose[3], double cost, double xv, double yv, double thetav);
/* the per-axis velocity samples of the last search (SimpleTrajectoryGenerator::initialise,
 * simple_trajectory_generator.cpp:60-135): counts_out = {nx, ny, nth}; samples_out = xs | ys | ths (float32, exactly
 * Eigen::Vector3f's values); sample index i = (ix * ny + iy) * nth + ith */
int navgpu_dwa_get_samples(navgpu_dwa* h, int32_t counts_out[3], float* samples_out, int capacity);
/* sample-range sharded variant for multi-GPU sweeps: scores enumerated samples [begin, end) only and returns this
 * shard's (cost, global index) minimum without touching the oscillation state; cost = +inf when none valid. */
int navgpu_dwa_score_range(navgpu_dwa* h, const double pose[3], const double vel[3], const double* footprint_xy,
                           int n_footprint, int64_t begin, int64_t end, double* best_cost, int64_t* best_index,
                           int64_t* n_samples_total);
/* finish a sharded sweep on every rank: given the all-gathered per-rank (cost,index) minima pick the winner exactly
 * as simple_scored_sampling_planner.cpp:111-116 would, regenerate its trajectory and update the oscillation flags */
int navgpu_dwa_finish_sharded(navgpu_dwa* h, const double pose[3], const double* costs, const int64_t* indices,
                              int n_ranks, navgpu_dwa_result* result, double* best_points, int points_capacity);
/* The same with the samples dealt out block-cyclically instead of in contiguous ranges: rank r of `world` scores the
 * 8-sample blocks r, r + world, r + 2 world, ... of the enumeration.  Trajectory length grows with the outer (vx)
 * index, so contiguous ranges leave the last rank with 1.6x the mean work at 8 ranks; block-cyclic shares are even.
 * The (cost, lowest index) winner does not depend on the partition (simple_scored_sampling_planner.cpp:111-116). */
int navgpu_dwa_score_strided(navgpu_dwa* h, const double pose[3], const double vel[3], const double* footprint_xy,
                             int n_footprint, int rank, int world, double* best_cost, int64_t* best_index,
                             int64_t* n_samples_total);

/* ---- multi-GPU sweep with the exchange on the device (SURVEY.md 8e, config C4) ----------------------------------
 * One planner handle per GPU (one process per GPU, or one process driving several).  Every rank scores its
 * block-cyclic share; the LAST CTA of its scoring kernel stores the rank's 16-byte (cost, index) minimum straight into
 * every peer's exchange buffer (peer-mapped device memory: the stores cross NVLink / NVSwitch), waits until all `world`
 * records of the sweep have arrived in its own buffer, picks the reference's winner and regenerates its trajectory --
 * all inside the one kernel launch.  No host round trip and no collective-library call between scoring and result;
 * every rank ends with the identical result and oscillation state.
 * Setup, once: each rank exports its buffer (a cudaIpcMemHandle_t, 64 bytes), the ranks exchange the handles by any
 * means (MPI, a socket, a file), each rank connects.  In one process: navgpu_dwa_shard_connect_local. */
#define NAVGPU_IPC_HANDLE_BYTES 64
int navgpu_dwa_shard_export(navgpu_dwa* h, void* ipc_handle_out /* NAVGPU_IPC_HANDLE_BYTES */);
int navgpu_dwa_shard_connect(navgpu_dwa* h, int rank, int world, const void* ipc_handles /* world x 64 bytes, rank order */);
int navgpu_dwa_shard_connect_local(navgpu_dwa* const* handles, int world); /* handles[r] becomes rank r */
/* DWAPlanner::findBestPath over all ranks; every rank must call it once per cycle with the same inputs (costmap, plan,
 * pose, velocity, footprint).  A rank whose peers do not answer within two seconds returns cost -7 (nothing valid). */
int navgpu_dwa_find_best_path_sharded(navgpu_dwa* h, const double pose[3], const double vel[3], const double* footprint_xy,
                                      int n_footprint, navgpu_dwa_result* result, double* best_points, int points_capacity);
/* the same split into enqueue and wait, for one host thread that drives several ranks' handles */
int navgpu_dwa_find_best_path_sharded_async(navgpu_dwa* h, const double pose[3], const double vel[3],
                                            const double* footprint_xy, int n_footprint);
int navgpu_dwa_sharded_collect(navgpu_dwa* h, const double pose[3], navgpu_dwa_result* result, double* best_points,
                               int points_capacity);
/* the four MapGrid distance fields after prepare(): which = 0 path, 1 goal, 2 goal_front, 3 alignment (fp64, host) */
int navgpu_dwa_get_grid(navgpu_dwa* h, int which, double* host_out);
/* enqueue one full scoring cycle without host synchronisation (timing) */
int navgpu_dwa_find_best_path_async(navgpu_dwa* h, const double pose[3], const double vel[3],
                                    const double* footprint_xy, int n_footprint);
int navgpu_dwa_synchronize(navgpu_dwa* h);
void* navgpu_dwa_stream(navgpu_dwa* h);

/* ---- Plan preprocessing of the local planners, batched (SURVEY.md 8f-4) ------------------------------------------
 * base_local_planner::transformGlobalPlan (base_local_planner/src/goal_functions.cpp:86-174) and prunePlan (:68-84) for
 * n_plans independent plans in one launch (one warp per plan).  Plans are concatenated: plan p owns poses
 * offsets[p] .. offsets[p + 1] - 1 of plan_xyz (x, y, z of pose.position, doubles).  tf's part stays with the caller
 * (tf is not in the reference tree): per plan the robot position expressed in the PLAN's frame (tf.transformPose,
 * :110-111) and plan_to_global_transform (:103-107) as a rigid transform.
 *   navgpu_plans_transform: first_out[p] = index of the first pose within dist_threshold[p] of the robot (the plan's
 *       size when there is none), count_out[p] = number of poses kept from there -- every pose up to and including the
 *       first one beyond the threshold, exactly the reference's two loops (:122-149); transformed_xyz[offsets[p] + k] =
 *       plan_to_global * (kept pose k).  The reference's dist_threshold is max(size_x, size_y) * resolution / 2 of the
 *       local costmap (:114-115).  Orientations are not transformed: the critics of this path read positions only.
 *   navgpu_plans_prune: erase_count_out[p] = number of way-points prunePlan erases from the front of plan p (and of
 *       the global plan): all before the first one closer than 1 m to the robot. */
typedef struct {
  double m[9]; /* rotation (tf::Matrix3x3 of the transform's basis), row-major */
  double t[3]; /* origin */
} navgpu_rigid_transform;
int navgpu_plans_transform(int n_plans, const int32_t* offsets, const double* plan_xyz, const double* robot_xy,
                           const navgpu_rigid_transform* plan_to_global, const double* dist_threshold,
                           int32_t* first_out, int32_t* count_out, double* transformed_xyz, int device);
int navgpu_plans_prune(int n_plans, const int32_t* offsets, const double* plan_xyz, const double* robot_xy,
                       int32_t* erase_count_out, int device);

/* ---- Fleet mode: N independent robots per control cycle (config C5) ------------------------------------------
 * Every robot has its own local costmap (raw obstacles in, inflated on the device exactly like a layered costmap
 * with a static-style layer + InflationLayer), plan, pose, velocity and oscillation state; one navgpu_fleet_step is
 * LayeredCostmap::updateMap + DWAPlanner::findBestPath for all of them in a handful of launches.  Robots are
 * independent, so a multi-GPU job gives each rank its own fleet with its share of the robots (no collective).  Every
 * fleet kind can plan with the legacy TrajectoryPlanner instead (navgpu_fleet_use_trajectory_planner, below). */
typedef struct navgpu_fleet navgpu_fleet;
int navgpu_fleet_create(navgpu_fleet** out, int n_robots, const navgpu_dwa_config* cfg, uint32_t size_x,
                        uint32_t size_y, double resolution, double inflation_radius, double cost_scaling_factor,
                        const double* footprint_xy, int n_footprint, int device);
int navgpu_fleet_destroy(navgpu_fleet* f);
/* raw (un-inflated) local maps [n][size_y][size_x] and their world origins [n][2], HOST memory */
int navgpu_fleet_set_maps(navgpu_fleet* f, const uint8_t* raw_maps, const double* origins_xy);  /* not on sensing fleets */
/* DWAPlanner::updatePlanAndLocalCosts for every robot: poses [n][3], concatenated plan points, offsets [n + 1] */
int navgpu_fleet_set_plans(navgpu_fleet* f, const double* poses, const double* plan_xy, const int32_t* plan_offsets);
int navgpu_fleet_reset_oscillation(navgpu_fleet* f);
/* one control cycle; poses, vels [n][3]; results: n entries (n_points = 0, winners' points are not materialised) */
int navgpu_fleet_step(navgpu_fleet* f, const double* poses, const double* vels, navgpu_dwa_result* results);
/* navgpu_fleet_step with device memory of the fleet's device: poses [n][3] and vels [n][3] (double) are read and
 * results [n] written on the fleet's stream (navgpu_fleet_stream); the call returns without waiting for the device.
 * After the stream has run, results, every costmap, layer, voxel column, window and origin, every oscillation mask and
 * distance grid, and all later behaviour are those of navgpu_fleet_step with the same poses and velocities.  One
 * exception by construction: a sensing fleet's footprint clearing takes cos / sin of each yaw from CUDA's sincos
 * instead of the host libm (as the scan projection does).  Robots navgpu_fleet_set_active left out keep their results
 * entry untouched; n_points is 0.  The caller orders its writes of poses and vels before the fleet's stream and reads
 * results after work ordered behind it.  Host and device steps, and every other call, may be mixed on one fleet: a
 * host call that reads the planner state (navgpu_fleet_step, _reset_oscillation, _get_oscillation_mask,
 * _check_trajectories, _get_geometry) first waits for the fleet's stream.  A device step that follows a device step,
 * with no set_plans, set_active, set_maps or reset_oscillation in between, neither waits for the host, allocates nor
 * copies from pageable memory, so it can be captured in a CUDA graph.  The scoring grid is sized from the
 * configuration: at most max(2, n) + 1 samples per axis configured with n.  Refused, with the fleet unchanged: null
 * or non-device pointers (NAVGPU_ERR_INVALID), TrajectoryPlanner fleets, use_dwa = 0 and more than 640 per-axis
 * samples by that bound (NAVGPU_ERR_UNSUPPORTED). */
int navgpu_fleet_step_device(navgpu_fleet* f, const double* poses, const double* vels, navgpu_dwa_result* results);
/* ---- Plan following on the device (DWAPlanner fleets of every kind) ---------------------------------------------
 * DWAPlannerROS runs, every control cycle before findBestPath: LocalPlannerUtil::getLocalPlan (transformGlobalPlan to
 * the stretch of the held global plan within max(size_x, size_y) * resolution / 2 of the robot; with prune_plan,
 * prunePlan erases the poses the robot has passed from that local plan and as many from the front of the held global
 * plan), returns without a command when the local plan is empty, else DWAPlanner::updatePlanAndLocalCosts.  The calls
 * below keep each robot's global plan on the device and run that per cycle for the whole fleet without a host wait.
 *
 * navgpu_fleet_set_global_plans: DWAPlannerROS::setPlan for robots[k], k < n_set: the (x, y) poses
 * plan_xy[offsets[k] .. offsets[k + 1]) (HOST memory, in the frame of the fleet's poses) become the robot's held global
 * plan, and its oscillation flags are reset (DWAPlanner::setPlan).  Other robots keep their plans and flags; empty plans
 * are accepted.  It may allocate and wait (a replan, <= 1 Hz); it sizes each robot's device slots so that later updates
 * never allocate.  Refused, with the fleet unchanged: a robot out of range or given twice, offsets that do not start at
 * 0 or that decrease, null pointers (NAVGPU_ERR_INVALID), TrajectoryPlanner fleets (NAVGPU_ERR_UNSUPPORTED). */
int navgpu_fleet_set_global_plans(navgpu_fleet* f, int n_set, const int32_t* robots, const double* plan_xy,
                                  const int32_t* offsets);
/* navgpu_fleet_update_plans_device: the per-cycle plan work above for EVERY robot, whatever navgpu_fleet_set_active
 * says (the wrappers update the plan at the goal too), with the identity transform, enqueued on the fleet's stream;
 * the call returns without waiting.  poses [n][3] (double) and status [n] (bytes, may be null) are device memory of the
 * fleet's device.  The kept poses go through the identity with navgpu_plans_transform's arithmetic (-0.0 becomes
 * +0.0, as tf's multiply does).  status[r] = 1: robot r has a local plan, and its MapGrid plans, alignment scale and
 * flags are those navgpu_fleet_set_plans would give it for that local plan and pose.  status[r] = 0: it has no global
 * plan or its local plan came out empty; its planner state is unchanged, and the following steps leave it out as
 * set_active would (results entry untouched, no wavefronts, no scoring) until an update gives it a local plan again
 * (navgpu_fleet_set_plans gives every robot one).  Exception by construction: the goal-front point takes atan2 / cos /
 * sin from CUDA, not the host libm (both within 2 ulp); everything else equals the host computation bit for bit.
 * An update followed by navgpu_fleet_step_device, repeated with no host call in between, neither waits for the host,
 * allocates nor copies from pageable memory, so the whole cycle can be captured in a CUDA graph.  Host calls may be
 * mixed in and see the plans the device computed: navgpu_fleet_step, _check_trajectories, _get_plan, _set_active,
 * _set_maps, _set_plans and _set_global_plans first wait for the fleet's stream; the update after them uploads the
 * plans again (waiting once).  navgpu_fleet_set_plans keeps its meaning: it sets every robot's local plan directly and
 * leaves the global plans alone; the next update replaces its result.  Refused, with the fleet unchanged: null or
 * non-device pointers (NAVGPU_ERR_INVALID), TrajectoryPlanner fleets (NAVGPU_ERR_UNSUPPORTED). */
int navgpu_fleet_update_plans_device(navgpu_fleet* f, const double* poses, int prune_plan, uint8_t* status);
/* robot's held global plan after the prunes (which = 0) or the local plan of the last update (which = 1, empty when it
 * had none), (x, y) doubles into HOST xy_out; *n_out = the number of poses; NAVGPU_ERR_CAPACITY when more than
 * capacity (the first capacity are written).  Waits for the fleet's stream first.  For tests and debugging. */
int navgpu_fleet_get_plan(navgpu_fleet* f, int robot, int which, double* xy_out, int capacity, int32_t* n_out);
/* inflated local costmap of one robot, HOST size_y x size_x */
int navgpu_fleet_get_costmap(navgpu_fleet* f, int robot, uint8_t* host_out);
int navgpu_fleet_get_oscillation_mask(navgpu_fleet* f, int robot, int* mask_out);
/* ---- Fleet mode with sensing: every robot runs move_base's local costmap itself --------------------------------
 * A second kind of fleet.  Every robot has a rolling size_x x size_y LayeredCostmap (rolling_window: true) with the
 * plugins [ObstacleLayer, InflationLayer], fed by the robot's own scans, followed by DWAPlanner.  navgpu_fleet_step then
 * runs, per robot, LayeredCostmap::updateMap(pose) (layered_costmap.cpp:79-150): the rolling origin, ObstacleLayer::
 * updateBounds (ray-trace clearing of every clearing source before any marking, then marking, then the footprint),
 * InflationLayer::updateBounds (its own last_* bounds per robot; the whole map on the first step), the cycle's window,
 * resetMap of the window, ObstacleLayer::updateCosts (footprint polygon to FREE_SPACE, then Overwrite or Max) and
 * InflationLayer::updateCosts with inflation mode 0 of navgpu_inflation_set_mode -- bit for bit what one
 * navgpu_costmap with an obstacle and an inflation layer computes -- and then DWAPlanner::findBestPath on the result.
 * Cells outside a robot's window keep their shifted previous values, as in the reference.  Every robot's maps start at
 * origin (0, 0) filled with the default value.  One CTA holds a robot's obstacle grid and master grid in shared
 * memory: maps, inflation radii and footprints beyond what fits it are refused with NAVGPU_ERR_UNSUPPORTED. */
typedef struct {
  double inflation_radius, cost_scaling_factor; /* InflationLayer (defaults 0.55, 10) */
  double max_obstacle_height;                   /* ObstacleLayer (default 2.0) */
  int32_t combination_method;                   /* 0 updateWithOverwrite, 1 updateWithMax (default) */
  int32_t footprint_clearing;                   /* default 1 */
  int32_t track_unknown;                        /* default value NO_INFORMATION (255) instead of FREE_SPACE (0) */
  int32_t pad_;
} navgpu_fleet_costmap_config;
int navgpu_fleet_create_sensing(navgpu_fleet** out, int n_robots, const navgpu_dwa_config* cfg, uint32_t size_x,
                                uint32_t size_y, double resolution, const navgpu_fleet_costmap_config* cm,
                                const double* footprint_xy, int n_footprint, int device);
/* Robot r's sources are scans[offsets[r] .. offsets[r + 1]) (navgpu_laser_scan records as navgpu_obstacle_set_scans
 * takes them: LaserScan ranges or is_cloud sensor-frame points).  They replace every robot's previous sources and
 * persist until the next call, like the observations of navgpu_obstacle_set_scans.  All robots' scans are projected in
 * one launch.  offsets: n_robots + 1 non-decreasing entries. */
int navgpu_fleet_set_scans(navgpu_fleet* f, const navgpu_laser_scan* scans, const int32_t* offsets);
/* Batched ingest for fleets whose robots all carry the same sensors: one source of every robot as dense arrays.  The
 * fields have navgpu_laser_scan's meaning; row r of data and of sensor_to_global belong to robot r. */
typedef struct {
  const float* data;              /* [n_robots][n_points] LaserScan ranges, or [n_robots][n_points][3] sensor-frame points (is_cloud) */
  const double* sensor_to_global; /* [n_robots][7]: translation x, y, z, then rotation x, y, z, w (tf order) */
  int32_t n_points;               /* per robot, >= 0 */
  int32_t is_cloud, inf_is_valid, marking, clearing;
  float angle_min, angle_increment, range_min, range_max;
  double min_obstacle_height, max_obstacle_height, obstacle_range, raytrace_range;
} navgpu_fleet_scan_source;
/* Equivalent to navgpu_fleet_set_scans with robot r's list [source 0, ..., source n_sources - 1], each entry built from
 * the source's shared fields, row r of data and row r of sensor_to_global: the same grids, columns, windows, origins
 * and planner results bit for bit.  The sources replace the previous ones and persist.  One kernel builds every
 * robot's observation records and projects every point; nothing per robot is built on the host.  n_sources = 0
 * empties every robot's list.  Sensing fleets of either kind, with either planner; NAVGPU_ERR_INVALID on a raw-map
 * fleet.  Refused, with the fleet's sources left as they were: a null handle or sources, n_sources < 0, a null
 * sensor_to_global, a null data with n_points > 0, n_points < 0 or is_cloud / marking / clearing outside {0, 1}
 * (NAVGPU_ERR_INVALID); more than 32 sources, or n_robots x the points of all sources beyond 2^31 - 1
 * (NAVGPU_ERR_UNSUPPORTED).
 * navgpu_fleet_set_scan_batch: the arrays are HOST memory, pageable or registered (navgpu_host_register); each is copied
 * to the device with its own copy, and the call returns once they were read.
 * navgpu_fleet_set_scan_batch_device: the arrays are device (or managed) memory of the fleet's device, anything else is
 * refused with NAVGPU_ERR_INVALID; the descriptors themselves are host memory.  The arrays are read in place on the
 * fleet's stream (navgpu_fleet_stream) and the call returns without waiting for it.  The caller orders its writes of
 * the arrays before that stream (for example cudaEventRecord on the writing stream, then cudaStreamWaitEvent on
 * navgpu_fleet_stream(f)), and must not change them until the fleet's stream has read them: the return of the next
 * navgpu_fleet_step / navgpu_fleet_step_tp is enough. */
int navgpu_fleet_set_scan_batch(navgpu_fleet* f, const navgpu_fleet_scan_source* sources, int n_sources);
int navgpu_fleet_set_scan_batch_device(navgpu_fleet* f, const navgpu_fleet_scan_source* sources, int n_sources);
/* the CUDA stream every kernel of this fleet runs on (cudaStream_t), like navgpu_costmap_stream / navgpu_dwa_stream */
void* navgpu_fleet_stream(navgpu_fleet* f);
/* per robot, after the last navgpu_fleet_step: the ObstacleLayer's own grid (HOST size_y x size_x) */
int navgpu_fleet_get_layer(navgpu_fleet* f, int robot, uint8_t* host_out);
/* per robot, after the last navgpu_fleet_step: the rolled origin and the cycle's window {x0, xn, y0, yn} */
int navgpu_fleet_get_geometry(navgpu_fleet* f, int robot, double origin_out[2], int32_t window_out[4]);
/* device time (ms, CUDA events) of the last scan projection (navgpu_fleet_set_scans; 0 when it had no points) and of the
 * last costmap update of all robots (navgpu_fleet_step); synchronises the fleet's stream */
int navgpu_fleet_last_timing(navgpu_fleet* f, float* project_ms, float* costmap_ms);
/* ---- Sensing fleet with a VoxelLayer (map_type: voxel) -----------------------------------------------------------
 * A third kind of fleet: every robot's rolling local costmap is [VoxelLayer, InflationLayer], the VoxelLayer of
 * navgpu_costmap_add_voxel_layer (3-D ray-trace clearing on columns of up to 16 voxels, so a ray that passes over a low
 * obstacle does not clear it; marking; the columns move with the rolling origin).  cm keeps its meaning
 * (max_obstacle_height, combination_method, footprint_clearing, track_unknown and the inflation parameters); voxel
 * gives the VoxelLayer's own parameters, checked like navgpu_costmap_add_voxel_layer's (same error codes; mark_threshold
 * must be 0).  Every robot's columns start unknown, as VoxelGrid does.  set_scans, set_plans, step, get_costmap,
 * get_geometry and last_timing work as on a sensing fleet; navgpu_fleet_get_layer returns the VoxelLayer's 2-D grid.
 * One CTA holds a robot's grids and its columns (4 B per cell) in shared memory: larger maps are refused with
 * NAVGPU_ERR_UNSUPPORTED (on a B200 with the default inflation at 0.05 m, up to about 188 x 188 cells). */
typedef struct {
  double origin_z, z_resolution; /* VoxelLayer (defaults 0.0, 0.2) */
  int32_t z_voxels;              /* defaults 10; same range as navgpu_costmap_add_voxel_layer */
  int32_t unknown_threshold;     /* default 15 (VoxelPlugin.cfg), before reconfigureCB's + (16 - z_voxels) */
  int32_t mark_threshold;        /* default 0 */
  int32_t pad_;
} navgpu_fleet_voxel_config;
int navgpu_fleet_create_sensing_voxel(navgpu_fleet** out, int n_robots, const navgpu_dwa_config* cfg, uint32_t size_x,
                                      uint32_t size_y, double resolution, const navgpu_fleet_costmap_config* cm,
                                      const navgpu_fleet_voxel_config* voxel, const double* footprint_xy,
                                      int n_footprint, int device);
/* per robot, after the last navgpu_fleet_step: the VoxelLayer's columns (HOST size_y x size_x uint32, the layout of
 * navgpu_layer_get_voxels); NAVGPU_ERR_INVALID on fleets without a VoxelLayer */
int navgpu_fleet_get_voxels(navgpu_fleet* f, int robot, uint32_t* host_out);


/* ---- legacy base_local_planner::TrajectoryPlanner (SURVEY.md 8f-4) ---------------------------------------------
 * The rollout planner behind TrajectoryPlannerROS (base_local_planner/src/trajectory_planner.cpp): the two MapGrid
 * wavefronts (path_map_, goal_map_) and generateTrajectory for every velocity sample of createTrajectories run on
 * the device; the sequential selection among the scored samples (in-place rotation / strafing / escape rules and
 * their oscillation flags, :560-905) is scalar bookkeeping and stays on the host.  Replaces
 * base_local_planner::TrajectoryPlanner::{updatePlan, findBestPath, scoreTrajectory, checkTrajectory}
 * (include/base_local_planner/trajectory_planner.h:116-212). */
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
  int32_t allow_unknown;
} navgpu_tp_config;

typedef struct {
  double cost, xv, yv, thetav; /* the returned Trajectory's cost_, xv_, yv_, thetav_ */
  int32_t n_points;
  /* bit0 stuck_left, 1 stuck_right, 2 stuck_left_strafe, 3 stuck_right_strafe, 4 rotating_left, 5 rotating_right,
   * 6 strafe_left, 7 strafe_right, 8 escaping_ (trajectory_planner.h:283-288) */
  int32_t flags;
} navgpu_tp_result;

typedef struct navgpu_tp navgpu_tp;

/* TrajectoryPlannerROS::initialize's defaults (trajectory_planner_ros.cpp:116-213) */
void navgpu_tp_default_config(navgpu_tp_config* cfg);
/* TrajectoryPlanner ctor (trajectory_planner.cpp:135-187) */
int navgpu_tp_create(navgpu_tp** out, const navgpu_tp_config* cfg, uint32_t size_x, uint32_t size_y, double resolution,
                     const double* footprint_xy, int n_footprint, int device);
int navgpu_tp_destroy(navgpu_tp* h);
/* TrajectoryPlanner::reconfigure (trajectory_planner.cpp:59-133); the oscillation / escape state is kept.  Validated
 * as navgpu_tp_create validates (a refused configuration leaves the handle unchanged); trajectories may grow longer
 * than at creation, and findBestPath still returns all of their points. */
int navgpu_tp_reconfigure(navgpu_tp* h, const navgpu_tp_config* cfg);
/* TrajectoryPlanner::setFootprint (trajectory_planner.h:195) */
int navgpu_tp_set_footprint(navgpu_tp* h, const double* footprint_xy, int n_footprint);
int navgpu_tp_set_costmap(navgpu_tp* h, const uint8_t* host_grid, double origin_x, double origin_y);
int navgpu_tp_set_costmap_device(navgpu_tp* h, const uint8_t* dev_grid, uint32_t pitch, double origin_x,
                                 double origin_y);
/* TrajectoryPlanner::updatePlan(new_plan, compute_dists = false), trajectory_planner.cpp:477-502 */
int navgpu_tp_update_plan(navgpu_tp* h, const double* plan_xy, int n);
/* TrajectoryPlanner::findBestPath (:908-980): footprint cells -> within_robot, both wavefronts, every sample of
 * createTrajectories scored, the reference's selection; points (nullable): 3 * points_capacity doubles */
int navgpu_tp_find_best_path(navgpu_tp* h, const double pose[3], const double vel[3], navgpu_tp_result* result,
                             double* points, int points_capacity);
/* TrajectoryPlanner::scoreTrajectory (:520-535; checkTrajectory is `cost >= 0`) on the maps of the last findBestPath */
int navgpu_tp_score_trajectory(navgpu_tp* h, const double pose[3], const double vel[3], const double vel_samples[3],
                               double* cost_out);
/* path_map_ (which = 0) / goal_map_ (1) target_dist after the last findBestPath, fp64, host */
int navgpu_tp_get_grid(navgpu_tp* h, int which, double* host_out);
/* number of velocity samples the last findBestPath scored on the device */
int navgpu_tp_last_sample_count(navgpu_tp* h, int* n_out);

/* ---- Fleets of legacy TrajectoryPlanners (TrajectoryPlannerROS, move_base's default base_local_planner) ---------
 * Any of the three fleet kinds can run base_local_planner::TrajectoryPlanner instead of DWAPlanner.  Its costmap side is
 * unchanged (set_maps / set_scans, get_costmap, get_layer, get_voxels, get_geometry and last_timing work as before).
 * navgpu_fleet_set_plans is then TrajectoryPlanner::updatePlan per robot (final goal, resolution-adjusted plan; empty
 * plans are accepted, as navgpu_tp_update_plan accepts them; the poses argument is not used), and each robot keeps its
 * own oscillation / escape state.  Per step, every robot's footprint cells, both wavefronts (path_map_, goal_map_) and
 * every robot's velocity samples run in one launch each; the samples are enumerated and the reference's selection is
 * made on the host, per robot, as navgpu_tp_find_best_path does.  One config for the whole fleet; the footprint is the
 * fleet's.  navgpu_fleet_step, navgpu_fleet_reset_oscillation and navgpu_fleet_get_oscillation_mask return
 * NAVGPU_ERR_INVALID on such a fleet, the calls below NAVGPU_ERR_INVALID on a DWA fleet. */
/* Makes f's planner base_local_planner::TrajectoryPlanner (trajectory_planner.cpp, TrajectoryPlannerROS's planner)
 * instead of DWAPlanner; cfg as for navgpu_tp_create (refused with its codes).  Any fleet kind; only between creation
 * and the first set_plans / step (NAVGPU_ERR_INVALID otherwise, and for a second call).  Footprints whose filled cells
 * could exceed the per-robot buffer (12000 cells, bounded from the circumscribed radius and the edge lengths) are
 * refused with NAVGPU_ERR_UNSUPPORTED. */
int navgpu_fleet_use_trajectory_planner(navgpu_fleet* f, const navgpu_tp_config* cfg);
/* one control cycle: every robot's costmap update (as navgpu_fleet_step), then TrajectoryPlanner::findBestPath per
 * robot; poses, vels [n][3]; results[r] as navgpu_tp_find_best_path returns it (points are not materialised, n_points
 * is their count) */
int navgpu_fleet_step_tp(navgpu_fleet* f, const double* poses, const double* vels, navgpu_tp_result* results);
/* navgpu_fleet_step_tp with device memory of the fleet's device, for any fleet kind: poses [n][3] and vels [n][3]
 * (double) are read and results [n] written on the fleet's stream (navgpu_fleet_stream); the call returns without
 * waiting for the device.  Per robot, the rounding through float, the samples of createTrajectories and the selection
 * with its oscillation / escape state run on the device too.  After the stream has run, results (n_points: the chosen
 * trajectory's point count), every costmap, layer, voxel column, window and origin, both distance grids of every robot
 * and all later behaviour are those of navgpu_fleet_step_tp with the same poses and velocities.  One exception by
 * construction: cos / sin of each robot's yaw (its footprint cells, a sensing fleet's footprint clearing) come from
 * CUDA's sincos instead of the host libm.  hypot is computed as glibc 2.35+ computes it (which is not correctly
 * rounded); where the process's libm hypot gives other bits on a fixed list of pairs, checked once per process, the
 * call is refused.  Robots navgpu_fleet_set_active left out keep their results entry untouched.  The caller orders its
 * writes of poses and vels before the fleet's stream and reads results after work ordered behind it.  Host and device
 * steps, and every other call, may be mixed on one fleet: a host call that reads or changes the planner state
 * (navgpu_fleet_step_tp, _set_plans, _check_trajectories, _get_geometry) first waits for the fleet's stream.  A device
 * step that follows a device step, with no set_plans, set_active or set_maps in between, neither waits for the host,
 * allocates nor copies from pageable memory, so it can be captured in a CUDA graph.  Each robot's samples sit in a slot
 * sized from the configuration: vx_samples * vtheta_samples + vtheta_samples + 1, plus 2 + n_y_vels when holonomic (87
 * with TrajectoryPlannerROS's defaults).  Refused, with the fleet unchanged: null or non-device pointers and fleets
 * that are not TrajectoryPlanner fleets (NAVGPU_ERR_INVALID), slots of more than 4096 samples and a libm whose hypot
 * differs (NAVGPU_ERR_UNSUPPORTED). */
int navgpu_fleet_step_tp_device(navgpu_fleet* f, const double* poses, const double* vels, navgpu_tp_result* results);
/* path_map_ (which = 0) / goal_map_ (1) of robot after the last step, fp64 HOST size_y x size_x (as navgpu_tp_get_grid) */
int navgpu_fleet_tp_get_grid(navgpu_fleet* f, int robot, int which, double* host_out);
/* device time (ms, CUDA events) of the last host step's (navgpu_fleet_step_tp) footprint-cell, wavefront and scoring
 * launches (0 before the first one); synchronises the fleet's stream.  Device steps (navgpu_fleet_step_tp_device)
 * record no events and leave these times as they were: time them with events of your own on navgpu_fleet_stream. */
int navgpu_fleet_tp_last_timing(navgpu_fleet* f, float* footprint_ms, float* wavefront_ms, float* score_ms);

/* ---- Goal handling for fleets: robots that stop and rotate ----------------------------------------------------
 * At the goal, DWAPlannerROS and TrajectoryPlannerROS stop searching: LatchedStopRotateController / rotateToGoal
 * propose one stop or rotate command and accept it if checkTrajectory scores it >= 0.  The two calls below let a
 * fleet do the same per robot; the goal tolerance and latch logic stay with the caller, as for single handles.
 * Both work on every fleet kind, with either planner. */
/* Which robots the following steps plan for: active[n_robots] bytes, 0 or 1; null means every robot.  The mask persists
 * until the next call; a new fleet starts with every robot active.  A robot with active[r] == 0 still gets its costmap
 * update in navgpu_fleet_step / navgpu_fleet_step_tp, but nothing of its planner runs: no MapGrid wavefronts (its
 * distance grids stay as its last planning step left them), no sample enumeration or scoring, no footprint cells
 * (TrajectoryPlanner), no change to its oscillation, result or escape state, and results[r] is not written.
 * navgpu_fleet_set_plans still applies every robot's plan.  NAVGPU_ERR_INVALID for any byte other than 0 or 1, and the
 * previous mask stays. */
int navgpu_fleet_set_active(navgpu_fleet* f, const uint8_t* active);
/* checkTrajectory of each robot's candidate commands: robot r's are vel_samples[offsets[r] .. offsets[r + 1]), 3 doubles
 * (vx, vy, vtheta) each; offsets has n_robots + 1 non-decreasing entries starting at 0; poses, vels [n][3]; costs_out
 * gets one cost per candidate (>= 0: legal).
 * DWAPlanner fleets: what navgpu_dwa_check_trajectory returns on a handle holding the robot's current costmap and
 * origin, its plans of the last set_plans (alignment scale included), the distance grids of its last planning step and
 * the fleet's footprint; a robot with candidates has its oscillation flags reset (dwa_planner.cpp:217), so the call
 * equals that handle's check of each candidate in order.
 * TrajectoryPlanner fleets: what navgpu_tp_score_trajectory returns (pose and velocity as given, not rounded through
 * float); no state changes.
 * Robots without candidates are untouched.  NAVGPU_ERR_INVALID, with no state changed, for null pointers, offsets that
 * decrease or do not start at 0, and candidates for a robot that was never active in a step.  One kernel launch
 * whatever the robots and candidates; returns once the costs are in costs_out. */
int navgpu_fleet_check_trajectories(navgpu_fleet* f, const double* poses, const double* vels, const int32_t* offsets,
                                    const double* vel_samples, double* costs_out);

#ifdef __cplusplus
}
#endif
#endif
