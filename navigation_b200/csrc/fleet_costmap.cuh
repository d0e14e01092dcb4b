// fleet_costmap.cuh -- the per-robot rolling local costmaps of a sensing fleet (navgpu_fleet_create_sensing), as the
// planner side of the fleet (dwa.cu) sees them.  Implemented next to the single costmap in costmap.cu, whose kernels
// and host arithmetic they share.
#pragma once

#include <cmath>

#include "common.cuh"

namespace navgpu {

struct FleetCostmap;

// one robot's scalars of one step: Costmap2D::updateOrigin (the new origin and the cell shift that got there) and the
// pose transformFootprint needs
struct FleetCmStep {
  double ox, oy;
  double rx, ry, cos_th, sin_th;
  int cell_dx, cell_dy;
};

// LayeredCostmap::updateMap's rolling origin (:86-91) and Costmap2D::updateOrigin's scalars, as roll_grid computes
// them, for a robot at pose whose grids are at (ox, oy); master and obstacle layer move together, so one origin serves
// both.  The host step (fleet_costmap_roll) and the device step (k_fleet_prepare) share it.  Everything but the
// footprint's cos / sin of the yaw is exact IEEE arithmetic; those come from the host libm on the host and from CUDA's
// sincos on the device, like the sincos of k_project_scans: the one input of a device step that is not the host
// step's by construction.
__host__ __device__ inline FleetCmStep fleet_roll_step(const double pose[3], double ox, double oy, unsigned sx,
                                                       unsigned sy, double res) {
  const double size_m_x = (sx - 1 + 0.5) * res, size_m_y = (sy - 1 + 0.5) * res;
  const double rx = pose[0], ry = pose[1], ryaw = pose[2];
  const double new_ox = rx - size_m_x / 2, new_oy = ry - size_m_y / 2;
  const int cell_ox = int((new_ox - ox) / res), cell_oy = int((new_oy - oy) / res);
  double s, c;
#ifdef __CUDA_ARCH__
  sincos(ryaw, &s, &c);
#else
  c = cos(ryaw);
  s = sin(ryaw);
#endif
  return FleetCmStep{ox + cell_ox * res, oy + cell_oy * res, rx, ry, c, s, cell_ox, cell_oy};
}

// n robots, each a rolling sx x sy LayeredCostmap [ObstacleLayer, InflationLayer] (voxel null) or [VoxelLayer,
// InflationLayer] with its origin at (0, 0); owns the CUDA stream the fleet runs on
int fleet_costmap_create(FleetCostmap** out, int n, unsigned sx, unsigned sy, double resolution,
                         const navgpu_fleet_costmap_config& cm, const navgpu_fleet_voxel_config* voxel,
                         const double* footprint_xy, int n_footprint, int device);
void fleet_costmap_destroy(FleetCostmap* fc);
cudaStream_t fleet_costmap_stream(const FleetCostmap* fc);
// the robots' master grids: robot r's is sy rows of `pitch` bytes at master + r * sy * pitch
const uint8_t* fleet_costmap_master(const FleetCostmap* fc, unsigned* pitch);
int fleet_costmap_set_scans(FleetCostmap* fc, const navgpu_laser_scan* scans, const int32_t* offsets);
// navgpu_fleet_set_scan_batch (device false: host arrays, staged and waited for) and _device (device true)
int fleet_costmap_set_scan_batch(FleetCostmap* fc, const navgpu_fleet_scan_source* sources, int n_sources, bool device);
// host part of one updateMap for every robot: the rolled origins (Costmap2D::updateOrigin's scalars) into origins_xy
// [n][2]; must be followed by fleet_costmap_enqueue before the next roll
int fleet_costmap_roll(FleetCostmap* fc, const double* poses, double* origins_xy);
// a device step's roll: the array of n step records the device writes (fleet_roll_step per robot, on the fleet's
// stream) in place of fleet_costmap_roll; fleet_costmap_enqueue(fc, true) then launches the update on them
FleetCmStep* fleet_costmap_device_steps(FleetCostmap* fc);
// the device part of that updateMap for every robot (one launch), on the fleet's stream; device_steps: the step
// records were written on the device, the host's origins stay as they are until fleet_costmap_set_origins
int fleet_costmap_enqueue(FleetCostmap* fc, bool device_steps = false);
// the origins [n][2] the grids on the device follow, after device steps rolled them
void fleet_costmap_set_origins(FleetCostmap* fc, const double* origins_xy);
// device or managed memory of `device`
bool on_device(const void* p, int device);
int fleet_costmap_get(FleetCostmap* fc, int robot, bool master, uint8_t* host_out);
// a voxel fleet's columns of one robot (NAVGPU_ERR_INVALID on a 2-D one)
int fleet_costmap_get_voxels(FleetCostmap* fc, int robot, uint32_t* host_out);
int fleet_costmap_geometry(FleetCostmap* fc, int robot, double origin_out[2], int32_t window_out[4]);
int fleet_costmap_last_timing(FleetCostmap* fc, float* project_ms, float* costmap_ms);

}  // namespace navgpu
