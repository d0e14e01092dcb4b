// fleet_costmap.cuh -- the per-robot rolling local costmaps of a sensing fleet (navgpu_fleet_create_sensing), as the
// planner side of the fleet (dwa.cu) sees them.  Implemented next to the single costmap in costmap.cu, whose kernels
// and host arithmetic they share.
#pragma once

#include "common.cuh"

namespace navgpu {

struct FleetCostmap;

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
// the device part of that updateMap for every robot (one launch), on the fleet's stream
int fleet_costmap_enqueue(FleetCostmap* fc);
int fleet_costmap_get(FleetCostmap* fc, int robot, bool master, uint8_t* host_out);
// a voxel fleet's columns of one robot (NAVGPU_ERR_INVALID on a 2-D one)
int fleet_costmap_get_voxels(FleetCostmap* fc, int robot, uint32_t* host_out);
int fleet_costmap_geometry(FleetCostmap* fc, int robot, double origin_out[2], int32_t window_out[4]);
int fleet_costmap_last_timing(FleetCostmap* fc, float* project_ms, float* costmap_ms);

}  // namespace navgpu
