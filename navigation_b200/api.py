"""ctypes binding of include/navgpu.h (libnavgpu.so).

Shaped like the checker binding (same method names) so parity tests drive both through the same scenario code, but
this module never imports or loads anything from oracle/.
"""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libnavgpu.so")

TRUE_OVERWRITE, OVERWRITE, MAX, ADDITION, NOTHING = 0, 1, 2, 3, 4


class NavGpuError(RuntimeError):
    pass


class Observation(C.Structure):
    _fields_ = [("origin_x", C.c_double), ("origin_y", C.c_double), ("origin_z", C.c_double),
                ("obstacle_range", C.c_double), ("raytrace_range", C.c_double),
                ("xyz", C.POINTER(C.c_float)), ("n_points", C.c_int32), ("marking", C.c_int32),
                ("clearing", C.c_int32), ("pad_", C.c_int32)]


class DwaConfig(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        "max_trans_vel", "min_trans_vel", "max_vel_x", "min_vel_x", "max_vel_y", "min_vel_y", "max_rot_vel",
        "min_rot_vel", "acc_lim_x", "acc_lim_y", "acc_lim_theta", "sim_time", "sim_granularity",
        "angular_sim_granularity", "sim_period", "path_distance_bias", "goal_distance_bias", "occdist_scale",
        "forward_point_distance", "cheat_factor", "oscillation_reset_dist", "oscillation_reset_angle",
        "scaling_speed", "max_scaling_factor")] + [(n, C.c_int32) for n in (
            "vx_samples", "vy_samples", "vth_samples", "use_dwa", "sum_scores", "allow_unknown")]


class DwaResult(C.Structure):
    _fields_ = [("cost", C.c_double), ("xv", C.c_double), ("yv", C.c_double), ("thetav", C.c_double),
                ("best_index", C.c_int32), ("n_samples", C.c_int32), ("n_scored", C.c_int32),
                ("n_points", C.c_int32)]


class LaserScan(C.Structure):
    """navgpu_laser_scan"""
    _fields_ = [("ranges", C.POINTER(C.c_float)), ("n_ranges", C.c_int32), ("inf_is_valid", C.c_int32),
                ("angle_min", C.c_float), ("angle_increment", C.c_float), ("range_min", C.c_float),
                ("range_max", C.c_float), ("translation", C.c_double * 3), ("rotation_xyzw", C.c_double * 4),
                ("min_obstacle_height", C.c_double), ("max_obstacle_height", C.c_double),
                ("obstacle_range", C.c_double), ("raytrace_range", C.c_double), ("marking", C.c_int32),
                ("clearing", C.c_int32), ("is_cloud", C.c_int32), ("pad_", C.c_int32)]


class FleetScanSource(C.Structure):
    """navgpu_fleet_scan_source: one sensor of every robot of a sensing fleet, as dense arrays"""
    _fields_ = [("data", C.c_void_p), ("sensor_to_global", C.c_void_p), ("n_points", C.c_int32),
                ("is_cloud", C.c_int32), ("inf_is_valid", C.c_int32), ("marking", C.c_int32), ("clearing", C.c_int32),
                ("angle_min", C.c_float), ("angle_increment", C.c_float), ("range_min", C.c_float),
                ("range_max", C.c_float), ("min_obstacle_height", C.c_double), ("max_obstacle_height", C.c_double),
                ("obstacle_range", C.c_double), ("raytrace_range", C.c_double)]


class FleetCostmapConfig(C.Structure):
    """navgpu_fleet_costmap_config"""
    _fields_ = [("inflation_radius", C.c_double), ("cost_scaling_factor", C.c_double),
                ("max_obstacle_height", C.c_double), ("combination_method", C.c_int32),
                ("footprint_clearing", C.c_int32), ("track_unknown", C.c_int32), ("pad_", C.c_int32)]


class FleetVoxelConfig(C.Structure):
    """navgpu_fleet_voxel_config (the VoxelLayer of navgpu_fleet_create_sensing_voxel)"""
    _fields_ = [("origin_z", C.c_double), ("z_resolution", C.c_double), ("z_voxels", C.c_int32),
                ("unknown_threshold", C.c_int32), ("mark_threshold", C.c_int32), ("pad_", C.c_int32)]


# cfg/VoxelPlugin.cfg
VOXEL_DEFAULTS = dict(origin_z=0.0, z_resolution=0.2, z_voxels=10, unknown_threshold=15, mark_threshold=0)


class TpConfig(C.Structure):
    """navgpu_tp_config: the legacy base_local_planner::TrajectoryPlanner's parameters."""
    _fields_ = [(n, C.c_double) for n in (
        "acc_lim_x", "acc_lim_y", "acc_lim_theta", "sim_time", "sim_granularity", "angular_sim_granularity",
        "sim_period", "pdist_scale", "gdist_scale", "occdist_scale", "heading_lookahead", "oscillation_reset_dist",
        "escape_reset_dist", "escape_reset_theta", "max_vel_x", "min_vel_x", "max_vel_th", "min_vel_th",
        "min_in_place_vel_th", "backup_vel", "heading_scoring_timestep", "stop_time_buffer")] + [
            ("y_vels", C.c_double * 8)] + [(n, C.c_int32) for n in (
                "n_y_vels", "vx_samples", "vtheta_samples", "holonomic_robot", "dwa", "heading_scoring",
                "simple_attractor", "allow_unknown")]


class TpResult(C.Structure):
    _fields_ = [("cost", C.c_double), ("xv", C.c_double), ("yv", C.c_double), ("thetav", C.c_double),
                ("n_points", C.c_int32), ("flags", C.c_int32)]


_u8p = C.POINTER(C.c_uint8)
_i8p = C.POINTER(C.c_int8)
_f64p = C.POINTER(C.c_double)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_vpp = C.POINTER(C.c_void_p)


def _p(a, t):
    return a.ctypes.data_as(t)


# name -> (restype, argtypes); every symbol include/navgpu.h declares
SIGNATURES = {
    "navgpu_last_error": (C.c_char_p, []),
    "navgpu_device_count": (C.c_int, []),
    "navgpu_launch_count": (C.c_uint64, []),
    "navgpu_costmap_create": (C.c_int, [_vpp, C.c_uint32, C.c_uint32, C.c_double, C.c_double, C.c_double, C.c_int,
                                        C.c_int, C.c_int]),
    "navgpu_costmap_destroy": (C.c_int, [C.c_void_p]),
    "navgpu_costmap_add_grid_layer": (C.c_int, [C.c_void_p, C.c_int, _i32p]),
    "navgpu_costmap_add_obstacle_layer": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_double, _i32p]),
    "navgpu_costmap_add_inflation_layer": (C.c_int, [C.c_void_p, C.c_double, C.c_double, _i32p]),
    "navgpu_costmap_add_voxel_layer": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int,
                                                 C.c_int, C.c_int, _i32p]),
    "navgpu_layer_get_voxels": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_uint32)]),
    "navgpu_costmap_set_footprint": (C.c_int, [C.c_void_p, _f64p, C.c_int]),
    "navgpu_grid_layer_set": (C.c_int, [C.c_void_p, C.c_int, _u8p]),
    "navgpu_grid_layer_set_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_uint32]),
    "navgpu_grid_layer_set_occupancy": (C.c_int, [C.c_void_p, C.c_int, _i8p, C.c_int, C.c_uint8, C.c_uint8, C.c_int]),
    "navgpu_grid_layer_touch": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]),
    "navgpu_layer_set_enabled": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "navgpu_obstacle_set_observations": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(Observation), C.c_int]),
    "navgpu_obstacle_set_scans": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(LaserScan), C.c_int]),
    "navgpu_obstacle_get_cloud": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float), C.c_int, _i32p]),
    "navgpu_inflation_set_params": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_double]),
    "navgpu_inflation_set_mode": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "navgpu_inflation_last_rounds": (C.c_int, [C.c_void_p, _i32p]),
    "navgpu_costmap_update_map": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_double, _i32p]),
    "navgpu_costmap_update_map_async": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_double]),
    "navgpu_costmap_synchronize": (C.c_int, [C.c_void_p]),
    "navgpu_costmap_stream": (C.c_void_p, [C.c_void_p]),
    "navgpu_costmap_set_profiling": (C.c_int, [C.c_void_p, C.c_int]),
    "navgpu_costmap_force_generic_sweep": (C.c_int, [C.c_void_p, C.c_int]),
    "navgpu_costmap_last_timing": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "navgpu_costmap_last_timing_split": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "navgpu_costmap_get": (C.c_int, [C.c_void_p, _u8p]),
    "navgpu_costmap_get_window": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, _u8p]),
    "navgpu_costmap_get_window_into": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, _u8p, C.c_uint32]),
    "navgpu_costmap_get_changed": (C.c_int, [C.c_void_p, _u8p, C.c_uint32, _i32p, C.c_int, C.POINTER(C.c_int32),
                                             C.POINTER(C.c_uint64)]),
    "navgpu_costmap_mirror_invalidate": (C.c_int, [C.c_void_p]),
    "navgpu_costmap_last_window": (C.c_int, [C.c_void_p, _i32p]),
    "navgpu_host_register": (C.c_int, [C.c_void_p, C.c_size_t]),
    "navgpu_host_unregister": (C.c_int, [C.c_void_p]),
    "navgpu_costmap_get_window_occupancy": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, _i8p]),
    "navgpu_costmap_set": (C.c_int, [C.c_void_p, _u8p]),
    "navgpu_layer_get": (C.c_int, [C.c_void_p, C.c_int, _u8p]),
    "navgpu_costmap_get_origin": (C.c_int, [C.c_void_p, _f64p]),
    "navgpu_costmap_device_grid": (C.c_int, [C.c_void_p, _vpp, C.POINTER(C.c_uint32)]),
    "navgpu_inflation_tables": (C.c_int, [C.c_void_p, C.c_int, _u8p, _f64p, C.c_int, _i32p]),
    "navgpu_inflate_host": (C.c_int, [_u8p, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int, _u8p,
                                      C.c_uint32, C.c_int]),
    "navgpu_merge_host": (C.c_int, [_u8p, _u8p, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.c_int]),
    "navgpu_build_cost_table": (C.c_int, [C.c_double, C.c_double, C.c_double, C.c_double, _u8p, _f64p, C.c_int, _i32p]),
    "navgpu_dwa_default_config": (None, [C.POINTER(DwaConfig)]),
    "navgpu_dwa_create": (C.c_int, [_vpp, C.POINTER(DwaConfig), C.c_uint32, C.c_uint32, C.c_double, C.c_int]),
    "navgpu_dwa_destroy": (C.c_int, [C.c_void_p]),
    "navgpu_dwa_reconfigure": (C.c_int, [C.c_void_p, C.POINTER(DwaConfig)]),
    "navgpu_dwa_set_costmap": (C.c_int, [C.c_void_p, _u8p, C.c_double, C.c_double]),
    "navgpu_dwa_set_costmap_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_double, C.c_double]),
    "navgpu_dwa_set_plan": (C.c_int, [C.c_void_p, _f64p, _f64p, C.c_int]),
    "navgpu_dwa_reset_oscillation": (C.c_int, [C.c_void_p]),
    "navgpu_dwa_get_oscillation_mask": (C.c_int, [C.c_void_p, _i32p]),
    "navgpu_dwa_find_best_path": (C.c_int, [C.c_void_p, _f64p, _f64p, _f64p, C.c_int, C.POINTER(DwaResult), _f64p,
                                            C.c_int, _f64p, C.c_int]),
    "navgpu_dwa_check_trajectory": (C.c_int, [C.c_void_p, _f64p, _f64p, _f64p, _f64p, C.c_int, _f64p]),
    "navgpu_dwa_score_range": (C.c_int, [C.c_void_p, _f64p, _f64p, _f64p, C.c_int, C.c_int64, C.c_int64, _f64p, _i64p,
                                         _i64p]),
    "navgpu_dwa_finish_sharded": (C.c_int, [C.c_void_p, _f64p, _f64p, _i64p, C.c_int, C.POINTER(DwaResult), _f64p,
                                            C.c_int]),
    "navgpu_plans_transform": (C.c_int, [C.c_int, _i32p, _f64p, _f64p, C.c_void_p, _f64p, _i32p, _i32p, _f64p, C.c_int]),
    "navgpu_plans_prune": (C.c_int, [C.c_int, _i32p, _f64p, _f64p, _i32p, C.c_int]),
    "navgpu_dwa_prepare": (C.c_int, [C.c_void_p]),
    "navgpu_dwa_score_trajectories": (C.c_int, [C.c_void_p, C.c_int, _i32p, _f64p, _f64p, _f64p, C.c_int, _f64p, _f64p]),
    "navgpu_dwa_update_oscillation": (C.c_int, [C.c_void_p, _f64p, C.c_double, C.c_double, C.c_double, C.c_double]),
    "navgpu_dwa_get_samples": (C.c_int, [C.c_void_p, _i32p, C.POINTER(C.c_float), C.c_int]),
    "navgpu_dwa_score_strided": (C.c_int, [C.c_void_p, _f64p, _f64p, _f64p, C.c_int, C.c_int, C.c_int,
                                           C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "navgpu_dwa_shard_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "navgpu_dwa_shard_connect": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "navgpu_dwa_shard_connect_local": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "navgpu_dwa_find_best_path_sharded": (C.c_int, [C.c_void_p, _f64p, _f64p, _f64p, C.c_int, C.POINTER(DwaResult),
                                                    _f64p, C.c_int]),
    "navgpu_dwa_find_best_path_sharded_async": (C.c_int, [C.c_void_p, _f64p, _f64p, _f64p, C.c_int]),
    "navgpu_dwa_sharded_collect": (C.c_int, [C.c_void_p, _f64p, C.POINTER(DwaResult), _f64p, C.c_int]),
    "navgpu_dwa_get_grid": (C.c_int, [C.c_void_p, C.c_int, _f64p]),
    "navgpu_dwa_find_best_path_async": (C.c_int, [C.c_void_p, _f64p, _f64p, _f64p, C.c_int]),
    "navgpu_dwa_synchronize": (C.c_int, [C.c_void_p]),
    "navgpu_dwa_stream": (C.c_void_p, [C.c_void_p]),
    "navgpu_fleet_create": (C.c_int, [_vpp, C.c_int, C.POINTER(DwaConfig), C.c_uint32, C.c_uint32, C.c_double, C.c_double,
                                      C.c_double, _f64p, C.c_int, C.c_int]),
    "navgpu_fleet_destroy": (C.c_int, [C.c_void_p]),
    "navgpu_fleet_set_maps": (C.c_int, [C.c_void_p, _u8p, _f64p]),
    "navgpu_fleet_set_plans": (C.c_int, [C.c_void_p, _f64p, _f64p, _i32p]),
    "navgpu_fleet_reset_oscillation": (C.c_int, [C.c_void_p]),
    "navgpu_fleet_step": (C.c_int, [C.c_void_p, _f64p, _f64p, C.POINTER(DwaResult)]),
    "navgpu_fleet_step_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "navgpu_fleet_get_costmap": (C.c_int, [C.c_void_p, C.c_int, _u8p]),
    "navgpu_fleet_get_oscillation_mask": (C.c_int, [C.c_void_p, C.c_int, _i32p]),
    "navgpu_fleet_create_sensing": (C.c_int, [_vpp, C.c_int, C.POINTER(DwaConfig), C.c_uint32, C.c_uint32, C.c_double,
                                              C.POINTER(FleetCostmapConfig), _f64p, C.c_int, C.c_int]),
    "navgpu_fleet_set_scans": (C.c_int, [C.c_void_p, C.POINTER(LaserScan), _i32p]),
    "navgpu_fleet_set_scan_batch": (C.c_int, [C.c_void_p, C.POINTER(FleetScanSource), C.c_int]),
    "navgpu_fleet_set_scan_batch_device": (C.c_int, [C.c_void_p, C.POINTER(FleetScanSource), C.c_int]),
    "navgpu_fleet_stream": (C.c_void_p, [C.c_void_p]),
    "navgpu_fleet_get_layer": (C.c_int, [C.c_void_p, C.c_int, _u8p]),
    "navgpu_fleet_get_geometry": (C.c_int, [C.c_void_p, C.c_int, _f64p, _i32p]),
    "navgpu_fleet_last_timing": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "navgpu_fleet_create_sensing_voxel": (C.c_int, [_vpp, C.c_int, C.POINTER(DwaConfig), C.c_uint32, C.c_uint32,
                                                    C.c_double, C.POINTER(FleetCostmapConfig),
                                                    C.POINTER(FleetVoxelConfig), _f64p, C.c_int, C.c_int]),
    "navgpu_fleet_get_voxels": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_uint32)]),
    "navgpu_tp_default_config": (None, [C.POINTER(TpConfig)]),
    "navgpu_tp_create": (C.c_int, [_vpp, C.POINTER(TpConfig), C.c_uint32, C.c_uint32, C.c_double, _f64p, C.c_int, C.c_int]),
    "navgpu_tp_destroy": (C.c_int, [C.c_void_p]),
    "navgpu_tp_reconfigure": (C.c_int, [C.c_void_p, C.POINTER(TpConfig)]),
    "navgpu_tp_set_footprint": (C.c_int, [C.c_void_p, _f64p, C.c_int]),
    "navgpu_tp_set_costmap": (C.c_int, [C.c_void_p, _u8p, C.c_double, C.c_double]),
    "navgpu_tp_set_costmap_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_double, C.c_double]),
    "navgpu_tp_update_plan": (C.c_int, [C.c_void_p, _f64p, C.c_int]),
    "navgpu_tp_find_best_path": (C.c_int, [C.c_void_p, _f64p, _f64p, C.POINTER(TpResult), _f64p, C.c_int]),
    "navgpu_tp_score_trajectory": (C.c_int, [C.c_void_p, _f64p, _f64p, _f64p, _f64p]),
    "navgpu_tp_get_grid": (C.c_int, [C.c_void_p, C.c_int, _f64p]),
    "navgpu_tp_last_sample_count": (C.c_int, [C.c_void_p, _i32p]),
    "navgpu_fleet_use_trajectory_planner": (C.c_int, [C.c_void_p, C.POINTER(TpConfig)]),
    "navgpu_fleet_step_tp": (C.c_int, [C.c_void_p, _f64p, _f64p, C.POINTER(TpResult)]),
    "navgpu_fleet_tp_get_grid": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _f64p]),
    "navgpu_fleet_tp_last_timing": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                              C.POINTER(C.c_float)]),
    "navgpu_fleet_set_active": (C.c_int, [C.c_void_p, _u8p]),
    "navgpu_fleet_check_trajectories": (C.c_int, [C.c_void_p, _f64p, _f64p, _i32p, _f64p, _f64p]),
}


def pack_scans(scans):
    """The navgpu_laser_scan array for a list of scan dicts (see Costmap.set_scans), and the arrays it points into."""
    arr = (LaserScan * max(1, len(scans)))()
    keep = []
    for k, sc in enumerate(scans):
        s = arr[k]
        if "points" in sc:  # a PointCloud(2) source: (n, 3) float32 in the sensor frame
            r = np.ascontiguousarray(sc["points"], dtype=np.float32).reshape(-1, 3)
            s.is_cloud = 1
        else:
            r = np.ascontiguousarray(sc["ranges"], dtype=np.float32)
            s.is_cloud = 0
            s.angle_min, s.angle_increment = sc["angle_min"], sc["angle_increment"]
            s.range_min, s.range_max = sc["range_min"], sc["range_max"]
        keep.append(r)
        s.ranges = r.ctypes.data_as(C.POINTER(C.c_float))
        s.n_ranges = len(r)
        s.inf_is_valid = int(sc.get("inf_is_valid", 0))
        for j in range(3):
            s.translation[j] = sc["translation"][j]
        for j in range(4):
            s.rotation_xyzw[j] = sc["rotation_xyzw"][j]
        s.min_obstacle_height, s.max_obstacle_height = sc["min_obstacle_height"], sc["max_obstacle_height"]
        s.obstacle_range, s.raytrace_range = sc["obstacle_range"], sc["raytrace_range"]
        s.marking, s.clearing = int(sc.get("marking", True)), int(sc.get("clearing", True))
    return arr, keep


class Costmap:
    """Device-resident LayeredCostmap (navgpu_costmap_*)."""

    def __init__(self, api, size_x, size_y, resolution, origin_x=0.0, origin_y=0.0, rolling=False,
                 track_unknown=False, device=0):
        self.api, self.lib = api, api.lib
        self.size_x, self.size_y, self.resolution = size_x, size_y, resolution
        h = C.c_void_p()
        api.check(self.lib.navgpu_costmap_create(C.byref(h), size_x, size_y, resolution, origin_x, origin_y,
                                                 int(rolling), int(track_unknown), device))
        self.h = h

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.navgpu_costmap_destroy(self.h)
            self.h = None

    def _layer(self, rc, out):
        self.api.check(rc)
        return int(out.value)

    def add_grid_layer(self, policy):
        out = C.c_int32()
        return self._layer(self.lib.navgpu_costmap_add_grid_layer(self.h, policy, C.byref(out)), out)

    def add_obstacle_layer(self, combination_method=1, footprint_clearing=True, max_obstacle_height=2.0):
        out = C.c_int32()
        return self._layer(self.lib.navgpu_costmap_add_obstacle_layer(self.h, combination_method,
                                                                      int(footprint_clearing), max_obstacle_height,
                                                                      C.byref(out)), out)

    def add_inflation_layer(self, inflation_radius=0.55, cost_scaling_factor=10.0):
        out = C.c_int32()
        return self._layer(self.lib.navgpu_costmap_add_inflation_layer(self.h, inflation_radius, cost_scaling_factor,
                                                                       C.byref(out)), out)

    def add_voxel_layer(self, combination_method=1, footprint_clearing=True, max_obstacle_height=2.0, origin_z=0.0,
                        z_resolution=0.2, z_voxels=10, unknown_threshold=15, mark_threshold=0):
        out = C.c_int32()
        return self._layer(self.lib.navgpu_costmap_add_voxel_layer(
            self.h, combination_method, int(footprint_clearing), max_obstacle_height, origin_z, z_resolution, z_voxels,
            unknown_threshold, mark_threshold, C.byref(out)), out)

    def get_voxels(self, layer):
        out = np.zeros((self.size_y, self.size_x), dtype=np.uint32)
        self.api.check(self.lib.navgpu_layer_get_voxels(self.h, layer, out.ctypes.data_as(C.POINTER(C.c_uint32))))
        return out

    def set_footprint(self, xy):
        a = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
        self.api.check(self.lib.navgpu_costmap_set_footprint(self.h, _p(a, _f64p), a.shape[0]))

    def set_grid_layer(self, layer, data):
        a = np.ascontiguousarray(data, dtype=np.uint8)
        assert a.size == self.size_x * self.size_y
        self.api.check(self.lib.navgpu_grid_layer_set(self.h, layer, _p(a, _u8p)))

    def set_grid_layer_device(self, layer, dev_ptr, pitch):
        self.api.check(self.lib.navgpu_grid_layer_set_device(self.h, layer, C.c_void_p(dev_ptr), pitch))

    def set_grid_layer_occupancy(self, layer, occupancy, track_unknown=True, unknown_cost_value=255,
                                 lethal_threshold=100, trinary=True):
        a = np.ascontiguousarray(occupancy, dtype=np.int8)
        assert a.size == self.size_x * self.size_y
        self.api.check(self.lib.navgpu_grid_layer_set_occupancy(self.h, layer, _p(a, _i8p), int(track_unknown),
                                                                unknown_cost_value, lethal_threshold, int(trinary)))

    def touch_grid_layer(self, layer, x, y, w, h):
        self.api.check(self.lib.navgpu_grid_layer_touch(self.h, layer, x, y, w, h))

    def set_enabled(self, layer, enabled):
        self.api.check(self.lib.navgpu_layer_set_enabled(self.h, layer, int(enabled)))

    @staticmethod
    def pack_observations(observations):
        """The navgpu_observation array for a list of observation dicts (what a C++ caller holds anyway); reusable."""
        arr = (Observation * max(1, len(observations)))()
        keep = []
        for k, o in enumerate(observations):
            pts = np.ascontiguousarray(o["points"], dtype=np.float32).reshape(-1, 3)
            keep.append(pts)
            arr[k].origin_x, arr[k].origin_y, arr[k].origin_z = [float(v) for v in o["origin"]]
            arr[k].obstacle_range = float(o.get("obstacle_range", 2.5))
            arr[k].raytrace_range = float(o.get("raytrace_range", 3.0))
            arr[k].xyz = _p(pts, C.POINTER(C.c_float))
            arr[k].n_points = pts.shape[0]
            arr[k].marking = int(o.get("marking", True))
            arr[k].clearing = int(o.get("clearing", True))
        return arr, len(observations), keep

    def set_observations(self, layer, observations):
        arr, n, _keep = self.pack_observations(observations)
        self.api.check(self.lib.navgpu_obstacle_set_observations(self.h, layer, arr, n))

    def set_packed_observations(self, layer, packed):
        self.api.check(self.lib.navgpu_obstacle_set_observations(self.h, layer, packed[0], packed[1]))

    def set_scans(self, layer, scans):
        """On-device observation ingest: scans = list of dicts (ranges, angle_min, angle_increment, range_min,
        range_max, translation, rotation_xyzw, min/max_obstacle_height, obstacle_range, raytrace_range, marking,
        clearing, inf_is_valid)."""
        arr, _keep = pack_scans(scans)
        self.api.check(self.lib.navgpu_obstacle_set_scans(self.h, layer, arr, len(scans)))

    def get_cloud(self, layer, index, capacity=1 << 16):
        out = np.zeros((capacity, 3), dtype=np.float32)
        n = C.c_int32()
        self.api.check(self.lib.navgpu_obstacle_get_cloud(self.h, layer, index, out.ctypes.data_as(C.POINTER(C.c_float)),
                                                          capacity, C.byref(n)))
        return out[:n.value].copy()

    def set_inflation_params(self, layer, inflation_radius, cost_scaling_factor):
        self.api.check(self.lib.navgpu_inflation_set_params(self.h, layer, inflation_radius, cost_scaling_factor))

    def set_inflation_mode(self, layer, mode):
        self.api.check(self.lib.navgpu_inflation_set_mode(self.h, layer, mode))

    def inflation_last_rounds(self):
        r = np.zeros(1, dtype=np.int32)
        self.api.check(self.lib.navgpu_inflation_last_rounds(self.h, _p(r, _i32p)))
        return int(r[0])

    def update_map(self, x=0.0, y=0.0, yaw=0.0):
        w = np.zeros(4, dtype=np.int32)
        self.api.check(self.lib.navgpu_costmap_update_map(self.h, x, y, yaw, _p(w, _i32p)))
        return tuple(int(v) for v in w)

    def update_map_async(self, x=0.0, y=0.0, yaw=0.0):
        self.api.check(self.lib.navgpu_costmap_update_map_async(self.h, x, y, yaw))

    def synchronize(self):
        self.api.check(self.lib.navgpu_costmap_synchronize(self.h))

    def stream(self):
        return self.lib.navgpu_costmap_stream(self.h)

    def force_generic_sweep(self, enabled=True):
        self.api.check(self.lib.navgpu_costmap_force_generic_sweep(self.h, int(enabled)))

    def set_profiling(self, enabled=True):
        self.api.check(self.lib.navgpu_costmap_set_profiling(self.h, int(enabled)))

    def last_timing(self):
        """(whole cycle ms, fused sweep kernel ms) of the last update_map_async, from CUDA events on the stream."""
        c, s = C.c_float(), C.c_float()
        self.api.check(self.lib.navgpu_costmap_last_timing(self.h, C.byref(c), C.byref(s)))
        return float(c.value), float(s.value)

    def last_timing_split(self):
        """(k_merge_seed ms, k_inflate ms) of the last profiled update_map_async."""
        m, i = C.c_float(), C.c_float()
        self.api.check(self.lib.navgpu_costmap_last_timing_split(self.h, C.byref(m), C.byref(i)))
        return float(m.value), float(i.value)

    def get(self):
        out = np.empty((self.size_y, self.size_x), dtype=np.uint8)
        self.api.check(self.lib.navgpu_costmap_get(self.h, _p(out, _u8p)))
        return out

    def get_window(self, x0, y0, xn, yn, out=None):
        if out is None:
            out = np.empty((yn - y0, xn - x0), dtype=np.uint8)
        self.api.check(self.lib.navgpu_costmap_get_window(self.h, x0, y0, xn, yn, _p(out, _u8p)))
        return out

    def get_window_into(self, x0, y0, xn, yn, host_grid):
        """Downloads the window straight into its place in a full-size host grid (size_y x size_x uint8)."""
        assert host_grid.dtype == np.uint8 and host_grid.flags["C_CONTIGUOUS"]
        self.api.check(self.lib.navgpu_costmap_get_window_into(self.h, x0, y0, xn, yn, _p(host_grid, _u8p),
                                                               host_grid.shape[1]))

    def get_changed(self, host_grid, max_rects=0):
        """Brings `host_grid` (the full-size host mirror, size_y x size_x uint8, the same array every call) up to date
        with the device master grid moving only the 128 x 16 tiles that changed; returns (number of changed tiles,
        bytes that crossed PCIe, rects [n][x0, y0, xn, yn] when max_rects > 0)."""
        assert host_grid.dtype == np.uint8 and host_grid.flags["C_CONTIGUOUS"]
        n, nbytes = C.c_int32(), C.c_uint64()
        rects = np.zeros((max(1, max_rects), 4), dtype=np.int32)
        self.api.check(self.lib.navgpu_costmap_get_changed(self.h, _p(host_grid, _u8p), host_grid.shape[1],
                                                           _p(rects, _i32p), max_rects, C.byref(n), C.byref(nbytes)))
        return int(n.value), int(nbytes.value), rects[:min(int(n.value), max_rects)]

    def prepared_cycle(self, obstacle_layer, grid_layer, mirror):
        """One end-to-end update cycle with its arguments marshalled once, the way a C++ caller holds them:
        cycle(packed_observations, robot) = navgpu_obstacle_set_observations + navgpu_grid_layer_touch (whole layer) +
        navgpu_costmap_update_map_async + navgpu_costmap_get_changed into `mirror`; returns the bytes that crossed
        PCIe on the way back."""
        assert mirror.dtype == np.uint8 and mirror.flags["C_CONTIGUOUS"]
        lib, h, check = self.lib, self.h, self.api.check
        mptr, pitch = _p(mirror, _u8p), mirror.shape[1]
        n, nbytes = C.c_int32(), C.c_uint64()
        nref, bref = C.byref(n), C.byref(nbytes)
        sx, sy = self.size_x, self.size_y

        def cycle(packed, robot):
            check(lib.navgpu_obstacle_set_observations(h, obstacle_layer, packed[0], packed[1]))
            check(lib.navgpu_grid_layer_touch(h, grid_layer, 0, 0, sx, sy))
            check(lib.navgpu_costmap_update_map_async(h, robot[0], robot[1], robot[2]))
            check(lib.navgpu_costmap_get_changed(h, mptr, pitch, None, 0, nref, bref))
            return nbytes.value
        return cycle

    def mirror_invalidate(self):
        self.api.check(self.lib.navgpu_costmap_mirror_invalidate(self.h))

    def last_window(self):
        w = np.zeros(4, dtype=np.int32)
        self.api.check(self.lib.navgpu_costmap_last_window(self.h, _p(w, _i32p)))
        return tuple(int(v) for v in w)

    def get_window_occupancy(self, x0, y0, xn, yn):
        out = np.empty((yn - y0, xn - x0), dtype=np.int8)
        self.api.check(self.lib.navgpu_costmap_get_window_occupancy(self.h, x0, y0, xn, yn, _p(out, _i8p)))
        return out

    def set(self, grid):
        a = np.ascontiguousarray(grid, dtype=np.uint8)
        self.api.check(self.lib.navgpu_costmap_set(self.h, _p(a, _u8p)))

    def get_layer(self, layer):
        out = np.empty((self.size_y, self.size_x), dtype=np.uint8)
        self.api.check(self.lib.navgpu_layer_get(self.h, layer, _p(out, _u8p)))
        return out

    def origin(self):
        o = np.zeros(2)
        self.api.check(self.lib.navgpu_costmap_get_origin(self.h, _p(o, _f64p)))
        return float(o[0]), float(o[1])

    def device_grid(self):
        ptr, pitch = C.c_void_p(), C.c_uint32()
        self.api.check(self.lib.navgpu_costmap_device_grid(self.h, C.byref(ptr), C.byref(pitch)))
        return ptr.value, int(pitch.value)

    def inflation_tables(self, layer):
        cap = 256 * 256
        costs = np.zeros(cap, dtype=np.uint8)
        dists = np.zeros(cap, dtype=np.float64)
        R = C.c_int32()
        self.api.check(self.lib.navgpu_inflation_tables(self.h, layer, _p(costs, _u8p), _p(dists, _f64p), cap,
                                                        C.byref(R)))
        n = R.value + 2
        return R.value, costs[:n * n].reshape(n, n).copy(), dists[:n * n].reshape(n, n).copy()


class Dwa:
    """DWAPlanner-shaped scorer (navgpu_dwa_*)."""

    def __init__(self, api, size_x, size_y, resolution, device=0, **overrides):
        self.api, self.lib = api, api.lib
        self.size_x, self.size_y, self.resolution = size_x, size_y, resolution
        self.cfg = DwaConfig()
        self.lib.navgpu_dwa_default_config(C.byref(self.cfg))
        for k, v in overrides.items():
            setattr(self.cfg, k, v)
        h = C.c_void_p()
        api.check(self.lib.navgpu_dwa_create(C.byref(h), C.byref(self.cfg), size_x, size_y, resolution, device))
        self.h = h

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.navgpu_dwa_destroy(self.h)
            self.h = None

    def set_costmap(self, grid, origin_x=0.0, origin_y=0.0):
        a = np.ascontiguousarray(grid, dtype=np.uint8)
        assert a.size == self.size_x * self.size_y
        self.api.check(self.lib.navgpu_dwa_set_costmap(self.h, _p(a, _u8p), origin_x, origin_y))

    def set_costmap_device(self, dev_ptr, pitch, origin_x, origin_y):
        self.api.check(self.lib.navgpu_dwa_set_costmap_device(self.h, C.c_void_p(dev_ptr), pitch, origin_x, origin_y))

    def set_plan(self, pose, plan_xy):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        a = np.ascontiguousarray(plan_xy, dtype=np.float64).reshape(-1, 2)
        self.api.check(self.lib.navgpu_dwa_set_plan(self.h, _p(p, _f64p), _p(a, _f64p), a.shape[0]))

    def reset_oscillation(self):
        self.api.check(self.lib.navgpu_dwa_reset_oscillation(self.h))

    def oscillation_mask(self):
        m = C.c_int32()
        self.api.check(self.lib.navgpu_dwa_get_oscillation_mask(self.h, C.byref(m)))
        return int(m.value)

    def find_best_path(self, pose, vel, footprint_xy, max_samples=1 << 21, max_points=4096, want_costs=True):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        v = np.ascontiguousarray(vel, dtype=np.float64)
        f = np.ascontiguousarray(footprint_xy, dtype=np.float64).reshape(-1, 2)
        res = DwaResult()
        costs = np.full(max_samples if want_costs else 1, np.nan)
        pts = getattr(self, "_pts", None)  # result buffer kept across calls (a C++ caller owns one, too)
        if pts is None or pts.shape[0] != max_points:
            pts = self._pts = np.zeros((max_points, 3))
        self.api.check(self.lib.navgpu_dwa_find_best_path(
            self.h, _p(p, _f64p), _p(v, _f64p), _p(f, _f64p), f.shape[0], C.byref(res),
            _p(costs, _f64p) if want_costs else None, max_samples if want_costs else 0, _p(pts, _f64p), max_points))
        return dict(ok=res.cost >= 0, cost=res.cost, xv=res.xv, yv=res.yv, thetav=res.thetav,
                    best_index=res.best_index, n_samples=res.n_samples, n_scored=res.n_scored,
                    costs=costs[:res.n_samples].copy() if want_costs else None, points=pts[:res.n_points].copy())

    def check_trajectory(self, pose, vel, vel_samples, footprint_xy):
        """DWAPlanner::checkTrajectory: cost of the single trajectory for vel_samples (>= 0 means legal)."""
        p = np.ascontiguousarray(pose, dtype=np.float64)
        v = np.ascontiguousarray(vel, dtype=np.float64)
        s = np.ascontiguousarray(vel_samples, dtype=np.float64)
        f = np.ascontiguousarray(footprint_xy, dtype=np.float64).reshape(-1, 2)
        cost = np.zeros(1)
        self.api.check(self.lib.navgpu_dwa_check_trajectory(self.h, _p(p, _f64p), _p(v, _f64p), _p(s, _f64p),
                                                            _p(f, _f64p), f.shape[0], _p(cost, _f64p)))
        return float(cost[0])

    def find_best_path_async(self, pose, vel, footprint_xy):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        v = np.ascontiguousarray(vel, dtype=np.float64)
        f = np.ascontiguousarray(footprint_xy, dtype=np.float64).reshape(-1, 2)
        self.api.check(self.lib.navgpu_dwa_find_best_path_async(self.h, _p(p, _f64p), _p(v, _f64p), _p(f, _f64p),
                                                                f.shape[0]))

    def score_range(self, pose, vel, footprint_xy, begin, end):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        v = np.ascontiguousarray(vel, dtype=np.float64)
        f = np.ascontiguousarray(footprint_xy, dtype=np.float64).reshape(-1, 2)
        cost, idx, total = C.c_double(), C.c_int64(), C.c_int64()
        self.api.check(self.lib.navgpu_dwa_score_range(self.h, _p(p, _f64p), _p(v, _f64p), _p(f, _f64p), f.shape[0],
                                                       begin, end, C.byref(cost), C.byref(idx), C.byref(total)))
        return cost.value, idx.value, total.value

    def prepare(self):
        """prepare() of the critics: the four MapGrid wavefronts on the current costmap and plan."""
        self.api.check(self.lib.navgpu_dwa_prepare(self.h))

    def score_trajectories(self, trajectories, vels, footprint_xy, want_terms=False):
        """The batched TrajectoryCostFunction: `trajectories` = list of [n_i][3] arrays (x, y, theta), vels [n][3]
        (xv_, yv_, thetav_); returns the total cost per trajectory (and the six per-critic terms)."""
        n = len(trajectories)
        offs = np.zeros(n + 1, dtype=np.int32)
        for i, t in enumerate(trajectories):
            offs[i + 1] = offs[i] + len(t)
        pts = (np.concatenate([np.asarray(t, dtype=np.float64).reshape(-1, 3) for t in trajectories])
               if n and offs[-1] else np.zeros((0, 3)))
        pts = np.ascontiguousarray(pts, dtype=np.float64)
        v = np.ascontiguousarray(vels, dtype=np.float64).reshape(-1, 3)
        f = np.ascontiguousarray(footprint_xy, dtype=np.float64).reshape(-1, 2)
        costs = np.zeros(n)
        terms = np.zeros((n, 6)) if want_terms else None
        self.api.check(self.lib.navgpu_dwa_score_trajectories(
            self.h, n, _p(offs, _i32p), _p(pts, _f64p), _p(v, _f64p), _p(f, _f64p), f.shape[0], _p(costs, _f64p),
            _p(terms, _f64p) if want_terms else None))
        return (costs, terms) if want_terms else costs

    def update_oscillation(self, pose, cost, xv, yv, thetav):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        self.api.check(self.lib.navgpu_dwa_update_oscillation(self.h, _p(p, _f64p), cost, xv, yv, thetav))

    def samples(self):
        """Per-axis velocity samples of the last search: (xs, ys, ths) float32 arrays."""
        counts = np.zeros(3, dtype=np.int32)
        buf = np.zeros(1 << 16, dtype=np.float32)
        self.api.check(self.lib.navgpu_dwa_get_samples(self.h, _p(counts, _i32p), _p(buf, C.POINTER(C.c_float)), buf.size))
        nx, ny, nth = (int(c) for c in counts)
        return buf[:nx].copy(), buf[nx:nx + ny].copy(), buf[nx + ny:nx + ny + nth].copy()

    def score_strided(self, pose, vel, footprint_xy, rank, world):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        v = np.ascontiguousarray(vel, dtype=np.float64)
        f = np.ascontiguousarray(footprint_xy, dtype=np.float64).reshape(-1, 2)
        cost, idx, total = C.c_double(), C.c_int64(), C.c_int64()
        self.api.check(self.lib.navgpu_dwa_score_strided(self.h, _p(p, _f64p), _p(v, _f64p), _p(f, _f64p), f.shape[0],
                                                         rank, world, C.byref(cost), C.byref(idx), C.byref(total)))
        return cost.value, idx.value, total.value

    def shard_export(self):
        """This rank's exchange buffer as a 64-byte CUDA IPC handle (bytes)."""
        buf = (C.c_ubyte * 64)()
        self.api.check(self.lib.navgpu_dwa_shard_export(self.h, buf))
        return bytes(buf)

    def shard_connect(self, rank, world, handles):
        """handles: the `world` exported handles in rank order (bytes each)."""
        blob = b"".join(handles)
        assert len(blob) == 64 * world
        buf = (C.c_ubyte * len(blob)).from_buffer_copy(blob)
        self.api.check(self.lib.navgpu_dwa_shard_connect(self.h, rank, world, buf))

    def find_best_path_sharded_async(self, pose, vel, footprint_xy):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        v = np.ascontiguousarray(vel, dtype=np.float64)
        f = np.ascontiguousarray(footprint_xy, dtype=np.float64).reshape(-1, 2)
        self.api.check(self.lib.navgpu_dwa_find_best_path_sharded_async(self.h, _p(p, _f64p), _p(v, _f64p), _p(f, _f64p),
                                                                        f.shape[0]))

    def sharded_collect(self, pose, max_points=4096):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        res = DwaResult()
        pts = np.zeros((max_points, 3))
        self.api.check(self.lib.navgpu_dwa_sharded_collect(self.h, _p(p, _f64p), C.byref(res), _p(pts, _f64p), max_points))
        return dict(ok=res.cost >= 0, cost=res.cost, xv=res.xv, yv=res.yv, thetav=res.thetav,
                    best_index=res.best_index, n_samples=res.n_samples, n_scored=res.n_scored,
                    points=pts[:res.n_points].copy())

    def prepared(self, pose, vel, footprint_xy, max_points=256):
        """The arguments of a search marshalled once, the way a C++ caller holds them (plain arrays and a result
        struct): repeated calls then cost the C-ABI call only.  Returns an object with find_best_path() and
        find_best_path_sharded()."""
        return _PreparedSearch(self, pose, vel, footprint_xy, max_points)

    def find_best_path_sharded(self, pose, vel, footprint_xy, max_points=4096):
        self.find_best_path_sharded_async(pose, vel, footprint_xy)
        return self.sharded_collect(pose, max_points)

    def finish_sharded(self, pose, costs, indices, max_points=4096):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        c = np.ascontiguousarray(costs, dtype=np.float64)
        i = np.ascontiguousarray(indices, dtype=np.int64)
        res = DwaResult()
        pts = np.zeros((max_points, 3))
        self.api.check(self.lib.navgpu_dwa_finish_sharded(self.h, _p(p, _f64p), _p(c, _f64p), _p(i, _i64p), c.size,
                                                          C.byref(res), _p(pts, _f64p), max_points))
        return dict(ok=res.cost >= 0, cost=res.cost, xv=res.xv, yv=res.yv, thetav=res.thetav,
                    best_index=res.best_index, n_samples=res.n_samples, points=pts[:res.n_points].copy())

    def synchronize(self):
        self.api.check(self.lib.navgpu_dwa_synchronize(self.h))

    def stream(self):
        return self.lib.navgpu_dwa_stream(self.h)

    def grid(self, which):
        out = np.empty((self.size_y, self.size_x), dtype=np.float64)
        self.api.check(self.lib.navgpu_dwa_get_grid(self.h, which, _p(out, _f64p)))
        return out


def tp_config(lib, overrides):
    """TrajectoryPlannerROS's defaults (navgpu_tp_default_config) with `overrides` (TpConfig field names; y_vels as a
    list) applied."""
    cfg = TpConfig()
    lib.navgpu_tp_default_config(C.byref(cfg))
    for k, v in overrides.items():
        if k == "y_vels":
            for j, y in enumerate(v):
                cfg.y_vels[j] = y
            cfg.n_y_vels = len(v)
        else:
            setattr(cfg, k, v)
    return cfg


class TrajectoryPlanner:
    """The legacy base_local_planner::TrajectoryPlanner (navgpu_tp_*)."""

    def __init__(self, api, size_x, size_y, resolution, footprint_xy, device=0, **overrides):
        self.api, self.lib = api, api.lib
        self.size_x, self.size_y = size_x, size_y
        self.cfg = tp_config(self.lib, overrides)
        f = np.ascontiguousarray(footprint_xy, dtype=np.float64).reshape(-1, 2)
        h = C.c_void_p()
        api.check(self.lib.navgpu_tp_create(C.byref(h), C.byref(self.cfg), size_x, size_y, resolution, _p(f, _f64p),
                                            f.shape[0], device))
        self.h = h

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.navgpu_tp_destroy(self.h)
            self.h = None

    def set_costmap(self, grid, origin_x=0.0, origin_y=0.0):
        a = np.ascontiguousarray(grid, dtype=np.uint8)
        assert a.size == self.size_x * self.size_y
        self.api.check(self.lib.navgpu_tp_set_costmap(self.h, _p(a, _u8p), origin_x, origin_y))

    def set_costmap_device(self, dev_ptr, pitch, origin_x, origin_y):
        self.api.check(self.lib.navgpu_tp_set_costmap_device(self.h, C.c_void_p(dev_ptr), pitch, origin_x, origin_y))

    def update_plan(self, plan_xy):
        a = np.ascontiguousarray(plan_xy, dtype=np.float64).reshape(-1, 2)
        self.api.check(self.lib.navgpu_tp_update_plan(self.h, _p(a, _f64p), a.shape[0]))

    def find_best_path(self, pose, vel, max_points=4096):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        v = np.ascontiguousarray(vel, dtype=np.float64)
        res = TpResult()
        pts = np.zeros((max_points, 3))
        self.api.check(self.lib.navgpu_tp_find_best_path(self.h, _p(p, _f64p), _p(v, _f64p), C.byref(res), _p(pts, _f64p),
                                                         max_points))
        return dict(cost=res.cost, xv=res.xv, yv=res.yv, thetav=res.thetav, flags=res.flags,
                    points=pts[:res.n_points].copy())

    def score_trajectory(self, pose, vel, vel_samples):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        v = np.ascontiguousarray(vel, dtype=np.float64)
        s = np.ascontiguousarray(vel_samples, dtype=np.float64)
        c = C.c_double()
        self.api.check(self.lib.navgpu_tp_score_trajectory(self.h, _p(p, _f64p), _p(v, _f64p), _p(s, _f64p), C.byref(c)))
        return float(c.value)

    def grid(self, which):
        out = np.empty((self.size_y, self.size_x), dtype=np.float64)
        self.api.check(self.lib.navgpu_tp_get_grid(self.h, which, _p(out, _f64p)))
        return out

    def last_sample_count(self):
        n = C.c_int32()
        self.api.check(self.lib.navgpu_tp_last_sample_count(self.h, C.byref(n)))
        return int(n.value)


class _PreparedSearch:
    def __init__(self, dwa, pose, vel, footprint_xy, max_points):
        self.dwa, self.lib, self.check = dwa, dwa.lib, dwa.api.check
        self.p = np.ascontiguousarray(pose, dtype=np.float64)
        self.v = np.ascontiguousarray(vel, dtype=np.float64)
        self.f = np.ascontiguousarray(footprint_xy, dtype=np.float64).reshape(-1, 2)
        self.res = DwaResult()
        self.pts = np.zeros((max_points, 3))
        self.max_points = max_points
        self._a = (_p(self.p, _f64p), _p(self.v, _f64p), _p(self.f, _f64p), self.f.shape[0])
        self._r = (C.byref(self.res), _p(self.pts, _f64p), max_points)

    def _result(self):
        r = self.res
        return dict(ok=r.cost >= 0, cost=r.cost, xv=r.xv, yv=r.yv, thetav=r.thetav, best_index=r.best_index,
                    n_samples=r.n_samples, n_scored=r.n_scored, points=self.pts[:min(r.n_points, self.max_points)])

    def find_best_path(self):
        self.check(self.lib.navgpu_dwa_find_best_path(self.dwa.h, *self._a, self._r[0], None, 0, self._r[1], self._r[2]))
        return self._result()

    def find_best_path_sharded(self):
        self.check(self.lib.navgpu_dwa_find_best_path_sharded(self.dwa.h, *self._a, *self._r))
        return self._result()


class Fleet:
    """N independent robots per control cycle (navgpu_fleet_*): local-costmap inflation + DWA scoring, batched."""

    def __init__(self, api, n_robots, size_x, size_y, resolution, footprint_xy, inflation_radius=0.55,
                 cost_scaling_factor=10.0, device=0, sensing=None, voxel=None, trajectory_planner=None, **overrides):
        """sensing: None for a raw-map fleet (set_maps), else a FleetCostmapConfig: every robot then builds its own
        rolling local costmap from its scans (set_scans; see Api.fleet_sensing).  voxel: with sensing, a
        FleetVoxelConfig makes that costmap's obstacle layer a VoxelLayer.  trajectory_planner: None for DWAPlanner
        (`overrides` are then DwaConfig fields), else a dict of TpConfig overrides, possibly empty: the robots run the
        legacy base_local_planner::TrajectoryPlanner (navgpu_fleet_use_trajectory_planner) and step() returns its
        results."""
        self.api, self.lib, self.n = api, api.lib, n_robots
        self.size_x, self.size_y = size_x, size_y
        self.device = device
        self._batch_keep = None  # the device arrays of the last set_scan_batch, alive until the next one
        self._active = None      # the set_active mask (None: every robot)
        self.cfg = DwaConfig()
        self.lib.navgpu_dwa_default_config(C.byref(self.cfg))
        for k, v in overrides.items():
            setattr(self.cfg, k, v)
        fp = np.ascontiguousarray(footprint_xy, dtype=np.float64).reshape(-1, 2)
        h = C.c_void_p()
        if sensing is None:
            api.check(self.lib.navgpu_fleet_create(C.byref(h), n_robots, C.byref(self.cfg), size_x, size_y, resolution,
                                                   inflation_radius, cost_scaling_factor, _p(fp, _f64p), fp.shape[0],
                                                   device))
        elif voxel is None:
            api.check(self.lib.navgpu_fleet_create_sensing(C.byref(h), n_robots, C.byref(self.cfg), size_x, size_y,
                                                           resolution, C.byref(sensing), _p(fp, _f64p), fp.shape[0],
                                                           device))
        else:
            api.check(self.lib.navgpu_fleet_create_sensing_voxel(C.byref(h), n_robots, C.byref(self.cfg), size_x,
                                                                 size_y, resolution, C.byref(sensing), C.byref(voxel),
                                                                 _p(fp, _f64p), fp.shape[0], device))
        self.h = h
        self.tp_cfg = None
        if trajectory_planner is None:
            self._results = (DwaResult * n_robots)()
        else:
            self.tp_cfg = tp_config(self.lib, trajectory_planner)
            api.check(self.lib.navgpu_fleet_use_trajectory_planner(self.h, C.byref(self.tp_cfg)))
            self._results = (TpResult * n_robots)()

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.navgpu_fleet_destroy(self.h)
            self.h = None

    def set_maps(self, raw_maps, origins_xy):
        m = np.ascontiguousarray(raw_maps, dtype=np.uint8)
        o = np.ascontiguousarray(origins_xy, dtype=np.float64)
        assert m.shape == (self.n, self.size_y, self.size_x) and o.shape == (self.n, 2)
        self.api.check(self.lib.navgpu_fleet_set_maps(self.h, _p(m, _u8p), _p(o, _f64p)))

    def set_plans(self, poses, plans):
        """plans: list of (k_i, 2) arrays, one per robot."""
        p = np.ascontiguousarray(poses, dtype=np.float64)
        off = np.zeros(self.n + 1, dtype=np.int32)
        off[1:] = np.cumsum([len(q) for q in plans])
        xy = np.ascontiguousarray(np.concatenate([np.asarray(q, dtype=np.float64).reshape(-1, 2) for q in plans]))
        self.api.check(self.lib.navgpu_fleet_set_plans(self.h, _p(p, _f64p), _p(xy, _f64p), _p(off, _i32p)))

    def reset_oscillation(self):
        self.api.check(self.lib.navgpu_fleet_reset_oscillation(self.h))

    def step(self, poses, vels):
        """One control cycle.  Per robot: cost, xv, yv, thetav, best_index, n_samples, n_scored with DWAPlanner;
        cost, xv, yv, thetav, flags, n_points with the TrajectoryPlanner (navgpu_tp_result); None for a robot that
        set_active left out."""
        p = np.ascontiguousarray(poses, dtype=np.float64)
        v = np.ascontiguousarray(vels, dtype=np.float64)
        assert p.shape == (self.n, 3) and v.shape == (self.n, 3)
        r = self.step_raw(p, v)
        act = self._active
        if self.tp_cfg is not None:
            out = [dict(cost=r[i].cost, xv=r[i].xv, yv=r[i].yv, thetav=r[i].thetav, flags=r[i].flags,
                        n_points=r[i].n_points) for i in range(self.n)]
        else:
            out = [dict(cost=r[i].cost, xv=r[i].xv, yv=r[i].yv, thetav=r[i].thetav, best_index=r[i].best_index,
                        n_samples=r[i].n_samples, n_scored=r[i].n_scored) for i in range(self.n)]
        return out if act is None else [g if a else None for g, a in zip(out, act)]

    def step_device(self, poses, vels, out=None):
        """step() on the device (navgpu_fleet_step_device), for a simulator that keeps its robots on the GPU: poses and
        vels are contiguous float64 CUDA tensors [n, 3] on the fleet's device.  The fleet's stream first waits for
        torch's current stream, and torch's current stream then waits for the fleet's, so torch work queued after
        this call sees the results; nothing waits on the host.  Returns views of one CUDA buffer of n result records:
        cost, xv, yv, thetav (float64), best_index, n_samples, n_scored (int32), and the buffer itself as `records`
        (uint8), which `out` may pass back to be written again.  A robot that set_active left out keeps its record as
        it was.  Wrong devices, dtypes or shapes raise ValueError."""
        import torch
        dev = torch.device("cuda", self.device)
        for what, x in (("poses", poses), ("vels", vels)):
            if not isinstance(x, torch.Tensor) or x.dtype != torch.float64 or tuple(x.shape) != (self.n, 3) or \
                    not x.is_cuda or x.device.index != self.device or not x.is_contiguous():
                raise ValueError(f"{what}: a contiguous float64 tensor of shape ({self.n}, 3) on cuda:{self.device}")
        nbytes = self.n * C.sizeof(DwaResult)
        if out is None:
            out = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        elif not isinstance(out, torch.Tensor) or out.dtype != torch.uint8 or tuple(out.shape) != (nbytes,) or \
                not out.is_cuda or out.device.index != self.device or not out.is_contiguous():
            raise ValueError(f"out: a contiguous uint8 tensor of {nbytes} bytes on cuda:{self.device}")
        fleet_stream = torch.cuda.ExternalStream(self.stream(), device=dev)
        fleet_stream.wait_stream(torch.cuda.current_stream(dev))
        # (no record_stream on the fleet's stream, which may be destroyed before the tensors are freed: torch's current
        # stream waits for the fleet's below, so memory torch reuses there is only written after the step read it)
        self.api.check(self.lib.navgpu_fleet_step_device(self.h, poses.data_ptr(), vels.data_ptr(), out.data_ptr()))
        torch.cuda.current_stream(dev).wait_stream(fleet_stream)
        words = C.sizeof(DwaResult) // 8
        f64 = out.view(torch.float64).view(self.n, words)
        i32 = out.view(torch.int32).view(self.n, 2 * words)
        return dict(cost=f64[:, 0], xv=f64[:, 1], yv=f64[:, 2], thetav=f64[:, 3], best_index=i32[:, 8],
                    n_samples=i32[:, 9], n_scored=i32[:, 10], records=out)

    def set_active(self, mask):
        """Which robots the following steps plan for (navgpu_fleet_set_active): n_robots booleans or 0 / 1 values, or
        None for every robot.  A left-out robot keeps its costmap updates but none of its planner runs, and step()
        returns None for it; check_trajectories still checks commands against its last planning step."""
        if mask is None:
            self.api.check(self.lib.navgpu_fleet_set_active(self.h, None))
            self._active = None
            return
        m = np.asarray(mask)
        assert m.shape == (self.n,)
        u = np.ascontiguousarray(np.where((m == 0) | (m == 1), m, 2), dtype=np.uint8)  # (other values are refused)
        self.api.check(self.lib.navgpu_fleet_set_active(self.h, _p(u, _u8p)))
        self._active = u.astype(bool)

    def check_trajectories(self, poses, vels, candidates):
        """checkTrajectory of each robot's candidate commands (navgpu_fleet_check_trajectories): candidates[r] is a
        (k_r, 3) array of (vx, vy, vtheta), possibly empty; returns one array of k_r costs per robot (>= 0: legal)."""
        p = np.ascontiguousarray(poses, dtype=np.float64)
        v = np.ascontiguousarray(vels, dtype=np.float64)
        assert p.shape == (self.n, 3) and v.shape == (self.n, 3) and len(candidates) == self.n
        cand = [np.asarray(c, dtype=np.float64).reshape(-1, 3) for c in candidates]
        off = np.zeros(self.n + 1, dtype=np.int32)
        off[1:] = np.cumsum([len(c) for c in cand])
        s = np.ascontiguousarray(np.concatenate(cand) if off[-1] else np.zeros((1, 3)))
        costs = np.zeros(max(int(off[-1]), 1))
        self.api.check(self.lib.navgpu_fleet_check_trajectories(self.h, _p(p, _f64p), _p(v, _f64p), _p(off, _i32p),
                                                                _p(s, _f64p), _p(costs, _f64p)))
        return [costs[off[r]:off[r + 1]].copy() for r in range(self.n)]

    def step_raw(self, poses, vels):
        """step() without building Python dicts (benchmarks); returns the ctypes result array."""
        step = self.lib.navgpu_fleet_step if self.tp_cfg is None else self.lib.navgpu_fleet_step_tp
        self.api.check(step(self.h, _p(poses, _f64p), _p(vels, _f64p), self._results))
        return self._results

    def tp_grid(self, robot, which):
        """TrajectoryPlanner fleets: path_map_ (which = 0) or goal_map_ (1) of robot after the last step."""
        out = np.empty((self.size_y, self.size_x), dtype=np.float64)
        self.api.check(self.lib.navgpu_fleet_tp_get_grid(self.h, robot, which, _p(out, _f64p)))
        return out

    def tp_timing(self):
        """TrajectoryPlanner fleets: device ms of the last step's footprint-cell, wavefront and scoring launches."""
        a, b, c = C.c_float(), C.c_float(), C.c_float()
        self.api.check(self.lib.navgpu_fleet_tp_last_timing(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return float(a.value), float(b.value), float(c.value)

    def costmap(self, robot):
        out = np.empty((self.size_y, self.size_x), dtype=np.uint8)
        self.api.check(self.lib.navgpu_fleet_get_costmap(self.h, robot, _p(out, _u8p)))
        return out

    def oscillation_mask(self, robot):
        m = C.c_int32()
        self.api.check(self.lib.navgpu_fleet_get_oscillation_mask(self.h, robot, C.byref(m)))
        return int(m.value)

    def set_scans(self, scans_per_robot):
        """Sensing fleets: scans_per_robot[r] = list of robot r's scan dicts (the format of Costmap.set_scans); they
        replace every robot's previous sources."""
        assert len(scans_per_robot) == self.n
        off = np.zeros(self.n + 1, dtype=np.int32)
        off[1:] = np.cumsum([len(s) for s in scans_per_robot])
        arr, _keep = pack_scans([s for robot in scans_per_robot for s in robot])
        self.api.check(self.lib.navgpu_fleet_set_scans(self.h, arr, _p(off, _i32p)))

    def set_scan_batch(self, sources):
        """Sensing fleets whose robots carry the same sensors: robot r's sources become [source 0, source 1, ...],
        each built from the source's shared fields and row r of its arrays -- set_scans with those lists, bit for bit.
        A source is a dict with the scan-dict fields (angle_min, angle_increment, range_min, range_max, inf_is_valid,
        min_obstacle_height, max_obstacle_height, obstacle_range, raytrace_range, marking, clearing), either `ranges`
        [n, B] float32 (LaserScan) or `points` [n, B, 3] float32 (sensor-frame cloud), and `sensor_to_global` [n, 7]
        float64 (translation x, y, z, rotation x, y, z, w).
        numpy arrays and CPU torch tensors are copied to the device and read before the call returns
        (navgpu_fleet_set_scan_batch).  Contiguous CUDA torch tensors on the fleet's device are read in place on the
        fleet's stream, after the work already queued on torch's current stream (navgpu_fleet_set_scan_batch_device):
        leave them unchanged until the next step returns.  Mixed host and device arrays, wrong shapes and wrong dtypes
        raise ValueError."""
        torch = sys.modules.get("torch")  # a torch tensor can only come from a caller that imported torch
        arr = (FleetScanSource * max(1, len(sources)))()
        keep, where = [], set()

        def take(x, what, dtype, shape):
            if torch is not None and isinstance(x, torch.Tensor):
                if x.dtype != getattr(torch, dtype) or x.dim() != len(shape) or \
                        any(s is not None and x.shape[i] != s for i, s in enumerate(shape)):
                    raise ValueError(f"{what}: a {dtype} tensor of shape {shape}, not {x.dtype} {tuple(x.shape)}")
                if x.is_cuda:
                    if x.device.index != self.device or not x.is_contiguous():
                        raise ValueError(f"{what}: a contiguous tensor on cuda:{self.device}")
                    where.add("device")
                    keep.append(x)
                    return x.data_ptr(), x.shape
                x = x.detach().numpy()
            if not isinstance(x, np.ndarray):
                raise ValueError(f"{what}: a numpy array or a torch tensor, not {type(x).__name__}")
            if x.dtype != np.dtype(dtype) or x.ndim != len(shape) or \
                    any(s is not None and x.shape[i] != s for i, s in enumerate(shape)):
                raise ValueError(f"{what}: a {dtype} array of shape {shape}, not {x.dtype} {x.shape}")
            x = np.ascontiguousarray(x)
            where.add("host")
            keep.append(x)
            return x.ctypes.data, x.shape

        for k, src in enumerate(sources):
            cloud = "points" in src
            if cloud == ("ranges" in src):
                raise ValueError(f"source {k}: give either ranges or points")
            s = arr[k]
            if cloud:
                s.data, shape = take(src["points"], f"source {k} points", "float32", (self.n, None, 3))
            else:
                s.data, shape = take(src["ranges"], f"source {k} ranges", "float32", (self.n, None))
                s.angle_min, s.angle_increment = src["angle_min"], src["angle_increment"]
                s.range_min, s.range_max = src["range_min"], src["range_max"]
            s.sensor_to_global, _ = take(src["sensor_to_global"], f"source {k} sensor_to_global", "float64", (self.n, 7))
            s.n_points, s.is_cloud = int(shape[1]), int(cloud)
            s.inf_is_valid = int(src.get("inf_is_valid", 0))
            s.min_obstacle_height, s.max_obstacle_height = src["min_obstacle_height"], src["max_obstacle_height"]
            s.obstacle_range, s.raytrace_range = src["obstacle_range"], src["raytrace_range"]
            s.marking, s.clearing = int(src.get("marking", True)), int(src.get("clearing", True))
        if len(where) > 1:
            raise ValueError("a batch is either host arrays or device arrays, not both")
        if where == {"device"}:
            dev = torch.device("cuda", self.device)
            torch.cuda.ExternalStream(self.stream(), device=dev).wait_stream(torch.cuda.current_stream(dev))
            self.api.check(self.lib.navgpu_fleet_set_scan_batch_device(self.h, arr, len(sources)))
            self._batch_keep = keep
        else:
            self.api.check(self.lib.navgpu_fleet_set_scan_batch(self.h, arr, len(sources)))
            self._batch_keep = None

    def stream(self):
        """The CUDA stream (cudaStream_t as an int) every kernel of this fleet runs on."""
        return self.lib.navgpu_fleet_stream(self.h)

    def layer(self, robot):
        """Sensing fleets: robot's ObstacleLayer (or VoxelLayer) grid after the last step."""
        out = np.empty((self.size_y, self.size_x), dtype=np.uint8)
        self.api.check(self.lib.navgpu_fleet_get_layer(self.h, robot, _p(out, _u8p)))
        return out

    def voxels(self, robot):
        """Voxel fleets: robot's VoxelLayer columns after the last step (size_y x size_x uint32: bit z = unknown or
        marked, bit z + 16 = marked)."""
        out = np.empty((self.size_y, self.size_x), dtype=np.uint32)
        self.api.check(self.lib.navgpu_fleet_get_voxels(self.h, robot, out.ctypes.data_as(C.POINTER(C.c_uint32))))
        return out

    def geometry(self, robot):
        """Sensing fleets: ((origin_x, origin_y), (x0, xn, y0, yn)) of robot's last step."""
        o = np.zeros(2)
        w = np.zeros(4, dtype=np.int32)
        self.api.check(self.lib.navgpu_fleet_get_geometry(self.h, robot, _p(o, _f64p), _p(w, _i32p)))
        return (float(o[0]), float(o[1])), tuple(int(v) for v in w)

    def last_timing(self):
        """Sensing fleets: device ms of the last scan projection and of the last costmap update of all robots."""
        a, b = C.c_float(), C.c_float()
        self.api.check(self.lib.navgpu_fleet_last_timing(self.h, C.byref(a), C.byref(b)))
        return float(a.value), float(b.value)


class Api:
    name = "cuda"

    def __init__(self, path=LIB_PATH):
        if not os.path.exists(path):
            raise NavGpuError(f"{path} is missing: run `python -m navigation_b200.build` (there is no CPU fallback)")
        self.lib = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(self.lib, name)
            f.restype = res
            f.argtypes = args

    def check(self, rc):
        if rc != 0:
            raise NavGpuError(f"navgpu error {rc}: {self.lib.navgpu_last_error().decode(errors='replace')}")

    def device_count(self):
        return self.lib.navgpu_device_count()

    def launch_count(self):
        return int(self.lib.navgpu_launch_count())

    def costmap(self, *a, **k):
        return Costmap(self, *a, **k)

    def dwa(self, *a, **k):
        return Dwa(self, *a, **k)

    def shard_connect_local(self, dwas):
        """One process driving several planner handles (one per GPU, or several on one GPU): dwas[r] becomes rank r."""
        arr = (C.c_void_p * len(dwas))(*[d.h for d in dwas])
        self.check(self.lib.navgpu_dwa_shard_connect_local(arr, len(dwas)))

    def fleet(self, *a, **k):
        """A raw-map fleet (see Fleet); trajectory_planner={...} runs the legacy TrajectoryPlanner instead of DWAPlanner."""
        return Fleet(self, *a, **k)

    def fleet_sensing(self, n, sx, sy, res, footprint, inflation_radius=0.55, cost_scaling_factor=10.0,
                      combination_method=1, footprint_clearing=True, max_obstacle_height=2.0, track_unknown=False,
                      device=0, voxel=None, trajectory_planner=None, **dwa_overrides):
        """A fleet whose robots each run a rolling sx x sy local costmap [ObstacleLayer, InflationLayer] fed by their
        own scans (Fleet.set_scans), then DWAPlanner (navgpu_fleet_create_sensing).  voxel: a FleetVoxelConfig or a
        dict of its fields (origin_z, z_resolution, z_voxels, unknown_threshold, mark_threshold; missing ones take
        VoxelPlugin.cfg's defaults) makes it [VoxelLayer, InflationLayer] (navgpu_fleet_create_sensing_voxel).
        trajectory_planner: a dict of TpConfig overrides, possibly empty, runs the legacy TrajectoryPlanner instead of
        DWAPlanner (see Fleet)."""
        cm = FleetCostmapConfig(inflation_radius=inflation_radius, cost_scaling_factor=cost_scaling_factor,
                                max_obstacle_height=max_obstacle_height, combination_method=combination_method,
                                footprint_clearing=int(footprint_clearing), track_unknown=int(track_unknown))
        if isinstance(voxel, dict):
            voxel = FleetVoxelConfig(**{**VOXEL_DEFAULTS, **voxel})
        return Fleet(self, n, sx, sy, res, footprint, device=device, sensing=cm, voxel=voxel,
                     trajectory_planner=trajectory_planner, **dwa_overrides)

    def trajectory_planner(self, *a, **k):
        return TrajectoryPlanner(self, *a, **k)

    def build_cost_table(self, resolution, inscribed_radius, inflation_radius, cost_scaling_factor):
        cap = 256 * 256
        costs = np.zeros(cap, dtype=np.uint8)
        dists = np.zeros(cap, dtype=np.float64)
        R = C.c_int32()
        self.check(self.lib.navgpu_build_cost_table(resolution, inscribed_radius, inflation_radius,
                                                    cost_scaling_factor, _p(costs, _u8p), _p(dists, _f64p), cap,
                                                    C.byref(R)))
        n = R.value + 2
        return R.value, costs[:n * n].reshape(n, n).copy(), dists[:n * n].reshape(n, n).copy()

    @staticmethod
    def _pack_plans(plans):
        offs = np.zeros(len(plans) + 1, dtype=np.int32)
        for i, p in enumerate(plans):
            offs[i + 1] = offs[i] + len(p)
        xyz = np.zeros((int(offs[-1]), 3))
        for i, p in enumerate(plans):
            a = np.asarray(p, dtype=np.float64).reshape(len(p), -1) if len(p) else np.zeros((0, 3))
            xyz[offs[i]:offs[i + 1], :a.shape[1]] = a
        return offs, np.ascontiguousarray(xyz)

    def plans_transform(self, plans, robot_xy, transforms, thresholds, device=0):
        """Batched base_local_planner::transformGlobalPlan: plans = list of [n_i][2 or 3] arrays, robot_xy [n][2] in the
        plans' frames, transforms [n][12] (3x3 rotation row-major, then the origin), thresholds [n]; returns
        (first index, list of transformed [count_i][3] arrays)."""
        n = len(plans)
        offs, xyz = self._pack_plans(plans)
        rob = np.ascontiguousarray(robot_xy, dtype=np.float64).reshape(n, 2)
        tf = np.ascontiguousarray(transforms, dtype=np.float64).reshape(n, 12)
        thr = np.ascontiguousarray(thresholds, dtype=np.float64).reshape(n)
        first, count = np.zeros(n, dtype=np.int32), np.zeros(n, dtype=np.int32)
        out = np.zeros_like(xyz)
        self.check(self.lib.navgpu_plans_transform(n, _p(offs, _i32p), _p(xyz, _f64p), _p(rob, _f64p),
                                                   C.c_void_p(tf.ctypes.data), _p(thr, _f64p), _p(first, _i32p),
                                                   _p(count, _i32p), _p(out, _f64p), device))
        return first, [out[offs[i]:offs[i] + count[i]].copy() for i in range(n)]

    def plans_prune(self, plans, robot_xy, device=0):
        """Batched base_local_planner::prunePlan: how many way-points are erased from the front of every plan."""
        n = len(plans)
        offs, xyz = self._pack_plans(plans)
        rob = np.ascontiguousarray(robot_xy, dtype=np.float64).reshape(n, 2)
        erase = np.zeros(n, dtype=np.int32)
        self.check(self.lib.navgpu_plans_prune(n, _p(offs, _i32p), _p(xyz, _f64p), _p(rob, _f64p), _p(erase, _i32p), device))
        return erase

    def host_register(self, array):
        """Page-locks a numpy array's buffer (navgpu_host_register); undo with host_unregister."""
        self.check(self.lib.navgpu_host_register(C.c_void_p(array.ctypes.data), array.nbytes))

    def host_unregister(self, array):
        self.check(self.lib.navgpu_host_unregister(C.c_void_p(array.ctypes.data)))

    def inflate_host(self, master, min_i, min_j, max_i, max_j, cost_table, radius, device=0):
        assert master.dtype == np.uint8 and master.flags.c_contiguous
        t = np.ascontiguousarray(cost_table, dtype=np.uint8)
        self.check(self.lib.navgpu_inflate_host(_p(master, _u8p), master.shape[1], master.shape[0], min_i, min_j,
                                                max_i, max_j, _p(t, _u8p), radius, device))
        return master

    def merge_host(self, master, layer, min_i, min_j, max_i, max_j, policy, device=0):
        assert master.dtype == np.uint8 and master.flags.c_contiguous
        a = np.ascontiguousarray(layer, dtype=np.uint8)
        self.check(self.lib.navgpu_merge_host(_p(master, _u8p), _p(a, _u8p), master.shape[1], master.shape[0], min_i,
                                              min_j, max_i, max_j, policy, device))
        return master


_api = None


def load():
    global _api
    if _api is None:
        _api = Api()
    return _api
