"""ctypes binding of oracle_api.h -- TEST INFRASTRUCTURE ONLY (see oracle/oracle_api.h).

Loads either checker:
    load("port")       -> oracle/libnavoracle.so   (our CPU restatement)
    load("reference")  -> oracle/_ref/libnavref.so (the reference's own compiled sources; may be absent)
    load("reference_hoisted") -> oracle/_ref/libnavref_hoisted.so (the same with map_grid.cpp:106 reading the default
                          value without copying the costmap: timing baseline only, see oracle/Makefile)
Nothing under navigation_b200/ imports this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

TRUE_OVERWRITE, OVERWRITE, MAX, ADDITION, NOTHING = 0, 1, 2, 3, 4


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
    _fields_ = [("ranges", C.POINTER(C.c_float)), ("n_ranges", C.c_int32), ("inf_is_valid", C.c_int32),
                ("angle_min", C.c_float), ("angle_increment", C.c_float), ("range_min", C.c_float),
                ("range_max", C.c_float), ("translation", C.c_double * 3), ("rotation_xyzw", C.c_double * 4),
                ("min_obstacle_height", C.c_double), ("max_obstacle_height", C.c_double), ("is_cloud", C.c_int32),
                ("pad_", C.c_int32)]


class TpConfig(C.Structure):
    """navo_tp_config / navgpu_tp_config: the legacy base_local_planner::TrajectoryPlanner's parameters."""
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
_f64p = C.POINTER(C.c_double)
_i32p = C.POINTER(C.c_int32)
_u32p = C.POINTER(C.c_uint32)


def _p(a, t):
    return a.ctypes.data_as(t)


def _declare(lib, prefix):
    """Declare argtypes; `prefix` is 'navo_' for the oracles (the product library has its own binding)."""
    g = lambda n: getattr(lib, prefix + n)
    vp, d, i, u = C.c_void_p, C.c_double, C.c_int, C.c_uint32
    sig = {
        "costmap_create": (vp, [u, u, d, d, d, i, i]),
        "costmap_destroy": (None, [vp]),
        "costmap_add_grid_layer": (i, [vp, i]),
        "costmap_add_obstacle_layer": (i, [vp, i, i, d]),
        "costmap_add_inflation_layer": (i, [vp, d, d]),
        "costmap_add_voxel_layer": (i, [vp, i, i, d, d, d, i, i, i]),
        "layer_get_voxels": (None, [vp, i, _u32p]),
        "voxel_line_cells": (i, [u, d, d, d, d, d, d, u, _u32p, _i32p, i]),
        "costmap_set_footprint": (None, [vp, _f64p, i]),
        "grid_layer_set": (None, [vp, i, _u8p]),
        "grid_layer_touch": (None, [vp, i, u, u, u, u]),
        "layer_set_enabled": (None, [vp, i, i]),
        "obstacle_set_observations": (None, [vp, i, C.POINTER(Observation), i]),
        "inflation_set_params": (None, [vp, i, d, d]),
        "inflation_set_variant": (i, [vp, i, i, C.c_uint64]),
        "inflation_last_rounds": (i, [vp, i]),
        "costmap_update_map": (None, [vp, d, d, d, _i32p]),
        "costmap_get": (None, [vp, _u8p]),
        "costmap_set": (None, [vp, _u8p]),
        "layer_get": (None, [vp, i, _u8p]),
        "costmap_get_origin": (None, [vp, _f64p]),
        "inflation_tables": (i, [vp, i, _u8p, _f64p, i]),
        "interpret_values": (None, [_u8p, _u8p, C.c_int64, i, C.c_uint8, C.c_uint8, i]),
        "raytrace_cells": (i, [u, u, u, u, u, u, _u32p, i]),
        "footprint_radii": (None, [_f64p, i, _f64p, _f64p]),
        "dwa_default_config": (None, [C.POINTER(DwaConfig)]),
        "dwa_create": (vp, [C.POINTER(DwaConfig), u, u, d]),
        "dwa_destroy": (None, [vp]),
        "dwa_set_costmap": (None, [vp, _u8p, d, d]),
        "dwa_set_plan": (None, [vp, _f64p, _f64p, i]),
        "dwa_reset_oscillation": (None, [vp]),
        "dwa_get_oscillation_mask": (i, [vp]),
        "dwa_find_best_path": (i, [vp, _f64p, _f64p, _f64p, i, C.POINTER(DwaResult), _f64p, i, _f64p, i]),
        "dwa_check_trajectory": (d, [vp, _f64p, _f64p, _f64p, _f64p, i]),
        "dwa_get_grid": (None, [vp, i, _f64p]),
        "dwa_prepare_only": (None, [vp]),
        "velocity_samples": (i, [d, d, i, _f64p, i]),
        "line_cells": (i, [i, i, i, i, _i32p, i]),
        "mapgrid_bfs": (None, [_u8p, u, u, _i32p, i, i, _f64p]),
        "impl_name": (C.c_char_p, []),
        "project_scan": (i, [C.POINTER(LaserScan), C.POINTER(C.c_float), i, _f64p]),
    }
    # the legacy TrajectoryPlanner and the reconfigure entry points (both checkers export them; tolerated as missing for
    # an older prebuilt library)
    optional = {
        "tp_default_config": (None, [C.POINTER(TpConfig)]),
        "tp_create": (vp, [C.POINTER(TpConfig), u, u, d, _f64p, i]),
        "tp_destroy": (None, [vp]),
        "tp_set_costmap": (None, [vp, _u8p, d, d]),
        "tp_update_plan": (None, [vp, _f64p, i]),
        "tp_find_best_path": (i, [vp, _f64p, _f64p, C.POINTER(TpResult), _f64p, i]),
        "tp_score_trajectory": (d, [vp, _f64p, _f64p, _f64p]),
        "tp_reconfigure": (None, [vp, C.POINTER(TpConfig)]),
        "tp_set_footprint": (None, [vp, _f64p, i]),
        "dwa_reconfigure": (None, [vp, C.POINTER(DwaConfig)]),
        "tp_get_grid": (None, [vp, i, _f64p]),
        "plan_transform": (i, [_f64p, i, _f64p, _f64p, _f64p, d, _i32p, _f64p]),
        "plan_prune": (i, [_f64p, i, _f64p]),
    }
    for name, (res, args) in sig.items():
        f = g(name)
        f.restype = res
        f.argtypes = args
    for name, (res, args) in optional.items():
        if hasattr(lib, prefix + name):
            f = g(name)
            f.restype = res
            f.argtypes = args
    return sig


def reference_dir():
    """The checkout of the reference's sources (ROS navigation) that oracle/_ref is compiled from: the directory the
    NAVIGATION_REFERENCE environment variable names, or None.  Without it the checkers under oracle/_ref are not
    built and the tests that run them skip."""
    d = os.environ.get("NAVIGATION_REFERENCE")
    return d if d and os.path.isdir(d) else None


def make(*targets):
    """oracle/Makefile; the targets under oracle/_ref need reference_dir()."""
    ref = reference_dir()
    subprocess.check_call(["make", "-s", "-C", HERE, *targets] + ([f"REF={ref}"] if ref else []))


def build(kind="port"):
    make({"port": "oracle", "reference": "ref", "reference_hoisted": "ref_hoisted"}[kind])


def lib_path(kind):
    return {"port": os.path.join(HERE, "libnavoracle.so"), "reference": os.path.join(HERE, "_ref", "libnavref.so"),
            "reference_hoisted": os.path.join(HERE, "_ref", "libnavref_hoisted.so")}[kind]


def available(kind):
    return os.path.exists(lib_path(kind))


class Costmap:
    """LayeredCostmap-shaped handle over an oracle library."""

    def __init__(self, api, size_x, size_y, resolution, origin_x=0.0, origin_y=0.0, rolling=False,
                 track_unknown=False):
        self.api, self.lib = api, api.lib
        self.size_x, self.size_y, self.resolution = size_x, size_y, resolution
        self.h = C.c_void_p(self.lib.navo_costmap_create(size_x, size_y, resolution, origin_x, origin_y,
                                                         int(rolling), int(track_unknown)))
        self._keep = []

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.navo_costmap_destroy(self.h)
            self.h = None

    def add_grid_layer(self, policy):
        return self.lib.navo_costmap_add_grid_layer(self.h, policy)

    def add_obstacle_layer(self, combination_method=1, footprint_clearing=True, max_obstacle_height=2.0):
        return self.lib.navo_costmap_add_obstacle_layer(self.h, combination_method, int(footprint_clearing),
                                                        max_obstacle_height)

    def add_inflation_layer(self, inflation_radius=0.55, cost_scaling_factor=10.0):
        return self.lib.navo_costmap_add_inflation_layer(self.h, inflation_radius, cost_scaling_factor)

    def add_voxel_layer(self, combination_method=1, footprint_clearing=True, max_obstacle_height=2.0, origin_z=0.0,
                        z_resolution=0.2, z_voxels=10, unknown_threshold=15, mark_threshold=0):
        """VoxelLayer with cfg/VoxelPlugin.cfg's defaults."""
        return self.lib.navo_costmap_add_voxel_layer(self.h, combination_method, int(footprint_clearing),
                                                     max_obstacle_height, origin_z, z_resolution, z_voxels,
                                                     unknown_threshold, mark_threshold)

    def get_voxels(self, layer):
        out = np.zeros((self.size_y, self.size_x), dtype=np.uint32)
        self.lib.navo_layer_get_voxels(self.h, layer, _p(out, _u32p))
        return out

    def set_footprint(self, xy):
        a = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
        self.lib.navo_costmap_set_footprint(self.h, _p(a, _f64p), a.shape[0])

    def set_grid_layer(self, layer, data):
        a = np.ascontiguousarray(data, dtype=np.uint8)
        assert a.size == self.size_x * self.size_y
        self.lib.navo_grid_layer_set(self.h, layer, _p(a, _u8p))

    def touch_grid_layer(self, layer, x, y, w, h):
        self.lib.navo_grid_layer_touch(self.h, layer, x, y, w, h)

    def set_enabled(self, layer, enabled):
        self.lib.navo_layer_set_enabled(self.h, layer, int(enabled))

    def set_observations(self, layer, observations):
        """observations: list of dicts(origin=(x,y,z), points=(n,3) float32, obstacle_range, raytrace_range,
        marking=True, clearing=True)"""
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
        self.lib.navo_obstacle_set_observations(self.h, layer, arr, len(observations))

    def set_inflation_params(self, layer, inflation_radius, cost_scaling_factor):
        self.lib.navo_inflation_set_params(self.h, layer, inflation_radius, cost_scaling_factor)

    def set_inflation_variant(self, layer, variant, seed=0):
        """0 reference heap order, 1 FIFO, 2 LIFO, 3 seeded random, 4 exact nearest-seed, 5 level-synchronous"""
        if self.lib.navo_inflation_set_variant(self.h, layer, variant, seed) != 0:
            raise ValueError(f"inflation variant {variant} is not available in this checker")

    def inflation_last_rounds(self, layer):
        return int(self.lib.navo_inflation_last_rounds(self.h, layer))

    def update_map(self, x=0.0, y=0.0, yaw=0.0):
        w = np.zeros(4, dtype=np.int32)
        self.lib.navo_costmap_update_map(self.h, x, y, yaw, _p(w, _i32p))
        return tuple(int(v) for v in w)

    def get(self):
        out = np.empty((self.size_y, self.size_x), dtype=np.uint8)
        self.lib.navo_costmap_get(self.h, _p(out, _u8p))
        return out

    def set(self, grid):
        a = np.ascontiguousarray(grid, dtype=np.uint8)
        self.lib.navo_costmap_set(self.h, _p(a, _u8p))

    def get_layer(self, layer):
        out = np.empty((self.size_y, self.size_x), dtype=np.uint8)
        self.lib.navo_layer_get(self.h, layer, _p(out, _u8p))
        return out

    def origin(self):
        o = np.zeros(2)
        self.lib.navo_costmap_get_origin(self.h, _p(o, _f64p))
        return float(o[0]), float(o[1])

    def inflation_tables(self, layer):
        cap = 256 * 256
        costs = np.zeros(cap, dtype=np.uint8)
        dists = np.zeros(cap, dtype=np.float64)
        R = self.lib.navo_inflation_tables(self.h, layer, _p(costs, _u8p), _p(dists, _f64p), cap)
        n = R + 2
        return R, costs[:n * n].reshape(n, n).copy(), dists[:n * n].reshape(n, n).copy()


class Dwa:
    """DWAPlanner-shaped handle over an oracle library."""

    def __init__(self, api, size_x, size_y, resolution, **overrides):
        self.api, self.lib = api, api.lib
        self.size_x, self.size_y, self.resolution = size_x, size_y, resolution
        self.cfg = DwaConfig()
        self.lib.navo_dwa_default_config(C.byref(self.cfg))
        for k, v in overrides.items():
            setattr(self.cfg, k, v)
        self.h = C.c_void_p(self.lib.navo_dwa_create(C.byref(self.cfg), size_x, size_y, resolution))

    def reconfigure(self, **overrides):
        """DWAPlanner::reconfigure with the current configuration and `overrides` (same signature as
        navigation_b200.api.Dwa.reconfigure)."""
        cfg = DwaConfig.from_buffer_copy(self.cfg)
        for k, v in overrides.items():
            setattr(cfg, k, v)
        self.lib.navo_dwa_reconfigure(self.h, C.byref(cfg))
        self.cfg = cfg

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.navo_dwa_destroy(self.h)
            self.h = None

    def set_costmap(self, grid, origin_x=0.0, origin_y=0.0):
        a = np.ascontiguousarray(grid, dtype=np.uint8)
        assert a.size == self.size_x * self.size_y
        self.lib.navo_dwa_set_costmap(self.h, _p(a, _u8p), origin_x, origin_y)

    def set_plan(self, pose, plan_xy):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        a = np.ascontiguousarray(plan_xy, dtype=np.float64).reshape(-1, 2)
        self.lib.navo_dwa_set_plan(self.h, _p(p, _f64p), _p(a, _f64p), a.shape[0])

    def reset_oscillation(self):
        self.lib.navo_dwa_reset_oscillation(self.h)

    def oscillation_mask(self):
        return self.lib.navo_dwa_get_oscillation_mask(self.h)

    def check_trajectory(self, pose, vel, vel_samples, footprint_xy):
        """DWAPlanner::checkTrajectory: cost of the single trajectory for vel_samples (>= 0 means legal)."""
        p = np.ascontiguousarray(pose, dtype=np.float64)
        v = np.ascontiguousarray(vel, dtype=np.float64)
        s = np.ascontiguousarray(vel_samples, dtype=np.float64)
        f = np.ascontiguousarray(footprint_xy, dtype=np.float64).reshape(-1, 2)
        return float(self.lib.navo_dwa_check_trajectory(self.h, _p(p, _f64p), _p(v, _f64p), _p(s, _f64p), _p(f, _f64p),
                                                        f.shape[0]))

    def find_best_path(self, pose, vel, footprint_xy, max_samples=1 << 21, max_points=4096):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        v = np.ascontiguousarray(vel, dtype=np.float64)
        f = np.ascontiguousarray(footprint_xy, dtype=np.float64).reshape(-1, 2)
        res = DwaResult()
        costs = np.full(max_samples, np.nan)
        pts = np.zeros((max_points, 3))
        ok = self.lib.navo_dwa_find_best_path(self.h, _p(p, _f64p), _p(v, _f64p), _p(f, _f64p), f.shape[0],
                                              C.byref(res), _p(costs, _f64p), max_samples, _p(pts, _f64p), max_points)
        return dict(ok=bool(ok), cost=res.cost, xv=res.xv, yv=res.yv, thetav=res.thetav, best_index=res.best_index,
                    n_samples=res.n_samples, n_scored=res.n_scored, costs=costs[:res.n_samples].copy(),
                    points=pts[:res.n_points].copy())

    def grid(self, which):
        out = np.empty((self.size_y, self.size_x), dtype=np.float64)
        self.lib.navo_dwa_get_grid(self.h, which, _p(out, _f64p))
        return out

    def prepare_only(self):
        self.lib.navo_dwa_prepare_only(self.h)


def _tp_override(cfg, overrides):
    for k, v in overrides.items():
        if k == "y_vels":
            for j, y in enumerate(v):
                cfg.y_vels[j] = y
            cfg.n_y_vels = len(v)
        else:
            setattr(cfg, k, v)


class TrajectoryPlanner:
    """The legacy base_local_planner::TrajectoryPlanner."""

    def __init__(self, api, size_x, size_y, resolution, footprint_xy, **overrides):
        self.lib = api.lib
        self.size_x, self.size_y = size_x, size_y
        self.cfg = TpConfig()
        self.lib.navo_tp_default_config(C.byref(self.cfg))
        _tp_override(self.cfg, overrides)
        f = np.ascontiguousarray(footprint_xy, dtype=np.float64).reshape(-1, 2)
        self.h = C.c_void_p(self.lib.navo_tp_create(C.byref(self.cfg), size_x, size_y, resolution, _p(f, _f64p),
                                                    f.shape[0]))

    def reconfigure(self, **overrides):
        """TrajectoryPlanner::reconfigure with the current configuration and `overrides` (y_vels as a list; same
        signature as navigation_b200.api.TrajectoryPlanner.reconfigure)."""
        cfg = TpConfig.from_buffer_copy(self.cfg)
        _tp_override(cfg, overrides)
        self.lib.navo_tp_reconfigure(self.h, C.byref(cfg))
        self.cfg = cfg

    def set_footprint(self, xy):
        f = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
        self.lib.navo_tp_set_footprint(self.h, _p(f, _f64p), f.shape[0])

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.navo_tp_destroy(self.h)
            self.h = None

    def set_costmap(self, grid, origin_x=0.0, origin_y=0.0):
        a = np.ascontiguousarray(grid, dtype=np.uint8)
        assert a.size == self.size_x * self.size_y
        self.lib.navo_tp_set_costmap(self.h, _p(a, _u8p), origin_x, origin_y)

    def update_plan(self, plan_xy):
        a = np.ascontiguousarray(plan_xy, dtype=np.float64).reshape(-1, 2)
        self.lib.navo_tp_update_plan(self.h, _p(a, _f64p), a.shape[0])

    def find_best_path(self, pose, vel, max_points=4096):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        v = np.ascontiguousarray(vel, dtype=np.float64)
        res = TpResult()
        pts = np.zeros((max_points, 3))
        self.lib.navo_tp_find_best_path(self.h, _p(p, _f64p), _p(v, _f64p), C.byref(res), _p(pts, _f64p), max_points)
        return dict(cost=res.cost, xv=res.xv, yv=res.yv, thetav=res.thetav, flags=res.flags,
                    points=pts[:res.n_points].copy())

    def score_trajectory(self, pose, vel, vel_samples):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        v = np.ascontiguousarray(vel, dtype=np.float64)
        s = np.ascontiguousarray(vel_samples, dtype=np.float64)
        return float(self.lib.navo_tp_score_trajectory(self.h, _p(p, _f64p), _p(v, _f64p), _p(s, _f64p)))

    def grid(self, which):
        out = np.empty((self.size_y, self.size_x), dtype=np.float64)
        self.lib.navo_tp_get_grid(self.h, which, _p(out, _f64p))
        return out


class Api:
    def __init__(self, kind):
        self.kind = kind
        self.lib = C.CDLL(lib_path(kind))
        _declare(self.lib, "navo_")
        self.name = self.lib.navo_impl_name().decode()

    def costmap(self, *a, **k):
        return Costmap(self, *a, **k)

    def dwa(self, *a, **k):
        return Dwa(self, *a, **k)

    def trajectory_planner(self, *a, **k):
        return TrajectoryPlanner(self, *a, **k)

    def plans_transform(self, plans, robot_xy, transforms, thresholds):
        """transformGlobalPlan plan by plan (same shape as navigation_b200.api.Api.plans_transform)."""
        first, outs = [], []
        for k, p in enumerate(plans):
            a = np.zeros((len(p), 3))
            q = np.asarray(p, dtype=np.float64).reshape(len(p), -1) if len(p) else np.zeros((0, 3))
            a[:, :q.shape[1]] = q
            a = np.ascontiguousarray(a)
            rob = np.ascontiguousarray(robot_xy[k], dtype=np.float64)
            tf = np.ascontiguousarray(transforms[k], dtype=np.float64).reshape(12)
            m, t = np.ascontiguousarray(tf[:9]), np.ascontiguousarray(tf[9:])
            f = np.zeros(1, dtype=np.int32)
            out = np.zeros_like(a)
            n = self.lib.navo_plan_transform(_p(a, _f64p), len(a), _p(rob, _f64p), _p(m, _f64p), _p(t, _f64p),
                                             float(thresholds[k]), _p(f, _i32p), _p(out, _f64p))
            first.append(int(f[0]))
            outs.append(out[:n].copy())
        return np.array(first, dtype=np.int32), outs

    def plans_prune(self, plans, robot_xy):
        out = []
        for k, p in enumerate(plans):
            a = np.zeros((len(p), 3))
            q = np.asarray(p, dtype=np.float64).reshape(len(p), -1) if len(p) else np.zeros((0, 3))
            a[:, :q.shape[1]] = q
            a = np.ascontiguousarray(a)
            rob = np.ascontiguousarray(robot_xy[k], dtype=np.float64)
            out.append(self.lib.navo_plan_prune(_p(a, _f64p), len(a), _p(rob, _f64p)))
        return np.array(out, dtype=np.int32)

    def interpret_values(self, values, track_unknown=True, unknown_cost_value=255, lethal_threshold=100,
                         trinary=True):
        a = np.ascontiguousarray(values, dtype=np.uint8)
        out = np.empty_like(a)
        self.lib.navo_interpret_values(_p(a, _u8p), _p(out, _u8p), a.size, int(track_unknown), unknown_cost_value,
                                       lethal_threshold, int(trinary))
        return out

    def raytrace_cells(self, size_x, x0, y0, x1, y1, max_length=0xFFFFFFFF):
        cap = 1 << 16
        out = np.zeros(cap, dtype=np.uint32)
        n = self.lib.navo_raytrace_cells(size_x, x0, y0, x1, y1, max_length, _p(out, _u32p), cap)
        return out[:n].copy()

    def voxel_line_cells(self, size_x, p0, p1, max_length=0xFFFFFFFF):
        """Voxels visited by VoxelGrid::raytraceLine from p0 to p1 (float voxel coordinates): (offset, z) rows."""
        cap = 1 << 14
        off = np.zeros(cap, dtype=np.uint32)
        z = np.zeros(cap, dtype=np.int32)
        n = self.lib.navo_voxel_line_cells(size_x, *[float(v) for v in p0], *[float(v) for v in p1], max_length,
                                           _p(off, _u32p), _p(z, _i32p), cap)
        return np.stack([off[:n].astype(np.int64), z[:n].astype(np.int64)], 1)

    def project_scan(self, scan):
        """Observation ingest restated (oracle/scan_ingest_restated.h): scan = dict(ranges, angle_min, angle_increment,
        range_min, range_max, translation, rotation_xyzw, min_obstacle_height, max_obstacle_height, inf_is_valid);
        returns (origin, float32 (n, 3) world-frame cloud)."""
        s = LaserScan()
        if "points" in scan:  # a PointCloud(2) source: (n, 3) float32 in the sensor frame
            r = np.ascontiguousarray(scan["points"], dtype=np.float32).reshape(-1, 3)
            s.is_cloud = 1
        else:
            r = np.ascontiguousarray(scan["ranges"], dtype=np.float32)
            s.is_cloud = 0
            s.angle_min, s.angle_increment = scan["angle_min"], scan["angle_increment"]
            s.range_min, s.range_max = scan["range_min"], scan["range_max"]
        s.ranges = r.ctypes.data_as(C.POINTER(C.c_float))
        s.n_ranges = len(r)
        s.inf_is_valid = int(scan.get("inf_is_valid", 0))
        for k in range(3):
            s.translation[k] = scan["translation"][k]
        for k in range(4):
            s.rotation_xyzw[k] = scan["rotation_xyzw"][k]
        s.min_obstacle_height, s.max_obstacle_height = scan["min_obstacle_height"], scan["max_obstacle_height"]
        out = np.zeros((max(1, len(r)), 3), dtype=np.float32)
        origin = np.zeros(3)
        n = self.lib.navo_project_scan(C.byref(s), out.ctypes.data_as(C.POINTER(C.c_float)), len(r), _p(origin, _f64p))
        return tuple(origin), out[:n].copy()

    def footprint_radii(self, xy):
        a = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
        i, c = C.c_double(), C.c_double()
        self.lib.navo_footprint_radii(_p(a, _f64p), a.shape[0], C.byref(i), C.byref(c))
        return i.value, c.value

    def velocity_samples(self, vmin, vmax, n):
        out = np.zeros(max(8, 2 * n + 8))
        k = self.lib.navo_velocity_samples(vmin, vmax, n, _p(out, _f64p), out.size)
        return out[:k].copy()

    def line_cells(self, x0, y0, x1, y1):
        cap = 1 << 14
        out = np.zeros((cap, 2), dtype=np.int32)
        n = self.lib.navo_line_cells(x0, y0, x1, y1, _p(out, _i32p), cap)
        return out[:n].copy()

    def mapgrid_bfs(self, costs, seeds_xy, allow_unknown=False):
        a = np.ascontiguousarray(costs, dtype=np.uint8)
        sy, sx = a.shape
        s = np.ascontiguousarray(seeds_xy, dtype=np.int32).reshape(-1, 2)
        out = np.empty((sy, sx), dtype=np.float64)
        self.lib.navo_mapgrid_bfs(_p(a, _u8p), sx, sy, _p(s, _i32p), s.shape[0], int(allow_unknown), _p(out, _f64p))
        return out


class GoalRef:
    """The reference's own transformGlobalPlan / prunePlan (oracle/_ref/libgoalref.so, `make -C oracle goalref`); same
    call shapes as Api.plans_transform / plans_prune.  Thresholds must be multiples of 0.5 (the harness expresses them
    as a costmap size)."""

    PATH = os.path.join(HERE, "_ref", "libgoalref.so")

    def __init__(self):
        self.lib = C.CDLL(self.PATH)
        self.lib.navref_plan_transform.restype = C.c_int
        self.lib.navref_plan_transform.argtypes = [_f64p, C.c_int, _f64p, _f64p, _f64p, C.c_double, _i32p, _f64p]
        self.lib.navref_plan_prune.restype = C.c_int
        self.lib.navref_plan_prune.argtypes = [_f64p, C.c_int, _f64p]

    @classmethod
    def available(cls):
        return os.path.exists(cls.PATH)

    @staticmethod
    def _xyz(p):
        a = np.zeros((len(p), 3))
        q = np.asarray(p, dtype=np.float64).reshape(len(p), -1) if len(p) else np.zeros((0, 3))
        a[:, :q.shape[1]] = q
        return np.ascontiguousarray(a)

    def plans_transform(self, plans, robot_xy, transforms, thresholds):
        outs = []
        for k, p in enumerate(plans):
            a = self._xyz(p)
            rob = np.ascontiguousarray(robot_xy[k], dtype=np.float64)
            tf = np.ascontiguousarray(transforms[k], dtype=np.float64).reshape(12)
            m, t = np.ascontiguousarray(tf[:9]), np.ascontiguousarray(tf[9:])
            f = np.zeros(1, dtype=np.int32)
            out = np.zeros_like(a)
            n = self.lib.navref_plan_transform(_p(a, _f64p), len(a), _p(rob, _f64p), _p(m, _f64p), _p(t, _f64p),
                                               float(thresholds[k]), _p(f, _i32p), _p(out, _f64p))
            assert n >= 0 or len(a) == 0, f"navref_plan_transform failed ({n})"
            outs.append(out[:max(n, 0)].copy())
        return outs

    def plans_prune(self, plans, robot_xy):
        return np.array([self.lib.navref_plan_prune(_p(self._xyz(p), _f64p), len(p),
                                                    _p(np.ascontiguousarray(robot_xy[k], dtype=np.float64), _f64p))
                         for k, p in enumerate(plans)], dtype=np.int32)


_cache = {}


def load(kind="port"):
    if kind not in _cache:
        if not available(kind):
            build(kind)
        _cache[kind] = Api(kind)
    return _cache[kind]
