"""Voxel sensing fleets without a GPU: the constructor refuses to run without a device (no CPU fallback), and the seeded
3-D worlds and clouds the tests and tools/bench_fleet_sensing.py --voxel feed them are reproducible, well formed and
cover what a VoxelLayer treats differently from a 2-D ObstacleLayer."""
import numpy as np
import pytest

import scenarios as sc
from navigation_b200 import synth

RES, N, Z_RES, MAX_H = 0.05, 120, 0.2, 2.0


def test_fleet_sensing_voxel_needs_a_device():
    import navigation_b200
    a = navigation_b200.load()
    if a.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(navigation_b200.api.NavGpuError, match="no CUDA device"):
        a.fleet_sensing(2, 120, 120, RES, sc.PENTAGON, voxel=dict(z_voxels=10))


def world_points(cloud):
    """The cloud in the world frame (a yaw-only sensor rotation) and the sensor position."""
    x, y, z = cloud["translation"]
    qz, qw = cloud["rotation_xyzw"][2:]
    yaw = 2 * np.arctan2(qz, qw)
    p = cloud["points"].astype(np.float64)
    cs, sn = np.cos(yaw), np.sin(yaw)
    return np.stack([x + cs * p[:, 0] - sn * p[:, 1], y + sn * p[:, 0] + cs * p[:, 1], z + p[:, 2]], 1), (x, y, z)


def dominant_axes(pts, sensor, origin_z=0.0):
    """Which axis dominates each ray's voxel walk (VoxelLayer::raytraceFreespace: the end point pulled 2 cells towards
    the sensor, clipped to [origin_z, max_obstacle_height - 0.01]; cells of RES x RES x Z_RES)."""
    s = np.asarray(sensor)
    d = pts - s
    dist = np.linalg.norm(d, axis=1)
    e = s + d * np.clip((dist - 2 * RES) / dist, 0, 1)[:, None]
    c = e[:, 2] - s[2]
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.where(e[:, 2] > MAX_H, (MAX_H - 0.01 - s[2]) / c, np.where(e[:, 2] < origin_z, (origin_z - s[2]) / c, 1.0))
    e = s + (e - s) * np.clip(t, 0, 1)[:, None]
    cell = lambda v: np.floor(np.stack([v[..., 0] / RES, v[..., 1] / RES, (v[..., 2] - origin_z) / Z_RES], -1))
    ad = np.abs(cell(e) - cell(s))
    return np.where(ad[:, 0] >= np.maximum(ad[:, 1], ad[:, 2]), 0, np.where(ad[:, 1] >= ad[:, 2], 1, 2))


def test_fleet_voxel_inputs_are_seeded_and_well_formed():
    r, again = synth.fleet_voxel_robot(7), synth.fleet_voxel_robot(7)
    flat = synth.fleet_sensing_robot(7)
    assert np.array_equal(r["world"], flat["world"]) and np.array_equal(r["poses"], flat["poses"])
    assert np.array_equal(r["top"], again["top"]) and np.array_equal(r["bottom"], again["bottom"])
    c, c2 = synth.fleet_cloud_3d(r, 5), synth.fleet_cloud_3d(again, 5)
    assert np.array_equal(c["points"], c2["points"])
    assert not np.array_equal(c["points"], synth.fleet_cloud_3d(r, 6)["points"])
    n_rows = len(synth.VOXEL_ELEVATIONS)
    assert c["points"].shape == (n_rows * 180, 3) and c["points"].dtype == np.float32
    assert np.isfinite(c["points"]).all()
    res, (ox, oy) = r["resolution"], r["origin"]
    for x, y, _ in r["poses"]:  # the robot drives through free space, 12 cells from any column
        cx, cy = int((x - ox) / res), int((y - oy) / res)
        assert np.isneginf(r["top"][cy - 11:cy + 12, cx - 11:cx + 12]).all()


@pytest.mark.parametrize("robot_id", [0, 7, 123])
def test_fleet_voxel_inputs_cover_the_voxel_cases(robot_id):
    r = synth.fleet_voxel_robot(robot_id)
    res, (ox, oy) = r["resolution"], r["origin"]
    axes = np.zeros(3, int)
    above = below = floor = 0
    low_marked = passed_over = False
    low = (r["top"] > 0) & (r["top"] < 0.3)  # below the sensor: the scan plane passes over it
    assert low.any() and ((r["bottom"] > 0.3) & np.isfinite(r["top"])).any()  # the low box and the overhang exist
    for cycle in range(0, 6):
        cloud = synth.fleet_cloud_3d(r, cycle)
        pts, sensor = world_points(cloud)
        axes += np.bincount(dominant_axes(pts, sensor), minlength=3)
        above += int((pts[:, 2] > MAX_H).sum())
        below += int((pts[:, 2] < 0.0).sum())
        floor += int((np.abs(pts[:, 2]) <= 0.03).sum())
        mx = np.floor((pts[:, 0] - ox) / res).astype(int)
        my = np.floor((pts[:, 1] - oy) / res).astype(int)
        ok = (mx >= 0) & (mx < low.shape[1]) & (my >= 0) & (my < low.shape[0])
        near = np.linalg.norm(pts - np.asarray(sensor), axis=1) < cloud["obstacle_range"]
        low_marked |= bool((low[my[ok & near], mx[ok & near]]).any())
        # scan-plane rays that cross a low cell before their end, inside raytrace_range
        plane = np.abs(pts[:, 2] - sensor[2]) < 1e-4
        for p in pts[plane]:
            d = np.hypot(p[0] - sensor[0], p[1] - sensor[1])
            s = np.arange(0.0, min(d, cloud["raytrace_range"]) - 3 * res, 0.5 * res)
            cx = np.floor((sensor[0] + (p[0] - sensor[0]) * s / d - ox) / res).astype(int)
            cy = np.floor((sensor[1] + (p[1] - sensor[1]) * s / d - oy) / res).astype(int)
            passed_over |= bool(low[cy, cx].any())
    assert (axes > 0).all(), f"rays by dominant axis (x, y, z): {axes}"
    assert above > 0 and below > 0 and floor > 0
    assert low_marked and passed_over


def test_fleet_cloud_3d_is_cheap_for_a_fleet():
    """Generating one cycle for 4096 robots has to stay a matter of seconds (the benchmark makes several)."""
    import time
    robots = [synth.fleet_voxel_robot(i) for i in range(32)]
    t = time.perf_counter()
    for rb in robots:
        synth.fleet_cloud_3d(rb, 0)
    assert (time.perf_counter() - t) / 32 * 4096 < 120
