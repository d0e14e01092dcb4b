"""Voxel sensing fleets (navgpu_fleet_create_sensing_voxel): every robot's rolling local costmap [VoxelLayer,
InflationLayer] built on the device from its own scans and 3-D clouds, then DWAPlanner::findBestPath on it.

1. Against one navgpu_costmap per robot (rolling, add_voxel_layer + add_inflation_layer) fed the identical scans:
   window, origin, the VoxelLayer's 2-D grid, its columns and the master grid bit-exact every cycle, over moving
   robots, LaserScan and 3-D cloud sources and the edge robots of the 2-D fleet's test.
2. Against the CPU checker robot by robot (its rolling LayeredCostmap with a VoxelLayer and the exact windowed inflation,
   then its DWAPlanner): costmaps and columns bit-exact; best index, sample counts, oscillation masks and velocities
   equal; cost within 1e-5 relative.  PointCloud sources only, as in test_gpu_fleet_sensing.py.
3. The benched configuration (tools/bench_fleet_sensing.py --voxel), sampled through the checker.
4. Argument errors, what one CTA cannot hold, and 2-D and voxel fleets sharing a process."""
import numpy as np
import pytest

import scenarios as sc
from navigation_b200 import synth
from navigation_b200.api import NavGpuError
from test_gpu_fleet_sensing import CFG, RES, assert_result, edge_pose, single_costmap

pytestmark = pytest.mark.gpu

VOXEL = dict(origin_z=0.0, z_resolution=0.2, z_voxels=10, unknown_threshold=15, mark_threshold=0)


def single_voxel_costmap(api, sx, sy, voxel, track_unknown=False, combination_method=1, footprint_clearing=True,
                         inflation_radius=0.55, cost_scaling_factor=10.0):
    """One robot's local costmap with map_type: voxel -- rolling, [VoxelLayer, InflationLayer]."""
    v = {**VOXEL, **voxel}
    cm = api.costmap(sx, sy, RES, 0.0, 0.0, rolling=True, track_unknown=track_unknown)
    o = cm.add_voxel_layer(combination_method, footprint_clearing, 2.0, v["origin_z"], v["z_resolution"],
                           v["z_voxels"], v["unknown_threshold"], v["mark_threshold"])
    il = cm.add_inflation_layer(inflation_radius, cost_scaling_factor)
    cm.set_footprint(sc.PENTAGON)
    return cm, o, il


def edge_sources(robots, i, cycle):
    """Robot 0 has no sources; robot 2's leave it after its jump; robot 3 has a second source whose sensor is off the
    map.  3-D clouds and LaserScans alternate between cycles and robots."""
    if i == 0 or (i == 2 and cycle >= 3):
        return []
    c = 0 if i == 1 else cycle
    three_d = (i + cycle) % 2 == 1
    out = [synth.fleet_cloud_3d(robots[i], c) if three_d else synth.fleet_scan(robots[i], c)]
    if i == 3:
        far = synth.fleet_cloud_3d(robots[i], cycle) if not three_d else synth.fleet_scan(robots[i], cycle, cloud=True)
        far["translation"] = (far["translation"][0] + 20.0, far["translation"][1], far["translation"][2])
        out.append(far)
    return out


@pytest.mark.parametrize("size,opts,voxel", [
    ((120, 120), dict(), dict()),
    ((120, 120), dict(track_unknown=True), dict(unknown_threshold=8, z_voxels=16)),
    ((120, 120), dict(combination_method=0), dict(origin_z=-0.1, z_voxels=4)),
    ((120, 120), dict(footprint_clearing=False), dict()),
    ((97, 131), dict(), dict()),
    ((120, 120), dict(inflation_radius=2.975, cost_scaling_factor=3.0), dict()),  # a cell radius of 60
], ids=["defaults", "track_unknown", "overwrite_low_column", "no_footprint_clearing", "97x131", "R60"])
def test_voxel_fleet_matches_single_costmaps(cuda, size, opts, voxel):
    sx, sy = size
    n, cycles = 6, 6
    zv = {**VOXEL, **voxel}["z_voxels"]
    robots = [synth.fleet_voxel_robot(40 + i, n=max(sx, sy)) for i in range(n)]
    fleet = cuda.fleet_sensing(n, sx, sy, RES, sc.PENTAGON, voxel=voxel, **opts, **CFG)
    flat = cuda.fleet_sensing(n, sx, sy, RES, sc.PENTAGON, **opts, **CFG)  # a 2-D ObstacleLayer fed the same sources
    singles = [single_voxel_costmap(cuda, sx, sy, voxel, **opts) for _ in range(n)]
    plans = [r["plan"] for r in robots]
    fleet.set_plans(np.array([edge_pose(robots, i, 0) for i in range(n)]), plans)
    flat.set_plans(np.array([edge_pose(robots, i, 0) for i in range(n)]), plans)
    seen = dict(marked=0, cleared=0, unknown=0, lethal=0, inflated=0, kept_over_2d=0)
    for cycle in range(cycles):
        scans = [edge_sources(robots, i, cycle) for i in range(n)]
        poses = np.array([edge_pose(robots, i, cycle) for i in range(n)])
        vels = np.array([r["vel"] for r in robots])
        for f in (fleet, flat):
            f.set_scans(scans)
            f.step(poses, vels)
        for i, (cm, o, _) in enumerate(singles):
            if scans[i]:
                cm.set_scans(o, scans[i])
            else:
                cm.set_observations(o, [])
            win = cm.update_map(*poses[i])
            where = f"cycle {cycle} robot {i}"
            origin, fwin = fleet.geometry(i)
            assert fwin == win, f"{where}: window {fwin} vs {win}"
            assert origin == cm.origin(), f"{where}: origin {origin} vs {cm.origin()}"
            layer, cols, master = fleet.layer(i), fleet.voxels(i), fleet.costmap(i)
            assert np.array_equal(layer, cm.get_layer(o)), f"{where}: voxel layer's grid differs"
            assert np.array_equal(cols, cm.get_voxels(o)), f"{where}: voxel columns differ"
            assert np.array_equal(master, cm.get()), f"{where}: master grid differs"
            in_column = np.uint32((1 << zv) - 1)
            seen["marked"] += int(((cols >> 16) & in_column).astype(bool).sum())
            seen["cleared"] += int((~cols & in_column).astype(bool).sum())
            touched = (cols & in_column) != in_column  # a ray reached the column
            seen["unknown"] += int(((layer == 255) & touched).sum())
            seen["lethal"] += int((master == 254).sum())
            seen["inflated"] += int(((master > 0) & (master < 253)).sum())
            seen["kept_over_2d"] += int(((layer == 254) & (flat.layer(i) == 0)).sum())
    # the scenario exercised what it claims
    assert seen["marked"] and seen["cleared"] and seen["lethal"] and seen["inflated"], seen
    if opts.get("track_unknown"):  # cells a ray reached that still hold too many unknown voxels
        assert seen["unknown"], seen
    assert seen["kept_over_2d"], seen  # obstacles a ray passed over or under: cleared in 2-D, kept in 3-D


def checker_robot(port, sx, sy):
    cm = port.costmap(sx, sy, RES, 0.0, 0.0, rolling=True)
    o = cm.add_voxel_layer(1, True, 2.0, **VOXEL)
    il = cm.add_inflation_layer(0.55, 10.0)
    sc.select_inflation(cm, il, "exact")
    cm.set_footprint(sc.PENTAGON)
    return cm, o


def checker_cycle(port, cm, o, scans, pose, plan, vel, d):
    """One robot's updateMap (with the checker's projection of the clouds as observations) and findBestPath."""
    obs = []
    for s_ in scans:
        org, pts = port.project_scan(s_)
        obs.append(dict(origin=org, points=pts, obstacle_range=s_["obstacle_range"],
                        raytrace_range=s_["raytrace_range"], marking=s_["marking"], clearing=s_["clearing"]))
    cm.set_observations(o, obs)
    win = cm.update_map(*pose)
    grid = cm.get()
    d.set_costmap(grid, *cm.origin())
    d.set_plan(pose, plan)
    return win, grid, d.find_best_path(pose, vel, sc.PENTAGON)


def test_voxel_fleet_matches_checker_robot_by_robot(cuda, port):
    sx = sy = 120
    n, cycles = 8, 5
    robots = [synth.fleet_voxel_robot(200 + i) for i in range(n)]
    fleet = cuda.fleet_sensing(n, sx, sy, RES, sc.PENTAGON, voxel=VOXEL, **CFG)
    refs = [checker_robot(port, sx, sy) for _ in range(n)]
    dwas = [port.dwa(sx, sy, RES, **CFG) for _ in range(n)]
    vels = np.array([r["vel"] for r in robots])
    valid = exact = 0
    for cycle in range(cycles):
        poses = np.array([r["poses"][cycle] for r in robots])
        scans = [[synth.fleet_cloud_3d(r, cycle)] for r in robots]
        fleet.set_scans(scans)
        fleet.set_plans(poses, [r["plan"] for r in robots])
        out = fleet.step(poses, vels)
        for i, ((cm, o), d) in enumerate(zip(refs, dwas)):
            win, grid, e = checker_cycle(port, cm, o, scans[i], poses[i], robots[i]["plan"], vels[i], d)
            assert fleet.geometry(i) == (cm.origin(), win), f"cycle {cycle} robot {i}"
            assert np.array_equal(fleet.layer(i), cm.get_layer(o)), f"cycle {cycle} robot {i}: voxel layer differs"
            assert np.array_equal(fleet.voxels(i), cm.get_voxels(o)), f"cycle {cycle} robot {i}: columns differ"
            assert np.array_equal(fleet.costmap(i), grid), f"cycle {cycle} robot {i}: master grid differs"
            v, x = assert_result(out[i], e, fleet, d, (cycle, i))
            valid, exact = valid + v, exact + x
        for i, g in enumerate(out):  # alternate the commanded direction so oscillation flags latch on some robots
            if g["cost"] >= 0:
                vels[i] = [g["xv"] * (-1 if cycle % 2 else 1), g["yv"], -g["thetav"]]
    assert valid > 0 and exact >= 0.99 * valid


def test_full_voxel_fleet_sampled_parity(cuda, port):
    """The benched configuration: 4096 robots, 120 x 120 at 0.05 m, [VoxelLayer, InflationLayer], 20 x 1 x 20 samples,
    one fresh 3-D cloud per robot; one step, every 64th robot replayed through the checker."""
    cfg = dict(vx_samples=20, vy_samples=1, vth_samples=20, max_vel_y=0.0, min_vel_y=0.0)
    n, sx, sy = 4096, 120, 120
    robots = [synth.fleet_voxel_robot(i) for i in range(n)]
    fleet = cuda.fleet_sensing(n, sx, sy, RES, sc.PENTAGON, voxel=VOXEL, **cfg)
    poses = np.array([r["poses"][0] for r in robots])
    vels = np.array([r["vel"] for r in robots])
    scans = [[synth.fleet_cloud_3d(r, 0)] for r in robots]
    fleet.set_scans(scans)
    fleet.set_plans(poses, [r["plan"] for r in robots])
    out = fleet.step(poses, vels)
    valid = exact = 0
    for i in range(0, n, 64):
        cm, o = checker_robot(port, sx, sy)
        d = port.dwa(sx, sy, RES, **cfg)
        win, grid, e = checker_cycle(port, cm, o, scans[i], poses[i], robots[i]["plan"], vels[i], d)
        assert fleet.geometry(i) == (cm.origin(), win), f"robot {i}"
        assert np.array_equal(fleet.voxels(i), cm.get_voxels(o)), f"robot {i}: columns differ"
        assert np.array_equal(fleet.costmap(i), grid), f"robot {i}: master grid differs"
        v, x = assert_result(out[i], e, fleet, d, (0, i))
        valid, exact = valid + v, exact + x
    assert valid >= 32 and exact >= 0.99 * valid


def test_errors(cuda):
    fp = sc.PENTAGON
    for bad in (dict(z_voxels=17), dict(z_voxels=-1), dict(z_resolution=0.0), dict(unknown_threshold=-1),
                dict(mark_threshold=-1)):
        with pytest.raises(NavGpuError, match="navgpu error 2"):
            cuda.fleet_sensing(2, 40, 40, RES, fp, voxel=bad, **CFG)
    # a positive mark_threshold is refused like navgpu_costmap_add_voxel_layer refuses it
    with pytest.raises(NavGpuError, match="navgpu error 3.*mark_threshold"):
        cuda.fleet_sensing(2, 40, 40, RES, fp, voxel=dict(mark_threshold=1), **CFG)
    with pytest.raises(NavGpuError, match="navgpu error 3.*mark_threshold"):
        single_voxel_costmap(cuda, 40, 40, dict(mark_threshold=1))
    with pytest.raises(NavGpuError, match="navgpu error 2"):
        cuda.fleet_sensing(2, 40, 40, RES, fp, combination_method=2, voxel=VOXEL, **CFG)
    raw = cuda.fleet(2, 40, 40, RES, fp, **CFG)
    flat = cuda.fleet_sensing(2, 40, 40, RES, fp, **CFG)
    vox = cuda.fleet_sensing(2, 40, 40, RES, fp, voxel=VOXEL, **CFG)
    for f in (raw, flat):
        with pytest.raises(NavGpuError, match="navgpu error 2"):
            f.voxels(0)
    with pytest.raises(NavGpuError, match="navgpu error 2"):
        vox.set_maps(np.zeros((2, 40, 40), np.uint8), np.zeros((2, 2)))
    with pytest.raises(NavGpuError, match="navgpu error 2"):
        vox.voxels(2)
    # before any step every column is unknown, as VoxelGrid starts
    assert (vox.voxels(1) == 0x0000ffff).all()
    # the columns add 4 B per cell to what one CTA holds: 200 x 200 fits a 2-D sensing fleet, not a voxel fleet
    with pytest.raises(NavGpuError, match="navgpu error 3.*shared memory"):
        cuda.fleet_sensing(2, 200, 200, RES, fp, voxel=VOXEL, **CFG)
    cuda.fleet_sensing(2, 200, 200, RES, fp, **CFG)


def test_flat_and_voxel_fleets_in_one_process(cuda):
    """Each kernel keeps its own shared-memory limit: a 200 x 200 2-D sensing fleet and a 120 x 120 voxel fleet,
    stepped alternately, both still equal their single costmaps."""
    flat_r = [synth.fleet_sensing_robot(300 + i, n=200) for i in range(2)]
    vox_r = [synth.fleet_voxel_robot(310 + i) for i in range(2)]
    flat = cuda.fleet_sensing(2, 200, 200, RES, sc.PENTAGON, inflation_radius=1.0, **CFG)
    vox = cuda.fleet_sensing(2, 120, 120, RES, sc.PENTAGON, voxel=VOXEL, **CFG)
    ref = {"flat": [single_costmap(cuda, 200, 200, inflation_radius=1.0) for _ in range(2)],
           "voxel": [single_voxel_costmap(cuda, 120, 120, VOXEL) for _ in range(2)]}
    for fl, robots in ((flat, flat_r), (vox, vox_r)):
        fl.set_plans(np.array([r["poses"][0] for r in robots]), [r["plan"] for r in robots])
    for cycle in range(3):
        for name, fl, robots in (("flat", flat, flat_r), ("voxel", vox, vox_r)):
            scans = [[synth.fleet_scan(r, cycle) if name == "flat" else synth.fleet_cloud_3d(r, cycle)] for r in robots]
            poses = np.array([r["poses"][cycle] for r in robots])
            fl.set_scans(scans)
            fl.step(poses, np.array([r["vel"] for r in robots]))
            for i, (cm, o, _) in enumerate(ref[name]):
                cm.set_scans(o, scans[i])
                win = cm.update_map(*poses[i])
                assert fl.geometry(i) == (cm.origin(), win), f"{name} cycle {cycle} robot {i}"
                assert np.array_equal(fl.costmap(i), cm.get()), f"{name} cycle {cycle} robot {i}: master grid differs"
                if name == "voxel":
                    assert np.array_equal(fl.voxels(i), cm.get_voxels(o)), f"voxel cycle {cycle} robot {i}: columns"
