"""Sensing fleets (navgpu_fleet_create_sensing): every robot's rolling local costmap [ObstacleLayer, InflationLayer] built
on the device from its own scans, then DWAPlanner::findBestPath on it.

1. Against one navgpu_costmap per robot (rolling, obstacle + inflation layer) fed the identical scans: window, origin,
   obstacle grid and master grid bit-exact every cycle, over moving robots, LaserScan and PointCloud sources and the
   edge cases (track_unknown, both combination methods, no footprint clearing, an odd map size, a robot without
   scans, a sensor off the map, a robot that stands still, a jump of more than a map width).
2. Against the CPU checker robot by robot (its rolling LayeredCostmap with the exact windowed inflation, then its
   DWAPlanner): costmaps bit-exact; best index, sample counts, oscillation masks and velocities equal; cost within
   1e-5 relative.  PointCloud sources only: a LaserScan's projection may differ from glibc's by one float ulp
   (test_gpu_scan_ingest.py)."""
import ctypes

import numpy as np
import pytest

import scenarios as sc
from navigation_b200 import synth
from navigation_b200.api import NavGpuError, pack_scans

pytestmark = pytest.mark.gpu

RTOL = 1e-5
RES = 0.05
CFG = dict(vx_samples=6, vy_samples=1, vth_samples=11, max_vel_y=0.0, min_vel_y=0.0)
CELL_RADII = {1.575: 32, 2.975: 60, 12.675: 254}  # inflation radius -> the cell radius it was chosen for


def single_costmap(api, sx, sy, track_unknown=False, combination_method=1, footprint_clearing=True,
                   inflation_radius=0.55, cost_scaling_factor=10.0):
    """One robot's local costmap as move_base configures it: rolling, [ObstacleLayer, InflationLayer]."""
    cm = api.costmap(sx, sy, RES, 0.0, 0.0, rolling=True, track_unknown=track_unknown)
    o = cm.add_obstacle_layer(combination_method, footprint_clearing, 2.0)
    il = cm.add_inflation_layer(inflation_radius, cost_scaling_factor)
    cm.set_footprint(sc.PENTAGON)
    return cm, o, il


def edge_pose(robots, i, cycle):
    """Robot 1 stands still, robot 2 jumps 2.5 map widths at cycle 3, the others drive their path."""
    p = robots[i]["poses"][0 if i == 1 else cycle].copy()
    if i == 2 and cycle >= 3:
        p[0] += 15.0
    return p


def edge_scans(robots, i, cycle):
    """Robot 0 has no scans; robot 3 has a second source whose sensor is off the map; LaserScan and PointCloud sources
    alternate between cycles and robots."""
    if i == 0:
        return []
    out = [synth.fleet_scan(robots[i], 0 if i == 1 else cycle, cloud=(i + cycle) % 2 == 1)]
    if i == 2 and cycle >= 3:
        out = []  # its sensor is where it was: the jump leaves an empty map
    if i == 3:
        far = synth.fleet_scan(robots[i], cycle, cloud=cycle % 2 == 0)
        far["translation"] = (far["translation"][0] + 20.0, far["translation"][1], 0.3)
        out.append(far)
    return out


@pytest.mark.parametrize("size,opts", [
    ((120, 120), dict()),
    ((120, 120), dict(track_unknown=True)),
    ((120, 120), dict(combination_method=0)),
    ((120, 120), dict(footprint_clearing=False, track_unknown=True)),
    ((97, 131), dict(combination_method=0)),
    # cell radii of 32, 60 and 254 (radius (R - 0.5) x resolution): the horizontal seed search reads a second 32-cell
    # word, and more
    ((120, 120), dict(inflation_radius=1.575, cost_scaling_factor=1.0)),
    ((120, 120), dict(inflation_radius=2.975, cost_scaling_factor=3.0, track_unknown=True)),
    ((120, 120), dict(inflation_radius=12.675, cost_scaling_factor=0.0)),
])
def test_fleet_matches_single_costmaps(cuda, size, opts):
    sx, sy = size
    radius = opts.get("inflation_radius", 0.55)
    R = cuda.build_cost_table(RES, 0.0, radius, 1.0)[0]
    assert R == CELL_RADII.get(radius, R), f"cell radius {R}"
    n, cycles = 6, 6
    robots = [synth.fleet_sensing_robot(40 + i, n=max(sx, sy)) for i in range(n)]
    fleet = cuda.fleet_sensing(n, sx, sy, RES, sc.PENTAGON, **opts, **CFG)
    singles = [single_costmap(cuda, sx, sy, **opts) for _ in range(n)]
    fleet.set_plans(np.array([edge_pose(robots, i, 0) for i in range(n)]), [r["plan"] for r in robots])
    for cycle in range(cycles):
        scans = [edge_scans(robots, i, cycle) for i in range(n)]
        poses = np.array([edge_pose(robots, i, cycle) for i in range(n)])
        fleet.set_scans(scans)
        fleet.step(poses, np.array([r["vel"] for r in robots]))
        for i, (cm, o, _) in enumerate(singles):
            if scans[i]:
                cm.set_scans(o, scans[i])
            else:
                cm.set_observations(o, [])
            win = cm.update_map(*poses[i])
            origin, fwin = fleet.geometry(i)
            assert fwin == win, f"cycle {cycle} robot {i}: window {fwin} vs {win}"
            assert origin == cm.origin(), f"cycle {cycle} robot {i}: origin {origin} vs {cm.origin()}"
            assert np.array_equal(fleet.layer(i), cm.get_layer(o)), f"cycle {cycle} robot {i}: obstacle layer differs"
            assert np.array_equal(fleet.costmap(i), cm.get()), f"cycle {cycle} robot {i}: master grid differs"
    # the scenario exercised what it claims: marks, inflation, an unknown default where asked
    last = fleet.costmap(4)
    assert (last == 254).any() and ((last > 0) & (last < 253)).any()
    if opts.get("track_unknown"):  # the robot without scans: unknown, but for its footprint where that is cleared
        assert (fleet.layer(0) == 255).any() and np.isin(fleet.layer(0), [0, 255]).all()


def checker_robot(port, sx, sy, inflation_radius=0.55, cost_scaling_factor=10.0):
    cm = port.costmap(sx, sy, RES, 0.0, 0.0, rolling=True)
    o = cm.add_obstacle_layer(1, True, 2.0)
    il = cm.add_inflation_layer(inflation_radius, cost_scaling_factor)
    sc.select_inflation(cm, il, "exact")
    cm.set_footprint(sc.PENTAGON)
    return cm, o


def checker_cycle(port, cm, o, scans, pose, plan, vel, d, sx, sy):
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


def assert_result(g, e, fleet, d, where):
    assert (g["best_index"], g["n_samples"], g["n_scored"]) == (e["best_index"], e["n_samples"], e["n_scored"]), \
        f"{where}: {g} vs best {e['best_index']} cost {e['cost']}"
    assert fleet.oscillation_mask(where[1]) == d.oscillation_mask(), where
    assert (g["cost"] >= 0) == bool(e["ok"]), f"{where}: fleet cost {g['cost']}, checker cost {e['cost']}"
    if e["ok"]:
        assert np.isclose(g["cost"], e["cost"], rtol=RTOL, atol=0), where
        assert (g["xv"], g["yv"], g["thetav"]) == (e["xv"], e["yv"], e["thetav"]), where
        return 1, int(g["cost"] == e["cost"])
    return 0, 0


def test_fleet_matches_checker_robot_by_robot(cuda, port):
    # the defaults, and a cell radius of 60 (2.975 m at 0.05 m)
    for infl in (dict(), dict(inflation_radius=2.975, cost_scaling_factor=3.0)):
        fleet_matches_checker(cuda, port, **infl)


def fleet_matches_checker(cuda, port, **infl):
    sx = sy = 120
    n, cycles = 8, 5
    robots = [synth.fleet_sensing_robot(200 + i) for i in range(n)]
    fleet = cuda.fleet_sensing(n, sx, sy, RES, sc.PENTAGON, **infl, **CFG)
    refs = [checker_robot(port, sx, sy, **infl) for _ in range(n)]
    dwas = [port.dwa(sx, sy, RES, **CFG) for _ in range(n)]
    vels = np.array([r["vel"] for r in robots])
    valid = exact = 0
    for cycle in range(cycles):
        poses = np.array([r["poses"][cycle] for r in robots])
        scans = [[synth.fleet_scan(r, cycle, cloud=True)] for r in robots]
        fleet.set_scans(scans)
        fleet.set_plans(poses, [r["plan"] for r in robots])
        out = fleet.step(poses, vels)
        for i, ((cm, o), d) in enumerate(zip(refs, dwas)):
            win, grid, e = checker_cycle(port, cm, o, scans[i], poses[i], robots[i]["plan"], vels[i], d, sx, sy)
            assert fleet.geometry(i) == (cm.origin(), win), f"cycle {cycle} robot {i}"
            assert np.array_equal(fleet.layer(i), cm.get_layer(o)), f"cycle {cycle} robot {i}: obstacle layer differs"
            assert np.array_equal(fleet.costmap(i), grid), f"cycle {cycle} robot {i}: master grid differs"
            v, x = assert_result(out[i], e, fleet, d, (cycle, i))
            valid, exact = valid + v, exact + x
        for i, g in enumerate(out):  # alternate the commanded direction so oscillation flags latch on some robots
            if g["cost"] >= 0:
                vels[i] = [g["xv"] * (-1 if cycle % 2 else 1), g["yv"], -g["thetav"]]
    assert valid > 0 and exact >= 0.99 * valid


def test_full_fleet_sampled_parity(cuda, port):
    """The benched configuration: 4096 robots, 120 x 120 at 0.05 m, 20 x 1 x 20 samples, one fresh scan per robot; one
    step, every 64th robot replayed through the checker."""
    cfg = dict(vx_samples=20, vy_samples=1, vth_samples=20, max_vel_y=0.0, min_vel_y=0.0)
    n, sx, sy = 4096, 120, 120
    robots = [synth.fleet_sensing_robot(i) for i in range(n)]
    fleet = cuda.fleet_sensing(n, sx, sy, RES, sc.PENTAGON, **cfg)
    poses = np.array([r["poses"][0] for r in robots])
    vels = np.array([r["vel"] for r in robots])
    scans = [[synth.fleet_scan(r, 0, cloud=True)] for r in robots]
    fleet.set_scans(scans)
    fleet.set_plans(poses, [r["plan"] for r in robots])
    out = fleet.step(poses, vels)
    valid = exact = 0
    for i in range(0, n, 64):
        cm, o = checker_robot(port, sx, sy)
        d = port.dwa(sx, sy, RES, **cfg)
        win, grid, e = checker_cycle(port, cm, o, scans[i], poses[i], robots[i]["plan"], vels[i], d, sx, sy)
        assert fleet.geometry(i) == (cm.origin(), win), f"robot {i}"
        assert np.array_equal(fleet.costmap(i), grid), f"robot {i}: master grid differs"
        v, x = assert_result(out[i], e, fleet, d, (0, i))
        valid, exact = valid + v, exact + x
    assert valid >= 32 and exact >= 0.99 * valid


def test_errors(cuda):
    fp = sc.PENTAGON
    raw = cuda.fleet(2, 40, 40, RES, fp, **CFG)
    sens = cuda.fleet_sensing(2, 40, 40, RES, fp, **CFG)
    r = synth.fleet_sensing_robot(1)
    with pytest.raises(NavGpuError, match="navgpu error 2"):
        sens.set_maps(np.zeros((2, 40, 40), np.uint8), np.zeros((2, 2)))
    with pytest.raises(NavGpuError, match="navgpu error 2"):
        raw.set_scans([[synth.fleet_scan(r, 0)], []])
    with pytest.raises(NavGpuError, match="navgpu error 2"):
        raw.layer(0)
    with pytest.raises(NavGpuError, match="navgpu error 2"):
        raw.geometry(0)
    arr, _keep = pack_scans([synth.fleet_scan(r, 0)] * 2)
    off = np.array([0, 2, 1], dtype=np.int32)  # robot 1's range ends before it starts
    with pytest.raises(NavGpuError, match="navgpu error 2"):
        cuda.check(cuda.lib.navgpu_fleet_set_scans(sens.h, arr, off.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))))
    with pytest.raises(NavGpuError, match="navgpu error 2"):
        raw.last_timing()
    with pytest.raises(NavGpuError, match="navgpu error 2"):
        cuda.fleet_sensing(2, 40, 40, RES, fp, combination_method=2, **CFG)
    # what one CTA's shared memory cannot hold
    with pytest.raises(NavGpuError, match="navgpu error 3.*shared memory"):
        cuda.fleet_sensing(2, 400, 400, RES, fp, **CFG)
    with pytest.raises(NavGpuError, match="navgpu error 3.*cell inflation radius 400 > 254"):
        cuda.fleet_sensing(2, 120, 120, RES, fp, inflation_radius=20.0, **CFG)
    # A cost table that is not a function of d^2 (upload_tables' check).  The host libm's hypot is not correctly
    # rounded: hypot(28, 47) and hypot(17, 52) differ in the last bit though 28^2 + 47^2 = 17^2 + 52^2.  With 1 m cells
    # and the inscribed radius exactly hypot(28, 47) -- the nearest point of this footprint, which keeps the origin
    # outside -- the first is INSCRIBED (253) and the second already decays (251).
    far = [(28.0, 47.0), (28.0, 100.0), (60.0, 100.0)]
    with pytest.raises(NavGpuError, match="navgpu error 3.*not a function of squared distance for R=55"):
        cuda.fleet_sensing(2, 40, 40, 1.0, far, inflation_radius=55.0, footprint_clearing=False, **CFG)
    # the same geometry with a radius whose table stops short of d^2 = 2993 is accepted
    cuda.fleet_sensing(2, 40, 40, 1.0, far, inflation_radius=54.0, footprint_clearing=False, **CFG)
    with pytest.raises(NavGpuError, match="navgpu error 3.*footprint"):
        cuda.fleet_sensing(2, 120, 120, RES, [(-2, -2), (-2, 2), (2, 2), (2, -2)], **CFG)
    # the same footprint is fine where it is never rasterised
    cuda.fleet_sensing(2, 120, 120, RES, [(-2, -2), (-2, 2), (2, 2), (2, -2)], footprint_clearing=False, **CFG)


def test_fleets_of_different_sizes_in_one_process(cuda):
    """The kernel's shared-memory limit is the device function's, not a fleet's: a large fleet still steps after a
    smaller one was created (and the other way round), and both still equal their single costmaps."""
    big_n, small_n = 200, 40
    big_r = [synth.fleet_sensing_robot(300 + i, n=big_n) for i in range(2)]
    small_r = [synth.fleet_sensing_robot(310 + i, n=120) for i in range(2)]
    big = cuda.fleet_sensing(2, big_n, big_n, RES, sc.PENTAGON, inflation_radius=1.0, **CFG)
    small = cuda.fleet_sensing(2, small_n, small_n, RES, sc.PENTAGON, **CFG)
    ref = {"big": [single_costmap(cuda, big_n, big_n, inflation_radius=1.0) for _ in range(2)],
           "small": [single_costmap(cuda, small_n, small_n) for _ in range(2)]}
    for fl, robots in ((big, big_r), (small, small_r)):
        fl.set_plans(np.array([r["poses"][0] for r in robots]), [r["plan"] for r in robots])
    for cycle in range(3):
        for name, fl, robots in (("big", big, big_r), ("small", small, small_r)):
            scans = [[synth.fleet_scan(r, cycle)] for r in robots]
            poses = np.array([r["poses"][cycle] for r in robots])
            fl.set_scans(scans)
            fl.step(poses, np.array([r["vel"] for r in robots]))
            for i, (cm, o, _) in enumerate(ref[name]):
                cm.set_scans(o, scans[i])
                win = cm.update_map(*poses[i])
                assert fl.geometry(i) == (cm.origin(), win), f"{name} cycle {cycle} robot {i}"
                assert np.array_equal(fl.costmap(i), cm.get()), f"{name} cycle {cycle} robot {i}: master grid differs"
