"""Batched scan ingest (navgpu_fleet_set_scan_batch / _device, Fleet.set_scan_batch): two fleets side by side, one fed
dense per-sensor arrays, one fed navgpu_fleet_set_scans with the per-robot scan lists the batch stands for
(synth.batch_scans).  Every robot's obstacle (or voxel) grid, master grid, origin, window, voxel columns, every result
field and the oscillation mask (DWAPlanner) or flags (TrajectoryPlanner) must be equal after every step.

Covered: moving robots (one standing still, one jumping more than a map width) with a LaserScan whose ranges hold
+inf under inf_is_valid, NaN and values below range_min and at or above range_max, next to a marking-only cloud;
track_unknown, Overwrite and an odd map; a clearing-only source without inf_is_valid, a source without points and an
empty batch; voxel fleets fed 3-D clouds; a sensing TrajectoryPlanner fleet; the device variant fed CUDA torch tensors
written on a side stream right before the call; and every refusal, after which the fleet steps as if it had never
been called."""
import ctypes as C

import numpy as np
import pytest

import scenarios as sc
from navigation_b200 import synth
from navigation_b200.api import FleetScanSource
from test_gpu_fleet_sensing import CFG, RES, edge_pose

pytestmark = pytest.mark.gpu

VOXEL = dict(origin_z=0.0, z_resolution=0.2, z_voxels=10, unknown_threshold=15, mark_threshold=0)


def moving_robots(n, cycles, size, voxel=False):
    """fleet_sensing_robot (fleet_voxel_robot) worlds whose poses follow edge_pose: robot 1 stands still, robot 2
    jumps 15 m at cycle 3."""
    make = synth.fleet_voxel_robot if voxel else synth.fleet_sensing_robot
    robots = [make(40 + i, n=size) for i in range(n)]
    for i, r in enumerate(robots):
        r["poses"] = np.array([edge_pose(robots, i, c) for c in range(cycles)])
    return robots


def hard_laser(robots, cycle):
    """fleet_scan_batch's LaserScan with every kind of range: +inf (inf_is_valid), NaN, below range_min, exactly
    range_max and beyond it."""
    b = synth.fleet_scan_batch(robots, cycle)
    r = b["ranges"]
    r[:, 3::17] = np.nan
    r[:, 5::29] = 0.01
    r[:, 7::31] = b["range_max"]
    r[:, 11::37] = 5.0
    assert np.isposinf(r).any() and b["inf_is_valid"] == 1
    return b


def marking_cloud(robots, cycle):
    b = synth.fleet_scan_batch(robots, cycle, cloud=True, n_beams=180)
    b["sensor_to_global"][:, 2] = 0.25
    b.update(clearing=False, marking=True)
    return b


def assert_same(a, b, n, step_a, step_b, where, voxel=False, tp=False):
    assert step_a == step_b, f"{where}: results differ"
    for i in range(n):
        w = f"{where} robot {i}"
        assert a.geometry(i) == b.geometry(i), w
        assert np.array_equal(a.layer(i), b.layer(i)), f"{w}: obstacle layer differs"
        assert np.array_equal(a.costmap(i), b.costmap(i)), f"{w}: master grid differs"
        if voxel:
            assert np.array_equal(a.voxels(i), b.voxels(i)), f"{w}: voxel columns differ"
        if not tp:
            assert a.oscillation_mask(i) == b.oscillation_mask(i), w


def twin_cycle(a, b, sources, n, poses, vels, where, **kw):
    """a takes the batch, b the equivalent per-robot lists; both step and must agree."""
    a.set_scan_batch(sources)
    b.set_scans(synth.batch_scans(sources, n))
    ra, rb = a.step(poses, vels), b.step(poses, vels)
    assert_same(a, b, n, ra, rb, where, **kw)
    return ra


@pytest.mark.parametrize("size,opts", [
    ((120, 120), dict()),
    ((120, 120), dict(track_unknown=True)),
    ((120, 120), dict(combination_method=0)),
    ((97, 131), dict()),
], ids=["defaults", "track_unknown", "overwrite", "97x131"])
def test_batch_equals_set_scans(cuda, size, opts):
    sx, sy = size
    n, cycles = 6, 6
    robots = moving_robots(n, cycles, max(sx, sy))
    a, b = (cuda.fleet_sensing(n, sx, sy, RES, sc.PENTAGON, **opts, **CFG) for _ in range(2))
    for f in (a, b):
        f.set_plans(robots_poses(robots, 0), [r["plan"] for r in robots])
    vels = np.array([r["vel"] for r in robots])
    for cycle in range(cycles):
        out = twin_cycle(a, b, [hard_laser(robots, cycle), marking_cloud(robots, cycle)], n,
                         robots_poses(robots, cycle), vels, f"cycle {cycle}")
        for i, g in enumerate(out):  # alternate the commanded direction so oscillation flags latch on some robots
            if g["cost"] >= 0:
                vels[i] = [g["xv"] * (-1 if cycle % 2 else 1), g["yv"], -g["thetav"]]
    last = a.costmap(4)
    assert (last == 254).any() and ((last > 0) & (last < 253)).any()


def robots_poses(robots, cycle):
    return np.array([r["poses"][cycle] for r in robots])


def test_clearing_only_empty_sources_and_empty_batch(cuda):
    n, cycles = 5, 4
    robots = moving_robots(n, cycles, 120)
    a, b = (cuda.fleet_sensing(n, 120, 120, RES, sc.PENTAGON, track_unknown=True, **CFG) for _ in range(2))
    for f in (a, b):
        f.set_plans(robots_poses(robots, 0), [r["plan"] for r in robots])
    vels = np.array([r["vel"] for r in robots])
    for cycle in range(cycles):
        clear_only = synth.fleet_scan_batch(robots, cycle)
        clear_only.update(marking=False, inf_is_valid=0)  # +inf is then dropped, not cleared along
        empty = marking_cloud(robots, cycle)
        empty["points"] = np.zeros((n, 0, 3), np.float32)
        empty["clearing"] = True
        batches = [[clear_only, empty], [empty], [], [synth.fleet_scan_batch(robots, cycle), empty]]
        twin_cycle(a, b, batches[cycle], n, robots_poses(robots, cycle), vels, f"cycle {cycle}")
    assert (a.layer(0) == 0).any() and (a.layer(0) == 255).any()


def test_voxel_fleet(cuda):
    n, cycles = 6, 5
    robots = moving_robots(n, cycles, 120, voxel=True)
    a, b = (cuda.fleet_sensing(n, 120, 120, RES, sc.PENTAGON, voxel=VOXEL, **CFG) for _ in range(2))
    for f in (a, b):
        f.set_plans(robots_poses(robots, 0), [r["plan"] for r in robots])
    vels = np.array([r["vel"] for r in robots])
    for cycle in range(cycles):
        sources = [synth.fleet_cloud_3d_batch(robots, cycle)]
        if cycle % 2:
            sources.append(hard_laser(robots, cycle))
        twin_cycle(a, b, sources, n, robots_poses(robots, cycle), vels, f"cycle {cycle}", voxel=True)
    assert (a.voxels(3) >> 16).any()


def test_trajectory_planner_fleet(cuda):
    n, cycles = 6, 4
    robots = moving_robots(n, cycles, 120)
    a, b = (cuda.fleet_sensing(n, 120, 120, RES, sc.PENTAGON, trajectory_planner={}) for _ in range(2))
    for f in (a, b):
        f.set_plans(robots_poses(robots, 0), [r["plan"] for r in robots])
    vels = np.array([r["vel"] for r in robots])
    for cycle in range(cycles):
        out = twin_cycle(a, b, [hard_laser(robots, cycle), marking_cloud(robots, cycle)], n,
                         robots_poses(robots, cycle), vels, f"cycle {cycle}", tp=True)
        for i in range(n):
            assert a.tp_grid(i, 0).tobytes() == b.tp_grid(i, 0).tobytes()
    assert any(g["cost"] >= 0 for g in out)


def test_device_tensors_equal_host_arrays(cuda):
    torch = pytest.importorskip("torch")
    n, cycles = 6, 4
    robots = moving_robots(n, cycles, 120)
    host, dev = (cuda.fleet_sensing(n, 120, 120, RES, sc.PENTAGON, **CFG) for _ in range(2))
    for f in (host, dev):
        f.set_plans(robots_poses(robots, 0), [r["plan"] for r in robots])
    vels = np.array([r["vel"] for r in robots])
    side = torch.cuda.Stream()
    for cycle in range(cycles):
        sources = [hard_laser(robots, cycle), marking_cloud(robots, cycle)]
        on_dev = []
        with torch.cuda.stream(side):
            for s in sources:
                d = dict(s)
                for k in ("ranges", "points", "sensor_to_global"):
                    if k in s:  # garbage first, then a long kernel, then the values: all queued on the side stream
                        t = torch.full(s[k].shape, -7.0, dtype=getattr(torch, str(s[k].dtype)), device="cuda")
                        torch.cuda._sleep(20_000_000)
                        t.copy_(torch.from_numpy(s[k]).pin_memory(), non_blocking=True)
                        d[k] = t
                on_dev.append(d)
            dev.set_scan_batch(on_dev)
        host.set_scan_batch(sources)
        poses = robots_poses(robots, cycle)
        assert_same(dev, host, n, dev.step(poses, vels), host.step(poses, vels), f"cycle {cycle}")
        assert dev.last_timing()[0] > 0
    torch.cuda.synchronize()
    # mixed host / device arrays and wrong dtypes or shapes never reach the C ABI
    s = sources[0]
    with pytest.raises(ValueError):
        dev.set_scan_batch([dict(s, ranges=torch.from_numpy(s["ranges"]).cuda())])
    with pytest.raises(ValueError):
        dev.set_scan_batch([dict(s, ranges=s["ranges"].astype(np.float64))])
    with pytest.raises(ValueError):
        dev.set_scan_batch([dict(s, sensor_to_global=s["sensor_to_global"][:, :6])])
    with pytest.raises(ValueError):
        dev.set_scan_batch([dict(s, ranges=torch.from_numpy(s["ranges"][:-1]))])


def packed(sources):
    """The navgpu_fleet_scan_source array of a host batch, and the arrays it points into."""
    arr = (FleetScanSource * max(1, len(sources)))()
    keep = []
    for k, s in enumerate(sources):
        key = "points" if "points" in s else "ranges"
        data, stg = np.ascontiguousarray(s[key]), np.ascontiguousarray(s["sensor_to_global"])
        keep += [data, stg]
        c = arr[k]
        c.data, c.sensor_to_global = data.ctypes.data, stg.ctypes.data
        c.n_points, c.is_cloud = data.shape[1], int(key == "points")
        c.inf_is_valid, c.marking, c.clearing = int(s.get("inf_is_valid", 0)), int(s["marking"]), int(s["clearing"])
        for f in ("angle_min", "angle_increment", "range_min", "range_max"):
            setattr(c, f, float(s.get(f, 0.0)))
        for f in ("min_obstacle_height", "max_obstacle_height", "obstacle_range", "raytrace_range"):
            setattr(c, f, s[f])
    return arr, keep


def test_refusals_leave_the_fleet_as_it_was(cuda):
    lib = cuda.lib
    n = 6
    robots = moving_robots(n, 3, 120)
    a, b = (cuda.fleet_sensing(n, 120, 120, RES, sc.PENTAGON, **CFG) for _ in range(2))
    raw = cuda.fleet(n, 40, 40, RES, sc.PENTAGON, **CFG)
    for f in (a, b):
        f.set_plans(robots_poses(robots, 0), [r["plan"] for r in robots])
    vels = np.array([r["vel"] for r in robots])
    good = [hard_laser(robots, 0), marking_cloud(robots, 0)]
    twin_cycle(a, b, good, n, robots_poses(robots, 0), vels, "cycle 0")

    other = [synth.fleet_scan_batch(robots, 2, cloud=True)]  # what a refused call must not install
    refusals = []

    def case(name, code, mutate=None, call=None, count=None):
        arr, keep = packed(other)
        if mutate:
            mutate(arr[0])
        refusals.append((name, code, call or (lambda: lib.navgpu_fleet_set_scan_batch(a.h, arr, count or 1)),
                         keep, arr))

    case("null handle", 2, call=lambda: lib.navgpu_fleet_set_scan_batch(None, packed(other)[0], 1))
    case("null handle, device", 2, call=lambda: lib.navgpu_fleet_set_scan_batch_device(None, packed(other)[0], 1))
    case("negative n_sources", 2, count=-1)
    case("null sources", 2, call=lambda: lib.navgpu_fleet_set_scan_batch(a.h, None, 1))
    case("null sensor_to_global", 2, lambda c: setattr(c, "sensor_to_global", None))
    case("null data", 2, lambda c: setattr(c, "data", None))
    case("negative n_points", 2, lambda c: setattr(c, "n_points", -1))
    case("is_cloud 2", 2, lambda c: setattr(c, "is_cloud", 2))
    case("marking 2", 2, lambda c: setattr(c, "marking", 2))
    case("clearing -1", 2, lambda c: setattr(c, "clearing", -1))
    case("beyond 2^31 points", 3, lambda c: setattr(c, "n_points", (1 << 31) // n + 1))
    arr33, keep33 = packed(other * 33)
    refusals.append(("33 sources", 3, lambda: lib.navgpu_fleet_set_scan_batch(a.h, arr33, 33), keep33, arr33))
    arr_h, keep_h = packed(other)
    refusals.append(("host memory to the device variant", 2,
                     lambda: lib.navgpu_fleet_set_scan_batch_device(a.h, arr_h, 1), keep_h, arr_h))
    refusals.append(("raw-map fleet", 2, lambda: lib.navgpu_fleet_set_scan_batch(raw.h, arr_h, 1), keep_h, arr_h))
    refusals.append(("raw-map fleet, device", 2, lambda: lib.navgpu_fleet_set_scan_batch_device(raw.h, arr_h, 1),
                     keep_h, arr_h))
    for cycle, (name, code, call, _keep, _arr) in enumerate(refusals, start=1):
        rc = call()
        assert rc == code, f"{name}: {rc} ({lib.navgpu_last_error().decode()})"
        poses = robots_poses(robots, cycle % 3)
        assert_same(a, b, n, a.step(poses, vels), b.step(poses, vels), f"after {name}")
    # the refused calls left the sources in place: a fresh batch still goes through both paths alike
    twin_cycle(a, b, good, n, robots_poses(robots, 2), vels, "after the refusals")
    assert lib.navgpu_fleet_stream(None) is None and a.stream() and raw.stream()
