"""Fleets of legacy TrajectoryPlanners (navgpu_fleet_use_trajectory_planner / navgpu_fleet_step_tp).

1. Robot by robot against single planners (navgpu_tp) fed the fleet's own costmap at the fleet's origin, over raw-map,
   2-D sensing and voxel fleets and three configurations: cost, velocities, flags and n_points bit-equal, both
   wavefront grids equal.  The same robots go through the CPU checker's TrajectoryPlanner (cost within 1e-5 relative,
   the rest identical).  The robots (fleet_tp_scenarios.py) take every branch of the selection between them.
2. 4096 robots of the benchmark's inputs, sampled through the checker.
3. A step's launch count does not grow with the robots; errors; DWA and TrajectoryPlanner fleets in one process."""
import numpy as np
import pytest

import fleet_tp_scenarios as ft
import scenarios as sc
from navigation_b200 import synth
from navigation_b200.api import DwaResult, NavGpuError, TpResult, _f64p, _p

pytestmark = pytest.mark.gpu

RTOL = 1e-5
CONFIGS = [dict(), dict(holonomic_robot=0, dwa=0), dict(heading_scoring=1)]
CYCLES = 9
ALL_BRANCHES = {"forward", "rotate", "strafe", "escape", "leave_escape", "stuck", "stuck_reset"}


def make_fleet(api, kind, n, cfg):
    if kind == "raw":
        return api.fleet(n, ft.N, ft.N, ft.RES, sc.PENTAGON, 0.55, 10.0, trajectory_planner=cfg)
    return api.fleet_sensing(n, ft.N, ft.N, ft.RES, sc.PENTAGON, voxel={} if kind == "voxel" else None,
                             trajectory_planner=cfg)


def same(g, e, rtol=0.0):
    if (g["xv"], g["yv"], g["thetav"], g["flags"], g["n_points"]) != (e["xv"], e["yv"], e["thetav"], e["flags"],
                                                                       len(e["points"])):
        return False
    return g["cost"] == e["cost"] if rtol == 0.0 else bool(np.isclose(g["cost"], e["cost"], rtol=rtol, atol=0))


@pytest.mark.parametrize("cfg", CONFIGS, ids=["defaults", "diff_drive_no_dwa", "heading_scoring"])
@pytest.mark.parametrize("kind", ["raw", "sensing", "voxel"])
def test_fleet_tp_matches_single_planners(cuda, port, kind, cfg):
    robots = ft.scenario(16)
    n = len(robots)
    fleet = make_fleet(cuda, kind, n, cfg)
    singles = [cuda.trajectory_planner(ft.N, ft.N, ft.RES, sc.PENTAGON, **cfg) for _ in robots]
    checkers = [port.trajectory_planner(ft.N, ft.N, ft.RES, sc.PENTAGON, **cfg) for _ in robots]
    traces = [[] for _ in robots]
    mixed_counts = False
    exact = total = 0
    for cycle in range(CYCLES):
        if kind == "raw" and cycle in (0, 3, 6):  # robot 6's box opens at 3, robot 5's slot closes at 6
            fleet.set_maps(*ft.scenario_raw(robots, cycle))
        elif kind != "raw":
            fleet.set_scans(ft.scenario_sources(robots, cycle, kind == "voxel"))
        if cycle in (0, 3):
            plans = [r.plan_at(cycle) for r in robots]
            fleet.set_plans(np.array([r.pose for r in robots]), plans)
            for p, tp, ck in zip(plans, singles, checkers):
                for h in (tp, ck):
                    if len(p):
                        h.update_plan(p)
        out = fleet.step(np.array([r.pose for r in robots]), np.array([r.vel for r in robots]))
        escaping = {bool(g["flags"] & 256) for g in out}
        mixed_counts |= len(escaping) == 2
        for i, (r, g) in enumerate(zip(robots, out)):
            origin = r.map_origin if kind == "raw" else fleet.geometry(i)[0]
            grid = fleet.costmap(i)
            grids = [fleet.tp_grid(i, 0), fleet.tp_grid(i, 1)]
            for h, rtol in ((singles[i], 0.0), (checkers[i], RTOL)):
                h.set_costmap(grid, *origin)
                e = h.find_best_path(r.pose, r.vel)
                assert same(g, e, rtol), f"{kind} cycle {cycle} robot {i}: fleet {g} vs {'single' if rtol == 0 else 'checker'} " \
                                         f"cost {e['cost']} v ({e['xv']}, {e['yv']}, {e['thetav']}) flags {e['flags']} " \
                                         f"points {len(e['points'])}"
                for k in (0, 1):
                    assert np.array_equal(grids[k], h.grid(k)), f"{kind} cycle {cycle} robot {i}: grid {k} differs"
                if rtol:
                    exact += g["cost"] == e["cost"]
                    total += 1
            traces[i].append((g, r.pose.copy()))
        ft.advance(robots, out)
    assert exact >= 0.99 * total  # costs are bit-equal in practice
    seen = set().union(*(ft.branches(t, cfg) for t in traces))
    if kind == "raw":
        want = ALL_BRANCHES if cfg.get("holonomic_robot", 1) else ALL_BRANCHES - {"strafe"}
        assert want <= seen, f"branches not taken: {want - seen}"
        assert mixed_counts, "no step had escaping (no forward samples) and other robots together"
        # the final-goal cap: 0.2 m to go (from the pose rounded through float) over sim_time 1 s
        assert 0.0 < traces[7][0][0]["xv"] <= 0.2 + 1e-6
        assert all(g["cost"] < 0 or g["xv"] < 0 for g, _ in traces[9])  # off its map: backing up
    else:
        assert {"forward", "rotate"} <= seen, seen
    assert all(g["xv"] < 0 for g, _ in traces[8])  # an empty plan: nothing reachable, backing up


def inflate_like_fleet(port, robot):
    cm = port.costmap(120, 120, 0.05, *robot["origin"])
    s = cm.add_grid_layer(0)
    cm.add_inflation_layer(0.55, 10.0)
    cm.set_footprint(sc.PENTAGON)
    cm.set_grid_layer(s, robot["raw"])
    cm.update_map(0, 0, 0)
    return cm.get()


def test_fleet_tp_full_size_sampled_through_checker(cuda, port):
    """tools/bench_fleet_tp.py's configuration: 4096 robots of synth.fleet_robot(i), TrajectoryPlannerROS's defaults,
    one step; every 64th robot and up to 24 that backed up are replayed through the checker."""
    n = 4096
    robots = [synth.fleet_robot(i) for i in range(n)]
    fleet = cuda.fleet(n, 120, 120, 0.05, sc.PENTAGON, 0.55, 10.0, trajectory_planner={})
    fleet.set_maps(np.stack([r["raw"] for r in robots]), np.array([r["origin"] for r in robots]))
    poses = np.array([r["pose"] for r in robots])
    vels = np.array([r["vel"] for r in robots])
    fleet.set_plans(poses, [r["plan"] for r in robots])
    out = fleet.step(poses, vels)
    backed = [i for i, g in enumerate(out) if g["xv"] < 0]
    sample = sorted(set(range(0, n, 64)) | set(backed[:24]))
    exact = 0
    for i in sample:
        grid = inflate_like_fleet(port, robots[i])
        assert np.array_equal(fleet.costmap(i), grid), f"robot {i}: inflated local costmap differs"
        tp = port.trajectory_planner(120, 120, 0.05, sc.PENTAGON)
        tp.set_costmap(grid, *robots[i]["origin"])
        tp.update_plan(robots[i]["plan"])
        e = tp.find_best_path(poses[i], vels[i])
        assert same(out[i], e, RTOL), f"robot {i}: fleet {out[i]} vs checker cost {e['cost']} flags {e['flags']}"
        for k in (0, 1):
            assert np.array_equal(fleet.tp_grid(i, k), tp.grid(k)), f"robot {i}: grid {k} differs"
        exact += out[i]["cost"] == e["cost"]
    assert exact >= 0.99 * len(sample)
    print(f"TrajectoryPlanner fleet: {sum(g['cost'] >= 0 for g in out)} of {n} robots valid, {len(backed)} backing up; "
          f"{len(sample)} replayed through the checker, {exact} costs bit-equal")


@pytest.mark.parametrize("kind", ["raw", "sensing"])
def test_fleet_tp_launch_count_does_not_grow_with_robots(cuda, kind):
    counts = []
    for n in (8, 64):
        robots = [synth.fleet_robot(i) for i in range(n)]
        fleet = make_fleet(cuda, kind, n, {})
        if kind == "raw":
            fleet.set_maps(np.stack([r["raw"] for r in robots]), np.array([r["origin"] for r in robots]))
        else:
            sens = [synth.fleet_sensing_robot(i) for i in range(n)]
            fleet.set_scans([[synth.fleet_scan(s, 0)] for s in sens])
        poses = np.array([r["pose"] for r in robots])
        vels = np.array([r["vel"] for r in robots])
        fleet.set_plans(poses, [r["plan"] for r in robots])
        fleet.step(poses, vels)
        before = cuda.launch_count()
        fleet.step(poses, vels)
        counts.append(cuda.launch_count() - before)
    assert counts[0] == counts[1], counts


def test_fleet_tp_errors(cuda):
    def raises(call, code, text):
        with pytest.raises(NavGpuError, match=f"error {code}: .*{text}"):
            call()

    poses, vels = np.zeros((2, 3)), np.zeros((2, 3))
    plans = [np.array([[0.0, 0.0], [1.0, 0.0]])] * 2
    tpf = cuda.fleet(2, 40, 40, 0.05, sc.PENTAGON, 0.55, 10.0, trajectory_planner={})
    lib = cuda.lib
    raises(lambda: tpf.reset_oscillation(), 2, "TrajectoryPlanner fleet")
    raises(lambda: tpf.oscillation_mask(0), 2, "TrajectoryPlanner fleet")
    raises(lambda: cuda.check(lib.navgpu_fleet_use_trajectory_planner(tpf.h, tpf.tp_cfg)), 2, "already")
    # navgpu_fleet_step itself refuses a TrajectoryPlanner fleet
    res = (DwaResult * 2)()
    raises(lambda: cuda.check(lib.navgpu_fleet_step(tpf.h, _p(poses, _f64p), _p(vels, _f64p), res)), 2,
           "navgpu_fleet_step_tp")
    # the TrajectoryPlanner calls refuse a DWA fleet
    dwa = cuda.fleet(2, 40, 40, 0.05, sc.PENTAGON, 0.55, 10.0)
    tres = (TpResult * 2)()
    raises(lambda: cuda.check(lib.navgpu_fleet_step_tp(dwa.h, _p(poses, _f64p), _p(vels, _f64p), tres)), 2,
           "not a TrajectoryPlanner fleet")
    raises(lambda: dwa.tp_grid(0, 0), 2, "not a TrajectoryPlanner fleet")
    # the planner is chosen before the first set_plans / step
    dwa.set_plans(poses, plans)
    raises(lambda: cuda.check(lib.navgpu_fleet_use_trajectory_planner(dwa.h, tpf.tp_cfg)), 2, "before the first")
    stepped = cuda.fleet(2, 40, 40, 0.05, sc.PENTAGON, 0.55, 10.0, trajectory_planner={})
    stepped.set_maps(np.zeros((2, 40, 40), np.uint8), np.zeros((2, 2)))
    stepped.set_plans(poses, plans)
    stepped.step(poses, vels)
    raises(lambda: cuda.check(lib.navgpu_fleet_use_trajectory_planner(stepped.h, stepped.tp_cfg)), 2, "already")
    # configs navgpu_tp_create refuses, refused with its codes
    raises(lambda: cuda.fleet(2, 40, 40, 0.05, sc.PENTAGON, trajectory_planner=dict(sim_time=0.0)), 2, "positive")
    raises(lambda: cuda.fleet(2, 40, 40, 0.05, sc.PENTAGON, trajectory_planner=dict(n_y_vels=9)), 2, "n_y_vels")
    raises(lambda: cuda.fleet_sensing(2, 40, 40, 0.05, sc.PENTAGON, trajectory_planner=dict(angular_sim_granularity=-1)),
           2, "positive")
    # footprints whose filled cells could overflow the per-robot buffer
    big = [(-3.0, -3.0), (-3.0, 3.0), (3.0, 3.0), (3.0, -3.0)]
    raises(lambda: cuda.fleet(2, 200, 200, 0.05, big, 0.0, 10.0, trajectory_planner={}), 3, "footprint")
    # grid arguments
    raises(lambda: stepped.tp_grid(2, 0), 2, "bad arguments")
    raises(lambda: stepped.tp_grid(0, 2), 2, "bad arguments")
    # empty plans are accepted, as navgpu_tp_update_plan accepts them: the robots back up
    stepped.set_plans(poses, [np.zeros((0, 2))] * 2)
    out = stepped.step(poses, vels)
    assert all(g["xv"] < 0 for g in out)


def test_dwa_and_tp_fleets_share_a_process(cuda):
    """A DWA fleet stepped alternately with a TrajectoryPlanner fleet gives what it gives stepped alone."""
    n = 12
    robots = [synth.fleet_robot(300 + i) for i in range(n)]
    maps = np.stack([r["raw"] for r in robots])
    origins = np.array([r["origin"] for r in robots])
    poses = np.array([r["pose"] for r in robots])
    vels = np.array([r["vel"] for r in robots])
    cfg = dict(vx_samples=6, vy_samples=1, vth_samples=11, max_vel_y=0.0, min_vel_y=0.0)

    def run(with_tp):
        dwa = cuda.fleet(n, 120, 120, 0.05, sc.PENTAGON, 0.55, 10.0, **cfg)
        dwa.set_maps(maps, origins)
        dwa.set_plans(poses, [r["plan"] for r in robots])
        if with_tp:
            tpf = cuda.fleet(n, 120, 120, 0.05, sc.PENTAGON, 0.55, 10.0, trajectory_planner={})
            tpf.set_maps(maps, origins)
            tpf.set_plans(poses, [r["plan"] for r in robots])
        trace = []
        p = poses.copy()
        for _ in range(4):
            trace.append(dwa.step(p, vels))
            if with_tp:
                t = tpf.step(p, vels)
                assert any(g["cost"] >= 0 for g in t)
            p = p + np.array([0.02, 0.0, 0.01])
        return trace

    assert run(True) == run(False)
