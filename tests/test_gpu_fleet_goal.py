"""Goal handling for fleets: per-robot planning masks (navgpu_fleet_set_active) and batched trajectory checks
(navgpu_fleet_check_trajectories).

1. Over raw-map, 2-D sensing and voxel fleets, with DWAPlanner and the TrajectoryPlanner, a changing subset of robots
   is left out of each step and every robot gets 0, 1 or several candidate commands.  Each robot has a single-handle
   twin fed the fleet's costmap and origin: active robots' twins search, inactive robots' twins do nothing, checked
   robots' twins check each candidate.  Costs are bit-equal to the twin's and within 1e-5 of the CPU checker's,
   oscillation masks and TrajectoryPlanner distance grids are equal, and step results stay equal after re-activation
   (a DWA robot with latched flags, a TrajectoryPlanner robot deactivated while escaping).
2. An all-ones mask, or set_active(None), changes nothing; refused calls change nothing.
3. The check call's launches do not grow with robots or candidates.
4. 4096 robots at full size, one candidate each, sampled through the checker."""
import ctypes

import numpy as np
import pytest

import fleet_tp_scenarios as ft
import scenarios as sc
from navigation_b200 import synth
from navigation_b200.api import NavGpuError, _f64p, _i32p, _p, _u8p

pytestmark = pytest.mark.gpu

RTOL = 1e-5
CYCLES = 7
# DWAPlanner with backward motion, so that a robot driven forward then backward latches forward_neg_only
DWA_CFG = dict(vx_samples=6, vy_samples=1, vth_samples=11, max_vel_y=0.0, min_vel_y=0.0, min_vel_x=-0.3)
# stop (the DWA generator rejects it), rotate either way, creep forward, too fast (rejected), back up
CANDIDATES = np.array([(0.0, 0.0, 0.0), (0.0, 0.0, 0.5), (0.2, 0.0, 0.0), (1.0, 0.0, 0.0), (0.0, 0.0, -0.5),
                       (-0.1, 0.0, 0.0)])
INTO_WALL = (0.5, 0.0, 0.0)  # robot 4 faces a wall 0.65 m ahead
LATCH = (10, 12, 13, 14)     # DWA: driven forward at cycle 1 and backward at cycle 2, which latches 10's and 12's flags
LATCH_CHECKED = (10, 13)     # checked at cycle 2; 12 and 14 keep their flags and are left out at cycle 3


def make_fleet(api, kind, n, tp_cfg):
    kw = dict(trajectory_planner=tp_cfg) if tp_cfg is not None else DWA_CFG
    if kind == "raw":
        return api.fleet(n, ft.N, ft.N, ft.RES, sc.PENTAGON, 0.55, 10.0, **kw)
    return api.fleet_sensing(n, ft.N, ft.N, ft.RES, sc.PENTAGON, voxel={} if kind == "voxel" else None, **kw)


def dwa_plan(r, cycle):
    """DWAPlanner needs a plan: the robot without one drives towards a point 1 m ahead."""
    p = r.plan_at(cycle)
    return p if len(p) else np.array([[r.pose[0], r.pose[1]], [r.pose[0] + 1.0, r.pose[1]]])


def candidates(i, cycle, dwa):
    if dwa and i in LATCH_CHECKED and cycle == 2:
        return np.array([(0.2, 0.0, 0.0), (0.0, 0.0, 0.0)])  # forward, which the latched flag forbids a search
    if dwa and i in LATCH and cycle in (1, 2, 3):
        return np.zeros((0, 3))  # a check would reset the flags the latch needs, or the latched ones
    k = (i + cycle) % 4
    out = [CANDIDATES[(i + cycle + j) % len(CANDIDATES)] for j in range(k if k < 3 else 4)]
    if i == 4:
        out.append(INTO_WALL)
    return np.array(out).reshape(-1, 3)


def same_tp(g, e, rtol=0.0):
    if (g["xv"], g["yv"], g["thetav"], g["flags"], g["n_points"]) != (e["xv"], e["yv"], e["thetav"], e["flags"],
                                                                       len(e["points"])):
        return False
    return g["cost"] == e["cost"] if rtol == 0.0 else bool(np.isclose(g["cost"], e["cost"], rtol=rtol, atol=0))


def same_dwa(g, e, rtol=0.0):
    if (g["best_index"], g["n_samples"], g["n_scored"]) != (e["best_index"], e["n_samples"], e["n_scored"]):
        return False
    if (g["cost"] >= 0) != (e["cost"] >= 0):
        return False
    if g["cost"] < 0:
        return True
    if (g["xv"], g["yv"], g["thetav"]) != (e["xv"], e["yv"], e["thetav"]):
        return False
    return g["cost"] == e["cost"] if rtol == 0.0 else bool(np.isclose(g["cost"], e["cost"], rtol=rtol, atol=0))


@pytest.mark.parametrize("planner", ["dwa", "tp"])
@pytest.mark.parametrize("kind", ["raw", "sensing", "voxel"])
def test_goal_handling_matches_single_handles(cuda, port, kind, planner):
    dwa = planner == "dwa"
    robots = ft.scenario(16)
    n = len(robots)
    fleet = make_fleet(cuda, kind, n, None if dwa else {})
    if dwa:
        twins = [cuda.dwa(ft.N, ft.N, ft.RES, **DWA_CFG) for _ in robots]
        checkers = [port.dwa(ft.N, ft.N, ft.RES, **DWA_CFG) for _ in robots]
    else:
        twins = [cuda.trajectory_planner(ft.N, ft.N, ft.RES, sc.PENTAGON) for _ in robots]
        checkers = [port.trajectory_planner(ft.N, ft.N, ft.RES, sc.PENTAGON) for _ in robots]
    seen = dict(rejected=0, negative=0, latched_checked=0, latched_reactivated=0, escaping_reactivated=0, inactive=0)
    escape_off = None  # the cycle the TrajectoryPlanner robot that was escaping is left out
    prev_out = [None] * n
    for cycle in range(CYCLES):
        if kind == "raw" and cycle in (0, 3, 6):
            fleet.set_maps(*ft.scenario_raw(robots, cycle))
        elif kind != "raw":
            fleet.set_scans(ft.scenario_sources(robots, cycle, kind == "voxel"))
        poses = np.array([r.pose for r in robots])
        vels = np.array([r.vel for r in robots])
        if dwa:
            for i in LATCH:
                if cycle in (1, 2):
                    vels[i] = (0.3 if cycle == 1 else -0.3, 0.0, 0.0)
            plans = [dwa_plan(r, cycle) for r in robots]  # updatePlanAndLocalCosts runs every cycle, at the goal too
            fleet.set_plans(poses, plans)
            for i, p in enumerate(plans):
                twins[i].set_plan(poses[i], p)
                checkers[i].set_plan(poses[i], p)
        elif cycle in (0, 3):
            plans = [r.plan_at(cycle) for r in robots]
            fleet.set_plans(poses, plans)
            for p, tw, ck in zip(plans, twins, checkers):
                if len(p):
                    tw.update_plan(p)
                    ck.update_plan(p)
        # who plans this cycle: everyone first, then a changing subset is left out
        active = np.array([cycle == 0 or (i * 7 + cycle * 3) % 5 != 0 for i in range(n)])
        if dwa:
            for i in LATCH:
                active[i] = cycle != 3 or i in LATCH_CHECKED
        else:
            if escape_off is None and cycle > 0 and prev_out[6] is not None and prev_out[6]["flags"] & 256:
                escape_off = cycle
            if escape_off is not None:
                active[6] = cycle != escape_off
        if dwa and cycle == 3:
            seen["latched_reactivated"] += sum(fleet.oscillation_mask(i) != 0 for i in LATCH if not active[i])
        if escape_off == cycle:
            seen["escaping_reactivated"] += 1
        seen["inactive"] += int((~active).sum())
        fleet.set_active(active)
        out = fleet.step(poses, vels)
        assert all((g is None) == (not a) for g, a in zip(out, active))
        for i, r in enumerate(robots):
            origin = r.map_origin if kind == "raw" else fleet.geometry(i)[0]
            grid = fleet.costmap(i)
            for h in (twins[i], checkers[i]):
                h.set_costmap(grid, *origin)
            if active[i]:
                for h, rtol in ((twins[i], 0.0), (checkers[i], RTOL)):
                    e = h.find_best_path(poses[i], vels[i], sc.PENTAGON) if dwa else h.find_best_path(poses[i], vels[i])
                    ok = same_dwa(out[i], e, rtol) if dwa else same_tp(out[i], e, rtol)
                    assert ok, f"{kind} {planner} cycle {cycle} robot {i}: fleet {out[i]} vs " \
                               f"{'twin' if rtol == 0 else 'checker'} cost {e['cost']} v ({e['xv']}, {e['yv']}, " \
                               f"{e['thetav']})"
            if dwa:
                assert fleet.oscillation_mask(i) == twins[i].oscillation_mask() == checkers[i].oscillation_mask(), \
                    f"{kind} cycle {cycle} robot {i}: oscillation mask after the step"
            else:
                for k in (0, 1):
                    assert np.array_equal(fleet.tp_grid(i, k), twins[i].grid(k)), f"cycle {cycle} robot {i}: grid {k}"
                    assert np.array_equal(fleet.tp_grid(i, k), checkers[i].grid(k)), f"cycle {cycle} robot {i}: grid {k}"
        # the stop / rotate commands of the goal controllers, checked against every robot's critics
        cands = [candidates(i, cycle, dwa) for i in range(n)]
        masks_before = [fleet.oscillation_mask(i) for i in range(n)] if dwa else None
        costs = fleet.check_trajectories(poses, vels, cands)
        for i in range(n):
            assert costs[i].shape == (len(cands[i]),)
            for j, c in enumerate(cands[i]):
                if dwa:
                    t = twins[i].check_trajectory(poses[i], vels[i], c, sc.PENTAGON)
                    e = checkers[i].check_trajectory(poses[i], vels[i], c, sc.PENTAGON)
                else:
                    t = twins[i].score_trajectory(poses[i], vels[i], c)
                    e = checkers[i].score_trajectory(poses[i], vels[i], c)
                where = f"{kind} {planner} cycle {cycle} robot {i} candidate {tuple(c)}"
                assert costs[i][j] == t, f"{where}: fleet {costs[i][j]} vs twin {t}"
                assert np.isclose(costs[i][j], e, rtol=RTOL, atol=0), f"{where}: fleet {costs[i][j]} vs checker {e}"
                seen["negative"] += costs[i][j] < 0
                seen["rejected"] += dwa and costs[i][j] == 0.0
            if dwa:
                assert fleet.oscillation_mask(i) == twins[i].oscillation_mask() == checkers[i].oscillation_mask(), \
                    f"{kind} cycle {cycle} robot {i}: oscillation mask after the check"
                if len(cands[i]):
                    assert fleet.oscillation_mask(i) == 0
                    seen["latched_checked"] += masks_before[i] != 0
                else:
                    assert fleet.oscillation_mask(i) == masks_before[i]
        prev_out = out
        ft.advance(robots, [g if g is not None else dict(cost=-1.0) for g in out])
    assert seen["negative"] > 0 and seen["inactive"] > 0, seen
    if dwa:
        assert seen["rejected"] > 0, seen
        if kind == "raw":
            assert seen["latched_checked"] > 0 and seen["latched_reactivated"] > 0, seen
    elif kind == "raw":
        assert seen["escaping_reactivated"] > 0, seen


def raw_fleet(cuda, tp, n=12):
    robots = [synth.fleet_robot(500 + i) for i in range(n)]
    fleet = cuda.fleet(n, 120, 120, 0.05, sc.PENTAGON, 0.55, 10.0, **(dict(trajectory_planner={}) if tp else DWA_CFG))
    fleet.set_maps(np.stack([r["raw"] for r in robots]), np.array([r["origin"] for r in robots]))
    poses = np.array([r["pose"] for r in robots])
    vels = np.array([r["vel"] for r in robots])
    fleet.set_plans(poses, [r["plan"] for r in robots])
    return fleet, robots, poses, vels


def run_cycles(fleet, robots, poses, vels, cycles=3):
    """Raw step results (bytes), oscillation masks and check costs over a few cycles with every robot planning."""
    trace = []
    cands = [CANDIDATES[:1 + i % 3] for i in range(len(robots))]
    p = poses.copy()
    for _ in range(cycles):
        fleet.set_plans(p, [r["plan"] for r in robots])
        res = bytes(fleet.step_raw(np.ascontiguousarray(p), vels))
        masks = [fleet.oscillation_mask(i) for i in range(len(robots))] if fleet.tp_cfg is None else None
        trace.append((res, masks, [c.tobytes() for c in fleet.check_trajectories(p, vels, cands)]))
        p = p + np.array([0.02, 0.0, 0.01])
    return trace


@pytest.mark.parametrize("tp", [False, True], ids=["dwa", "tp"])
def test_all_active_masks_change_nothing(cuda, tp):
    want = run_cycles(*raw_fleet(cuda, tp))
    ones = raw_fleet(cuda, tp)
    ones[0].set_active(np.ones(len(ones[1]), bool))
    assert run_cycles(*ones) == want
    reset = raw_fleet(cuda, tp)
    reset[0].set_active(np.arange(len(reset[1])) % 2 == 0)
    reset[0].set_active(None)
    assert run_cycles(*reset) == want


@pytest.mark.parametrize("tp", [False, True], ids=["dwa", "tp"])
def test_refusals_change_nothing(cuda, tp):
    def raises(call, text):
        with pytest.raises(NavGpuError, match=f"error 2: .*{text}"):
            call()

    fleet, robots, poses, vels = raw_fleet(cuda, tp)
    twin = raw_fleet(cuda, tp)[0]
    n = len(robots)
    lib = cuda.lib
    mask = np.arange(n) % 3 != 0  # robots 0, 3, 6, 9 are never planned
    for f in (fleet, twin):
        f.set_active(mask)
        f.step(poses, vels)
    # a refused mask leaves the previous one in place
    bad = np.ones(n, np.uint8)
    bad[5] = 2
    raises(lambda: cuda.check(lib.navgpu_fleet_set_active(fleet.h, _p(bad, _u8p))), "not 0 or 1")
    # checks: null pointers, offsets that decrease or do not start at 0, candidates of a never-planned robot
    cands = [CANDIDATES[:2] if i % 3 else np.zeros((0, 3)) for i in range(n)]
    off = np.zeros(n + 1, np.int32)
    off[1:] = np.cumsum([len(c) for c in cands])
    s = np.ascontiguousarray(np.concatenate(cands))
    costs = np.zeros(len(s))
    args = [_p(poses, _f64p), _p(vels, _f64p), _p(off, _i32p), _p(s, _f64p), _p(costs, _f64p)]
    for k in range(5):
        nulled = list(args)
        nulled[k] = None
        raises(lambda: cuda.check(lib.navgpu_fleet_check_trajectories(fleet.h, *nulled)), "bad arguments")
    dec = off.copy()
    dec[4] = dec[5] + 1
    raises(lambda: cuda.check(lib.navgpu_fleet_check_trajectories(fleet.h, *args[:2], _p(dec, _i32p), *args[3:])),
           "decrease")
    shifted = off + 1
    raises(lambda: cuda.check(lib.navgpu_fleet_check_trajectories(fleet.h, *args[:2], _p(shifted, _i32p), *args[3:])),
           "start at 0")
    with pytest.raises(NavGpuError, match="error 2: .*robot 0 .*never"):
        fleet.check_trajectories(poses, vels, [CANDIDATES[:1]] * n)
    assert not costs.any()
    # the fleet then works as its twin, which made none of these calls
    if not tp:
        assert [fleet.oscillation_mask(i) for i in range(n)] == [twin.oscillation_mask(i) for i in range(n)]
    a, b = fleet.check_trajectories(poses, vels, cands), twin.check_trajectories(poses, vels, cands)
    assert [x.tobytes() for x in a] == [y.tobytes() for y in b]
    for _ in range(2):
        a, b = fleet.step(poses, vels), twin.step(poses, vels)
        assert a == b and all((g is None) == (not m) for g, m in zip(a, mask))
        if not tp:
            assert [fleet.oscillation_mask(i) for i in range(n)] == [twin.oscillation_mask(i) for i in range(n)]


@pytest.mark.parametrize("tp", [False, True], ids=["dwa", "tp"])
def test_check_launch_count_does_not_grow(cuda, tp):
    counts = []
    for n, k in ((8, 1), (64, 32)):
        robots = [synth.fleet_robot(i) for i in range(n)]
        fleet = cuda.fleet(n, 120, 120, 0.05, sc.PENTAGON, 0.55, 10.0,
                           **(dict(trajectory_planner={}) if tp else DWA_CFG))
        fleet.set_maps(np.stack([r["raw"] for r in robots]), np.array([r["origin"] for r in robots]))
        poses = np.array([r["pose"] for r in robots])
        vels = np.array([r["vel"] for r in robots])
        fleet.set_plans(poses, [r["plan"] for r in robots])
        fleet.step(poses, vels)
        cands = [np.tile(CANDIDATES, (k // len(CANDIDATES) + 1, 1))[:k]] * n
        before = cuda.launch_count()
        fleet.check_trajectories(poses, vels, cands)
        counts.append(cuda.launch_count() - before)
    assert counts[0] == counts[1] == 1, counts


def inflate_like_fleet(port, robot):
    cm = port.costmap(120, 120, 0.05, *robot["origin"])
    s = cm.add_grid_layer(0)
    cm.add_inflation_layer(0.55, 10.0)
    cm.set_footprint(sc.PENTAGON)
    cm.set_grid_layer(s, robot["raw"])
    cm.update_map(0, 0, 0)
    return cm.get()


@pytest.mark.parametrize("tp", [False, True], ids=["dwa", "tp"])
def test_full_size_checks_sampled_through_checker(cuda, port, tp):
    """4096 robots of config C5's inputs, half of them left out of the second step, then one candidate each; every
    128th robot is replayed through the checker."""
    n = 4096
    robots = [synth.fleet_robot(i) for i in range(n)]
    cfg = dict(vx_samples=20, vy_samples=1, vth_samples=20, max_vel_y=0.0, min_vel_y=0.0)
    fleet = cuda.fleet(n, 120, 120, 0.05, sc.PENTAGON, 0.55, 10.0, **(dict(trajectory_planner={}) if tp else cfg))
    fleet.set_maps(np.stack([r["raw"] for r in robots]), np.array([r["origin"] for r in robots]))
    poses = np.array([r["pose"] for r in robots])
    vels = np.array([r["vel"] for r in robots])
    fleet.set_plans(poses, [r["plan"] for r in robots])
    fleet.step(poses, vels)
    active = np.arange(n) % 2 == 1
    fleet.set_active(active)
    poses2 = poses + np.array([0.03, -0.01, 0.02])
    if not tp:
        fleet.set_plans(poses2, [r["plan"] for r in robots])
    out = fleet.step(poses2, vels)
    cands = [CANDIDATES[i % len(CANDIDATES)][None, :] for i in range(n)]
    costs = fleet.check_trajectories(poses2, vels, cands)
    sample = range(0, n, 128)
    exact = 0
    for i in list(sample) + [i + 1 for i in sample]:
        grid = inflate_like_fleet(port, robots[i])
        if tp:
            h = port.trajectory_planner(120, 120, 0.05, sc.PENTAGON)
            h.set_costmap(grid, *robots[i]["origin"])
            h.update_plan(robots[i]["plan"])
            h.find_best_path(poses[i], vels[i])
            if active[i]:
                e = h.find_best_path(poses2[i], vels[i])
                assert same_tp(out[i], e, RTOL), f"robot {i}: {out[i]} vs cost {e['cost']}"
            c = h.score_trajectory(poses2[i], vels[i], cands[i][0])
        else:
            h = port.dwa(120, 120, 0.05, **cfg)
            h.set_costmap(grid, *robots[i]["origin"])
            h.set_plan(poses[i], robots[i]["plan"])
            h.find_best_path(poses[i], vels[i], sc.PENTAGON)
            h.set_plan(poses2[i], robots[i]["plan"])
            if active[i]:
                e = h.find_best_path(poses2[i], vels[i], sc.PENTAGON)
                assert same_dwa(out[i], e, RTOL), f"robot {i}: {out[i]} vs cost {e['cost']}"
            c = h.check_trajectory(poses2[i], vels[i], cands[i][0], sc.PENTAGON)
        assert np.isclose(costs[i][0], c, rtol=RTOL, atol=0), f"robot {i}: fleet {costs[i][0]} vs checker {c}"
        exact += costs[i][0] == c
    print(f"{'TrajectoryPlanner' if tp else 'DWA'} fleet goal checks: {exact} of {2 * len(sample)} checker costs "
          f"bit-equal")
