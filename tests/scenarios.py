"""Seeded random scenarios shared by the oracle-vs-reference and GPU-vs-oracle parity tests."""
import numpy as np

from oracle import pyoracle as po


def square_footprint(half=0.325):
    return [(half, half), (half, -half), (-half, -half), (-half, half)]


PENTAGON = [(-0.325, -0.325), (-0.325, 0.325), (0.325, 0.325), (0.46, 0.0), (0.325, -0.325)]  # costmap_params.yaml:21


def random_layer(rng, sy, sx, kind):
    """kind: 'blocks' axis-aligned thick structure (tie-free), 'salt' single cells, 'values' arbitrary bytes."""
    g = np.zeros((sy, sx), np.uint8)
    if kind == "blocks":
        for _ in range(max(2, sx * sy // 2500)):
            w, h = rng.integers(3, max(4, sx // 5)), rng.integers(3, max(4, sy // 5))
            x, y = rng.integers(0, sx - 2), rng.integers(0, sy - 2)
            g[y:y + h, x:x + w] = 254
    elif kind == "salt":
        g[rng.random((sy, sx)) < 0.01] = 254
    elif kind == "values":
        g = rng.choice(np.array([0, 0, 0, 1, 50, 100, 128, 200, 252, 253, 254, 255], np.uint8), size=(sy, sx))
    elif kind == "values_nolethal":  # no isolated LETHAL cells: keeps a scenario in the tie-free class
        g = rng.choice(np.array([0, 0, 0, 1, 50, 100, 128, 200, 252, 253, 255, 255], np.uint8), size=(sy, sx))
    return g


def random_observations(rng, sx, sy, res, ox, oy, n_obs, n_pts, spread=1.3):
    obs = []
    for _ in range(n_obs):
        # origins mostly inside the map, sometimes outside (whole observation skipped for clearing)
        o = (ox + rng.uniform(-0.1, 1.1) * sx * res, oy + rng.uniform(-0.1, 1.1) * sy * res, rng.uniform(0, 1))
        ang = rng.uniform(0, 2 * np.pi, n_pts)
        rad = rng.uniform(0.0, spread * max(sx, sy) * res, n_pts)
        pts = np.stack([o[0] + rad * np.cos(ang), o[1] + rad * np.sin(ang), rng.uniform(-0.2, 2.5, n_pts)], 1)
        obs.append(dict(origin=o, points=pts.astype(np.float32), obstacle_range=float(rng.uniform(1.0, 8.0)),
                        raytrace_range=float(rng.uniform(1.0, 8.0)), marking=bool(rng.random() < 0.8),
                        clearing=bool(rng.random() < 0.8)))
    return obs


def build_stack(api, rng, sx, sy, res, ox, oy, rolling, track_unknown, layer_kind="blocks", with_obstacle=True,
                with_inflation=True, radius=0.55, scaling=10.0, extra_policy=None):
    """static(TrueOverwrite|Max) [+ extra grid layer] [+ obstacle] [+ inflation]; returns (costmap, ids)."""
    cm = api.costmap(sx, sy, res, ox, oy, rolling=rolling, track_unknown=track_unknown)
    ids = {}
    if not rolling:
        ids["static"] = cm.add_grid_layer(po.TRUE_OVERWRITE if rng.random() < 0.7 else po.MAX)
    if extra_policy is not None:
        ids["extra"] = cm.add_grid_layer(extra_policy)
    if with_obstacle:
        ids["obstacle"] = cm.add_obstacle_layer(int(rng.integers(0, 2)), bool(rng.random() < 0.7), 2.0)
    if with_inflation:
        ids["inflation"] = cm.add_inflation_layer(radius, scaling)
    cm.set_footprint(square_footprint())
    return cm, ids


def local_costmap(api, rng, n=120, res=0.05, ox=0.0, oy=0.0, style="corridor"):
    """A C2-style local costmap (no NO_INFORMATION cells): walls/boxes inflated by the oracle itself."""
    cm = api.costmap(n, n, res, ox, oy)
    s = cm.add_grid_layer(po.TRUE_OVERWRITE)
    cm.add_inflation_layer(0.55, 10.0)
    cm.set_footprint(PENTAGON)
    g = np.zeros((n, n), np.uint8)
    if style == "corridor":
        lo, hi = int(n * 0.25), int(n * 0.75)
        g[:lo - 1, :] = 0
        g[lo - 4:lo - 1, :] = 254
        g[hi + 1:hi + 4, :] = 254
        bx, by = int(rng.integers(n // 2, n - 20)), int(rng.integers(lo + 8, hi - 14))
        g[by:by + 6, bx:bx + 6] = 254
    elif style == "clutter":
        for _ in range(int(rng.integers(3, 9))):
            x, y = rng.integers(0, n - 8, 2)
            w, h = rng.integers(2, 8, 2)
            g[y:y + h, x:x + w] = 254
    elif style == "empty":
        pass
    cm.set_grid_layer(s, g)
    cm.update_map(0, 0, 0)
    return cm.get()


def dwa_scenario(rng, n=120, res=0.05, style=None):
    """Returns dict(origin, pose, vel, plan) for a local map of n x n cells."""
    style = style or str(rng.choice(["corridor", "clutter", "empty"]))
    ox, oy = float(rng.uniform(-5, 5)), float(rng.uniform(-5, 5))
    size = n * res
    pose = (ox + size * rng.uniform(0.2, 0.5), oy + size * rng.uniform(0.4, 0.6), float(rng.uniform(-0.6, 0.6)))
    vel = (float(rng.uniform(0.0, 0.5)), 0.0, float(rng.uniform(-0.5, 0.5)))
    # plan: polyline from behind the robot to beyond the map edge (so it leaves the window), some sparse gaps
    npts = int(rng.integers(20, 200))
    t = np.linspace(-0.1, 1.3, npts)
    px = pose[0] + t * size * 0.7
    py = pose[1] + 0.3 * np.sin(t * rng.uniform(1, 4)) * rng.uniform(0, 1.5)
    return dict(style=style, origin=(ox, oy), pose=pose, vel=vel, plan=np.stack([px, py], 1))


INFLATION_SEMANTICS = {
    # name: (checker variant of navo_inflation_set_variant, libnavgpu mode of navgpu_inflation_set_mode)
    "reference": (0, None),   # libstdc++ heap order, the reference as compiled (checker only)
    "fifo": (1, None), "lifo": (2, None), "random": (3, None),
    "exact": (4, 0),          # exact windowed nearest-seed inflation
    "propagate": (5, 1),      # level-synchronous nearest-source propagation
    "certificate": (6, None),
}
# the sampled tie policies whose disagreement with the reference defines a scenario's tie-variant mask
TIE_POLICIES = [("fifo", 0), ("lifo", 0)] + [("random", s) for s in range(1, 17)]


def select_inflation(cm, layer, which, seed=0):
    """Pick the inflation semantics on a checker costmap (variant) or a CUDA costmap (mode)."""
    if which is None:
        return
    variant, mode = INFLATION_SEMANTICS[which]
    if hasattr(cm, "set_inflation_variant"):
        cm.set_inflation_variant(layer, variant, seed)
    else:
        assert mode is not None, f"libnavgpu has no inflation mode for '{which}'"
        cm.set_inflation_mode(layer, mode)


def run_costmap_scenario(api, seed, cycles=4, max_size=90, tie_free=False, inflation=None, inflation_seed=0,
                         on_cycle=None):
    """Multi-cycle LayeredCostmap scenario; returns per cycle (window, master, obstacle-layer grid, origin).
    `inflation` (a key of INFLATION_SEMANTICS) selects which execution of InflationLayer::updateCosts runs.

    `api` is anything shaped like oracle.pyoracle.Api (the oracles and the CUDA binding all are).
    tie_free=True restricts obstacle sources to thick axis-aligned blocks (no marking of single points), the class on
    which every tie policy of the reference's priority queue gives the same grid (SURVEY.md section 7).
    """
    rng = np.random.default_rng(seed)
    sx, sy = int(rng.integers(20, max_size)), int(rng.integers(20, max_size))
    res = float(rng.choice([0.05, 0.1, 0.25]))
    ox, oy = float(rng.uniform(-3, 3)), float(rng.uniform(-3, 3))
    rolling = bool(rng.random() < 0.4)
    tu = bool(rng.random() < 0.4)
    kind = "blocks" if tie_free else str(rng.choice(["blocks", "salt", "values"]))
    extra = [None, po.OVERWRITE, po.MAX, po.ADDITION][int(rng.integers(0, 4))]
    radius = float(rng.choice([0.3, 0.55, 1.0]))
    scaling = float(rng.choice([1.0, 10.0]))
    cm, ids = build_stack(api, rng, sx, sy, res, ox, oy, rolling, tu, kind, radius=radius, scaling=scaling,
                          extra_policy=extra)
    select_inflation(cm, ids["inflation"], inflation, inflation_seed)
    trace = []
    rx, ry = ox + sx * res / 2, oy + sy * res / 2
    for cyc in range(cycles):
        if "static" in ids and (cyc == 0 or rng.random() < 0.3):
            cm.set_grid_layer(ids["static"], random_layer(rng, sy, sx, kind))
        if "extra" in ids and (cyc == 0 or rng.random() < 0.5):
            cm.set_grid_layer(ids["extra"], random_layer(rng, sy, sx, "values_nolethal" if tie_free else "values"))
        obs = random_observations(rng, sx, sy, res, ox, oy, int(rng.integers(0, 4)), 40)
        if tie_free:
            for o in obs:
                o["marking"] = False
        cm.set_observations(ids["obstacle"], obs)
        rx += rng.uniform(-0.5, 0.5)
        ry += rng.uniform(-0.5, 0.5)
        w = cm.update_map(rx, ry, float(rng.uniform(-3, 3)))
        if on_cycle is not None:
            on_cycle(cm, cyc, w)
        trace.append((w, cm.get().copy(), cm.get_layer(ids["obstacle"]).copy(), cm.origin()))
    return trace


def tie_mask_trace(port, seed, **kw):
    """Per cycle: the cells of the master grid on which some sampled tie policy of the reference's priority queue
    (TIE_POLICIES, each a full run of the scenario) disagrees with the reference's own heap order."""
    base = run_costmap_scenario(port, seed, inflation="reference", **kw)
    masks = [np.zeros_like(c[1], bool) for c in base]
    for which, s in TIE_POLICIES:
        tr = run_costmap_scenario(port, seed, inflation=which, inflation_seed=s, **kw)
        for m, a, b in zip(masks, tr, base):
            m |= a[1] != b[1]
    return base, masks


def run_dwa_scenario(api, grid_api, seed, cycles=5):
    """Multi-cycle DWAPlanner scenario; the local costmap is produced by `grid_api` (an oracle)."""
    rng = np.random.default_rng(seed)
    s = dwa_scenario(rng)
    grid = local_costmap(grid_api, np.random.default_rng(seed + 1000), ox=s["origin"][0], oy=s["origin"][1],
                         style=s["style"])
    over = dict(vx_samples=int(rng.integers(1, 12)), vy_samples=int(rng.integers(1, 4)),
                vth_samples=int(rng.integers(1, 25)))
    if rng.random() < 0.3:
        over.update(max_vel_y=0.0, min_vel_y=0.0)
    if rng.random() < 0.2:
        over.update(use_dwa=0)
    if rng.random() < 0.2:
        over.update(sum_scores=1)
    if rng.random() < 0.3:
        over.update(min_vel_x=-0.2)
    d = api.dwa(120, 120, 0.05, **over)
    d.set_costmap(grid, *s["origin"])
    out = []
    pose = np.array(s["pose"])
    vel = np.array(s["vel"])
    for cyc in range(cycles):
        d.set_plan(pose, s["plan"])
        r = d.find_best_path(pose, vel, PENTAGON)
        r["mask"] = d.oscillation_mask()
        r["grids"] = [d.grid(k) for k in range(4)]
        out.append(r)
        # alternate forward/backward so the oscillation flags latch
        vel = np.array([r["xv"] * (-1 if cyc % 2 else 1), r["yv"], -r["thetav"]]) if r["ok"] else vel * 0
        pose = pose + np.array([0.01 * vel[0], 0, 0.01 * vel[2]])
    return out


def dwa_results_equal(a, b, rtol=0.0):
    """Exact (rtol=0) or relative comparison of two find_best_path result dicts."""
    if (a["ok"], a["best_index"], a["n_samples"], a["n_scored"], a["mask"]) != \
       (b["ok"], b["best_index"], b["n_samples"], b["n_scored"], b["mask"]):
        return False
    if not all(np.array_equal(x, y) for x, y in zip(a["grids"], b["grids"])):
        return False
    if rtol == 0.0:
        return (a["cost"] == b["cost"] and (a["xv"], a["yv"], a["thetav"]) == (b["xv"], b["yv"], b["thetav"]) and
                np.array_equal(a["costs"], b["costs"], equal_nan=True) and np.array_equal(a["points"], b["points"]))
    ok = np.isclose(a["cost"], b["cost"], rtol=rtol, atol=0) and \
        np.allclose(a["costs"], b["costs"], rtol=rtol, atol=0, equal_nan=True) and \
        np.allclose(a["points"], b["points"], rtol=rtol, atol=1e-12)
    return bool(ok)


def run_voxel_scenario(api, seed, cycles=4, max_size=70, inflation=None):
    """Multi-cycle LayeredCostmap scenario with a VoxelLayer (3-D ray-trace clearing + marking) [+ inflation];
    returns per cycle (window, master, voxel layer's 2-D grid, voxel columns, origin).  mark_threshold stays 0 (the
    reference's default): with a positive threshold the reference's bounds depend on the order of the cloud points."""
    rng = np.random.default_rng(seed)
    sx, sy = int(rng.integers(20, max_size)), int(rng.integers(20, max_size))
    res = float(rng.choice([0.05, 0.1, 0.25]))
    ox, oy = float(rng.uniform(-3, 3)), float(rng.uniform(-3, 3))
    rolling = bool(rng.random() < 0.4)
    tu = bool(rng.random() < 0.5)
    z_voxels = int(rng.choice([4, 10, 16]))
    z_res = float(rng.choice([0.1, 0.2]))
    origin_z = float(rng.choice([0.0, -0.1]))
    unknown_threshold = int(rng.choice([0, 8, 15]))
    max_h = float(rng.choice([1.0, 2.0]))
    cm = api.costmap(sx, sy, res, ox, oy, rolling=rolling, track_unknown=tu)
    ids = {}
    if not rolling:
        ids["static"] = cm.add_grid_layer(po.TRUE_OVERWRITE)
    ids["voxel"] = cm.add_voxel_layer(int(rng.integers(0, 2)), bool(rng.random() < 0.7), max_h, origin_z, z_res, z_voxels,
                                      unknown_threshold, 0)
    with_inflation = bool(rng.random() < 0.5)
    if with_inflation:
        ids["inflation"] = cm.add_inflation_layer(0.3, 10.0)
        select_inflation(cm, ids["inflation"], inflation)
    cm.set_footprint(square_footprint())
    trace = []
    rx, ry = ox + sx * res / 2, oy + sy * res / 2
    for cyc in range(cycles):
        if "static" in ids and cyc == 0:
            cm.set_grid_layer(ids["static"], random_layer(rng, sy, sx, "blocks"))
        obs = random_observations(rng, sx, sy, res, ox, oy, int(rng.integers(1, 4)), 60)
        for o in obs:  # sensor heights and point heights inside and outside the voxel column
            o["origin"] = (o["origin"][0], o["origin"][1], float(rng.uniform(-0.3, z_voxels * z_res + 0.3)))
            o["points"][:, 2] = rng.uniform(-0.4, z_voxels * z_res + 0.5, len(o["points"])).astype(np.float32)
        cm.set_observations(ids["voxel"], obs)
        rx += rng.uniform(-0.5, 0.5)
        ry += rng.uniform(-0.5, 0.5)
        w = cm.update_map(rx, ry, float(rng.uniform(-3, 3)))
        trace.append((w, cm.get().copy(), cm.get_layer(ids["voxel"]).copy(), cm.get_voxels(ids["voxel"]).copy(), cm.origin()))
    return trace, with_inflation


def run_tp_scenario(api, grid_api, seed, cycles=6):
    """Multi-cycle scenario of the legacy base_local_planner::TrajectoryPlanner (findBestPath + scoreTrajectory).
    `api` needs .trajectory_planner (the CUDA binding and the compiled reference have it); the local costmap comes from
    `grid_api`.  A third of the seeds start the robot against a wall or turned away from the plan, so that the
    in-place-rotation, strafing and back-up branches of createTrajectories and their latched flags are exercised."""
    rng = np.random.default_rng(seed + 5000)
    s = dwa_scenario(rng)
    grid = local_costmap(grid_api, np.random.default_rng(seed + 6000), ox=s["origin"][0], oy=s["origin"][1],
                         style=s["style"])
    over = dict(vx_samples=int(rng.integers(1, 9)), vtheta_samples=int(rng.integers(1, 21)),
                holonomic_robot=int(rng.random() < 0.6), dwa=int(rng.random() < 0.7),
                sim_time=float(rng.choice([1.0, 1.7, 0.5])))
    if rng.random() < 0.15:
        over.update(simple_attractor=1)
    if rng.random() < 0.3:
        over.update(angular_sim_granularity=0.1)
    if rng.random() < 0.3:
        over.update(y_vels=[-0.2, 0.2])
    if rng.random() < 0.2:
        over.update(min_vel_x=-0.1)
    if seed % 5 == 4:  # heading scoring: distances and the heading difference of the one step at heading_scoring_timestep
        over.update(heading_scoring=1, heading_scoring_timestep=float([0.1, 0.8, 0.45][(seed // 5) % 3]))
        over.pop("simple_attractor", None)
    tp = api.trajectory_planner(120, 120, 0.05, PENTAGON, **over)
    tp.set_costmap(grid, *s["origin"])
    tp.update_plan(s["plan"])
    pose = np.array(s["pose"])
    vel = np.array(s["vel"])
    mode = int(rng.integers(0, 3))
    if mode == 1:  # nose against the lower corridor wall / a random heading
        pose[2] = float(rng.uniform(-3.1, 3.1))
        if s["style"] == "corridor":
            pose[1] = s["origin"][1] + (0.25 * 120 + rng.uniform(6, 12)) * 0.05
    elif mode == 2:  # inside an inflated / lethal area: nothing but backing up is legal
        ys, xs = np.nonzero(grid >= 253)
        if len(xs):
            k = int(rng.integers(0, len(xs)))
            pose[0] = s["origin"][0] + (xs[k] + 0.5) * 0.05
            pose[1] = s["origin"][1] + (ys[k] + 0.5) * 0.05
    out = []
    for cyc in range(cycles):
        if cyc == 3 and rng.random() < 0.5:
            tp.update_plan(s["plan"][: max(2, len(s["plan"]) // 2)])
        r = tp.find_best_path(pose, vel)
        r["grids"] = [tp.grid(0), tp.grid(1)]
        probes = [(0.3, 0.0, 0.2), (float(rng.uniform(-0.2, 0.5)), float(rng.choice([0.0, 0.1])), float(rng.uniform(-1, 1)))]
        r["scores"] = np.array([tp.score_trajectory(pose, vel, p) for p in probes])
        out.append(r)
        vel = np.array([r["xv"], r["yv"], r["thetav"]]) if r["cost"] >= 0 else vel * 0
        step = float(rng.choice([0.02, 0.2]))  # below / above oscillation_reset_dist and escape_reset_dist
        pose = pose + np.array([step * vel[0] * np.cos(pose[2]), step * vel[0] * np.sin(pose[2]), step * vel[2]])
    return out


def tp_results_equal(a, b, rtol=0.0):
    if a["flags"] != b["flags"] or len(a["points"]) != len(b["points"]):
        return False
    if not all(np.array_equal(x, y) for x, y in zip(a["grids"], b["grids"])):
        return False
    if (a["xv"], a["yv"], a["thetav"]) != (b["xv"], b["yv"], b["thetav"]):
        return False
    if rtol == 0.0:
        return a["cost"] == b["cost"] and np.array_equal(a["points"], b["points"]) and np.array_equal(a["scores"], b["scores"])
    return bool(np.isclose(a["cost"], b["cost"], rtol=rtol, atol=0) and
                np.allclose(a["points"], b["points"], rtol=rtol, atol=1e-12) and
                np.allclose(a["scores"], b["scores"], rtol=rtol, atol=0))


def run_tp_boxed_scenario(api, cycles=9, reconfigure=None):
    """The legacy TrajectoryPlanner in a slot just wider than the robot, open along y: driving forward and rotating in
    place collide, so createTrajectories falls through to strafing (trajectory_planner.cpp:752-797); the plan is then
    reversed (the other strafing direction wins and the first one is latched as stuck), and finally the slot is closed
    on both sides, which leaves backing up and escape mode (:851-903).  `reconfigure`: {cycle: overrides} applied
    before that cycle's findBestPath."""
    n, res = 120, 0.05
    grid = np.zeros((n, n), np.uint8)
    grid[:, 50:52] = 254   # wall behind the robot: x in [2.50, 2.60)
    grid[:, 70:72] = 254   # wall ahead: x in [3.50, 3.60)
    tp = api.trajectory_planner(n, n, res, PENTAGON, holonomic_robot=1, vx_samples=4, vtheta_samples=10)
    tp.set_costmap(grid, 0.0, 0.0)
    plan = np.stack([np.full(60, 3.0), np.linspace(3.0, 5.9, 60)], 1)  # the plan runs along the slot
    tp.update_plan(plan)
    pose = np.array([3.0, 3.0, 0.0])
    vel = np.zeros(3)
    out = []
    for cyc in range(cycles):
        if cyc == 3:
            tp.update_plan(np.stack([np.full(60, 3.0), np.linspace(3.0, 0.1, 60)], 1))
        if cyc == 6:
            closed = grid.copy()
            closed[49:51, :] = 254
            closed[70:72, :] = 254
            tp.set_costmap(closed, 0.0, 0.0)
        if reconfigure and cyc in reconfigure:
            tp.reconfigure(**reconfigure[cyc])
        r = tp.find_best_path(pose, vel)
        r["grids"] = [tp.grid(0), tp.grid(1)]
        r["scores"] = np.array([tp.score_trajectory(pose, vel, (0.0, 0.1, 0.0)), tp.score_trajectory(pose, vel, (0.1, 0.0, 0.0))])
        out.append(r)
        vel = np.array([r["xv"], r["yv"], r["thetav"]]) if r["cost"] >= 0 else vel * 0
        pose = pose + np.array([0.0, 0.01 * vel[1], 0.0])  # creep: below oscillation_reset_dist, the flags stay latched
    return out


def tp_utest_footprint_obstacles(api):
    """base_local_planner/test/utest.cpp:86-110 (TrajectoryPlannerTest::footprintObstacles) through scoreTrajectory:
    10 x 10 map at 1 m, square footprint of +-2 m, the robot at (4.5, 4.5) heading +y, an obstacle at cell (4, 6).
    Driving into it with (vx 4, acc 4) and rotating with (vtheta pi/2, acc pi/4) must both come back as -1."""
    fp = [(2, 2), (2, -2), (-2, -2), (-2, 2)]
    grid = np.zeros((10, 10), np.uint8)
    grid[6, 4] = 254
    out = []
    for acc, samp in (((4.0, 0.0, 0.0), (4.0, 0.0, 0.0)), ((0.0, 0.0, np.pi / 4), (0.0, 0.0, np.pi / 2))):
        tp = api.trajectory_planner(10, 10, 1.0, fp, acc_lim_x=acc[0], acc_lim_y=acc[1], acc_lim_theta=acc[2], sim_time=1.0,
                                    sim_granularity=1.0, vx_samples=2)
        tp.set_costmap(grid, 0.0, 0.0)
        out.append(tp.score_trajectory((4.5, 4.5, np.pi / 2), (0.0, 0.0, 0.0), samp))
    # and with the obstacle out of the footprint's way the same commands are legal
    grid2 = np.zeros((10, 10), np.uint8)
    grid2[9, 9] = 254
    tp = api.trajectory_planner(10, 10, 1.0, fp, acc_lim_x=4.0, acc_lim_y=0.0, acc_lim_theta=0.0, sim_time=1.0,
                                sim_granularity=1.0, vx_samples=2, simple_attractor=1)
    tp.set_costmap(grid2, 0.0, 0.0)
    tp.update_plan([(4.5, 4.5), (4.5, 6.5)])
    out.append(tp.score_trajectory((4.5, 4.5, np.pi / 2), (0.0, 0.0, 0.0), (1.0, 0.0, 0.0)))
    return out


def run_tp_edge_cases(api, grid_api):
    """Corner cases of the legacy TrajectoryPlanner: no plan at all, a degenerate (2-vertex) and an empty footprint,
    a one-pose plan, a robot outside the map, unknown cells with allow_unknown on and off (allow_unknown is honoured by
    the CUDA path and the restatement; the reference's own flag is uninitialised, so unknown cells stay out of the way
    of anything it is compared on)."""
    rng = np.random.default_rng(77)
    s = dwa_scenario(rng, style="corridor")
    grid = local_costmap(grid_api, np.random.default_rng(78), ox=s["origin"][0], oy=s["origin"][1], style="corridor")
    out = []
    cases = [
        dict(fp=PENTAGON, plan=None, pose=s["pose"]),
        dict(fp=[(-0.2, 0.0), (0.3, 0.0)], plan=s["plan"], pose=s["pose"]),
        dict(fp=[], plan=s["plan"], pose=s["pose"]),
        dict(fp=PENTAGON, plan=s["plan"][:1], pose=s["pose"]),
        dict(fp=PENTAGON, plan=s["plan"], pose=(s["origin"][0] - 1.0, s["origin"][1] + 3.0, 0.0)),
    ]
    for c in cases:
        tp = api.trajectory_planner(120, 120, 0.05, c["fp"], vx_samples=3, vtheta_samples=5)
        tp.set_costmap(grid, *s["origin"])
        if c["plan"] is not None:
            tp.update_plan(c["plan"])
        for cyc in range(2):
            r = tp.find_best_path(c["pose"], s["vel"])
            r["grids"] = [tp.grid(0), tp.grid(1)]
            r["scores"] = np.array([tp.score_trajectory(c["pose"], s["vel"], (0.2, 0.0, 0.1))])
            out.append(r)
    return out


def run_dwa_sequence(api, grid, origin, pose, plan, vel, ops, **create):
    """A DWAPlanner handle driven through `ops` on one local costmap.  Ops: ("reconfigure", overrides), ("plan",) =
    updatePlanAndLocalCosts at the current pose, ("plan_at", pose, plan), ("find",), ("check", [vel_samples, ...]),
    ("follow",) = take the last result as the next velocity, alternating forward and backward so that the oscillation
    flags latch (as run_dwa_scenario does), ("costmap", grid).  Returns one record per "find" / "check"."""
    d = api.dwa(120, 120, 0.05, **create)
    d.set_costmap(grid, *origin)
    pose, vel = np.array(pose, dtype=np.float64), np.array(vel, dtype=np.float64)
    out, last, n_find = [], None, 0
    for op in ops:
        if op[0] == "reconfigure":
            d.reconfigure(**op[1])
        elif op[0] == "plan":
            d.set_plan(pose, plan)
        elif op[0] == "plan_at":
            d.set_plan(op[1], op[2])
        elif op[0] == "costmap":
            d.set_costmap(op[1], *origin)
        elif op[0] == "find":
            last = d.find_best_path(pose, vel, PENTAGON)
            last["mask"] = d.oscillation_mask()
            last["grids"] = [d.grid(k) for k in range(4)]
            last["cfg"] = bytes(d.cfg)
            last["pose"], last["vel"] = pose.copy(), vel.copy()
            out.append(last)
            n_find += 1
        elif op[0] == "check":
            out.append(dict(checks=[d.check_trajectory(pose, vel, v, PENTAGON) for v in op[1]], mask=d.oscillation_mask()))
        elif op[0] == "follow":
            vel = (np.array([last["xv"] * (-1 if n_find % 2 == 0 else 1), last["yv"], -last["thetav"]]) if last["ok"]
                   else vel * 0)
            pose = pose + np.array([0.01 * vel[0], 0, 0.01 * vel[2]])
    return out


def run_tp_sequence(api, grid, origin, pose, plan, vel, ops, footprint=PENTAGON, **create):
    """A legacy TrajectoryPlanner handle driven through `ops`: ("reconfigure", overrides), ("footprint", xy),
    ("plan", plan), ("find",) = findBestPath + both distance maps + two scoreTrajectory probes, ("follow", step) = take
    the last result as the next velocity and move by step x velocity.  Returns one record per "find"."""
    tp = api.trajectory_planner(120, 120, 0.05, footprint, **create)
    tp.set_costmap(grid, *origin)
    if plan is not None:
        tp.update_plan(plan)
    pose, vel = np.array(pose, dtype=np.float64), np.array(vel, dtype=np.float64)
    out = []
    for op in ops:
        if op[0] == "reconfigure":
            tp.reconfigure(**op[1])
        elif op[0] == "footprint":
            tp.set_footprint(op[1])
        elif op[0] == "plan":
            tp.update_plan(op[1])
        elif op[0] == "find":
            r = tp.find_best_path(pose, vel)
            r["grids"] = [tp.grid(0), tp.grid(1)]
            r["scores"] = np.array([tp.score_trajectory(pose, vel, p) for p in ((0.3, 0.0, 0.2), (0.0, 0.1, -0.6))])
            out.append(r)
        elif op[0] == "follow":
            vel = np.array([out[-1]["xv"], out[-1]["yv"], out[-1]["thetav"]]) if out[-1]["cost"] >= 0 else vel * 0
            pose = pose + np.array([op[1] * vel[0] * np.cos(pose[2]), op[1] * vel[0] * np.sin(pose[2]), op[1] * vel[2]])
    return out


def reconfigure_world(seed=3, style="corridor", unknown=False):
    """A local costmap, pose, velocity and plan of dwa_scenario for the reconfigure sequences; `unknown` marks a band of
    NO_INFORMATION cells across the robot's way."""
    from oracle import pyoracle
    rng = np.random.default_rng(seed)
    s = dwa_scenario(rng, style=style)
    grid = local_costmap(pyoracle.load("port"), np.random.default_rng(seed + 1000), ox=s["origin"][0],
                         oy=s["origin"][1], style=style)
    if unknown:
        cx = int((s["pose"][0] - s["origin"][0]) / 0.05)
        grid[:, cx + 8:cx + 11] = 255
    return dict(grid=grid, origin=s["origin"], pose=s["pose"], plan=s["plan"], vel=s["vel"])


def dwa_reconfigure_cases():
    """name -> (world, create overrides, ops) of the DWAPlanner reconfigure sequences."""
    find = [("plan",), ("find",), ("check", [(0.3, 0.0, 0.2), (0.0, 0.0, 0.0), (0.5, 0.1, -0.7)]), ("follow",)]
    cases = {}
    # per-axis sample counts across the 640 values carried inline in the kernel parameters, and back, at one velocity:
    # the staged set of the second and the fourth search is the same
    xy0 = dict(max_vel_y=0.0, min_vel_y=0.0)
    cases["samples_inline_staged"] = (dict(seed=3), dict(vx_samples=20, vy_samples=1, vth_samples=20, **xy0), [
        ("plan",), ("find",), ("reconfigure", dict(vx_samples=400, vth_samples=400)), ("plan",), ("find",),
        ("reconfigure", dict(vx_samples=3, vy_samples=10, vth_samples=20, max_vel_y=0.1, min_vel_y=-0.1)), ("plan",),
        ("find",), ("reconfigure", dict(vx_samples=400, vy_samples=1, vth_samples=400, **xy0)), ("plan",), ("find",)])
    # the goal-front target and the alignment scale come from the configuration of set_plan; the reconfigure between
    # set_plan and findBestPath restores the alignment scale, which set_plan zeroed near the goal
    crit = dict(forward_point_distance=0.6, cheat_factor=2.0, path_distance_bias=20.0, goal_distance_bias=40.0)
    crit2 = dict(forward_point_distance=0.1, cheat_factor=0.5, path_distance_bias=32.0, goal_distance_bias=24.0)
    for where in ("near", "far", "far_then_near"):
        ops = []
        for k in range(3):
            near = where == "near" or (where == "far_then_near" and k > 0)
            ops += [("plan_at", None, near), ("reconfigure", crit if k % 2 == 0 else crit2), ("find",),
                    ("check", [(0.3, 0.0, 0.2), (0.1, 0.0, -0.5)])]
        cases[f"critics_{where}"] = (dict(seed=5, style="empty"), dict(vx_samples=6, vy_samples=1, vth_samples=9), ops)
    # oscillation flags latched by alternating commands, then new reset distance / angle, then further cycles
    # (without checkTrajectory, which resets the flags)
    step = [("plan",), ("find",), ("follow",)]
    cases["oscillation_reset"] = (dict(seed=11), dict(vx_samples=5, vy_samples=3, vth_samples=7, min_vel_x=-0.2),
                                  step * 4 + [("reconfigure", dict(oscillation_reset_dist=0.001,
                                                                   oscillation_reset_angle=0.01))] + step * 3)
    cases["use_dwa_sum_scores"] = (dict(seed=7), dict(vx_samples=5, vy_samples=2, vth_samples=8), find + [
        ("reconfigure", dict(use_dwa=0))] + find + [("reconfigure", dict(use_dwa=1, sum_scores=1))] + find + [
        ("reconfigure", dict(sum_scores=0))] + find)
    cases["allow_unknown"] = (dict(seed=7, unknown=True), dict(vx_samples=5, vy_samples=1, vth_samples=8), find + [
        ("reconfigure", dict(allow_unknown=1))] + find + [("reconfigure", dict(allow_unknown=0))] + find)
    cases["limits_and_horizon"] = (dict(seed=13), dict(vx_samples=6, vy_samples=3, vth_samples=9), find + [
        ("reconfigure", dict(max_vel_x=0.3, max_trans_vel=0.35, min_rot_vel=0.2, max_rot_vel=0.6, acc_lim_x=1.0,
                             acc_lim_theta=6.0))] + find + [
        ("reconfigure", dict(sim_time=3.0, sim_granularity=0.01, angular_sim_granularity=0.05, sim_period=0.2))] + find + [
        ("reconfigure", dict(sim_time=0.8, sim_granularity=0.05, angular_sim_granularity=0.2))] + find)
    cases["zero_samples"] = (dict(seed=13), dict(vx_samples=4, vy_samples=2, vth_samples=6), find + [
        ("reconfigure", dict(vx_samples=0, vy_samples=0, vth_samples=0))] + find + [
        ("reconfigure", dict(vx_samples=-3, vy_samples=1, vth_samples=5))] + find + [
        ("reconfigure", dict(vx_samples=4, vy_samples=2, vth_samples=6))] + find)
    return cases


def dwa_case_world(case):
    world, create, ops = dwa_reconfigure_cases()[case]
    w = reconfigure_world(**world)
    resolved = []
    for op in ops:
        if op[0] == "plan_at":  # near: a plan that ends 0.3 m ahead of the robot; far: the scenario's plan
            if op[2]:
                p = np.array(w["pose"][:2])
                resolved.append(("plan_at", w["pose"], np.stack([np.linspace(p[0] - 0.5, p[0] + 0.3, 17),
                                                                  np.full(17, p[1])], 1)))
            else:
                resolved.append(("plan_at", w["pose"], w["plan"]))
        else:
            resolved.append(op)
    return w, create, resolved


def run_dwa_reconfigure_case(api, case):
    w, create, ops = dwa_case_world(case)
    return run_dwa_sequence(api, w["grid"], w["origin"], w["pose"], w["plan"], w["vel"], ops, **create)


def tp_points_stride(cfg):
    """The points per sample a TrajectoryPlanner handle sizes for `cfg` (tp_check_config of tp_host.inc)."""
    vmax = max(abs(cfg.max_vel_x), abs(cfg.min_vel_x), abs(cfg.backup_vel))
    vymax = max([0.1] + [abs(cfg.y_vels[i]) for i in range(cfg.n_y_vels)])
    wmax = max(abs(cfg.max_vel_th), abs(cfg.min_vel_th), abs(cfg.min_in_place_vel_th))
    return int(max(max(np.hypot(vmax, vymax) * cfg.sim_time, cfg.sim_time) / cfg.sim_granularity,
                   wmax / cfg.angular_sim_granularity) + 2.0)


def tp_open_world():
    """An empty 6 m x 6 m map, the robot at (1, 3) heading along the plan (+x) at 0.5 m/s."""
    plan = np.stack([np.arange(1.0, 5.9, 0.05), np.full(98, 3.0)], 1)
    return dict(grid=np.zeros((120, 120), np.uint8), origin=(0.0, 0.0), pose=(1.0, 3.0, 0.0), plan=plan,
                vel=(0.5, 0.0, 0.0))


def tp_reconfigure_cases():
    """name -> (world, create overrides, ops, lengthening) of the TrajectoryPlanner reconfigure sequences; a
    lengthening case returns trajectories longer than the handle's creation configuration allows."""
    f = [("find",), ("follow", 0.02)]
    turn = dict(pose=(1.0, 3.0, 1.2), vel=(0.3, 0.0, -0.8))  # heading away from the plan: the winner turns
    cases = {
        "longer_sim_time": (dict(), dict(), f + [("reconfigure", dict(sim_time=3.0))] + f * 2, True),
        "finer_angular_granularity": (turn, dict(dwa=0), f + [("reconfigure", dict(angular_sim_granularity=0.005))] + f * 2,
                                      True),
        "finer_granularity": (dict(), dict(), f + [("reconfigure", dict(sim_granularity=0.01))] + f * 2, True),
        "faster_max_vel_x": (dict(vel=(1.4, 0.0, 0.0)), dict(), f + [("reconfigure", dict(max_vel_x=1.5))] + f * 2, True),
        "faster_max_vel_th": (turn, dict(dwa=0), f + [("reconfigure", dict(max_vel_th=4.0, min_vel_th=-4.0,
                                                                          acc_lim_theta=8.0))] + f * 2, True),
        "shorter": (dict(), dict(sim_time=2.0, sim_granularity=0.01), f + [
            ("reconfigure", dict(sim_time=0.5, sim_granularity=0.05, angular_sim_granularity=0.1))] + f * 2, False),
        # 30 x 40 forward samples: past the 256 samples the buffers start with, regrown together with the stride
        "sample_capacity": (dict(), dict(), f + [("reconfigure", dict(vx_samples=30, vtheta_samples=40, sim_time=2.5))] +
                            f + [("reconfigure", dict(vx_samples=3, vtheta_samples=20, sim_time=1.0))] + f + [
                                ("reconfigure", dict(vx_samples=30, vtheta_samples=40, sim_time=2.5))] + f, True),
        "zero_samples": (dict(), dict(), f + [("reconfigure", dict(vx_samples=0, vtheta_samples=0))] + f + [
            ("reconfigure", dict(vx_samples=3, vtheta_samples=20))] + f, False),
        "modes": (dict(seed=21), dict(), f + [("reconfigure", dict(heading_scoring=1, heading_scoring_timestep=0.45))] + f + [
            ("plan", None)] + f + [("reconfigure", dict(heading_scoring=0, dwa=0))] + f + [
            ("reconfigure", dict(holonomic_robot=0, dwa=1, y_vels=[-0.2, 0.2]))] + f + [
            ("reconfigure", dict(holonomic_robot=1, heading_scoring=1, heading_scoring_timestep=0.1))] + f, False),
        "footprints": (dict(seed=21), dict(), f + [("footprint", square_footprint(0.4))] + f + [
            ("footprint", square_footprint(0.15))] + f + [
            ("footprint", [(0.3 * np.cos(a), 0.3 * np.sin(a)) for a in np.linspace(0, 2 * np.pi, 16, endpoint=False)])] +
            f + [("footprint", PENTAGON)] + f, False),
    }
    return cases


def run_tp_reconfigure_case(api, case):
    world, create, ops, _ = tp_reconfigure_cases()[case]
    if "seed" in world:  # a corridor of dwa_scenario; ("plan", None) halves its plan
        w = reconfigure_world(seed=world["seed"])
        ops = [("plan", w["plan"][:len(w["plan"]) // 2]) if op == ("plan", None) else op for op in ops]
    else:
        w = dict(tp_open_world(), **world)
    return run_tp_sequence(api, w["grid"], w["origin"], w["pose"], w["plan"], w["vel"], ops, **create)
