"""Footprint clearing (ObstacleLayer::updateCosts -> setConvexPolygonCost) beyond the square footprint, against the CPU
checker, bit for bit: window, origin, every obstacle or voxel layer grid, voxel columns and master grid.

The device rasteriser runs in four places: the tail of k_obstacle_update (outline + bounding box <= 2048 cells, mode
1), the stand-alone k_polygon_clear (<= 12288 cells, mode 2), the last CTA of k_voxel_commit, and step 3 of the fleet
kernels.  Its fill is per column for closed outlines spanning two columns or more; an outline whose vertices all fall
in one column replays the reference's column walk.  Every case asserts the path it was written for (polygon_path
restates footprint_polygon's choice) and that k_polygon_clear ran exactly in the mode-2 cycles (launch counts against
a twin handle whose footprint is empty).

Clearing is made visible twice in every stack: a "bare" layer that never observes anything on a track_unknown map
(its FREE cells are exactly the cells cleared), and a "marked" layer with a marking point on every cell of the
footprint's bounding box and 2400 clearing rays (300 CTAs of k_obstacle_update), whose marks inside the footprint only
the fill after the last mark turns FREE.

Footprints the rasteriser cannot take (more than 32 vertices, more than 12288 cells at the pose, a map wider or taller
than 65535 cells) are refused with NAVGPU_ERR_UNSUPPORTED before the cycle changes anything."""
import numpy as np
import pytest

import scenarios as sc
from navigation_b200 import synth
from navigation_b200.api import NavGpuError
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu

POLY_SMALL, POLY_MAX = 2048, 12288  # kPolySmallCells, kPolyMaxCells


def polygon_path(fp, pose, res, sx, sy, ox, oy):
    """footprint_polygon's choice for a footprint at a pose on a layer grid at (ox, oy): 'refused', 'none' (fewer than
    three vertices, or one off the map), 'mode1' or 'mode2', with ' W1' / ' H1' when every vertex lies in one column /
    row; and the cells it counts (outline + bounding box)."""
    w = sc.transform_footprint(fp, pose)
    if len(w) > 32:
        return "refused", 0
    vx, vy = [], []
    for x, y in w:  # worldToMap
        if x < ox or y < oy:
            return "none", 0
        mx, my = int((x - ox) / res), int((y - oy) / res)
        if not (mx < sx and my < sy):
            return "none", 0
        vx.append(mx)
        vy.append(my)
    n = len(vx)
    if n < 3:
        return "none", 0
    outline = sum(max(abs(vx[(k + 1) % n] - vx[k]), abs(vy[(k + 1) % n] - vy[k])) + 1 for k in range(n))
    W, H = max(vx) - min(vx) + 1, max(vy) - min(vy) + 1
    cells = outline + W * H
    if cells > POLY_MAX or sx > 65535 or sy > 65535:
        return "refused", cells
    label = "mode1" if cells <= POLY_SMALL else "mode2"
    return label + (" W1" if W == 1 else "") + (" H1" if H == 1 else ""), cells


# the paths each catalogue entry was written for (on the fixed map)
EXPECT = {
    "rect_8x0.2": {"mode1", "mode2"}, "rect_8x0.2_ccw": {"mode1", "mode2"}, "rect_2x0.5_fine": {"mode2"},
    "square_cw": {"mode1"}, "square_ccw": {"mode1"}, "triangle_ccw": {"mode1"}, "triangle_cw": {"mode1"},
    "ngon16": {"mode1"}, "ngon32": {"mode1"}, "ngon32_large": {"mode2"}, "l_shape": {"mode1"}, "u_shape": {"mode1"},
    "star8": {"mode1"}, "bowtie": {"mode1"}, "repeated": {"mode1"}, "collinear": {"mode1"},
    "one_cell": {"mode1 W1 H1"}, "sliver": {"mode1 W1", "mode1 H1"}, "sliver_tall": {"mode2 W1"},
    "sliver_wide": {"mode2 H1"}, "no_vertex": {"none"}, "one_vertex": {"none"}, "two_vertices": {"none"},
}


def records_equal(a, b, what):
    assert a.keys() == b.keys(), what
    assert a["window"] == b["window"], f"{what}: window {a['window']} != checker's {b['window']}"
    assert a["origin"] == b["origin"], f"{what}: origin {a['origin']} != checker's {b['origin']}"
    for k in sorted(a):
        if k in ("window", "origin", "master"):
            continue
        assert np.array_equal(a[k], b[k]), f"{what}: {k} differs on {int((a[k] != b[k]).sum())} cells"
    assert np.array_equal(a["master"], b["master"]), f"{what}: {int((a['master'] != b['master']).sum())} master cells differ"


def record(cm, ids, window, voxel):
    rec = dict(window=window, origin=cm.origin(), master=cm.get())
    for k in ("bare", "marked"):
        if k in ids:
            rec[k] = cm.get_layer(ids[k])
            if voxel:
                rec[k + "_voxels"] = cm.get_voxels(ids[k])
    return rec


# ---- 1: the catalogue on every host ------------------------------------------------------------------------------------
@pytest.mark.parametrize("host", sc.FOOTPRINT_HOSTS)
@pytest.mark.parametrize("case", list(sc.FOOTPRINT_CASES))
def test_catalogue_matches_checker(cuda, port, case, host):
    fp, res, (sx, sy), yaws = sc.FOOTPRINT_CASES[case]
    cm, ids = sc.footprint_stack(cuda, case, host)
    twin, twin_ids = sc.footprint_stack(cuda, case, host)  # the same stack and calls with an empty footprint
    twin.set_footprint([])
    chk, chk_ids = sc.footprint_stack(port, case, host)
    clearing = [k for k in ("bare", "marked") if k in ids]
    paths, prev_free = [], None
    for cycle in range(len(yaws)):
        what = f"{case} on {host}, cycle {cycle} (yaw {yaws[cycle]:.4f})"
        n0 = cuda.launch_count()
        pose, w = sc.footprint_cycle(cm, ids, case, host, cycle)
        n1 = cuda.launch_count()
        sc.footprint_cycle(twin, twin_ids, case, host, cycle)
        n2 = cuda.launch_count()
        _, cw = sc.footprint_cycle(chk, chk_ids, case, host, cycle)
        got, want = record(cm, ids, w, host == "voxel"), record(chk, chk_ids, cw, host == "voxel")
        path, cells = polygon_path(fp, pose, res, sx, sy, *want["origin"])
        paths.append(path)
        what += f" {path} ({cells} cells)"
        assert path != "refused", what
        assert (n1 - n0) - (n2 - n1) == (len(clearing) if path.startswith("mode2") else 0), \
            f"{what}: {n1 - n0} launches, {n2 - n1} without the footprint"
        records_equal(got, want, what)
        # clearing is visible: the bare layer is FREE exactly where a polygon was cleared, and there only; on a fixed
        # map the marked layer is FREE on every cell this cycle freed in the bare layer (its marks there were cleared
        # after the last mark landed), with marks around the footprint still LETHAL
        if "bare" in ids:
            free = got["bare"] == 0
            assert np.isin(got["bare"], [0, 255]).all(), what
            assert free.any() == any(p != "none" for p in paths), what
            if host != "rolling":
                new = free & ~prev_free if cycle else free
                assert (got["marked"][new] == 0).all(), f"{what}: marks left under the footprint"
                prev_free = free
        assert (got["marked"] == 254).any(), what
    if host == "obstacle":
        assert EXPECT[case] <= set(paths), f"{case}: paths {paths}, written for {sorted(EXPECT[case])}"


# ---- 2: vertices on and just off the map edge --------------------------------------------------------------------------
EDGE_SX, EDGE_SY, EDGE_RES, EDGE_HALF = 60, 50, 0.05, 0.5
EDGE_CASES = {
    # name: robot pose (the footprint is the square of half-size 0.5 m; the named vertex is the one placed)
    "vertex_at_origin": (0.5, 0.5),  # vertex (-0.5, -0.5) lands exactly on the map origin
    "vertex_on_last_cell": ((EDGE_SX - 0.5) * EDGE_RES - 0.5, (EDGE_SY - 0.5) * EDGE_RES - 0.5),
    "off_left": (0.5 - 1e-9, 1.2),
    "off_bottom": (1.2, 0.5 - 1e-9),
    "off_right": (EDGE_SX * EDGE_RES - 0.5 + 1e-9, 1.2),
    "off_top": (1.2, EDGE_SY * EDGE_RES - 0.5 + 1e-9),
}


@pytest.mark.parametrize("voxel", [False, True], ids=["obstacle", "voxel"])
@pytest.mark.parametrize("where", list(EDGE_CASES))
def test_vertices_on_and_off_the_map_edge(cuda, port, where, voxel):
    """A vertex on the map's first or last cell is cleared with the rest; one just off any side clears nothing, but
    the footprint's bounds still make the window."""
    fp = sc.square_footprint(EDGE_HALF)
    pose = (*EDGE_CASES[where], 0.0)
    outs = []
    for api in (cuda, port):
        cm = api.costmap(EDGE_SX, EDGE_SY, EDGE_RES, 0.0, 0.0, track_unknown=True)
        ids = dict(bare=cm.add_voxel_layer(1, True, 2.0) if voxel else cm.add_obstacle_layer(1, True, 2.0))
        cm.set_footprint(fp)
        outs.append(record(cm, ids, cm.update_map(*pose), voxel))
    got, want = outs
    path, _ = polygon_path(fp, pose, EDGE_RES, EDGE_SX, EDGE_SY, 0.0, 0.0)
    assert path == ("none" if where.startswith("off_") else "mode1"), f"{where}: {path}"
    records_equal(got, want, where)
    x0, xn, y0, yn = got["window"]
    assert xn > x0 and yn > y0, f"{where}: the footprint did not touch the window {got['window']}"
    free = got["bare"] == 0
    assert free.any() == (path != "none"), where
    if where == "vertex_at_origin":
        assert free[0, 0]
    elif where == "vertex_on_last_cell":
        assert free[-1, -1]


# ---- 3: refusals leave the handle as it was ----------------------------------------------------------------------------
RECT = sc.rectangle(8.0, 0.2)
REFUSALS = ["33_vertices", "rect_pi4_static_pending", "rect_pi4_rolling", "voxel_rolling", "second_layer_clears",
            "map_65536_wide"]


def refusal_handle(api, case):
    """(costmap, ids, accepted footprint, refused footprint, pose of the first cycle, refused pose, pose after)."""
    if case == "map_65536_wide":
        sx, sy, res, rolling = 65536, 4, 0.05, False
    elif case == "33_vertices":
        sx, sy, res, rolling = 90, 80, 0.05, False
    else:
        sx, sy, res, rolling = 200, 200, 0.05, case.endswith("rolling")
    cm = api.costmap(sx, sy, res, 0.0, 0.0, rolling=rolling, track_unknown=True)
    ids = {}
    if not rolling:
        ids["static"] = cm.add_grid_layer(po.TRUE_OVERWRITE)
    if case == "voxel_rolling":
        ids["marked"] = cm.add_voxel_layer(1, True, 2.0)
    elif case == "second_layer_clears":
        ids["first"] = cm.add_obstacle_layer(1, False, 2.0)
        ids["marked"] = cm.add_obstacle_layer(0, True, 2.0)
    else:
        ids["marked"] = cm.add_obstacle_layer(1, True, 2.0)
    if case != "map_65536_wide":
        ids["inflation"] = cm.add_inflation_layer(0.3, 3.0)
        sc.select_inflation(cm, ids["inflation"], "exact")
    c = (sx // 2 + 0.5) * res, (sy // 2 + 0.5) * res
    if case == "33_vertices":
        good, bad = sc.regular_polygon(32, 0.6), sc.regular_polygon(33, 0.6)
        poses = [(*c, 0.0), (*c, 0.0), (*c, 0.0)]
    elif case == "map_65536_wide":  # a footprint half off the map's bottom is accepted (nothing to clear)
        good = bad = sc.square_footprint(0.06)
        poses = [(1000.0, 0.05, 0.0), (1000.0, 0.1, 0.0), (1000.3, 0.05, 0.0)]
    else:  # the 8 m x 0.2 m rectangle: 13925 cells at pi/4
        good = bad = RECT
        step = (0.37, 0.21) if rolling else (0.0, 0.0)
        poses = [(*c, 0.0), (c[0] + step[0], c[1] + step[1], np.pi / 4), (c[0] + 2 * step[0], c[1] + 2 * step[1], 0.0)]
    cm.set_footprint(good)
    return cm, ids, (sx, sy, res), good, bad, poses


def refusal_observations(cm, ids, pose, res, sx, sy, seed):
    for k in ("first", "marked"):
        if k in ids:
            ox, oy = cm.origin()
            obs = sc.footprint_marks(sc.square_footprint(0.8), pose, res, sx, sy, ox, oy, n_rays=400)
            rng = np.random.default_rng(seed + len(k))
            obs[1]["points"] = obs[1]["points"][rng.random(len(obs[1]["points"])) < 0.3]
            cm.set_observations(ids[k], obs)


def refusal_state(cm, ids, window, voxel):
    st = dict(master=cm.get(), origin=cm.origin(), window=window)
    for k in ("first", "marked", "static"):
        if k in ids:
            st[k] = cm.get_layer(ids[k])
    if voxel:
        st["voxels"] = cm.get_voxels(ids["marked"])
    return st


@pytest.mark.parametrize("case", REFUSALS)
def test_refused_footprint_leaves_the_handle_as_it_was(cuda, port, case):
    """A cycle refused for its footprint raises NAVGPU_ERR_UNSUPPORTED before it rolls a grid, clears an update flag or
    launches an obstacle kernel: master grid, layer grids, voxel columns, origin, window and host mirror unchanged.
    The next accepted cycle equals a checker that received the same calls but skipped the refused cycle -- a static
    layer update that was pending, observations that were set, a map that moves."""
    voxel = case == "voxel_rolling"
    (cm, ids, (sx, sy, res), good, bad, poses), (twin, t_ids, *_) = refusal_handle(cuda, case), refusal_handle(port, case)
    static = np.zeros((sy, sx), np.uint8)
    static[::3, ::4] = 254
    for h, i in ((cm, ids), (twin, t_ids)):
        if "static" in i:
            h.set_grid_layer(i["static"], static)
        refusal_observations(h, i, poses[0], res, sx, sy, 1)
    first = [h.update_map(*poses[0]) for h in (cm, twin)]
    assert first[0] == first[1] and np.array_equal(cm.get(), twin.get())
    # a windowed cycle, so that the one after the refusal is windowed too (the inflation layer adds the last bounds)
    for h, i in ((cm, ids), (twin, t_ids)):
        refusal_observations(h, i, poses[0], res, sx, sy, 3)
    second = [h.update_map(*poses[0]) for h in (cm, twin)]
    assert second[0] == second[1] and np.array_equal(cm.get(), twin.get())
    mirror = np.zeros((sy, sx), np.uint8)
    cm.get_changed(mirror)
    # the refused cycle's calls, on both: a pending static-layer update in a small box, fresh observations
    y0 = max(0, sy // 2 - 20)
    pending = static.copy()
    pending[y0:y0 + 3, 1:7] = 254
    for h, i in ((cm, ids), (twin, t_ids)):
        if "static" in i:
            h.set_grid_layer(i["static"], pending)
            h.touch_grid_layer(i["static"], 0, y0, 8, 3)
        refusal_observations(h, i, poses[1], res, sx, sy, 2)
        if bad is not good:
            h.set_footprint(bad)
    path, cells = polygon_path(bad, poses[1], res, sx, sy, *cm.origin())
    assert path == "refused" or (case.endswith("rolling") and cells > POLY_MAX), f"{case}: {path} {cells}"
    before = refusal_state(cm, ids, cm.last_window(), voxel)
    with pytest.raises(NavGpuError, match="navgpu error 3: .*(more than 32 vertices|too many cells)"):
        cm.update_map(*poses[1])
    after = refusal_state(cm, ids, cm.last_window(), voxel)
    for k in before:
        assert np.array_equal(np.asarray(before[k]), np.asarray(after[k])), f"{case}: the refused cycle changed {k}"
    cm.get_changed(mirror)
    assert np.array_equal(mirror, before["master"]), f"{case}: the host mirror moved"
    # back to an accepted footprint / pose
    for h in (cm, twin):
        if bad is not good:
            h.set_footprint(good)
    out = [refusal_state(h, i, h.update_map(*poses[2]), voxel) for h, i in ((cm, ids), (twin, t_ids))]
    records_equal(out[0], out[1], f"{case}: the cycle after the refusal")
    if case in ("rect_pi4_static_pending", "map_65536_wide"):
        assert out[0]["window"] != (0, sx, 0, sy), f"{case}: a whole-map cycle hides a lost window"
    if "static" in ids:
        assert (out[0]["master"][y0:y0 + 3, 1:7] == 254).all(), f"{case}: the pending static update was lost"
    cm.get_changed(mirror)
    assert np.array_equal(mirror, cm.get()), f"{case}: the host mirror differs from the master grid"


# ---- 4: fleets -----------------------------------------------------------------------------------------------------------
RES = 0.05
FLEET_CFG = dict(vx_samples=4, vy_samples=1, vth_samples=5, max_vel_y=0.0, min_vel_y=0.0)
FLEET_CASES = ["square_cw", "square_ccw", "triangle_ccw", "triangle_cw", "ngon16", "l_shape", "u_shape", "star8",
               "bowtie", "repeated", "collinear", "one_cell", "sliver"]
INSIDE_BOUND, OUTSIDE_BOUND = sc.square_footprint(0.70), sc.square_footprint(0.71)


def fleet_bound(fp, res=RES):
    """fleet_costmap_create's bound on the cells the footprint polygon can cover at any pose."""
    n = len(fp)
    rc = max(np.hypot(*p) for p in fp)
    outline = sum(np.ceil(np.hypot(fp[(i + 1) % n][0] - fp[i][0], fp[(i + 1) % n][1] - fp[i][1]) / res) + 2
                  for i in range(n))
    span = np.ceil(2 * rc / res) + 3
    return span * span + outline


def fleet_checker(port, fp, voxel):
    cm = port.costmap(120, 120, RES, 0.0, 0.0, rolling=True, track_unknown=True)
    o = cm.add_voxel_layer(1, True, 2.0) if voxel else cm.add_obstacle_layer(1, True, 2.0)
    il = cm.add_inflation_layer(0.55, 10.0)
    sc.select_inflation(cm, il, "exact")
    cm.set_footprint(fp)
    return cm, o


def run_fleet(cuda, port, fp, voxel, yaws_of_cycle, n=6):
    """n robots of fleet_sensing_robot, turned to the yaws yaws_of_cycle(cycle, robot), with one PointCloud source
    each; every robot's layer, columns, master grid, origin and window against its own checker costmap."""
    robots = [synth.fleet_sensing_robot(500 + i) for i in range(n)]
    fleet = cuda.fleet_sensing(n, 120, 120, RES, fp, track_unknown=True, voxel={} if voxel else None, **FLEET_CFG)
    refs = [fleet_checker(port, fp, voxel) for _ in range(n)]
    vels = np.array([r["vel"] for r in robots])
    cycles = len(yaws_of_cycle) if isinstance(yaws_of_cycle, list) else 3
    cleared = 0
    for cycle in range(cycles):
        for i, r in enumerate(robots):
            r["poses"][cycle][2] = yaws_of_cycle[cycle] if isinstance(yaws_of_cycle, list) else yaws_of_cycle(cycle, i)
        poses = np.array([r["poses"][cycle] for r in robots])
        scans = [[synth.fleet_scan(r, cycle, cloud=True)] for r in robots]
        fleet.set_scans(scans)
        fleet.set_plans(poses, [r["plan"] for r in robots])
        fleet.step(poses, vels)
        for i, (cm, o) in enumerate(refs):
            obs = []
            for s_ in scans[i]:
                org, pts = port.project_scan(s_)
                obs.append(dict(origin=org, points=pts, obstacle_range=s_["obstacle_range"],
                                raytrace_range=s_["raytrace_range"], marking=s_["marking"], clearing=s_["clearing"]))
            cm.set_observations(o, obs)
            win = cm.update_map(*poses[i])
            where = f"cycle {cycle} robot {i} yaw {poses[i][2]:.4f}"
            assert fleet.geometry(i) == (cm.origin(), win), where
            layer = fleet.layer(i)
            assert np.array_equal(layer, cm.get_layer(o)), f"{where}: layer differs on {(layer != cm.get_layer(o)).sum()}"
            if voxel:
                assert np.array_equal(fleet.voxels(i), cm.get_voxels(o)), f"{where}: columns differ"
            assert np.array_equal(fleet.costmap(i), cm.get()), f"{where}: master grid differs"
            ox, oy = cm.origin()
            cleared += polygon_path(fp, tuple(poses[i]), RES, 120, 120, ox, oy)[0] != "none"
    assert cleared > 0


@pytest.mark.parametrize("voxel", [False, True], ids=["sensing", "voxel"])
@pytest.mark.parametrize("case", FLEET_CASES)
def test_fleet_catalogue_matches_checker(cuda, port, case, voxel):
    fp = sc.FOOTPRINT_CASES[case][0]
    assert len(fp) <= 16 and fleet_bound(fp) <= POLY_SMALL
    run_fleet(cuda, port, fp, voxel, lambda cycle, i: 0.37 * i + 1.1 * cycle)


@pytest.mark.parametrize("voxel", [False, True], ids=["sensing", "voxel"])
def test_fleet_footprint_at_the_creation_bound(cuda, port, voxel):
    """The largest square the creation bound admits, turned through 0 ... pi/2 in pi/32 steps: the per-robot
    rasteriser's scratch (2048 entries, no capacity check on the outline) holds it at every pose; one 0.01 m larger
    is refused at creation."""
    assert fleet_bound(INSIDE_BOUND) <= POLY_SMALL < fleet_bound(OUTSIDE_BOUND)
    run_fleet(cuda, port, INSIDE_BOUND, voxel, [k * np.pi / 32 for k in range(17)], n=4)
    with pytest.raises(NavGpuError, match="navgpu error 3.*footprint polygon can cover"):
        cuda.fleet_sensing(2, 120, 120, RES, OUTSIDE_BOUND, voxel={} if voxel else None, **FLEET_CFG)
