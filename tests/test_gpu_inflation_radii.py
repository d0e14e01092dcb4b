"""Inflation beyond the fast path, against the CPU checker: cell radii above 31 (the generic sweep k_update_costs, up to
the largest accepted radius and across the 48 KB shared-memory opt-in), propagation mode at large radii, refused radii,
one handle moved between every sweep by set_inflation_params / set_inflation_mode, stacks in which inflation is not
the last layer, and the host mirror behind the generic and propagation sweeps.

Radii are chosen as (R - 0.5) * resolution, so that Costmap2D::cellDistance gives exactly R cells, and every case
asserts its cell radius (and reports its effective reach, the largest distance whose cost is non-zero) before it
compares anything.  The checker's exact variant is brute force (about pi R^2 work per seed), so worlds with large radii
hold few LETHAL cells (seed_budget)."""
import numpy as np
import pytest

import scenarios as sc
from navigation_b200.api import NavGpuError
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu

RES = 0.05


def radius_of(R):
    """An inflation radius whose cell distance is exactly R."""
    return (R - 0.5) * RES


def effective_reach(costs, R):
    """The largest cell distance within R whose cached cost is non-zero (what launch_sweep picks k_inflate<N> by)."""
    n = R + 2
    i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    d2 = i * i + j * j
    live = (d2 <= R * R) & (costs > 0)
    return int(np.sqrt(d2[live].max() + 0.5)) if R > 0 and live.any() else 0


def cell_radius_and_reach(cm, layer, R):
    """Asserts the layer's cell radius; returns its effective reach."""
    got, costs, _ = cm.inflation_tables(layer)
    assert got == R, f"cell radius {got}, meant {R}"
    return effective_reach(costs, R)


def last_rounds(cm, layer):
    """Rounds of the last propagation sweep (the CUDA handle has one counter, the checker one per layer)."""
    return cm.inflation_last_rounds() if hasattr(cm, "get_changed") else cm.inflation_last_rounds(layer)


def seed_budget(R):
    """LETHAL cells a world may hold at cell radius R, so that the checker's exact variant stays fast."""
    return int(min(1500, max(120, 3e7 / (np.pi * R * R))))


def sparse_world(sx, sy, n_lethal, seed):
    """Free, mid-cost and NO_INFORMATION cells with about n_lethal LETHAL ones: a wall, a diagonal line, isolated seeds
    each with a NO_INFORMATION neighbour, and LETHAL / NO_INFORMATION cells alternating down the last column."""
    rng = np.random.default_rng(seed)
    g = rng.choice(np.array([0, 0, 0, 0, 0, 0, 40, 128, 200, 252, 253], np.uint8), size=(sy, sx))
    g[rng.random((sy, sx)) < 0.03] = 255
    ys = np.arange(sy)
    g[ys % 9 == 0, sx - 1] = 254
    g[ys % 9 == 1, sx - 1] = 255
    budget = n_lethal - int((ys % 9 == 0).sum())
    wall = max(0, min(sx - 4, budget // 4))
    g[sy // 3, 2:2 + wall] = 254
    diag = max(0, min(sx - sx // 5, sy - 2, budget // 4))
    k = np.arange(diag)
    g[sy - 2 - k, sx // 5 + k] = 254
    for _ in range(max(1, (budget - wall - diag) // 2)):
        x, y = int(rng.integers(0, sx - 1)), int(rng.integers(0, sy - 1))
        g[y, x] = 254
        if rng.random() < 0.5:
            g[y, x + 1] = 255
        else:
            g[y + 1, x] = 255
    return g


def extra_world(sx, sy, seed):
    """A second grid layer: NO_INFORMATION but for a patch of values and a few LETHAL cells, so that what it merges
    depends on the policy."""
    rng = np.random.default_rng(seed)
    g = np.full((sy, sx), 255, np.uint8)
    patch = rng.random((sy, sx)) < 0.3
    g[patch] = rng.choice(np.array([0, 0, 1, 60, 130, 252, 253], np.uint8), size=int(patch.sum()))
    g.flat[rng.choice(sx * sy, 6, replace=False)] = 254
    return g


def marks(sx, sy, seed, n=6):
    """Marked points in the middle of the map, seen from its centre: the window they make has its edges inside tiles."""
    rng = np.random.default_rng(seed)
    pts = np.stack([rng.uniform(0.35 * sx, 0.65 * sx, n) * RES, rng.uniform(0.35 * sy, 0.65 * sy, n) * RES,
                    np.full(n, 0.5)], 1).astype(np.float32)
    return dict(origin=(0.5 * sx * RES + 0.01, 0.5 * sy * RES + 0.01, 0.5), points=pts, obstacle_range=100.0,
                raytrace_range=100.0, marking=True, clearing=False)


def clears(mark):
    """Clearing rays from the same origin through (and past) the marked points of `mark`."""
    o = np.array(mark["origin"][:2], np.float32)
    pts = mark["points"].copy()
    pts[:, :2] = o + 1.3 * (pts[:, :2] - o)
    return dict(mark, points=pts, marking=False, clearing=True)


def moving_scan(sx, sy, cycle, seed, n=30, spread=2.0):
    """One observation from a sensor that moves along x with the cycle: marks up to `spread` m around it, clearing rays
    to them; returns (observations, robot pose)."""
    rng = np.random.default_rng(seed + 101 * cycle)
    ox, oy = (0.25 + 0.05 * cycle) * sx * RES, 0.5 * sy * RES
    ang, rad = rng.uniform(0, 2 * np.pi, n), rng.uniform(0.2 * spread, spread, n)
    pts = np.stack([ox + rad * np.cos(ang), oy + rad * np.sin(ang), np.full(n, 0.5)], 1).astype(np.float32)
    return [dict(origin=(ox, oy, 0.5), points=pts, obstacle_range=spread + 0.5, raytrace_range=spread + 1.0,
                 marking=True, clearing=True)], (ox, oy, 0.1 * cycle)


def assert_cycles_equal(a, b, what):
    """a, b: per cycle (window, master grid, [layer grids]) of the CUDA handle and the checker."""
    for cycle, ((wa, ga, la), (wb, gb, lb)) in enumerate(zip(a, b)):
        assert wa == wb, f"{what} cycle {cycle}: window {wa} != checker's {wb}"
        for k, (x, y) in enumerate(zip(la, lb)):
            assert np.array_equal(x, y), f"{what} cycle {cycle}: layer {k} differs on {int((x != y).sum())} cells"
        assert np.array_equal(ga, gb), f"{what} cycle {cycle}: {int((ga != gb).sum())} master cells differ"


# ---- 1a: the generic sweep against the exact variant ------------------------------------------------------------------
# 32 / 33: the first generic radii; 63 / 64 / 65: the horizontal search crosses its second and third 32-bit word;
# 92 / 93: the last radius within 48 KB of shared memory and the first beyond; 254: the largest accepted
GENERIC_RADII = [32, 33, 63, 64, 65, 92, 93, 127, 128, 200, 254]
GENERIC_SHAPES = ["below_2R", "129x33", "250x200"]
MERGE_POLICIES = [po.OVERWRITE, po.MAX, po.ADDITION]
SCALINGS = [0.0, 1.0, 3.0]


def generic_shape(R, shape):
    if shape == "below_2R":  # narrower and shorter than 2R
        return min(R + 7, 250), R // 2 + 9
    return {"129x33": (129, 33), "250x200": (250, 200)}[shape]


def run_generic(api, R, sx, sy, policy, track_unknown, scaling, seed):
    cm = api.costmap(sx, sy, RES, track_unknown=track_unknown)
    s = cm.add_grid_layer(po.TRUE_OVERWRITE)
    e = cm.add_grid_layer(policy)
    o = cm.add_obstacle_layer(1, True, 2.0)
    il = cm.add_inflation_layer(radius_of(R), scaling)
    cm.set_footprint(sc.square_footprint())
    sc.select_inflation(cm, il, "exact")
    cm.set_grid_layer(s, sparse_world(sx, sy, min(seed_budget(R), sx * sy // 40), seed))
    cm.set_grid_layer(e, extra_world(sx, sy, seed + 1))
    first = marks(sx, sy, seed + 2)
    obs = [[], [first], [clears(first), marks(sx, sy, seed + 3)], [marks(sx, sy, seed + 4, n=2)]]
    trace = []
    # the whole map; marks (the inflation layer still adds the last cycle's bounds: the whole map again); clearing rays
    # through them and new marks; two more marks
    for cycle in range(4):
        cm.set_observations(o, obs[cycle])
        w = cm.update_map(0.5 * sx * RES, 0.5 * sy * RES, 0.0)
        trace.append((w, cm.get(), [cm.get_layer(k) for k in (s, e, o)]))
    return cm, il, trace


@pytest.mark.parametrize("shape", GENERIC_SHAPES)
@pytest.mark.parametrize("R", GENERIC_RADII)
def test_generic_sweep_matches_exact(cuda, port, R, shape, record_property):
    ri, si = GENERIC_RADII.index(R), GENERIC_SHAPES.index(shape)
    policy = MERGE_POLICIES[(ri + si) % 3]
    track_unknown = (ri + si) % 2 == 1
    scaling = SCALINGS[(ri + 2 * si) % 3]
    sx, sy = generic_shape(R, shape)
    outs = []
    for api in (cuda, port):
        cm, il, trace = run_generic(api, R, sx, sy, policy, track_unknown, scaling, 1000 * R + si)
        if api is cuda:
            reach = cell_radius_and_reach(cm, il, R)
            record_property("R", R)
            record_property("reach", reach)
        outs.append(trace)
    what = f"R={R} reach={reach} {sx}x{sy} policy={policy} track_unknown={track_unknown} scaling={scaling}"
    assert outs[0][0][0] == (0, sx, 0, sy), what
    if shape == "250x200" and R <= 65:  # the last two cycles really are windowed
        assert all(w[1] - w[0] < sx and w[3] - w[2] < sy for w, _, _ in outs[0][2:]), what
    assert_cycles_equal(outs[0], outs[1], what)
    master = outs[0][0][1]
    assert ((master > 0) & (master < 253)).any(), what
    if track_unknown:  # (without it the obstacle layer's FREE cells replace every NO_INFORMATION of the window)
        assert (master == 255).any(), what


# ---- 1b: propagation mode against the level-synchronous variant --------------------------------------------------------
PROPAGATE_RADII = [21, 31, 32, 64, 100, 127]


def propagation_world(sx, sy, seed):
    """Isolated seeds and diagonal lines of several slopes: propagated and nearest-seed costs differ behind them."""
    rng = np.random.default_rng(seed)
    g = np.zeros((sy, sx), np.uint8)
    for x0, y0, dx, dy, n in ((10, 10, 1, 1, 120), (sx - 12, 15, -1, 2, 70), (20, sy - 12, 3, -1, 60)):
        k = np.arange(n)
        x, y = x0 + dx * k, y0 + dy * k
        ok = (x >= 0) & (x < sx) & (y >= 0) & (y < sy)
        g[y[ok], x[ok]] = 254
    for _ in range(60):
        g[int(rng.integers(0, sy)), int(rng.integers(0, sx))] = 254
    g[rng.random((sy, sx)) < 0.01] = 255
    return g


def run_propagation(api, R, scaling, seed, which="propagate", sx=210, sy=170):
    cm = api.costmap(sx, sy, RES)
    s = cm.add_grid_layer(po.TRUE_OVERWRITE)
    o = cm.add_obstacle_layer(1, True, 2.0)
    il = cm.add_inflation_layer(radius_of(R), scaling)
    cm.set_footprint(sc.square_footprint())
    sc.select_inflation(cm, il, which)
    cm.set_grid_layer(s, propagation_world(sx, sy, seed))
    first = marks(sx, sy, seed + 1)
    obs = [[], [first], [clears(first), marks(sx, sy, seed + 2)], [marks(sx, sy, seed + 3, n=3)]]
    trace = []
    for cycle in range(4):
        cm.set_observations(o, obs[cycle])
        w = cm.update_map(0.5 * sx * RES, 0.5 * sy * RES, 0.0)
        trace.append((w, cm.get(), [cm.get_layer(o)], last_rounds(cm, il) if which == "propagate" else None))
    return cm, il, trace


@pytest.mark.parametrize("R", PROPAGATE_RADII)
def test_propagation_mode_matches_propagate(cuda, port, R, record_property):
    scaling = 1.0 if R >= 64 else 3.0
    outs = []
    for api in (cuda, port):
        cm, il, trace = run_propagation(api, R, scaling, 77 + R)
        if api is cuda:
            reach = cell_radius_and_reach(cm, il, R)
            record_property("R", R)
            record_property("reach", reach)
        outs.append(trace)
    what = f"propagation R={R} reach={reach} scaling={scaling}"
    assert_cycles_equal([t[:3] for t in outs[0]], [t[:3] for t in outs[1]], what)
    assert [t[3] for t in outs[0]] == [t[3] for t in outs[1]], f"{what}: rounds"
    assert all(t[3] > 0 for t in outs[0]), what
    # a world on which propagation and the nearest seed disagree, in every cycle
    _, _, exact = run_propagation(port, R, scaling, 77 + R, which="exact")
    assert all((t[1] != e[1]).any() for t, e in zip(outs[1], exact)), what


# ---- 1c: refused radii -------------------------------------------------------------------------------------------------
REFUSALS = {
    # name: (mode, refused cell radius, how the handle gets back to an accepted configuration)
    "mode0_R255": (0, 255, ("params", 40)),
    "mode1_R128": (1, 128, ("params", 64)),
    "mode1_R128_then_mode0": (1, 128, ("mode", 0)),  # R = 128 is accepted by the generic sweep
}


def stack_with_obstacles(api, sx, sy, R, scaling, seed, track_unknown=False):
    cm = api.costmap(sx, sy, RES, track_unknown=track_unknown)
    s = cm.add_grid_layer(po.TRUE_OVERWRITE)
    o = cm.add_obstacle_layer(1, True, 2.0)
    il = cm.add_inflation_layer(radius_of(R), scaling)
    cm.set_footprint(sc.square_footprint())
    cm.set_grid_layer(s, sparse_world(sx, sy, 400, seed))
    return cm, s, o, il


def set_mode(cm, il, mode):
    sc.select_inflation(cm, il, ("exact", "propagate")[mode])


@pytest.mark.parametrize("case", list(REFUSALS))
def test_refused_radius_leaves_the_handle_as_it_was(cuda, port, case):
    """A cycle refused for its radius raises NAVGPU_ERR_UNSUPPORTED before any sweep and leaves the handle as if it had
    not been asked for: the master grid unchanged, and after going back to an accepted configuration the next cycle
    equals a checker that received the same calls but skipped the refused cycle (both reinflate the whole map), with
    the host mirror equal to the master grid."""
    mode, bad, (how, to) = REFUSALS[case]
    # a map wider than the window of marks in its middle grown by R = 128: reinflating the whole map must be asked for
    sx, sy, scaling, good = 420, 320, 3.0, 40 if mode == 0 else 64
    robot = (0.5 * sx * RES, 0.5 * sy * RES, 0.0)
    sides = []
    for api in (cuda, port):
        cm, s, o, il = stack_with_obstacles(api, sx, sy, good, scaling, 5)
        set_mode(cm, il, mode)
        cm.set_observations(o, [marks(sx, sy, 6)])
        w = cm.update_map(*robot)
        sides.append((cm, o, il, w))
    (cm, o, il, w), (twin, t_o, t_il, tw) = sides
    assert w == tw == (0, sx, 0, sy) and np.array_equal(cm.get(), twin.get())
    mirror = np.zeros((sy, sx), np.uint8)
    cm.get_changed(mirror)
    before = cm.get()
    for h, layer in ((cm, il), (twin, t_il)):
        h.set_inflation_params(layer, radius_of(bad), scaling)
    cm.set_observations(o, [])
    with pytest.raises(NavGpuError, match=f"navgpu error 3: .*R={bad} > 127" if mode else "navgpu error 3: .* 255 > 254"):
        cm.update_map(*robot)
    assert np.array_equal(cm.get(), before), "the refused cycle wrote the master grid"
    for h, layer in ((cm, il), (twin, t_il)):
        if how == "params":
            h.set_inflation_params(layer, radius_of(to), scaling)
        else:
            set_mode(h, layer, to)
    for h, layer in ((cm, o), (twin, t_o)):
        h.set_observations(layer, [])
    out = [(h.update_map(*robot), h.get(), [h.get_layer(k)]) for h, k in ((cm, o), (twin, t_o))]
    assert out[0][0] == (0, sx, 0, sy), f"{case}: the cycle after the refusal did not reinflate the whole map"
    assert twin.update_map(*robot) != (0, sx, 0, sy)  # (the cycle after that one is windowed)
    assert_cycles_equal([out[0]], [out[1]], case)
    cm.get_changed(mirror)
    assert np.array_equal(mirror, cm.get()), f"{case}: the host mirror differs from the master grid"


# ---- 1d: one live handle through every sweep ---------------------------------------------------------------------------
# ("params", R): set_inflation_params; ("mode", m, R): set_inflation_mode, then set_inflation_params
WALK = [("params", 11), ("params", 45), ("params", 150), ("params", 20), ("params", 31), ("params", 32),
        ("mode", 1, 100), ("mode", 0, 11), ("params", 0), ("params", 11)]


def run_walk(api, sx, sy, seed):
    cm, s, o, il = stack_with_obstacles(api, sx, sy, 11, 3.0, seed)
    set_mode(cm, il, 0)
    trace, radii = [], []
    for cycle, step in enumerate(WALK):
        R = step[-1]
        if step[0] == "mode":
            set_mode(cm, il, step[1])
        scaling = (3.0, 1.0)[cycle % 2]
        cm.set_inflation_params(il, radius_of(R) if R else 0.0, scaling)
        obs, robot = moving_scan(sx, sy, cycle, seed)
        cm.set_observations(o, obs)
        w = cm.update_map(*robot)
        rounds = last_rounds(cm, il) if step[0] == "mode" and step[1] == 1 else None
        trace.append((w, cm.get(), [cm.get_layer(o)], rounds))
        if hasattr(cm, "get_changed"):
            radii.append((R, cell_radius_and_reach(cm, il, R)))
    return trace, radii


def test_one_handle_through_every_sweep(cuda, port, record_property):
    """set_inflation_params / set_inflation_mode before every cycle move one handle between the fast path (k_inflate<12>,
    <20>, <31>), the generic sweep (also past the 48 KB opt-in), propagation mode and radius 0, regrowing its tables
    and buffers on the way; scans move every cycle.  Every cycle equals the checker driven through the same calls."""
    sx, sy = 200, 150
    a, radii = run_walk(cuda, sx, sy, 31)
    b, _ = run_walk(port, sx, sy, 31)
    record_property("radii_and_reaches", radii)
    for cycle, ((x, y), step) in enumerate(zip(zip(a, b), WALK)):
        what = f"cycle {cycle} {step} (R, reach) = {radii[cycle]}"
        assert_cycles_equal([x[:3]], [y[:3]], what)
        assert x[3] == y[3], f"{what}: rounds {x[3]} != {y[3]}"
    # the fast-path steps took each k_inflate instantiation, the others the generic sweep (past 48 KB at R = 150)
    fast = [reach for (R, reach), step in zip(radii, WALK) if 0 < R <= 31 and not (step[0] == "mode" and step[1] == 1)]
    assert min(fast) <= 12 and any(12 < r <= 20 for r in fast) and max(fast) > 20, radii


# ---- 1e: stacks where inflation is not the last layer ------------------------------------------------------------------
STACKS = {
    "inflation_then_obstacle": [("static",), ("inflation", 25), ("obstacle",)],
    "two_inflations": [("static",), ("obstacle",), ("inflation", 11), ("inflation", 45)],
    "inflate_merge_inflate": [("static",), ("inflation", 20), ("extra", po.MAX), ("inflation", 64)],
    "inflation_disabled_once": [("static",), ("obstacle",), ("inflation", 30)],
}


# the inflation layer of "inflation_disabled_once" is off in cycle 2 and on again from cycle 3
STACK_CYCLES = ["first", "window", "window", "window", "whole", "whole", "window", "window"]


def run_stack(api, name, mode, sx, sy, seed):
    """Windowed cycles (a block added to the static layer inside a touched rectangle, moving scans) and whole-map cycles
    (the static layer touched whole, moving scans: the early-release path); a cycle after a whole-map one is whole too
    (the inflation layer adds the last cycle's bounds).  The CUDA handle's host mirror is brought up to date every
    cycle.  Returns per cycle (window, master grid, [obstacle layer grids])."""
    rng = np.random.default_rng(seed)
    cm = api.costmap(sx, sy, RES)
    ids = []
    for layer in STACKS[name]:
        if layer[0] == "static":
            ids.append(cm.add_grid_layer(po.TRUE_OVERWRITE))
        elif layer[0] == "extra":
            ids.append(cm.add_grid_layer(layer[1]))
        elif layer[0] == "obstacle":
            ids.append(cm.add_obstacle_layer(1, True, 2.0))
        else:
            ids.append(cm.add_inflation_layer(radius_of(layer[1]), 3.0))
    cm.set_footprint(sc.square_footprint())
    kinds = [layer[0] for layer in STACKS[name]]
    infl = [i for i, k in zip(ids, kinds) if k == "inflation"]
    obst = [i for i, k in zip(ids, kinds) if k == "obstacle"]
    s = ids[kinds.index("static")]
    for il in infl:
        set_mode(cm, il, mode)
    static = sparse_world(sx, sy, 1200, seed)
    cm.set_grid_layer(s, static)
    if "extra" in kinds:
        cm.set_grid_layer(ids[kinds.index("extra")], extra_world(sx, sy, seed + 1))
    mirror = np.full((sy, sx), 7, np.uint8) if hasattr(cm, "get_changed") else None
    trace = []
    for cycle, kind in enumerate(STACK_CYCLES):
        if name == "inflation_disabled_once" and cycle in (2, 3):
            cm.set_enabled(infl[0], cycle == 3)
        if kind == "window":
            x0, y0 = int(rng.integers(sx // 4, sx // 2)), int(rng.integers(sy // 4, sy // 2))
            static = static.copy()
            static[y0:y0 + 5, x0:x0 + 8] = 254
            cm.set_grid_layer(s, static)
            cm.touch_grid_layer(s, x0 - 3, y0 - 3, 14, 11)
        elif kind == "whole":
            cm.touch_grid_layer(s, 0, 0, sx, sy)
        obs, robot = moving_scan(sx, sy, cycle, seed, spread=0.8)
        for o in obst:
            cm.set_observations(o, obs)
        w = cm.update_map(*robot)
        grid = cm.get()
        trace.append((w, grid, [cm.get_layer(o) for o in obst]))
        if mirror is not None:
            cm.get_changed(mirror)
            assert np.array_equal(mirror, grid), f"{name} mode {mode} cycle {cycle}: the host mirror differs"
    if hasattr(cm, "get_changed"):
        for il, layer in zip(infl, [layer for layer in STACKS[name] if layer[0] == "inflation"]):
            assert cm.inflation_tables(il)[0] == layer[1]
    return trace


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("name", list(STACKS))
def test_stacks_with_inflation_not_last(cuda, port, name, mode):
    sx, sy = 320, 220
    a = run_stack(cuda, name, mode, sx, sy, 9)
    b = run_stack(port, name, mode, sx, sy, 9)
    assert a[0][0] == a[4][0] == a[5][0] == (0, sx, 0, sy)
    assert any(a[c][0] != (0, sx, 0, sy) for c in (3, 7)), "no windowed cycle"
    assert_cycles_equal(a, b, f"{name} mode {mode}")


# ---- 1f: the host mirror behind the generic and propagation sweeps -----------------------------------------------------
@pytest.mark.parametrize("registered", [False, True], ids=["pageable", "page-locked"])
@pytest.mark.parametrize("mode,R", [(0, 45), (1, 64)])
def test_host_mirror_behind_generic_and_propagation_sweeps(cuda, port, mode, R, registered):
    """test_host_mirror_tracks_the_master_grid's recipe at a radius the fast sweep does not take: windowed cycles,
    whole-map cycles (refinable from the second one on: the grid is clean and no layer content changed), a windowed
    cycle that changes the static layer, a last whole-map cycle.  After every cycle the mirror equals the device grid,
    every changed cell lies in a reported rectangle, and the grid equals the checker."""
    sx, sy, seed = 300, 200, 21
    static = sparse_world(sx, sy, 1500, seed)
    hs = []
    for api in (cuda, port):
        cm = api.costmap(sx, sy, RES)
        s = cm.add_grid_layer(po.TRUE_OVERWRITE)
        o = cm.add_obstacle_layer(1, True, 2.0)
        il = cm.add_inflation_layer(radius_of(R), 3.0)
        cm.set_footprint(sc.square_footprint())
        set_mode(cm, il, mode)
        cm.set_grid_layer(s, static)
        hs.append((cm, s, o, il))
    cm = hs[0][0]
    assert cell_radius_and_reach(cm, hs[0][3], R) > 31
    mirror = np.full((sy, sx), 7, np.uint8)
    if registered:
        cuda.host_register(mirror)
    try:
        prev = None
        for cycle, kind in enumerate(["first", "window", "window", "whole", "whole", "whole", "static", "whole"]):
            outs = []
            for h, s, o, _ in hs:
                if kind == "whole":
                    h.touch_grid_layer(s, 0, 0, sx, sy)
                elif kind == "static":
                    changed = static.copy()
                    changed[150:156, 40:52] = 254
                    h.set_grid_layer(s, changed)
                    h.touch_grid_layer(s, 37, 147, 18, 12)
                obs, robot = moving_scan(sx, sy, cycle, seed)
                h.set_observations(o, obs)
                outs.append((h.update_map(*robot), h.get(), [h.get_layer(o)]))
            assert_cycles_equal([outs[0]], [outs[1]], f"mode {mode} R={R} cycle {cycle} ({kind})")
            w, now = outs[0][0], outs[0][1]
            n, nbytes, rects = cm.get_changed(mirror, max_rects=4096)
            assert cm.last_window() == w
            assert np.array_equal(mirror, now), f"cycle {cycle} ({kind}): the mirror differs from the device grid"
            if prev is not None:
                covered = np.zeros((sy, sx), bool)
                for x0, y0, xn, yn in rects[:n]:
                    covered[y0:yn, x0:xn] = True
                assert not ((prev != now) & ~covered).any(), f"cycle {cycle} ({kind}): a changed cell was not reported"
            prev = now
    finally:
        if registered:
            cuda.host_unregister(mirror)
