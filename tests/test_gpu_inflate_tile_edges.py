"""k_inflate works on tiles of 128 columns x 64 rows, and each lane reads and writes four cells of a row as one 32-bit
word.  These cases put the map edges, the update window's edges and NO_INFORMATION cells where that shape can get them
wrong: widths of 4k + 1, 4k + 2 and 4k + 3 cells, so that the last word of a row holds 1-3 cells of the map and the
rest is row padding; maps narrower or shorter than one tile; window edges inside a tile; NO_INFORMATION next to LETHAL
in the last columns; and effective reaches that select each of the three instantiations (reach <= 12, 20, 31).

launch_sweep picks the instantiation by the effective reach -- the largest distance whose cost is non-zero -- not by
the cell radius R: with a steep cost scaling the reach is well below R, and k_merge_seed's seed region (R) is wider
than k_inflate's halo rows (the reach).  The device grid must equal the checker's exact nearest-seed variant cell for
cell."""
import numpy as np
import pytest

import scenarios as sc

pytestmark = pytest.mark.gpu

RES = 0.05
# (inflation radius in m, cost scaling) -> (cell radius R, effective reach).  With scaling 1.0 the cost stays non-zero
# out to the radius, so the reach is R: k_inflate<12>, <20> and <31>.  Then a reach well below R (12 of 31: <12>;
# 17 of 25: <20>), the smallest reach that takes <31> (21), and scaling 0 (cost 252 out to R = 31).
RADII = {(0.55, 1.0): (11, 11), (0.95, 1.0): (19, 19), (1.5, 1.0): (30, 30), (1.525, 20.0): (31, 12),
         (1.225, 10.0): (25, 17), (1.025, 1.0): (21, 21), (1.525, 0.0): (31, 31)}
# widths 4k + 1 / 4k + 2 / 4k + 3, narrower than one tile and spanning several; heights not multiples of 64
SHAPES = [(37, 45), (102, 130), (127, 63), (257, 200), (262, 71), (391, 133)]


def edge_world(sx, sy, seed):
    """Walls, pillars and single seeds, with LETHAL and NO_INFORMATION cells packed into the last three columns."""
    rng = np.random.default_rng(seed)
    g = np.zeros((sy, sx), np.uint8)
    g[sy // 3, 2:max(3, sx - 7)] = 254
    g[3:max(4, sy - 4), sx // 2] = 254
    for _ in range(max(2, sx * sy // 900)):
        x, y = int(rng.integers(0, sx)), int(rng.integers(0, sy))
        g[y:y + int(rng.integers(1, 4)), x:x + int(rng.integers(1, 4))] = 254
    ys = np.arange(sy)
    g[ys % 5 == 0, sx - 1] = 254
    g[ys % 5 == 1, sx - 1] = 255
    g[ys % 7 == 2, sx - 2] = 255
    g[ys % 7 == 3, sx - 2] = 254
    g[ys % 3 == 0, sx - 3] = 255
    g[(ys % 11 == 4), sx - 4] = 254
    g[rng.random((sy, sx)) < 0.02] = 255  # NO_INFORMATION scattered everywhere, also inside the reach of seeds
    return g


def marks(sx, sy, seed):
    """A few marked points in the middle of the map: the update window they make has its edges inside tiles."""
    rng = np.random.default_rng(seed)
    xs = rng.uniform(0.3 * sx, 0.7 * sx, 6) * RES
    ys = rng.uniform(0.3 * sy, 0.7 * sy, 6) * RES
    pts = np.stack([xs, ys, np.full(6, 0.5)], 1).astype(np.float32)
    return [dict(origin=(0.5 * sx * RES, 0.5 * sy * RES, 0.5), points=pts, obstacle_range=100.0,
                 raytrace_range=100.0, marking=True, clearing=False)]


@pytest.mark.parametrize("radius,scaling", list(RADII))
@pytest.mark.parametrize("sx,sy", SHAPES)
def test_tile_edges_exact(cuda, port, sx, sy, radius, scaling):
    static = edge_world(sx, sy, sx * 1000 + sy)
    outs = []
    for api in (cuda, port):
        cm = api.costmap(sx, sy, RES)
        s = cm.add_grid_layer(0)
        o = cm.add_obstacle_layer(1, False, 2.0)
        il = cm.add_inflation_layer(radius, scaling)
        cm.set_footprint(sc.square_footprint())
        cm.set_grid_layer(s, static)
        sc.select_inflation(cm, il, "exact", 0)
        R, costs, _ = cm.inflation_tables(il)
        n = np.arange(R + 2)
        d2 = n[:, None] ** 2 + n[None, :] ** 2
        reach = int(np.sqrt(d2[(d2 <= R * R) & (costs > 0)].max() + 0.5))
        assert (R, reach) == RADII[(radius, scaling)], f"{api.name}: (R, reach) = {(R, reach)}"
        trace = [(cm.update_map(), cm.get())]
        # second cycle: only the marks changed, so the window is their bounds grown by the radius
        cm.set_observations(o, marks(sx, sy, sx + sy))
        trace.append((cm.update_map(), cm.get()))
        outs.append(trace)
    for cycle, ((wa, ga), (wb, gb)) in enumerate(zip(*outs)):
        assert wa == wb, f"cycle {cycle}: window {wa} != checker's {wb}"
        assert np.array_equal(ga, gb), f"cycle {cycle}: {int((ga != gb).sum())} cells differ from the checker"
