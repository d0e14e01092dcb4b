"""Seeded synthetic worlds and scans for the named configurations (SURVEY.md section 8d): used by bench.py and the
full-size parity tests.  Pure numpy, host side only.
"""
import numpy as np

LETHAL = 254


def warehouse_static(size_x, size_y, clutter=0.0, seed=1):
    """1-cell border + shelves: 6-cell-thick bars every 80 rows, 160 cells long per 200 columns (axis-aligned, thick:
    the class on which the reference's inflation does not depend on its priority-queue tie order)."""
    g = np.zeros((size_y, size_x), np.uint8)
    g[0, :] = g[-1, :] = LETHAL
    g[:, 0] = g[:, -1] = LETHAL
    for y in range(40, size_y - 10, 80):
        for x in range(20, size_x - 10, 200):
            g[y:y + 6, x:min(x + 160, size_x - 1)] = LETHAL
    if clutter > 0:
        rng = np.random.default_rng(seed)
        g[rng.random((size_y, size_x)) < clutter] = LETHAL
    return g


def pallets(size_x, size_y, centers, half=3):
    """Axis-aligned boxes that exist only in the scans (>= 3 cells thick)."""
    g = np.zeros((size_y, size_x), bool)
    for (cx, cy) in centers:
        g[max(0, cy - half):cy + half + 1, max(0, cx - half):cx + half + 1] = True
    return g


def raycast_scan(occupied, resolution, origin_xy, sensor_xy, n_beams=360, max_range=10.0, z=0.3, phase=0.0):
    """Casts n_beams rays from sensor_xy through the boolean world `occupied`; returns float32 (n,3) end points: the
    centre of the first occupied cell hit, or the point at max_range when nothing is hit."""
    sy, sx = occupied.shape
    ang = phase + np.arange(n_beams) * (2 * np.pi / n_beams)
    step = 0.5 * resolution
    n_steps = int(max_range / step)
    t = (np.arange(1, n_steps + 1) * step)[None, :]
    px = sensor_xy[0] + np.cos(ang)[:, None] * t
    py = sensor_xy[1] + np.sin(ang)[:, None] * t
    mx = np.floor((px - origin_xy[0]) / resolution).astype(np.int64)
    my = np.floor((py - origin_xy[1]) / resolution).astype(np.int64)
    inside = (mx >= 0) & (mx < sx) & (my >= 0) & (my < sy)
    hit = np.zeros_like(inside)
    hit[inside] = occupied[my[inside], mx[inside]]
    stop = hit | ~inside
    first = np.where(stop.any(axis=1), stop.argmax(axis=1), n_steps - 1)
    rows = np.arange(n_beams)
    hx, hy = mx[rows, first], my[rows, first]
    was_hit = hit[rows, first]
    ex = np.where(was_hit, origin_xy[0] + (hx + 0.5) * resolution, px[rows, first])
    ey = np.where(was_hit, origin_xy[1] + (hy + 0.5) * resolution, py[rows, first])
    return np.stack([ex, ey, np.full(n_beams, z)], axis=1).astype(np.float32)


def warehouse_c3(size=4000, resolution=0.05, n_obs=8, n_beams=360, scan_range=10.0, seed=1, cycle=0):
    """Config C3: static warehouse + K observations x 360 beams obtained by ray-casting the world (static + pallets)
    from sensor poses along an aisle.  Returns (static_grid, observations, robot_pose, footprint)."""
    static = warehouse_static(size, size)
    rng = np.random.default_rng(seed)
    aisle_y = (40 + 6 + 80 + 40) // 2 + 80 * (size // 160)  # middle of an aisle near the map centre
    x_start = size // 2 - 200 + 7 * cycle
    centers = [(x_start + int(rng.integers(-60, 160)), aisle_y + int(rng.integers(-20, 20))) for _ in range(6)]
    world = (static == LETHAL) | pallets(size, size, centers)
    obs = []
    for k in range(n_obs):
        sx_cell = x_start + 12 * k
        sensor = ((sx_cell + 0.5) * resolution, (aisle_y + 0.5) * resolution)
        while world[int(sensor[1] / resolution), int(sensor[0] / resolution)]:
            sensor = (sensor[0] + 7 * resolution, sensor[1])
        pts = raycast_scan(world, resolution, (0.0, 0.0), sensor, n_beams, scan_range, phase=0.001 * k)
        obs.append(dict(origin=(sensor[0], sensor[1], 0.3), points=pts, obstacle_range=scan_range,
                        raytrace_range=scan_range, marking=True, clearing=True))
    robot = (obs[-1]["origin"][0], obs[-1]["origin"][1], 0.0)
    half = 0.325
    footprint = [(half, half), (half, -half), (-half, -half), (-half, half)]
    return static, obs, robot, footprint


def blocks_c1(size=400, seed=1, adversarial=False):
    """Config C1: 400x400 border walls + rectangular blocks >= 3 cells thick; adversarial adds 1 % single cells."""
    rng = np.random.default_rng(seed)
    g = np.zeros((size, size), np.uint8)
    g[0:3, :] = g[-3:, :] = LETHAL
    g[:, 0:3] = g[:, -3:] = LETHAL
    for _ in range(25):
        w, h = int(rng.integers(3, 40)), int(rng.integers(3, 40))
        x, y = int(rng.integers(0, size - w)), int(rng.integers(0, size - h))
        g[y:y + h, x:x + w] = LETHAL
    if adversarial:
        g[rng.random((size, size)) < 0.01] = LETHAL
    return g


def fleet_robot(robot_id, n=120, res=0.05):
    """Config C5: the independent inputs of one robot of the fleet, seeded by its id -- a raw (un-inflated) n x n local
    map made of thick axis-aligned structure (corridor walls and boxes; the class on which the reference's inflation
    is tie-order independent), its world origin, pose, velocity and a plan through it."""
    rng = np.random.default_rng(1_000_003 * 7 + robot_id)
    raw = np.zeros((n, n), np.uint8)
    lo, hi = int(n * rng.uniform(0.15, 0.3)), int(n * rng.uniform(0.7, 0.85))
    raw[lo - 4:lo - 1, :] = 254
    raw[hi + 1:hi + 4, :] = 254
    for _ in range(int(rng.integers(1, 4))):
        bx, by = int(rng.integers(n // 2, n - 12)), int(rng.integers(lo + 6, hi - 12))
        w, h = int(rng.integers(3, 9)), int(rng.integers(3, 9))
        raw[by:by + h, bx:bx + w] = 254
    ox, oy = float(rng.uniform(-50, 50)), float(rng.uniform(-50, 50))
    size = n * res
    mid = oy + (lo + hi) / 2 * res
    pose = (ox + size * rng.uniform(0.15, 0.35), mid + rng.uniform(-0.3, 0.3), float(rng.uniform(-0.4, 0.4)))
    vel = (float(rng.uniform(0.0, 0.5)), 0.0, float(rng.uniform(-0.4, 0.4)))
    t = np.linspace(-0.05, 1.2, int(rng.integers(40, 160)))
    plan = np.stack([pose[0] + t * size * 0.75, mid + 0.25 * np.sin(t * rng.uniform(1, 3)) * rng.uniform(0, 1)], 1)
    return dict(raw=raw, origin=(ox, oy), pose=pose, vel=vel, plan=plan)


def fleet_sensing_robot(robot_id, n=120, res=0.05, cycles=64):
    """Config C5 with sensing: one robot's world, seeded by its id -- a 2n x 2n boolean grid with a corridor of thick
    axis-aligned walls and boxes and a few one-cell posts (point-like obstacles such as table legs), kept clear of the
    robot's path -- its origin, a pose per cycle driving along the corridor, a velocity and a plan.  The robot senses it
    through fleet_scan; its local n x n costmap is built from those scans alone."""
    rng = np.random.default_rng(2_000_003 * 7 + robot_id)
    wn = 2 * n
    world = np.zeros((wn, wn), bool)
    lo, hi = int(wn * rng.uniform(0.3, 0.38)), int(wn * rng.uniform(0.62, 0.7))
    world[lo - 4:lo, :] = True
    world[hi:hi + 4, :] = True
    mid_cell = (lo + hi) // 2

    def off_path(h):  # a row band that keeps an obstacle of height h at least 12 cells from the corridor's middle
        return int(rng.integers(mid_cell + 12, hi - h - 1)) if rng.random() < 0.5 else int(rng.integers(lo + 1, mid_cell - 12 - h))
    for _ in range(int(rng.integers(1, 4))):
        w, h = int(rng.integers(3, 9)), int(rng.integers(3, 9))
        bx, by = int(rng.integers(0, wn - w)), off_path(h)
        world[by:by + h, bx:bx + w] = True
    for _ in range(int(rng.integers(3, 7))):
        world[off_path(1), int(rng.integers(0, wn))] = True
    ox, oy = float(rng.uniform(-20, 20)), float(rng.uniform(-20, 20))
    mid = oy + (mid_cell + 0.5) * res
    x0 = ox + wn * res * rng.uniform(0.3, 0.4)
    speed, yaw0, ph = float(rng.uniform(0.01, 0.06)), float(rng.uniform(-0.4, 0.4)), float(rng.uniform(0, 6.28))
    c = np.arange(cycles)
    poses = np.stack([x0 + speed * c, mid + 0.1 * np.sin(0.3 * c + ph), yaw0 + 0.05 * np.sin(0.2 * c + ph)], 1)
    vel = (float(rng.uniform(0.0, 0.5)), 0.0, float(rng.uniform(-0.4, 0.4)))
    t = np.linspace(-0.05, 1.2, int(rng.integers(40, 160)))
    plan = np.stack([x0 + t * n * res * 0.75, mid + 0.15 * np.sin(t * rng.uniform(1, 3)) * rng.uniform(0, 1)], 1)
    return dict(world=world, origin=(ox, oy), resolution=res, poses=poses, vel=vel, plan=plan)


def fleet_scan(robot, cycle, cloud=False, n_beams=360, range_max=4.0):
    """One scan of `robot` (fleet_sensing_robot) at its pose of `cycle`: n_beams rays cast through its world from a
    sensor 0.3 m above the robot's centre, as a navgpu_laser_scan dict (the format Costmap.set_scans takes).  Beams
    without a return read +inf with inf_is_valid (laserScanValidInfCallback clears along them).  cloud=True gives the
    same end points as a PointCloud source (sensor-frame points) instead of ranges."""
    x, y, yaw = (float(v) for v in robot["poses"][cycle % len(robot["poses"])])
    phase = 0.001 * cycle
    pts = raycast_scan(robot["world"], robot["resolution"], robot["origin"], (x, y), n_beams, range_max, phase=phase)
    dx, dy = pts[:, 0].astype(np.float64) - x, pts[:, 1].astype(np.float64) - y
    scan = dict(translation=(x, y, 0.3), rotation_xyzw=(0.0, 0.0, float(np.sin(yaw / 2)), float(np.cos(yaw / 2))),
                min_obstacle_height=0.0, max_obstacle_height=2.0, obstacle_range=2.5, raytrace_range=3.0,
                marking=True, clearing=True)
    if cloud:
        cs, sn = np.cos(yaw), np.sin(yaw)
        scan["points"] = np.stack([cs * dx + sn * dy, -sn * dx + cs * dy, np.zeros_like(dx)], 1).astype(np.float32)
        return scan
    ranges = np.hypot(dx, dy).astype(np.float32)
    ranges[ranges >= np.float32(range_max - 1e-3)] = np.inf
    scan.update(ranges=ranges, angle_min=np.float32(phase - yaw), angle_increment=np.float32(2 * np.pi / n_beams),
                range_min=np.float32(0.05), range_max=np.float32(range_max), inf_is_valid=1)
    return scan


def _sensor_to_global(poses, z):
    """[n][7] tf transforms (translation, rotation xyzw) of sensors z above robots at poses [n][3]."""
    poses = np.asarray(poses, dtype=np.float64)
    yaw = poses[:, 2]
    zeros = np.zeros(len(poses))
    return np.ascontiguousarray(np.stack([poses[:, 0], poses[:, 1], np.full(len(poses), z), zeros, zeros,
                                          np.sin(yaw / 2), np.cos(yaw / 2)], 1))


def fleet_scan_batch(robots, cycle, cloud=False, n_beams=360, range_max=4.0):
    """One scan of every robot (fleet_sensing_robot) at its pose of `cycle`, as one source of Fleet.set_scan_batch:
    dense [n, n_beams] ranges (or [n, n_beams, 3] sensor-frame points with cloud=True) and [n, 7] sensor transforms.
    Unlike fleet_scan, every robot's scan shares one sensor-frame angle_min, so the rays are cast at world angle
    yaw + angle_min + i * angle_increment; the other fields are fleet_scan's."""
    angle_min, inc = np.float32(0.001 * cycle), np.float32(2 * np.pi / n_beams)
    poses = np.array([r["poses"][cycle % len(r["poses"])] for r in robots], dtype=np.float64)
    out = dict(sensor_to_global=_sensor_to_global(poses, 0.3), min_obstacle_height=0.0, max_obstacle_height=2.0,
               obstacle_range=2.5, raytrace_range=3.0, marking=True, clearing=True)
    rows = []
    for r, (x, y, yaw) in zip(robots, poses):
        pts = raycast_scan(r["world"], r["resolution"], r["origin"], (x, y), n_beams, range_max,
                           phase=yaw + float(angle_min))
        dx, dy = pts[:, 0].astype(np.float64) - x, pts[:, 1].astype(np.float64) - y
        if cloud:
            cs, sn = np.cos(yaw), np.sin(yaw)
            rows.append(np.stack([cs * dx + sn * dy, -sn * dx + cs * dy, np.zeros_like(dx)], 1).astype(np.float32))
        else:
            ranges = np.hypot(dx, dy).astype(np.float32)
            ranges[ranges >= np.float32(range_max - 1e-3)] = np.inf
            rows.append(ranges)
    if cloud:
        out["points"] = np.ascontiguousarray(np.stack(rows))
    else:
        out.update(ranges=np.ascontiguousarray(np.stack(rows)), angle_min=angle_min, angle_increment=inc,
                   range_min=np.float32(0.05), range_max=np.float32(range_max), inf_is_valid=1)
    return out


def fleet_cloud_3d_batch(robots, cycle, **kw):
    """fleet_cloud_3d of every robot (fleet_voxel_robot) as one source of Fleet.set_scan_batch: the clouds are in the
    sensor frame with shared fields, so the batch is their stack ([n, points, 3]) and the robots' [n, 7] transforms."""
    clouds = [fleet_cloud_3d(r, cycle, **kw) for r in robots]
    out = {k: v for k, v in clouds[0].items() if k not in ("points", "translation", "rotation_xyzw")}
    out["points"] = np.ascontiguousarray(np.stack([c["points"] for c in clouds]))
    out["sensor_to_global"] = np.ascontiguousarray([list(c["translation"]) + list(c["rotation_xyzw"]) for c in clouds],
                                                   dtype=np.float64)
    return out


def batch_scans(sources, n):
    """The per-robot scan-dict lists (Fleet.set_scans) that a batch of sources (Fleet.set_scan_batch) stands for:
    robot r's list holds, per source, its shared fields with row r of its arrays."""
    out = [[] for _ in range(n)]
    for src in sources:
        shared = {k: v for k, v in src.items() if k not in ("ranges", "points", "sensor_to_global")}
        key = "points" if "points" in src else "ranges"
        data, stg = np.asarray(src[key]), np.asarray(src["sensor_to_global"], dtype=np.float64)
        for r in range(n):
            out[r].append(dict(shared, **{key: data[r]}, translation=tuple(stg[r, :3]), rotation_xyzw=tuple(stg[r, 3:])))
    return out


# elevation rows of fleet_cloud_3d, degrees: straight down (floor returns under the robot: z-dominant rays), a shallow
# downward row (low obstacles; its floor return is beyond obstacle_range, so the floor only clears), the scan plane,
# two upward rows (tall obstacles, overhangs) and a steep upward one (z-dominant, ends above max_obstacle_height)
VOXEL_ELEVATIONS = (-80.0, -6.0, 0.0, 4.0, 25.0, 80.0)


def fleet_voxel_robot(robot_id, n=120, res=0.05, cycles=64):
    """fleet_sensing_robot's world with heights, for VoxelLayer fleets: every occupied cell gets a column [bottom, top]
    in metres -- the corridor walls 2.5 m (above the default max_obstacle_height), boxes and posts 0.12 .. 1.2 m in 8 x 8
    cell patches -- plus, next to the start of the path (off it by 14 cells or more), a 0.15 m high box below the scan
    plane and a tabletop from 0.7 to 0.75 m above it (an overhang the scan plane passes under).  Adds `bottom`, `top`
    (float32, top = -inf where free) and `seed` to fleet_sensing_robot's dict."""
    r = fleet_sensing_robot(robot_id, n=n, res=res, cycles=cycles)
    rng = np.random.default_rng(3_000_017 * 7 + robot_id)
    world = r["world"]
    wn = world.shape[0]
    patch = rng.uniform(0.12, 1.2, (wn // 8 + 1, wn // 8 + 1)).astype(np.float32)
    ys, xs = np.mgrid[0:wn, 0:wn]
    top = np.where(world, patch[ys // 8, xs // 8], -np.inf).astype(np.float32)
    top[world.all(axis=1), :] = 2.5
    bottom = np.zeros((wn, wn), np.float32)
    (ox, oy), poses = r["origin"], r["poses"]
    cx = int((poses[0, 0] - ox) / res)
    mc = int(round((poses[:, 1].mean() - oy) / res - 0.5))  # the corridor's middle row, to a cell or two
    low_y, low_x = mc + 14 + int(rng.integers(0, 3)), cx + int(rng.integers(30, 40))
    top[low_y:low_y + 4, low_x:low_x + 4] = 0.15
    tab_y, tab_x = mc - 24 + int(rng.integers(0, 3)), cx + int(rng.integers(8, 16))
    top[tab_y:tab_y + 8, tab_x:tab_x + 8] = 0.75
    bottom[tab_y:tab_y + 8, tab_x:tab_x + 8] = 0.7
    r.update(bottom=bottom, top=top, seed=robot_id)
    return r


def fleet_cloud_3d(robot, cycle, n_az=180, range_max=4.0, sensor_z=0.3):
    """One 3-D cloud of `robot` (fleet_voxel_robot) at its pose of `cycle`: len(VOXEL_ELEVATIONS) rows of n_az beams
    from a sensor sensor_z above the robot's centre, as an is_cloud navgpu_laser_scan dict (sensor-frame points, the
    format Costmap.set_scans takes).  A beam ends where it first enters an occupied column, on the floor (z = 0 with
    seeded noise of -3 .. +2 cm, so some returns lie below origin_z = 0) or, without a return, at range_max (the steep
    upward row then ends far above max_obstacle_height).  The projection keeps every point (heights -0.5 .. 5 m); the
    layer applies its own max_obstacle_height.  Vectorised over beams: the horizontal march is shared by the rows."""
    x, y, yaw = (float(v) for v in robot["poses"][cycle % len(robot["poses"])])
    res, (ox, oy) = robot["resolution"], robot["origin"]
    top, bottom = robot["top"], robot["bottom"]
    wn_y, wn_x = top.shape
    az = 0.001 * cycle + np.arange(n_az) * (2 * np.pi / n_az)
    step = 0.5 * res
    t = np.arange(1, int(range_max / step) + 1) * step  # horizontal distance of every march step
    px = x + np.cos(az)[:, None] * t
    py = y + np.sin(az)[:, None] * t
    mx = np.floor((px - ox) / res).astype(np.int64)
    my = np.floor((py - oy) / res).astype(np.int64)
    inside = (mx >= 0) & (mx < wn_x) & (my >= 0) & (my < wn_y)
    col_top = np.full(px.shape, -np.inf, np.float32)
    col_bot = np.zeros(px.shape, np.float32)
    col_top[inside] = top[my[inside], mx[inside]]
    col_bot[inside] = bottom[my[inside], mx[inside]]
    el = np.radians(np.asarray(VOXEL_ELEVATIONS))
    z = sensor_z + np.tan(el)[:, None] * t  # (rows, steps): the same for every azimuth
    hit = (z[:, None, :] <= col_top[None]) & (z[:, None, :] >= col_bot[None])
    floor = np.broadcast_to((z <= 0.0)[:, None, :], hit.shape)
    far = np.broadcast_to((t[None, :] / np.cos(el)[:, None] > range_max)[:, None, :] | ~inside[None], hit.shape)
    stop = hit | floor | far
    first = np.where(stop.any(axis=2), stop.argmax(axis=2), len(t) - 1)  # (rows, azimuths)
    took = lambda a: np.take_along_axis(a, first[..., None], axis=2)[..., 0]
    was_hit, was_floor = took(hit), took(floor) & ~took(hit)
    r3 = np.where(was_hit, t[first] / np.cos(el)[:, None], range_max)  # 3-D range along the beam
    tf = sensor_z / -np.tan(np.minimum(el, -1e-9))  # horizontal distance to the floor (downward rows)
    rng = np.random.default_rng((robot.get("seed", 0), cycle))
    floor_z = rng.uniform(-0.03, 0.02, first.shape)
    h = np.where(was_floor, np.broadcast_to(tf[:, None], first.shape), r3 * np.cos(el)[:, None])
    ez = np.where(was_floor, floor_z, sensor_z + r3 * np.sin(el)[:, None])
    dx, dy = (np.cos(az)[None, :] * h).ravel(), (np.sin(az)[None, :] * h).ravel()
    cs, sn = np.cos(yaw), np.sin(yaw)
    pts = np.stack([cs * dx + sn * dy, -sn * dx + cs * dy, ez.ravel() - sensor_z], 1).astype(np.float32)
    return dict(points=pts, translation=(x, y, sensor_z),
                rotation_xyzw=(0.0, 0.0, float(np.sin(yaw / 2)), float(np.cos(yaw / 2))),
                min_obstacle_height=-0.5, max_obstacle_height=5.0, obstacle_range=2.5, raytrace_range=3.0,
                marking=True, clearing=True)
