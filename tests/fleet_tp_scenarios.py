"""Robots for fleets of legacy TrajectoryPlanners (tests/test_gpu_fleet_tp.py): between them they take every branch of
TrajectoryPlanner::createTrajectories' selection -- a forward choice, rotation in place facing a wall, strafing in a
slot then backing up into escape mode and leaving it, oscillation flags latching and resetting, the final-goal cap,
plans that leave the map, an empty plan and a robot off its raw map -- so that robots with different sample counts
share every step.

Every robot lives in a 12 x 12 m world at 0.05 m (a 240 x 240 boolean grid with heights for VoxelLayer clouds) whose
middle 6 x 6 m is its raw local map.  Raw-map fleets get that middle (scenario_raw); sensing fleets scan the whole world
from the robot's current pose (scenario_sources)."""
import numpy as np

from navigation_b200 import synth

RES = 0.05
N = 120          # local map cells a side
WN = 2 * N       # world cells a side
WALL_TOP = 1.0   # metres: below the default max_obstacle_height


class Robot:
    def __init__(self, rid, world_origin, pose, vel, plan, dt=0.1, world=None, closes_at=None, plan2=None,
                 plan2_at=None):
        self.rid = rid
        self.world_origin = world_origin            # world cell (0, 0) in metres; the map's origin is 3 m further
        self.pose = np.array(pose, float)
        self.vel = np.array(vel, float)
        self.plan = np.asarray(plan, float).reshape(-1, 2)
        self.dt = dt                                # seconds the pose advances per cycle at the chosen velocity
        self.world = np.zeros((WN, WN), bool) if world is None else world
        self.closed = None                          # the world from cycle closes_at on
        self.closes_at = closes_at
        self.plan2, self.plan2_at = plan2, plan2_at  # a new plan from cycle plan2_at on

    @property
    def map_origin(self):
        return (self.world_origin[0] + N / 2 * RES, self.world_origin[1] + N / 2 * RES)

    def world_at(self, cycle):
        return self.closed if self.closes_at is not None and cycle >= self.closes_at else self.world

    def plan_at(self, cycle):
        return self.plan2 if self.plan2_at is not None and cycle >= self.plan2_at else self.plan


def _cell(v):  # map metres (origin at the local map's corner) to a world cell index
    return int(round(v / RES)) + N // 2


def scenario(n=16):
    """n >= 12 robots; ids 0-9 take the branches, the rest are corridor robots with varied headings and speeds."""
    assert n >= 12
    rng = np.random.default_rng(424242)
    robots = []
    for i in range(n):
        wo = (float(rng.uniform(-40, 40)), float(rng.uniform(-40, 40)))
        mo = (wo[0] + 3.0, wo[1] + 3.0)  # the local map's origin
        world = np.zeros((WN, WN), bool)
        if i == 4:  # nose against a wall, the plan to its left: rotation in place, then the way along the wall
            world[_cell(0.5):_cell(5.5), _cell(2.75):_cell(2.9)] = True
            r = Robot(i, wo, (mo[0] + 2.1, mo[1] + 2.0, 0.0), (0.0, 0.0, 0.0),
                      np.stack([np.full(40, mo[0] + 2.1), np.linspace(mo[1] + 2.0, mo[1] + 5.5, 40)], 1), dt=0.3,
                      world=world)
        elif i == 5:  # a slot just wider than the robot, open along y: strafing, then closed: backing up, escape
            world[:, _cell(2.5):_cell(2.6)] = True
            world[:, _cell(3.5):_cell(3.6)] = True
            closed = world.copy()
            closed[_cell(2.45):_cell(2.55), :] = True
            closed[_cell(3.5):_cell(3.6), :] = True
            r = Robot(i, wo, (mo[0] + 3.0, mo[1] + 3.0, 0.0), (0.0, 0.0, 0.0),
                      np.stack([np.full(60, mo[0] + 3.0), np.linspace(mo[1] + 3.0, mo[1] + 5.9, 60)], 1), dt=0.1,
                      world=world, closes_at=6,
                      plan2=np.stack([np.full(60, mo[0] + 3.0), np.linspace(mo[1] + 3.0, mo[1] + 0.1, 60)], 1),
                      plan2_at=3)
            r.closed = closed
        elif i == 6:  # boxed in from the start, then released: backs up into escape mode, leaves it once it moved
            world[_cell(2.45):_cell(3.55), _cell(2.45):_cell(2.55)] = True
            world[_cell(2.45):_cell(3.55), _cell(3.45):_cell(3.55)] = True
            world[_cell(2.45):_cell(2.55), _cell(2.45):_cell(3.55)] = True
            world[_cell(3.45):_cell(3.55), _cell(2.45):_cell(3.55)] = True
            r = Robot(i, wo, (mo[0] + 3.0, mo[1] + 3.0, 0.0), (0.0, 0.0, 0.0),
                      np.stack([np.linspace(mo[0] + 3.0, mo[0] + 5.5, 50), np.full(50, mo[1] + 3.0)], 1), dt=1.5,
                      world=world, closes_at=3)
            r.closed = np.zeros_like(world)
        elif i == 7:  # the goal 0.2 m ahead: max_vel_x capped at its distance / sim_time
            r = Robot(i, wo, (mo[0] + 2.0, mo[1] + 3.0, 0.0), (0.5, 0.0, 0.0),
                      np.stack([np.linspace(mo[0] + 1.8, mo[0] + 2.2, 9), np.full(9, mo[1] + 3.0)], 1), dt=0.1,
                      world=world)
        elif i == 8:  # an empty plan: nothing is reachable, the robot backs up
            r = Robot(i, wo, (mo[0] + 2.0, mo[1] + 3.0, 0.3), (0.2, 0.0, 0.0), np.zeros((0, 2)), world=world)
        elif i == 9:  # off its raw map (raw-map fleets; a sensing robot's rolling window always holds it)
            r = Robot(i, wo, (mo[0] - 1.0, mo[1] + 3.0, 0.0), (0.2, 0.0, 0.0),
                      np.stack([np.linspace(mo[0] - 1.0, mo[0] + 4.0, 60), np.full(60, mo[1] + 3.0)], 1), world=world)
        else:  # corridor robots; their plans run off the map
            lo, hi = float(rng.uniform(1.2, 1.8)), float(rng.uniform(4.2, 4.8))
            world[_cell(lo) - 3:_cell(lo), :] = True
            world[_cell(hi):_cell(hi) + 3, :] = True
            for _ in range(int(rng.integers(0, 3))):
                bx, by = _cell(float(rng.uniform(3.5, 5.0))), _cell(float(rng.uniform(lo + 0.4, hi - 0.8)))
                world[by:by + int(rng.integers(3, 8)), bx:bx + int(rng.integers(3, 8))] = True
            mid = (lo + hi) / 2
            yaw = float(rng.uniform(-0.5, 0.5)) if i not in (2, 11) else float(rng.choice([2.5, -2.8]))
            t = np.linspace(-0.05, 1.2, int(rng.integers(40, 120)))
            plan = np.stack([mo[0] + 1.0 + t * 6.0, mo[1] + mid + 0.25 * np.sin(t * rng.uniform(1, 3))], 1)
            r = Robot(i, wo, (mo[0] + float(rng.uniform(0.8, 1.4)), mo[1] + mid + float(rng.uniform(-0.3, 0.3)), yaw),
                      (float(rng.uniform(0.0, 0.5)), 0.0, float(rng.uniform(-0.4, 0.4))), plan,
                      dt=float(rng.choice([0.1, 0.3])), world=world)
        robots.append(r)
    return robots


def scenario_raw(robots, cycle):
    """Raw local maps [n][N][N] and their origins [n][2] of a raw-map fleet at `cycle`."""
    maps = np.stack([np.where(r.world_at(cycle)[N // 2:N // 2 + N, N // 2:N // 2 + N], 254, 0).astype(np.uint8)
                     for r in robots])
    return maps, np.array([r.map_origin for r in robots])


def scenario_sources(robots, cycle, voxel):
    """Every robot's sensor source at `cycle` from its current pose: a LaserScan, or a 3-D cloud for VoxelLayers."""
    out = []
    for r in robots:
        w = r.world_at(cycle)
        d = dict(world=w, origin=r.world_origin, resolution=RES, poses=r.pose[None, :], seed=r.rid,
                 top=np.where(w, np.float32(WALL_TOP), np.float32(-np.inf)), bottom=np.zeros(w.shape, np.float32))
        out.append([synth.fleet_cloud_3d(d, cycle) if voxel else synth.fleet_scan(d, cycle)])
    return out


def advance(robots, results):
    """Every pose moves by its robot's dt at the velocity the planner chose (zero when it found none)."""
    for r, g in zip(robots, results):
        v = np.array([g["xv"], g["yv"], g["thetav"]]) if g["cost"] >= 0 else np.zeros(3)
        c, s = np.cos(r.pose[2]), np.sin(r.pose[2])
        r.pose = r.pose + r.dt * np.array([v[0] * c - v[1] * s, v[0] * s + v[1] * c, v[2]])
        r.vel = v


def branches(trace, cfg):
    """Which selection branches a robot's results took: trace = [(result, pose)] over its cycles."""
    seen = set()
    prev = None
    for g, _ in trace:
        f = g["flags"]
        if g["cost"] >= 0 and g["xv"] > 0:
            seen.add("forward")
        if g["cost"] >= 0 and g["xv"] == 0 and g["yv"] == 0 and g["thetav"] != 0:
            seen.add("rotate")
        if g["cost"] >= 0 and g["xv"] == 0 and g["yv"] != 0:
            seen.add("strafe")
        if g["xv"] == cfg.get("backup_vel", -0.1) and f & 256:
            seen.add("escape")
        if prev is not None and prev & 256 and not f & 256:
            seen.add("leave_escape")
        if f & 15:
            seen.add("stuck")
        if prev is not None and prev & 15 and not f & 15:
            seen.add("stuck_reset")
        prev = f
    return seen
