"""Plan following on the device (navgpu_fleet_set_global_plans, navgpu_fleet_update_plans_device, Fleet.plan).

1. Raw-map, 2-D sensing and voxel fleets that follow their global plans on the device beside host twins that run
   DWAPlannerROS's loop on the host: the checker's transformGlobalPlan / prunePlan, global-plan erasure in Python, then
   set_plans and a host step.  Robots advance along their plans (poses are pruned, the local plan slides, the alignment
   cheat switches on at the goal); one robot is teleported beyond the plan threshold and one more than 1 m off its
   path, so that their local plans come out empty.  Every cycle: held and local plans bit for bit, status, results,
   left-out robots' untouched records and oscillation masks; check_trajectories costs every third cycle.  Robot-cycles
   whose goal-front point differs between CUDA's and the host libm's trig are counted and left out of the results
   comparison only.
2. A few robots' cycles replayed through the checker's DWA with the host-derived local plans.
3. set_global_plans on a subset: only those robots' plans and oscillation flags change; a retained alignment plan
   longer than the new plan's slots survives.
4. prune_plan = 0.
5. Host calls between device updates: host steps, set_plans, set_active, set_maps, check_trajectories.
6. Refusals leave the fleet bit-identical to its twin at the next step.
7. update_plans_device + step_device in steady state capture into a CUDA graph (discarded unlaunched).
8. How often CUDA's and the host libm's goal-front points differ over 10^6 random robot / goal pairs.
9. 4096 robots with long plans, sampled through the checker."""
import ctypes as C
import math

import numpy as np
import pytest

import scenarios as sc
from navigation_b200 import synth
from navigation_b200.api import DwaResult
from test_gpu_fleet_device_step import CFG, SENTINEL, World, host_records, make_fleet

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

RES = 0.05
THRESHOLD = max(120 * RES / 2.0, 120 * RES / 2.0)  # transformGlobalPlan's dist_threshold of a 120 x 120 local map
IDENTITY = np.array([1.0, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0])
FPD = 0.325  # forward_point_distance (default)


def front_points(goals, poses):
    """The goal-front point of DWAPlanner::updatePlanAndLocalCosts from the host libm and from CUDA (torch), for goals
    [k][2] and robot poses [k][2] (rounded through float as the planner does)."""
    pf = poses.astype(np.float32).astype(np.float64)
    host = np.array([(gx + FPD * math.cos(a), gy + FPD * math.sin(a))
                     for (gx, gy), a in ((g, math.atan2(g[1] - p[1], g[0] - p[0])) for g, p in zip(goals, pf))])
    g, p = torch.from_numpy(goals).cuda(), torch.from_numpy(pf).cuda()
    a = torch.atan2(g[:, 1] - p[:, 1], g[:, 0] - p[:, 0])
    dev = torch.stack([g[:, 0] + FPD * torch.cos(a), g[:, 1] + FPD * torch.sin(a)], 1).cpu().numpy()
    return host.reshape(-1, 2), dev


class Twin:
    """DWAPlannerROS's plan loop on the host for every robot of a host-stepped fleet: the checker's transformGlobalPlan
    (identity transform) and prunePlan, erasure from the held global plans, then set_plans.  A robot whose local plan
    comes out empty is left out (set_active) and its planner state kept: set_plans replays its last pose and plan,
    which gives the same plans again."""

    def __init__(self, fleet, plans):
        self.fleet, self.n = fleet, fleet.n
        self.held = [np.asarray(p, dtype=np.float64).reshape(-1, 2) for p in plans]
        self.last = [None] * self.n
        self.mask = None

    def set_global(self, robots, plans):
        for r, p in zip(robots, plans):
            self.held[r] = np.asarray(p, dtype=np.float64).reshape(-1, 2)

    def update(self, port, poses, prune=True, user_active=None):
        xy = np.ascontiguousarray(poses[:, :2])
        _, local = port.plans_transform(self.held, xy, [IDENTITY] * self.n, [THRESHOLD] * self.n)
        if prune:
            erase = port.plans_prune(local, xy)
            local = [q[e:] for q, e in zip(local, erase)]
            self.held = [h[e:] for h, e in zip(self.held, erase)]
        local = [np.ascontiguousarray(q[:, :2]) for q in local]
        status = np.array([len(q) > 0 for q in local])
        for r in range(self.n):
            if status[r]:
                self.last[r] = (poses[r].copy(), local[r])
        assert all(s is not None for s in self.last), "every robot needs a local plan at its first update"
        self.fleet.set_plans(np.array([s[0] for s in self.last]), [s[1] for s in self.last])
        mask = status if user_active is None else status & user_active
        self.fleet.set_active(None if mask.all() else mask)
        self.mask = mask
        return status, local


def robot_plans(kind, world):
    return [np.asarray(r["plan"], dtype=np.float64) for r in world.robots]


def drive_poses(plans, cycle, rng, schedule):
    """Each robot's pose on its plan at the cycle's fraction of the way (schedule), with a little noise; yaw along the plan."""
    out = []
    for p in plans:
        i = min(int(schedule[cycle] * (len(p) - 1)), len(p) - 1)
        j = min(i + 1, len(p) - 1)
        yaw = math.atan2(p[j, 1] - p[i, 1], p[j, 0] - p[i, 0]) if j != i else 0.0
        out.append((p[i, 0] + rng.uniform(-0.03, 0.03), p[i, 1] + rng.uniform(-0.03, 0.03), yaw + rng.uniform(-0.2, 0.2)))
    return np.array(out)


def assert_plans(dev, twin, local, status, where):
    for r in range(dev.n):
        assert dev.plan(r, 0).tobytes() == twin.held[r].tobytes(), f"{where} robot {r}: held global plan differs"
        assert dev.plan(r, 1).tobytes() == local[r].tobytes(), f"{where} robot {r}: local plan differs"


def update_and_step(dev, twin, port, poses, vels, where, prune=True, user_active=None, out=None, record=None):
    """One cycle on both: the device update + device step, the twin's host loop + host step.  Returns the robots left
    out of the results comparison for the trig exception, the local plans and the status."""
    n = dev.n
    P = torch.from_numpy(poses).cuda()
    status = dev.update_plans_device(P, prune_plan=prune).cpu().numpy()
    exp_status, local = twin.update(port, poses, prune, user_active)
    assert (status == exp_status).all(), f"{where}: status {status} != {exp_status.astype(int)}"
    assert_plans(dev, twin, local, status, where)
    if out is None:
        out = torch.empty(n * C.sizeof(DwaResult), dtype=torch.uint8, device="cuda")
    out.fill_(SENTINEL)
    r = dev.step_device(P, torch.from_numpy(vels).cuda(), out=out)
    torch.cuda.synchronize()
    got = host_records(dev, r, twin.mask)
    exp = twin.fleet.step(poses, vels)
    # the goal-front points of the robots with a local plan, from the host libm and from CUDA
    have = [i for i in range(n) if status[i]]
    trig = set()
    if have:
        h, d = front_points(np.array([local[i][-1] for i in have]), poses[have, :2])
        trig = {i for k, i in enumerate(have) if h[k].tobytes() != d[k].tobytes()}
    for i in range(n):
        if i not in trig:
            assert got[i] == exp[i], f"{where} robot {i}: results differ"
    after = out.cpu().numpy().reshape(n, -1)
    assert (after[~twin.mask] == SENTINEL).all(), f"{where}: a left-out robot's record changed"
    for i in range(n):
        assert dev.oscillation_mask(i) == twin.fleet.oscillation_mask(i), f"{where} robot {i}: oscillation flags"
    if record is not None:
        record.append(len(trig))
    return trig, local, status


def check_costs(dev, host, poses, vels, trig, where):
    cand = [np.array([(0.2, 0.0, 0.0), (0.0, 0.0, 0.5), (0.1, 0.0, -0.3)]) for _ in range(dev.n)]
    a, b = dev.check_trajectories(poses, vels, cand), host.check_trajectories(poses, vels, cand)
    for i in range(dev.n):
        if i not in trig:
            assert a[i].tobytes() == b[i].tobytes(), f"{where} robot {i}: check_trajectories costs differ"


SCHEDULE = [0.0, 0.12, 0.25, 0.4, 0.55, 0.7, 0.85, 1.0, 1.0, 1.0]


@pytest.mark.parametrize("kind", ["raw", "sensing", "voxel"])
def test_plan_following_matches_host_twin(cuda, port, kind, record_property):
    n = 10
    w = World(kind, n, seed=21)
    dev, host = make_fleet(cuda, kind, n), make_fleet(cuda, kind, n)
    if kind == "raw":
        for f in (dev, host):
            f.set_maps(np.stack([r["raw"] for r in w.robots]), np.array([r["origin"] for r in w.robots]))
    plans = robot_plans(kind, w)
    dev.set_global_plans(plans)
    twin = Twin(host, plans)
    rng = np.random.default_rng(5)
    skipped, cheats, empties, pruned = [], 0, 0, 0
    for cycle in range(len(SCHEDULE)):
        poses, vels = drive_poses(plans, cycle, rng, SCHEDULE), w.vels()
        if cycle == 3:
            poses[1, :2] += (0.0, THRESHOLD + 5.0)  # beyond dist_threshold of every pose: nothing is transformed
            poses[2, :2] += (0.0, 1.6)              # within it, but more than 1 m off the path: all pruned
        before = sum(len(h) for h in twin.held)
        w.feed(dev, host, cycle)
        trig, local, status = update_and_step(dev, twin, port, poses, vels, f"cycle {cycle}", record=skipped)
        pruned += before - sum(len(h) for h in twin.held)
        empties += int((~status.astype(bool)).sum())
        cheats += sum(1 for i in range(n) if status[i] and np.hypot(*(poses[i, :2].astype(np.float32) - local[i][-1])) <= FPD)
        if cycle % 3 == 2:
            check_costs(dev, host, poses, vels, trig, f"cycle {cycle}")
    assert empties >= 2 and pruned > 0 and cheats > 0, (empties, pruned, cheats)
    record_property("trig_skipped_robot_cycles", sum(skipped))
    print(f"{kind}: {sum(skipped)} robot-cycles left out of the results comparison for the trig exception")


def test_checker_replay(cuda, port):
    """A few robots' cycles through the checker's DWA with the host-derived local plans: the device fleet's results
    equal the checker's (cost to the usual relative tolerance)."""
    n = 6
    w = World("raw", n, seed=23)
    dev = make_fleet(cuda, "raw", n)
    dev.set_maps(np.stack([r["raw"] for r in w.robots]), np.array([r["origin"] for r in w.robots]))
    plans = robot_plans("raw", w)
    dev.set_global_plans(plans)
    held = [p.copy() for p in plans]
    checkers = [port.dwa(120, 120, RES, **CFG) for _ in range(n)]
    rng = np.random.default_rng(9)
    compared = 0
    for cycle in range(6):
        poses, vels = drive_poses(plans, cycle, rng, SCHEDULE), w.vels()
        status = dev.update_plans_device(torch.from_numpy(poses).cuda()).cpu().numpy()
        r = dev.step_device(torch.from_numpy(poses).cuda(), torch.from_numpy(vels).cuda())
        got = host_records(dev, r)
        xy = np.ascontiguousarray(poses[:, :2])
        _, local = port.plans_transform(held, xy, [IDENTITY] * n, [THRESHOLD] * n)
        erase = port.plans_prune(local, xy)
        held = [h[e:] for h, e in zip(held, erase)]
        for i in range(n):
            q = local[i][erase[i]:, :2]
            assert bool(status[i]) == (len(q) > 0)
            if not len(q):
                continue
            d = checkers[i]
            cm = port.costmap(120, 120, RES, *w.robots[i]["origin"])
            s = cm.add_grid_layer(0)
            cm.add_inflation_layer(0.55, 10.0)
            cm.set_footprint(sc.PENTAGON)
            cm.set_grid_layer(s, w.robots[i]["raw"])
            cm.update_map(0, 0, 0)
            d.set_costmap(cm.get(), *w.robots[i]["origin"])
            d.set_plan(poses[i], np.ascontiguousarray(q))
            e = d.find_best_path(poses[i], vels[i], sc.PENTAGON)
            g = got[i]
            assert (g["best_index"], g["n_samples"], g["n_scored"]) == (e["best_index"], e["n_samples"], e["n_scored"])
            if e["ok"]:
                assert np.isclose(g["cost"], e["cost"], rtol=1e-5, atol=0)
                assert (g["xv"], g["yv"], g["thetav"]) == (e["xv"], e["yv"], e["thetav"])
            assert dev.oscillation_mask(i) == d.oscillation_mask()
            compared += 1
    assert compared >= 20


def test_set_global_plans_on_a_subset(cuda, port):
    n = 8
    w = World("raw", n, seed=25)
    dev, host = make_fleet(cuda, "raw", n), make_fleet(cuda, "raw", n)
    for f in (dev, host):
        f.set_maps(np.stack([r["raw"] for r in w.robots]), np.array([r["origin"] for r in w.robots]))
    plans = robot_plans("raw", w)
    dev.set_global_plans(plans)
    twin = Twin(host, plans)
    rng = np.random.default_rng(13)
    for cycle in range(4):
        poses, vels = drive_poses(plans, cycle, rng, SCHEDULE), w.vels()
        if cycle in (1, 2):  # forward then backward: flags latch
            vels[:] = (0.3, 0.0, 0.0) if cycle == 1 else (-0.3, 0.0, 0.0)
        update_and_step(dev, twin, port, poses, vels, f"cycle {cycle}")
    masks = [dev.oscillation_mask(i) for i in range(n)]
    # robots 0-3 get short new plans that end just ahead of them: the alignment critic keeps the longer poses it had
    subset = [0, 1, 2, 3]
    new = [np.array([poses[i, :2], poses[i, :2] + (0.05, 0.0), poses[i, :2] + (0.1, 0.0)]) for i in subset]
    dev.set_global_plans(new, robots=subset)
    host.set_global_plans(new, robots=subset)  # (the host twin's oscillation flags: setPlan resets them)
    twin.set_global(subset, new)
    after = [dev.oscillation_mask(i) for i in range(n)]
    assert after[:4] == [0] * 4 and after[4:] == masks[4:]
    assert any(masks[:4]), masks
    for i in range(4, n):
        assert dev.plan(i, 0).tobytes() == twin.held[i].tobytes()
    for cycle in range(4, 7):
        p2 = drive_poses(plans, cycle, rng, SCHEDULE)
        p2[subset] = poses[subset]
        trig, local, status = update_and_step(dev, twin, port, p2, w.vels(), f"cycle {cycle}")
        check_costs(dev, host, p2, w.vels(), trig, f"cycle {cycle}")
        for i in subset:
            assert status[i] and len(local[i]) == 3


def test_without_prune(cuda, port):
    n = 6
    w = World("raw", n, seed=27)
    dev, host = make_fleet(cuda, "raw", n), make_fleet(cuda, "raw", n)
    for f in (dev, host):
        f.set_maps(np.stack([r["raw"] for r in w.robots]), np.array([r["origin"] for r in w.robots]))
    plans = robot_plans("raw", w)
    dev.set_global_plans(plans)
    twin = Twin(host, plans)
    rng = np.random.default_rng(15)
    for cycle in range(5):
        poses = drive_poses(plans, cycle, rng, SCHEDULE)
        update_and_step(dev, twin, port, poses, w.vels(), f"cycle {cycle}", prune=False)
    assert [len(dev.plan(i, 0)) for i in range(n)] == [len(p) for p in plans]


@pytest.mark.parametrize("kind", ["raw", "sensing"])
def test_mixed_host_calls(cuda, port, kind):
    n, cycles = 9, 10
    w = World(kind, n, seed=29)
    dev, host = make_fleet(cuda, kind, n), make_fleet(cuda, kind, n)
    if kind == "raw":
        for f in (dev, host):
            f.set_maps(np.stack([r["raw"] for r in w.robots]), np.array([r["origin"] for r in w.robots]))
    plans = robot_plans(kind, w)
    dev.set_global_plans(plans)
    twin = Twin(host, plans)
    rng = np.random.default_rng(17)
    user = None
    for cycle in range(cycles):
        poses, vels = drive_poses(plans, cycle, rng, SCHEDULE), w.vels()
        w.feed(dev, host, cycle)
        op = cycle % 5
        if op == 1:  # set_active after a device update: the device's plan records must survive it
            user = np.array([(i + cycle) % 3 != 0 for i in range(n)])
            dev.set_active(user)
        if op == 2 and kind == "raw":
            maps = np.stack([np.roll(r["raw"], cycle, axis=1) for r in w.robots])
            for f in (dev, host):
                f.set_maps(maps, np.array([r["origin"] for r in w.robots]))
        if op == 3:  # set_plans between updates (the twin's host loop then runs its own set_plans)
            for f in (dev, host):
                f.set_plans(poses, [p[:5] for p in plans])
        if op == 4:
            user = None
            dev.set_active(None)
        trig, local, status = update_and_step(dev, twin, port, poses, vels, f"cycle {cycle}", user_active=user)
        if op == 0 and cycle:  # a host step on both, after the device update
            a, b = dev.step(poses, vels), twin.fleet.step(poses, vels)
            assert [x for x, m in zip(a, twin.mask) if m] == [x for x, m in zip(b, twin.mask) if m], \
                f"cycle {cycle}: host steps differ"
        if op == 2:
            check_costs(dev, host, poses, vels, trig, f"cycle {cycle}")


def test_refusals_leave_the_fleet_as_it_was(cuda, port):
    lib = cuda.lib
    n = 6
    w = World("raw", n, seed=31)
    dev, host = make_fleet(cuda, "raw", n), make_fleet(cuda, "raw", n)
    for f in (dev, host):
        f.set_maps(np.stack([r["raw"] for r in w.robots]), np.array([r["origin"] for r in w.robots]))
    plans = robot_plans("raw", w)
    dev.set_global_plans(plans)
    twin = Twin(host, plans)
    tp = cuda.fleet(n, 40, 40, RES, sc.PENTAGON, trajectory_planner={})
    rng = np.random.default_rng(19)
    P = torch.zeros((n, 3), dtype=torch.float64, device="cuda")
    S = torch.zeros(n, dtype=torch.uint8, device="cuda")
    hp, hs = np.zeros((n, 3)), np.zeros(n, dtype=np.uint8)
    xy = np.zeros((4, 2))
    f64 = xy.ctypes.data_as(C.POINTER(C.c_double))
    ptr = lambda t: C.c_void_p(t.data_ptr())
    keep = []

    def arr(a):
        keep.append(np.ascontiguousarray(a, dtype=np.int32))
        return keep[-1].ctypes.data_as(C.POINTER(C.c_int32))

    cases = [
        ("update: null handle", 2, lambda: lib.navgpu_fleet_update_plans_device(None, ptr(P), 1, ptr(S))),
        ("update: null poses", 2, lambda: lib.navgpu_fleet_update_plans_device(dev.h, None, 1, ptr(S))),
        ("update: host poses", 2, lambda: lib.navgpu_fleet_update_plans_device(dev.h, C.c_void_p(hp.ctypes.data), 1, ptr(S))),
        ("update: host status", 2, lambda: lib.navgpu_fleet_update_plans_device(dev.h, ptr(P), 1, C.c_void_p(hs.ctypes.data))),
        ("update: TrajectoryPlanner fleet", 3, lambda: lib.navgpu_fleet_update_plans_device(tp.h, ptr(P), 1, ptr(S))),
        ("set: robot out of range", 2, lambda: lib.navgpu_fleet_set_global_plans(dev.h, 1, arr([n]), f64, arr([0, 2]))),
        ("set: negative robot", 2, lambda: lib.navgpu_fleet_set_global_plans(dev.h, 1, arr([-1]), f64, arr([0, 2]))),
        ("set: repeated robot", 2, lambda: lib.navgpu_fleet_set_global_plans(dev.h, 2, arr([1, 1]), f64, arr([0, 2, 4]))),
        ("set: offsets not from 0", 2, lambda: lib.navgpu_fleet_set_global_plans(dev.h, 1, arr([1]), f64, arr([1, 2]))),
        ("set: decreasing offsets", 2, lambda: lib.navgpu_fleet_set_global_plans(dev.h, 2, arr([1, 2]), f64, arr([0, 3, 2]))),
        ("set: null robots", 2, lambda: lib.navgpu_fleet_set_global_plans(dev.h, 1, None, f64, arr([0, 2]))),
        ("set: null plan", 2, lambda: lib.navgpu_fleet_set_global_plans(dev.h, 1, arr([1]), None, arr([0, 2]))),
        ("set: null offsets", 2, lambda: lib.navgpu_fleet_set_global_plans(dev.h, 1, arr([1]), f64, None)),
        ("set: TrajectoryPlanner fleet", 3, lambda: lib.navgpu_fleet_set_global_plans(tp.h, 1, arr([1]), f64, arr([0, 2]))),
    ]
    update_and_step(dev, twin, port, drive_poses(plans, 0, rng, SCHEDULE), w.vels(), "before")
    for cycle, (name, code, call) in enumerate(cases, start=1):
        rc = call()
        assert rc == code, f"{name}: {rc} ({lib.navgpu_last_error().decode()})"
        poses = drive_poses(plans, min(cycle, len(SCHEDULE) - 1), rng, SCHEDULE)
        update_and_step(dev, twin, port, poses, w.vels(), f"after {name}")
    for bad in (P.float(), P[:-1], P.cpu()):
        with pytest.raises(ValueError):
            dev.update_plans_device(bad)


@pytest.mark.parametrize("kind", ["raw", "sensing", "voxel"])
def test_steady_state_cycle_captures(cuda, kind):
    """Two cycles of update + step size every buffer; the third, enqueued under thread-local stream capture, must
    capture without a host wait, an allocation or a pageable copy.  The graph is discarded unlaunched."""
    cu = C.CDLL("libcuda.so.1")
    n = 8
    w = World(kind, n, seed=33)
    dev, host = make_fleet(cuda, kind, n), make_fleet(cuda, kind, n)
    if kind == "raw":
        dev.set_maps(np.stack([r["raw"] for r in w.robots]), np.array([r["origin"] for r in w.robots]))
    plans = robot_plans(kind, w)
    dev.set_global_plans(plans)
    P = torch.from_numpy(drive_poses(plans, 1, np.random.default_rng(3), SCHEDULE)).cuda()
    V = torch.from_numpy(w.vels()).cuda()
    R = torch.zeros(n * C.sizeof(DwaResult), dtype=torch.uint8, device="cuda")
    S = torch.zeros(n, dtype=torch.uint8, device="cuda")
    for cycle in range(2):
        w.feed(dev, host, cycle)
        dev.update_plans_device(P)
        dev.step_device(P, V, out=R)
    torch.cuda.synchronize()
    stream = C.c_void_p(dev.stream())
    assert cu.cuStreamBeginCapture_v2(stream, 1) == 0  # CU_STREAM_CAPTURE_MODE_THREAD_LOCAL
    rc1 = cuda.lib.navgpu_fleet_update_plans_device(dev.h, C.c_void_p(P.data_ptr()), 1, C.c_void_p(S.data_ptr()))
    msg1 = cuda.lib.navgpu_last_error().decode()
    rc2 = cuda.lib.navgpu_fleet_step_device(dev.h, C.c_void_p(P.data_ptr()), C.c_void_p(V.data_ptr()),
                                            C.c_void_p(R.data_ptr()))
    msg2 = cuda.lib.navgpu_last_error().decode()
    graph = C.c_void_p()
    end = cu.cuStreamEndCapture(stream, C.byref(graph))
    assert rc1 == 0, msg1
    assert rc2 == 0, msg2
    assert end == 0 and graph.value
    assert cu.cuGraphDestroy(graph) == 0
    del dev


def test_cuda_and_libm_front_points(record_property):
    """The goal-front point takes atan2 / cos / sin from CUDA on the device and from the host libm on the host.  Counts
    how often the two points differ over 10^6 random robot / goal pairs; CUDA's atan2, cos and sin stay within 2 ulp of
    the libm's."""
    rng = np.random.default_rng(37)
    k = 1_000_000
    goals = rng.uniform(-60, 60, (k, 2))
    poses = goals + rng.uniform(-3, 3, (k, 2))
    h, d = front_points(goals, poses)
    differ = int((h != d).any(axis=1).sum())
    record_property("front_points_differ", differ)
    record_property("pairs", k)
    print(f"goal-front points: {differ} of {k} differ between CUDA and the host libm")
    pf = poses.astype(np.float32).astype(np.float64)
    dy, dx = goals[:, 1] - pf[:, 1], goals[:, 0] - pf[:, 0]
    ang = np.array([math.atan2(y, x) for y, x in zip(dy, dx)])
    t = torch.from_numpy(ang).cuda()
    for name, dev, host in (("atan2", torch.atan2(torch.from_numpy(dy).cuda(), torch.from_numpy(dx).cuda()), ang),
                            ("cos", torch.cos(t), np.array([math.cos(v) for v in ang])),
                            ("sin", torch.sin(t), np.array([math.sin(v) for v in ang]))):
        ulps = np.abs(dev.cpu().numpy().view(np.int64) - host.view(np.int64))
        assert ulps.max() <= 2, name


def test_c5_fleet_with_long_plans(cuda, port):
    """4096 robots with C5's inputs and global plans of thousands of poses through and beyond their maps: two cycles
    of update + step, every 64th robot's plans, result and flags checked against the checker's loop."""
    cfg = dict(vx_samples=20, vy_samples=1, vth_samples=20, max_vel_y=0.0, min_vel_y=0.0)
    n = 4096
    robots = [synth.fleet_robot(i) for i in range(n)]
    dev = cuda.fleet(n, 120, 120, RES, sc.PENTAGON, 0.55, 10.0, **cfg)
    dev.set_maps(np.stack([r["raw"] for r in robots]), np.array([r["origin"] for r in robots]))
    plans = []
    for i, r in enumerate(robots):
        t = np.arange(-200, 1800 + (i % 7) * 100) * 0.025  # 0.025 m apart, from 5 m behind to 45+ m ahead
        x0, y0, yaw = r["pose"]
        plans.append(np.stack([x0 + t * math.cos(yaw * 0.2), y0 + t * math.sin(yaw * 0.2) + 0.2 * np.sin(t)], 1))
    dev.set_global_plans(plans)
    held = [p.copy() for p in plans]
    sample = list(range(0, n, 64))
    checkers = {i: port.dwa(120, 120, RES, **cfg) for i in sample}
    valid = 0
    for cycle in range(2):
        poses = np.array([(p[200 + 20 * cycle, 0], p[200 + 20 * cycle, 1], robots[i]["pose"][2])
                          for i, p in enumerate(plans)])
        vels = np.array([r["vel"] for r in robots])
        P = torch.from_numpy(poses).cuda()
        status = dev.update_plans_device(P).cpu().numpy()
        out = host_records(dev, dev.step_device(P, torch.from_numpy(vels).cuda()))
        assert status.all()
        xy = np.ascontiguousarray(poses[sample, :2])
        _, local = port.plans_transform([held[i] for i in sample], xy, [IDENTITY] * len(sample),
                                        [THRESHOLD] * len(sample))
        erase = port.plans_prune(local, xy)
        for k, i in enumerate(sample):
            held[i] = held[i][erase[k]:]
            q = np.ascontiguousarray(local[k][erase[k]:, :2])
            assert dev.plan(i, 0).tobytes() == held[i].tobytes(), f"robot {i}"
            assert dev.plan(i, 1).tobytes() == q.tobytes(), f"robot {i}"
            cm = port.costmap(120, 120, RES, *robots[i]["origin"])
            s = cm.add_grid_layer(0)
            cm.add_inflation_layer(0.55, 10.0)
            cm.set_footprint(sc.PENTAGON)
            cm.set_grid_layer(s, robots[i]["raw"])
            cm.update_map(0, 0, 0)
            d = checkers[i]
            d.set_costmap(cm.get(), *robots[i]["origin"])
            d.set_plan(poses[i], q)
            e = d.find_best_path(poses[i], vels[i], sc.PENTAGON)
            g = out[i]
            assert (g["best_index"], g["n_samples"], g["n_scored"]) == (e["best_index"], e["n_samples"], e["n_scored"])
            assert dev.oscillation_mask(i) == d.oscillation_mask()
            if e["ok"]:
                assert np.isclose(g["cost"], e["cost"], rtol=1e-5, atol=0)
                valid += 1
    assert valid >= 32
