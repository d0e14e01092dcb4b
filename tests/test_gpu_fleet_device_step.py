"""Device-resident DWAPlanner fleet steps (navgpu_fleet_step_device, Fleet.step_device): poses and velocities in device
memory, results written on the fleet's stream.

1. Raw-map, 2-D sensing and voxel fleets beside host-stepped twins over multi-step runs with random poses and
   velocities (sensing fleets fed through set_scan_batch_device): every step results, master grids, layers, voxel
   columns, windows and origins are bit-equal; oscillation masks at the end of chains of device steps.  A few robots
   of the raw-map run are replayed through the CPU checker.
2. Oscillation flags that latch and are later reset by distance and by angle.
3. Host calls between device steps: host steps, set_plans, set_active with a changing subset, check_trajectories
   (whose costs read the distance grids), reset_oscillation, get_oscillation_mask, get_geometry and set_maps.
   Left-out robots keep a sentinel byte pattern in their result records.
4. Refusals leave the fleet bit-identical to its twin at the next step.
5. A steady-state device step is captured under cudaStreamBeginCapture (thread-local mode, which rejects host waits
   and allocations) without error; the graph is discarded without being launched.
6. How often CUDA's and numpy's cos / sin differ over 10^6 random yaws (a sensing fleet's footprint transform).
7. 4096 robots with C5's inputs, sampled through the CPU checker."""
import ctypes as C

import numpy as np
import pytest

import scenarios as sc
from navigation_b200 import synth
from navigation_b200.api import DwaResult

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

RES = 0.05
RTOL = 1e-5
# vy pinned, backward motion allowed: a robot driven forward then backward latches forward_neg_only
CFG = dict(vx_samples=6, vy_samples=1, vth_samples=11, max_vel_y=0.0, min_vel_y=0.0, min_vel_x=-0.3)
FIELDS = ("cost", "xv", "yv", "thetav", "best_index", "n_samples", "n_scored")
SENTINEL = 0xA5


def make_fleet(api, kind, n, **cfg):
    cfg = dict(CFG, **cfg)
    if kind == "raw":
        return api.fleet(n, 120, 120, RES, sc.PENTAGON, 0.55, 10.0, **cfg)
    return api.fleet_sensing(n, 120, 120, RES, sc.PENTAGON, voxel={} if kind == "voxel" else None, **cfg)


class World:
    """n robots of one fleet kind and their per-cycle inputs: noisy poses around the robots' own, random velocities."""

    def __init__(self, kind, n, seed=0):
        self.kind, self.n = kind, n
        self.rng = np.random.default_rng(seed)
        if kind == "raw":
            self.robots = [synth.fleet_robot(100 + i) for i in range(n)]
            self.base = np.array([r["pose"] for r in self.robots])
        else:
            make = synth.fleet_voxel_robot if kind == "voxel" else synth.fleet_sensing_robot
            self.robots = [make(300 + i) for i in range(n)]
            self.base = None

    def poses(self, cycle):
        base = self.base if self.base is not None else np.array([r["poses"][cycle] for r in self.robots])
        noise = self.rng.uniform(-1, 1, (self.n, 3)) * np.array([0.02, 0.02, 0.3])
        return np.ascontiguousarray(base + noise)

    def vels(self):
        v = np.zeros((self.n, 3))
        v[:, 0] = self.rng.uniform(-0.35, 0.6, self.n)
        v[:, 2] = self.rng.uniform(-1.0, 1.0, self.n)
        v[::5, 1] = 0.2  # outside the pinned y window: n samples on that axis
        return v

    def plans(self, poses):
        return [r["plan"] for r in self.robots]

    def setup(self, *fleets):
        for f in fleets:
            if self.kind == "raw":
                f.set_maps(np.stack([r["raw"] for r in self.robots]), np.array([r["origin"] for r in self.robots]))
            f.set_plans(self.base if self.base is not None else np.array([r["poses"][0] for r in self.robots]),
                        self.plans(None))

    def sources(self, cycle):
        if self.kind == "voxel":
            return [synth.fleet_cloud_3d_batch(self.robots, cycle)]
        return [synth.fleet_scan_batch(self.robots, cycle), synth.fleet_scan_batch(self.robots, cycle, cloud=True,
                                                                                  n_beams=120)]

    def feed(self, dev, host, cycle):
        """Scans of the cycle: CUDA tensors to the device-stepped fleet, the same host arrays to its twin."""
        if self.kind == "raw":
            return
        src = self.sources(cycle)
        on_dev = []
        for s in src:
            d = dict(s)
            for k in ("ranges", "points", "sensor_to_global"):
                if k in s:
                    d[k] = torch.from_numpy(s[k]).cuda()
            on_dev.append(d)
        dev.set_scan_batch(on_dev)
        host.set_scan_batch(src)


def dev_step(fleet, poses, vels, out=None):
    r = fleet.step_device(torch.from_numpy(poses).cuda(), torch.from_numpy(vels).cuda(), out=out)
    torch.cuda.synchronize()
    return r


def host_records(fleet, dev_out, active=None):
    """The device results as step()'s list of dicts (None for left-out robots)."""
    cols = {k: dev_out[k].cpu().numpy() for k in FIELDS}
    out = [{k: cols[k][i].item() for k in FIELDS} for i in range(fleet.n)]
    return out if active is None else [g if a else None for g, a in zip(out, active)]


def assert_twins(dev, host, kind, where, state=True):
    for i in range(dev.n):
        w = f"{where} robot {i}"
        assert np.array_equal(dev.costmap(i), host.costmap(i)), f"{w}: master grid differs"
        if kind != "raw":
            assert np.array_equal(dev.layer(i), host.layer(i)), f"{w}: obstacle layer differs"
        if kind == "voxel":
            assert np.array_equal(dev.voxels(i), host.voxels(i)), f"{w}: voxel columns differ"
        if state:  # (these bring the device state back to the host: the next device step uploads it again)
            assert dev.oscillation_mask(i) == host.oscillation_mask(i), w
            if kind != "raw":
                assert dev.geometry(i) == host.geometry(i), w


def step_pair(dev, host, poses, vels, where, active=None, out=None):
    r = dev_step(dev, poses, vels, out)
    got = host_records(dev, r, active)
    exp = host.step(poses, vels)
    assert got == exp, f"{where}: results differ"
    return r, exp


@pytest.mark.parametrize("kind", ["raw", "sensing", "voxel"])
def test_device_steps_match_host_twin(cuda, port, kind):
    n, cycles = 12, 9
    w = World(kind, n, seed=1)
    dev, host = make_fleet(cuda, kind, n), make_fleet(cuda, kind, n)
    w.setup(dev, host)
    latched = valid = 0
    for cycle in range(cycles):
        poses, vels = w.poses(cycle), w.vels()
        if cycle in (1, 4):  # the same robots forward, then backward: flags latch
            vels[:4] = (0.3, 0.0, 0.0)
        if cycle in (2, 5):
            vels[:4] = (-0.3, 0.0, 0.0)
        w.feed(dev, host, cycle)
        _, exp = step_pair(dev, host, poses, vels, f"cycle {cycle}")
        valid += sum(g["cost"] >= 0 for g in exp)
        # the planner state is compared at the end of chains of three device steps
        assert_twins(dev, host, kind, f"cycle {cycle}", state=cycle % 3 == 2)
        if cycle % 3 == 2:
            latched += sum(host.oscillation_mask(i) != 0 for i in range(n))
    assert valid > n * cycles // 2 and latched > 0
    if kind == "raw":  # a few robots through the CPU checker, on the last cycle's inputs
        for i in (0, 5, 11):
            r = w.robots[i]
            cm = port.costmap(120, 120, RES, *r["origin"])
            s = cm.add_grid_layer(0)
            cm.add_inflation_layer(0.55, 10.0)
            cm.set_footprint(sc.PENTAGON)
            cm.set_grid_layer(s, r["raw"])
            cm.update_map(0, 0, 0)
            assert np.array_equal(dev.costmap(i), cm.get()), f"robot {i}"


def test_oscillation_latches_and_resets(cuda):
    """Robots 0-3 driven forward then backward latch forward_neg_only; 4-5 are then reset by distance, 6-7 by
    angle; the twins agree at every step."""
    n = 8
    w = World("raw", n)
    dev, host = make_fleet(cuda, "raw", n), make_fleet(cuda, "raw", n)
    w.setup(dev, host)
    for f in (dev, host):
        f.set_plans(w.base, [np.array([[p[0], p[1]], [p[0] + 1.5, p[1]]]) for p in w.base])
    poses = w.base.copy()
    poses[:, 2] = 0.0
    fwd, back = np.tile([0.3, 0.0, 0.0], (n, 1)), np.tile([-0.3, 0.0, 0.0], (n, 1))
    masks = []
    for cycle, vels in enumerate([fwd, back, back, back, back]):
        p = poses.copy()
        if cycle >= 3:
            p[4:6, 0] += 0.1 * (cycle - 2)  # beyond oscillation_reset_dist (0.05 m)
            p[6:8, 2] += 0.3 * (cycle - 2)  # beyond oscillation_reset_angle (0.2 rad)
        step_pair(dev, host, p, vels, f"cycle {cycle}")
        masks.append([dev.oscillation_mask(i) for i in range(n)])
        assert masks[-1] == [host.oscillation_mask(i) for i in range(n)]
    latched = [i for i in range(n) if masks[2][i] & 2]  # forward_neg_only
    assert len(latched) >= 4, masks
    reset = [i for i in latched if i >= 4 and masks[3][i] == 0]
    assert any(i < 6 for i in reset) and any(i >= 6 for i in reset), masks  # by distance (4, 5), by angle (6, 7)


@pytest.mark.parametrize("kind", ["raw", "sensing"])
def test_mixed_host_calls(cuda, kind):
    n, cycles = 10, 12
    w = World(kind, n, seed=3)
    dev, host = make_fleet(cuda, kind, n), make_fleet(cuda, kind, n)
    w.setup(dev, host)
    out = torch.full((n * C.sizeof(DwaResult),), SENTINEL, dtype=torch.uint8, device="cuda")
    cand = [np.array([(0.2, 0.0, 0.0), (0.0, 0.0, 0.5)]) if i % 3 else np.zeros((0, 3)) for i in range(n)]
    left_out = 0
    active = None  # the set_active mask in force (it holds until the next set_active)
    for cycle in range(cycles):
        poses, vels = w.poses(cycle), w.vels()
        w.feed(dev, host, cycle)
        op = cycle % 6
        if op == 1:
            for f in (dev, host):
                f.set_plans(poses, w.plans(poses))
        if op in (2, 4):
            active = np.array([(i + cycle) % 3 != 0 for i in range(n)])
            for f in (dev, host):
                f.set_active(active)
        if op == 3:
            assert [c.tobytes() for c in dev.check_trajectories(poses, vels, cand)] == \
                [c.tobytes() for c in host.check_trajectories(poses, vels, cand)]
        if op == 5:
            for f in (dev, host):
                f.reset_oscillation()
                f.set_active(None)
            active = None
            if kind == "raw":
                for f in (dev, host):
                    f.set_maps(np.stack([np.roll(r["raw"], cycle, axis=1) for r in w.robots]),
                               np.array([r["origin"] for r in w.robots]))
        if op == 0 and cycle:  # a host step on both
            assert dev.step(poses, vels) == host.step(poses, vels), f"cycle {cycle}: host steps differ"
            assert_twins(dev, host, kind, f"cycle {cycle} (host step)")
            continue
        out.fill_(SENTINEL)
        step_pair(dev, host, poses, vels, f"cycle {cycle}", active=active, out=out)
        after = out.cpu().numpy().reshape(n, -1)
        if active is not None:
            assert (after[~active] == SENTINEL).all(), f"cycle {cycle}: a left-out robot's record changed"
            assert not (after[active] == SENTINEL).all(axis=1).any()
            left_out += int((~active).sum())
        assert_twins(dev, host, kind, f"cycle {cycle}", state=op in (2, 3, 4))
    assert left_out > 0


def test_refusals_leave_the_fleet_as_it_was(cuda):
    lib = cuda.lib
    n = 6
    w = World("sensing", n, seed=5)
    dev, host = make_fleet(cuda, "sensing", n), make_fleet(cuda, "sensing", n)
    w.setup(dev, host)
    tp = cuda.fleet(n, 40, 40, RES, sc.PENTAGON, trajectory_planner={})
    no_dwa = make_fleet(cuda, "raw", n, use_dwa=0)
    wide = make_fleet(cuda, "raw", n, vth_samples=700)
    P = torch.zeros((n, 3), dtype=torch.float64, device="cuda")
    V = torch.zeros((n, 3), dtype=torch.float64, device="cuda")
    R = torch.zeros(n * C.sizeof(DwaResult), dtype=torch.uint8, device="cuda")
    hp, hv, hr = np.zeros((n, 3)), np.zeros((n, 3)), (DwaResult * n)()
    ptr = lambda t: C.c_void_p(t.data_ptr())
    cases = [
        ("null handle", 2, lambda: lib.navgpu_fleet_step_device(None, ptr(P), ptr(V), ptr(R))),
        ("null poses", 2, lambda: lib.navgpu_fleet_step_device(dev.h, None, ptr(V), ptr(R))),
        ("null results", 2, lambda: lib.navgpu_fleet_step_device(dev.h, ptr(P), ptr(V), None)),
        ("host poses", 2, lambda: lib.navgpu_fleet_step_device(dev.h, C.c_void_p(hp.ctypes.data), ptr(V), ptr(R))),
        ("host vels", 2, lambda: lib.navgpu_fleet_step_device(dev.h, ptr(P), C.c_void_p(hv.ctypes.data), ptr(R))),
        ("host results", 2, lambda: lib.navgpu_fleet_step_device(dev.h, ptr(P), ptr(V), C.cast(hr, C.c_void_p))),
        ("TrajectoryPlanner fleet", 3, lambda: lib.navgpu_fleet_step_device(tp.h, ptr(P), ptr(V), ptr(R))),
        ("use_dwa = 0", 3, lambda: lib.navgpu_fleet_step_device(no_dwa.h, ptr(P), ptr(V), ptr(R))),
        ("more than 640 per-axis samples", 3, lambda: lib.navgpu_fleet_step_device(wide.h, ptr(P), ptr(V), ptr(R))),
    ]
    step_pair(dev, host, w.poses(0), w.vels(), "before")
    for cycle, (name, code, call) in enumerate(cases, start=1):
        rc = call()
        assert rc == code, f"{name}: {rc} ({lib.navgpu_last_error().decode()})"
        w.feed(dev, host, cycle)
        step_pair(dev, host, w.poses(cycle), w.vels(), f"after {name}")
        assert_twins(dev, host, "sensing", f"after {name}", state=cycle % 3 == 0)
    for bad in (dict(poses=P.float()), dict(poses=P[:-1]), dict(poses=P.cpu()), dict(vels=V.t()),
                dict(out=R[:-1])):
        args = dict(poses=P, vels=V, out=None)
        args.update(bad)
        with pytest.raises(ValueError):
            dev.step_device(args["poses"], args["vels"], out=args["out"])


@pytest.mark.parametrize("kind", ["raw", "sensing", "voxel"])
def test_steady_state_step_captures(cuda, kind):
    """Two device steps size every buffer; the third, enqueued under thread-local stream capture, must capture without
    a host wait, an allocation or a pageable copy.  The graph is discarded unlaunched, then the fleet is destroyed."""
    cu = C.CDLL("libcuda.so.1")
    n = 8
    w = World(kind, n, seed=7)
    dev, host = make_fleet(cuda, kind, n), make_fleet(cuda, kind, n)
    w.setup(dev, host)
    P = torch.from_numpy(w.poses(0)).cuda()
    V = torch.from_numpy(w.vels()).cuda()
    R = torch.zeros(n * C.sizeof(DwaResult), dtype=torch.uint8, device="cuda")
    for cycle in range(2):
        w.feed(dev, host, cycle)
        dev.step_device(P, V, out=R)
    torch.cuda.synchronize()
    stream = C.c_void_p(dev.stream())
    assert cu.cuStreamBeginCapture_v2(stream, 1) == 0  # CU_STREAM_CAPTURE_MODE_THREAD_LOCAL
    rc = cuda.lib.navgpu_fleet_step_device(dev.h, C.c_void_p(P.data_ptr()), C.c_void_p(V.data_ptr()),
                                           C.c_void_p(R.data_ptr()))
    msg = cuda.lib.navgpu_last_error().decode()
    graph = C.c_void_p()
    end = cu.cuStreamEndCapture(stream, C.byref(graph))
    assert rc == 0, msg
    assert end == 0 and graph.value
    assert cu.cuGraphDestroy(graph) == 0
    del dev


def test_cuda_and_numpy_cos_sin(record_property):
    """A sensing fleet's footprint transform takes cos / sin of the yaw from CUDA's sincos on a device step and from
    the host libm on a host step.  Counts how often CUDA's and numpy's values differ over 10^6 random yaws; they stay
    within two ulp."""
    yaw = np.random.default_rng(11).uniform(-np.pi, np.pi, 1_000_000)
    t = torch.from_numpy(yaw).cuda()
    total = 0
    for name, dev_f, np_f in (("cos", torch.cos, np.cos), ("sin", torch.sin, np.sin)):
        d, h = dev_f(t).cpu().numpy(), np_f(yaw)
        differ = int((d != h).sum())
        record_property(f"{name}_differ", differ)
        total += differ
        ulps = np.abs(d.view(np.int64) - h.view(np.int64))
        assert ulps.max() <= 2, name
    record_property("yaws", len(yaw))
    print(f"cos / sin: {total} of {2 * len(yaw)} values differ between CUDA and numpy")


def test_c5_full_fleet_device_step(cuda, port):
    """4096 robots with bench.py's C5 inputs: a device step equals a host step on a twin, and every 64th robot is
    replayed through the CPU checker."""
    cfg = dict(vx_samples=20, vy_samples=1, vth_samples=20, max_vel_y=0.0, min_vel_y=0.0)
    n = 4096
    robots = [synth.fleet_robot(i) for i in range(n)]
    dev, host = (cuda.fleet(n, 120, 120, RES, sc.PENTAGON, 0.55, 10.0, **cfg) for _ in range(2))
    poses = np.array([r["pose"] for r in robots])
    vels = np.array([r["vel"] for r in robots])
    for f in (dev, host):
        f.set_maps(np.stack([r["raw"] for r in robots]), np.array([r["origin"] for r in robots]))
        f.set_plans(poses, [r["plan"] for r in robots])
    _, out = step_pair(dev, host, poses, vels, "cycle 0")
    valid = exact = 0
    for i in range(0, n, 64):
        cm = port.costmap(120, 120, RES, *robots[i]["origin"])
        s = cm.add_grid_layer(0)
        cm.add_inflation_layer(0.55, 10.0)
        cm.set_footprint(sc.PENTAGON)
        cm.set_grid_layer(s, robots[i]["raw"])
        cm.update_map(0, 0, 0)
        assert np.array_equal(dev.costmap(i), cm.get()), f"robot {i}"
        d = port.dwa(120, 120, RES, **cfg)
        d.set_costmap(cm.get(), *robots[i]["origin"])
        d.set_plan(poses[i], robots[i]["plan"])
        e = d.find_best_path(poses[i], vels[i], sc.PENTAGON)
        g = out[i]
        assert (g["best_index"], g["n_samples"], g["n_scored"]) == (e["best_index"], e["n_samples"], e["n_scored"])
        assert dev.oscillation_mask(i) == d.oscillation_mask()
        if e["ok"]:
            assert np.isclose(g["cost"], e["cost"], rtol=RTOL, atol=0)
            assert (g["xv"], g["yv"], g["thetav"]) == (e["xv"], e["yv"], e["thetav"])
            exact += g["cost"] == e["cost"]
            valid += 1
    assert valid >= 32 and exact >= 0.99 * valid
    step_pair(dev, host, poses, vels, "cycle 1")
