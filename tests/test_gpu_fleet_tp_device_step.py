"""Device-resident TrajectoryPlanner fleet steps (navgpu_fleet_step_tp_device, Fleet.step_tp_device): poses and velocities
in device memory, the enumeration, scoring and selection on the fleet's stream.

1. Raw-map, 2-D sensing and voxel fleets beside host-stepped twins over multi-cycle runs of fleet_tp_scenarios' robots
   (sensing fleets fed through set_scan_batch_device), holonomic and differential-drive configurations, heading scoring
   on and off: every cycle results (flags and n_points included), master grids, both distance grids, layers, voxel
   columns, windows and origins are bit-equal, and the robots take every selection branch between them.  Three robots
   of the raw-map runs are replayed through the CPU checker's TrajectoryPlanner.
2. glibc_hypot on the device equals glibc_hypot on the host over 2 x 10^6 pairs (a test kernel built here with nvcc).
3. Host calls between device steps: host steps, set_plans, set_active with a changing subset, check_trajectories,
   get_geometry and set_maps; left-out robots keep a sentinel byte pattern in their result records.  New plans
   followed by a host step and then a device step, with heading scoring and with the simple attractor (both read
   each robot's plan or goal in the scoring records).
4. Refusals leave the fleet bit-identical to its twin at the next step.
5. A steady-state device step captures under cuStreamBeginCapture in thread-local mode; the graph is discarded unlaunched.
6. 4096 robots of tools/bench_fleet_tp.py's inputs: the device step equals a host step on a twin, and every 64th robot
   is replayed through the checker."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import fleet_tp_scenarios as ft
import scenarios as sc
from navigation_b200 import synth
from navigation_b200.api import TpResult

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL = 1e-5
CONFIGS = [dict(), dict(holonomic_robot=0, dwa=0), dict(heading_scoring=1)]
CFG_IDS = ["defaults", "diff_drive_no_dwa", "heading_scoring"]
ALL_BRANCHES = {"forward", "rotate", "strafe", "escape", "leave_escape", "stuck", "stuck_reset"}
CYCLES = 9
SENTINEL = 0xA5
REC = C.sizeof(TpResult)


def make_fleet(api, kind, n, cfg):
    if kind == "raw":
        return api.fleet(n, ft.N, ft.N, ft.RES, sc.PENTAGON, 0.55, 10.0, trajectory_planner=cfg)
    return api.fleet_sensing(n, ft.N, ft.N, ft.RES, sc.PENTAGON, voxel={} if kind == "voxel" else None,
                             trajectory_planner=cfg)


def scan_batch(robots, cycle, voxel):
    """fleet_tp_scenarios.scenario_sources as one batch source: every robot's scan of its world from its current pose."""
    ds = []
    for r in robots:
        w = r.world_at(cycle)
        ds.append(dict(world=w, origin=r.world_origin, resolution=ft.RES, poses=r.pose[None, :], seed=r.rid,
                       top=np.where(w, np.float32(ft.WALL_TOP), np.float32(-np.inf)), bottom=np.zeros(w.shape, np.float32)))
    return [synth.fleet_cloud_3d_batch(ds, cycle) if voxel else synth.fleet_scan_batch(ds, 0)]


def on_device(sources):
    out = []
    for s in sources:
        d = dict(s)
        for k in ("ranges", "points", "sensor_to_global"):
            if k in s:
                d[k] = torch.from_numpy(s[k]).cuda()
        out.append(d)
    return out


def feed(kind, dev, host, robots, cycle):
    if kind == "raw":
        if cycle in (0, 3, 6):  # robot 6's box opens at 3, robot 5's slot closes at 6
            for f in (dev, host):
                f.set_maps(*ft.scenario_raw(robots, cycle))
        return
    src = scan_batch(robots, cycle, kind == "voxel")
    dev.set_scan_batch(on_device(src))
    host.set_scan_batch(src)


def dev_step(fleet, poses, vels, out=None):
    r = fleet.step_tp_device(torch.from_numpy(np.ascontiguousarray(poses)).cuda(),
                             torch.from_numpy(np.ascontiguousarray(vels)).cuda(), out=out)
    torch.cuda.synchronize()
    return r


def records(fleet, raw):
    """Result records [n][40 bytes] of a device step (its `records`) or of a host step (the ctypes array)."""
    if isinstance(raw, dict):
        return raw["records"].cpu().numpy().reshape(fleet.n, REC)
    return np.frombuffer(C.string_at(C.addressof(raw), fleet.n * REC), np.uint8).reshape(fleet.n, REC)


def as_dicts(fleet, raw):
    r = raw["records"].cpu().numpy()
    f64, i32 = r.view(np.float64).reshape(fleet.n, -1), r.view(np.int32).reshape(fleet.n, -1)
    return [dict(cost=f64[i, 0], xv=f64[i, 1], yv=f64[i, 2], thetav=f64[i, 3], n_points=int(i32[i, 8]),
                 flags=int(i32[i, 9])) for i in range(fleet.n)]


def step_pair(dev, host, poses, vels, where, active=None, out=None):
    """A device step and a host step on the twin: their records are bit-equal (active robots only)."""
    d = dev_step(dev, poses, vels, out)
    h = host.step_raw(np.ascontiguousarray(poses, dtype=np.float64), np.ascontiguousarray(vels, dtype=np.float64))
    got, exp = records(dev, d), records(host, h)
    rows = np.ones(dev.n, bool) if active is None else np.asarray(active, bool)
    bad = [i for i in range(dev.n) if rows[i] and not np.array_equal(got[i], exp[i])]
    assert not bad, f"{where}: results of robots {bad} differ"
    return d


def assert_twins(dev, host, kind, where, state=True):
    for i in range(dev.n):
        w = f"{where} robot {i}"
        assert np.array_equal(dev.costmap(i), host.costmap(i)), f"{w}: master grid differs"
        for k in (0, 1):
            assert np.array_equal(dev.tp_grid(i, k), host.tp_grid(i, k)), f"{w}: distance grid {k} differs"
        if kind != "raw":
            assert np.array_equal(dev.layer(i), host.layer(i)), f"{w}: obstacle layer differs"
        if kind == "voxel":
            assert np.array_equal(dev.voxels(i), host.voxels(i)), f"{w}: voxel columns differ"
        if state and kind != "raw":  # (brings the device state back: the next device step uploads it again)
            assert dev.geometry(i) == host.geometry(i), w


@pytest.mark.parametrize("cfg", CONFIGS, ids=CFG_IDS)
@pytest.mark.parametrize("kind", ["raw", "sensing", "voxel"])
def test_device_steps_match_host_twin(cuda, port, kind, cfg):
    robots = ft.scenario(16)
    n = len(robots)
    dev, host = make_fleet(cuda, kind, n, cfg), make_fleet(cuda, kind, n, cfg)
    checked = (4, 5, 6)
    checkers = {i: port.trajectory_planner(ft.N, ft.N, ft.RES, sc.PENTAGON, **cfg) for i in checked}
    traces = [[] for _ in robots]
    for cycle in range(CYCLES):
        feed(kind, dev, host, robots, cycle)
        if cycle in (0, 3):
            plans = [r.plan_at(cycle) for r in robots]
            for f in (dev, host):
                f.set_plans(np.array([r.pose for r in robots]), plans)
            for i, ck in checkers.items():
                if len(plans[i]):
                    ck.update_plan(plans[i])
        poses, vels = np.array([r.pose for r in robots]), np.array([r.vel for r in robots])
        out = as_dicts(dev, step_pair(dev, host, poses, vels, f"{kind} cycle {cycle}"))
        assert_twins(dev, host, kind, f"{kind} cycle {cycle}", state=cycle % 3 == 2)
        if kind == "raw":
            for i, ck in checkers.items():
                ck.set_costmap(dev.costmap(i), *robots[i].map_origin)
                e = ck.find_best_path(robots[i].pose, robots[i].vel)
                g = out[i]
                assert (g["xv"], g["yv"], g["thetav"], g["flags"], g["n_points"]) == \
                    (e["xv"], e["yv"], e["thetav"], e["flags"], len(e["points"])), f"cycle {cycle} robot {i}: {g} vs {e}"
                assert np.isclose(g["cost"], e["cost"], rtol=RTOL, atol=0), f"cycle {cycle} robot {i}"
        for i, g in enumerate(out):
            traces[i].append((g, robots[i].pose.copy()))
        ft.advance(robots, out)
    seen = set().union(*(ft.branches(t, cfg) for t in traces))
    if kind == "raw":
        want = ALL_BRANCHES if cfg.get("holonomic_robot", 1) else ALL_BRANCHES - {"strafe"}
        assert want <= seen, f"branches not taken: {want - seen}"
    else:
        assert {"forward", "rotate"} <= seen, seen


@pytest.fixture(scope="module")
def hypot_kernel(tmp_path_factory):
    """glibc_hypot on the device and on the host of one library, built here with the project's nvcc flags."""
    from navigation_b200 import build as nb
    d = tmp_path_factory.mktemp("glibc_hypot")
    src = d / "hypot_test.cu"
    src.write_text(f'#include "{ROOT}/navigation_b200/csrc/glibc_hypot.cuh"\n' + r'''
__global__ void k_hypot(const double* x, const double* y, double* out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = glibc_hypot(x[i], y[i]);
}
extern "C" int hypot_device(const double* x, const double* y, double* out, int n) {
  k_hypot<<<(n + 255) / 256, 256>>>(x, y, out, n);
  return (int)cudaDeviceSynchronize();
}
extern "C" void hypot_host(const double* x, const double* y, double* out, int n) {
  for (int i = 0; i < n; ++i) out[i] = glibc_hypot(x[i], y[i]);
}
''')
    lib = d / "libhypot_test.so"
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    flags = [f for f in nb.NVCC_FLAGS if f != "-lineinfo"]
    subprocess.check_call([nvcc] + flags + ["-o", str(lib), str(src)])
    return C.CDLL(str(lib))


def hypot_pairs(n, seed=5):
    """Random magnitudes over the whole exponent range, the planner's range, integers, equal arguments, zeros,
    subnormals, values around the cutoffs, and non-finite ones."""
    rng = np.random.default_rng(seed)
    q = n // 6
    sgn = lambda k: rng.choice([-1.0, 1.0], k)
    wide = lambda k: np.ldexp(1.0 + rng.random(k), rng.integers(-1074, 1024, k)) * sgn(k)
    planner = lambda k: np.exp(rng.uniform(np.log(1e-9), np.log(2e4), k)) * sgn(k)
    x = np.concatenate([wide(q), planner(q), rng.integers(0, 100000, q).astype(np.float64), wide(q), wide(q),
                        np.ldexp(1.0 + rng.random(q), rng.choice([511, 510, -459, -460, -511], q))])
    y = np.concatenate([wide(q), planner(q), rng.integers(0, 100000, q).astype(np.float64), -x[3 * q:4 * q],
                        np.where(rng.random(q) < 0.5, 0.0, np.ldexp(rng.random(q), -1022)),
                        x[5 * q:] * np.ldexp(1.0 + rng.random(q), -rng.integers(0, 60, q))])
    special = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1.0, 5e-324, 1.7976931348623157e308])
    sx, sy = np.meshgrid(special, special)
    return np.concatenate([x, sx.ravel()]), np.concatenate([y, sy.ravel()])


def test_glibc_hypot_device_matches_host(hypot_kernel):
    x, y = hypot_pairs(2_000_000)
    n = len(x)
    host = np.empty(n)
    f64 = C.POINTER(C.c_double)
    hypot_kernel.hypot_host(x.ctypes.data_as(f64), y.ctypes.data_as(f64), host.ctypes.data_as(f64), n)
    X, Y = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    D = torch.empty(n, dtype=torch.float64, device="cuda")
    assert hypot_kernel.hypot_device(C.c_void_p(X.data_ptr()), C.c_void_p(Y.data_ptr()), C.c_void_p(D.data_ptr()), n) == 0
    dev = D.cpu().numpy()
    nan = np.isnan(host)
    assert np.array_equal(nan, np.isnan(dev))
    differ = np.flatnonzero(host[~nan].view(np.int64) != dev[~nan].view(np.int64))
    assert differ.size == 0, f"{differ.size} of {n} pairs differ, e.g. {x[~nan][differ[:3]]} {y[~nan][differ[:3]]}"


@pytest.mark.parametrize("kind", ["raw", "sensing"])
def test_mixed_host_calls(cuda, kind):
    robots = ft.scenario(12)
    n = len(robots)
    dev, host = make_fleet(cuda, kind, n, {}), make_fleet(cuda, kind, n, {})
    out = torch.full((n * REC,), SENTINEL, dtype=torch.uint8, device="cuda")
    cand = [np.array([(0.2, 0.0, 0.0), (0.0, 0.0, 0.5)]) if i % 3 else np.zeros((0, 3)) for i in range(n)]
    active, left_out, cycles = None, 0, 12
    for cycle in range(cycles):
        feed(kind, dev, host, robots, cycle)
        poses, vels = np.array([r.pose for r in robots]), np.array([r.vel for r in robots])
        op = cycle % 6
        if op == 1 or cycle == 0:
            for f in (dev, host):
                f.set_plans(poses, [r.plan_at(cycle) for r in robots])
        if op in (2, 4):
            active = np.array([(i + cycle) % 3 != 0 for i in range(n)])
            for f in (dev, host):
                f.set_active(active)
        if op == 3:
            assert [c.tobytes() for c in dev.check_trajectories(poses, vels, cand)] == \
                [c.tobytes() for c in host.check_trajectories(poses, vels, cand)]
        if op == 5:
            for f in (dev, host):
                f.set_active(None)
            active = None
            if kind == "raw":
                maps, origins = ft.scenario_raw(robots, cycle)
                for f in (dev, host):
                    f.set_maps(np.roll(maps, cycle, axis=2), origins)
        if op == 0 and cycle:  # a host step on both
            h = [f.step(poses, vels) for f in (dev, host)]
            assert h[0] == h[1], f"cycle {cycle}: host steps differ"
            assert_twins(dev, host, kind, f"cycle {cycle} (host step)")
            ft.advance(robots, h[1])
            continue
        out.fill_(SENTINEL)
        r = step_pair(dev, host, poses, vels, f"cycle {cycle}", active=active, out=out)
        after = out.cpu().numpy().reshape(n, REC)
        if active is not None:
            assert (after[~active] == SENTINEL).all(), f"cycle {cycle}: a left-out robot's record changed"
            assert not (after[active] == SENTINEL).all(axis=1).any()
            left_out += int((~active).sum())
        assert_twins(dev, host, kind, f"cycle {cycle}", state=op in (2, 3, 4))
        res = as_dicts(dev, r)
        ft.advance(robots, [g if active is None or active[i] else dict(g, cost=-1.0) for i, g in enumerate(res)])
    assert left_out > 0


@pytest.mark.parametrize("cfg", [dict(heading_scoring=1), dict(simple_attractor=1)], ids=["heading_scoring",
                                                                                      "simple_attractor"])
def test_new_plans_then_host_step_then_device_step(cuda, cfg):
    """set_plans, a host step, then a device step: the device step scores against the new plans (goals, raw plans)."""
    robots = ft.scenario(12)
    n = len(robots)
    dev, host = make_fleet(cuda, "raw", n, cfg), make_fleet(cuda, "raw", n, cfg)
    feed("raw", dev, host, robots, 0)
    poses, vels = np.array([r.pose for r in robots]), np.array([r.vel for r in robots])
    plans = [r.plan for r in robots]
    for f in (dev, host):
        f.set_plans(poses, plans)
    for cycle in range(2):
        last = records(dev, step_pair(dev, host, poses, vels, f"first plans, cycle {cycle}")).copy()
    changed = 0
    for k, shift in enumerate((0.6, -0.9)):
        # every robot's plan moves and gets shorter: new goals, raw-plan offsets and lengths
        new = [p[: max(len(p) - 7 * (k + 1), 2)] + np.array([shift, 0.5 * shift]) if len(p) else p for p in plans]
        for f in (dev, host):
            f.set_plans(poses, new)
        h = [f.step_raw(poses, vels) for f in (dev, host)]  # host steps upload the new plans on both fleets
        assert np.array_equal(records(dev, h[0]), records(host, h[1])), f"plans {k}: host steps differ"
        got = records(dev, step_pair(dev, host, poses, vels, f"plans {k}: device step after a host step"))
        for i in range(n):
            for j in (0, 1):
                assert np.array_equal(dev.tp_grid(i, j), host.tp_grid(i, j)), f"plans {k} robot {i}: grid {j}"
        changed += int((got != last).any(axis=1).sum())
        last = got.copy()
    assert changed > 0  # the new plans change what the robots choose


def test_refusals_leave_the_fleet_as_it_was(cuda):
    lib = cuda.lib
    robots = ft.scenario(12)
    n = len(robots)
    dev, host = make_fleet(cuda, "sensing", n, {}), make_fleet(cuda, "sensing", n, {})
    dwa = cuda.fleet(n, 40, 40, ft.RES, sc.PENTAGON)
    wide = make_fleet(cuda, "raw", n, dict(vx_samples=60, vtheta_samples=70))  # 60 x 70 + 70 + 7 samples per robot
    P = torch.zeros((n, 3), dtype=torch.float64, device="cuda")
    V = torch.zeros((n, 3), dtype=torch.float64, device="cuda")
    R = torch.zeros(n * REC, dtype=torch.uint8, device="cuda")
    hp, hv, hr = np.zeros((n, 3)), np.zeros((n, 3)), (TpResult * n)()
    ptr = lambda t: C.c_void_p(t.data_ptr())
    cases = [
        ("null handle", 2, lambda: lib.navgpu_fleet_step_tp_device(None, ptr(P), ptr(V), ptr(R))),
        ("null poses", 2, lambda: lib.navgpu_fleet_step_tp_device(dev.h, None, ptr(V), ptr(R))),
        ("null vels", 2, lambda: lib.navgpu_fleet_step_tp_device(dev.h, ptr(P), None, ptr(R))),
        ("null results", 2, lambda: lib.navgpu_fleet_step_tp_device(dev.h, ptr(P), ptr(V), None)),
        ("host poses", 2, lambda: lib.navgpu_fleet_step_tp_device(dev.h, C.c_void_p(hp.ctypes.data), ptr(V), ptr(R))),
        ("host vels", 2, lambda: lib.navgpu_fleet_step_tp_device(dev.h, ptr(P), C.c_void_p(hv.ctypes.data), ptr(R))),
        ("host results", 2, lambda: lib.navgpu_fleet_step_tp_device(dev.h, ptr(P), ptr(V), C.cast(hr, C.c_void_p))),
        ("DWAPlanner fleet", 2, lambda: lib.navgpu_fleet_step_tp_device(dwa.h, ptr(P), ptr(V), ptr(R))),
        ("slot of 4277 samples", 3, lambda: lib.navgpu_fleet_step_tp_device(wide.h, ptr(P), ptr(V), ptr(R))),
        ("the DWA device step", 3, lambda: lib.navgpu_fleet_step_device(dev.h, ptr(P), ptr(V), ptr(R))),
    ]
    feed("sensing", dev, host, robots, 0)
    for f in (dev, host):
        f.set_plans(np.array([r.pose for r in robots]), [r.plan for r in robots])
    step_pair(dev, host, np.array([r.pose for r in robots]), np.array([r.vel for r in robots]), "before")
    for cycle, (name, code, call) in enumerate(cases, start=1):
        rc = call()
        assert rc == code, f"{name}: {rc} ({lib.navgpu_last_error().decode()})"
        feed("sensing", dev, host, robots, cycle)
        r = step_pair(dev, host, np.array([r.pose for r in robots]), np.array([r.vel for r in robots]), f"after {name}")
        assert_twins(dev, host, "sensing", f"after {name}", state=cycle % 3 == 0)
        ft.advance(robots, as_dicts(dev, r))
    assert "not a TrajectoryPlanner fleet" in (cases[7][2](), lib.navgpu_last_error().decode())[1]
    assert "navgpu_fleet_step_tp_device" in (cases[9][2](), lib.navgpu_last_error().decode())[1]
    for bad in (dict(poses=P.float()), dict(poses=P[:-1]), dict(poses=P.cpu()), dict(vels=V.t()), dict(out=R[:-1])):
        args = dict(poses=P, vels=V, out=None)
        args.update(bad)
        with pytest.raises(ValueError):
            dev.step_tp_device(args["poses"], args["vels"], out=args["out"])


@pytest.mark.parametrize("kind", ["raw", "sensing", "voxel"])
def test_steady_state_step_captures(cuda, kind):
    """Two device steps size every buffer; the third, enqueued under thread-local stream capture, must capture without
    a host wait, an allocation or a pageable copy.  The graph is discarded unlaunched, then the fleet is destroyed."""
    cu = C.CDLL("libcuda.so.1")
    robots = ft.scenario(12)
    n = len(robots)
    dev, host = make_fleet(cuda, kind, n, {}), make_fleet(cuda, kind, n, {})
    for f in (dev, host):
        f.set_plans(np.array([r.pose for r in robots]), [r.plan for r in robots])
    P = torch.from_numpy(np.array([r.pose for r in robots])).cuda()
    V = torch.from_numpy(np.array([r.vel for r in robots])).cuda()
    R = torch.zeros(n * REC, dtype=torch.uint8, device="cuda")
    for cycle in range(2):
        feed(kind, dev, host, robots, cycle)
        dev.step_tp_device(P, V, out=R)
    torch.cuda.synchronize()
    stream = C.c_void_p(dev.stream())
    assert cu.cuStreamBeginCapture_v2(stream, 1) == 0  # CU_STREAM_CAPTURE_MODE_THREAD_LOCAL
    rc = cuda.lib.navgpu_fleet_step_tp_device(dev.h, C.c_void_p(P.data_ptr()), C.c_void_p(V.data_ptr()),
                                              C.c_void_p(R.data_ptr()))
    msg = cuda.lib.navgpu_last_error().decode()
    graph = C.c_void_p()
    end = cu.cuStreamEndCapture(stream, C.byref(graph))
    assert rc == 0, msg
    assert end == 0 and graph.value
    assert cu.cuGraphDestroy(graph) == 0
    del dev


def test_full_size_device_step(cuda, port):
    """tools/bench_fleet_tp.py's inputs: 4096 robots of synth.fleet_robot(i), TrajectoryPlannerROS's defaults.  Two
    device steps equal host steps on a twin; every 64th robot of the first is replayed through the checker."""
    n = 4096
    robots = [synth.fleet_robot(i) for i in range(n)]
    dev, host = (cuda.fleet(n, 120, 120, 0.05, sc.PENTAGON, 0.55, 10.0, trajectory_planner={}) for _ in range(2))
    poses = np.array([r["pose"] for r in robots])
    vels = np.array([r["vel"] for r in robots])
    for f in (dev, host):
        f.set_maps(np.stack([r["raw"] for r in robots]), np.array([r["origin"] for r in robots]))
        f.set_plans(poses, [r["plan"] for r in robots])
    out = as_dicts(dev, step_pair(dev, host, poses, vels, "cycle 0"))
    exact = 0
    sample = range(0, n, 64)
    for i in sample:
        cm = port.costmap(120, 120, 0.05, *robots[i]["origin"])
        s = cm.add_grid_layer(0)
        cm.add_inflation_layer(0.55, 10.0)
        cm.set_footprint(sc.PENTAGON)
        cm.set_grid_layer(s, robots[i]["raw"])
        cm.update_map(0, 0, 0)
        grid = cm.get()
        assert np.array_equal(dev.costmap(i), grid), f"robot {i}: inflated local costmap differs"
        tp = port.trajectory_planner(120, 120, 0.05, sc.PENTAGON)
        tp.set_costmap(grid, *robots[i]["origin"])
        tp.update_plan(robots[i]["plan"])
        e = tp.find_best_path(poses[i], vels[i])
        g = out[i]
        assert (g["xv"], g["yv"], g["thetav"], g["flags"], g["n_points"]) == \
            (e["xv"], e["yv"], e["thetav"], e["flags"], len(e["points"])), f"robot {i}: {g} vs {e}"
        assert np.isclose(g["cost"], e["cost"], rtol=RTOL, atol=0), f"robot {i}"
        for k in (0, 1):
            assert np.array_equal(dev.tp_grid(i, k), tp.grid(k)), f"robot {i}: grid {k} differs"
        exact += g["cost"] == e["cost"]
    assert exact >= 0.99 * len(sample)
    step_pair(dev, host, poses + np.array([0.02, 0.0, 0.05]), vels, "cycle 1")
