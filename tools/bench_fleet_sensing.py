"""Sensing fleet throughput (navgpu_fleet_create_sensing): 4096 robots, each a rolling 120 x 120 local costmap at 0.05 m
[ObstacleLayer, InflationLayer] fed one fresh 360-beam LaserScan per step, then DWAPlanner with 20 x 1 x 20 samples and the
pentagon footprint.  Prints one JSON line:
  sensing_step_ms   host wall time of set_scans + step (the step ends in a device synchronise), mean over the timed steps
  set_scans_ms, step_ms   the same split: host wall time of the set call alone and of the step alone
  project_ms, costmap_ms   device time (CUDA events) of the scan projection (k_project_scans) and of k_fleet_costmap,
                    means over the timed steps, and their sum
  raw_step_ms       the raw-map fleet (config C5, navgpu_fleet_create + set_maps) step in the same process, for comparison
  gpu, power_limit  the card and its power limit, read in the same run
--check N replays N evenly spaced robots through the CPU checker (rolling LayeredCostmap with the exact windowed
inflation, then DWAPlanner) over every step and reports how many agree (costmaps bit for bit, results as in
the tests).  LaserScan projection may differ from glibc's in the last float bit (tests/test_gpu_scan_ingest.py), so a
disagreement is reported, not fatal.

The scans of K distinct cycles are ray-cast once before timing (ray casting 4096 x 360 beams in numpy takes seconds);
step k uses cycle k mod K, so every step still uploads and projects a new scan per robot.

--voxel benches the same fleet with map_type: voxel -- every robot's costmap is [VoxelLayer, InflationLayer]
(cfg/VoxelPlugin.cfg's defaults: 10 voxels of 0.2 m from z = 0) fed one fresh 3-D cloud per step instead of the scan
(synth.fleet_cloud_3d: 6 rows of 180 beams through a world with heights, 1080 points per robot) -- and adds
"voxel": true to the JSON line.  costmap_ms is then the device time of k_fleet_costmap_voxel.

--ingest picks how the scans reach the fleet (the JSON line's "ingest"):
  list    Fleet.set_scans with one scan dict per robot (navgpu_fleet_set_scans), the default
  host    Fleet.set_scan_batch with dense numpy arrays, one per sensor (navgpu_fleet_set_scan_batch)
  device  the same arrays as CUDA torch tensors, as a GPU simulator holds them (navgpu_fleet_set_scan_batch_device);
          they are uploaded before timing, and set_scans_ms is then the enqueue alone: the kernel (project_ms) runs
          on the fleet's stream and its time is part of step_ms
The batch modes ray-cast every robot's LaserScan at one sensor-frame angle_min (synth.fleet_scan_batch; the clouds of
--voxel are the same either way); project_ms is the device time of k_fleet_scan_batch there."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

PENTAGON = [(-0.325, -0.325), (-0.325, 0.325), (0.325, 0.325), (0.46, 0.0), (0.325, -0.325)]
CFG = dict(vx_samples=20, vy_samples=1, vth_samples=20, max_vel_y=0.0, min_vel_y=0.0)
VOXEL = dict(origin_z=0.0, z_resolution=0.2, z_voxels=10, unknown_threshold=15, mark_threshold=0)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception as e:  # the numbers are still reported, without the card's limit
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--robots", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--cycles", type=int, default=4, help="distinct scan cycles ray-cast before timing")
    ap.add_argument("--check", type=int, default=0)
    ap.add_argument("--voxel", action="store_true", help="[VoxelLayer, InflationLayer] fed 3-D clouds")
    ap.add_argument("--ingest", choices=("list", "host", "device"), default="list")
    args = ap.parse_args()
    if args.steps < 1 or args.robots < 1 or args.cycles < 1:
        ap.error("--steps, --robots and --cycles must be positive")

    import navigation_b200
    from navigation_b200 import build, synth
    build.build()
    cuda = navigation_b200.load()
    if cuda.device_count() == 0:
        sys.exit("bench_fleet_sensing needs a CUDA device (libnavgpu has no CPU path)")
    n, sx, res = args.robots, 120, 0.05

    t0 = time.perf_counter()
    if args.voxel:
        robots = [synth.fleet_voxel_robot(i, n=sx, res=res) for i in range(n)]
    else:
        robots = [synth.fleet_sensing_robot(i, n=sx, res=res) for i in range(n)]
    if args.ingest == "list":
        one = synth.fleet_cloud_3d if args.voxel else synth.fleet_scan
        scans = [[[one(r, c)] for r in robots] for c in range(args.cycles)]
        inputs = scans
    else:
        batch = synth.fleet_cloud_3d_batch if args.voxel else synth.fleet_scan_batch
        inputs = [[batch(robots, c)] for c in range(args.cycles)]
        scans = None  # per-robot dicts only for the robots --check replays (synth.batch_scans)
        if args.ingest == "device":
            import torch
            gpu = torch.device("cuda", 0)
            inputs = [[{k: torch.from_numpy(v).to(gpu) if isinstance(v, np.ndarray) else v for k, v in s.items()}
                       for s in srcs] for srcs in inputs]
            torch.cuda.synchronize()
    poses = [np.ascontiguousarray([r["poses"][c] for r in robots]) for c in range(args.cycles)]
    vels = np.ascontiguousarray([r["vel"] for r in robots])
    prep_s = time.perf_counter() - t0

    fleet = cuda.fleet_sensing(n, sx, sx, res, PENTAGON, voxel=VOXEL if args.voxel else None, **CFG)
    fleet.set_plans(poses[0], [r["plan"] for r in robots])
    sample = list(range(0, n, max(1, n // args.check)))[:args.check] if args.check else []
    history = {i: [] for i in sample}
    set_call = fleet.set_scans if args.ingest == "list" else fleet.set_scan_batch
    wall, set_ms, step_ms, proj, dev = [], [], [], [], []
    for k in range(args.warmup + args.steps):
        c = k % args.cycles
        t = time.perf_counter()
        set_call(inputs[c])
        t1 = time.perf_counter()
        res_arr = fleet.step_raw(poses[c], vels)
        t2 = time.perf_counter()
        dt = t2 - t
        for i in sample:
            g = res_arr[i]
            history[i].append((g.cost, g.xv, g.yv, g.thetav, g.best_index, g.n_samples, g.n_scored, fleet.oscillation_mask(i)))
        if k >= args.warmup:
            wall.append(dt * 1e3)
            set_ms.append((t1 - t) * 1e3)
            step_ms.append((t2 - t1) * 1e3)
            p_ms, c_ms = fleet.last_timing()
            proj.append(p_ms)
            dev.append(c_ms)
    valid = sum(1 for i in range(n) if res_arr[i].cost >= 0)

    # the raw-map fleet (config C5) in the same process
    raw_robots = [synth.fleet_robot(i) for i in range(n)]
    raw = cuda.fleet(n, sx, sx, res, PENTAGON, 0.55, 10.0, **CFG)
    raw.set_maps(np.stack([r["raw"] for r in raw_robots]), np.array([r["origin"] for r in raw_robots]))
    rposes = np.ascontiguousarray([r["pose"] for r in raw_robots])
    rvels = np.ascontiguousarray([r["vel"] for r in raw_robots])
    raw.set_plans(rposes, [r["plan"] for r in raw_robots])
    raw_ms = []
    for k in range(args.warmup + args.steps):
        t = time.perf_counter()
        raw.step_raw(rposes, rvels)
        if k >= args.warmup:
            raw_ms.append((time.perf_counter() - t) * 1e3)

    checked = agree = 0
    if sample:
        from oracle import pyoracle
        port = pyoracle.load("port")
        final = {i: fleet.costmap(i) for i in sample}
        if scans is None:  # the batch modes: robot i's scan of cycle c is its row of the batch
            to_np = lambda v: v.cpu().numpy() if hasattr(v, "cpu") else v  # noqa: E731
            scans = [synth.batch_scans([{k: to_np(v) for k, v in s.items()} for s in srcs], n) for srcs in inputs]
        for i in sample:
            cm = port.costmap(sx, sx, res, 0.0, 0.0, rolling=True)
            o = cm.add_voxel_layer(1, True, 2.0, **VOXEL) if args.voxel else cm.add_obstacle_layer(1, True, 2.0)
            il = cm.add_inflation_layer(0.55, 10.0)
            cm.set_inflation_variant(il, 4)  # exact windowed nearest-seed inflation (inflation mode 0)
            cm.set_footprint(PENTAGON)
            d = port.dwa(sx, sx, res, **CFG)
            ok = True
            for k in range(args.warmup + args.steps):
                c = k % args.cycles
                org, pts = port.project_scan(scans[c][i][0])
                s_ = scans[c][i][0]
                cm.set_observations(o, [dict(origin=org, points=pts, obstacle_range=s_["obstacle_range"],
                                             raytrace_range=s_["raytrace_range"])])
                cm.update_map(*poses[c][i])
                d.set_costmap(cm.get(), *cm.origin())
                if k == 0:
                    d.set_plan(poses[0][i], robots[i]["plan"])
                e = d.find_best_path(poses[c][i], vels[i], PENTAGON)
                got = history[i][k]
                want = (e["cost"], e["xv"], e["yv"], e["thetav"], e["best_index"], e["n_samples"], e["n_scored"],
                        d.oscillation_mask())
                same = got[4:] == want[4:] and (got[0] < 0) == (want[0] < 0) and \
                    (want[0] < 0 or (np.isclose(got[0], want[0], rtol=1e-5, atol=0) and got[1:4] == want[1:4]))
                ok = ok and same
            ok = ok and np.array_equal(final[i], cm.get())
            checked += 1
            agree += ok

    name, limit = gpu_info()
    out = dict(robots=n, map=f"{sx}x{sx}@{res}", samples="20x1x20", steps=args.steps, warmup=args.warmup,
               scan_cycles=args.cycles, beams=360, ingest=args.ingest,
               sensing_step_ms=float(np.mean(wall)), sensing_step_ms_min=float(np.min(wall)),
               set_scans_ms=float(np.mean(set_ms)), step_ms=float(np.mean(step_ms)),
               project_ms=float(np.mean(proj)), costmap_ms=float(np.mean(dev)),
               project_plus_costmap_ms=float(np.mean(np.add(proj, dev))),
               raw_step_ms=float(np.mean(raw_ms)), raw_step_ms_min=float(np.min(raw_ms)),
               valid_robots=valid, checked=checked, checked_agree=agree, input_prep_s=round(prep_s, 1),
               gpu=name, power_limit=limit)
    if args.voxel:
        out.update(voxel=True, beams=len(synth.VOXEL_ELEVATIONS) * 180)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
