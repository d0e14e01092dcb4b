"""Fleet of legacy TrajectoryPlanners (navgpu_fleet_use_trajectory_planner): 4096 robots of config C5's inputs
(synth.fleet_robot(i): 120 x 120 raw local maps at 0.05 m, inflated on the device), TrajectoryPlannerROS's defaults
(3 x 20 forward samples, holonomic, dwa) and the pentagon footprint.  Prints one JSON line:
  tp_step_ms        host wall time of one navgpu_fleet_step_tp (it ends in a device synchronise), mean over the timed
                    steps; it includes the costmap update, the copies and the host's enumeration and selection
  footprint_ms, wavefront_ms, score_ms   device time (CUDA events) of k_tp_fleet_footprint, the MapGrid launch (two
                    wavefronts per robot) and k_tp_fleet_score, means over the timed steps
  h2d_bytes, d2h_bytes   bytes copied each way per step by the planner side, computed from the sample counts (the
                    previous step's escape flags decide them): samples (24 B each) and per-robot records (112 B) up,
                    scored samples (24 B each) down.  Costmap inputs (maps, scans) are not included.
  dwa_step_ms       the DWA raw-map fleet (config C5, 20 x 1 x 20 samples) step in the same process
  valid_robots      robots whose result has a cost >= 0 in the last step
  gpu, power_limit  the card and its power limit, read in the same run
--sensing runs the same planner on a 2-D sensing fleet ([ObstacleLayer, InflationLayer] per robot) fed one fresh
synth.fleet_scan per robot and step (K distinct cycles ray-cast before timing, step k uses cycle k mod K), and adds
"sensing": true; tp_step_ms then includes set_scans.
--check N replays N evenly spaced robots through the CPU checker (its LayeredCostmap, then its TrajectoryPlanner) over
every step and reports how many agree: costmaps bit for bit, velocities, flags and n_points equal, cost within 1e-5
relative."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PENTAGON = [(-0.325, -0.325), (-0.325, 0.325), (0.325, 0.325), (0.46, 0.0), (0.325, -0.325)]
DWA_CFG = dict(vx_samples=20, vy_samples=1, vth_samples=20, max_vel_y=0.0, min_vel_y=0.0)
SAMPLE_BYTES = 24       # (vx, vy, vtheta) doubles up, TpSampleResult down
ROBOT_RECORD_BYTES = 112  # TpFleetRobot: 12 doubles + 4 int32


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception as e:  # the numbers are still reported, without the card's limit
        return f"unknown ({e})", "unknown"


def sample_count(cfg, escaping):
    """createTrajectories' samples of one robot (tp_enumerate): no forward ones while escaping."""
    forward = 0 if escaping else cfg.vx_samples * cfg.vtheta_samples + (2 if cfg.holonomic_robot else 0)
    return forward + cfg.vtheta_samples + (cfg.n_y_vels if cfg.holonomic_robot else 0) + 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--robots", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--cycles", type=int, default=4, help="distinct scan cycles ray-cast before timing (--sensing)")
    ap.add_argument("--check", type=int, default=0)
    ap.add_argument("--sensing", action="store_true", help="a 2-D sensing fleet fed synth.fleet_scan")
    args = ap.parse_args()
    if args.steps < 1 or args.robots < 1 or args.cycles < 1 or args.warmup < 0:
        ap.error("--steps, --robots and --cycles must be positive")

    import navigation_b200
    from navigation_b200 import build, synth
    build.build()
    cuda = navigation_b200.load()
    if cuda.device_count() == 0:
        sys.exit("bench_fleet_tp needs a CUDA device (libnavgpu has no CPU path)")
    n, sx, res = args.robots, 120, 0.05
    total = args.warmup + args.steps

    t0 = time.perf_counter()
    if args.sensing:
        robots = [synth.fleet_sensing_robot(i, n=sx, res=res) for i in range(n)]
        scans = [[[synth.fleet_scan(r, c)] for r in robots] for c in range(args.cycles)]
        poses = [np.ascontiguousarray([r["poses"][c] for r in robots]) for c in range(args.cycles)]
        fleet = cuda.fleet_sensing(n, sx, sx, res, PENTAGON, trajectory_planner={})
    else:
        robots = [synth.fleet_robot(i) for i in range(n)]
        poses = [np.ascontiguousarray([r["pose"] for r in robots])]
        fleet = cuda.fleet(n, sx, sx, res, PENTAGON, 0.55, 10.0, trajectory_planner={})
        fleet.set_maps(np.stack([r["raw"] for r in robots]), np.array([r["origin"] for r in robots]))
    vels = np.ascontiguousarray([r["vel"] for r in robots])
    prep_s = time.perf_counter() - t0
    cfg = fleet.tp_cfg

    fleet.set_plans(poses[0], [r["plan"] for r in robots])
    sample = list(range(0, n, max(1, n // args.check)))[:args.check] if args.check else []
    history = {i: [] for i in sample}
    wall, t_fp, t_wf, t_sc, h2d, d2h = [], [], [], [], [], []
    escaping = np.zeros(n, bool)
    for k in range(total):
        c = k % len(poses)
        t = time.perf_counter()
        if args.sensing:
            fleet.set_scans(scans[k % args.cycles])
        r = fleet.step_raw(poses[c], vels)
        dt = time.perf_counter() - t
        n_samples = sum(sample_count(cfg, e) for e in escaping)
        escaping = np.array([bool(r[i].flags & 256) for i in range(n)])
        for i in sample:
            history[i].append((r[i].cost, r[i].xv, r[i].yv, r[i].thetav, r[i].flags, r[i].n_points))
        if k >= args.warmup:
            wall.append(dt * 1e3)
            a, b, s = fleet.tp_timing()
            t_fp.append(a)
            t_wf.append(b)
            t_sc.append(s)
            h2d.append(n_samples * SAMPLE_BYTES + n * ROBOT_RECORD_BYTES)
            d2h.append(n_samples * SAMPLE_BYTES)
    valid = sum(1 for i in range(n) if r[i].cost >= 0)
    backing_up = sum(1 for i in range(n) if r[i].xv < 0)

    # the DWA raw-map fleet (config C5) in the same process
    raw_robots = [synth.fleet_robot(i) for i in range(n)]
    dwa = cuda.fleet(n, sx, sx, res, PENTAGON, 0.55, 10.0, **DWA_CFG)
    dwa.set_maps(np.stack([q["raw"] for q in raw_robots]), np.array([q["origin"] for q in raw_robots]))
    rposes = np.ascontiguousarray([q["pose"] for q in raw_robots])
    rvels = np.ascontiguousarray([q["vel"] for q in raw_robots])
    dwa.set_plans(rposes, [q["plan"] for q in raw_robots])
    dwa_ms = []
    for k in range(total):
        t = time.perf_counter()
        dwa.step_raw(rposes, rvels)
        if k >= args.warmup:
            dwa_ms.append((time.perf_counter() - t) * 1e3)

    checked = agree = 0
    if sample:
        from oracle import pyoracle
        port = pyoracle.load("port")
        final = {i: fleet.costmap(i) for i in sample}
        for i in sample:
            if args.sensing:
                cm = port.costmap(sx, sx, res, 0.0, 0.0, rolling=True)
                o = cm.add_obstacle_layer(1, True, 2.0)
                il = cm.add_inflation_layer(0.55, 10.0)
                cm.set_inflation_variant(il, 4)  # exact windowed nearest-seed inflation (inflation mode 0)
            else:
                cm = port.costmap(sx, sx, res, *robots[i]["origin"])
                s_layer = cm.add_grid_layer(0)
                cm.add_inflation_layer(0.55, 10.0)
                cm.set_grid_layer(s_layer, robots[i]["raw"])
            cm.set_footprint(PENTAGON)
            tp = port.trajectory_planner(sx, sx, res, PENTAGON)
            tp.update_plan(robots[i]["plan"])
            ok = True
            for k in range(total):
                c = k % len(poses)
                if args.sensing:
                    s_ = scans[k % args.cycles][i][0]
                    org, pts = port.project_scan(s_)
                    cm.set_observations(o, [dict(origin=org, points=pts, obstacle_range=s_["obstacle_range"],
                                                 raytrace_range=s_["raytrace_range"])])
                    cm.update_map(*poses[c][i])
                elif k == 0:
                    cm.update_map(0, 0, 0)
                tp.set_costmap(cm.get(), *cm.origin())
                e = tp.find_best_path(poses[c][i], vels[i])
                got = history[i][k]
                want = (e["cost"], e["xv"], e["yv"], e["thetav"], e["flags"], len(e["points"]))
                ok = ok and got[1:] == want[1:] and bool(np.isclose(got[0], want[0], rtol=1e-5, atol=0))
            ok = ok and np.array_equal(final[i], cm.get())
            checked += 1
            agree += ok

    name, limit = gpu_info()
    out = dict(robots=n, map=f"{sx}x{sx}@{res}", planner="TrajectoryPlanner", samples_per_robot=sample_count(cfg, False),
               steps=args.steps, warmup=args.warmup,
               tp_step_ms=float(np.mean(wall)), tp_step_ms_min=float(np.min(wall)),
               footprint_ms=float(np.mean(t_fp)), wavefront_ms=float(np.mean(t_wf)), score_ms=float(np.mean(t_sc)),
               h2d_bytes=int(np.mean(h2d)), d2h_bytes=int(np.mean(d2h)),
               dwa_step_ms=float(np.mean(dwa_ms)), dwa_step_ms_min=float(np.min(dwa_ms)),
               valid_robots=valid, backing_up=backing_up, checked=checked, checked_agree=agree,
               input_prep_s=round(prep_s, 1), gpu=name, power_limit=limit)
    if args.sensing:
        out.update(sensing=True, scan_cycles=args.cycles, beams=360)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
