"""Goal handling for fleets (navgpu_fleet_set_active, navgpu_fleet_check_trajectories) at config C5's inputs: 4096 robots of
synth.fleet_robot(i) (120 x 120 raw local maps at 0.05 m, inflated on the device), the pentagon footprint, DWAPlanner
with C5's 20 x 1 x 20 samples and TrajectoryPlannerROS's defaults (the inputs of tools/bench_fleet_tp.py).  Prints one
JSON line; for each planner (dwa_*, tp_*):
  step_ms_100, step_ms_50, step_ms_10   host wall time of one step (it ends in a device synchronise) with 100 %, 50 %
                    and 10 % of the robots active (every robot, every 2nd, every 10th), means over the timed steps
  check_ms_1, check_ms_32   host wall time of one navgpu_fleet_check_trajectories call (it returns once the costs are on
                    the host) with 1 and 32 candidates per robot, means over the timed calls
  check_kernel_ms_1, check_kernel_ms_32   device time of the call's scoring kernel (k_fleet_check, k_tp_fleet_score), and
  check_device_ms_1, check_device_ms_32   of everything the call put on the GPU (kernel and copies), per call, from a
                    separate torch.profiler pass with CUDA activities
  gpu, power_limit  the card and its power limit, read in the same run
Candidates are stop, rotate and creep commands of the goal controllers (and variations of them), cycled over robots."""
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
FRACTIONS = (100, 50, 10)
KERNELS = {"dwa": "k_fleet_check", "tp": "k_tp_fleet_score"}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception as e:  # the numbers are still reported, without the card's limit
        return f"unknown ({e})", "unknown"


def candidates(n, k):
    """k commands per robot: stop, rotate either way, creep forward, varied by the robot's index."""
    base = np.array([(0.0, 0.0, 0.0), (0.0, 0.0, 0.4), (0.0, 0.0, -0.4), (0.1, 0.0, 0.0)])
    j = (np.arange(n)[:, None] + np.arange(k)[None, :]) % len(base)
    scale = 1.0 + 0.01 * (np.arange(k)[None, :, None] // len(base))
    return list(base[j] * scale)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--robots", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if args.steps < 1 or args.robots < 1 or args.warmup < 0:
        ap.error("--steps and --robots must be positive")

    import torch
    import navigation_b200
    from navigation_b200 import build, synth
    build.build()
    cuda = navigation_b200.load()
    if cuda.device_count() == 0:
        sys.exit("bench_fleet_goal needs a CUDA device (libnavgpu has no CPU path)")
    n, sx, res = args.robots, 120, 0.05
    robots = [synth.fleet_robot(i) for i in range(n)]
    maps = np.stack([r["raw"] for r in robots])
    origins = np.array([r["origin"] for r in robots])
    poses = np.ascontiguousarray([r["pose"] for r in robots])
    vels = np.ascontiguousarray([r["vel"] for r in robots])
    plans = [r["plan"] for r in robots]
    cands = {k: candidates(n, k) for k in (1, 32)}

    out = dict(robots=n, map=f"{sx}x{sx}@{res}", steps=args.steps, warmup=args.warmup)
    for planner in ("dwa", "tp"):
        kw = DWA_CFG if planner == "dwa" else dict(trajectory_planner={})
        fleet = cuda.fleet(n, sx, sx, res, PENTAGON, 0.55, 10.0, **kw)
        fleet.set_maps(maps, origins)
        fleet.set_plans(poses, plans)
        for pct in FRACTIONS:
            fleet.set_active(np.arange(n) % (100 // pct) == 0)
            wall = []
            for s in range(args.warmup + args.steps):
                t = time.perf_counter()
                fleet.step_raw(poses, vels)
                if s >= args.warmup:
                    wall.append((time.perf_counter() - t) * 1e3)
            out[f"{planner}_step_ms_{pct}"] = float(np.mean(wall))
        fleet.set_active(None)
        fleet.step_raw(poses, vels)
        for k, c in cands.items():
            wall = []
            for s in range(args.warmup + args.steps):
                t = time.perf_counter()
                costs = fleet.check_trajectories(poses, vels, c)
                if s >= args.warmup:
                    wall.append((time.perf_counter() - t) * 1e3)
            out[f"{planner}_check_ms_{k}"] = float(np.mean(wall))
            out[f"{planner}_check_legal_{k}"] = int(sum((x >= 0).sum() for x in costs))
        # device time, in a profiled pass of its own
        from torch.profiler import ProfilerActivity, profile
        for k, c in cands.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.steps):
                    fleet.check_trajectories(poses, vels, c)
                torch.cuda.synchronize()
            kern = dev = 0.0
            for e in prof.events():
                if e.device_type != torch.autograd.DeviceType.CUDA:
                    continue
                us = e.time_range.elapsed_us()  # a kernel or copy on the device
                dev += us
                if KERNELS[planner] in e.name:
                    kern += us
            out[f"{planner}_check_kernel_ms_{k}"] = kern / 1e3 / args.steps
            out[f"{planner}_check_device_ms_{k}"] = dev / 1e3 / args.steps
        del fleet
    name, limit = gpu_info()
    out.update(gpu=name, power_limit=limit)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
