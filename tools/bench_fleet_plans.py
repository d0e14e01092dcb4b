"""Plan following for a sensing fleet: the host loop a caller runs today against navgpu_fleet_update_plans_device, on
one GPU.  4096 synth.fleet_sensing_robot(i) robots (120 x 120 rolling local costmaps at 0.05 m, one LaserScan source
per robot, DWAPlanner with 20 x 1 x 20 samples), each with a global plan of about 2000 poses 0.025 m apart that starts
5 m behind the robot and runs far beyond its map; the robots advance 0.1 m along their plans per cycle.  Per cycle:
  (a) host path    navgpu_plans_transform + navgpu_plans_prune on host arrays, the erasure bookkeeping in numpy,
                   navgpu_fleet_set_plans, then navgpu_fleet_step_device
  (b) device path  navgpu_fleet_update_plans_device, then navgpu_fleet_step_device
each on its own fleet, alternating, both fed the same scans (set_scan_batch_device, outside the timed window).
Prints one JSON line with, as means over the timed cycles:
  host_path_ms, device_path_ms          host wall time of the cycle, ending in a synchronise
  host_path_stream_ms, device_path_stream_ms   CUDA-event time on the fleet's stream (the host path's transform and
                                        prune run on their own stream, before its events)
  update_kernel_us                      k_fleet_update_plans' device time per cycle (torch.profiler, a separate pass)
  results_equal                         every result record of (a) and (b) bit-equal in every cycle
  gpu, power_limit                      the card and its power limit, read in the same run"""
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
CFG = dict(vx_samples=20, vy_samples=1, vth_samples=20, max_vel_y=0.0, min_vel_y=0.0)
IDENTITY = [1.0, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0]


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
    ap.add_argument("--cycles", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch
    import navigation_b200
    from navigation_b200 import synth
    api = navigation_b200.load()
    n = args.robots
    robots = [synth.fleet_sensing_robot(i) for i in range(n)]
    plans = []
    for i, r in enumerate(robots):
        x0, y0, _ = r["poses"][0]
        t = np.arange(-200, 1800 + (i % 5) * 50) * 0.025
        plans.append(np.stack([x0 + t, y0 + 0.2 * np.sin(0.3 * t + i)], 1))
    fleets = [api.fleet_sensing(n, 120, 120, 0.05, PENTAGON, **CFG) for _ in range(2)]
    host_f, dev_f = fleets
    dev_f.set_global_plans(plans)
    held = [p.copy() for p in plans]
    vels = torch.from_numpy(np.array([r["vel"] for r in robots])).cuda()
    streams = [torch.cuda.ExternalStream(f.stream()) for f in fleets]

    def poses(c):
        out = np.array([(p[200 + 4 * c, 0], p[200 + 4 * c, 1] + 0.02 * np.sin(c + i), 0.1 * np.sin(c))
                        for i, p in enumerate(plans)])
        return out, torch.from_numpy(out).cuda()

    def feed(c):
        src = synth.fleet_scan_batch(robots, c)
        d = {k: (torch.from_numpy(v).cuda() if k in ("ranges", "sensor_to_global") else v) for k, v in src.items()}
        for f in fleets:
            f.set_scan_batch([d])
        torch.cuda.synchronize()

    def host_cycle(c, hp, P):
        nonlocal held
        _, local = api.plans_transform(held, hp[:, :2], [IDENTITY] * n, [3.0] * n)
        erase = api.plans_prune(local, hp[:, :2])
        held = [h[e:] for h, e in zip(held, erase)]
        host_f.set_plans(hp, [q[e:, :2] for q, e in zip(local, erase)])
        return host_f.step_device(P, vels)

    def dev_cycle(c, hp, P):
        dev_f.update_plans_device(P)
        return dev_f.step_device(P, vels)

    times = {"host": [], "device": []}
    events = {"host": [], "device": []}
    equal = True
    total = args.warmup + args.cycles
    for c in range(total):
        feed(c)
        hp, P = poses(c)
        recs = {}
        for name, run, s in (("host", host_cycle, streams[0]), ("device", dev_cycle, streams[1])):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0.record(s)
            out = run(c, hp, P)
            e1.record(s)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            recs[name] = out["records"].cpu().numpy()
            if c >= args.warmup:
                times[name].append((t1 - t0) * 1e3)
                events[name].append(e0.elapsed_time(e1))
        equal &= bool(np.array_equal(recs["host"], recs["device"]))
    # the update kernel's own time, from a profiled pass of device cycles
    from torch.profiler import ProfilerActivity, profile
    prof_cycles = 5
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for c in range(total, total + prof_cycles):
            _, P = poses(c)
            dev_cycle(c, None, P)
        torch.cuda.synchronize()
    kern = [e for e in prof.key_averages() if "k_fleet_update_plans" in e.key]
    dt = (lambda e: getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0))
    update_us = sum(dt(e) for e in kern) / prof_cycles if kern else None
    gpu, limit = gpu_info()
    print(json.dumps(dict(
        kind="sensing", robots=n, plan_poses=int(np.mean([len(p) for p in plans])), cycles=args.cycles,
        host_path_ms=round(float(np.mean(times["host"])), 3), device_path_ms=round(float(np.mean(times["device"])), 3),
        host_path_stream_ms=round(float(np.mean(events["host"])), 3),
        device_path_stream_ms=round(float(np.mean(events["device"])), 3),
        update_kernel_us=None if update_us is None else round(update_us, 2), results_equal=equal, gpu=gpu,
        power_limit=limit)))


if __name__ == "__main__":
    main()
