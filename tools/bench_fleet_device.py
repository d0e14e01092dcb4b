"""Device fleet steps (navgpu_fleet_step_device) against host fleet steps (navgpu_fleet_step) on one GPU.  Prints one
JSON line per fleet kind:
  raw       config C5's inputs: 4096 robots of synth.fleet_robot(i) (120 x 120 raw local maps at 0.05 m), the
            pentagon footprint, DWAPlanner with 20 x 1 x 20 samples
  sensing   4096 synth.fleet_sensing_robot(i) robots, 120 x 120, one LaserScan source per robot (set_scan_batch)
  voxel     the same with a VoxelLayer fed one 3-D cloud source per robot
with, as means over the timed steps:
  host_step_ms        host wall time of navgpu_fleet_step (it ends in a device synchronise)
  device_enqueue_ms   host wall time of the navgpu_fleet_step_device call alone (it returns without waiting)
  device_step_ms      CUDA-event time of the device step on the fleet's stream
  host_scan_ms, device_scan_ms   (sensing kinds) the scan batch's host call (host arrays, waited for) and the device
                      batch's event time on the fleet's stream, fed right before each step
  score_host_us, score_device_us   k_fleet_score's device time per step on each path (torch.profiler, a separate
                      pass): the host path sizes its grid from the robots' real sample counts, the device path from
                      the configuration's bound, whose extra CTAs exit at once
  gpu, power_limit    the card and its power limit, read in the same run
Host and device steps alternate, each on its own fleet, so that each fleet's state stays on its own path."""
import argparse
import ctypes as C
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


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception as e:  # the numbers are still reported, without the card's limit
        return f"unknown ({e})", "unknown"


def build(api, synth, kind, n):
    if kind == "raw":
        robots = [synth.fleet_robot(i) for i in range(n)]
        fleets = [api.fleet(n, 120, 120, 0.05, PENTAGON, 0.55, 10.0, **CFG) for _ in range(2)]
        for f in fleets:
            f.set_maps(np.stack([r["raw"] for r in robots]), np.array([r["origin"] for r in robots]))
        poses = lambda c: np.array([r["pose"] for r in robots])
        sources = None
    else:
        make = synth.fleet_voxel_robot if kind == "voxel" else synth.fleet_sensing_robot
        robots = [make(i) for i in range(n)]
        fleets = [api.fleet_sensing(n, 120, 120, 0.05, PENTAGON, voxel={} if kind == "voxel" else None, **CFG)
                  for _ in range(2)]
        poses = lambda c: np.array([r["poses"][c % len(r["poses"])] for r in robots])
        sources = (lambda c: [synth.fleet_cloud_3d_batch(robots, c)]) if kind == "voxel" else \
            (lambda c: [synth.fleet_scan_batch(robots, c)])
    for f in fleets:
        f.set_plans(poses(0), [r["plan"] for r in robots])
    return fleets, poses, sources, np.array([r["vel"] for r in robots])


def to_device(torch, sources):
    out = []
    for s in sources:
        d = dict(s)
        for k in ("ranges", "points", "sensor_to_global"):
            if k in s:
                d[k] = torch.from_numpy(s[k]).cuda()
        out.append(d)
    return out


def run_kind(api, synth, torch, kind, n, steps, warmup):
    (host, dev), poses, sources, vels = build(api, synth, kind, n)
    lib = api.lib
    stream = torch.cuda.ExternalStream(dev.stream())
    R = torch.empty(n * 48, dtype=torch.uint8, device="cuda")
    V = torch.from_numpy(vels).cuda()
    P = [torch.from_numpy(np.ascontiguousarray(poses(c))).cuda() for c in range(warmup + steps)]
    S = [(sources(c), to_device(torch, sources(c))) for c in range(warmup + steps)] if sources else None
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    acc = dict(host_step_ms=0.0, device_enqueue_ms=0.0, device_step_ms=0.0, host_scan_ms=0.0, device_scan_ms=0.0)
    torch.cuda.synchronize()
    for c in range(warmup + steps):
        p_host = np.ascontiguousarray(poses(c))
        if S:
            t0 = time.perf_counter()
            host.set_scan_batch(S[c][0])
            t_scan = time.perf_counter() - t0
        t0 = time.perf_counter()
        host.step_raw(p_host, vels)
        t_host = time.perf_counter() - t0
        torch.cuda.synchronize()
        if S:
            ev[2].record(stream)
            dev.set_scan_batch(S[c][1])
            ev[3].record(stream)
        ev[0].record(stream)
        t0 = time.perf_counter()
        rc = lib.navgpu_fleet_step_device(dev.h, C.c_void_p(P[c].data_ptr()), C.c_void_p(V.data_ptr()),
                                          C.c_void_p(R.data_ptr()))
        t_enq = time.perf_counter() - t0
        ev[1].record(stream)
        api.check(rc)
        torch.cuda.synchronize()
        if c >= warmup:
            acc["host_step_ms"] += t_host * 1e3
            acc["device_enqueue_ms"] += t_enq * 1e3
            acc["device_step_ms"] += ev[0].elapsed_time(ev[1])
            if S:
                acc["host_scan_ms"] += t_scan * 1e3
                acc["device_scan_ms"] += ev[2].elapsed_time(ev[3])
    res = {k: round(v / steps, 4) for k, v in acc.items() if S or "scan" not in k}
    # k_fleet_score on each path, in a profiled pass of its own
    from torch.profiler import ProfilerActivity, profile
    score = {}
    for name, fleet, call in (("host", host, lambda c: host.step_raw(np.ascontiguousarray(poses(c)), vels)),
                              ("device", dev, lambda c: api.check(lib.navgpu_fleet_step_device(
                                  dev.h, C.c_void_p(P[c].data_ptr()), C.c_void_p(V.data_ptr()),
                                  C.c_void_p(R.data_ptr()))))):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for c in range(steps):
                call(c)
            torch.cuda.synchronize()
        tot = cnt = 0
        for e in prof.events():
            if "k_fleet_score" in e.name and e.device_type.name == "CUDA":
                tot += e.device_time if hasattr(e, "device_time") else e.cuda_time
                cnt += 1
        score[f"score_{name}_us"] = round(tot / max(cnt, 1), 2)
    res.update(score)
    # the two paths computed the same results on the last step
    host_r = host.step_raw(np.ascontiguousarray(poses(0)), vels)
    api.check(lib.navgpu_fleet_step_device(dev.h, C.c_void_p(P[0].data_ptr()), C.c_void_p(V.data_ptr()),
                                           C.c_void_p(R.data_ptr())))
    torch.cuda.synchronize()
    res["results_equal"] = bytes(R.cpu().numpy()) == C.string_at(C.addressof(host_r), n * 48)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--robots", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--kinds", default="raw,sensing,voxel")
    args = ap.parse_args()
    import torch
    import navigation_b200
    from navigation_b200 import build as nbuild, synth
    nbuild.build()
    api = navigation_b200.load()
    name, limit = gpu_info()
    for kind in args.kinds.split(","):
        res = dict(kind=kind, robots=args.robots, steps=args.steps)
        res.update(run_kind(api, synth, torch, kind, args.robots, args.steps, args.warmup))
        res.update(gpu=name, power_limit=limit)
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
