"""Measurement helper: where the C3 cycle's time goes -- obstacle layer on / off / without observations, flushed and
hot L2."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import navigation_b200  # noqa: E402

api = navigation_b200.load()
size = int(os.environ.get("PROBE_SIZE", 4000))
cm, (s, o, il), sets = bench.build_c3(lambda *a: api.costmap(*a), size=size)
obs, robot = sets[0]
stream = torch.cuda.ExternalStream(cm.stream())
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")


def measure(label):
    for _ in range(5):
        cm.touch_grid_layer(s, 0, 0, size, size)
        cm.update_map(*robot)
    n = 100
    e0 = [torch.cuda.Event(enable_timing=True) for _ in range(n)]
    e1 = [torch.cuda.Event(enable_timing=True) for _ in range(n)]
    for k in range(n):
        with torch.cuda.stream(stream):
            flush.zero_()
            e0[k].record(stream)
        cm.touch_grid_layer(s, 0, 0, size, size)
        cm.update_map_async(*robot)
        e1[k].record(stream)
    torch.cuda.synchronize()
    cold = np.mean([a.elapsed_time(b) for a, b in zip(e0, e1)])
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for k in range(n):
        cm.touch_grid_layer(s, 0, 0, size, size)
        cm.update_map_async(*robot)
    b.record(stream)
    torch.cuda.synchronize()
    print(f"{label:34s} flushed_us={1e3 * cold:.1f} hot_us={1e3 * a.elapsed_time(b) / n:.1f}", flush=True)


cm.set_observations(o, obs)
measure("full C3 (8 x 360 rays)")
cm.set_observations(o, [])
measure("obstacle layer, no observations")
cm.set_enabled(o, False)
measure("obstacle layer disabled")
cm.set_enabled(o, True)
cm.set_observations(o, obs[:1])
measure("one observation (360 rays)")
