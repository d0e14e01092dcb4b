"""Measurement helper (not part of the product): times the fused sweep kernel of the C3 cycle with CUDA events."""
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
cm.set_profiling(True)
obs, robot = sets[0]
cm.set_observations(o, obs)
stream = torch.cuda.ExternalStream(cm.stream())
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
for _ in range(5):
    cm.touch_grid_layer(s, 0, 0, size, size)
    cm.update_map(*robot)
cyc, swp = [], []
for k in range(20):
    with torch.cuda.stream(stream):
        flush.zero_()
    cm.touch_grid_layer(s, 0, 0, size, size)
    cm.update_map_async(*robot)
    c, w = cm.last_timing()
    cyc.append(c)
    swp.append(w)
print(f"size={size} cycle_ms={np.mean(cyc):.4f} sweep_ms={np.mean(swp):.4f} "
      f"min_sweep={np.min(swp):.4f}")
