"""Batched scan ingest without a GPU: the ctypes descriptor has navgpu_fleet_scan_source's layout, and the dense
batches synth makes for Fleet.set_scan_batch are well formed and stand for the per-robot scan lists synth.batch_scans
derives from them."""
import ctypes
import os
import subprocess

import numpy as np

from navigation_b200 import synth
from navigation_b200.api import FleetScanSource

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = [f for f, _ in FleetScanSource._fields_]


def test_descriptor_layout_matches_the_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "navgpu.h"\nint main(void) {\n'
                   '  printf("%zu", sizeof(navgpu_fleet_scan_source));\n' +
                   "".join(f'  printf(" %zu", offsetof(navgpu_fleet_scan_source, {f}));\n' for f in FIELDS) +
                   "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    want = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    got = [ctypes.sizeof(FleetScanSource)] + [getattr(FleetScanSource, f).offset for f in FIELDS]
    assert got == want


def test_batches_are_dense_and_match_their_scan_lists():
    robots = [synth.fleet_sensing_robot(i) for i in range(3)]
    laser = synth.fleet_scan_batch(robots, 2)
    cloud = synth.fleet_scan_batch(robots, 2, cloud=True, n_beams=90)
    assert laser["ranges"].shape == (3, 360) and laser["ranges"].dtype == np.float32
    assert cloud["points"].shape == (3, 90, 3) and cloud["points"].dtype == np.float32
    assert laser["sensor_to_global"].shape == (3, 7) and laser["sensor_to_global"].dtype == np.float64
    assert np.isposinf(laser["ranges"]).any() and np.isfinite(laser["ranges"]).any()
    lists = synth.batch_scans([laser, cloud], 3)
    for r, (rb, scans) in enumerate(zip(robots, lists)):
        x, y, yaw = rb["poses"][2]
        assert len(scans) == 2 and np.array_equal(scans[0]["ranges"], laser["ranges"][r])
        assert scans[0]["translation"] == (x, y, 0.3) and scans[0]["angle_min"] == laser["angle_min"]
        assert np.isclose(2 * np.arctan2(scans[1]["rotation_xyzw"][2], scans[1]["rotation_xyzw"][3]), yaw)
        assert "ranges" not in scans[1] and np.array_equal(scans[1]["points"], cloud["points"][r])
        # the shared sensor-frame angle: beam i of the scan ends where the cloud's beam i of the same cycle does (the
        # centre of the cell it hit, so near the beam's direction rather than on it)
        ang = float(laser["angle_min"]) + np.arange(360) * float(laser["angle_increment"])
        rng = laser["ranges"][r]
        ok = np.isfinite(rng)
        same = synth.fleet_scan_batch([rb], 2, cloud=True)["points"][0]
        assert np.allclose(np.hypot(same[ok, 0], same[ok, 1]), rng[ok], rtol=1e-5)
        err = np.angle(np.exp(1j * (np.arctan2(same[ok, 1], same[ok, 0]) - ang[ok])))
        assert (np.abs(err) * rng[ok] < 0.05).all()
    assert synth.batch_scans([], 3) == [[], [], []]


def test_cloud_3d_batch_stacks_the_robots_clouds():
    robots = [synth.fleet_voxel_robot(i) for i in range(2)]
    b = synth.fleet_cloud_3d_batch(robots, 1)
    for r, rb in enumerate(robots):
        c = synth.fleet_cloud_3d(rb, 1)
        assert np.array_equal(b["points"][r], c["points"])
        assert list(b["sensor_to_global"][r]) == list(c["translation"]) + list(c["rotation_xyzw"])
        assert all(b[k] == c[k] for k in c if k not in ("points", "translation", "rotation_xyzw"))
