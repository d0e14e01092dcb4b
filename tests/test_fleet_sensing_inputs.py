"""Sensing fleets without a GPU: the constructor refuses to run without a device (no CPU fallback), and the seeded
inputs the tests and tools/bench_fleet_sensing.py feed them are well formed and reproducible."""
import numpy as np
import pytest

import scenarios as sc
from navigation_b200 import synth


def test_fleet_sensing_needs_a_device():
    import navigation_b200
    a = navigation_b200.load()
    if a.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(navigation_b200.api.NavGpuError, match="no CUDA device"):
        a.fleet_sensing(2, 120, 120, 0.05, sc.PENTAGON)


def test_fleet_sensing_inputs_are_seeded_and_well_formed():
    r, again = synth.fleet_sensing_robot(7), synth.fleet_sensing_robot(7)
    assert np.array_equal(r["world"], again["world"]) and np.array_equal(r["poses"], again["poses"])
    assert r["world"].shape == (240, 240) and r["poses"].shape == (64, 3)
    res, (ox, oy) = r["resolution"], r["origin"]
    for x, y, _ in r["poses"]:  # the robot drives through free space, 12 cells from anything
        cx, cy = int((x - ox) / res), int((y - oy) / res)
        assert not r["world"][cy - 11:cy + 12, cx - 11:cx + 12].any()
    scan, cloud = synth.fleet_scan(r, 5), synth.fleet_scan(r, 5, cloud=True)
    assert scan["ranges"].dtype == np.float32 and scan["ranges"].shape == (360,)
    assert np.isinf(scan["ranges"]).any() and np.isfinite(scan["ranges"]).any() and scan["inf_is_valid"] == 1
    assert cloud["points"].shape == (360, 3) and cloud["points"].dtype == np.float32
    finite = np.isfinite(scan["ranges"])
    assert np.allclose(np.hypot(cloud["points"][finite, 0], cloud["points"][finite, 1]), scan["ranges"][finite], atol=1e-5)
