"""Drop-in check of the C++ adapters (navigation_b200/plugin) next to the reference's own classes.

oracle/_ref/dropin_harness is built where NAVIGATION_REFERENCE names the reference's sources (`make -C oracle dropin
REF=...`): the adapters and tests/cpp/dropin_harness.cpp are compiled against the reference's headers and linked with
the reference's unmodified hot-path sources (oracle/_ref/libnavref.so) and libnavgpu.so.  A harness built on one
machine may be run on another that has the library but not the sources."""
import os
import subprocess

import pytest

from oracle import pyoracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS = os.path.join(ROOT, "oracle", "_ref", "dropin_harness")


def build_harness():
    from navigation_b200 import build
    build.build()
    pyoracle.make("ref", "dropin")


def test_dropin_harness_builds_against_reference_headers():
    """GpuInflationLayer : costmap_2d::Layer, GpuLayeredCostmap and GpuScoredSamplingPlanner : TrajectorySearch compile
    against the reference's own headers and link with its compiled sources (no GPU needed for that)."""
    if not pyoracle.reference_dir():
        pytest.skip("needs NAVIGATION_REFERENCE")
    build_harness()
    assert os.access(HARNESS, os.X_OK)


@pytest.mark.gpu
def test_adapters_match_reference_classes(cuda):
    """A1: reference LayeredCostmap with GpuInflationLayer as its plugin == with costmap_2d::InflationLayer (4 cycles);
    A2: GpuLayeredCostmap == reference stack; B: GpuScoredSamplingPlanner through base_local_planner::TrajectorySearch
    == the reference's generator + critics + SimpleScoredSamplingPlanner (best index, cost <= 1e-5 rel, velocities,
    point count, explored count, oscillation flags) over 6 control cycles; C: GpuTrajectoryPlanner == the reference's
    TrajectoryPlanner through the same public calls; D: GpuLayeredCostmap fed with LaserScans == the checker's stack fed
    with the clouds of the restated ingest path."""
    if not os.path.exists(HARNESS):
        if pyoracle.reference_dir():
            build_harness()
        else:
            pytest.skip("oracle/_ref/dropin_harness was not built (needs NAVIGATION_REFERENCE)")
    r = subprocess.run([HARNESS], capture_output=True, text=True, timeout=300)
    print(r.stdout)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "DROP-IN OK" in r.stdout
