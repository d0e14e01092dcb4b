"""SURVEY.md 8f-4: the legacy base_local_planner::TrajectoryPlanner on the GPU (navgpu_tp_*) against the CPU restatement
(oracle/navoracle.cpp, pinned bit-for-bit to the compiled reference), the reference's own compiled class (oracle/_ref,
when it travelled with the repository) and golden fixtures generated from it.

Everything that is integer or decided by integers (both MapGrid wavefronts with within_robot cells, the chosen
velocities, the oscillation / escape flags, the number of trajectory points) must be identical; costs and points are
asserted bit-exact first and may differ by 1e-5 relative only where CUDA's sin/cos differs from glibc's in the last bit.
"""
import numpy as np
import pytest

import golden_util as gu
import scenarios as sc

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def assert_cycles_match(a, b, what):
    for c, (x, y) in enumerate(zip(a, b)):
        assert sc.tp_results_equal(x, y, rtol=RTOL), (
            f"{what} cycle {c}: cost {x['cost']} vs {y['cost']}, v ({x['xv']}, {x['yv']}, {x['thetav']}) vs "
            f"({y['xv']}, {y['yv']}, {y['thetav']}), flags {x['flags']} vs {y['flags']}, "
            f"points {len(x['points'])} vs {len(y['points'])}, scores {x['scores']} vs {y['scores']}")


@pytest.mark.parametrize("seed", range(52))  # 40-51 are also compared with the reference where it is built
def test_tp_scenarios_match_checker(cuda, port, seed):
    assert_cycles_match(sc.run_tp_scenario(cuda, port, seed), sc.run_tp_scenario(port, port, seed), f"seed {seed}")


@pytest.mark.parametrize("seed", range(40, 52))
def test_tp_scenarios_match_reference(cuda, port, ref, seed):
    """... and against the reference's own compiled class where oracle/_ref travelled with the repository"""
    assert_cycles_match(sc.run_tp_scenario(cuda, port, seed), sc.run_tp_scenario(ref, port, seed), f"seed {seed}")


@pytest.mark.parametrize("seed,path", gu.tp_cases())
def test_tp_golden_fixtures(cuda, port, seed, path):
    assert_cycles_match(gu.run_tp_case(cuda, port, seed), gu.load_tp_case(path), f"golden seed {seed}")


def test_tp_boxed_in_matches_checker(cuda, port):
    """Strafing in both directions with its stuck flag latching, then backing up with nothing legal left."""
    got, want = sc.run_tp_boxed_scenario(cuda), sc.run_tp_boxed_scenario(port)
    assert_cycles_match(got, want, "boxed")
    assert any(r["yv"] > 0 for r in got) and any(r["yv"] < 0 for r in got) and any(r["xv"] < 0 for r in got)
    assert got[-1]["flags"] & 4  # stuck_left_strafe


def test_tp_edge_cases_match_checker(cuda, port):
    """No plan, degenerate and empty footprints, a one-pose plan, the robot outside the map."""
    assert_cycles_match(sc.run_tp_edge_cases(cuda, port), sc.run_tp_edge_cases(port, port), "edge cases")


def test_tp_utest_footprint_obstacles(cuda):
    """base_local_planner/test/utest.cpp:86-110: trajectories that run or rotate the footprint into an obstacle are
    invalid (-1); the same command on a clear map is legal."""
    a, b, c = sc.tp_utest_footprint_obstacles(cuda)
    assert a == -1.0 and b == -1.0 and c >= 0.0


def test_tp_scores_every_sample_on_the_device(cuda, port):
    """3 x 20 forward samples + 2 holonomic + 20 in-place + 4 strafing + 1 back-up, all scored by one k_tp_score."""
    rng = np.random.default_rng(7)
    s = sc.dwa_scenario(rng, style="corridor")
    grid = sc.local_costmap(port, rng, ox=s["origin"][0], oy=s["origin"][1], style="corridor")
    tp = cuda.trajectory_planner(120, 120, 0.05, sc.PENTAGON)
    tp.set_costmap(grid, *s["origin"])
    tp.update_plan(s["plan"])
    before = cuda.launch_count()
    r = tp.find_best_path(s["pose"], s["vel"])
    assert cuda.launch_count() - before == 2  # the MapGrid wavefronts (one launch, two CTAs) + k_tp_score
    assert tp.last_sample_count() == 3 * 20 + 2 + 20 + 4 + 1
    assert r["cost"] >= 0 and len(r["points"]) > 0


def test_tp_heading_scoring_matches_checker(cuda, port):
    """heading_scoring_ (trajectory_planner.cpp:318-331, 372-387): line of sight to the farthest visible plan pose;
    atan2 / fmod on the device may differ from glibc in the last bit, hence the 1e-5 comparison."""
    for seed in (4, 9, 14, 19, 24, 29):
        assert_cycles_match(sc.run_tp_scenario(cuda, port, seed), sc.run_tp_scenario(port, port, seed), f"heading seed {seed}")
