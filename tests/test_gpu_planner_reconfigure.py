"""Reconfigured planner handles: navgpu_dwa_reconfigure, navgpu_tp_reconfigure and navgpu_tp_set_footprint (what every
dynamic_reconfigure change of a running move_base reaches) on live handles against the CPU checker driven through the
same calls.  A fresh handle never holds what these keep across a configuration change: cached velocity samples and
grown buffers, plans adjusted with the old configuration, latched oscillation / escape flags, the last result.

Comparisons are those of test_gpu_dwa.py and test_gpu_tp.py: bit-exact where integers decide (grids, sample counts,
indices, flags, velocities, the number of trajectory points), 1e-5 relative where CUDA's cos/sin may differ from
glibc's in the last bit.
"""
import numpy as np
import pytest

from navigation_b200.api import NavGpuError
import scenarios as sc

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def assert_dwa_records_match(got, want, what):
    assert len(got) == len(want)
    for c, (x, y) in enumerate(zip(got, want)):
        if "checks" in y:
            assert x["mask"] == y["mask"] and np.allclose(x["checks"], y["checks"], rtol=RTOL, atol=0), (
                f"{what} record {c}: checks {x['checks']} vs {y['checks']}")
            continue
        assert sc.dwa_results_equal(x, y, rtol=RTOL), (
            f"{what} record {c}: best {x['best_index']} vs {y['best_index']}, cost {x['cost']} vs {y['cost']}, "
            f"n {x['n_samples']}/{x['n_scored']} vs {y['n_samples']}/{y['n_scored']}, mask {x['mask']} vs {y['mask']}")


def assert_tp_records_match(got, want, what):
    assert len(got) == len(want)
    for c, (x, y) in enumerate(zip(got, want)):
        assert sc.tp_results_equal(x, y, rtol=RTOL), (
            f"{what} cycle {c}: cost {x['cost']} vs {y['cost']}, v ({x['xv']}, {x['yv']}, {x['thetav']}) vs "
            f"({y['xv']}, {y['yv']}, {y['thetav']}), flags {x['flags']} vs {y['flags']}, "
            f"points {len(x['points'])} vs {len(y['points'])}")


# ---- DWAPlanner -------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", sorted(sc.dwa_reconfigure_cases()))
def test_dwa_reconfigure_sequence_matches_checker(cuda, port, case):
    assert_dwa_records_match(sc.run_dwa_reconfigure_case(cuda, case), sc.run_dwa_reconfigure_case(port, case), case)


def test_dwa_samples_across_the_inline_bound_match_a_fresh_handle(cuda, port):
    """navgpu_dwa_get_samples after every reconfigure of the sample counts equals what a handle created with that
    configuration enumerates at the same pose and velocity (the staged samples cached on the device are replaced)."""
    w, create, ops = sc.dwa_case_world("samples_inline_staged")
    d = cuda.dwa(120, 120, 0.05, **create)
    d.set_costmap(w["grid"], *w["origin"])
    sizes = []
    for op in ops:
        if op[0] == "reconfigure":
            d.reconfigure(**op[1])
        elif op[0] == "plan":
            d.set_plan(w["pose"], w["plan"])
        elif op[0] == "find":
            r = d.find_best_path(w["pose"], w["vel"], sc.PENTAGON, want_costs=False)
            fresh = cuda.dwa(120, 120, 0.05, **{k: getattr(d.cfg, k) for k, _ in d.cfg._fields_})
            fresh.set_costmap(w["grid"], *w["origin"])
            fresh.set_plan(w["pose"], w["plan"])
            rf = fresh.find_best_path(w["pose"], w["vel"], sc.PENTAGON, want_costs=False)
            got, want = d.samples(), fresh.samples()
            assert all(np.array_equal(a, b) for a, b in zip(got, want))
            assert (r["best_index"], r["cost"], r["n_samples"]) == (rf["best_index"], rf["cost"], rf["n_samples"])
            sizes.append(sum(len(a) for a in got))
    assert [s > 640 for s in sizes] == [False, True, False, True]


def test_dwa_trajectory_cost_function_after_reconfigure(cuda, port):
    """navgpu_dwa_prepare + navgpu_dwa_score_trajectories on a handle reconfigured from another configuration: the
    winner of the checker's search, handed back as an explicit trajectory, scores the checker's search cost."""
    w = sc.reconfigure_world(seed=5, style="empty")
    new = dict(path_distance_bias=20.0, goal_distance_bias=40.0, occdist_scale=0.05, forward_point_distance=0.5,
               sum_scores=1, vx_samples=6, vy_samples=1, vth_samples=9)
    ref = port.dwa(120, 120, 0.05, vx_samples=3, vy_samples=1, vth_samples=5)
    ref.set_costmap(w["grid"], *w["origin"])
    ref.set_plan(w["pose"], w["plan"])
    ref.reconfigure(**new)
    want = ref.find_best_path(w["pose"], w["vel"], sc.PENTAGON)
    assert want["ok"]
    d = cuda.dwa(120, 120, 0.05, vx_samples=3, vy_samples=1, vth_samples=5)
    d.set_costmap(w["grid"], *w["origin"])
    d.set_plan(w["pose"], w["plan"])
    d.reconfigure(**new)
    d.prepare()
    v = (want["xv"], want["yv"], want["thetav"])
    costs, terms = d.score_trajectories([want["points"], want["points"][:1]], [v, v], sc.PENTAGON, want_terms=True)
    assert costs[0] == pytest.approx(want["cost"], rel=RTOL) and costs[0] == np.add.reduce(terms[0])
    assert costs[1] >= 0
    for k in range(4):
        assert np.array_equal(d.grid(k), ref.grid(k))


def test_dwa_sharded_handles_reconfigured_alike(cuda, port):
    """Two handles on one GPU joined by navgpu_dwa_shard_connect_local, reconfigured identically between cycles: the
    sharded winner is the single reconfigured handle's, and the checker's."""
    w = sc.reconfigure_world(seed=3)
    create = dict(vx_samples=20, vy_samples=1, vth_samples=20, max_vel_y=0.0, min_vel_y=0.0)
    steps = [dict(vx_samples=60, vy_samples=3, vth_samples=60, max_vel_y=0.1, min_vel_y=-0.1, acc_lim_x=20.0,
                  acc_lim_theta=20.0), dict(vx_samples=7, vth_samples=11, path_distance_bias=20.0, sim_time=1.2),
             dict(vx_samples=300, vy_samples=1, vth_samples=300, max_vel_y=0.0, min_vel_y=0.0)]
    handles = []
    for api in (cuda, cuda, cuda, port):
        d = api.dwa(120, 120, 0.05, **create)
        d.set_costmap(w["grid"], *w["origin"])
        handles.append(d)
    whole, ranks, ref = handles[0], handles[1:3], handles[3]
    cuda.shard_connect_local(ranks)
    for over in steps:
        for d in handles:
            d.set_plan(w["pose"], w["plan"])
            d.reconfigure(**over)
        rw = whole.find_best_path(w["pose"], w["vel"], sc.PENTAGON, want_costs=False)
        for d in ranks:
            d.find_best_path_sharded_async(w["pose"], w["vel"], sc.PENTAGON)
        for r, o in enumerate(d.sharded_collect(w["pose"]) for d in ranks):
            assert (o["best_index"], o["cost"], o["n_samples"]) == (rw["best_index"], rw["cost"], rw["n_samples"]), r
            assert np.array_equal(o["points"], rw["points"])
        rr = ref.find_best_path(w["pose"], w["vel"], sc.PENTAGON)
        assert rr["best_index"] == rw["best_index"] and rr["cost"] == pytest.approx(rw["cost"], rel=RTOL)
        assert all(d.oscillation_mask() == whole.oscillation_mask() == ref.oscillation_mask() for d in ranks)


# ---- legacy TrajectoryPlanner -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", sorted(sc.tp_reconfigure_cases()))
def test_tp_reconfigure_sequence_matches_checker(cuda, port, case):
    got, want = sc.run_tp_reconfigure_case(cuda, case), sc.run_tp_reconfigure_case(port, case)
    assert_tp_records_match(got, want, case)
    world, create, _, lengthening = sc.tp_reconfigure_cases()[case]
    stride = sc.tp_points_stride(cuda.trajectory_planner(120, 120, 0.05, sc.PENTAGON, **create).cfg)
    # the lengthening cases return trajectories longer than the creation configuration's, in full
    assert (max(len(r["points"]) for r in want) > stride) == lengthening


def test_tp_escape_and_oscillation_kept_across_reconfigure(cuda, port):
    """Strafing flags latched against the walls of run_tp_boxed_scenario, then backing up; reconfigures in the middle
    of both keep that state, on the device as in the checker."""
    over = {4: dict(oscillation_reset_dist=0.02, sim_time=1.5), 7: dict(escape_reset_dist=0.3, escape_reset_theta=0.5,
                                                                       backup_vel=-0.2, vtheta_samples=7)}
    got, want = sc.run_tp_boxed_scenario(cuda, reconfigure=over), sc.run_tp_boxed_scenario(port, reconfigure=over)
    assert_tp_records_match(got, want, "boxed")
    assert got[5]["flags"] & 4 and got[-1]["flags"] & 4  # stuck_left_strafe stays latched across both
    assert got[6]["xv"] < 0 and got[-1]["xv"] == pytest.approx(-0.2)  # backing up, at the reconfigured backup_vel


REFUSED = {
    "n_y_vels_9": dict(n_y_vels=9),
    "sim_time_0": dict(sim_time=0.0),
    "million_steps": dict(sim_granularity=1e-7),
}


@pytest.mark.parametrize("what", sorted(REFUSED) + ["footprint_17"])
def test_tp_refused_change_leaves_the_handle_as_it_was(cuda, what):
    """A refused reconfigure or footprint returns an error; the handle's next findBestPath is that of an untouched
    twin, and the wrapper keeps its configuration."""
    w = sc.tp_open_world()
    handles = []
    for _ in range(2):
        tp = cuda.trajectory_planner(120, 120, 0.05, sc.PENTAGON, vx_samples=4, vtheta_samples=9)
        tp.set_costmap(w["grid"], *w["origin"])
        tp.update_plan(w["plan"])
        tp.find_best_path(w["pose"], w["vel"])
        handles.append(tp)
    tp, twin = handles
    before = bytes(tp.cfg)
    with pytest.raises(NavGpuError):
        if what == "footprint_17":
            tp.set_footprint([(0.3 * np.cos(a), 0.3 * np.sin(a)) for a in np.linspace(0, 2 * np.pi, 17, endpoint=False)])
        else:
            tp.reconfigure(**REFUSED[what])
    assert bytes(tp.cfg) == before
    for pose in (w["pose"], (1.2, 3.1, 0.3)):
        a, b = tp.find_best_path(pose, w["vel"]), twin.find_best_path(pose, w["vel"])
        a["grids"] = [tp.grid(0), tp.grid(1)]
        b["grids"] = [twin.grid(0), twin.grid(1)]
        a["scores"] = b["scores"] = np.zeros(1)
        assert sc.tp_results_equal(a, b, rtol=0.0)
