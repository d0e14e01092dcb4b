"""The checker's reconfigure entry points (navo_dwa_reconfigure, navo_tp_reconfigure, navo_tp_set_footprint), which the
GPU tests of reconfigured planner handles compare against: a reconfigure before the first call is a handle created with
the new configuration, and one in the middle of a sequence keeps the state the reference keeps."""
import numpy as np

import scenarios as sc


def test_dwa_reconfigured_before_first_call_is_a_fresh_handle(port):
    w = sc.reconfigure_world(seed=7)
    b = dict(vx_samples=7, vy_samples=2, vth_samples=9, path_distance_bias=20.0, goal_distance_bias=30.0,
             forward_point_distance=0.5, cheat_factor=2.0, sim_time=1.2, use_dwa=0, sum_scores=1, acc_lim_x=1.5)
    ops = [("plan",), ("find",), ("follow",), ("plan",), ("find",)]
    fresh = sc.run_dwa_sequence(port, w["grid"], w["origin"], w["pose"], w["plan"], w["vel"], ops, **b)
    moved = sc.run_dwa_sequence(port, w["grid"], w["origin"], w["pose"], w["plan"], w["vel"],
                                [("reconfigure", b)] + ops, vx_samples=3, vy_samples=1, vth_samples=4)
    for x, y in zip(moved, fresh):
        assert sc.dwa_results_equal(x, y)


def test_dwa_reconfigure_keeps_latched_oscillation_flags(port):
    """Flags latched by alternating commands survive a reconfigure; the next search starts from them."""
    out = sc.run_dwa_reconfigure_case(port, "oscillation_reset")
    assert out[3]["mask"] != 0 and out[4]["mask"] & out[3]["mask"] == out[3]["mask"]
    w, create, ops = sc.dwa_case_world("oscillation_reset")
    d = port.dwa(120, 120, 0.05, **create)
    d.set_costmap(w["grid"], *w["origin"])
    d.set_plan(w["pose"], w["plan"])
    for xv in (0.3, -0.2):  # forward, then backward: forward_neg_only latches
        d.find_best_path(w["pose"], (xv, 0.0, 0.0), sc.PENTAGON)
    mask = d.oscillation_mask()
    assert mask != 0
    d.reconfigure(oscillation_reset_dist=0.001, vx_samples=9, sim_time=1.0)
    assert d.oscillation_mask() == mask


def test_tp_reconfigured_before_first_call_is_a_fresh_handle(port):
    w = sc.tp_open_world()
    b = dict(sim_time=2.0, sim_granularity=0.02, vx_samples=5, vtheta_samples=7, holonomic_robot=0, dwa=0,
             y_vels=[-0.2, 0.2], pdist_scale=0.9, max_vel_x=0.8, sim_period=0.1)
    ops = [("find",), ("follow", 0.2), ("find",)]
    fresh = sc.run_tp_sequence(port, w["grid"], w["origin"], w["pose"], w["plan"], w["vel"], ops, **b)
    moved = sc.run_tp_sequence(port, w["grid"], w["origin"], w["pose"], w["plan"], w["vel"], [("reconfigure", b)] + ops)
    assert all(sc.tp_results_equal(x, y) for x, y in zip(moved, fresh))
    fp = sc.square_footprint(0.2)
    fresh = sc.run_tp_sequence(port, w["grid"], w["origin"], w["pose"], w["plan"], w["vel"], ops, footprint=fp)
    moved = sc.run_tp_sequence(port, w["grid"], w["origin"], w["pose"], w["plan"], w["vel"], [("footprint", fp)] + ops)
    assert all(sc.tp_results_equal(x, y) for x, y in zip(moved, fresh))


def test_tp_reconfigure_keeps_latched_flags(port):
    """Reconfiguring to the very same configuration in the middle of the boxed-in run changes nothing: the latched
    strafing flags and the plan are kept; the reference's clamp of zero sample counts to one applies."""
    same = {k: {} for k in (2, 4, 7)}
    assert all(sc.tp_results_equal(x, y) for x, y in zip(sc.run_tp_boxed_scenario(port, reconfigure=same),
                                                          sc.run_tp_boxed_scenario(port)))
    w = sc.tp_open_world()
    ops = [("find",)]
    zero = sc.run_tp_sequence(port, w["grid"], w["origin"], w["pose"], w["plan"], w["vel"],
                              [("reconfigure", dict(vx_samples=0, vtheta_samples=-2))] + ops)
    one = sc.run_tp_sequence(port, w["grid"], w["origin"], w["pose"], w["plan"], w["vel"], ops, vx_samples=1,
                             vtheta_samples=1)
    assert sc.tp_results_equal(zero[0], one[0]) and np.all(zero[0]["points"][:, 1] == w["pose"][1])
