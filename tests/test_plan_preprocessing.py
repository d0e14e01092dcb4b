"""Plan preprocessing (SURVEY.md 8f-4): base_local_planner::transformGlobalPlan / prunePlan
(base_local_planner/src/goal_functions.cpp:68-174).

CPU part: the checker's restatement (oracle/plan_restated.h) on hand-worked cases and against the REFERENCE'S OWN
functions -- goal_functions.cpp compiled unmodified into oracle/_ref/libgoalref.so against a tf stand-in
(oracle/shim_tf; tf is not in the reference tree, so the transform arithmetic itself stays "parity unpinned", the loops
do not) -- plus golden vectors generated from it (tests/golden/plan_*.npz).  GPU part: the batched kernels (navgpu_plans_transform / navgpu_plans_prune, one warp per plan)
against the restatement on random batches, bit for bit."""
import numpy as np
import pytest

IDENTITY = [1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0]


def line_plan(n, x0=0.0, step=0.5):
    return np.stack([x0 + step * np.arange(n), np.zeros(n), np.zeros(n)], 1)


def test_transform_keeps_the_first_pose_beyond_the_threshold(port):
    """Poses every 0.5 m along x, robot at x = 5, threshold 2: the first pose within 2 m is x = 3 (index 6); poses are
    pushed while the PREVIOUS one was within the threshold, so x = 7.5 (index 15, 2.5 m away) is the last one kept
    (goal_functions.cpp:135-149)."""
    first, outs = port.plans_transform([line_plan(40)], [(5.0, 0.0)], [IDENTITY], [2.0])
    assert first[0] == 6 and len(outs[0]) == 10
    assert outs[0][0, 0] == 3.0 and outs[0][-1, 0] == 7.5


def test_transform_applies_the_rigid_transform(port):
    c, s = np.cos(0.3), np.sin(0.3)
    tf = [c, -s, 0, s, c, 0, 0, 0, 1, 10.0, -4.0, 0.5]
    plan = line_plan(5)
    plan[:, 1] = [0.0, 0.1, 0.2, 0.1, 0.0]
    first, outs = port.plans_transform([plan], [(1.0, 0.0)], [tf], [100.0])
    assert first[0] == 0 and len(outs[0]) == 5
    want = np.stack([c * plan[:, 0] + -s * plan[:, 1] + 0 * plan[:, 2] + 10.0,
                     s * plan[:, 0] + c * plan[:, 1] + 0 * plan[:, 2] - 4.0, plan[:, 2] + 0.5], 1)
    assert np.allclose(outs[0], want, rtol=0, atol=1e-15)


def test_transform_edge_cases(port):
    plan = line_plan(10)
    # robot far from every pose: nothing is kept, first = plan size
    first, outs = port.plans_transform([plan], [(100.0, 0.0)], [IDENTITY], [2.0])
    assert first[0] == 10 and len(outs[0]) == 0
    # everything within the threshold: the whole plan
    first, outs = port.plans_transform([plan], [(2.0, 0.0)], [IDENTITY], [50.0])
    assert first[0] == 0 and len(outs[0]) == 10
    # the plan re-enters the threshold later: only the first stretch (and the pose that left it) is kept
    loop = np.array([[0, 0, 0], [1, 0, 0], [5, 0, 0], [6, 0, 0], [1, 0.5, 0], [0, 0.5, 0]], float)
    first, outs = port.plans_transform([loop], [(0.0, 0.0)], [IDENTITY], [2.0])
    assert first[0] == 0 and len(outs[0]) == 3
    # an empty plan
    first, outs = port.plans_transform([np.zeros((0, 3))], [(0.0, 0.0)], [IDENTITY], [2.0])
    assert first[0] == 0 and len(outs[0]) == 0


def test_prune_erases_up_to_the_first_waypoint_within_one_metre(port):
    plan = line_plan(20)
    assert list(port.plans_prune([plan, plan, plan, plan], [(5.0, 0.0), (0.0, 0.0), (100.0, 0.0), (5.0, 1.0)])) == \
        [9, 0, 20, 20]  # 4.5 is the first with d^2 < 1; strictly less: (5, 1) is exactly 1 m from x = 5


def random_batch(rng, n):
    plans, robots, tfs, thr = [], [], [], []
    for _ in range(n):
        m = int(rng.integers(0, 400))
        t = np.linspace(0, rng.uniform(2, 30), max(m, 1))[:m]
        plan = np.stack([rng.uniform(-20, 20) + t * np.cos(0.2 * t), rng.uniform(-20, 20) + t * np.sin(0.3 * t),
                         rng.uniform(-0.1, 0.1, m)], 1)
        plans.append(plan)
        if m and rng.random() < 0.8:
            k = int(rng.integers(0, m))
            robots.append(plan[k, :2] + rng.uniform(-1.5, 1.5, 2))
        else:
            robots.append(rng.uniform(-40, 40, 2))
        yaw, q = rng.uniform(-3.1, 3.1), rng.uniform(-0.2, 0.2)
        cz, sz, cx, sx = np.cos(yaw), np.sin(yaw), np.cos(q), np.sin(q)
        rot = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]]) @ np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
        tfs.append(list(rot.reshape(9)) + list(rng.uniform(-50, 50, 3)))
        thr.append(rng.choice([3.0, 2.0, 0.5, 10.0]))
    return plans, np.array(robots), np.array(tfs), np.array(thr)


@pytest.mark.gpu
@pytest.mark.parametrize("seed,n", [(1, 1), (2, 37), (3, 1000), (4, 4096)])
def test_batched_kernels_match_the_restatement(cuda, port, seed, n):
    rng = np.random.default_rng(seed)
    plans, robots, tfs, thr = random_batch(rng, n)
    f_gpu, o_gpu = cuda.plans_transform(plans, robots, tfs, thr)
    f_ref, o_ref = port.plans_transform(plans, robots, tfs, thr)
    assert np.array_equal(f_gpu, f_ref)
    for k, (a, b) in enumerate(zip(o_gpu, o_ref)):
        assert a.shape == b.shape and np.array_equal(a, b), f"plan {k}: transformed poses differ"
    assert np.array_equal(cuda.plans_prune(plans, robots), port.plans_prune(plans, robots))
    assert sum(len(o) for o in o_ref) > 0 or n == 1


@pytest.mark.gpu
def test_batched_kernels_edge_cases(cuda, port):
    plan = line_plan(10)
    loop = np.array([[0, 0, 0], [1, 0, 0], [5, 0, 0], [6, 0, 0], [1, 0.5, 0], [0, 0.5, 0]], float)
    nan_plan = line_plan(6)
    nan_plan[3, 0] = np.nan
    plans = [plan, plan, loop, np.zeros((0, 3)), nan_plan, line_plan(100, step=0.01)]
    robots = [(100.0, 0.0), (2.0, 0.0), (0.0, 0.0), (0.0, 0.0), (0.0, 0.0), (0.5, 0.0)]
    tfs = [IDENTITY] * 6
    thr = [2.0, 50.0, 2.0, 2.0, 5.0, 0.25]
    f_gpu, o_gpu = cuda.plans_transform(plans, robots, tfs, thr)
    f_ref, o_ref = port.plans_transform(plans, robots, tfs, thr)
    assert np.array_equal(f_gpu, f_ref) and [len(o) for o in o_gpu] == [len(o) for o in o_ref] == [0, 10, 3, 0, 4, 52]
    for a, b in zip(o_gpu, o_ref):
        assert np.array_equal(a, b, equal_nan=True)
    assert np.array_equal(cuda.plans_prune(plans, robots), port.plans_prune(plans, robots))


def reference_goal_functions():
    from oracle import pyoracle
    if not pyoracle.GoalRef.available():
        if pyoracle.reference_dir():
            pyoracle.make("goalref")
        else:
            pytest.skip("oracle/_ref/libgoalref.so not present (needs NAVIGATION_REFERENCE to build)")
    return pyoracle.GoalRef()


@pytest.mark.parametrize("seed,n", [(11, 50), (12, 400)])
def test_restatement_equals_the_reference_functions(port, seed, n):
    """The restated loops against base_local_planner::transformGlobalPlan / prunePlan themselves: the kept poses (which
    poses, how many, their transformed positions) and the number of pruned way-points, bit for bit."""
    ref = reference_goal_functions()
    rng = np.random.default_rng(seed)
    plans, robots, tfs, thr = random_batch(rng, n)
    _, o_port = port.plans_transform(plans, robots, tfs, thr)
    o_ref = ref.plans_transform(plans, robots, tfs, thr)
    for k, (a, b) in enumerate(zip(o_port, o_ref)):
        assert a.shape == b.shape and np.array_equal(a, b), f"plan {k}: {a.shape} vs {b.shape}"
    assert np.array_equal(port.plans_prune(plans, robots), ref.plans_prune(plans, robots))
    assert sum(len(o) for o in o_ref) > 0


GOLDEN_PLAN_SEEDS = [21, 22, 23]


@pytest.mark.parametrize("seed", GOLDEN_PLAN_SEEDS)
def test_restatement_equals_the_golden_vectors(port, seed):
    import os
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", f"plan_{seed}.npz")
    g = np.load(path)
    plans, robots, tfs, thr = random_batch(np.random.default_rng(seed), 64)
    first, outs = port.plans_transform(plans, robots, tfs, thr)
    assert np.array_equal(np.array([len(o) for o in outs]), g["counts"])
    assert np.array_equal(np.concatenate(outs) if sum(map(len, outs)) else np.zeros((0, 3)), g["xyz"])
    assert np.array_equal(port.plans_prune(plans, robots), g["pruned"])


@pytest.mark.gpu
@pytest.mark.parametrize("seed", GOLDEN_PLAN_SEEDS)
def test_batched_kernels_equal_the_golden_vectors(cuda, seed):
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", f"plan_{seed}.npz"))
    plans, robots, tfs, thr = random_batch(np.random.default_rng(seed), 64)
    first, outs = cuda.plans_transform(plans, robots, tfs, thr)
    assert np.array_equal(np.array([len(o) for o in outs]), g["counts"])
    assert np.array_equal(np.concatenate(outs), g["xyz"])
    assert np.array_equal(cuda.plans_prune(plans, robots), g["pruned"])
