"""Digests of what the CPU restatement (oracle/libnavoracle.so) computes on the cases that test_oracle_vs_reference.py,
test_oracle_tie_variants.py and test_plan_preprocessing.py compare live against the reference's own compiled code.

The live comparisons need the reference's sources (NAVIGATION_REFERENCE) and skip without them; the golden fixtures
of make_golden.py hold the reference's outputs for a subset of these seeds only.  The digests in
golden/restatement_digests.json pin the restatement on every case of those live comparisons, so a change to the
checker that the GPU tests compare against is caught without the reference: where the reference is given, the live
tests show the restatement equal to it on exactly these cases, and a restatement that keeps these digests keeps that.

Regenerate (only after such a change has been checked against the reference):   python tests/restatement_snapshots.py
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import scenarios as sc  # noqa: E402

DIGESTS = os.path.join(HERE, "golden", "restatement_digests.json")


def digest(obj):
    """sha256 over the exact bits of (nested dicts / lists / tuples of) arrays and scalars, with dtypes and shapes."""
    h = hashlib.sha256()

    def feed(x):
        if isinstance(x, dict):
            for k in sorted(x):
                h.update(repr(k).encode())
                feed(x[k])
        elif isinstance(x, (list, tuple)):
            h.update(f"seq{len(x)}".encode())
            for v in x:
                feed(v)
        else:
            a = np.ascontiguousarray(np.asarray(x))
            h.update(f"{a.dtype.str}{a.shape}".encode())
            h.update(a.tobytes())
    feed(obj)
    return h.hexdigest()


def c1_salt(api):
    """test_inflation_larger_map_port_equals_reference: 400x400 @0.05, R = 11, 1% salt-and-pepper."""
    g = sc.random_layer(np.random.default_rng(7), 400, 400, "salt")
    cm = api.costmap(400, 400, 0.05)
    s = cm.add_grid_layer(0)
    cm.add_inflation_layer(0.55, 10.0)
    cm.set_footprint(sc.square_footprint())
    cm.set_grid_layer(s, g)
    cm.update_map()
    return cm.get()


def check_trajectory(api):
    """test_check_trajectory_restatement_matches_reference (the local maps come from the same checker)."""
    outs = []
    for seed in range(6):
        s = sc.dwa_scenario(np.random.default_rng(seed))
        grid = sc.local_costmap(api, np.random.default_rng(seed + 1000), ox=s["origin"][0], oy=s["origin"][1],
                                style=s["style"])
        d = api.dwa(120, 120, 0.05, vx_samples=5, vy_samples=1, vth_samples=7)
        d.set_costmap(grid, *s["origin"])
        d.set_plan(s["pose"], s["plan"])
        d.find_best_path(s["pose"], s["vel"], sc.PENTAGON)
        costs = [d.check_trajectory(s["pose"], s["vel"], v, sc.PENTAGON)
                 for v in [(0.3, 0.0, 0.2), (0.55, 0.0, -1.0), (0.0, 0.0, 0.0), (0.05, 0.0, 0.1), (0.5, 0.1, 0.9),
                           (2.0, 0.0, 0.0)]]
        outs.append((costs, d.oscillation_mask()))
    return outs


def tie_world(kind, radius):
    """test_tie_worlds: the restatement in the reference's own heap order."""
    def run(api):
        from test_gpu_costmap import world_from_kind
        from test_oracle_tie_variants import inflate
        return inflate(api, world_from_kind(kind, 400, 1), radius, "reference")[0]
    return run


def blocked_three_seeds(api):
    """test_blocked_propagation_three_seeds."""
    from test_oracle_tie_variants import inflate
    g = np.zeros((60, 60), np.uint8)
    for dx, dy in ((3, 3), (4, 1), (0, 5)):
        g[20 + dy, 21 + dx] = 254
    return inflate(api, g, 0.5, "reference", scaling=3.0, half=0.1)[0]


def plans(seed, n):
    """test_restatement_equals_the_reference_functions: transformGlobalPlan / prunePlan on a random batch."""
    def run(api):
        from test_plan_preprocessing import random_batch
        p, robots, tfs, thr = random_batch(np.random.default_rng(seed), n)
        return api.plans_transform(p, robots, tfs, thr)[1], api.plans_prune(p, robots)
    return run


def cases():
    out = {}
    for seed in range(40):
        out[f"costmap_{seed}"] = lambda api, s=seed: sc.run_costmap_scenario(api, s)
    for seed in range(24):
        out[f"dwa_{seed}"] = lambda api, s=seed: sc.run_dwa_scenario(api, api, s)
    out["c1_salt"] = c1_salt
    out["check_trajectory"] = check_trajectory
    for seed in range(200, 230):
        out[f"voxel_{seed}"] = lambda api, s=seed: sc.run_voxel_scenario(api, s)[0]
    for seed in range(52):  # 40-51: the seeds test_gpu_tp.py compares with the reference only
        out[f"tp_{seed}"] = lambda api, s=seed: sc.run_tp_scenario(api, api, s)
    out["tp_boxed"] = sc.run_tp_boxed_scenario
    out["tp_edge_cases"] = lambda api: sc.run_tp_edge_cases(api, api)
    out["tp_utest_footprint_obstacles"] = sc.tp_utest_footprint_obstacles
    for kind in ("axis1", "ring", "salt", "diag3", "diag1"):
        for radius in (0.55, 1.0):
            out[f"tie_{kind}_{radius}"] = tie_world(kind, radius)
    out["blocked_three_seeds"] = blocked_three_seeds
    out["plans_11"] = plans(11, 50)
    out["plans_12"] = plans(12, 400)
    return out


def stored():
    with open(DIGESTS) as f:
        return json.load(f)


if __name__ == "__main__":
    from oracle import pyoracle
    port = pyoracle.load("port")
    with open(DIGESTS, "w") as f:
        json.dump({name: digest(run(port)) for name, run in cases().items()}, f, indent=1, sort_keys=True)
        f.write("\n")
    print("digests written to", DIGESTS)
