"""Generates the golden fixtures in this directory from the REFERENCE's own compiled code (oracle/_ref/libnavref.so).

Run with NAVIGATION_REFERENCE naming the reference's sources:   python tests/golden/make_golden.py
Inputs are regenerated from the seed by tests/scenarios.py; only the reference's outputs are stored.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import pyoracle as po  # noqa: E402
import scenarios as sc  # noqa: E402

COSTMAP_SEEDS = [0, 1, 2, 3, 5, 8, 13, 21]
COSTMAP_TIEFREE_SEEDS = [100, 101, 102, 103, 104, 105]
DWA_SEEDS = [0, 1, 3, 4, 9, 20, 32]
TP_SEEDS = [0, 2, 4, 5, 7, 9, 11, 16, 23, 31, 9000]  # 9000 = sc.run_tp_boxed_scenario (golden_util.TP_BOXED)


def main():
    ref = po.load("reference")
    assert ref.name == "reference"
    for tie_free, seeds in ((False, COSTMAP_SEEDS), (True, COSTMAP_TIEFREE_SEEDS)):
        for seed in seeds:
            tr = sc.run_costmap_scenario(ref, seed, tie_free=tie_free)
            d = {}
            for c, (w, m, o, org) in enumerate(tr):
                d[f"w{c}"] = np.array(w, np.int32)
                d[f"m{c}"] = m
                d[f"o{c}"] = o
                d[f"org{c}"] = np.array(org)
            np.savez_compressed(os.path.join(HERE, f"costmap_{'tf' if tie_free else 'any'}_{seed}.npz"), **d)
    for seed in DWA_SEEDS:
        out = sc.run_dwa_scenario(ref, ref, seed)
        d = {}
        for c, r in enumerate(out):
            d[f"scalars{c}"] = np.array([r["ok"], r["cost"], r["xv"], r["yv"], r["thetav"], r["best_index"],
                                         r["n_samples"], r["n_scored"], r["mask"]], np.float64)
            d[f"costs{c}"] = r["costs"]
            d[f"points{c}"] = r["points"]
            for k in range(4):
                d[f"grid{c}_{k}"] = r["grids"][k].astype(np.int32)
        np.savez_compressed(os.path.join(HERE, f"dwa_{seed}.npz"), **d)
    port = po.load("port")  # the local costmaps come from the restatement, as in the tests
    for seed in TP_SEEDS:
        out = sc.run_tp_boxed_scenario(ref) if seed == 9000 else sc.run_tp_scenario(ref, port, seed)
        d = {}
        for c, r in enumerate(out):
            d[f"scalars{c}"] = np.array([r["cost"], r["xv"], r["yv"], r["thetav"], r["flags"]], np.float64)
            d[f"points{c}"] = r["points"]
            d[f"scores{c}"] = r["scores"]
            for k in range(2):
                d[f"grid{c}_{k}"] = r["grids"][k].astype(np.int32)
        np.savez_compressed(os.path.join(HERE, f"tp_{seed}.npz"), **d)
    # plan preprocessing: the reference's own transformGlobalPlan / prunePlan (oracle/_ref/libgoalref.so)
    import test_plan_preprocessing as tpp
    goal = po.GoalRef()
    for seed in tpp.GOLDEN_PLAN_SEEDS:
        plans, robots, tfs, thr = tpp.random_batch(np.random.default_rng(seed), 64)
        outs = goal.plans_transform(plans, robots, tfs, thr)
        np.savez_compressed(os.path.join(HERE, f"plan_{seed}.npz"), counts=np.array([len(o) for o in outs]),
                            xyz=np.concatenate(outs), pruned=goal.plans_prune(plans, robots))
    print("golden fixtures written to", HERE)


if __name__ == "__main__":
    main()
