#!/usr/bin/env python
"""Cost of the exact Hessian of the fast log-likelihood on the BASELINE configs[1] forest (10 000 trees x 6 generations), resident:
  eval           one fast evaluation (ggp_loglik, the rule "fast" picks)
  grad           the 11-direction gradient (ggp_loglik_grad, same rule)
  hess           the 11-parameter Hessian (ggp_loglik_hess, same rule): 66 evaluations; one vector's state (14 GB) exceeds the
                 default 8 GB budget, so they run in direction ranges
  hess_16gb      the same with GGP_B200_STATE_BUDGET = 16 GB: all 66 evaluations in one launch sequence
  num_hess_grad  num_hessian_grad at epsilon 1e-5: central differences of the gradient, 22 vectors in one call
  num_hess_ll    the command line's error bars before --exact_errors: three num_hessian_ll stencils (epsilon 5e-2, 1e-2, 5e-3) of
                 4 n^2 = 484 vectors each, in the fast mode with the same rule and in the strict mode (three calls each)
Each is warmed up, then timed over --reps calls: device time from the handle's CUDA events (ggp_last_kernel_ms, summed over the
calls of one repetition) and wall time around it (every call ends in a stream synchronise).  Medians are printed with the card's
name, power limit and maximum SM clock, read in the same run.

  python tools/hess_probe.py [--reps 10] [--out profiles/r04_hess_probe.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import gfp_gaussian_process_b200 as ggp  # noqa: E402
from grad_probe import card  # noqa: E402


def timed(calls, forest, reps, warmup):
    """calls: functions run one after the other as one repetition"""
    for _ in range(warmup):
        for fn in calls:
            fn()
    dev, wall = [], []
    for _ in range(reps):
        ms = 0.0
        t0 = time.perf_counter()
        for fn in calls:
            fn()
            ms += forest.last_kernel_ms
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append(ms)
    return {"device_ms_median": float(np.median(dev)), "device_ms_min": float(np.min(dev)), "wall_ms_median": float(np.median(wall)),
            "launches_last_call": int(forest.last_launch_count)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    P = ggp.PARAMS_CONST_GAUSS
    idx = list(range(11))
    d = ggp.simulate_forest(10000, 6, seed=20261018)
    f = ggp.Forest(d)
    f.set_mode("fast")
    ggp.total_likelihood(P, f)
    n = f.last_fast_nodes
    f.set_mode(n)
    os.environ["GGP_B200_STATE_BUDGET"] = str(16 << 30)
    f16 = ggp.Forest(d)
    del os.environ["GGP_B200_STATE_BUDGET"]
    f16.set_mode(n)
    res = {"card": card(), "forest": {"n_cells": int(d.n_cells), "n_ctp": int(d.n_ctp), "n_generations": int(f.n_generations)},
           "nodes": int(n), "reps": a.reps}
    res["eval"] = timed([lambda: ggp.total_likelihood(P, f)], f, a.reps, a.warmup)
    res["grad"] = timed([lambda: ggp.total_likelihood_grad(P, f)], f, a.reps, a.warmup)
    res["hess"] = timed([lambda: ggp.total_likelihood_hess(P, f)], f, a.reps, a.warmup)
    res["hess_16gb"] = timed([lambda: ggp.total_likelihood_hess(P, f16)], f16, a.reps, a.warmup)
    assert all(np.array_equal(x, y) for x, y in zip(ggp.total_likelihood_hess(P, f), ggp.total_likelihood_hess(P, f16)))
    f16.close()
    res["num_hess_grad"] = timed([lambda: ggp.num_hessian_grad(f, P, idx, 1e-5)], f, a.reps, a.warmup)
    stencils = [lambda e=e: ggp.num_hessian_ll(f, P, idx, e) for e in (5e-2, 1e-2, 5e-3)]
    res["num_hess_ll_fast"] = timed(stencils, f, max(2, a.reps // 4), 1)
    f.set_mode("strict")
    res["num_hess_ll_strict"] = timed(stencils, f, max(2, a.reps // 4), 1)
    f.close()
    for k in ("grad", "hess", "hess_16gb", "num_hess_grad", "num_hess_ll_fast", "num_hess_ll_strict"):
        res[k]["over_eval"] = res[k]["device_ms_median"] / res["eval"]["device_ms_median"]
    print(f"card: {res['card']}")
    print(f"configs[1]: {d.n_cells} cells, {d.n_ctp} points, {n}-node rule, medians of timed repetitions")
    for k in ("eval", "grad", "hess", "hess_16gb", "num_hess_grad", "num_hess_ll_fast", "num_hess_ll_strict"):
        r = res[k]
        print(f"  {k:18s} device {r['device_ms_median']:10.3f} ms (min {r['device_ms_min']:.3f})  wall {r['wall_ms_median']:10.3f} ms  "
              f"= {r.get('over_eval', 1.0):7.1f} evaluations")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
        print("wrote", a.out)


if __name__ == "__main__":
    main()
