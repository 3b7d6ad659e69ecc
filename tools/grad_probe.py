#!/usr/bin/env python
"""Cost of the gradient of the fast log-likelihood on the BASELINE configs[1] forest (10 000 trees x 6 generations), resident:
  eval      one fast evaluation (ggp_loglik, the rule "fast" picks)
  grad      the 11-direction gradient (ggp_loglik_grad, same rule)
  stencil   the 23 vectors of a central-difference gradient (centre + 2 x 11 shifts) as one ggp_loglik call, same rule
Each is warmed up, then timed over --reps calls: device time from the handle's CUDA events (ggp_last_kernel_ms) and wall time
around the call (every call ends in a stream synchronise).  Medians are printed with the card's name, power limit and
maximum SM clock, read in the same run.

  python tools/grad_probe.py [--reps 20] [--out profiles/r03_grad_probe.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import gfp_gaussian_process_b200 as ggp  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed(fn, forest, reps, warmup):
    for _ in range(warmup):
        fn()
    dev, wall = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append(forest.last_kernel_ms)
    return {"device_ms_median": float(np.median(dev)), "device_ms_min": float(np.min(dev)), "wall_ms_median": float(np.median(wall)),
            "launches": int(forest.last_launch_count)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(10000, 6, seed=20261018)
    f = ggp.Forest(d)
    f.set_mode("fast")
    ggp.total_likelihood(P, f)
    n = f.last_fast_nodes
    f.set_mode(n)
    h = 1e-5 * np.abs(P)
    vecs = np.repeat(P[None, :], 23, axis=0)
    for i in range(11):
        vecs[2 * i, i] += h[i]
        vecs[2 * i + 1, i] -= h[i]
    res = {"card": card(), "forest": {"n_cells": int(d.n_cells), "n_ctp": int(d.n_ctp), "n_generations": int(f.n_generations)},
           "nodes": int(n), "reps": a.reps}
    res["eval"] = timed(lambda: ggp.total_likelihood(P, f), f, a.reps, a.warmup)
    res["grad"] = timed(lambda: ggp.total_likelihood_grad(P, f), f, a.reps, a.warmup)
    res["stencil"] = timed(lambda: ggp.total_likelihood(vecs, f), f, a.reps, a.warmup)
    res["grad_over_eval"] = res["grad"]["device_ms_median"] / res["eval"]["device_ms_median"]
    res["grad_over_stencil"] = res["grad"]["device_ms_median"] / res["stencil"]["device_ms_median"]
    f.close()
    print(f"card: {res['card']}")
    print(f"configs[1]: {d.n_cells} cells, {d.n_ctp} points, {n}-node rule, {a.reps} timed calls each (medians)")
    for k in ("eval", "grad", "stencil"):
        r = res[k]
        print(f"  {k:8s} device {r['device_ms_median']:8.3f} ms (min {r['device_ms_min']:.3f})  wall {r['wall_ms_median']:8.3f} ms  "
              f"launches {r['launches']}")
    print(f"  gradient / one evaluation {res['grad_over_eval']:.2f}, gradient / 23-vector stencil {res['grad_over_stencil']:.2f}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
        print("wrote", a.out)


if __name__ == "__main__":
    main()
