#!/usr/bin/env python
"""Cost of ggp_simulate and a first look at the calibration of the fast likelihood's error bars, on one GPU:
  sim            device time of one simulation (CUDA events around its launches, ggp_last_kernel_ms; warm-up, median of --reps),
                 8 sub-steps, on the BASELINE configs[1] genealogy (10 000 trees x 6 generations, const / gauss) and on the 1 M-cell
                 target forest (15 873 trees x 6 generations, scaled / binomial), as time points per second; wall time of the
                 call with its copy-out beside it
  synthetic      synthetic.simulate_forest's host time for the configs[1] forest, for scale
  calibration    on 10 000-tree forests simulated at PARAMS_CONST_GAUSS (one per seed, root prior fixed), from the fast gradient g
                 and the exact fast Hessian H at the simulating parameters theta_0, per parameter i:
                   newton_t  (-H^-1 g)_i / sqrt(-(H^-1)_ii): the one-step Newton estimate's distance from theta_0 in units of
                             its error bar (approximately (theta_hat - theta_0) / sigma without a refit)
                   score_z   g_i / sqrt(-H_ii): the score over its standard deviation
                 both are ~ N(0, 1) over replicates when the model is right and the error bars are calibrated
The card's name, power limit and maximum SM clock are read in the same run.

  python tools/sim_probe.py [--reps 20] [--replicates 8] [--out profiles/r05_sim_probe.json]
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


def time_sim(data, P, reps, warmup=3):
    f = ggp.Forest(data)
    prior = data.init_stats()
    for s in range(warmup):
        ggp.simulate_series(f, P, seed=s, root_prior=prior, copy_out=False)
    dev, wall = [], []
    for s in range(reps):
        t0 = time.perf_counter()
        ggp.simulate_series(f, P, seed=100 + s, root_prior=prior)
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append(f.last_kernel_ms)
    r = {"n_cells": int(data.n_cells), "n_ctp": int(data.n_ctp), "launches": int(f.last_launch_count),
         "device_ms_median": float(np.median(dev)), "device_ms_min": float(np.min(dev)),
         "ctp_per_s": data.n_ctp / (np.median(dev) * 1e-3), "wall_ms_median_with_copy_out": float(np.median(wall))}
    f.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--replicates", type=int, default=8)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = {"card": card(), "substeps": 8}
    t0 = time.perf_counter()
    cfg1 = ggp.simulate_forest(10000, 6, seed=20261018)
    out["synthetic_host_s_configs1"] = time.perf_counter() - t0
    out["sim_configs1"] = time_sim(cfg1, ggp.PARAMS_CONST_GAUSS, a.reps)
    print("configs[1]:", out["sim_configs1"], "synthetic.py on the host: %.2f s" % out["synthetic_host_s_configs1"], flush=True)
    tgt = ggp.simulate_forest(15873, 6, noise_model="scaled", division_model="binomial", seed=20261018)
    out["sim_target_1m"] = time_sim(tgt, ggp.PARAMS_SCALED_BINOMIAL, a.reps)
    print("1 M cells:", out["sim_target_1m"], flush=True)
    del tgt
    P = ggp.PARAMS_CONST_GAUSS
    f = ggp.Forest(cfg1)
    prior = cfg1.init_stats()
    t, z = [], []
    for s in range(a.replicates):
        ggp.simulate_series(f, P, seed=1000 + s, root_prior=prior, copy_out=False)
        _, g, H = ggp.total_likelihood_hess(P, f)
        Hi = np.linalg.inv(H)
        t.append(-(Hi @ g) / np.sqrt(-np.diag(Hi)))
        z.append(g / np.sqrt(-np.diag(H)))
        print(f"replicate {s}: newton_t = {np.array2string(t[-1], precision=2)}  score_z = {np.array2string(z[-1], precision=2)}",
              flush=True)
    cal = {"params": ggp.PARAM_NAMES, "n_trees": 10000, "replicates": a.replicates}
    for name, v in (("newton_t", np.array(t)), ("score_z", np.array(z))):
        cal[name] = v.tolist()
        cal[name + "_mean"] = v.mean(axis=0).tolist()
        cal[name + "_sd"] = v.std(axis=0, ddof=1).tolist() if a.replicates > 1 else None
        print(name, "mean", np.array2string(v.mean(axis=0), precision=2), "sd", np.array2string(v.std(axis=0, ddof=1), precision=2))
    out["calibration"] = cal
    f.close()
    print(json.dumps({k: v for k, v in out.items() if k != "calibration"}))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
