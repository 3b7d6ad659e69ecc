#!/usr/bin/env python
"""Cost of the per-tree scores and a first look at the tree-robust (sandwich) error bars, on one GPU:
  cost         on the BASELINE configs[1] forest (10 000 trees x 6 generations, const / gauss), resident, with the 5-node rule,
               all 11 directions: device time (CUDA events around the launches, ggp_last_kernel_ms; warm-up, median of --reps) of
               ggp_loglik_grad and of ggp_loglik_tree_grad, and their wall times
  ab           with --parent-lib: ggp_loglik_grad of that library build against this one, alternating in one run (one child
               process per round and build), medians of --reps calls each
  calibration  on 10 000-tree forests simulated at PARAMS_CONST_GAUSS (one per seed, root prior fixed), evaluated at the
               simulating parameters theta_0, per parameter i: ratio robust_var / hess_var (about 1 where the model is right), and
               t_i = (-H^-1 g)_i / sqrt(var_i), the one-step Newton estimate's distance from theta_0 in units of either error bar
               (DESIGN.md 5.8), whose spread over the replicates is about 1 when that error bar is calibrated
The card's name, power limit and maximum SM clock are read in the same run.

  python tools/tree_probe.py [--reps 20] [--replicates 8] [--parent-lib PATH] [--rounds 3] [--out profiles/r06_tree_probe.json]
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
sys.path.insert(0, os.path.join(ROOT, "tools"))


def configs1():
    import gfp_gaussian_process_b200 as ggp
    return ggp.simulate_forest(10000, 6, seed=20261018)


def time_calls(fn, f, reps, warmup=3):
    for _ in range(warmup):
        fn()
    dev, wall = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append(f.last_kernel_ms)
    return {"device_ms_median": float(np.median(dev)), "device_ms_min": float(np.min(dev)), "device_ms_max": float(np.max(dev)),
            "wall_ms_median": float(np.median(wall)), "launches": int(f.last_launch_count)}


def grad_only(reps):
    """child process of the A/B: ggp_loglik_grad of the library GGP_B200_LIB names on configs[1], one JSON line"""
    import ctypes
    from gfp_gaussian_process_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in [n for n in _lib.SIGNATURES if not hasattr(lib, n)]:   # an older build lacks the newer entry points
        del _lib.SIGNATURES[name]
    import gfp_gaussian_process_b200 as ggp
    f = ggp.Forest(configs1())
    f.set_mode(5)
    P = ggp.PARAMS_CONST_GAUSS
    r = time_calls(lambda: ggp.total_likelihood_grad(P, f), f, reps)
    r["grad"] = ggp.total_likelihood_grad(P, f)[1].tolist()
    print("RESULT " + json.dumps(r), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--replicates", type=int, default=8)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--grad-only", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.grad_only:
        return grad_only(a.reps)
    import gfp_gaussian_process_b200 as ggp
    from grad_probe import card
    out = {"card": card(), "forest": "configs[1]: 10 000 trees x 6 generations, const / gauss", "nodes": 5, "directions": 11}
    if a.parent_lib:
        runs = {"parent": [], "this": []}
        for _ in range(a.rounds):
            for name, lib in (("parent", os.path.abspath(a.parent_lib)), ("this", None)):
                env = dict(os.environ)
                if lib:
                    env["GGP_B200_LIB"] = lib
                else:
                    env.pop("GGP_B200_LIB", None)
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--grad-only", "--reps", str(a.reps)], env=env,
                                   capture_output=True, text=True)
                if r.returncode:
                    sys.exit(r.stdout + r.stderr)
                res = json.loads([line for line in r.stdout.split("\n") if line.startswith("RESULT ")][0][7:])
                runs[name].append(res)
                print(f"A/B {name}: ggp_loglik_grad {res['device_ms_median']:.3f} ms (min {res['device_ms_min']:.3f})", flush=True)
        same = all(r["grad"] == runs["parent"][0]["grad"] for r in runs["parent"] + runs["this"])
        out["ab_grad"] = {k: [{kk: vv for kk, vv in r.items() if kk != "grad"} for r in v] for k, v in runs.items()}
        out["ab_grad"]["same_gradient_bits"] = same
        print("A/B gradient bits identical:", same, flush=True)
    d = configs1()
    f = ggp.Forest(d)
    f.set_mode(5)
    P = ggp.PARAMS_CONST_GAUSS
    out["n_cells"], out["n_ctp"], out["n_trees"] = int(d.n_cells), int(d.n_ctp), int(f.n_roots)
    for name, fn in (("grad", lambda: ggp.total_likelihood_grad(P, f)), ("tree_grad", lambda: ggp.tree_scores(P, f)),
                     ("grad_again", lambda: ggp.total_likelihood_grad(P, f)), ("tree_grad_again", lambda: ggp.tree_scores(P, f))):
        out[name] = time_calls(fn, f, a.reps)
        print(f"{name}: {out[name]}", flush=True)
    ll, g = ggp.total_likelihood_grad(P, f)
    tl, tg = ggp.tree_scores(P, f)[2:]
    out["tree_rows_finite"] = bool(np.all(np.isfinite(tg)) and np.all(np.isfinite(tl)))
    prior = d.init_stats()
    ratio, t_h, t_r = [], [], []
    for s in range(a.replicates):
        ggp.simulate_series(f, P, seed=1000 + s, root_prior=prior, copy_out=False)
        hv, rv, H, _ = ggp.sandwich_error_bars(P, f)
        _, g = ggp.total_likelihood_grad(P, f)
        shift = -np.linalg.solve(H, g)
        ratio.append(rv / hv)
        t_h.append(shift / np.sqrt(hv))
        t_r.append(shift / np.sqrt(rv))
        print(f"replicate {s}: robust/hess {np.array2string(ratio[-1], precision=2)}", flush=True)
    cal = {"params": ggp.PARAM_NAMES, "n_trees": int(f.n_roots), "replicates": a.replicates}
    for name, v in (("ratio_robust_over_hess", np.array(ratio)), ("newton_t_hess", np.array(t_h)), ("newton_t_robust", np.array(t_r))):
        cal[name] = v.tolist()
        cal[name + "_mean"] = v.mean(axis=0).tolist()
        cal[name + "_sd"] = v.std(axis=0, ddof=1).tolist() if a.replicates > 1 else None
        print(name, "mean", np.array2string(v.mean(axis=0), precision=2), "sd",
              np.array2string(v.std(axis=0, ddof=1), precision=2) if a.replicates > 1 else "-", flush=True)
    out["calibration"] = cal
    f.close()
    print(json.dumps({k: v for k, v in out.items() if k not in ("calibration", "ab_grad")}))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
