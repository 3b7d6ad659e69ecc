#!/usr/bin/env python
"""GPU timing of one fast log-likelihood evaluation on bench.py's headline forest (configs[1]: 10 000 trees, 6 generations,
seed 20261018, the rule the fast mode picks):
  * the evaluation: CUDA events around ggp_loglik_device on the library's stream, median over the repetitions;
  * each kernel of it: mean device time per evaluation from torch.profiler (CUDA activities), in a run of its own, for the
    constants table (ggp_fast_consts_kernel), the generations (ggp_fast_loglik_kernel) and the reduction (ggp_reduce_kernel).
GGP_B200_LIB selects the library build, so two builds can be compared in one session.

  python tools/eval_probe.py [--trees 10000] [--reps 200] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import gfp_gaussian_process_b200 as ggp  # noqa: E402
from gfp_gaussian_process_b200 import _lib  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trees", type=int, default=10000)
    ap.add_argument("--generations", type=int, default=6)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--out")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("eval_probe: no CUDA device")
    lib = _lib.load()
    d = ggp.simulate_forest(args.trees, args.generations, seed=20261018)
    f = ggp.Forest(d)
    f.set_mode("fast")
    dp = torch.tensor(ggp.PARAMS_CONST_GAUSS, dtype=torch.float64, device="cuda").reshape(1, 11)
    out = torch.zeros(1, dtype=torch.float64, device="cuda")
    kms = np.zeros(1)

    def evaluate():
        _lib.check(lib.ggp_loglik_device(f.handle, dp.data_ptr(), 1, out.data_ptr()))

    for _ in range(20):   # warm-up: module load, upload, the rule's first pick
        evaluate()
    _lib.check(lib.ggp_sync_kernel_ms(f.handle, kms.ctypes.data_as(_lib.c_double_p)))
    ms = []
    for _ in range(args.reps):
        evaluate()
        _lib.check(lib.ggp_sync_kernel_ms(f.handle, kms.ctypes.data_as(_lib.c_double_p)))
        ms.append(float(kms[0]))
    loglik = float(out.item())

    from torch.profiler import ProfilerActivity, profile
    n_prof = 50
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n_prof):
            evaluate()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        for key in ("ggp_fast_consts_kernel", "ggp_fast_loglik_kernel", "ggp_reduce_kernel", "ggp_fill64_kernel"):
            if key in ev.key:
                k = kern.setdefault(key, [0.0, 0])
                k[0] += max(ev.self_device_time_total, ev.device_time_total)   # us
                k[1] += ev.count
    per_eval_us = {k: {"us_per_eval": v[0] / n_prof, "launches_per_eval": v[1] / n_prof} for k, v in kern.items()}
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {"lib": _lib.LIB_PATH, "gpu": smi, "n_ctp": int(d.n_ctp), "nodes": int(f.last_fast_nodes),
           "eval_ms_median": float(np.median(ms)), "eval_ms_min": float(np.min(ms)), "eval_ms_p90": float(np.percentile(ms, 90)),
           "loglik": loglik, "kernels": per_eval_us}
    f.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
