#!/usr/bin/env python
"""Generates tests/golden/ref_wrapper_vectors.npz from the REFERENCE'S OWN WRAPPER SOURCE: likelihood.h, predictions.h,
correlation_tree.h, Gaussians.h and moma_input.h compiled unmodified over oracle/eigen_shim (oracle/ref_wrappers.cpp ->
oracle/_ref/libggp_ref_wrappers.so).  Run in the build container, where /root/reference is mounted; the GPU box and any
machine without the reference only see the committed file (tests/test_ref_wrappers.py::test_oracle_matches_wrapper_golden).

Cases (all tiny, so that the dense joints matrix of the reference stays small):
  four model combinations on 2 trees x 3 generations; a ragged two-segment forest (single-daughter mothers, one-point
  cells, parents stored after daughters, fp_auto != 0); per case: genealogy, init statistics, log-likelihood of three
  successive evaluations (fresh, then carried, SURVEY.md H3) with the per-cell sums of the first, the three prediction
  passes, the cell state the backward pass leaves, and every joint at tolerance 1e-10.
  The example data set: log-likelihood (fresh, second, third evaluation), per-cell sums and the predictions at every 97th point.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
OUT = os.path.join(ROOT, "tests", "golden", "ref_wrapper_vectors.npz")

import gfp_gaussian_process_b200 as ggp  # noqa: E402
from oracle.oracle_py import RefWrappers  # noqa: E402
from conftest import ragged_forest, example_data  # noqa: E402


def wrapper_cases():
    """(name, data, parameter sets [n_seg][11])"""
    out = []
    for noise, division in (("const", "gauss"), ("scaled", "binomial"), ("scaled", "gauss"), ("const", "binomial")):
        P = ggp.PARAMS_CONST_GAUSS if noise == "const" else ggp.PARAMS_SCALED_BINOMIAL
        d = ggp.simulate_forest(2, 3, params=P, noise_model=noise, division_model=division, seed=21, pts_range=(3, 6))
        out.append((f"{noise}_{division}", d, np.asarray([P])))
    P2 = np.stack([ggp.PARAMS_SCALED_BINOMIAL, ggp.PARAMS_SCALED_BINOMIAL * np.array([1, 1, 1, 2, 1, 1, 1, 1, 1, 1, 1.])])
    out.append(("ragged_segments", ragged_forest(), P2))
    return out


def run_case(r, P, joints=True, keep_records=True):
    res = {}
    res["d1"], res["d2"] = r.daughters()
    res["init_f"], res["init_r"] = r.init_stats()
    if P.shape[0] == 1:
        res["cell_ll"] = r.total_loglik(P[0], per_cell=True)
        r.reset()
        res["loglik_chain"] = np.array([r.total_loglik(P[0], fresh=False), r.total_loglik(P[0] * 1.01, fresh=False),
                                        r.total_loglik(P[0], fresh=False)])
    pr = r.predictions(P)
    for k in ("forward", "backward", "prediction"):
        res[k + "_mean"], res[k + "_cov"] = pr[k]
    res["state_mean"], res["state_cov"] = r.state()
    if joints:
        n, row, col, rec = r.joints(1e-10, 1 << 20)
        assert n <= 1 << 20
        # a SHA-256 of the records' bytes in (row, col) order (bit-exact check); the records themselves only on request
        order = np.lexsort((col, row))
        res["j_row"], res["j_col"] = row[order], col[order]
        res["j_sha256"] = np.frombuffer(hashlib.sha256(np.ascontiguousarray(rec[order]).tobytes()).digest(), dtype=np.uint8)
        if keep_records:
            res["j_rec"] = rec[order]
    return res


def main():
    z = {}
    for name, d, P in wrapper_cases():
        r = RefWrappers(d)
        for k, v in run_case(r, P, keep_records=False).items():   # the hash keeps the file under 1 MB
            z[f"{name}/{k}"] = v
        print(name, "cells", d.n_cells, "ctp", d.n_ctp, "joints", len(z[f"{name}/j_row"]))
        r.close()
    data, ez = example_data(os.path.join(ROOT, "tests", "golden"))
    r = RefWrappers(data)
    P = np.asarray(ez["params"])
    z["example/cell_ll"] = r.total_loglik(P, per_cell=True)
    r.reset()
    z["example/loglik_chain"] = np.array([r.total_loglik(P, fresh=False) for _ in range(3)])
    pr = r.predictions([P])
    for k in ("forward", "backward", "prediction"):
        z[f"example/{k}_mean"], z[f"example/{k}_cov"] = pr[k][0][::97], pr[k][1][::97]
    print("example", z["example/loglik_chain"])
    np.savez_compressed(OUT, **z)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
