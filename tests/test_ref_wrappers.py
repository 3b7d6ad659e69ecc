"""The oracle (oracle/ggp_oracle.cpp, the restatement every GPU parity test compares with) against the REFERENCE'S OWN
WRAPPER SOURCE: likelihood.h, predictions.h, correlation_tree.h, Gaussians.h, moma_input.h compiled unmodified over
oracle/eigen_shim (oracle/ref_wrappers.cpp -> oracle/_ref/libggp_ref_wrappers.so).  Bit for bit: genealogy, init statistics,
log-likelihood (fresh and carried), per-cell sums, forward / backward / combined predictions, the cell state the backward
pass leaves, and every joint.  What stays an assumption is how Eigen 3.3 evaluates the dense kernels (the shim's header
lists them: E1-E5); the reference's own logic is no longer transcribed.

Live tests need the build, which needs the reference's sources (oracle/Makefile, REF); the golden test, and the five
small live cases, run everywhere on the fixture tools/make_wrapper_golden.py made from that build.  CPU only."""
import hashlib
import os
import sys

import numpy as np
import pytest

from conftest import same_bits, example_data, ragged_forest, ROOT
from oracle.oracle_py import Oracle, ref_wrappers, RefWrappers
import gfp_gaussian_process_b200 as ggp

sys.path.insert(0, os.path.join(ROOT, "tools"))
from make_wrapper_golden import wrapper_cases, run_case  # noqa: E402

live = pytest.mark.skipif(ref_wrappers() is None, reason="oracle/_ref/libggp_ref_wrappers.so needs /root/reference")


def oracle_case(d, P, joints=True):
    """the quantities of make_wrapper_golden.run_case from the oracle"""
    o = Oracle(d)
    res = {"d1": np.asarray(d.daughter1), "d2": np.asarray(d.daughter2)}
    res["init_f"], res["init_r"] = o.init_stats()
    if P.shape[0] == 1:
        res["cell_ll"] = o.total_loglik(P[0], per_cell=True)[1]
        o.reset()
        res["loglik_chain"] = np.array([o.total_loglik(P[0], fresh=False), o.total_loglik(P[0] * 1.01, fresh=False),
                                        o.total_loglik(P[0], fresh=False)])
    pr = o.predictions(P)
    for k in ("forward", "backward", "prediction"):
        res[k + "_mean"], res[k + "_cov"] = pr[k]
    res["state_mean"], res["state_cov"] = o.cell_mean.copy(), o.cell_cov.copy()
    if joints:
        n, row, col, rec = o.joints(1e-10, 1 << 20)
        order = np.lexsort((col, row))
        res["j_row"], res["j_col"], res["j_rec"] = row[order], col[order], rec[order]
        res["j_sha256"] = np.frombuffer(hashlib.sha256(np.ascontiguousarray(rec[order]).tobytes()).digest(), dtype=np.uint8)
    return res


def assert_same(got, want, what):
    for k, w in want.items():
        g = got[k]
        if np.asarray(w).dtype.kind == "f":
            assert same_bits(g, w), f"{what}: {k}"
        else:
            assert np.array_equal(g, w), f"{what}: {k}"


@pytest.mark.parametrize("case", range(5))
def test_oracle_matches_the_reference_wrappers_live(case, golden_dir):
    """against the reference-wrapper build where it exists, else against that build's committed outputs for the same case"""
    name, d, P = wrapper_cases()[case]
    if ref_wrappers() is None:
        z = np.load(os.path.join(golden_dir, "ref_wrapper_vectors.npz"))
        want = {k.split("/", 1)[1]: z[k] for k in z.files if k.startswith(name + "/")}
        assert "j_sha256" in want
    else:
        r = RefWrappers(d)
        want = run_case(r, P)
        r.close()
    assert_same(oracle_case(d, P), want, name)


@live
@pytest.mark.parametrize("noise,division,seed", [("const", "gauss", 31), ("scaled", "binomial", 32), ("scaled", "gauss", 33), ("const", "binomial", 34)])
def test_oracle_matches_the_reference_wrappers_on_larger_forests(noise, division, seed):
    """6 trees x 4 generations, the size of the GPU joints parity test (9 000 joints, rows of 280 columns)"""
    P = ggp.PARAMS_CONST_GAUSS if noise == "const" else ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(6, 4, params=P, noise_model=noise, division_model=division, seed=seed, pts_range=(4, 8))
    r = RefWrappers(d)
    assert_same(oracle_case(d, np.asarray([P])), run_case(r, np.asarray([P])), f"{noise}/{division}")
    r.close()


@live
def test_oracle_matches_the_reference_wrappers_on_the_example_data_set(golden_dir):
    """config 1's data: total of three successive evaluations (the reference's one running sum in depth-first order,
    history dependent), per-cell sums, and all 22 065 x 3 predictions"""
    data, z = example_data(golden_dir)
    P = np.asarray(z["params"])
    o, r = Oracle(data), RefWrappers(data)
    assert same_bits(o.total_loglik(P, per_cell=True)[1], r.total_loglik(P, per_cell=True))
    o.reset(); r.reset()
    for _ in range(3):
        assert o.total_loglik(P, fresh=False) == r.total_loglik(P, fresh=False)
    po, pr = o.predictions([P]), r.predictions([P])
    for k in ("forward", "backward", "prediction"):
        assert same_bits(po[k][0], pr[k][0]) and same_bits(po[k][1], pr[k][1]), k
    ms, cs = r.state()
    assert same_bits(ms, o.cell_mean) and same_bits(cs, o.cell_cov)
    r.close()


def test_oracle_matches_wrapper_golden(golden_dir):
    """same comparison against the committed outputs of the reference-wrapper build (runs without /root/reference)"""
    z = np.load(os.path.join(golden_dir, "ref_wrapper_vectors.npz"))
    for name, d, P in wrapper_cases():
        want = {k.split("/", 1)[1]: z[k] for k in z.files if k.startswith(name + "/")}
        assert {"forward_mean", "state_cov", "j_row", "j_sha256"} <= set(want)
        assert_same(oracle_case(d, P), want, name)
    data, ez = example_data(golden_dir)
    P = np.asarray(ez["params"])
    o = Oracle(data)
    assert same_bits(o.total_loglik(P, per_cell=True)[1], z["example/cell_ll"])
    o.reset()
    assert same_bits([o.total_loglik(P, fresh=False) for _ in range(3)], z["example/loglik_chain"])
    pr = o.predictions([P])
    for k in ("forward", "backward", "prediction"):
        assert same_bits(pr[k][0][::97], z[f"example/{k}_mean"]) and same_bits(pr[k][1][::97], z[f"example/{k}_cov"]), k
