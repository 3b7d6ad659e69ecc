"""The gradient of the FAST log-likelihood on the host, without a GPU: the dual-number evaluation of ggp_fast.cuh
(csrc/ggp_dual.cuh, compiled by tests/hostcheck/gradcheck.cpp; the device gradient kernel runs the same code with FMA contraction)
against the binary128 central difference of the 16-node binary128 evaluation, and against central differences of the oracle's
strict log-likelihood (the reference's own model).  The error of direction i is scaled as |p_i| |g_i - t_i| / |loglik|."""
import os
import sys

import numpy as np
import pytest

from conftest import example_data, ROOT
from oracle.oracle_py import Oracle
import gfp_gaussian_process_b200 as ggp

sys.path.insert(0, os.path.join(ROOT, "tools"))
from fast_gate import fast_loglik  # noqa: E402
from grad_check import grad_host, grad_quad, scaled_error  # noqa: E402

QUAD_BAR = 1e-11     # against the binary128 truth
ORACLE_BAR = 1e-6    # against central differences of the reference's strict arithmetic (its rounding noise over the step)


def oracle_central_difference(data, P, rel_step=1e-4):
    o = Oracle(data)
    g = np.empty(11)
    for i in range(11):
        h = rel_step * abs(P[i])
        up, dn = P.copy(), P.copy()
        up[i] += h
        dn[i] -= h
        g[i] = (o.total_loglik(up) - o.total_loglik(dn)) / (2 * h)
    return g


def check(data, P, nodes):
    ll, g, valid = grad_host(data, P, nodes)
    fast, fvalid, _, _ = fast_loglik(data, P, n_nodes=nodes)
    q, gq, qvalid = grad_quad(data, P)
    assert valid[0] == 1 and fvalid[0] == 1 and qvalid[0] == 1
    # the value part is the fast evaluation itself
    assert abs(ll[0] - fast[0]) / abs(fast[0]) <= 1e-15
    e_quad = scaled_error(P, g[0], gq[0], q[0])
    e_orc = scaled_error(P, g[0], oracle_central_difference(data, P), q[0])
    print(f"N={nodes}: scaled error vs binary128 max {e_quad.max():.2e}, vs oracle central differences max {e_orc.max():.2e}")
    assert np.all(np.isfinite(g[0]))
    assert e_quad.max() <= QUAD_BAR
    assert e_orc.max() <= ORACLE_BAR


@pytest.mark.parametrize("noise,division,nodes", [("const", "gauss", 5), ("scaled", "binomial", 6), ("scaled", "gauss", 6), ("const", "binomial", 5)])
def test_dual_gradient_matches_binary128_and_the_oracle(noise, division, nodes):
    P = ggp.PARAMS_CONST_GAUSS if noise == "const" else ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(12, 4, params=P, noise_model=noise, division_model=division, seed=71)
    check(d, P, nodes)


def test_dual_gradient_on_the_example_data_set(golden_dir):
    data, z = example_data(golden_dir)
    check(data, np.asarray(z["params"]), 5)


def test_dual_gradient_flags_steps_outside_the_validity_range():
    """the vectors test_fast_host flags are flagged by the dual evaluation too"""
    P = ggp.PARAMS_CONST_GAUSS.copy()
    d = ggp.simulate_forest(3, 3, seed=72)
    assert grad_host(d, P, 5)[2][0] == 1
    P[4] = 2.0
    assert grad_host(d, P, 5)[2][0] == 0 and grad_host(d, P, 10)[2][0] == 0
    P[4] = 0.25
    assert grad_host(d, P, 6)[2][0] == 0 and grad_host(d, P, 8)[2][0] == 1
