"""The Hessian of the FAST log-likelihood on the host, without a GPU: the second-order Taylor evaluation of ggp_fast.cuh
(GgpTaylor2, csrc/ggp_dual.cuh, compiled by tests/hostcheck/hesscheck.cpp with the device's directions, scales and unscaling;
the device kernels run the same code with FMA contraction) against binary128 second differences of the 16-node binary128
evaluation, which share no code with the Taylor numbers, and against central differences of the host dual gradient.
The error of entry (i, j) is scaled as |p_i| |p_j| |H_ij - T_ij| / |loglik|.  Polarization subtracts terms of size
s_i^2 |H_ii|, so its rounding error is about that ratio to |loglik| times the double epsilon; the tests print the ratio."""
import os
import sys

import numpy as np
import pytest

from conftest import example_data, ROOT
import gfp_gaussian_process_b200 as ggp

sys.path.insert(0, os.path.join(ROOT, "tools"))
from fast_gate import fast_loglik  # noqa: E402
from grad_check import grad_host, hess_host, hess_quad, polarization_ratio, scaled_error, scaled_hess_error  # noqa: E402

QUAD_BAR = 1e-10     # against the binary128 second differences
CD_BAR = 1e-6        # against central differences of the host dual gradient (step 1e-5 relative)


def central_difference_of_gradient(data, P, dirs, nodes, rel_step=1e-5):
    """H[:, j] = (g(x + h_j e_j) - g(x - h_j e_j)) / (2 h_j) of the host dual gradient, rows and columns over dirs"""
    h = rel_step * np.abs(P[dirs])
    vecs = np.repeat(P[None, :], 2 * len(dirs), axis=0)
    for k, i in enumerate(dirs):
        vecs[2 * k, i] += h[k]
        vecs[2 * k + 1, i] -= h[k]
    _, g, valid = grad_host(data, vecs, nodes)
    assert valid.all()
    g = g[:, dirs]
    return ((g[0::2] - g[1::2]) / (2 * h[:, None])).T


def check(data, P, nodes, dirs=None):
    d = list(range(11)) if dirs is None else list(dirs)
    ll, g, H, valid = hess_host(data, P, nodes, dirs=d)
    fast, fvalid, _, _ = fast_loglik(data, P, n_nodes=nodes)
    _, gd, gvalid = grad_host(data, P, nodes)
    q, Hq, qvalid = hess_quad(data, P, dirs=d)
    assert valid[0] == 1 and fvalid[0] == 1 and gvalid[0] == 1 and qvalid[0] == 1
    H, g = H[0], g[0]
    assert np.all(np.isfinite(H)) and np.array_equal(H, H.T)
    # the value part is the fast evaluation, the gradient part the dual gradient
    assert abs(ll[0] - fast[0]) / abs(fast[0]) <= 1e-15
    e_grad = scaled_error(P[d], g, gd[0][d], ll[0])
    e_quad = scaled_hess_error(P, d, H, Hq[0], q[0])
    e_cd = scaled_hess_error(P, d, H, central_difference_of_gradient(data, P, d, nodes), q[0])
    ratio = polarization_ratio(P, d, H, ll[0])
    print(f"N={nodes} dirs={d}: scaled Hessian error vs binary128 max {e_quad.max():.2e}, vs central differences of the gradient "
          f"max {e_cd.max():.2e}; gradient part vs dual gradient {e_grad.max():.2e}; s_i^2 |H_ii| / |loglik| max {ratio.max():.2e}")
    assert e_grad.max() <= 1e-15
    assert e_quad.max() <= QUAD_BAR
    assert e_cd.max() <= CD_BAR


@pytest.mark.parametrize("noise,division,nodes", [("const", "gauss", 5), ("scaled", "binomial", 6), ("scaled", "gauss", 6), ("const", "binomial", 5)])
def test_taylor2_hessian_matches_binary128_and_gradient_differences(noise, division, nodes):
    P = ggp.PARAMS_CONST_GAUSS if noise == "const" else ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(12, 4, params=P, noise_model=noise, division_model=division, seed=71)
    check(d, P, nodes)


def test_taylor2_hessian_on_the_example_data_set(golden_dir):
    """a direction subset: all 11 take 243 binary128 evaluations of the data set; the subset couples a rate (gamma_lambda), a
    mean (mean_q), the measurement noise (var_x) and a division noise (var_dg)"""
    data, z = example_data(golden_dir)
    check(data, np.asarray(z["params"]), 5, dirs=[1, 3, 7, 10])


def test_taylor2_flags_steps_outside_the_validity_range():
    """the vectors test_dual_gradient_flags_steps_outside_the_validity_range flags are flagged by the Taylor evaluation too"""
    P = ggp.PARAMS_CONST_GAUSS.copy()
    d = ggp.simulate_forest(3, 3, seed=72)
    dirs = [0, 4]
    assert hess_host(d, P, 5, dirs)[3][0] == 1
    P[4] = 2.0
    assert hess_host(d, P, 5, dirs)[3][0] == 0 and hess_host(d, P, 10, dirs)[3][0] == 0
    P[4] = 0.25
    assert hess_host(d, P, 6, dirs)[3][0] == 0 and hess_host(d, P, 8, dirs)[3][0] == 1
