"""Per-tree scores of the FAST log-likelihood on the host, without a GPU: the dual-number evaluation of ggp_fast.cuh added into
every lineage tree (tests/hostcheck/treecheck.cpp; the device gradient kernels run the same per-cell code, then add the cells
per tree) against binary128 central differences of every tree's 16-node binary128 log-likelihood, and the sandwich algebra
of tree_scores' consumer, api.sandwich.  The error of tree t along direction i is |p_i| |s_ti - t_ti| / sum_{c in t} |ll_c|:
a tree's log-likelihood itself can come close to 0."""
import os
import sys

import numpy as np
import pytest

from conftest import ROOT
import gfp_gaussian_process_b200 as ggp
from gfp_gaussian_process_b200.api import sandwich

sys.path.insert(0, os.path.join(ROOT, "tools"))
from grad_check import grad_host, scaled_error, scaled_tree_error, tree_host, tree_quad  # noqa: E402

QUAD_BAR = 1e-13   # per tree, against the binary128 truth
SUM_BAR = 1e-15    # the trees' scores added up, against the forest's gradient (scaled as scaled_error)

COMBOS = [("const", "gauss", 5), ("scaled", "binomial", 6), ("scaled", "gauss", 6), ("const", "binomial", 5)]


@pytest.mark.parametrize("noise,division,nodes", COMBOS)
def test_tree_scores_match_binary128_per_tree(noise, division, nodes):
    P = ggp.PARAMS_CONST_GAUSS if noise == "const" else ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(30, 3, params=P, noise_model=noise, division_model=division, seed=81)
    ll, g, ab, valid = tree_host(d, P, nodes)
    q, gq, qvalid = tree_quad(d, P)
    assert valid[0] == 1 and qvalid[0] == 1
    assert ll.shape == (1, 30) and np.all(ab[0] > 0)
    e = scaled_tree_error(P, g[0], gq[0], ab[0])
    print(f"{noise}/{division} N={nodes}: per-tree scaled error vs binary128 max {e.max():.2e}")
    assert np.all(np.isfinite(g[0]))
    assert e.max() <= QUAD_BAR


@pytest.mark.parametrize("noise,division,nodes", COMBOS)
def test_tree_scores_add_up_to_the_gradient(noise, division, nodes):
    P = ggp.PARAMS_CONST_GAUSS if noise == "const" else ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(30, 4, params=P, noise_model=noise, division_model=division, seed=82)
    ll, g, _, _ = tree_host(d, P, nodes)
    total, grad, _ = grad_host(d, P, nodes)
    assert abs(ll[0].sum() - total[0]) / abs(total[0]) <= SUM_BAR * 10
    assert scaled_error(P, g[0].sum(axis=0), grad[0], total[0]).max() <= SUM_BAR


def _numpy_sandwich(H, S):
    T = S.shape[0]
    sbar = S.mean(axis=0)
    J = sum(np.outer(s - sbar, s - sbar) for s in S) * T / (T - 1)
    Hi = np.linalg.inv(H)
    return -np.diag(Hi), np.diag(Hi @ J @ Hi)


@pytest.mark.parametrize("n,T", [(1, 2), (3, 4), (5, 40), (11, 200)])
def test_sandwich_matches_a_direct_transcription(n, T):
    rng = np.random.default_rng(n * 1000 + T)
    A = rng.normal(size=(n, n))
    H = -(A @ A.T + n * np.eye(n))
    S = rng.normal(size=(T, n)) * rng.uniform(0.1, 10.0, size=n) + rng.normal(size=n)
    hv, rv = sandwich(H, S)
    hv2, rv2 = _numpy_sandwich(H, S)
    np.testing.assert_allclose(hv, hv2, rtol=1e-12)
    np.testing.assert_allclose(rv, rv2, rtol=1e-10)
    assert np.all(hv > 0) and np.all(rv >= 0)


def test_sandwich_is_centred_and_is_the_hessian_variance_for_matching_information():
    """J is centred (a common shift of every score changes nothing); with J = -H (scores whose covariance is the information)
    the sandwich is -diag(H^-1)"""
    rng = np.random.default_rng(3)
    n, T = 3, 5000
    L = np.linalg.cholesky(np.array([[4.0, 1.0, 0.5], [1.0, 3.0, 0.2], [0.5, 0.2, 2.0]]))
    S = rng.normal(size=(T, n)) @ L.T
    S -= S.mean(axis=0)
    C = S.T @ S * T / (T - 1) / 1.0
    H = -C
    hv, rv = sandwich(H, S)
    np.testing.assert_allclose(rv, hv, rtol=1e-10)
    hv2, rv2 = sandwich(H, S + np.array([5.0, -2.0, 1e3]))
    np.testing.assert_allclose(rv2, rv, rtol=1e-9)


def test_sandwich_refuses_too_few_trees():
    H = -np.eye(3)
    with pytest.raises(ValueError, match="3 lineage trees for 3 free parameters"):
        sandwich(H, np.ones((3, 3)))
    with pytest.raises(ValueError, match="1 lineage trees for 1 free parameters"):
        sandwich(-np.eye(1), np.ones((1, 1)))
    with pytest.raises(ValueError):
        sandwich(-np.eye(2), np.ones((10, 3)))
    sandwich(H, np.arange(12.0).reshape(4, 3) ** 2)   # T - 1 = n is enough
