"""The gradient of the FAST log-likelihood on the GPU (ggp_loglik_grad, ggp_group_loglik_grad, total_likelihood_grad,
num_hessian_grad): the device kernels against the host build of the same dual-number code (tests/hostcheck/gradcheck.cpp), the
fast log-likelihood, and central differences of it; reproducibility, chunking, the re-run ladder and the error rows."""
import os
import sys

import numpy as np
import pytest

from conftest import same_bits, example_data, max_rel, ROOT
from oracle.oracle_py import Oracle
import gfp_gaussian_process_b200 as ggp
from gfp_gaussian_process_b200 import _lib

sys.path.insert(0, os.path.join(ROOT, "tools"))
from grad_check import grad_host, scaled_error  # noqa: E402

pytestmark = pytest.mark.gpu

COMBOS = [("const", "gauss"), ("scaled", "binomial"), ("scaled", "gauss"), ("const", "binomial")]


def params_of(noise):
    return ggp.PARAMS_CONST_GAUSS if noise == "const" else ggp.PARAMS_SCALED_BINOMIAL


def raw_grad(f, vecs, dirs=None):
    """ggp_loglik_grad through the C ABI: (rc, loglik, grad, [(cell, t_index)])"""
    lib = _lib.load()
    p = np.ascontiguousarray(vecs, dtype=np.float64).reshape(-1, 11)
    n = p.shape[0]
    d = None if dirs is None else np.ascontiguousarray(dirs, dtype=np.int32)
    nd = 11 if d is None else d.size
    ll, g = np.empty(n), np.empty((n, nd))
    nan = (_lib.NanInfo * n)()
    rc = lib.ggp_loglik_grad(f.handle, p.ctypes.data_as(_lib.c_double_p), n, None if d is None else d.ctypes.data_as(_lib.c_int32_p),
                             nd, ll.ctypes.data_as(_lib.c_double_p), g.ctypes.data_as(_lib.c_double_p), nan)
    return rc, ll, g, [(nan[v].cell, nan[v].t_index) for v in range(n)]


@pytest.mark.parametrize("noise,division", COMBOS)
def test_device_gradient_matches_the_host_dual_evaluation(noise, division):
    P = params_of(noise)
    d = ggp.simulate_forest(60, 5, params=P, noise_model=noise, division_model=division, seed=51)
    vecs = np.stack([P, P * 1.03, P * 0.96])
    f = ggp.Forest(d)
    f.set_mode(6)
    ll, g = ggp.total_likelihood_grad(vecs, f)
    assert f.last_fast_nodes == 6 and g.shape == (3, 11)
    fast = ggp.total_likelihood(vecs, f)
    hl, hg, valid = grad_host(d, vecs, 6)
    assert valid.all()
    for i in range(3):
        e = scaled_error(vecs[i], g[i], hg[i], hl[i])
        print(f"{noise}/{division} vector {i}: scaled error vs host {e.max():.2e}, value vs fast loglik {abs(ll[i] - fast[i]) / abs(fast[i]):.2e}")
        assert e.max() <= 1e-13
        assert abs(ll[i] - fast[i]) / abs(fast[i]) <= 1e-14
    # the mode picks its rule as fast ggp_loglik does; the strict mode of the handle does not change the arithmetic
    f.set_mode("strict")
    ll_s, g_s = ggp.total_likelihood_grad(vecs, f)
    n_auto = f.last_fast_nodes
    assert n_auto in (4, 5, 6, 8, 10)
    f.set_mode(n_auto)
    assert same_bits(ggp.total_likelihood_grad(vecs, f)[1], g_s)
    # the sign of the objective
    nl, ng = ggp.total_likelihood_grad(P, f, negative=True)
    assert nl == -ggp.total_likelihood_grad(P, f)[0] and ng.shape == (11,)
    f.close()


def test_direction_subsets_are_columns_of_the_full_gradient_and_calls_repeat_bit_for_bit():
    P = ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(50, 5, params=P, noise_model="scaled", division_model="binomial", seed=53)
    vecs = np.stack([P, P * 1.05])
    f = ggp.Forest(d)
    ll, g = ggp.total_likelihood_grad(vecs, f)
    ll2, g2 = ggp.total_likelihood_grad(vecs, f)
    assert same_bits(ll, ll2) and same_bits(g, g2)
    for dirs in ([4], [10, 0, 3], [0, 1, 2, 3, 4, 5, 6]):
        lls, gs = ggp.total_likelihood_grad(vecs, f, dirs=dirs)
        assert same_bits(gs, g[:, dirs]) and same_bits(lls, ll)
    for bad in ([11], [-1], [2, 2]):
        with pytest.raises(_lib.GgpError) as e:
            ggp.total_likelihood_grad(vecs, f, dirs=bad)
        assert e.value.code == _lib.GGP_ERR_BAD_ARG
    lib = _lib.load()
    p = np.ascontiguousarray(P)
    out, gr = np.empty(1), np.empty(11)
    dirs = np.zeros(1, dtype=np.int32)
    for nd, dp in ((0, dirs.ctypes.data_as(_lib.c_int32_p)), (5, None)):
        assert lib.ggp_loglik_grad(f.handle, p.ctypes.data_as(_lib.c_double_p), 1, dp, nd, out.ctypes.data_as(_lib.c_double_p),
                                   gr.ctypes.data_as(_lib.c_double_p), None) == _lib.GGP_ERR_BAD_ARG
    f.close()


def test_vectors_outside_every_rule_and_nan_vectors_get_nan_rows():
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(30, 4, seed=52)
    wide = P.copy()
    wide[4] = 2.0   # gamma_q = 2: the exponent varies by 7 over a step, no rule covers it
    bad = P.copy()
    bad[7] = -1.0   # negative measurement variance: NaN in the reference
    f = ggp.Forest(d)
    strict = ggp.total_likelihood(np.stack([P, wide, bad]), f, raise_on_nan=False)
    o = Oracle(d)
    assert np.isnan(o.total_loglik(bad))
    rc0, ll0, g0, _ = raw_grad(f, P)
    assert rc0 == _lib.GGP_OK and np.all(np.isfinite(g0))
    # all three kinds in one batch: every row filled, BAD_ARG names the uncovered vector
    rc, ll, g, nan = raw_grad(f, np.stack([P, wide, P * 1.01, bad]))
    assert rc == _lib.GGP_ERR_BAD_ARG and "vector(s) 1 " in _lib.load().ggp_last_error().decode()
    assert same_bits(ll[0], ll0) and same_bits(g[0], g0[0]) and np.all(np.isfinite(g[2]))
    assert ll[1] == strict[1] and np.all(np.isnan(g[1])) and nan[1] == (-1, -1)
    assert np.isnan(ll[3]) and np.all(np.isnan(g[3])) and nan[3] == o.nan
    assert nan[0] == (-1, -1) and nan[2] == (-1, -1)
    assert f.last_strict_reruns == 2
    # NaN vectors only: GGP_ERR_NAN, and LikelihoodNaN from Python
    rc, ll, g, nan = raw_grad(f, np.stack([P, bad]))
    assert rc == _lib.GGP_ERR_NAN and same_bits(g[0], g0[0]) and np.all(np.isnan(g[1])) and nan[1] == o.nan
    with pytest.raises(ggp.LikelihoodNaN) as e:
        ggp.total_likelihood_grad(np.stack([P, bad]), f)
    assert e.value.vec_index == 1 and (e.value.cell, e.value.t_index) == o.nan
    with pytest.raises(_lib.GgpError):
        ggp.total_likelihood_grad(wide, f)
    # gamma_q = 0.25 leaves a 5- and 6-node rule but not the 8-node one: the ladder gives the 8-node gradient
    mid = P.copy()
    mid[4] = 0.25
    f.set_mode(5)
    rc, ll5, g5, _ = raw_grad(f, mid)
    assert rc == _lib.GGP_OK and f.last_strict_reruns == 0
    f.set_mode(8)
    rc, ll8, g8, _ = raw_grad(f, mid)
    assert rc == _lib.GGP_OK and same_bits(g5, g8) and same_bits(ll5, ll8)
    f.close()


def test_vector_chunks_give_the_same_bits(monkeypatch):
    P = ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(40, 5, params=P, noise_model="scaled", division_model="binomial", seed=54)
    vecs = P * np.exp(np.random.default_rng(3).uniform(-0.05, 0.05, size=(5, 11)))
    f = ggp.Forest(d)
    ll, g = ggp.total_likelihood_grad(vecs, f)
    f.close()
    # one vector's 11 evaluations fit the budget, two do not: five chunks
    monkeypatch.setenv("GGP_B200_STATE_BUDGET", str(d.n_cells * 14 * 2 * 8 * 11 + 8))
    fc = ggp.Forest(d)
    llc, gc = ggp.total_likelihood_grad(vecs, fc)
    monkeypatch.delenv("GGP_B200_STATE_BUDGET")
    assert same_bits(llc, ll) and same_bits(gc, g)
    fc.close()


def test_gradient_after_upload_series_equals_a_fresh_forest(monkeypatch):
    monkeypatch.setenv("GGP_B200_UPLOAD_CHUNKS", "3")
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(40, 4, seed=31)
    f = ggp.Forest(d)
    ggp.total_likelihood_grad(P, f)
    rng = np.random.default_rng(5)
    x2 = d.log_length + rng.normal(0, 1e-3, d.n_ctp)
    g2 = d.fp * (1 + rng.normal(0, 1e-3, d.n_ctp))
    f.upload_series(None, x2.ctypes.data, g2.ctypes.data)
    vecs = np.stack([P, P * 1.01])
    ll, g = ggp.total_likelihood_grad(vecs, f)
    d2 = ggp.LineageData(cell_offset=d.cell_offset, parent=d.parent, time=d.time, log_length=x2, fp=g2, segment=d.segment,
                         noise_model=d.noise_model, division_model=d.division_model, fp_auto=d.fp_auto)
    f2 = ggp.Forest(d2)
    ll2, gg2 = ggp.total_likelihood_grad(vecs, f2)
    assert same_bits(ll, ll2) and same_bits(g, gg2)
    f.close()
    f2.close()


def test_other_calls_return_the_same_bits_after_a_gradient():
    P = ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(40, 5, params=P, noise_model="scaled", division_model="binomial", seed=55)
    vecs = np.stack([P, P * 1.02, P * 0.98])
    f = ggp.Forest(d)
    before_s = ggp.total_likelihood(vecs, f, per_cell=True)
    f.set_mode("fast")
    before_f = ggp.total_likelihood(vecs, f, per_cell=True)
    n_before = f.last_fast_nodes
    f.set_mode("strict")
    ggp.total_likelihood_grad(np.tile(P, (7, 1)), f)
    after_s = ggp.total_likelihood(vecs, f, per_cell=True)
    f.set_mode("fast")
    ggp.total_likelihood_grad(P, f)
    after_f = ggp.total_likelihood(vecs, f, per_cell=True)
    assert same_bits(before_s[0], after_s[0]) and same_bits(before_s[1], after_s[1])
    assert same_bits(before_f[0], after_f[0]) and same_bits(before_f[1], after_f[1]) and f.last_fast_nodes == n_before
    f.close()


def test_group_gradient_agrees_with_the_single_forest():
    P = ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(40, 5, params=P, noise_model="scaled", division_model="binomial", seed=56)
    vecs = np.stack([P, P * 1.03])
    f = ggp.Forest(d)
    f.set_mode(6)
    ll, g = ggp.total_likelihood_grad(vecs, f)
    grp = ggp.ForestGroup(d, [0, 0])
    grp.set_mode(6)
    llg, gg = ggp.total_likelihood_grad(vecs, grp)
    assert max_rel(llg, ll) <= 1e-13
    for i in range(2):
        assert np.max(scaled_error(vecs[i], gg[i], g[i], ll[i])) <= 1e-13
    lls, gs = ggp.total_likelihood_grad(vecs, grp, dirs=[2, 5])
    assert same_bits(gs, gg[:, [2, 5]]) and same_bits(lls, llg)
    grp.close()
    f.close()


def test_gradient_at_configs1_size_matches_device_central_differences():
    """BASELINE configs[1] (10 000 trees x 6 generations): the gradient is finite and agrees with central differences of the fast
    log-likelihood (22 shifted vectors and the centre in one call, step 1e-5 relative, the same rule)"""
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(10000, 6, seed=20261018)
    f = ggp.Forest(d)
    ll, g = ggp.total_likelihood_grad(P, f)
    assert np.all(np.isfinite(g)) and f.last_strict_reruns == 0
    f.set_mode(f.last_fast_nodes)
    h = 1e-5 * np.abs(P)
    vecs = np.repeat(P[None, :], 23, axis=0)
    for i in range(11):
        vecs[2 * i, i] += h[i]
        vecs[2 * i + 1, i] -= h[i]
    fl = ggp.total_likelihood(vecs, f)
    cd = (fl[0:22:2] - fl[1:22:2]) / (2 * h)
    e = scaled_error(P, g, cd, ll)
    print(f"configs[1]: loglik {ll!r}, scaled error vs central differences max {e.max():.2e}")
    assert abs(fl[22] - ll) / abs(ll) <= 1e-14
    assert e.max() <= 1e-6
    f.close()


def test_num_hessian_grad_is_symmetric_and_matches_num_hessian_ll(golden_dir):
    """num_hessian_ll's diagonal is a second difference with step 2 h: the log-likelihood's rounding noise e |ll| becomes up to
    e |ll| / h^2 in it.  On the fast log-likelihood (e ~ 1e-15) that is below the 1e-3 bar on every diagonal entry; on the
    strict one (e up to 2.3e-11 on this data set, the reference's own envelope) it dominates where |H_ii| h^2 is small against
    |ll| (var_dg: 0.87), so there the bar is 1e-3 plus that noise bound."""
    data, z = example_data(golden_dir)
    P = np.asarray(z["params"])
    idx = list(range(11))
    eps = 1e-3
    f = ggp.Forest(data)
    H = ggp.num_hessian_grad(f, P, idx, eps)
    assert H.shape == (11, 11) and same_bits(H, H.T) and np.all(np.isfinite(H))
    ll = ggp.total_likelihood(P, f)
    h = np.maximum(np.abs(P) * eps, 1e-12)
    strict = ggp.num_hessian_ll(f, P, idx, eps)
    f.set_mode("fast")
    fast = ggp.num_hessian_ll(f, P, idx, eps)
    r_fast = np.abs(np.diag(H) - np.diag(fast)) / np.abs(np.diag(fast))
    r_strict = np.abs(np.diag(H) - np.diag(strict)) / np.abs(np.diag(strict))
    noise = 2.3e-11 * abs(ll) / h ** 2 / np.abs(np.diag(H))
    print("example data set, diagonal of num_hessian_grad against num_hessian_ll (relative):")
    print(f"  fast   {np.array2string(r_fast, precision=1)}")
    print(f"  strict {np.array2string(r_strict, precision=1)}")
    print(f"  strict second-difference noise bound {np.array2string(noise, precision=1)}")
    assert r_fast.max() <= 1e-3
    assert np.all(r_strict <= 1e-3 + noise)
    f.close()
