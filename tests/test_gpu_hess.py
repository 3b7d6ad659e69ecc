"""The exact Hessian of the FAST log-likelihood on the GPU (ggp_loglik_hess, ggp_group_loglik_hess, total_likelihood_hess and
the command line's --exact_errors): the device kernels against the host build of the same GgpTaylor2 code
(tests/hostcheck/hesscheck.cpp), the fast log-likelihood and its gradient; symmetry, reproducibility, direction subsets,
chunking, the re-run ladder and the error rows."""
import os
import sys

import numpy as np
import pytest

from conftest import same_bits, max_rel, ROOT
from oracle.oracle_py import Oracle
import gfp_gaussian_process_b200 as ggp
from gfp_gaussian_process_b200 import _lib
from test_gpu_cli import write_inputs, write_params, run, read_table

sys.path.insert(0, os.path.join(ROOT, "tools"))
from grad_check import hess_host, scaled_error, scaled_hess_error  # noqa: E402

pytestmark = pytest.mark.gpu

COMBOS = [("const", "gauss"), ("scaled", "binomial"), ("scaled", "gauss"), ("const", "binomial")]


def params_of(noise):
    return ggp.PARAMS_CONST_GAUSS if noise == "const" else ggp.PARAMS_SCALED_BINOMIAL


def raw_hess(f, vecs, dirs=None):
    """ggp_loglik_hess through the C ABI: (rc, loglik, grad, hess, [(cell, t_index)])"""
    lib = _lib.load()
    p = np.ascontiguousarray(vecs, dtype=np.float64).reshape(-1, 11)
    n = p.shape[0]
    d = None if dirs is None else np.ascontiguousarray(dirs, dtype=np.int32)
    nd = 11 if d is None else d.size
    ll, g, h = np.empty(n), np.empty((n, nd)), np.empty((n, nd, nd))
    nan = (_lib.NanInfo * n)()
    rc = lib.ggp_loglik_hess(f.handle, p.ctypes.data_as(_lib.c_double_p), n, None if d is None else d.ctypes.data_as(_lib.c_int32_p),
                             nd, ll.ctypes.data_as(_lib.c_double_p), g.ctypes.data_as(_lib.c_double_p),
                             h.ctypes.data_as(_lib.c_double_p), nan)
    return rc, ll, g, h, [(nan[v].cell, nan[v].t_index) for v in range(n)]


@pytest.mark.parametrize("noise,division", COMBOS)
def test_device_hessian_matches_the_host_taylor_evaluation(noise, division):
    P = params_of(noise)
    d = ggp.simulate_forest(30, 4, params=P, noise_model=noise, division_model=division, seed=61)
    vecs = np.stack([P, P * 1.03])
    f = ggp.Forest(d)
    f.set_mode(6)
    ll, g, H = ggp.total_likelihood_hess(vecs, f)
    assert f.last_fast_nodes == 6 and g.shape == (2, 11) and H.shape == (2, 11, 11)
    fast = ggp.total_likelihood(vecs, f)
    lg, gg = ggp.total_likelihood_grad(vecs, f)
    hl, hg, hH, valid = hess_host(d, vecs, 6)
    assert valid.all()
    for i in range(2):
        assert same_bits(H[i], H[i].T)
        e = scaled_hess_error(vecs[i], None, H[i], hH[i], hl[i])
        eg = scaled_error(vecs[i], g[i], gg[i], lg[i])
        print(f"{noise}/{division} vector {i}: scaled Hessian error vs host {e.max():.2e}, gradient vs ggp_loglik_grad {eg.max():.2e}, "
              f"value vs fast loglik {abs(ll[i] - fast[i]) / abs(fast[i]):.2e}")
        assert e.max() <= 1e-13
        assert eg.max() <= 1e-13
        assert abs(ll[i] - fast[i]) / abs(fast[i]) <= 1e-14
    # the strict mode of the handle does not change the arithmetic; the sign of the objective
    f.set_mode("strict")
    ls, gs, Hs = ggp.total_likelihood_hess(vecs, f)
    f.set_mode(f.last_fast_nodes)
    assert same_bits(ggp.total_likelihood_hess(vecs, f)[2], Hs)
    nl, ng, nH = ggp.total_likelihood_hess(P, f, negative=True)
    pl, pg, pH = ggp.total_likelihood_hess(P, f)
    assert nl == -pl and same_bits(ng, -pg) and same_bits(nH, -pH) and nH.shape == (11, 11)
    f.close()


def test_direction_subsets_are_blocks_of_the_full_hessian_and_calls_repeat_bit_for_bit():
    P = ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(40, 5, params=P, noise_model="scaled", division_model="binomial", seed=63)
    vecs = np.stack([P, P * 1.05])
    f = ggp.Forest(d)
    ll, g, H = ggp.total_likelihood_hess(vecs, f)
    ll2, g2, H2 = ggp.total_likelihood_hess(vecs, f)
    assert same_bits(ll, ll2) and same_bits(g, g2) and same_bits(H, H2)
    for dirs in ([4], [10, 0, 3], [0, 1, 2, 3, 4, 5, 6]):
        lls, gs, Hs = ggp.total_likelihood_hess(vecs, f, dirs=dirs)
        assert same_bits(lls, ll) and same_bits(gs, g[:, dirs]) and same_bits(Hs, H[:, dirs][:, :, dirs])
    for bad in ([11], [-1], [2, 2]):
        with pytest.raises(_lib.GgpError) as e:
            ggp.total_likelihood_hess(vecs, f, dirs=bad)
        assert e.value.code == _lib.GGP_ERR_BAD_ARG
    lib = _lib.load()
    p = np.ascontiguousarray(P)
    out, gr, he = np.empty(1), np.empty(11), np.empty(121)
    dirs = np.zeros(1, dtype=np.int32)
    dp = _lib.c_double_p
    for nd, dirp, hp in ((0, dirs.ctypes.data_as(_lib.c_int32_p), he.ctypes.data_as(dp)), (5, None, he.ctypes.data_as(dp)), (11, None, None)):
        assert lib.ggp_loglik_hess(f.handle, p.ctypes.data_as(dp), 1, dirp, nd, out.ctypes.data_as(dp), gr.ctypes.data_as(dp), hp,
                                   None) == _lib.GGP_ERR_BAD_ARG
    f.close()


def test_vectors_outside_every_rule_and_nan_vectors_get_nan_rows():
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(30, 4, seed=52)
    wide = P.copy()
    wide[4] = 2.0   # gamma_q = 2: no rule covers it
    bad = P.copy()
    bad[7] = -1.0   # negative measurement variance: NaN in the reference
    dirs = [0, 4, 7]
    f = ggp.Forest(d)
    strict = ggp.total_likelihood(np.stack([P, wide, bad]), f, raise_on_nan=False)
    o = Oracle(d)
    assert np.isnan(o.total_loglik(bad))
    rc0, ll0, g0, H0, _ = raw_hess(f, P, dirs)
    assert rc0 == _lib.GGP_OK and np.all(np.isfinite(H0))
    rc, ll, g, H, nan = raw_hess(f, np.stack([P, wide, P * 1.01, bad]), dirs)
    assert rc == _lib.GGP_ERR_BAD_ARG and "vector(s) 1 " in _lib.load().ggp_last_error().decode()
    assert same_bits(ll[0], ll0) and same_bits(g[0], g0[0]) and same_bits(H[0], H0[0]) and np.all(np.isfinite(H[2]))
    assert ll[1] == strict[1] and np.all(np.isnan(g[1])) and np.all(np.isnan(H[1])) and nan[1] == (-1, -1)
    assert np.isnan(ll[3]) and np.all(np.isnan(g[3])) and np.all(np.isnan(H[3])) and nan[3] == o.nan
    assert nan[0] == (-1, -1) and nan[2] == (-1, -1)
    assert f.last_strict_reruns == 2
    rc, ll, g, H, nan = raw_hess(f, np.stack([P, bad]), dirs)
    assert rc == _lib.GGP_ERR_NAN and same_bits(H[0], H0[0]) and np.all(np.isnan(H[1])) and nan[1] == o.nan
    with pytest.raises(ggp.LikelihoodNaN) as e:
        ggp.total_likelihood_hess(np.stack([P, bad]), f, dirs=dirs)
    assert e.value.vec_index == 1 and (e.value.cell, e.value.t_index) == o.nan
    with pytest.raises(_lib.GgpError):
        ggp.total_likelihood_hess(wide, f, dirs=dirs)
    # gamma_q = 0.25 leaves the 5- and 6-node rules but not the 8-node one: the ladder gives the 8-node Hessian
    mid = P.copy()
    mid[4] = 0.25
    f.set_mode(5)
    rc, ll5, g5, H5, _ = raw_hess(f, mid, dirs)
    assert rc == _lib.GGP_OK and f.last_strict_reruns == 0
    f.set_mode(8)
    rc, ll8, g8, H8, _ = raw_hess(f, mid, dirs)
    assert rc == _lib.GGP_OK and same_bits(H5, H8) and same_bits(g5, g8) and same_bits(ll5, ll8)
    f.close()


def test_state_budget_chunks_give_the_same_bits(monkeypatch):
    P = ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(40, 5, params=P, noise_model="scaled", division_model="binomial", seed=64)
    vecs = P * np.exp(np.random.default_rng(4).uniform(-0.05, 0.05, size=(3, 11)))
    f = ggp.Forest(d)
    ref = ggp.total_likelihood_hess(vecs, f)
    f.close()
    one_eval = d.n_cells * 14 * 3 * 8
    # one vector's 66 evaluations fit, two vectors' do not: vector chunks; then 10 evaluations per launch: direction ranges
    for budget in (one_eval * 66 + 8, one_eval * 10 + 8):
        monkeypatch.setenv("GGP_B200_STATE_BUDGET", str(budget))
        fc = ggp.Forest(d)
        got = ggp.total_likelihood_hess(vecs, fc)
        fc.close()
        for a, b in zip(got, ref):
            assert same_bits(a, b)
    monkeypatch.delenv("GGP_B200_STATE_BUDGET")


def test_hessian_after_upload_series_equals_a_fresh_forest(monkeypatch):
    monkeypatch.setenv("GGP_B200_UPLOAD_CHUNKS", "3")
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(40, 4, seed=31)
    f = ggp.Forest(d)
    ggp.total_likelihood_hess(P, f, dirs=[0, 1])
    rng = np.random.default_rng(5)
    x2 = d.log_length + rng.normal(0, 1e-3, d.n_ctp)
    g2 = d.fp * (1 + rng.normal(0, 1e-3, d.n_ctp))
    f.upload_series(None, x2.ctypes.data, g2.ctypes.data)
    vecs = np.stack([P, P * 1.01])
    got = ggp.total_likelihood_hess(vecs, f)
    d2 = ggp.LineageData(cell_offset=d.cell_offset, parent=d.parent, time=d.time, log_length=x2, fp=g2, segment=d.segment,
                         noise_model=d.noise_model, division_model=d.division_model, fp_auto=d.fp_auto)
    f2 = ggp.Forest(d2)
    ref = ggp.total_likelihood_hess(vecs, f2)
    for a, b in zip(got, ref):
        assert same_bits(a, b)
    f.close()
    f2.close()


def test_other_calls_return_the_same_bits_after_a_hessian():
    P = ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(40, 5, params=P, noise_model="scaled", division_model="binomial", seed=65)
    vecs = np.stack([P, P * 1.02, P * 0.98])
    f = ggp.Forest(d)
    before_s = ggp.total_likelihood(vecs, f, per_cell=True)
    before_g = ggp.total_likelihood_grad(vecs, f)
    f.set_mode("fast")
    before_f = ggp.total_likelihood(vecs, f, per_cell=True)
    n_before = f.last_fast_nodes
    f.set_mode("strict")
    ggp.total_likelihood_hess(np.tile(P, (3, 1)), f)
    after_s = ggp.total_likelihood(vecs, f, per_cell=True)
    after_g = ggp.total_likelihood_grad(vecs, f)
    f.set_mode("fast")
    ggp.total_likelihood_hess(P, f)
    after_f = ggp.total_likelihood(vecs, f, per_cell=True)
    assert same_bits(before_s[0], after_s[0]) and same_bits(before_s[1], after_s[1])
    assert same_bits(before_g[0], after_g[0]) and same_bits(before_g[1], after_g[1])
    assert same_bits(before_f[0], after_f[0]) and same_bits(before_f[1], after_f[1]) and f.last_fast_nodes == n_before
    f.close()


def test_group_hessian_agrees_with_the_single_forest():
    P = ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(40, 5, params=P, noise_model="scaled", division_model="binomial", seed=66)
    vecs = np.stack([P, P * 1.03])
    f = ggp.Forest(d)
    f.set_mode(6)
    ll, g, H = ggp.total_likelihood_hess(vecs, f)
    grp = ggp.ForestGroup(d, [0, 0])
    grp.set_mode(6)
    llg, gg, Hg = ggp.total_likelihood_hess(vecs, grp)
    assert max_rel(llg, ll) <= 1e-13
    for i in range(2):
        assert np.max(scaled_error(vecs[i], gg[i], g[i], ll[i])) <= 1e-13
        assert np.max(scaled_hess_error(vecs[i], None, Hg[i], H[i], ll[i])) <= 1e-13
        assert same_bits(Hg[i], Hg[i].T)
    lls, gs, Hs = ggp.total_likelihood_hess(vecs, grp, dirs=[2, 5])
    assert same_bits(gs, gg[:, [2, 5]]) and same_bits(Hs, Hg[:, [2, 5]][:, :, [2, 5]]) and same_bits(lls, llg)
    grp.close()
    f.close()


def test_hessian_at_configs1_size_is_finite_and_matches_num_hessian_grad(monkeypatch):
    """BASELINE configs[1] (10 000 trees x 6 generations, several upload chunks): one vector's 66 evaluations need 14 GB of
    state against the default 8 GB budget, so its directions run in ranges; with a 16 GB budget they run in one pass, with the
    same bits.  The diagonal agrees with central differences of the gradient."""
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(10000, 6, seed=20261018)
    assert d.n_cells * 14 * 3 * 66 * 8 > 8 << 30
    f = ggp.Forest(d)
    ll, g, H = ggp.total_likelihood_hess(P, f)
    assert np.all(np.isfinite(H)) and same_bits(H, H.T) and f.last_strict_reruns == 0
    vecs = np.stack([P, P * 1.01])
    two = ggp.total_likelihood_hess(vecs, f, dirs=[0, 4, 10])
    monkeypatch.setenv("GGP_B200_STATE_BUDGET", str(16 << 30))
    f16 = ggp.Forest(d)
    monkeypatch.delenv("GGP_B200_STATE_BUDGET")
    assert all(same_bits(a, b) for a, b in zip(ggp.total_likelihood_hess(P, f16), (ll, g, H)))
    assert all(same_bits(a, b) for a, b in zip(ggp.total_likelihood_hess(vecs, f16, dirs=[0, 4, 10]), two))
    f16.close()
    lg, gg = ggp.total_likelihood_grad(P, f)
    assert np.max(scaled_error(P, g, gg, lg)) <= 1e-13 and abs(ll - lg) <= 1e-14 * abs(lg)
    Hn = ggp.num_hessian_grad(f, P, list(range(11)), 1e-5)
    r = np.abs(np.diag(H) - np.diag(Hn)) / np.abs(np.diag(H))
    print(f"configs[1]: diagonal of the exact Hessian against num_hessian_grad(1e-5), relative: {np.array2string(r, precision=1)}")
    assert r.max() <= 1e-5
    f.close()


def test_exact_errors_option_writes_the_inverse_hessian_diagonal(tmp_path):
    """-m --fast --exact_errors on the small forest of test_minimization_scan_and_error_bars_replay_on_the_oracle: the new
    _final.csv section equals -diag(inv(H)) of total_likelihood_hess at the final parameters; without the option the file
    holds what it held before"""
    P = ggp.PARAMS_SCALED_BINOMIAL
    data = ggp.simulate_forest(8, 3, noise_model="scaled", division_model="binomial", seed=21)
    csv, cfg = write_inputs(tmp_path, data)
    pf = write_params(tmp_path / "p.txt", P * np.array([1.1, 1, 1, 0.9, 1, 1, 1, 1, 1, 1, 1]), free=(0, 3), bound=(8,))
    finals = {}
    for name, extra in (("plain", []), ("exact", ["--exact_errors"])):
        out = str(tmp_path / name)
        run(["-i", csv, "-b", pf, "-c", cfg, "-m", "--fast", "-t", "1e-2", "-o", out] + extra)
        finals[name] = open(os.path.join(out, "forest_f03_b8_final.csv")).read()
    head = "\nerrors^2 (exact Hessian of the fast log-likelihood):\n"
    assert head not in finals["plain"]
    assert finals["exact"].startswith(finals["plain"])
    section = finals["exact"][len(finals["plain"]):]
    assert section.startswith(head)
    names, values = section[len(head):].strip().split("\n")
    assert names == "mean_lambda,mean_q,var_g"
    # the final parameters: _parameter_file.txt prints them to 6 digits, the iterations file to 20 (the best logged vector)
    out = str(tmp_path / "exact")
    pfile = open(os.path.join(out, "forest_f03_b8_parameter_file.txt")).read().split("\n")[1:12]
    x6 = np.array([float(line.split(" = ")[1]) for line in pfile])
    it = read_table(os.path.join(out, "forest_f03_b8_iterations.csv"), "iteration,")
    logged = np.array([[float(v) for v in r[1:]] for r in it])
    x = logged[np.argmax(logged[:, 11]), :11]
    assert np.all(np.abs(x - x6) <= 1e-5 * np.abs(x))
    dirs = [0, 3, 8]   # the parameters that are not fixed: free mean_lambda and mean_q, bound var_g
    f = ggp.Forest(data)
    _, _, H = ggp.total_likelihood_hess(x, f, dirs=dirs)
    want = -np.diag(np.linalg.inv(H))
    got = np.array([float(v) for v in values.split(",")])
    print(f"--exact_errors {got} vs -diag(inv(H)) {want}")
    assert np.all(np.abs(got - want) <= 1e-10 * np.abs(want))
    f.close()
