"""CPU tests of the strict math: the product's host+device headers compiled for the host (tests/hostcheck)
and the oracle, against (a) the committed golden vectors generated from the reference's own code and libm,
(b) the host's libm and the reference build oracle/_ref when it is present, (c) Faddeeva's Maple values and mpmath."""
import ctypes as C
import ctypes.util
import json
import os

import numpy as np
import pytest

from conftest import ROOT, same_bits, max_rel
from oracle import oracle_py

dp = C.POINTER(C.c_double)


@pytest.fixture(scope="module")
def hc():
    L = C.CDLL(os.path.join(ROOT, "tests", "hostcheck", "libhostcheck.so"))
    return L


def _p(a):
    return a.ctypes.data_as(dp)


def _call1(fn, x):
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.empty_like(x)
    fn(C.c_long(x.size), _p(x), _p(y))
    return y


def test_exp_log_pow_match_glibc_bits(hc, golden_dir):
    z = np.load(os.path.join(golden_dir, "libm_bits.npz"))
    assert same_bits(_call1(hc.hc_exp, z["exp_x"]), z["exp_y"])
    assert same_bits(_call1(hc.hc_log, z["log_x"]), z["log_y"])
    x, e = np.ascontiguousarray(z["pow_x"]), np.ascontiguousarray(z["pow_e"])
    y = np.empty_like(x)
    hc.hc_pow(C.c_long(x.size), _p(x), _p(e), _p(y))
    assert same_bits(y, z["pow_y"])


def test_exp_log_pow_match_live_libm(hc):
    """the host's libm itself: the reference calls exp / log of glibc (oracle/ref_shim.cpp routes them unchanged)"""
    libm = C.CDLL(ctypes.util.find_library("m"))
    for name in ("exp", "log"):
        getattr(libm, name).restype = C.c_double
        getattr(libm, name).argtypes = [C.c_double]
    rng = np.random.default_rng(11)
    x = rng.uniform(-30, 30, 20000)
    assert same_bits(_call1(hc.hc_exp, x), np.array([libm.exp(v) for v in x]))
    x = 10 ** rng.uniform(-10, 10, 20000)
    assert same_bits(_call1(hc.hc_log, x), np.array([libm.log(v) for v in x]))


def test_dawson_known_answers(hc, golden_dir):
    g = json.load(open(os.path.join(golden_dir, "dawson_known_answers.json")))
    # Faddeeva.cc:2378-2512, the self-test's real-argument entries (relative 1e-13 there, :2514)
    xs = np.array([float(e["x"]) for e in g["maple_real"]])
    ws = np.array([float(e["dawson"]) for e in g["maple_real"]])
    assert len(xs) >= 4
    for fn in (lambda v: _call1(hc.hc_dawson, v), lambda v: np.array([oracle_py.oracle().ggp_oracle_dawson(t) for t in v])):
        assert max_rel(fn(xs), ws) < 1e-13
    xs = np.array([float.fromhex(e["x"]) for e in g["mpmath"]])
    ws = np.array([float(e["dawson"]) for e in g["mpmath"]])
    nz = ws != 0
    assert max_rel(_call1(hc.hc_dawson, xs)[nz], ws[nz]) < 2e-13
    assert same_bits(_call1(hc.hc_dawson, xs), np.array([oracle_py.oracle().ggp_oracle_dawson(t) for t in xs]))


def test_dawson_matches_reference_bits(hc):
    R = oracle_py.ref()
    if R is None:
        pytest.skip("reference build not present")
    rng = np.random.default_rng(5)
    x = np.concatenate([rng.uniform(-60, 60, 30000), 10 ** rng.uniform(-12, 9, 5000), -10 ** rng.uniform(-12, 9, 5000)])
    ref = np.array([R.ggp_ref_dawson(v) for v in x])
    assert same_bits(_call1(hc.hc_dawson, x), ref)
    assert same_bits(np.array([oracle_py.oracle().ggp_oracle_dawson(v) for v in x]), ref)


def _propagate_host(hc, mean, cov16, dt, p7):
    n = mean.shape[0]
    c = cov16.reshape(n, 4, 4)
    iu = np.triu_indices(4)
    out = np.empty((n, 14))
    for i in range(n):   # hc_propagate takes one parameter set per call
        s = np.ascontiguousarray(np.concatenate([mean[i], c[i][iu]]))
        o = np.empty(14)
        hc.hc_propagate(C.c_long(1), _p(s), _p(np.array([dt[i]])), _p(np.ascontiguousarray(p7[i])), _p(o))
        out[i] = o
    return out


def test_step_matches_reference_golden(hc, golden_dir):
    """the CSE'd propagation step (ggp_step.cuh) and the oracle reproduce the reference's mean_cov_model and
    cross_cov_model bit for bit on the committed vectors (tests.h literals + states along filter runs)"""
    z = np.load(os.path.join(golden_dir, "ref_step_vectors.npz"))
    iu = np.triu_indices(4)
    out = _propagate_host(hc, z["mean"], z["cov"], z["dt"], z["p7"])
    assert same_bits(out[:, :4], z["mean_out"])
    assert same_bits(out[:, 4:], z["cov_out"].reshape(-1, 4, 4)[:, iu[0], iu[1]])
    for i in range(z["mean"].shape[0]):
        mo, co = oracle_py.mean_cov_model(z["mean"][i], z["cov"][i], z["dt"][i], z["p7"][i])
        assert same_bits(mo, z["mean_out"][i]) and same_bits(co, z["cov_out"][i])
        assert same_bits(oracle_py.cross_cov_model(z["mean"][i], z["cov"][i], z["dt"][i], z["p7"][i]), z["cross_out"][i])
    L = oracle_py.oracle()
    got = np.array([[L.ggp_oracle_tauint(k, *row) for k in range(4)] for row in z["tauint_args"]])
    assert same_bits(got, z["tauint_out"])


def test_step_matches_live_reference(hc):
    R = oracle_py.ref()
    if R is None:
        pytest.skip("reference build not present")
    from gfp_gaussian_process_b200 import simulate_forest, PARAMS_SCALED_BINOMIAL
    d = simulate_forest(8, 4, noise_model="scaled", division_model="binomial", seed=21)
    o = oracle_py.Oracle(d)
    mf, cf = o.predictions([PARAMS_SCALED_BINOMIAL])["forward"]
    idx = np.arange(0, d.n_ctp, 7)
    p7 = np.tile(PARAMS_SCALED_BINOMIAL[:7], (len(idx), 1))
    dt = np.full(len(idx), 15.0)
    out = _propagate_host(hc, mf[idx], cf[idx].reshape(-1, 16), dt, p7)
    iu = np.triu_indices(4)
    for k, i in enumerate(idx):
        mo, co = oracle_py.mean_cov_model(mf[i], cf[i], 15.0, PARAMS_SCALED_BINOMIAL[:7], which="ref")
        assert same_bits(out[k, :4], mo)
        assert same_bits(out[k, 4:], co.reshape(4, 4)[iu])


def test_log_evidence_finish_matches_numpy_on_ordinary_input(hc):
    """hc_ll_finish (the product's ggp_log_evidence_finish on the host, the reference of the device self-test fn 6)
    against a direct numpy evaluation of likelihood.h:26-32 from the quadratic form on"""
    rng = np.random.default_rng(2)
    n = 2000
    S00 = 10 ** rng.uniform(-3, 5, n); S11 = 10 ** rng.uniform(-3, 5, n)
    S01 = rng.uniform(-0.9, 0.9, n) * np.sqrt(S00 * S11)
    qf = -rng.uniform(0, 30, n)
    cases = np.ascontiguousarray(np.stack([qf, S00, S01, S01, S11], axis=1))
    out = np.empty(n)
    hc.hc_ll_finish(C.c_long(n), _p(cases), _p(out))
    ref = qf - 0.5 * np.log(S00 * S11 - S01 * S01) - 2 * np.log(2 * np.pi)
    assert np.max(np.abs(out - ref) / np.abs(ref)) < 1e-12
