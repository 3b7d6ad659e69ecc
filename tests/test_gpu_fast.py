"""The FAST likelihood mode (ggp_forest_set_mode, csrc/ggp_fast.cuh) on the GPU.  It is NOT bit-identical to the reference:
its gate is the north-star tolerance |dloglik| / |loglik| <= 1e-10 against the oracle, written here, never widened; beside it
the kernel must agree with its own host build (tests/hostcheck/fastcheck.cpp, same code without FMA contraction) to 1e-12,
fall back to the strict path bit for bit outside the quadrature's validity range, and report NaNs like the reference."""
import os
import sys

import numpy as np
import pytest

from conftest import same_bits, example_data, max_rel, ROOT
from oracle.oracle_py import Oracle
import gfp_gaussian_process_b200 as ggp

sys.path.insert(0, os.path.join(ROOT, "tools"))
from fast_gate import fast_loglik  # noqa: E402

pytestmark = pytest.mark.gpu
GATE = 1e-10


def rel(a, b):
    return abs(a - b) / abs(b)


@pytest.mark.parametrize("noise,division", [("const", "gauss"), ("scaled", "binomial"), ("scaled", "gauss"), ("const", "binomial")])
def test_fast_gate_on_small_forests(noise, division):
    P = ggp.PARAMS_CONST_GAUSS if noise == "const" else ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(60, 5, params=P, noise_model=noise, division_model=division, seed=51)
    f = ggp.Forest(d)
    f.set_mode(6)
    assert f.mode == "fast6"
    vecs = np.stack([P, P * 1.03, P * 0.96])
    ll, pc = ggp.total_likelihood(vecs, f, per_cell=True)
    assert f.last_strict_reruns == 0
    o = Oracle(d)
    for i in range(3):
        assert rel(ll[i], o.total_loglik(vecs[i])) <= GATE
    host, valid, pc_h, _ = fast_loglik(d, vecs, n_nodes=6, per_cell=True)
    assert valid.all() and np.max(np.abs(ll - host) / np.abs(host)) <= 1e-13
    assert np.max(np.abs(pc - pc_h) / np.abs(pc_h)) <= 1e-11
    # single calls equal the batch, run to run identical
    assert ggp.total_likelihood(vecs[1], f) == ll[1] and same_bits(ggp.total_likelihood(vecs, f), ll)
    # "fast" picks the rule from the parameters and the forest's time step (5 nodes at dt = 3.5, 6 at dt = 15): same gate
    f.set_mode("fast")
    ll_auto = ggp.total_likelihood(vecs, f)
    assert f.last_fast_nodes == (5 if noise == "const" else 6) and f.last_strict_reruns == 0
    assert np.max(np.abs(ll_auto - ll) / np.abs(ll)) <= 1e-13
    # back to strict: the bit-exact path again
    f.set_mode("strict")
    assert same_bits(ggp.total_likelihood(P, f, per_cell=True)[1], o.total_loglik(P, per_cell=True)[1])
    f.close()


def test_fast_gate_on_the_example_data_set(golden_dir):
    data, z = example_data(golden_dir)
    P = np.asarray(z["params"])
    f = ggp.Forest(data)
    f.set_mode("fast")
    ll = ggp.total_likelihood(P, f)
    ref = Oracle(data).total_loglik(P)
    print(f"example data set: fast {ll!r} reference {ref!r} rel {rel(ll, ref):.2e}")
    assert f.last_strict_reruns == 0 and rel(ll, ref) <= GATE
    f.close()


def test_fast_gate_at_full_size():
    """BASELINE configs[1] (10 000 trees x 6 generations): fast against the strict kernels (== oracle per cell, other tests)"""
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(10000, 6, seed=20261018)
    f = ggp.Forest(d)
    strict = ggp.total_likelihood(P, f)
    f.set_mode(6)
    vecs = np.stack([P, P * 1.02])
    fast = ggp.total_likelihood(vecs, f)
    print(f"configs[1]: fast {fast[0]!r} strict {strict!r} rel {rel(fast[0], strict):.2e}")
    assert f.last_strict_reruns == 0 and rel(fast[0], strict) <= GATE
    sub, cells, ctp = d.subset(d.roots()[100:110])
    host, valid, _, _ = fast_loglik(sub, vecs, n_nodes=6)
    fs = ggp.Forest(sub)
    fs.set_mode(6)
    assert np.max(np.abs(ggp.total_likelihood(vecs, fs) - host) / np.abs(host)) <= 1e-13
    fs.close()
    f.close()


def test_fast_falls_back_to_strict_outside_its_validity_range():
    """a vector with gamma_q = 2 (exponent varies by 7 over a step) is outside the 6-node rule's range: ggp_loglik re-runs it
    strictly (bits of the strict path, NaN records of the reference); the others stay fast"""
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(30, 4, seed=52)
    wide = P.copy()
    wide[4] = 2.0
    bad = P.copy()
    bad[7] = -1.0   # negative measurement variance: NaN in the reference
    vecs = np.stack([P, wide, P * 1.01, bad])
    f = ggp.Forest(d)
    strict, pc_s = ggp.total_likelihood(vecs, f, per_cell=True, raise_on_nan=False)
    f.set_mode(6)
    fast, pc_f = ggp.total_likelihood(vecs, f, per_cell=True, raise_on_nan=False)
    assert f.last_strict_reruns == 2
    assert fast[1] == strict[1] and same_bits(pc_f[1], pc_s[1]) and np.isnan(fast[3]) and np.isnan(strict[3])
    assert rel(fast[0], strict[0]) <= GATE and rel(fast[2], strict[2]) <= GATE and fast[0] != strict[0]
    o = Oracle(d)
    assert np.isnan(o.total_loglik(bad))
    with pytest.raises(ggp.LikelihoodNaN) as e:
        ggp.total_likelihood(vecs, f)
    assert e.value.vec_index == 3 and (e.value.cell, e.value.t_index) == o.nan
    # more nodes widen the range (gamma_q = 0.25: the exponent varies by ~0.95 over a step): "fast" chooses 8 nodes; a forced
    # 5-node rule climbs the ladder 5 -> 6 -> 8 without reaching the strict kernels
    wide[4] = 0.25
    f.set_mode("fast")
    ll_w = ggp.total_likelihood(wide, f)
    assert f.last_strict_reruns == 0 and f.last_fast_nodes == 8
    f.set_mode(5)
    assert ggp.total_likelihood(wide, f) == ll_w and f.last_strict_reruns == 0
    f.set_mode("strict")
    assert rel(ll_w, ggp.total_likelihood(wide, f)) <= GATE
    f.close()


@pytest.mark.parametrize("grid", ["two_steps", "many_steps"])
def test_fast_gate_on_irregular_time_grids(grid):
    """the constants' table of the fast kernels: 2 distinct time steps (table in shared memory, per-point index) and hundreds
    (table read through L1); a uniform grid takes the index-free path (every other test).  Random parameter vectors around the
    example's values: the gate against the strict kernels (== oracle per cell), and against the oracle itself for the first"""
    P = ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(40, 4, params=P, noise_model="scaled", division_model="binomial", seed=77, dt=6.0)
    k = np.rint(d.time / 6.0)
    if grid == "two_steps":
        d.time = 6.0 * k + np.where(k % 2 == 1, 1.5, 0.0)          # steps of 7.5 and 4.5
    else:
        d.time = 6.0 * k + 1.7 * np.sin(k * 0.37)                   # every step different
    rng = np.random.default_rng(11)
    vecs = P * np.exp(rng.uniform(-0.4, 0.4, size=(12, 11)))
    vecs[0] = P
    f = ggp.Forest(d)
    strict = ggp.total_likelihood(vecs, f, raise_on_nan=False)
    f.set_mode("fast")
    fast = ggp.total_likelihood(vecs, f, raise_on_nan=False)
    ok = np.isfinite(strict)
    assert ok.sum() >= 10 and np.array_equal(np.isfinite(fast), ok)
    assert np.max(np.abs(fast[ok] - strict[ok]) / np.abs(strict[ok])) <= GATE
    assert f.last_strict_reruns <= 2 and np.any(fast[ok] != strict[ok])
    assert rel(fast[0], Oracle(d).total_loglik(vecs[0])) <= GATE
    f.close()


def test_fast_mode_runs_a_batch_with_an_uncovered_vector_on_the_strict_kernels():
    """mode "fast" picks one rule for the batch: if no rule covers one of its vectors (gamma_q = 2), the whole batch returns
    the strict kernels' bits, nothing counts as re-run, and ggp_last_fast_nodes keeps the rule of the last covered batch"""
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(30, 4, seed=52)
    wide, mid = P.copy(), P.copy()
    wide[4] = 2.0
    mid[4] = 0.25
    vecs = np.stack([P, wide, P * 1.01])
    f = ggp.Forest(d)
    strict, pc_s = ggp.total_likelihood(vecs, f, per_cell=True)
    f.set_mode("fast")
    ggp.total_likelihood(mid, f)
    assert f.last_fast_nodes == 8
    fast, pc_f = ggp.total_likelihood(vecs, f, per_cell=True)
    assert same_bits(fast, strict) and same_bits(pc_f, pc_s)
    assert f.last_strict_reruns == 0 and f.last_fast_nodes == 8
    f.close()


def test_ladder_behind_a_streamed_upload(monkeypatch):
    """after ggp_forest_upload_series the first pass of a small batch carries its parameters in the launch arguments and runs
    chunk by chunk behind the copies; the vector it flags (gamma_q = 0.25) climbs 5 -> 6 -> 8 nodes.  Per-cell rows as on a
    forest created from the new series, the climbed vector's as an 8-node call; totals to 1e-14 (other block partials)"""
    monkeypatch.setenv("GGP_B200_UPLOAD_CHUNKS", "3")
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(30, 4, seed=52)
    mid = P.copy()
    mid[4] = 0.25
    vecs = np.stack([P, mid, P * 1.01])
    f = ggp.Forest(d)
    f.set_mode(5)
    rng = np.random.default_rng(5)
    x2 = d.log_length + rng.normal(0, 1e-3, d.n_ctp)
    g2 = d.fp * (1 + rng.normal(0, 1e-3, d.n_ctp))
    f.upload_series(None, x2.ctypes.data, g2.ctypes.data)
    ll, pc = ggp.total_likelihood(vecs, f, per_cell=True)
    assert f.last_strict_reruns == 0
    d2 = ggp.LineageData(cell_offset=d.cell_offset, parent=d.parent, time=d.time, log_length=x2, fp=g2, segment=d.segment,
                         noise_model=d.noise_model, division_model=d.division_model, fp_auto=d.fp_auto)
    f2 = ggp.Forest(d2)
    f2.set_mode(5)
    ll2, pc2 = ggp.total_likelihood(vecs, f2, per_cell=True)
    assert same_bits(pc, pc2) and max_rel(ll, ll2) < 1e-14
    f2.set_mode(8)
    assert same_bits(ggp.total_likelihood(mid, f2, per_cell=True)[1], pc[1])
    f.close()
    f2.close()


def test_launch_count_adds_the_passes_of_the_ladder():
    """ggp_last_launch_count of a call whose vector climbs 5 -> 6 -> 8 nodes is the sum of one pass of each rule, for the
    likelihood and for its gradient"""
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(30, 4, seed=52)
    mid = P.copy()
    mid[4] = 0.25
    f = ggp.Forest(d)
    for run in (ggp.total_likelihood, ggp.total_likelihood_grad):
        single = 0
        for n in (5, 6, 8):
            f.set_mode(n)
            run(P, f)
            single += f.last_launch_count
        f.set_mode(5)
        run(np.stack([P, mid]), f)
        assert f.last_strict_reruns == 0 and f.last_launch_count == single
    f.close()
