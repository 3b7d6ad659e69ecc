"""The series simulator without a GPU: csrc/ggp_sim.cuh compiled for the host (tests/hostcheck/simcheck.cpp, the device kernel's
per-cell body and bits).  Philox known answers, the same process as synthetic.py (two-sample statistics per generation and
point index), and exact limits of the dynamics."""
import os
import sys

import numpy as np
import pytest

from conftest import ROOT
import gfp_gaussian_process_b200 as ggp

sys.path.insert(0, os.path.join(ROOT, "tools"))
from sim_check import philox, sim_host  # noqa: E402


@pytest.mark.parametrize("ctr,key,expect", [
    ([0, 0, 0, 0], 0, [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
    ([0xffffffff] * 4, 0xffffffffffffffff, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
    ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], (0x299f31d0 << 32) | 0xa4093822, [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]),
])
def test_philox_known_answers(ctr, key, expect):
    """Random123's known-answer vectors of Philox4x32-10 (key word 0 = the seed's low 32 bits)"""
    assert list(philox(ctr, key)) == expect


def root_prior(P, noise):
    g_mean = 2.0 * P[3] / (P[0] + P[6]) * (1.0 if noise == "const" else 0.5)
    return np.array([np.log(2.0), g_mean, 0.01, (0.1 * g_mean) ** 2])


def point_table(data):
    """generation and point index of every time point of a simulate_forest forest (tree-major, breadth-first cells)"""
    n = np.diff(data.cell_offset)
    cells_per_tree = int(np.flatnonzero(data.parent < 0)[1]) if (data.parent < 0).sum() > 1 else data.n_cells
    b = np.arange(data.n_cells) % cells_per_tree
    gen = np.floor(np.log2(b + 1)).astype(int)
    k = np.arange(data.n_ctp) - np.repeat(data.cell_offset[:-1], n)
    last = np.repeat(data.cell_offset[1:] - 1, n)
    return np.repeat(gen, n), k, np.arange(data.n_ctp) < last


def z_scores(a, b):
    """two-sample z of the means and of the variances (variance of a sample variance from the fourth central moment)"""
    ma, mb, va, vb = a.mean(), b.mean(), a.var(), b.var()
    zm = (ma - mb) / np.sqrt(va / a.size + vb / b.size)
    m4a, m4b = ((a - ma) ** 4).mean(), ((b - mb) ** 4).mean()
    zv = (va - vb) / np.sqrt((m4a - va ** 2) / a.size + (m4b - vb ** 2) / b.size)
    return zm, zv


@pytest.mark.parametrize("noise,division", [("const", "gauss"), ("scaled", "binomial")])
def test_same_process_as_synthetic(noise, division):
    """for every (generation, point index): mean and variance of x_obs, g_obs and of the x_obs increments against a
    synthetic.py sample on the same genealogy, |z| < 5"""
    P = ggp.PARAMS_CONST_GAUSS if noise == "const" else ggp.PARAMS_SCALED_BINOMIAL
    data = ggp.simulate_forest(20000, 4, noise_model=noise, division_model=division, seed=20261022, substeps=8)
    x, g, bad = sim_host(data, P, seed=11, substeps=8, root_prior=root_prior(P, noise))
    assert bad == -1
    gen, k, has_next = point_table(data)
    nxt = np.flatnonzero(has_next)
    worst, n_groups = 0.0, 0
    for gi in range(4):
        for ki in range(int(k.max()) + 1):
            sel = np.flatnonzero((gen == gi) & (k == ki))
            if sel.size < 200:
                continue
            inc = np.intersect1d(sel, nxt)
            pairs = [(x[sel], data.log_length[sel]), (g[sel], data.fp[sel])]
            if inc.size >= 200:
                pairs.append((x[inc + 1] - x[inc], data.log_length[inc + 1] - data.log_length[inc]))
            for a, b in pairs:
                zm, zv = z_scores(a, b)
                worst = max(worst, abs(zm), abs(zv))
                n_groups += 1
                assert abs(zm) < 5 and abs(zv) < 5, (gi, ki, zm, zv)
    print(f"{noise}/{division}: {n_groups} comparisons, max |z| {worst:.2f}")
    assert n_groups > 200


def test_deterministic_x_without_its_noise():
    """var_x = var_lambda = var_dx = 0: lambda stays mean_lambda and every x_obs increment is the sum of mean_lambda * h"""
    P = ggp.PARAMS_CONST_GAUSS.copy()
    P[[2, 7, 9]] = 0.0
    data = ggp.simulate_forest(50, 3, seed=5)
    for substeps in (1, 3, 8):
        x, _, _ = sim_host(data, P, seed=3, substeps=substeps)
        _, _, has_next = point_table(data)
        i = np.flatnonzero(has_next)
        h = (data.time[i + 1] - data.time[i]) / substeps
        y = x[i].copy()
        for _ in range(substeps):
            y = y + P[0] * h
        assert np.array_equal(y, x[i + 1])


def test_binomial_division_gives_whole_molecules():
    """var_g = 0 with binomial division: a daughter's first g_obs is var_dg times an integer"""
    P = ggp.PARAMS_SCALED_BINOMIAL.copy()
    P[8] = 0.0
    data = ggp.simulate_forest(50, 3, noise_model="scaled", division_model="binomial", seed=5)
    _, g, _ = sim_host(data, P, seed=3)
    first = data.cell_offset[:-1][data.parent >= 0]
    n_mol = np.rint(g[first] / P[10])
    assert np.all(n_mol >= 1) and np.array_equal(P[10] * n_mol, g[first])


def test_seeds():
    """the same seed gives the same bits, different seeds give different series"""
    P = ggp.PARAMS_SCALED_BINOMIAL
    data = ggp.simulate_forest(20, 3, noise_model="scaled", division_model="binomial", seed=5)
    a = sim_host(data, P, seed=1)
    b = sim_host(data, P, seed=1)
    c = sim_host(data, P, seed=2)
    assert np.array_equal(a[0].view(np.uint64), b[0].view(np.uint64)) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))
    assert not np.any(a[0] == c[0]) and not np.any(a[1] == c[1])
