"""The series simulator on the GPU (ggp_simulate, ggp_group_simulate, simulate_series and the command line's --simulate): the
device bits against the host build of the same code (tests/hostcheck/simcheck.cpp), groups against one forest, the handle's
state afterwards against a forest made from the simulated series, streamed uploads, argument errors."""
import ctypes as C
import glob
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, ragged_forest, same_bits
import gfp_gaussian_process_b200 as ggp
from gfp_gaussian_process_b200 import _lib, io
from test_gpu_cli import write_inputs, write_params, run

sys.path.insert(0, os.path.join(ROOT, "tools"))
from sim_check import sim_host  # noqa: E402

pytestmark = pytest.mark.gpu

COMBOS = [("const", "gauss"), ("scaled", "binomial"), ("scaled", "gauss"), ("const", "binomial")]


def params_of(noise):
    return ggp.PARAMS_CONST_GAUSS if noise == "const" else ggp.PARAMS_SCALED_BINOMIAL


def irregular(data, seed=4):
    """every time jittered by up to 40 % of the step: irregular steps, daughters whose first times differ"""
    rng = np.random.default_rng(seed)
    dt = np.min(np.diff(data.time[:2]))
    t = data.time + rng.uniform(0.0, 0.4 * dt, data.n_ctp)
    return ggp.LineageData(cell_offset=data.cell_offset, parent=data.parent, time=t, log_length=data.log_length, fp=data.fp,
                           segment=data.segment, noise_model=data.noise_model, division_model=data.division_model, fp_auto=data.fp_auto)


def with_series(data, x, g, **kw):
    return ggp.LineageData(cell_offset=data.cell_offset, parent=data.parent, time=data.time, log_length=x, fp=g, segment=data.segment,
                           noise_model=data.noise_model, division_model=data.division_model, fp_auto=data.fp_auto, **kw)


def cases():
    out = []
    for i, (noise, division) in enumerate(COMBOS):
        out.append((f"{noise}/{division}", ggp.simulate_forest(30, 4, noise_model=noise, division_model=division, seed=40 + i),
                    params_of(noise), (1, 8, 3)[i % 3]))
    rf = ragged_forest()
    out.append(("ragged", rf, np.stack([ggp.PARAMS_SCALED_BINOMIAL, ggp.PARAMS_SCALED_BINOMIAL * 1.1]), 3))
    out.append(("irregular", irregular(ggp.simulate_forest(30, 4, seed=45)), ggp.PARAMS_CONST_GAUSS, 8))
    return out


@pytest.mark.parametrize("case", range(6))
def test_device_series_equal_the_host_build(case):
    name, data, P, substeps = cases()[case]
    f = ggp.Forest(data)
    for root in (np.array([0.7, 30.0, 0.01, 4.0]), None):
        x, g = ggp.simulate_series(f, P, seed=7, substeps=substeps, root_prior=root)
        hx, hg, bad = sim_host(data, P, 7, substeps, root)
        assert bad == -1
        print(f"{name}, {substeps} sub-steps: {data.n_ctp} points, bit-identical {same_bits(x, hx) and same_bits(g, hg)}")
        assert same_bits(x, hx) and same_bits(g, hg)
        data = with_series(data, x, g)   # the next call's default root prior is the simulated series' init_f
    f.close()


@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]])
@pytest.mark.parametrize("layout", ["contiguous", "bin-packed"])
def test_group_gives_the_single_forest_bits(devices, layout):
    data, P = (ggp.simulate_forest(30, 4, noise_model="scaled", division_model="binomial", seed=46), ggp.PARAMS_SCALED_BINOMIAL) \
        if layout == "contiguous" else (ragged_forest(), np.stack([ggp.PARAMS_SCALED_BINOMIAL, ggp.PARAMS_SCALED_BINOMIAL * 1.1]))
    grp = ggp.ForestGroup(data, devices)
    assert grp.contiguous == (layout == "contiguous")
    f = ggp.Forest(data)
    for seed in (1, 2):
        x, g = ggp.simulate_series(f, P, seed=seed, substeps=3)
        gx, gg = ggp.simulate_series(grp, P, seed=seed, substeps=3)
        assert same_bits(x, gx) and same_bits(g, gg)
        # the group against a new group made from the simulated series: the same likelihood bits
        fresh = ggp.ForestGroup(with_series(data, x, g), devices)
        p0 = P if P.ndim == 1 else P[0]
        a, ac = grp.total_likelihood(p0, per_cell=True)
        b, bc = fresh.total_likelihood(p0, per_cell=True)
        assert same_bits(a, b) and same_bits(ac, bc)
        assert same_bits(ggp.total_likelihood_grad(p0, grp)[1], ggp.total_likelihood_grad(p0, fresh)[1])
        pa, pb = grp.predictions(P), fresh.predictions(P)
        assert all(same_bits(pa[k], pb[k]) for k in pa)
        fresh.close()
    grp.close()
    f.close()


def test_handle_state_after_a_simulation_equals_a_new_forest():
    data = ggp.simulate_forest(40, 4, noise_model="scaled", division_model="binomial", seed=47)
    P = ggp.PARAMS_SCALED_BINOMIAL
    f = ggp.Forest(data)
    ll0 = ggp.total_likelihood(P, f)
    ggp.prediction_forward_backward(f, [P])   # predictions of the original series, to be invalidated
    x, g = ggp.simulate_series(f, P, seed=9)
    n = ggp.Forest(with_series(data, x, g))
    assert all(same_bits(a, b) for a, b in zip(f.init_stats(), n.init_stats()))
    for mode in ("strict", "fast"):
        f.set_mode(mode)
        n.set_mode(mode)
        a, ac = ggp.total_likelihood(P, f, per_cell=True)
        b, bc = ggp.total_likelihood(P, n, per_cell=True)
        assert same_bits(a, b) and same_bits(ac, bc)
    ga, gb = ggp.total_likelihood_grad(P, f), ggp.total_likelihood_grad(P, n)
    assert same_bits(ga[0], gb[0]) and same_bits(ga[1], gb[1])
    pa, pb = ggp.prediction_forward_backward(f, [P]), ggp.prediction_forward_backward(n, [P])
    assert all(same_bits(pa[k][i], pb[k][i]) for k in pa for i in range(2))
    # the original series back: the original log-likelihood bits
    f.set_mode("strict")
    f.upload_series(None, data.log_length.ctypes.data, data.fp.ctypes.data)
    assert same_bits(ggp.total_likelihood(P, f), ll0)
    f.close()
    n.close()


def test_simulation_behind_a_streamed_upload(monkeypatch):
    monkeypatch.setenv("GGP_B200_UPLOAD_CHUNKS", "3")
    data = ggp.simulate_forest(40, 4, seed=48)
    P = ggp.PARAMS_CONST_GAUSS
    f = ggp.Forest(data)
    x0, g0 = ggp.simulate_series(f, P, seed=3, root_prior=data.init_stats())
    rng = np.random.default_rng(1)
    x2, g2 = data.log_length + rng.normal(0, 1e-3, data.n_ctp), data.fp * (1 + rng.normal(0, 1e-3, data.n_ctp))
    f.upload_series(None, x2.ctypes.data, g2.ctypes.data)   # pending on the copy stream
    x1, g1 = ggp.simulate_series(f, P, seed=3, root_prior=data.init_stats())
    assert same_bits(x0, x1) and same_bits(g0, g1)
    f.close()


def raw_simulate(f, P, substeps=8, root=None):
    p = np.ascontiguousarray(P, dtype=np.float64).reshape(-1, 11)
    r = None if root is None else np.ascontiguousarray(root, dtype=np.float64)
    cp = lambda a: None if a is None else a.ctypes.data_as(_lib.c_double_p)  # noqa: E731
    return _lib.load().ggp_simulate(f.handle, cp(p), p.shape[0], C.c_uint64(1), substeps, cp(r), None, None)


def test_argument_errors_leave_the_series_untouched():
    data = ggp.simulate_forest(10, 3, noise_model="scaled", division_model="binomial", seed=49)
    P = ggp.PARAMS_SCALED_BINOMIAL
    f = ggp.Forest(data)
    ll = ggp.total_likelihood(P, f)
    bad = []
    for i, v in ((1, 0.0), (4, -1.0), (2, -1e-9), (5, -1.0), (7, -1e-9), (8, -1.0), (9, -1e-9), (10, -1.0), (10, 0.0)):
        Q = P.copy()
        Q[i] = v
        bad.append((Q, 8, None))
    bad += [(P, 0, None), (P, 8, np.array([0.7, 30.0, -0.01, 4.0]))]
    for Q, substeps, root in bad:
        assert raw_simulate(f, Q, substeps, root) == _lib.GGP_ERR_BAD_ARG, (Q, substeps, root)
    assert same_bits(ggp.total_likelihood(P, f), ll)
    f.close()
    # a negative time step
    t = data.time.copy()
    o = data.cell_offset
    t[o[3]:o[4]] = t[o[3]:o[4]][::-1].copy()
    neg = ggp.LineageData(cell_offset=o, parent=data.parent, time=t, log_length=data.log_length, fp=data.fp, noise_model="scaled",
                          division_model="binomial")
    fn = ggp.Forest(neg)
    lln = ggp.total_likelihood(P, fn, raise_on_nan=False)
    assert raw_simulate(fn, P) == _lib.GGP_ERR_BAD_ARG
    assert same_bits(ggp.total_likelihood(P, fn, raise_on_nan=False), lln)
    fn.close()
    # statistics of a larger data set (compute_init = 0)
    fi, ri = data.init_stats()
    fz = ggp.Forest(with_series(data, data.log_length, data.fp, init_f=fi, init_r=ri))
    llz = ggp.total_likelihood(P, fz)
    assert raw_simulate(fz, P) == _lib.GGP_ERR_BAD_ARG
    assert same_bits(ggp.total_likelihood(P, fz), llz)
    fz.close()


def test_command_line_simulate(tmp_path):
    P = ggp.PARAMS_SCALED_BINOMIAL
    data = ggp.simulate_forest(8, 3, noise_model="scaled", division_model="binomial", seed=21)
    csv, cfg = write_inputs(tmp_path, data)
    pf = write_params(tmp_path / "p.txt", P * np.array([1.1, 1, 1, 0.9, 1, 1, 1, 1, 1, 1, 1]), free=(0, 3), bound=(8,))
    start = P * np.array([1.1, 1, 1, 0.9, 1, 1, 1, 1, 1, 1, 1])
    out = str(tmp_path / "sim")
    run(["-i", csv, "-b", pf, "-c", cfg, "--simulate", "7", "-o", out])
    sim, _, _ = io.read_forest_binary(os.path.join(out, "forest_simulated_7.bin"))
    f = ggp.Forest(data)
    x, g = ggp.simulate_series(f, start, seed=7)
    f.close()
    assert same_bits(sim.log_length, x) and same_bits(sim.fp, g) and same_bits(sim.time, data.time)
    # -m --fast on the simulated table = -m --fast on the written file
    finals = {}
    for name, args in (("sim", ["-i", csv, "--simulate", "7"]), ("bin", ["-i", os.path.join(out, "forest_simulated_7.bin")])):
        o = str(tmp_path / ("fit_" + name))
        run(args + ["-b", pf, "-c", cfg, "-m", "--fast", "--exact_errors", "-t", "1e-2", "-o", o])
        (path,) = glob.glob(os.path.join(o, "*_final.csv"))
        assert os.path.basename(path).startswith("forest_simulated_7_")   # named after the simulated table either way
        finals[name] = [line for line in open(path) if "forest" not in line]
    assert finals["sim"] == finals["bin"] and len(finals["sim"]) > 5


def test_command_line_bootstrap_loop_keeps_every_replicate(tmp_path):
    """the real data's fit and two replicates in ONE output directory: every run keeps its own files"""
    P = ggp.PARAMS_SCALED_BINOMIAL
    data = ggp.simulate_forest(8, 3, noise_model="scaled", division_model="binomial", seed=22)
    csv, cfg = write_inputs(tmp_path, data)
    pf = write_params(tmp_path / "p.txt", P, free=(0, 3))
    out = str(tmp_path / "boot")
    for extra in ([], ["--simulate", "1"], ["--simulate", "2"]):
        run(["-i", csv, "-b", pf, "-c", cfg, "-m", "--fast", "-t", "1e-2", "-o", out] + extra)
    finals = sorted(os.path.basename(p) for p in glob.glob(os.path.join(out, "*_final.csv")))
    iters = sorted(os.path.basename(p) for p in glob.glob(os.path.join(out, "*_iterations.csv")))
    logs = sorted(os.path.basename(p) for p in glob.glob(os.path.join(out, "*_success.log")))
    assert [f.split("_f")[0] for f in finals] == ["forest", "forest_simulated_1", "forest_simulated_2"], finals
    assert len(iters) == 3 and len(logs) == 3 and len(set(open(os.path.join(out, f)).read() for f in finals)) == 3


def test_root_prior_forms_and_group_init_stats():
    """root_prior as a 4-tuple, a list, an array or an (init_f, init_r) pair; ForestGroup.init_stats is the shards' statistics"""
    data = ggp.simulate_forest(20, 3, seed=50)
    P = ggp.PARAMS_CONST_GAUSS
    f = ggp.Forest(data)
    grp = ggp.ForestGroup(data, [0, 0])
    fi, ri = data.init_stats()
    assert all(same_bits(a, b) for a, b in zip(grp.init_stats(), f.init_stats()))
    assert same_bits(grp.init_stats()[0], fi)
    want = ggp.simulate_series(f, P, seed=4, root_prior=fi)
    for prior in (tuple(float(v) for v in fi), list(fi), (fi, ri), [fi, ri], np.stack([fi, ri]), grp.init_stats()):
        got = ggp.simulate_series(f, P, seed=4, root_prior=prior)
        assert same_bits(got[0], want[0]) and same_bits(got[1], want[1])
    with pytest.raises(ValueError):
        ggp.simulate_series(f, P, seed=4, root_prior=fi[:3])
    grp.close()
    f.close()
