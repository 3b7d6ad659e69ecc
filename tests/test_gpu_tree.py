"""Per-tree scores of the FAST log-likelihood on the GPU (ggp_loglik_tree_grad, ggp_group_loglik_tree_grad, tree_scores,
sandwich_error_bars and the command line's --robust_errors): the device rows against the host build of the same dual-number
code added per tree (tests/hostcheck/treecheck.cpp), against the totals, and against ggp_loglik_grad's bits; reproducibility,
direction subsets, chunking, the re-run ladder, the error rows and the group.  With 6 or more nodes the lanes of a warp share a
polynomial level (ggp_fast.cuh), so a cell's bits depend on its warp neighbours: device against host, and group against single
forest, are compared by tolerance."""
import os
import sys

import numpy as np
import pytest

from conftest import same_bits, max_rel, ROOT
import gfp_gaussian_process_b200 as ggp
from gfp_gaussian_process_b200 import _lib
from test_gpu_cli import write_inputs, write_params, run, read_table

sys.path.insert(0, os.path.join(ROOT, "tools"))
from grad_check import scaled_error, scaled_tree_error, tree_host  # noqa: E402

pytestmark = pytest.mark.gpu

COMBOS = [("const", "gauss"), ("scaled", "binomial"), ("scaled", "gauss"), ("const", "binomial")]


def params_of(noise):
    return ggp.PARAMS_CONST_GAUSS if noise == "const" else ggp.PARAMS_SCALED_BINOMIAL


def raw_tree(f, vecs, dirs=None, with_ll=True, with_grad=True, n_vec=None):
    """ggp_loglik_tree_grad (Forest) or ggp_group_loglik_tree_grad (ForestGroup) through the C ABI:
    (rc, loglik, grad, tree_ll, tree_grad, [(cell, t_index)])"""
    lib = _lib.load()
    p = np.ascontiguousarray(vecs, dtype=np.float64).reshape(-1, 11)
    n = p.shape[0]
    d = None if dirs is None else np.ascontiguousarray(dirs, dtype=np.int32)
    nd = 11 if d is None else d.size
    group = isinstance(f, ggp.ForestGroup)
    R = lib.ggp_group_n_roots(f.handle) if group else f.n_roots
    ll, g, tl, tg = np.full(n, -7.0), np.full((n, nd), -7.0), np.full((n, R), -7.0), np.full((n, R, nd), -7.0)
    nan = (_lib.NanInfo * n)()
    c = _lib.c_double_p
    fn = lib.ggp_group_loglik_tree_grad if group else lib.ggp_loglik_tree_grad
    rc = fn(f.handle, p.ctypes.data_as(c), n if n_vec is None else n_vec, None if d is None else d.ctypes.data_as(_lib.c_int32_p), nd,
            ll.ctypes.data_as(c), g.ctypes.data_as(c), tl.ctypes.data_as(c) if with_ll else None, tg.ctypes.data_as(c) if with_grad else None,
            nan)
    return rc, ll, g, tl, tg, [(nan[v].cell, nan[v].t_index) for v in range(n)]


def roots_of(data):
    """tree number of every cell (roots numbered in cell order)"""
    parent = np.asarray(data.parent)
    tree = -np.ones(data.n_cells, dtype=np.int64)
    roots = np.flatnonzero(parent < 0)
    tree[roots] = np.arange(len(roots))
    for c in range(data.n_cells):
        chain, u = [], c
        while tree[u] < 0:
            chain.append(u)
            u = parent[u]
        tree[chain] = tree[u]
    return tree


def check_sums(f, data, vecs, ll, g, tl, tg):
    """sum_t tree_grad against out_grad (1e-13 scaled), sum_t tree_ll against out_loglik (1e-14) and against the fast per-cell
    rows added per tree (1e-14)"""
    mode = _lib.load().ggp_forest_get_mode(f.handle) if isinstance(f, ggp.Forest) else None
    for i in range(len(vecs)):
        assert np.max(scaled_error(vecs[i], tg[i].sum(axis=0), g[i], ll[i])) <= 1e-13
        assert abs(tl[i].sum() - ll[i]) / abs(ll[i]) <= 1e-14
    if mode is not None:
        f.set_mode(f.last_fast_nodes)
        fast, cells = ggp.total_likelihood(vecs, f, per_cell=True)
        tree = roots_of(data)
        for i in range(len(vecs)):
            per_tree = np.bincount(tree, weights=cells[i], minlength=tl.shape[1])
            assert max_rel(tl[i], per_tree) <= 1e-14
        f.set_mode(mode)


@pytest.mark.parametrize("nodes", [5, 6])
@pytest.mark.parametrize("noise,division", COMBOS)
def test_device_tree_rows_match_the_host_per_tree_evaluation(noise, division, nodes):
    P = params_of(noise)
    d = ggp.simulate_forest(40, 5, params=P, noise_model=noise, division_model=division, seed=61)
    vecs = np.stack([P, P * 1.02])
    f = ggp.Forest(d)
    f.set_mode(nodes)
    rc, ll, g, tl, tg, _ = raw_tree(f, vecs)
    assert rc == _lib.GGP_OK and f.last_fast_nodes == nodes and tl.shape == (2, 40) and tg.shape == (2, 40, 11)
    for i in range(2):
        # the ladder: a vector the rule flags takes its rows from the next larger rule that accepts it
        rule = nodes
        while not tree_host(d, vecs[i], rule)[3][0]:
            rule = {5: 6, 6: 8, 8: 10}[rule]
        if noise == "const":
            assert rule == nodes
        hl, hg, ab, _ = tree_host(d, vecs[i], rule)
        e = scaled_tree_error(vecs[i], tg[i], hg[0], ab[0])
        el = np.abs(tl[i] - hl[0]) / ab[0]
        print(f"{noise}/{division} N={nodes} (accepted by {rule}) vector {i}: tree scores vs host {e.max():.2e}, tree values {el.max():.2e}")
        assert e.max() <= 1e-13 and el.max() <= 1e-13
    check_sums(f, d, vecs, ll, g, tl, tg)
    f.close()


def test_tree_call_gives_the_gradient_bits_repeats_and_subsets_are_columns(monkeypatch):
    P = ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(50, 5, params=P, noise_model="scaled", division_model="binomial", seed=62)
    vecs = P * np.exp(np.random.default_rng(4).uniform(-0.04, 0.04, size=(3, 11)))
    f = ggp.Forest(d)
    gl, gg = ggp.total_likelihood_grad(vecs, f)
    ll, g, tl, tg = ggp.tree_scores(vecs, f)
    assert same_bits(ll, gl) and same_bits(g, gg)
    ll2, g2, tl2, tg2 = ggp.tree_scores(vecs, f)
    assert same_bits(ll2, ll) and same_bits(g2, g) and same_bits(tl2, tl) and same_bits(tg2, tg)
    for dirs in ([4], [10, 0, 3], [0, 1, 2, 3, 4, 5, 6]):
        lls, gs, tls, tgs = ggp.tree_scores(vecs, f, dirs=dirs)
        assert same_bits(gs, g[:, dirs]) and same_bits(lls, ll) and same_bits(tls, tl) and same_bits(tgs, tg[:, :, dirs])
        assert same_bits(gs, ggp.total_likelihood_grad(vecs, f, dirs=dirs)[1])
    # one vector and the objective's sign
    l1, g1, t1, s1 = ggp.tree_scores(vecs[0], f, negative=True)
    assert same_bits(l1, -ll[0]) and same_bits(s1, -tg[0]) and t1.shape == (50,)
    # NULL tree_ll: the same gradient rows
    rc, _, gn, _, tgn, _ = raw_tree(f, vecs, with_ll=False)
    assert rc == _lib.GGP_OK and same_bits(tgn, tg) and same_bits(gn, g)
    f.close()
    # chunking: one vector's 11 evaluations fit the budget, two do not; then only 4 evaluations of one vector per launch
    for budget in (d.n_cells * 14 * 2 * 8 * 11 + 8, d.n_cells * 14 * 2 * 8 * 4 + 8):
        monkeypatch.setenv("GGP_B200_STATE_BUDGET", str(budget))
        fc = ggp.Forest(d)
        llc, gc, tlc, tgc = ggp.tree_scores(vecs, fc)
        monkeypatch.delenv("GGP_B200_STATE_BUDGET")
        assert same_bits(llc, ll) and same_bits(gc, g) and same_bits(tlc, tl) and same_bits(tgc, tg)
        assert same_bits(gc, ggp.total_likelihood_grad(vecs, fc)[1])
        fc.close()


def test_tree_rows_after_upload_series_equal_a_fresh_forest(monkeypatch):
    monkeypatch.setenv("GGP_B200_UPLOAD_CHUNKS", "3")
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(40, 4, seed=63)
    f = ggp.Forest(d)
    ggp.tree_scores(P, f)
    rng = np.random.default_rng(6)
    x2 = d.log_length + rng.normal(0, 1e-3, d.n_ctp)
    g2 = d.fp * (1 + rng.normal(0, 1e-3, d.n_ctp))
    f.upload_series(None, x2.ctypes.data, g2.ctypes.data)
    vecs = np.stack([P, P * 1.01])
    r = ggp.tree_scores(vecs, f)
    d2 = ggp.LineageData(cell_offset=d.cell_offset, parent=d.parent, time=d.time, log_length=x2, fp=g2, segment=d.segment,
                         noise_model=d.noise_model, division_model=d.division_model, fp_auto=d.fp_auto)
    f2 = ggp.Forest(d2)
    r2 = ggp.tree_scores(vecs, f2)
    assert all(same_bits(a, b) for a, b in zip(r, r2))
    f.close()
    f2.close()


def test_uncovered_and_nan_vectors_get_nan_tree_rows_and_arguments_are_refused():
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(30, 4, seed=64)
    wide = P.copy()
    wide[4] = 2.0   # no rule covers it
    bad = P.copy()
    bad[7] = -1.0   # a NaN term
    f = ggp.Forest(d)
    lib = _lib.load()
    vecs = np.stack([P, wide, P * 1.01, bad])
    rc0, ll0, g0, tl0, tg0, _ = raw_tree(f, vecs[[0, 2]])
    assert rc0 == _lib.GGP_OK
    rg = lib.ggp_loglik_grad
    rcg = rg(f.handle, np.ascontiguousarray(vecs).ctypes.data_as(_lib.c_double_p), 4, None, 11,
             np.empty(4).ctypes.data_as(_lib.c_double_p), np.empty((4, 11)).ctypes.data_as(_lib.c_double_p), None)
    msg_g = lib.ggp_last_error().decode()
    rc, ll, g, tl, tg, nan = raw_tree(f, vecs)
    msg = lib.ggp_last_error().decode()
    assert rc == rcg == _lib.GGP_ERR_BAD_ARG and msg == msg_g and "vector(s) 1 " in msg
    for i, j in ((0, 0), (2, 1)):
        assert same_bits(tl[i], tl0[j]) and same_bits(tg[i], tg0[j]) and same_bits(g[i], g0[j])
    for i in (1, 3):
        assert np.all(np.isnan(g[i])) and np.all(np.isnan(tl[i])) and np.all(np.isnan(tg[i]))
    assert np.isnan(ll[3]) and nan[3][0] >= 0 and nan[1] == (-1, -1)
    rc, _, _, tl, tg, _ = raw_tree(f, np.stack([P, bad]))
    assert rc == _lib.GGP_ERR_NAN and same_bits(tg[0], tg0[0]) and np.all(np.isnan(tg[1]))
    with pytest.raises(ggp.LikelihoodNaN):
        ggp.tree_scores(np.stack([P, bad]), f)
    with pytest.raises(_lib.GgpError):
        ggp.tree_scores(wide, f)
    # refused before anything is written
    for kw in (dict(with_grad=False), dict(n_vec=0), dict(n_vec=-1), dict(dirs=[11]), dict(dirs=[2, 2])):
        rc, ll, g, tl, tg, _ = raw_tree(f, P, **kw)
        assert rc == _lib.GGP_ERR_BAD_ARG
        assert np.all(ll == -7.0) and np.all(g == -7.0) and np.all(tl == -7.0) and np.all(tg == -7.0)
    f.close()


def test_other_calls_return_the_same_bits_after_a_tree_call():
    P = ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(40, 5, params=P, noise_model="scaled", division_model="binomial", seed=65)
    vecs = np.stack([P, P * 1.02, P * 0.98])
    f = ggp.Forest(d)
    before_s = ggp.total_likelihood(vecs, f, per_cell=True)
    f.set_mode("fast")
    before_f = ggp.total_likelihood(vecs, f, per_cell=True)
    n_before = f.last_fast_nodes
    before_g = ggp.total_likelihood_grad(vecs, f)
    f.set_mode("strict")
    ggp.tree_scores(np.tile(P, (7, 1)), f)
    after_s = ggp.total_likelihood(vecs, f, per_cell=True)
    f.set_mode("fast")
    ggp.tree_scores(P, f)
    after_f = ggp.total_likelihood(vecs, f, per_cell=True)
    assert same_bits(before_s[0], after_s[0]) and same_bits(before_s[1], after_s[1])
    assert same_bits(before_f[0], after_f[0]) and same_bits(before_f[1], after_f[1]) and f.last_fast_nodes == n_before
    after_g = ggp.total_likelihood_grad(vecs, f)
    assert same_bits(before_g[0], after_g[0]) and same_bits(before_g[1], after_g[1])
    f.close()


def shuffled_trees(d, seed):
    """the same forest with its trees interleaved in the cell order (not stored tree by tree: the group bin-packs)"""
    order = np.random.default_rng(seed).permutation(d.n_cells)
    parent = np.asarray(d.parent)
    remap = np.empty(d.n_cells, dtype=np.int64)
    remap[order] = np.arange(d.n_cells)
    n = np.diff(d.cell_offset)[order]
    off = np.concatenate([[0], np.cumsum(n)])
    ctp = np.repeat(d.cell_offset[order] - off[:-1], n) + np.arange(off[-1])
    par = parent[order]
    return ggp.LineageData(cell_offset=off, parent=np.where(par >= 0, remap[np.maximum(par, 0)], -1), time=d.time[ctp],
                           log_length=d.log_length[ctp], fp=d.fp[ctp], segment=d.segment[ctp], noise_model=d.noise_model,
                           division_model=d.division_model, fp_auto=d.fp_auto)


@pytest.mark.parametrize("layout", ["contiguous", "bin-packed"])
def test_group_tree_rows_agree_with_the_single_forest(layout):
    P = ggp.PARAMS_SCALED_BINOMIAL
    d = ggp.simulate_forest(40, 5, params=P, noise_model="scaled", division_model="binomial", seed=66)
    if layout == "bin-packed":
        d = shuffled_trees(d, 7)
    vecs = np.stack([P, P * 1.03])
    f = ggp.Forest(d)
    f.set_mode(6)
    ll, g, tl, tg = ggp.tree_scores(vecs, f)
    grp = ggp.ForestGroup(d, [0, 0])
    grp.set_mode(6)
    assert grp.contiguous == (layout == "contiguous")
    assert _lib.load().ggp_group_n_roots(grp.handle) == f.n_roots == grp.n_roots
    llg, gg, tlg, tgg = ggp.tree_scores(vecs, grp)
    _, gref = ggp.total_likelihood_grad(vecs, grp)
    assert same_bits(gg, gref)
    assert max_rel(llg, ll) <= 1e-13
    _, _, ab, _ = tree_host(d, vecs, 6)
    for i in range(2):
        assert np.max(scaled_tree_error(vecs[i], tgg[i], tg[i], ab[i])) <= 1e-13
        assert np.max(np.abs(tlg[i] - tl[i]) / ab[i]) <= 1e-13
        assert np.max(scaled_error(vecs[i], tgg[i].sum(axis=0), gg[i], llg[i])) <= 1e-13
    lls, gs, tls, tgs = ggp.tree_scores(vecs, grp, dirs=[2, 5])
    assert same_bits(gs, gg[:, [2, 5]]) and same_bits(tgs, tgg[:, :, [2, 5]]) and same_bits(tls, tlg)
    hv, rv, H, J = ggp.sandwich_error_bars(P, grp, dirs=[0, 3])
    hv1, rv1, H1, J1 = ggp.sandwich_error_bars(P, f, dirs=[0, 3])
    assert max_rel(hv, hv1) <= 1e-9 and max_rel(rv, rv1) <= 1e-9
    grp.close()
    f.close()


def test_tree_rows_at_configs1_size():
    """BASELINE configs[1] (10 000 trees x 6 generations), resident: every tree row is finite and the rows add up to the totals"""
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(10000, 6, seed=20261018)
    f = ggp.Forest(d)
    f.set_mode(5)
    vecs = P[None, :]
    ll, g, tl, tg = ggp.tree_scores(vecs, f)
    assert tl.shape == (1, 10000) and tg.shape == (1, 10000, 11)
    assert np.all(np.isfinite(tl)) and np.all(np.isfinite(tg)) and f.last_strict_reruns == 0
    gl, gg = ggp.total_likelihood_grad(vecs, f)
    assert same_bits(gl, ll) and same_bits(gg, g)
    check_sums(f, d, vecs, ll, g, tl, tg)
    f.close()


def test_sandwich_error_bars_on_a_forest():
    P = ggp.PARAMS_CONST_GAUSS
    d = ggp.simulate_forest(200, 4, params=P, seed=67)
    f = ggp.Forest(d)
    dirs = [0, 3, 6]
    hv, rv, H, J = ggp.sandwich_error_bars(P, f, dirs=dirs)
    _, _, Hh = ggp.total_likelihood_hess(P, f, dirs=dirs)
    _, _, _, S = ggp.tree_scores(P, f, dirs=dirs)
    assert same_bits(H, Hh) and np.all(hv > 0) and np.all(rv > 0)
    assert max_rel(hv, -np.diag(np.linalg.inv(H))) <= 1e-12
    hs, rs = ggp.sandwich(H, S)
    assert same_bits(hs, hv) and same_bits(rs, rv)
    # simulated from the model: the sandwich is of the size of the model-based variance
    print(f"robust / hessian variance on data from the model: {rv / hv}")
    assert np.all(rv / hv > 0.2) and np.all(rv / hv < 5.0)
    with pytest.raises(ValueError, match="lineage trees for 11 free parameters"):
        ggp.sandwich_error_bars(P, ggp.Forest(ggp.simulate_forest(5, 3, seed=1)))
    f.close()


def test_robust_errors_option_writes_the_sandwich_and_the_trees_file(tmp_path):
    """-m --fast --robust_errors on 60 trees x 3 generations, three parameters not fixed: the new _final.csv section equals
    sandwich_error_bars at the best logged parameters; <base>_trees.csv has one row per tree whose score columns add up to the
    gradient; the --exact_errors section is the same bytes with and without the option; without it nothing changes; a single tree
    writes the 'not available' line"""
    P = ggp.PARAMS_SCALED_BINOMIAL
    data = ggp.simulate_forest(60, 3, noise_model="scaled", division_model="binomial", seed=68)
    csv, cfg = write_inputs(tmp_path, data)
    pf = write_params(tmp_path / "p.txt", P * np.array([1.1, 1, 1, 0.9, 1, 1, 1, 1, 1, 1, 1]), free=(0, 3), bound=(8,))
    finals = {}
    for name, extra in (("plain", []), ("exact", ["--exact_errors"]), ("robust", ["--robust_errors"]),
                        ("both", ["--exact_errors", "--robust_errors"])):
        out = str(tmp_path / name)
        run(["-i", csv, "-b", pf, "-c", cfg, "-m", "--fast", "-t", "1e-2", "-o", out] + extra)
        finals[name] = open(os.path.join(out, "forest_f03_b8_final.csv")).read()
        assert os.path.exists(os.path.join(out, "forest_f03_b8_trees.csv")) == ("robust" in name or name == "both")
    head = "\nerrors^2 (sandwich over lineage trees, fast log-likelihood):\n"
    assert head not in finals["plain"] and head not in finals["exact"]
    assert finals["robust"].startswith(finals["plain"]) and finals["both"].startswith(finals["exact"])
    section = finals["robust"][len(finals["plain"]):]
    assert section == finals["both"][len(finals["exact"]):]
    assert section.startswith(head)
    names, values = section[len(head):].strip().split("\n")
    assert names == "mean_lambda,mean_q,var_g"
    out = str(tmp_path / "robust")
    it = read_table(os.path.join(out, "forest_f03_b8_iterations.csv"), "iteration,")
    logged = np.array([[float(v) for v in r[1:]] for r in it])
    x = logged[np.argmax(logged[:, 11]), :11]
    dirs = [0, 3, 8]
    f = ggp.Forest(data)
    hv, rv, _, _ = ggp.sandwich_error_bars(x, f, dirs=dirs)
    got = np.array([float(v) for v in values.split(",")])
    print(f"--robust_errors {got} vs sandwich_error_bars {rv} (hessian {hv})")
    assert max_rel(got, rv) <= 1e-10
    trees = open(os.path.join(out, "forest_f03_b8_trees.csv")).read().strip().split("\n")
    assert trees[0] == "tree,root_cell_id,n_cells,n_points,log_likelihood,mean_lambda,mean_q,var_g"
    rows = [r.split(",") for r in trees[1:]]
    assert len(rows) == 60 and [int(r[0]) for r in rows] == list(range(60))
    assert sum(int(r[2]) for r in rows) == data.n_cells and sum(int(r[3]) for r in rows) == data.n_ctp
    S = np.array([[float(v) for v in r[5:]] for r in rows])
    tll = np.array([float(r[4]) for r in rows])
    ll, g = ggp.total_likelihood_grad(x, f, dirs=dirs)
    assert max_rel(S.sum(axis=0), g) <= 1e-9 and abs(tll.sum() - ll) / abs(ll) <= 1e-9
    f.close()
    # one tree: the 'not available' line, exit status 0
    one = ggp.simulate_forest(1, 4, noise_model="scaled", division_model="binomial", seed=69)
    (tmp_path / "one").mkdir()
    csv1, cfg1 = write_inputs(tmp_path / "one", one)
    out = str(tmp_path / "one" / "out")
    run(["-i", csv1, "-b", pf, "-c", cfg1, "-m", "--fast", "-t", "1e-2", "-o", out, "--robust_errors"])
    text = open(os.path.join(out, "forest_f03_b8_final.csv")).read()
    assert text.endswith(head + "mean_lambda,mean_q,var_g\nnot available: 1 lineage trees for 3 free parameters\n")
    assert len(open(os.path.join(out, "forest_f03_b8_trees.csv")).read().strip().split("\n")) == 2
