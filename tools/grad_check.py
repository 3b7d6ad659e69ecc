#!/usr/bin/env python
"""Host evaluations of the gradient and the Hessian of the FAST log-likelihood (tests/hostcheck/gradcheck.cpp and
hesscheck.cpp, no GPU needed):
  grad_host   dual numbers over ggp_fast.cuh in double with an N-node rule: the device gradient kernel's arithmetic up to FMA
              contraction
  grad_quad   central differences of the binary128 16-node evaluation, differenced in binary128: the truth
  hess_host   second-order Taylor numbers (GgpTaylor2) in double through the library's evaluation plan (GgpEvalPlan): the
              device's evaluations, seeding and unscaling
  hess_quad   second differences of the binary128 16-node evaluation, differenced in binary128: the truth
  tree_host   grad_host per lineage tree (tests/hostcheck/treecheck.cpp): every cell's dual number added into its tree
  tree_quad   central differences of every tree's binary128 16-node log-likelihood: the per-tree truth
The libraries are compiled on first use (g++, -lquadmath) next to their sources, or in a temporary directory if that is read-only.

  python tools/grad_check.py     prints the scaled errors of both on the example data set
"""
import ctypes as C
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from gfp_gaussian_process_b200 import _lib  # noqa: E402
from hostpass import make_desc  # noqa: E402

HC = os.path.join(ROOT, "tests", "hostcheck")
DEPS = [os.path.join(HC, "gradcheck.cpp"), os.path.join(HC, "fastcheck.cpp")] + \
       [os.path.join(ROOT, "gfp_gaussian_process_b200", "csrc", f) for f in ("ggp_fast.cuh", "ggp_dual.cuh", "ggp_types.cuh")]
_libs = {}


def _load(name):
    """tests/hostcheck/<name>.cpp as lib<name>.so, compiled on first use (next to the source, or in a temporary directory if
    that is read-only)"""
    if name not in _libs:
        src = os.path.join(HC, name + ".cpp")
        newest = max(os.path.getmtime(s) for s in DEPS + [src])
        lib = os.path.join(HC, f"lib{name}.so")
        if not os.access(HC, os.W_OK):
            lib = os.path.join(tempfile.gettempdir(), f"lib{name}-{os.getuid()}-{int(newest)}.so")
        if not os.path.exists(lib) or os.path.getmtime(lib) < newest:
            tmp = lib + f".{os.getpid()}.tmp"
            subprocess.check_call(["g++", "-std=gnu++17", "-O2", "-fPIC", "-shared", "-o", tmp, src, "-lquadmath"])
            os.replace(tmp, lib)
        _libs[name] = C.CDLL(lib)
    return _libs[name]


def gradcheck():
    return _load("gradcheck")


def hesscheck():
    return _load("hesscheck")


def treecheck():
    return _load("treecheck")


def _call(fn, data, params, *extra):
    p = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, 11)
    n = p.shape[0]
    total, grad, valid = np.zeros(n), np.zeros((n, 11)), np.zeros(n, dtype=np.int32)
    d = make_desc(data)
    dp = _lib.c_double_p
    rc = fn(C.byref(d), p.ctypes.data_as(dp), n, *extra, total.ctypes.data_as(dp), grad.ctypes.data_as(dp),
            valid.ctypes.data_as(C.POINTER(C.c_int)))
    assert rc == 0, rc
    return total, grad, valid


def grad_host(data, params, n_nodes):
    """(loglik [n], grad [n][11], valid [n]) of the dual-number evaluation in double"""
    return _call(gradcheck().gc_loglik_grad, data, params, C.c_int(n_nodes))


def grad_quad(data, params, rel_step=1e-9):
    """(loglik [n], grad [n][11], valid [n]): binary128 value and central differences with step rel_step |p_i|"""
    return _call(gradcheck().gc_grad_quad, data, params, C.c_double(rel_step))


def _dirs(dirs):
    d = np.arange(11, dtype=np.int32) if dirs is None else np.ascontiguousarray(dirs, dtype=np.int32).reshape(-1)
    return d, d.ctypes.data_as(C.POINTER(C.c_int)), C.c_int(d.size)


def hess_host(data, params, n_nodes, dirs=None):
    """(loglik [n], grad [n][k], hess [n][k][k], valid [n]) of the GgpTaylor2 evaluation in double over dirs (None = all 11)"""
    p = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, 11)
    n = p.shape[0]
    d, dp, nd = _dirs(dirs)
    total, grad, hess, valid = np.zeros(n), np.zeros((n, d.size)), np.zeros((n, d.size, d.size)), np.zeros(n, dtype=np.int32)
    desc = make_desc(data)
    c = _lib.c_double_p
    rc = hesscheck().gc_loglik_hess(C.byref(desc), p.ctypes.data_as(c), n, C.c_int(n_nodes), dp, nd, total.ctypes.data_as(c),
                                    grad.ctypes.data_as(c), hess.ctypes.data_as(c), valid.ctypes.data_as(C.POINTER(C.c_int)))
    assert rc == 0, rc
    return total, grad, hess, valid


def hess_quad(data, params, dirs=None, rel_step=1e-8):
    """(loglik [n], hess [n][k][k], valid [n]): binary128 value and second differences with steps rel_step |p_i| over dirs"""
    p = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, 11)
    n = p.shape[0]
    d, dp, nd = _dirs(dirs)
    total, hess, valid = np.zeros(n), np.zeros((n, d.size, d.size)), np.zeros(n, dtype=np.int32)
    desc = make_desc(data)
    c = _lib.c_double_p
    rc = hesscheck().gc_hess_quad(C.byref(desc), p.ctypes.data_as(c), n, C.c_double(rel_step), dp, nd, total.ctypes.data_as(c),
                                  hess.ctypes.data_as(c), valid.ctypes.data_as(C.POINTER(C.c_int)))
    assert rc == 0, rc
    return total, hess, valid


def _n_roots(data):
    return int(np.sum(np.asarray(data.parent) < 0))


def tree_host(data, params, n_nodes):
    """(tree_ll [n][R], tree_grad [n][R][11], tree_abs [n][R], valid [n]) of the dual-number evaluation in double, per tree (roots
    in cell order); tree_abs: the sum of |cell log-likelihood| over the tree's cells"""
    p = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, 11)
    n, R = p.shape[0], _n_roots(data)
    ll, grad, ab, valid = np.zeros((n, R)), np.zeros((n, R, 11)), np.zeros((n, R)), np.zeros(n, dtype=np.int32)
    desc = make_desc(data)
    c = _lib.c_double_p
    rc = treecheck().tc_tree_grad(C.byref(desc), p.ctypes.data_as(c), n, C.c_int(n_nodes), ll.ctypes.data_as(c), grad.ctypes.data_as(c),
                                  ab.ctypes.data_as(c), valid.ctypes.data_as(C.POINTER(C.c_int)))
    assert rc == 0, rc
    return ll, grad, ab, valid


def tree_quad(data, params, rel_step=1e-9):
    """(tree_ll [n][R], tree_grad [n][R][11], valid [n]): every tree's binary128 value and central differences with step
    rel_step |p_i|"""
    p = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, 11)
    n, R = p.shape[0], _n_roots(data)
    ll, grad, valid = np.zeros((n, R)), np.zeros((n, R, 11)), np.zeros(n, dtype=np.int32)
    desc = make_desc(data)
    c = _lib.c_double_p
    rc = treecheck().tc_tree_quad(C.byref(desc), p.ctypes.data_as(c), n, C.c_double(rel_step), ll.ctypes.data_as(c), grad.ctypes.data_as(c),
                                  valid.ctypes.data_as(C.POINTER(C.c_int)))
    assert rc == 0, rc
    return ll, grad, valid


def scaled_tree_error(params, g, truth, tree_abs):
    """|p_i| |s_ti - t_ti| / sum over the cells c of tree t of |ll_c|, per (tree, direction): g, truth [R][n], tree_abs [R]"""
    return np.abs(np.asarray(params))[None, :] * np.abs(np.asarray(g) - np.asarray(truth)) / np.asarray(tree_abs)[:, None]


def scaled_hess_error(params, dirs, H, truth, loglik):
    """|p_i| |p_j| |H_ij - T_ij| / |loglik| over the directions dirs (None = all 11)"""
    p = np.abs(np.asarray(params, dtype=np.float64)[np.arange(11) if dirs is None else np.asarray(dirs)])
    return np.outer(p, p) * np.abs(np.asarray(H) - np.asarray(truth)) / abs(loglik)


def polarization_ratio(params, dirs, H, loglik):
    """s_i^2 |H_ii| / |loglik|: the size of the terms polarization subtracts against the log-likelihood (DESIGN.md 5.7)"""
    p = np.asarray(params, dtype=np.float64)[np.arange(11) if dirs is None else np.asarray(dirs)]
    s = np.array([hess_scale(x) for x in p])
    return s ** 2 * np.abs(np.diag(H)) / abs(loglik)


def hess_scale(p):
    """ggp_hess_scale: the power of two nearest |p|, 1 for 0"""
    a = abs(float(p))
    if not (a > 0.0) or not np.isfinite(a):
        return 1.0
    m, e = np.frexp(a)
    return float(np.ldexp(1.0, int(e) if m >= 0.75 else int(e) - 1))


def scaled_error(params, g, truth, loglik):
    """|p_i| |g_i - t_i| / |loglik| per direction"""
    return np.abs(params) * np.abs(np.asarray(g) - np.asarray(truth)) / abs(loglik)


def main():
    from conftest import example_data
    data, z = example_data(os.path.join(ROOT, "tests", "golden"))
    P = np.asarray(z["params"])
    q, gq, _ = grad_quad(data, P)
    for n in (5, 6, 8):
        ll, g, valid = grad_host(data, P, n)
        e = scaled_error(P, g[0], gq[0], q[0])
        print(f"N={n} valid={valid[0]} value vs quad {abs(ll[0] - q[0]) / abs(q[0]):.2e}  scaled gradient error max {e.max():.2e}  "
              f"per direction {np.array2string(e, precision=1)}")


if __name__ == "__main__":
    main()
