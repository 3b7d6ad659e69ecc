#!/usr/bin/env python
"""Host evaluations of the gradient of the FAST log-likelihood (tests/hostcheck/gradcheck.cpp, no GPU needed):
  grad_host   dual numbers over ggp_fast.cuh in double with an N-node rule: the device gradient kernel's arithmetic up to FMA
              contraction
  grad_quad   central differences of the binary128 16-node evaluation, differenced in binary128: the truth
The library is compiled on first use (g++, -lquadmath) next to its source, or in a temporary directory if that is read-only.

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
SOURCES = [os.path.join(HC, "gradcheck.cpp"), os.path.join(HC, "fastcheck.cpp")] + \
          [os.path.join(ROOT, "gfp_gaussian_process_b200", "csrc", f) for f in ("ggp_fast.cuh", "ggp_dual.cuh")]
_gc = None


def gradcheck():
    global _gc
    if _gc is None:
        newest = max(os.path.getmtime(s) for s in SOURCES)
        lib = os.path.join(HC, "libgradcheck.so")
        if not os.access(HC, os.W_OK):
            lib = os.path.join(tempfile.gettempdir(), f"libgradcheck-{os.getuid()}-{int(newest)}.so")
        if not os.path.exists(lib) or os.path.getmtime(lib) < newest:
            tmp = lib + f".{os.getpid()}.tmp"
            subprocess.check_call(["g++", "-std=gnu++17", "-O2", "-fPIC", "-shared", "-o", tmp, SOURCES[0], "-lquadmath"])
            os.replace(tmp, lib)
        _gc = C.CDLL(lib)
    return _gc


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
