#!/usr/bin/env python
"""Gate report of the FAST likelihood step on the CPU (no GPU needed): total log-likelihood of
  ref    the oracle (== the reference's own source bit for bit, tests/test_ref_wrappers.py)
  fastN  ggp_fast.cuh in double with an N-node Gauss-Legendre rule (tests/hostcheck/fastcheck.cpp; the device kernel's arithmetic
         up to FMA contraction)
  quad   ggp_fast.cuh in binary128 with a 16-node rule: the value both are measured against
on the example data set, a configs[1] sample and a scaled/binomial forest, next to the reference's own +-1-ulp envelope
(profiles/r02_ulp_envelope.json, tools/ulp_envelope.py).  The gate of the fast mode is |fast - ref| / |ref| <= 1e-10.

  python tools/fast_gate.py [--small] [--out profiles/r02_fast_gate_cpu.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import gfp_gaussian_process_b200 as ggp  # noqa: E402
from gfp_gaussian_process_b200 import _lib  # noqa: E402
from oracle import oracle_py  # noqa: E402
from hostpass import make_desc  # noqa: E402

FC = os.path.join(ROOT, "tests", "hostcheck", "libfastcheck.so")


def fastcheck():
    """the host build of the fast step, compiled on first use next to its source, or in a temporary directory if that is
    read-only and holds no up-to-date build"""
    src = os.path.join(ROOT, "tests", "hostcheck", "fastcheck.cpp")
    hdr = os.path.join(ROOT, "gfp_gaussian_process_b200", "csrc", "ggp_fast.cuh")
    newest = max(os.path.getmtime(src), os.path.getmtime(hdr))
    lib = FC
    if not (os.path.exists(lib) and os.path.getmtime(lib) >= newest) and not os.access(os.path.dirname(lib), os.W_OK):
        lib = os.path.join(tempfile.gettempdir(), f"libfastcheck-{os.getuid()}-{int(newest)}.so")
    if not os.path.exists(lib) or os.path.getmtime(lib) < newest:
        tmp = lib + f".{os.getpid()}.tmp"
        subprocess.check_call(["g++", "-std=gnu++17", "-O2", "-fPIC", "-shared", "-o", tmp, src, "-lquadmath"])
        os.replace(tmp, lib)
    return C.CDLL(lib)


def fast_loglik(data, params, n_nodes=4, quad=False, per_cell=False, state=False):
    L = fastcheck()
    p = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, 11)
    n_vec = p.shape[0]
    total, valid = np.zeros(n_vec), np.zeros(n_vec, dtype=np.int32)
    pc = np.zeros((n_vec, data.n_cells)) if per_cell else None
    st = np.zeros((data.n_cells, 14)) if state else None
    d = make_desc(data)
    dp = _lib.c_double_p
    args = [C.byref(d), p.ctypes.data_as(dp), n_vec]
    if not quad:
        args.append(n_nodes)
    args += [pc.ctypes.data_as(dp) if per_cell else None, total.ctypes.data_as(dp), valid.ctypes.data_as(C.POINTER(C.c_int)),
             st.ctypes.data_as(dp) if state else None]
    rc = (L.fc_loglik_quad if quad else L.fc_loglik)(*args)
    assert rc == 0, rc
    return total, valid, pc, st


def datasets(small):
    from conftest import example_data
    ex, z = example_data(os.path.join(ROOT, "tests", "golden"))
    yield "example data set (scaled/binomial)", ex, np.asarray(z["params"])
    yield ("configs[1] sample (const/gauss)", ggp.simulate_forest(40 if small else 1500, 6, seed=20261018), ggp.PARAMS_CONST_GAUSS)
    yield ("scaled/binomial forest", ggp.simulate_forest(20 if small else 400, 6, noise_model="scaled", division_model="binomial",
                                                         seed=20261018), ggp.PARAMS_SCALED_BINOMIAL)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--small", action="store_true")
    ap.add_argument("--nodes", default="3,4,5,6,8")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r02_fast_gate_cpu.json"))
    a = ap.parse_args()
    res = {}
    for name, d, P in datasets(a.small):
        o = oracle_py.Oracle(d)
        ref, pc_ref = o.total_loglik(P, per_cell=True)
        q, vq, pc_q, _ = fast_loglik(d, P, quad=True, per_cell=True)
        row = {"n_ctp": int(d.n_ctp), "ref": ref, "quad": float(q[0]), "ref_vs_quad": abs(ref - q[0]) / abs(q[0]),
               "cell_ref_vs_quad_max": float(np.max(np.abs(pc_ref - pc_q[0]) / np.abs(pc_q[0]))), "fast": {}}
        print(f"{name}: {d.n_ctp} ctp  ref {ref!r}  quad {q[0]!r}  |ref-quad|/|quad| = {row['ref_vs_quad']:.2e}  (per cell max {row['cell_ref_vs_quad_max']:.1e})")
        for n in [int(v) for v in a.nodes.split(",")]:
            f, vf, pc_f, _ = fast_loglik(d, P, n_nodes=n, per_cell=True)
            r = {"loglik": float(f[0]), "valid": int(vf[0]), "vs_ref": abs(f[0] - ref) / abs(ref), "vs_quad": abs(f[0] - q[0]) / abs(q[0]),
                 "cell_vs_ref_max": float(np.max(np.abs(pc_f[0] - pc_ref) / np.abs(pc_ref))),
                 "cell_vs_quad_max": float(np.max(np.abs(pc_f[0] - pc_q[0]) / np.abs(pc_q[0])))}
            row["fast"][n] = r
            print(f"   N={n:2d} valid={r['valid']}  |fast-ref|/|ref| = {r['vs_ref']:.2e}   |fast-quad|/|quad| = {r['vs_quad']:.2e}   "
                  f"per cell: vs ref {r['cell_vs_ref_max']:.1e}, vs quad {r['cell_vs_quad_max']:.1e}")
        res[name] = row
    json.dump(res, open(a.out, "w"), indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
