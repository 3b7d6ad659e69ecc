#!/usr/bin/env python
"""Host build of the series simulator (tests/hostcheck/simcheck.cpp, no GPU needed): the per-cell body of csrc/ggp_sim.cuh
compiled with g++ -ffp-contract=off, which returns the bits ggp_simulate returns on the device.
  philox(ctr, key)                                     Philox4x32-10 of one counter (4 x uint32), key a uint64
  sim_host(data, params, seed, substeps, root_prior)   (log_length [n_ctp], fp [n_ctp], first non-finite cell or -1)
The library is compiled on first use (g++) next to its source, or in a temporary directory if that is read-only.

  python tools/sim_check.py     simulates on the example data set's genealogy and prints summary statistics
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
CSRC = os.path.join(ROOT, "gfp_gaussian_process_b200", "csrc")
DEPS = [os.path.join(HC, "simcheck.cpp"), os.path.join(ROOT, "include", "ggp_b200.h")] + \
       [os.path.join(CSRC, f) for f in ("ggp_sim.cuh", "ggp_libm.cuh", "ggp_types.cuh", "ggp_layout.hpp", "ggp_tables_data.h")]
_lib_sim = None


def simcheck():
    """tests/hostcheck/simcheck.cpp as libsimcheck.so, compiled on first use"""
    global _lib_sim
    if _lib_sim is None:
        newest = max(os.path.getmtime(s) for s in DEPS)
        lib = os.path.join(HC, "libsimcheck.so")
        if not os.access(HC, os.W_OK):
            lib = os.path.join(tempfile.gettempdir(), f"libsimcheck-{os.getuid()}-{int(newest)}.so")
        if not os.path.exists(lib) or os.path.getmtime(lib) < newest:
            tmp = lib + f".{os.getpid()}.tmp"
            subprocess.check_call(["g++", "-std=gnu++17", "-O2", "-fPIC", "-ffp-contract=off", "-shared", "-o", tmp, DEPS[0]])
            os.replace(tmp, lib)
        _lib_sim = C.CDLL(lib)
        _lib_sim.sc_simulate.argtypes = [C.c_void_p, _lib.c_double_p, C.c_uint64, C.c_int, _lib.c_double_p, _lib.c_double_p,
                                         _lib.c_double_p, C.POINTER(C.c_longlong)]
        _lib_sim.sc_philox.argtypes = [C.POINTER(C.c_uint32), C.c_uint64, C.POINTER(C.c_uint32)]
    return _lib_sim


def philox(ctr, key):
    c = np.ascontiguousarray(ctr, dtype=np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    simcheck().sc_philox(c.ctypes.data_as(C.POINTER(C.c_uint32)), C.c_uint64(int(key)), out.ctypes.data_as(C.POINTER(C.c_uint32)))
    return out


def sim_host(data, params, seed, substeps=8, root_prior=None):
    p = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, 11)
    x, g = np.empty(data.n_ctp), np.empty(data.n_ctp)
    bad = C.c_longlong(0)
    d = make_desc(data)
    r = None if root_prior is None else np.ascontiguousarray(root_prior, dtype=np.float64)
    rc = simcheck().sc_simulate(C.byref(d), p.ctypes.data_as(_lib.c_double_p), C.c_uint64(int(seed)), int(substeps),
                                None if r is None else r.ctypes.data_as(_lib.c_double_p), x.ctypes.data_as(_lib.c_double_p),
                                g.ctypes.data_as(_lib.c_double_p), C.byref(bad))
    assert rc == 0, rc
    return x, g, bad.value


def main():
    from conftest import example_data
    data, z = example_data(os.path.join(ROOT, "tests", "golden"))
    P = np.asarray(z["params"])
    x, g, bad = sim_host(data, P, 7)
    print(f"example genealogy: {data.n_cells} cells, {data.n_ctp} points; simulated log_length mean {x.mean():.4f} sd {x.std():.4f} "
          f"(data {data.log_length.mean():.4f} / {data.log_length.std():.4f}), fp mean {g.mean():.1f} sd {g.std():.1f} "
          f"(data {data.fp.mean():.1f} / {data.fp.std():.1f}), first non-finite cell {bad}")


if __name__ == "__main__":
    main()
