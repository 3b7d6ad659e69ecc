"""Host-side mirror of the reference's entry points for the hot path, above the C ABI.

Names, argument meaning and error behaviour follow the reference:
  total_likelihood(params_vec, cells)        likelihood.h:170-174 (returns +log-likelihood; the nlopt objective
                                             :125-159 returns the negative, `total_likelihood(..., negative=True)`)
  run_bound_1dscan                           main.cpp:77-112 (all samples of one parameter in ONE launch)
  num_hessian_ll                             likelihood.h:211-258 (the whole stencil in ONE launch)
  total_likelihood_grad, num_hessian_grad    no reference counterpart: the gradient of the fast log-likelihood (forward mode)
                                             and a Hessian as central differences of it
  total_likelihood_hess                      no reference counterpart: the exact Hessian of the fast log-likelihood (forward
                                             mode, second order)
  prediction_forward/backward + combine      predictions.h:166, 438, 466 (main.cpp:132-140)
A NaN running sum raises LikelihoodNaN carrying the first offending (cell, time index) in the reference's
depth-first order, where the reference throws std::domain_error("Likelihood is Nan") (likelihood.h:71-93).
"""
import ctypes as C

import numpy as np

from . import _lib
from .forest import Forest, ForestGroup


class LikelihoodNaN(ArithmeticError):
    def __init__(self, vec_index, cell, t_index):
        super().__init__(f"Likelihood is Nan (parameter vector {vec_index}, cell {cell}, time index {t_index})")
        self.vec_index, self.cell, self.t_index = vec_index, cell, t_index


def _as_params(params):
    p = np.ascontiguousarray(params, dtype=np.float64)
    single = p.ndim == 1
    p = p.reshape(-1, _lib.N_PARAMS)
    return p, single


def total_likelihood(params_vec, forest: Forest, root_carry=None, per_cell=False, negative=False, raise_on_nan=True):
    """+log-likelihood of one parameter vector (11 doubles) or of a batch [n_vec][11].

    root_carry: None = first ("fresh") evaluation; an array [n_roots][16] (zeros to start) reproduces the
    reference's history dependence across successive evaluations (SURVEY.md H3) and is updated in place.
    """
    lib = _lib.load()
    p, single = _as_params(params_vec)
    n_vec = p.shape[0]
    out = np.empty(n_vec)
    cell_ll = np.empty((n_vec, forest.n_cells)) if per_cell else None
    nan = (_lib.NanInfo * n_vec)()
    carry_p = None
    if root_carry is not None:
        if root_carry.dtype != np.float64 or not root_carry.flags.c_contiguous or root_carry.size != forest.n_roots * 16:
            raise ValueError("root_carry must be a C-contiguous float64 array [n_roots][16]")
        carry_p = root_carry.ctypes.data_as(_lib.c_double_p)
    rc = lib.ggp_loglik(forest.handle, p.ctypes.data_as(_lib.c_double_p), n_vec, carry_p,
                        out.ctypes.data_as(_lib.c_double_p),
                        cell_ll.ctypes.data_as(_lib.c_double_p) if per_cell else None, nan)
    _lib.check(rc, allow=(_lib.GGP_ERR_NAN,))
    if rc == _lib.GGP_ERR_NAN and raise_on_nan:
        for v in range(n_vec):
            if nan[v].cell >= 0:
                raise LikelihoodNaN(v, nan[v].cell, nan[v].t_index)
    if negative:
        out = -out
    res = out[0] if single else out
    if per_cell:
        return res, (cell_ll[0] if single else cell_ll)
    return res


def total_likelihood_grad(params_vec, forest, dirs=None, negative=False):
    """(log-likelihood, gradient) of one parameter vector (11 doubles) or of a batch [n_vec][11], natural space.

    The fast arithmetic whatever the forest's mode (ggp_loglik_grad): the log-likelihood is the fast value, the gradient its
    exact derivative by forward-mode dual numbers.  dirs: None = all 11 parameters, else the parameter indices to differentiate
    (gradient columns in that order).  negative: the objective's sign (-log-likelihood and its gradient).  forest: a Forest or a
    ForestGroup.  A vector that meets a NaN term raises LikelihoodNaN; one that no quadrature rule covers raises GgpError.
    """
    lib = _lib.load()
    p, single = _as_params(params_vec)
    n_vec = p.shape[0]
    d = None if dirs is None else np.ascontiguousarray(dirs, dtype=np.int32).reshape(-1)
    n_dirs = _lib.N_PARAMS if d is None else d.size
    ll = np.empty(n_vec)
    grad = np.empty((n_vec, n_dirs))
    nan = (_lib.NanInfo * n_vec)()
    fn = lib.ggp_group_loglik_grad if isinstance(forest, ForestGroup) else lib.ggp_loglik_grad
    rc = fn(forest.handle, p.ctypes.data_as(_lib.c_double_p), n_vec, None if d is None else d.ctypes.data_as(_lib.c_int32_p), n_dirs,
            ll.ctypes.data_as(_lib.c_double_p), grad.ctypes.data_as(_lib.c_double_p), nan)
    _lib.check(rc, allow=(_lib.GGP_ERR_NAN,))
    if rc == _lib.GGP_ERR_NAN:
        for v in range(n_vec):
            if nan[v].cell >= 0:
                raise LikelihoodNaN(v, nan[v].cell, nan[v].t_index)
    if negative:
        ll, grad = -ll, -grad
    return (ll[0], grad[0]) if single else (ll, grad)


def total_likelihood_hess(params_vec, forest, dirs=None, negative=False):
    """(log-likelihood, gradient, Hessian) of one parameter vector (11 doubles) or of a batch [n_vec][11], natural space.

    The fast arithmetic whatever the forest's mode (ggp_loglik_hess): the log-likelihood is the fast value, the gradient and the
    Hessian its exact derivatives (second-order Taylor numbers and polarization, no step size; the Hessian is symmetric bit for
    bit).  dirs: None = all 11 parameters, else the parameter indices to differentiate (rows and columns in that order).
    negative: the objective's sign.  forest: a Forest or a ForestGroup.  A vector that meets a NaN term raises LikelihoodNaN;
    one that no quadrature rule covers raises GgpError.  Error bars: -diag(inv(H)).
    """
    lib = _lib.load()
    p, single = _as_params(params_vec)
    n_vec = p.shape[0]
    d = None if dirs is None else np.ascontiguousarray(dirs, dtype=np.int32).reshape(-1)
    n_dirs = _lib.N_PARAMS if d is None else d.size
    ll = np.empty(n_vec)
    grad = np.empty((n_vec, n_dirs))
    hess = np.empty((n_vec, n_dirs, n_dirs))
    nan = (_lib.NanInfo * n_vec)()
    fn = lib.ggp_group_loglik_hess if isinstance(forest, ForestGroup) else lib.ggp_loglik_hess
    rc = fn(forest.handle, p.ctypes.data_as(_lib.c_double_p), n_vec, None if d is None else d.ctypes.data_as(_lib.c_int32_p), n_dirs,
            ll.ctypes.data_as(_lib.c_double_p), grad.ctypes.data_as(_lib.c_double_p), hess.ctypes.data_as(_lib.c_double_p), nan)
    _lib.check(rc, allow=(_lib.GGP_ERR_NAN,))
    if rc == _lib.GGP_ERR_NAN:
        for v in range(n_vec):
            if nan[v].cell >= 0:
                raise LikelihoodNaN(v, nan[v].cell, nan[v].t_index)
    if negative:
        ll, grad, hess = -ll, -grad, -hess
    return (ll[0], grad[0], hess[0]) if single else (ll, grad, hess)


def arange(start, stop, step=1.0):
    """utils.h:96-103: accumulating `value += step` (NOT numpy's start + i*step)."""
    vals = []
    value = float(start)
    while value < stop:
        vals.append(value)
        value += step
    return np.array(vals)


def run_bound_1dscan(forest: Forest, params_vec, index, lower, upper, step, root_carry=None):
    """1-d scan of parameter `index` over arange(lower, upper, step) (main.cpp:77-112).
    Returns (sampling, loglik[sampling])."""
    sampling = arange(lower, upper, step)
    P = np.tile(np.asarray(params_vec, dtype=np.float64), (sampling.shape[0], 1))
    P[:, index] = sampling
    return sampling, total_likelihood(P, forest, root_carry=root_carry, raise_on_nan=False)


def hessian_stencil(params_vec, idx_non_fixed, epsilon):
    """the 4 * n^2 parameter vectors num_hessian_ll evaluates, in its order (likelihood.h:228-254)."""
    x = np.asarray(params_vec, dtype=np.float64)
    vecs, hs = [], []
    for ii in idx_non_fixed:
        for jj in idx_non_fixed:
            h1 = max(x[ii] * epsilon, 1e-12)
            h2 = max(x[jj] * epsilon, 1e-12)
            for s1, s2 in ((+1, +1), (+1, -1), (-1, +1), (-1, -1)):
                v = x.copy()
                v[ii] = v[ii] + s1 * h1
                v[jj] = v[jj] + s2 * h2
                vecs.append(v)
            hs.append((h1, h2))
    return np.array(vecs), hs


def num_hessian_ll(forest: Forest, params_vec, idx_non_fixed, epsilon, root_carry=None):
    """Numerical Hessian of the log-likelihood (likelihood.h:211-258), all stencil points in one launch."""
    vecs, hs = hessian_stencil(params_vec, idx_non_fixed, epsilon)
    ll = total_likelihood(vecs, forest, root_carry=root_carry, raise_on_nan=False).reshape(-1, 4)
    n = len(idx_non_fixed)
    H = np.empty((n, n))
    for k, (h1, h2) in enumerate(hs):
        lij, li_j, l_ij, l_i_j = ll[k]
        H[k // n, k % n] = (lij - li_j - l_ij + l_i_j) / (4 * h1 * h2)
    return H


def num_hessian_grad(forest, params_vec, idx_non_fixed, epsilon):
    """Hessian of the log-likelihood over the parameters idx_non_fixed as central differences of the exact gradient
    (total_likelihood_grad): row i is (g(x + h_i e_i) - g(x - h_i e_i)) / (2 h_i) with num_hessian_ll's step
    h_i = max(|x_i| epsilon, 1e-12); all 2 n vectors in one call; the result is symmetrised.  The rounding noise of the
    log-likelihood is divided by h once, not by h^2 as in second differences."""
    x = np.asarray(params_vec, dtype=np.float64)
    idx = [int(i) for i in idx_non_fixed]
    n = len(idx)
    hs = np.array([max(abs(x[i]) * epsilon, 1e-12) for i in idx])
    vecs = np.repeat(x[None, :], 2 * n, axis=0)
    for k, i in enumerate(idx):
        vecs[2 * k, i] += hs[k]
        vecs[2 * k + 1, i] -= hs[k]
    _, g = total_likelihood_grad(vecs, forest, dirs=idx)
    H = (g[0::2] - g[1::2]) / (2.0 * hs[:, None])
    return 0.5 * (H + H.T)


def prediction_forward_backward(forest: Forest, params_vecs, forward=True, backward=True, combined=True):
    """prediction_forward, prediction_backward, combine_predictions (main.cpp:132-140).
    params_vecs: [n_seg][11].  Returns dict name -> (mean [n_ctp][4], cov [n_ctp][4][4])."""
    lib = _lib.load()
    p, _ = _as_params(params_vecs)
    M = forest.n_ctp
    bufs = {k: (np.empty((M, 20)) if want else None)
            for k, want in (("forward", forward), ("backward", backward), ("prediction", combined))}

    def ptr(a):
        return a.ctypes.data_as(_lib.c_double_p) if a is not None else None

    _lib.check(lib.ggp_predict(forest.handle, p.ctypes.data_as(_lib.c_double_p), p.shape[0],
                               ptr(bufs["forward"]), ptr(bufs["backward"]), ptr(bufs["prediction"])))
    return {k: (a[:, :4], a[:, 4:].reshape(M, 4, 4)) for k, a in bufs.items() if a is not None}


def prediction_upper14(forest: Forest, params_vecs, forward=True, backward=True, combined=True, out=None):
    """the same passes, outputs as [n_ctp][14] = 4 means + upper triangle (xx xg xl xq gg gl gq ll lq qq): the numbers
    write_predictions_to_file prints (predictions.h:575-578), packed on the device (ggp_predict14).  out: optional dict of
    preallocated (e.g. pinned) [n_ctp][14] float64 arrays to copy into."""
    lib = _lib.load()
    p, _ = _as_params(params_vecs)
    M = forest.n_ctp
    bufs = {k: ((out[k] if out and k in out else np.empty((M, 14))) if want else None)
            for k, want in (("forward", forward), ("backward", backward), ("prediction", combined))}

    def ptr(a):
        return a.ctypes.data_as(_lib.c_double_p) if a is not None else None

    _lib.check(lib.ggp_predict14(forest.handle, p.ctypes.data_as(_lib.c_double_p), p.shape[0],
                                 ptr(bufs["forward"]), ptr(bufs["backward"]), ptr(bufs["prediction"])))
    return {k: a for k, a in bufs.items() if a is not None}


def collect_joint_distributions(forest: Forest, params_vecs, tolerance_joint=1e-10, row_begin=0, row_end=None, cap=None, out=None):
    """collect_joint_distributions (correlation_tree.h:629-648) as a sparse list instead of the dense CSV.
    prediction_forward_backward must have been run on `forest` with the same params_vecs (the reference's -j
    implies -p, main.cpp:265-268).  Rows are the start points row_begin <= ctp < row_end.
    Returns (row_ctp, col_ctp, mean [n][8], cov_upper [n][36]), sorted by (row, col): the joint of
    z at `col` (first four means) and z at `row` (last four), tolerance as --rel_tolerance_joints.
    out: optional preallocated (row int64 [cap], col int64 [cap], rec float64 [cap][44]) arrays, e.g. pinned host memory (the
    copy into fresh pageable numpy arrays is bound by the host's first-touch page faults, not by the GPU)."""
    lib = _lib.load()
    p, _ = _as_params(params_vecs)
    if row_end is None:
        row_end = forest.n_ctp
    cnt = C.c_int64(0)
    args = (forest.handle, p.ctypes.data_as(_lib.c_double_p), p.shape[0], C.c_double(tolerance_joint), row_begin, row_end)
    if out is not None:
        row, col, rec = out
        cap = min(len(row), len(col), len(rec))
        if row.dtype != np.int64 or col.dtype != np.int64 or rec.dtype != np.float64 or rec.shape[1:] != (44,) or not rec.flags.c_contiguous:
            raise ValueError("out = (int64 [cap], int64 [cap], float64 [cap][44])")
    else:
        if cap is None:
            _lib.check(lib.ggp_joints(*args, 0, C.byref(cnt), None, None, None))
            cap = cnt.value
        row = np.empty(max(cap, 1), dtype=np.int64)
        col = np.empty(max(cap, 1), dtype=np.int64)
        rec = np.empty((max(cap, 1), 44))
    _lib.check(lib.ggp_joints(*args, cap, C.byref(cnt), row.ctypes.data_as(_lib.c_int64_p), col.ctypes.data_as(_lib.c_int64_p),
                              rec.ctypes.data_as(_lib.c_double_p)))
    n = min(cnt.value, cap)
    return row[:n], col[:n], rec[:n, :8], rec[:n, 8:]


def count_joints(forest: Forest, params_vecs, tolerance_joint=1e-10, row_begin=0, row_end=None):
    """number of joints the start points row_begin <= ctp < row_end emit (the walk without storing records)"""
    lib = _lib.load()
    p, _ = _as_params(params_vecs)
    cnt = C.c_int64(0)
    _lib.check(lib.ggp_joints(forest.handle, p.ctypes.data_as(_lib.c_double_p), p.shape[0], C.c_double(tolerance_joint), row_begin,
                              forest.n_ctp if row_end is None else row_end, 0, C.byref(cnt), None, None, None))
    return cnt.value


def correlation_sums(forest: Forest, params_vecs, dt_step, n_bins, tolerance_joint=1e-10, atol=None, normalize_time=False):
    """lag-binned moment sums of the correlation functions, accumulated on the device (ggp_correlation_sums): what
    python_src/correlation_from_joint.py accumulates from the joints and prediction files.  Returns (sums [n_bins][50] as
    numpy longdouble, number of emitted joints); prediction_forward_backward must have run with the same params_vecs."""
    lib = _lib.load()
    p, _ = _as_params(params_vecs)
    hi, lo = np.zeros((n_bins, 50)), np.zeros((n_bins, 50))
    nj = C.c_int64(0)
    _lib.check(lib.ggp_correlation_sums(forest.handle, p.ctypes.data_as(_lib.c_double_p), p.shape[0], C.c_double(tolerance_joint),
                                        C.c_double(dt_step), n_bins, C.c_double(0.2 * dt_step if atol is None else atol),
                                        1 if normalize_time else 0, hi.ctypes.data_as(_lib.c_double_p), lo.ctypes.data_as(_lib.c_double_p),
                                        C.byref(nj)))
    return hi.astype(np.longdouble) + lo.astype(np.longdouble), nj.value


def backward_cell_state(forest: Forest):
    """each cell's MOMAdata::mean/cov as the backward pass leaves them (sign-flipped frame)."""
    lib = _lib.load()
    out = np.empty((forest.n_cells, 20))
    _lib.check(lib.ggp_backward_cell_state(forest.handle, out.ctypes.data_as(_lib.c_double_p)))
    return out[:, :4], out[:, 4:].reshape(-1, 4, 4)


def math_eval(fn, x, y=None, device=0):
    """device self-test of the strict exp/log/pow/dawson (ggp_math_eval)."""
    lib = _lib.load()
    code = {"exp": 0, "log": 1, "pow": 2, "dawson": 3, "div": 4, "powexp": 5, "ll_finish": 6}[fn]
    x = np.ascontiguousarray(x, dtype=np.float64)
    if fn == "ll_finish":     # x [n][5]: quadratic form, S00, S01, S10, S11 -> out [n]
        n = x.shape[0]
        out = np.empty(n)
        _lib.check(lib.ggp_math_eval(device, code, n, x.ctypes.data_as(_lib.c_double_p), None, out.ctypes.data_as(_lib.c_double_p)))
        return out
    if fn == "powexp":        # x [n] bases, y [n] exp arguments -> out [n][5]: pow(x, 1.5 + i % 3), exp(y), exp(y/2), exp(-y), exp(y+1)
        y = np.ascontiguousarray(np.broadcast_to(y, x.shape), dtype=np.float64)
        out = np.empty((x.size, 5))
        _lib.check(lib.ggp_math_eval(device, code, x.size, x.ctypes.data_as(_lib.c_double_p), y.ctypes.data_as(_lib.c_double_p),
                                     out.ctypes.data_as(_lib.c_double_p)))
        return out
    out = np.empty_like(x)
    yp = None
    if y is not None:
        y = np.ascontiguousarray(np.broadcast_to(y, x.shape), dtype=np.float64)
        yp = y.ctypes.data_as(_lib.c_double_p)
    _lib.check(lib.ggp_math_eval(device, code, x.size, x.ctypes.data_as(_lib.c_double_p), yp, out.ctypes.data_as(_lib.c_double_p)))
    return out


def propagate_eval(state14, dt, p7, cross=False, device=0):
    """device mean_cov_model / cross_cov_model on n independent states (ggp_propagate_eval)."""
    lib = _lib.load()
    s = np.ascontiguousarray(state14, dtype=np.float64).reshape(-1, 14)
    n = s.shape[0]
    dt = np.ascontiguousarray(np.broadcast_to(dt, (n,)), dtype=np.float64)
    p7 = np.ascontiguousarray(np.broadcast_to(p7, (n, 7)), dtype=np.float64)
    out = np.empty((n, 14))
    cr = np.empty((n, 16)) if cross else None
    _lib.check(lib.ggp_propagate_eval(device, n, s.ctypes.data_as(_lib.c_double_p), dt.ctypes.data_as(_lib.c_double_p),
                                      p7.ctypes.data_as(_lib.c_double_p), out.ctypes.data_as(_lib.c_double_p),
                                      cr.ctypes.data_as(_lib.c_double_p) if cross else None))
    return (out, cr) if cross else out
