"""Host-side data model: the flattened lineage forest (the reference's std::vector<MOMAdata>,
moma_input.h:22-80) and the device handle built from it."""
import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _lib

NOISE_MODELS = {"const": 0, "scaled": 1}          # MOMAdata::noise_model (likelihood.h:59-64)
DIVISION_MODELS = {"gauss": 0, "binomial": 1}     # MOMAdata::cell_division_model (predictions.h:40-60)
PARAM_NAMES = ["mean_lambda", "gamma_lambda", "var_lambda", "mean_q", "gamma_q", "var_q", "beta",
               "var_x", "var_g", "var_dx", "var_dg"]   # Parameters.h:175


@dataclass
class LineageData:
    """Cells in input-file order; per-cell series concatenated (cell_offset).  parent/daughter indices as
    build_cell_genealogy leaves them (moma_input.h:125-151): daughter1 = first cell in file order whose
    parent is this cell, daughter2 = the second."""
    cell_offset: np.ndarray
    parent: np.ndarray
    time: np.ndarray
    log_length: np.ndarray
    fp: np.ndarray
    segment: np.ndarray = None
    daughter1: np.ndarray = None
    daughter2: np.ndarray = None
    noise_model: str = "scaled"        # code defaults, main.cpp:218-223
    division_model: str = "binomial"
    fp_auto: float = 0.0
    init_f: np.ndarray = None          # init_cells_f statistics (moma_input.h:675-704); None = derive
    init_r: np.ndarray = None          # init_cells_r statistics (moma_input.h:706-735)

    def __post_init__(self):
        self.cell_offset = np.ascontiguousarray(self.cell_offset, dtype=np.int64)
        self.parent = np.ascontiguousarray(self.parent, dtype=np.int32)
        self.time = np.ascontiguousarray(self.time, dtype=np.float64)
        self.log_length = np.ascontiguousarray(self.log_length, dtype=np.float64)
        self.fp = np.ascontiguousarray(self.fp, dtype=np.float64)
        if self.segment is None:
            self.segment = np.zeros(self.n_ctp, dtype=np.int32)
        self.segment = np.ascontiguousarray(self.segment, dtype=np.int32)
        if self.daughter1 is None or self.daughter2 is None:
            self.daughter1, self.daughter2 = build_daughters(self.parent)
        self.daughter1 = np.ascontiguousarray(self.daughter1, dtype=np.int32)
        self.daughter2 = np.ascontiguousarray(self.daughter2, dtype=np.int32)
        if self.noise_model not in NOISE_MODELS or self.division_model not in DIVISION_MODELS:
            raise ValueError("unknown noise or cell division model")

    @property
    def n_cells(self):
        return int(self.parent.shape[0])

    @property
    def n_ctp(self):
        return int(self.time.shape[0])

    def roots(self):
        """get_roots (moma_input.h:177-189): cells without parent, in file order."""
        return np.flatnonzero(self.parent < 0)

    def init_stats(self):
        """init_cells_f / init_cells_r (moma_input.h:663-735): mean and E[x^2]-E[x]^2 of the first / last
        point over all cells with more than one point, accumulated left to right like std::accumulate."""
        n = np.diff(self.cell_offset)
        sel = n > 1
        out = []
        for idx in (self.cell_offset[:-1][sel], self.cell_offset[1:][sel] - 1):
            x, g = self.log_length[idx], self.fp[idx]
            cnt = x.shape[0]
            # np.cumsum accumulates sequentially in float64, i.e. std::accumulate / std::inner_product order
            mx = (np.cumsum(x)[-1] if cnt else 0.0) / cnt
            mg = (np.cumsum(g)[-1] if cnt else 0.0) / cnt
            vx = np.cumsum(x * x)[-1] / cnt - mx * mx
            vg = np.cumsum(g * g)[-1] / cnt - mg * mg
            out.append(np.array([mx, mg, vx, vg]))
        return out[0], out[1]

    def subset(self, roots):
        """The trees hanging off the given roots (file order kept), for sharding across GPUs.  The init
        statistics of the WHOLE data set are frozen into the shard (they are population statistics)."""
        init_f, init_r = (self.init_f, self.init_r) if self.init_f is not None else self.init_stats()
        keep = np.zeros(self.n_cells, dtype=bool)
        stack = list(int(r) for r in roots)
        while stack:
            u = stack.pop()
            keep[u] = True
            for d in (self.daughter1[u], self.daughter2[u]):
                if d >= 0:
                    stack.append(int(d))
        cells = np.flatnonzero(keep)
        remap = -np.ones(self.n_cells, dtype=np.int64)
        remap[cells] = np.arange(cells.shape[0])
        n = np.diff(self.cell_offset)[cells]
        new_off = np.concatenate([[0], np.cumsum(n)])
        ctp = np.repeat(self.cell_offset[cells] - new_off[:-1], n) + np.arange(new_off[-1])

        def rm(a):
            a = a[cells]
            return np.where(a >= 0, remap[np.maximum(a, 0)], -1).astype(np.int32)

        return LineageData(cell_offset=new_off, parent=rm(self.parent), time=self.time[ctp], log_length=self.log_length[ctp],
                           fp=self.fp[ctp], segment=self.segment[ctp], daughter1=rm(self.daughter1), daughter2=rm(self.daughter2),
                           noise_model=self.noise_model, division_model=self.division_model, fp_auto=self.fp_auto,
                           init_f=np.array(init_f), init_r=np.array(init_r)), cells, ctp


def build_daughters(parent):
    """daughter1/daughter2 as build_cell_genealogy assigns them (moma_input.h:125-151)."""
    parent = np.asarray(parent)
    n = parent.shape[0]
    d1 = -np.ones(n, dtype=np.int32)
    d2 = -np.ones(n, dtype=np.int32)
    child = np.flatnonzero(parent >= 0)
    order = np.argsort(parent[child], kind="stable")
    child = child[order]
    par = parent[child]
    first = np.ones(child.shape[0], dtype=bool)
    first[1:] = par[1:] != par[:-1]
    second = np.zeros(child.shape[0], dtype=bool)
    second[1:] = first[:-1] & ~first[1:]
    d1[par[first]] = child[first]
    d2[par[second]] = child[second]
    return d1, d2


def _make_desc(data: LineageData, device: int = 0):
    d = _lib.ForestDesc()
    d.n_cells, d.n_ctp = data.n_cells, data.n_ctp
    d.cell_offset = data.cell_offset.ctypes.data_as(_lib.c_int64_p)
    d.parent = data.parent.ctypes.data_as(_lib.c_int32_p)
    d.daughter1 = data.daughter1.ctypes.data_as(_lib.c_int32_p)
    d.daughter2 = data.daughter2.ctypes.data_as(_lib.c_int32_p)
    d.time = data.time.ctypes.data_as(_lib.c_double_p)
    d.log_length = data.log_length.ctypes.data_as(_lib.c_double_p)
    d.fp = data.fp.ctypes.data_as(_lib.c_double_p)
    d.segment = data.segment.ctypes.data_as(_lib.c_int32_p)
    d.noise_model = NOISE_MODELS[data.noise_model]
    d.division_model = DIVISION_MODELS[data.division_model]
    d.fp_auto = data.fp_auto
    if data.init_f is not None and data.init_r is not None:
        d.init_f = (C.c_double * 4)(*[float(v) for v in data.init_f])
        d.init_r = (C.c_double * 4)(*[float(v) for v in data.init_r])
        d.compute_init = 0
    else:
        d.compute_init = 1
    d.device = device
    return d


class Forest:
    """Device-resident forest (ggp_forest handle)."""

    def __init__(self, data: LineageData, device: int = 0):
        self._lib = _lib.load()
        self.data = data
        d = _make_desc(data, device)
        h = C.c_void_p()
        _lib.check(self._lib.ggp_forest_create(C.byref(d), C.byref(h)))
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ggp_forest_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    @property
    def n_cells(self):
        return self._lib.ggp_forest_n_cells(self._h)

    @property
    def n_ctp(self):
        return self._lib.ggp_forest_n_ctp(self._h)

    @property
    def n_roots(self):
        return self._lib.ggp_forest_n_roots(self._h)

    @property
    def n_generations(self):
        return self._lib.ggp_forest_n_generations(self._h)

    def init_stats(self):
        f4 = np.zeros(4)
        r4 = np.zeros(4)
        _lib.check(self._lib.ggp_forest_get_init(self._h, f4.ctypes.data_as(_lib.c_double_p), r4.ctypes.data_as(_lib.c_double_p)))
        return f4, r4

    def set_mode(self, mode):
        """likelihood arithmetic: "strict" (bit-exact, default), "fast" (quadrature + FMA, gate 1e-10) or a node count"""
        code = {"strict": _lib.GGP_MODE_STRICT, "fast": _lib.GGP_MODE_FAST}.get(mode, mode)
        _lib.check(self._lib.ggp_forest_set_mode(self._h, int(code)))

    @property
    def mode(self):
        n = self._lib.ggp_forest_get_mode(self._h)
        return "strict" if n == 0 else ("fast" if n == 1 else f"fast{n}")

    @property
    def last_fast_nodes(self):
        """quadrature order the fast mode chose for the last ggp_loglik"""
        return self._lib.ggp_last_fast_nodes(self._h)

    @property
    def last_strict_reruns(self):
        return self._lib.ggp_last_strict_reruns(self._h)

    def set_stream(self, cuda_stream_ptr):
        _lib.check(self._lib.ggp_forest_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def upload_series(self, time_ptr, x_ptr, g_ptr, init_f=None, init_r=None):
        """Re-upload measurement arrays from host pointers (pinned memory gives async copies); a pointer of None / 0 leaves
        that array as it is.  init_f / init_r: the init_cells statistics of the new measurements (moma_input.h:675-735);
        None = re-derived by the library (forests created without explicit statistics only)."""
        fi = ri = None
        if init_f is not None:
            fi = (C.c_double * 4)(*[float(v) for v in init_f])
            ri = (C.c_double * 4)(*[float(v) for v in init_r])
        _lib.check(self._lib.ggp_forest_upload_series(self._h, C.c_void_p(time_ptr or None), C.c_void_p(x_ptr or None),
                                                      C.c_void_p(g_ptr or None), fi, ri))

    @property
    def last_kernel_ms(self):
        return self._lib.ggp_last_kernel_ms(self._h)

    @property
    def last_launch_count(self):
        return self._lib.ggp_last_launch_count(self._h)


class ForestGroup:
    """One data set sharded over several GPUs behind one handle (ggp_group): one host process drives them all."""

    def __init__(self, data: LineageData, devices):
        self._lib = _lib.load()
        self.data = data
        d = _make_desc(data, 0)
        dev = (C.c_int32 * len(devices))(*[int(v) for v in devices])
        h = C.c_void_p()
        _lib.check(self._lib.ggp_group_create(C.byref(d), dev, len(devices), C.byref(h)))
        self._h = h
        self.n_cells, self.n_ctp, self.n_roots = data.n_cells, data.n_ctp, len(data.roots())

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ggp_group_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    @property
    def size(self):
        return self._lib.ggp_group_size(self._h)

    @property
    def contiguous(self):
        return bool(self._lib.ggp_group_is_contiguous(self._h))

    def init_stats(self):
        """(init_f, init_r): the init_cells statistics of the whole data set the shards evaluate with (every shard holds the same)"""
        f4 = np.zeros(4)
        r4 = np.zeros(4)
        for k in range(self.size):
            h = self._lib.ggp_group_member(self._h, k)
            if h:
                _lib.check(self._lib.ggp_forest_get_init(h, f4.ctypes.data_as(_lib.c_double_p), r4.ctypes.data_as(_lib.c_double_p)))
                break
        return f4, r4

    def member_ctp(self, k):
        n = self._lib.ggp_group_member_ctp(self._h, k, None)
        a = np.empty(n, dtype=np.int64)
        self._lib.ggp_group_member_ctp(self._h, k, a.ctypes.data_as(_lib.c_int64_p))
        return a

    def set_mode(self, mode):
        code = {"strict": _lib.GGP_MODE_STRICT, "fast": _lib.GGP_MODE_FAST}.get(mode, mode)
        _lib.check(self._lib.ggp_group_set_mode(self._h, int(code)))

    def total_likelihood(self, params_vec, root_carry=None, per_cell=False):
        p = np.ascontiguousarray(params_vec, dtype=np.float64)
        single = p.ndim == 1
        p = p.reshape(-1, _lib.N_PARAMS)
        n_vec = p.shape[0]
        out = np.empty(n_vec)
        cell_ll = np.empty((n_vec, self.n_cells)) if per_cell else None
        nan = (_lib.NanInfo * n_vec)()
        rc = self._lib.ggp_group_loglik(self._h, p.ctypes.data_as(_lib.c_double_p), n_vec,
                                        root_carry.ctypes.data_as(_lib.c_double_p) if root_carry is not None else None,
                                        out.ctypes.data_as(_lib.c_double_p),
                                        cell_ll.ctypes.data_as(_lib.c_double_p) if per_cell else None, nan)
        _lib.check(rc, allow=(_lib.GGP_ERR_NAN,))
        self.nan = [(nan[v].cell, nan[v].t_index) for v in range(n_vec)]
        res = out[0] if single else out
        return (res, (cell_ll[0] if single else cell_ll)) if per_cell else res

    def predictions(self, params_vecs, packed=False, out=None):
        """forward / backward / combined for the whole data set in the caller's order; packed: 14 columns per time point"""
        p = np.ascontiguousarray(params_vecs, dtype=np.float64).reshape(-1, _lib.N_PARAMS)
        w = 14 if packed else 20
        bufs = out or {k: np.empty((self.n_ctp, w)) for k in ("forward", "backward", "prediction")}
        fn = self._lib.ggp_group_predict14 if packed else self._lib.ggp_group_predict
        _lib.check(fn(self._h, p.ctypes.data_as(_lib.c_double_p), p.shape[0], *[bufs[k].ctypes.data_as(_lib.c_double_p) if k in bufs else None
                                                                               for k in ("forward", "backward", "prediction")]))
        return bufs

    def joints(self, params_vecs, tolerance_joint=1e-10, row_begin=0, row_end=None):
        """collect_joint_distributions over the shards (ggp_group_joints): (row_ctp, col_ctp, mean [n][8], cov_upper [n][36]) in the
        caller's time-point indices, sorted by (row, col); predictions() must have run with the same params_vecs"""
        p = np.ascontiguousarray(params_vecs, dtype=np.float64).reshape(-1, _lib.N_PARAMS)
        row_end = self.n_ctp if row_end is None else row_end
        cnt = C.c_int64(0)
        args = (self._h, p.ctypes.data_as(_lib.c_double_p), p.shape[0], C.c_double(tolerance_joint), row_begin, row_end)
        _lib.check(self._lib.ggp_group_joints(*args, 0, C.byref(cnt), None, None, None))
        n = cnt.value
        row, col, rec = np.empty(max(n, 1), dtype=np.int64), np.empty(max(n, 1), dtype=np.int64), np.empty((max(n, 1), 44))
        _lib.check(self._lib.ggp_group_joints(*args, n, C.byref(cnt), row.ctypes.data_as(_lib.c_int64_p), col.ctypes.data_as(_lib.c_int64_p),
                                              rec.ctypes.data_as(_lib.c_double_p)))
        return row[:n], col[:n], rec[:n, :8], rec[:n, 8:]

    def correlation_sums(self, params_vecs, dt_step, n_bins, tolerance_joint=1e-10, atol=None, normalize_time=False):
        """lag-binned moment sums of the correlation functions over all shards (ggp_group_correlation_sums)"""
        p = np.ascontiguousarray(params_vecs, dtype=np.float64).reshape(-1, _lib.N_PARAMS)
        hi, lo = np.zeros((n_bins, 50)), np.zeros((n_bins, 50))
        nj = C.c_int64(0)
        _lib.check(self._lib.ggp_group_correlation_sums(self._h, p.ctypes.data_as(_lib.c_double_p), p.shape[0], C.c_double(tolerance_joint),
                                                        C.c_double(dt_step), n_bins, C.c_double(0.2 * dt_step if atol is None else atol),
                                                        1 if normalize_time else 0, hi.ctypes.data_as(_lib.c_double_p),
                                                        lo.ctypes.data_as(_lib.c_double_p), C.byref(nj)))
        return hi.astype(np.longdouble) + lo.astype(np.longdouble), nj.value
