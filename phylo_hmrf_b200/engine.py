"""Thin object layer over the C ABI (include/phmrf.h): a :class:`Model` (K states, d leaf
species, one device) and its :class:`Region` handles (one synteny region or one row band).

Also the two third-party callables the reference's hot path goes through, re-hosted on
the library with their original signatures:

* :func:`log_multivariate_normal_density`  (sklearn 0.18; phylo_hmrf.py:266-268)
* :func:`cut_general_graph`                (pygco; phylo_hmrf.py:496-498)
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import PhmrfError, as_f64, check, dptr, i32ptr, i64ptr

def pinned_empty(shape, dtype):
    """NumPy array in page-locked host memory (phmrf_host_alloc): copies to and from it run at
    the PCIe rate and overlap with kernels and with copies in the other direction.  The memory
    is released when the array (and every view of it) is garbage collected."""
    import weakref
    dtype = np.dtype(dtype)
    count = int(np.prod(shape, dtype=np.int64))
    nbytes = max(1, count * dtype.itemsize)
    p = C.c_void_p()
    check(_lib.lib().phmrf_host_alloc(nbytes, C.byref(p)))
    buf = (C.c_byte * nbytes).from_address(p.value)
    weakref.finalize(buf, _lib.lib().phmrf_host_free, C.c_void_p(p.value))
    return np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)


class Model:
    """Device-side model state: means_ [K,d], _covars_ [K,d,d], edge_potential [K,K]."""

    def __init__(self, n_states, n_features, device=0):
        self.K, self.d, self.device = int(n_states), int(n_features), int(device)
        h = C.c_void_p()
        check(_lib.lib().phmrf_ctx_create(self.device, self.K, self.d, C.byref(h)))
        self._h = h
        self.stats_len = int(_lib.lib().phmrf_stats_len(h))

    def set_model(self, means, covars, V):
        means, covars, V = as_f64(means), as_f64(covars), as_f64(V)
        if means.shape != (self.K, self.d) or covars.shape != (self.K, self.d, self.d) or V.shape != (self.K, self.K):
            raise ValueError("model arrays must be means[K,d], covars[K,d,d], V[K,K]")
        rc = _lib.lib().phmrf_set_model(self._h, dptr(means), dptr(covars), dptr(V))
        if rc == _lib.PHMRF_E_NOT_SPD:
            raise ValueError("'covars' must be symmetric, positive-definite")
        check(rc)

    def set_quantiser(self, unary_precision=100000, pairwise_precision=1000, smooth_precision=100):
        """Scale factors of pygco's float->int conversion (see phmrf_set_quantiser); the defaults
        are pygco's _UNARY_FLOAT_PRECISION / _PAIRWISE_FLOAT_PRECISION / _SMOOTH_COST_PRECISION."""
        check(_lib.lib().phmrf_set_quantiser(self._h, float(unary_precision), float(pairwise_precision),
                                             float(smooth_precision)))

    def quantiser(self):
        u, w, v = C.c_double(), C.c_double(), C.c_double()
        check(_lib.lib().phmrf_get_quantiser(self._h, C.byref(u), C.byref(w), C.byref(v)))
        return u.value, w.value, v.value

    def region(self, X, edge_ids, edge_w, n_window=None, own_offset=0, stream=None):
        return Region(self, X, edge_ids, edge_w, n_window, own_offset, stream)

    def region_grid(self, X_window, kind, n1, n2, row0=0, row1=None, num_neighbor=8, beta1=0.5, stream=None):
        """Region (or row band [row0,row1)) built on the device from the grid geometry; see
        phmrf_region_create_grid.  kind: 1 diagonal region (n1 == n2 bins), 0 rectangle."""
        return GridRegion(self, X_window, kind, n1, n2, row0, row1, num_neighbor, beta1, stream)

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().phmrf_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Region:
    """One region (or row band) resident on the device; see phmrf_region_create."""
    has_logp = False     # a log-likelihood is on the device (emitted or uploaded)

    def __init__(self, model, X, edge_ids, edge_w, n_window=None, own_offset=0, stream=None):
        X = as_f64(X)
        if X.ndim != 2 or X.shape[1] != model.d:
            raise ValueError("X must be [n, %d]" % model.d)
        e = np.ascontiguousarray(edge_ids, dtype=np.int64).reshape(-1, 2)
        w = as_f64(edge_w).reshape(-1)
        if len(e) != len(w):
            raise ValueError("edge_ids and edge_w disagree in length")
        self.model = model
        self.n = int(X.shape[0])
        self.n_window = self.n if n_window is None else int(n_window)
        self.own_offset = int(own_offset)
        self.n_edges = len(e)
        h = C.c_void_p()
        check(_lib.lib().phmrf_region_create(model._h, dptr(X), self.n, self.n_window, self.own_offset, i64ptr(e),
                                             dptr(w), len(e), C.c_void_p(stream) if stream else None, C.byref(h)))
        self._h = h

    def update_X(self, X):
        X = as_f64(X)
        if X.shape != (self.n, self.model.d):
            raise ValueError("X must be [%d, %d]" % (self.n, self.model.d))
        self._x_keepalive = X
        check(_lib.lib().phmrf_region_update_X(self._h, dptr(X)))

    # ---- phase A
    def emit_loglik(self, want_absmax=False):
        if want_absmax:
            v = C.c_double()
            check(_lib.lib().phmrf_emit_loglik(self._h, C.byref(v)))
            self.has_logp = True
            return v.value
        check(_lib.lib().phmrf_emit_loglik(self._h, None))
        self.has_logp = True
        return None

    def logprob(self):
        out = np.empty((self.n, self.model.K), dtype=np.float64)
        check(_lib.lib().phmrf_get_logprob(self._h, dptr(out)))
        return out

    def set_logprob(self, logprob):
        lp = as_f64(logprob)
        if lp.shape != (self.n, self.model.K):
            raise ValueError("logprob must be [%d, %d]" % (self.n, self.model.K))
        check(_lib.lib().phmrf_set_logprob(self._h, dptr(lp)))
        self.has_logp = True

    def pairwise_potential(self, estimate_type):
        out = np.empty((self.n, self.model.K), dtype=np.float64)
        check(_lib.lib().phmrf_pairwise_potential(self._h, int(estimate_type), dptr(out)))
        return out

    def quantise(self, dwf=0.0, tol=1e-9, want_unary=True, want_edges=True, boundary_cap=1 << 16, staged=False):
        """-> dict(unary_i32, w_i32, V_i32, dwf, boundary_idx, n_boundary)

        staged=True returns the integer arrays as views of the region's own page-locked staging
        buffers (allocated once, overwritten by the next staged call on this region): the
        per-iteration product path, where the arrays go straight into the graph cut."""
        K = self.model.K
        if staged:
            if getattr(self, "_pin_unary", None) is None:
                self._pin_unary = pinned_empty((self.n, K), np.int32)
                self._pin_w = pinned_empty((self.n_edges,), np.int32)
            u = self._pin_unary if want_unary else None
            wi = self._pin_w if want_edges else None
        else:
            u = np.empty((self.n, K), dtype=np.int32) if want_unary else None
            wi = np.empty(self.n_edges, dtype=np.int32) if want_edges else None
        Vi = np.empty((K, K), dtype=np.int32)
        d = C.c_double()
        nb = C.c_int64()
        bl = np.empty(max(1, boundary_cap), dtype=np.int64)
        check(_lib.lib().phmrf_quantise(self._h, float(dwf), float(tol), i32ptr(u), i32ptr(wi), i32ptr(Vi), C.byref(d),
                                        i64ptr(bl), int(boundary_cap), C.byref(nb)))
        m = min(int(nb.value), boundary_cap)
        return dict(unary_i32=u, w_i32=wi, V_i32=Vi, dwf=d.value, boundary_idx=bl[:m].copy(), n_boundary=int(nb.value))

    def label_staging(self):
        """Page-locked int32 buffer covering the label window: the graph cut writes its result here
        (gco_cut_int(..., out=...)) and set_labels() uploads it without a pageable detour."""
        if getattr(self, "_pin_labels", None) is None:
            self._pin_labels = pinned_empty((self.n_window,), np.int32)
        return self._pin_labels

    # ---- phase B
    def set_labels(self, labels_window):
        lab = np.ascontiguousarray(labels_window, dtype=np.int32)
        if lab.shape != (self.n_window,):
            raise ValueError("labels must cover the %d-node window" % self.n_window)
        rc = _lib.lib().phmrf_set_labels(self._h, i32ptr(lab))
        if rc == _lib.PHMRF_E_INVALID:
            raise ValueError(_lib.lib().phmrf_last_error().decode())
        check(rc)

    def labels_argmin_unary(self):
        out = np.empty(self.n, dtype=np.int32)
        check(_lib.lib().phmrf_labels_argmin_unary(self._h, i32ptr(out)))
        return out

    def graph_cut(self, init_labels=None, n_iter=5000, return_energy=False):
        """Alpha-beta swap on the region's own integer arrays from the last quantise() (phmrf_region_graph_cut):
        the labels of gco_cut_int(..., algorithm='swap') on those arrays, without downloading them.  The labels
        stay on the device for estep_stats(); they are also returned (with the energy after and before the cut
        when return_energy).  Whole regions only."""
        init = None
        if init_labels is not None:
            init = np.ascontiguousarray(init_labels, dtype=np.int32)
            if init.shape != (self.n,):
                raise ValueError("init_labels must hold %d labels" % self.n)
        out = np.empty(self.n, dtype=np.int32)
        en, en0 = C.c_longlong(), C.c_longlong()
        check(_lib.lib().phmrf_region_graph_cut(self._h, i32ptr(init), int(n_iter), i32ptr(out), C.byref(en),
                                                C.byref(en0)))
        return (out, en.value, en0.value) if return_energy else out

    def estep_stats(self, estimate_type, want_post=False):
        """-> (stats dict like phylo_hmrf.py:311-314, cost_sums[3], posteriors or None)"""
        K, d = self.model.K, self.model.d
        flat = np.empty(K * (1 + d + d * d), dtype=np.float64)
        sums = np.empty(3, dtype=np.float64)
        post = np.empty((self.n, K), dtype=np.float64) if want_post else None
        check(_lib.lib().phmrf_estep_stats(self._h, int(estimate_type), dptr(post), dptr(flat), dptr(sums)))
        return unpack_stats(flat, K, d), sums, post

    # ---- enqueue-only (bench)
    def emit_loglik_async(self):
        check(_lib.lib().phmrf_emit_loglik_async(self._h))
        self.has_logp = True

    def quantise_async(self, dwf=0.0, tol=1e-9):
        check(_lib.lib().phmrf_quantise_async(self._h, float(dwf), float(tol)))

    def estep_stats_async(self, estimate_type):
        check(_lib.lib().phmrf_estep_stats_async(self._h, int(estimate_type)))

    def sync(self):
        check(_lib.lib().phmrf_region_sync(self._h))

    def absmax_device_ptr(self):
        return int(_lib.lib().phmrf_absmax_device_ptr(self._h))

    def weight_max(self):
        return float(_lib.lib().phmrf_region_weight_max(self._h))

    def set_weight_max(self, wmax):
        check(_lib.lib().phmrf_region_set_weight_max(self._h, float(wmax)))

    def stats_device_ptr(self):
        return int(_lib.lib().phmrf_stats_device_ptr(self._h))

    def device_bytes(self):
        return int(_lib.lib().phmrf_region_device_bytes(self._h))

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().phmrf_region_destroy(self._h)
            self._h = None
        self._pin_unary = self._pin_w = self._pin_labels = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GridRegion(Region):
    """A region whose graph was built by kernels from the grid geometry (SURVEY 8 f-1)."""

    def __init__(self, model, X_window, kind, n1, n2, row0, row1, num_neighbor, beta1, stream=None):
        X = as_f64(X_window)
        rows = n2 if kind == 1 else n1
        row1 = rows if row1 is None else row1

        def start(row):  # first node of a row in the region's node order
            return row * n2 if kind == 0 else row * n2 - (row * (row - 1)) // 2

        expect = start(min(row1 + 1, rows)) - start(max(row0 - 1, 0))
        if X.ndim != 2 or X.shape != (expect, model.d):
            raise ValueError("X_window must be [%d, %d]: rows [row0-1, row1+1) of the region" % (expect, model.d))
        self.model = model
        h = C.c_void_p()
        check(_lib.lib().phmrf_region_create_grid(model._h, dptr(X), int(kind), int(n1), int(n2), int(row0), int(row1),
                                                  int(num_neighbor), float(beta1), C.c_void_p(stream) if stream else None,
                                                  C.byref(h)))
        self._h = h
        L = _lib.lib()
        self.n = int(L.phmrf_region_n_own(h))
        self.n_window = int(L.phmrf_region_n_window(h))
        self.own_offset = int(L.phmrf_region_own_offset(h))
        self.n_edges = int(L.phmrf_region_n_edges(h))

    def set_edge_weights(self, edge_w):
        """Use the caller's host edge weights (same order as edges()) for the integer conversion; see
        phmrf_region_set_edge_weights."""
        w = as_f64(edge_w).reshape(-1)
        check(_lib.lib().phmrf_region_set_edge_weights(self._h, dptr(w), len(w)))

    def edges(self):
        """-> (edge_ids [E,2] int64 window-local, edge_w [E]) for the host graph cut."""
        ids = np.empty((self.n_edges, 2), dtype=np.int64)
        w = np.empty(self.n_edges, dtype=np.float64)
        check(_lib.lib().phmrf_region_edges(self._h, i64ptr(ids), dptr(w)))
        return ids, w


def unpack_stats(flat, K, d):
    """post[K] | obs[K,d] | obs*obs.T[K,d,d]  ->  the reference's stats dict keys."""
    return {
        'post': flat[:K].copy(),
        'obs': flat[K:K + K * d].reshape(K, d).copy(),
        'obs*obs.T': flat[K + K * d:K + K * d + K * d * d].reshape(K, d, d).copy(),
    }


def costs_from_sums(sums, n):
    """The four scalars of _compute_cost_v1 (phylo_hmrf.py:374-396) from the device sums."""
    pairwise_cost = sums[0] * 1.0 / n
    pairwise_cost_normalize = -sums[1] * 1.0 / n
    unary_cost = -sums[2] * 1.0 / n
    return pairwise_cost, pairwise_cost_normalize, unary_cost, unary_cost + pairwise_cost_normalize


# -------------------------------------------------------------------------------------
# Re-hosted third-party callables
# -------------------------------------------------------------------------------------
def log_multivariate_normal_density(X, means, covars, covariance_type='full', device=0):
    """sklearn 0.18 signature (phylo_hmrf.py:266-268); only 'full' is on the hot path
    (phylo_hmrf.py:57: the constructor default, never overridden by run())."""
    if covariance_type != 'full':
        raise ValueError("only covariance_type='full' is implemented on the device path")
    X = as_f64(X)
    means = as_f64(means)
    K, d = means.shape
    m = Model(K, d, device)
    try:
        m.set_model(means, covars, np.zeros((K, K)))
        r = m.region(X, np.zeros((0, 2), dtype=np.int64), np.zeros(0))
        try:
            r.emit_loglik()
            return r.logprob()
        finally:
            r.close()
    finally:
        m.close()


def gco_cut_int(unary_i32, edge_ids, w_i32, V_i32, n_iter=-1, algorithm='expansion', init_labels=None,
                return_energy=False, out=None):
    """Host graph cut on already quantised arrays (include/phmrf_gco.h).  `out`: int32 [n] buffer
    the labels are written to (e.g. Region.label_staging())."""
    u = np.ascontiguousarray(unary_i32, dtype=np.int32)
    n, K = u.shape
    e = np.ascontiguousarray(edge_ids, dtype=np.int64).reshape(-1, 2)
    w = np.ascontiguousarray(w_i32, dtype=np.int32)
    V = np.ascontiguousarray(V_i32, dtype=np.int32)
    init = None if init_labels is None else np.ascontiguousarray(init_labels, dtype=np.int32)
    if out is None:
        out = np.empty(n, dtype=np.int32)
    elif out.dtype != np.int32 or out.shape != (n,) or not out.flags.c_contiguous:
        raise ValueError("out must be a contiguous int32 array of %d labels" % n)
    en, en0 = C.c_longlong(), C.c_longlong()
    alg = {'swap': 0, 'expansion': 1}[algorithm]
    g = _lib.gco()
    rc = g.phmrf_gco_cut_general_graph(n, K, i32ptr(u), i64ptr(e), i32ptr(w), len(e), i32ptr(V), i32ptr(init),
                                       int(n_iter), alg, i32ptr(out), C.byref(en), C.byref(en0))
    if rc != 0:
        raise RuntimeError(g.phmrf_gco_last_error().decode("utf-8", "replace"))
    return (out, en.value, en0.value) if return_energy else out


def swap_supported(V_i32, w_min):
    """True when the device swap runs these costs: no negative edge weight and V[a][b] + V[b][a] >=
    V[a][a] + V[b][b] for every pair of labels, so that every swap move is submodular.  The host cut also runs
    the other cases (with negative capacities)."""
    V = np.asarray(V_i32, dtype=np.int64)
    d = np.diag(V)
    return bool(w_min >= 0 and np.all(V + V.T >= d[:, None] + d[None, :]))


def gco_swap_device(unary_i32, edge_ids, w_i32, V_i32, n_iter=-1, init_labels=None, return_energy=False, device=0):
    """gco_cut_int(..., algorithm='swap') on the GPU (phmrf_graph_cut_swap): the same labels and energies.
    Costs swap_supported() refuses raise PhmrfError with code PHMRF_E_UNSUPPORTED."""
    u = np.ascontiguousarray(unary_i32, dtype=np.int32)
    n, K = u.shape
    e = np.ascontiguousarray(edge_ids, dtype=np.int64).reshape(-1, 2)
    w = np.ascontiguousarray(w_i32, dtype=np.int32)
    V = np.ascontiguousarray(V_i32, dtype=np.int32)
    if len(w) != len(e) or V.shape != (K, K):
        raise ValueError("need w_i32 [%d] and V_i32 [%d, %d]" % (len(e), K, K))
    init = None if init_labels is None else np.ascontiguousarray(init_labels, dtype=np.int32)
    if init is not None and init.shape != (n,):
        raise ValueError("init_labels must hold %d labels" % n)
    out = np.empty(n, dtype=np.int32)
    en, en0 = C.c_longlong(), C.c_longlong()
    check(_lib.lib().phmrf_graph_cut_swap(int(device), n, K, i32ptr(u), i64ptr(e), i32ptr(w), len(e), i32ptr(V),
                                          i32ptr(init), int(n_iter), i32ptr(out), C.byref(en), C.byref(en0)))
    return (out, en.value, en0.value) if return_energy else out


def cut_general_graph(edges, edge_weights, unary_cost, pairwise_cost, n_iter=-1, algorithm='expansion',
                      init_labels=None, down_weight_factor=None):
    """pygco.cut_general_graph signature (call site phylo_hmrf.py:496-498), integer-cost
    form: pygco passes integer arrays to GCO untouched, and so does this.  Float costs are
    NOT converted on the host -- the float->int conversion of the hot path runs on the GPU
    (Region.quantise / phmrf_quantise) and its output is what this function consumes."""
    for name, arr in (("unary_cost", unary_cost), ("edge_weights", edge_weights), ("pairwise_cost", pairwise_cost)):
        if not np.issubdtype(np.asarray(arr).dtype, np.integer):
            raise TypeError("%s must be an integer array: quantise float costs on the device with "
                            "Region.quantise() (there is no host conversion path)" % name)
    if down_weight_factor is not None:
        raise ValueError("down_weight_factor applies to float costs only")
    return gco_cut_int(unary_cost, edges, edge_weights, pairwise_cost, n_iter, algorithm, init_labels)


def probe(which, device=0):
    """Pipe probes (lib/libphmrf_probe.so, include/phmrf_probe.h): measured roofline denominators for bench.py."""
    v = C.c_double()
    L = _lib.probe_lib()
    rc = L.phmrf_probe(int(device), int(which), C.byref(v))
    if rc != 0:
        raise PhmrfError(rc, L.phmrf_probe_last_error().decode("utf-8", "replace"))
    return v.value


def launch_count():
    return int(_lib.lib().phmrf_launch_count())
