"""ctypes bindings of the C ABI in include/phmrf.h and include/phmrf_gco.h.

There is no CPU fallback: when ``lib/libphmrf.so`` is missing, importing the bindings
raises, and when no CUDA device is present every compute entry point returns
``PHMRF_E_CUDA`` which surfaces as :class:`PhmrfError`.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "lib", "libphmrf.so")
GCO_LIB_PATH = os.path.join(_PKG, "lib", "libphmrf_gco.so")
PROBE_LIB_PATH = os.path.join(_PKG, "lib", "libphmrf_probe.so")

PHMRF_OK, PHMRF_E_INVALID, PHMRF_E_CUDA, PHMRF_E_NOT_SPD, PHMRF_E_STATE, PHMRF_E_UNSUPPORTED = 0, -1, -2, -3, -4, -5


class PhmrfError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libphmrf error %d: %s" % (code, msg))
        self.code = code


_c_double_p = C.POINTER(C.c_double)
_c_int32_p = C.POINTER(C.c_int32)
_c_int64_p = C.POINTER(C.c_int64)
_vp = C.c_void_p

# name -> (restype, argtypes); kept in step with include/phmrf.h (tests/test_abi.py checks it)
SIGNATURES = {
    "phmrf_abi_version": (C.c_int, []),
    "phmrf_last_error": (C.c_char_p, []),
    "phmrf_host_alloc": (C.c_int, [C.c_int64, C.POINTER(_vp)]),
    "phmrf_host_free": (C.c_int, [_vp]),
    "phmrf_ctx_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    "phmrf_ctx_destroy": (C.c_int, [_vp]),
    "phmrf_set_model": (C.c_int, [_vp, _c_double_p, _c_double_p, _c_double_p]),
    "phmrf_set_quantiser": (C.c_int, [_vp, C.c_double, C.c_double, C.c_double]),
    "phmrf_get_quantiser": (C.c_int, [_vp, _c_double_p, _c_double_p, _c_double_p]),
    "phmrf_region_create": (C.c_int, [_vp, _c_double_p, C.c_int64, C.c_int64, C.c_int64, _c_int64_p, _c_double_p,
                                      C.c_int64, _vp, C.POINTER(_vp)]),
    "phmrf_region_update_X": (C.c_int, [_vp, _c_double_p]),
    "phmrf_region_destroy": (C.c_int, [_vp]),
    "phmrf_region_sync": (C.c_int, [_vp]),
    "phmrf_region_device_bytes": (C.c_int64, [_vp]),
    "phmrf_emit_loglik": (C.c_int, [_vp, _c_double_p]),
    "phmrf_get_logprob": (C.c_int, [_vp, _c_double_p]),
    "phmrf_set_logprob": (C.c_int, [_vp, _c_double_p]),
    "phmrf_pairwise_potential": (C.c_int, [_vp, C.c_int, _c_double_p]),
    "phmrf_quantise": (C.c_int, [_vp, C.c_double, C.c_double, _c_int32_p, _c_int32_p, _c_int32_p, _c_double_p,
                                 _c_int64_p, C.c_int64, _c_int64_p]),
    "phmrf_set_labels": (C.c_int, [_vp, _c_int32_p]),
    "phmrf_labels_argmin_unary": (C.c_int, [_vp, _c_int32_p]),
    "phmrf_estep_stats": (C.c_int, [_vp, C.c_int, _c_double_p, _c_double_p, _c_double_p]),
    "phmrf_stats_device_ptr": (_vp, [_vp]),
    "phmrf_stats_len": (C.c_int64, [_vp]),
    "phmrf_absmax_device_ptr": (_vp, [_vp]),
    "phmrf_region_set_weight_max": (C.c_int, [_vp, C.c_double]),
    "phmrf_region_weight_max": (C.c_double, [_vp]),
    "phmrf_emit_loglik_async": (C.c_int, [_vp]),
    "phmrf_quantise_async": (C.c_int, [_vp, C.c_double, C.c_double]),
    "phmrf_estep_stats_async": (C.c_int, [_vp, C.c_int]),
    "phmrf_launch_count": (C.c_int64, []),
    "phmrf_region_create_grid": (C.c_int, [_vp, _c_double_p, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                                           C.c_double, _vp, C.POINTER(_vp)]),
    "phmrf_region_n_edges": (C.c_int64, [_vp]),
    "phmrf_region_n_own": (C.c_int64, [_vp]),
    "phmrf_region_n_window": (C.c_int64, [_vp]),
    "phmrf_region_own_offset": (C.c_int64, [_vp]),
    "phmrf_region_edges": (C.c_int, [_vp, _c_int64_p, _c_double_p]),
    "phmrf_region_set_edge_weights": (C.c_int, [_vp, _c_double_p, C.c_int64]),
    "phmrf_graph_cut_swap": (C.c_int, [C.c_int, C.c_int64, C.c_int32, _c_int32_p, _c_int64_p, _c_int32_p, C.c_int64,
                                       _c_int32_p, _c_int32_p, C.c_int32, _c_int32_p, C.POINTER(C.c_longlong),
                                       C.POINTER(C.c_longlong)]),
    "phmrf_region_graph_cut": (C.c_int, [_vp, _c_int32_p, C.c_int32, _c_int32_p, C.POINTER(C.c_longlong),
                                         C.POINTER(C.c_longlong)]),
    "phmrf_grid_edge_count":(C.c_int64, [C.c_int, C.c_int64, C.c_int64, C.c_int]),
    "phmrf_grid_edges": (C.c_int, [C.c_int, _c_double_p, C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_int, _c_double_p,
                                   C.c_int64]),
    "phmrf_prep_normalise": (C.c_int, [C.c_int, _c_double_p, C.c_int64, C.c_int, _c_double_p, _c_double_p, _c_double_p,
                                       C.c_int]),
    "phmrf_prep_region_image": (C.c_int, [C.c_int, _c_double_p, _c_int64_p, C.c_int64, C.c_int, C.c_int, C.c_int64,
                                          C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_double,
                                          C.c_double, _c_double_p, _c_double_p]),
}

# measurement tool (lib/libphmrf_probe.so, include/phmrf_probe.h): not part of the product library
PROBE_SIGNATURES = {
    "phmrf_probe_fp64_tflops": (C.c_int, [C.c_int, _c_double_p]),
    "phmrf_probe": (C.c_int, [C.c_int, C.c_int, _c_double_p]),
    "phmrf_probe_last_error": (C.c_char_p, []),
}

GCO_SIGNATURES = {
    "phmrf_gco_cut_general_graph": (C.c_int, [C.c_int64, C.c_int32, _c_int32_p, _c_int64_p, _c_int32_p, C.c_int64,
                                              _c_int32_p, _c_int32_p, C.c_int32, C.c_int32, _c_int32_p,
                                              C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]),
    "phmrf_gco_last_error": (C.c_char_p, []),
}

_lib = None
_gco = None
_probe = None


def _bind(path, sigs, what):
    if not os.path.exists(path):
        raise ImportError("%s not built: %s is missing (run `python -m phylo_hmrf_b200.build`); "
                          "there is no CPU fallback" % (what, path))
    lib = C.CDLL(path)
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    return lib


def lib():
    global _lib
    if _lib is None:
        _lib = _bind(LIB_PATH, SIGNATURES, "CUDA extension")
    return _lib


def probe_lib():
    global _probe
    if _probe is None:
        _probe = _bind(PROBE_LIB_PATH, PROBE_SIGNATURES, "pipe probes")
    return _probe


def gco():
    global _gco
    if _gco is None:
        _gco = _bind(GCO_LIB_PATH, GCO_SIGNATURES, "GCO graph-cut wrapper")
    return _gco


def check(rc):
    if rc != 0:
        raise PhmrfError(rc, lib().phmrf_last_error().decode("utf-8", "replace"))


def dptr(a):
    return None if a is None else a.ctypes.data_as(_c_double_p)


def i32ptr(a):
    return None if a is None else a.ctypes.data_as(_c_int32_p)


def i64ptr(a):
    return None if a is None else a.ctypes.data_as(_c_int64_p)


def as_f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)
