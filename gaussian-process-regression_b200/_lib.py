"""ctypes binding of libgprc (include/gprc.h).  The library is the product; there is no CPU fallback: if the shared
object is missing or no CUDA device is present every entry point raises."""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgprc.so")

c_double_p = C.POINTER(C.c_double)
c_long_p = C.POINTER(C.c_long)
c_int_p = C.POINTER(C.c_int)

(CONSTANT, LINEAR, POLYNOMIAL, SQREXP, GAMMAEXP, RATQUAD, PRECOMPUTED) = range(7)
KERNEL_IDS = dict(constant=CONSTANT, linear=LINEAR, polynomial=POLYNOMIAL, sqrexp=SQREXP, gammaexp=GAMMAEXP,
                  rationalquadratic=RATQUAD)
GET_L, GET_ALPHA, GET_LINV, GET_FHAT, GET_SQRTW = range(5)
GRAD_AS_CODED, GRAD_TEXTBOOK = 0, 1
OPT_GRAM_DMMA = 1
OPT_PREDICT_PATH = 2
OPT_OZAKI_DIGITS = 3
OPT_INT8_AUTO = 4
OPT_INT8_TILE = 5
INT8_TILE_DEFAULT = 2  # kernel variant of the INT8 pass the library starts with (csrc/common.cuh: opt_int8_tile)
OPT_INT8_TEST_SHRINK = 6
OPT_TRSV = 7
OPT_CHOL_TILES = 8
CHOL_TILES_DEFAULT = 128  # csrc/common.cuh: opt_chol_tiles
TRSV_DEFAULT = 1  # csrc/common.cuh: opt_trsv
T_NAMES = ["build_k", "chol", "solve", "trtri", "build_ks", "var", "newton", "predict"]


class GprcKernel(C.Structure):
    _fields_ = [("id", C.c_int), ("c", C.c_double), ("sigma", C.c_double), ("p", C.c_double), ("l", C.c_double),
                ("gamma", C.c_double), ("alpha", C.c_double), ("sigma_vec", c_double_p), ("sigma_len", C.c_int)]


class GprcError(RuntimeError):
    pass


# every symbol include/gprc.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_K = C.POINTER(GprcKernel)
# gprc_objective_fn / gprc_gradient_fn: int (*)(const double* par, int npar, void* user, double* out)
OBJECTIVE_FN = C.CFUNCTYPE(C.c_int, c_double_p, C.c_int, C.c_void_p, c_double_p)
SIGNATURES = {
    "gprc_ctx_create": (C.c_int, [C.POINTER(_P), C.c_int]),
    "gprc_ctx_free": (None, [_P]),
    "gprc_ctx_set_option": (C.c_int, [_P, C.c_int, C.c_int]),
    "gprc_ctx_sync": (C.c_int, [_P]),
    "gprc_ctx_set_interrupt": (C.c_int, [_P, C.CFUNCTYPE(C.c_int, C.c_void_p), _P]),
    "gprc_ctx_reset_timers": (None, [_P]),
    "gprc_ctx_get_timers": (C.c_int, [_P, c_double_p, c_long_p]),
    "gprc_ctx_trim": (C.c_int, [_P, C.POINTER(C.c_ulonglong)]),
    "gprc_ctx_last_predict_path": (C.c_int, [_P]),
    "gprc_ctx_last_predict_chunks": (C.c_long, [_P]),
    "gprc_ctx_mark": (C.c_int, [_P, C.c_int]),
    "gprc_ctx_elapsed_ms": (C.c_int, [_P, C.c_int, C.c_int, c_double_p]),
    "gprc_last_error": (C.c_char_p, []),
    "gprc_version": (C.c_int, []),
    "gprc_dev_malloc": (C.c_int, [_P, C.POINTER(_P), C.c_ulonglong]),
    "gprc_dev_free": (C.c_int, [_P, _P]),
    "gprc_dev_h2d": (C.c_int, [_P, _P, _P, C.c_ulonglong]),
    "gprc_dev_d2h": (C.c_int, [_P, _P, _P, C.c_ulonglong]),
    "gprc_host_register": (C.c_int, [_P, C.c_ulonglong]),
    "gprc_host_unregister": (C.c_int, [_P]),
    "gprc_cov_matrix": (C.c_int, [_P, _K, c_double_p, C.c_int, C.c_long, c_double_p, C.c_long, c_double_p]),
    "gprc_cov_pointwise": (C.c_int, [_P, _K, c_double_p, c_double_p, C.c_int, C.c_long, c_double_p]),
    "gprc_gpr_fit": (C.c_int, [_P, _K, c_double_p, C.c_int, C.c_long, c_double_p, C.c_double, C.POINTER(_P),
                               c_double_p, c_long_p]),
    "gprc_gpr_fit_dev": (C.c_int, [_P, _K, _P, C.c_int, C.c_long, _P, C.c_double, C.POINTER(_P), c_double_p,
                                   c_long_p]),
    "gprc_gpr_fit_precomputed": (C.c_int, [_P, c_double_p, C.c_long, c_double_p, C.c_double, C.POINTER(_P),
                                           c_double_p, c_long_p]),
    "gprc_gpr_append": (C.c_int, [_P, c_double_p, C.c_long, c_double_p, c_double_p, c_long_p]),
    "gprc_gpr_predict": (C.c_int, [_P, c_double_p, C.c_long, c_double_p, c_double_p]),
    "gprc_gpr_predict_dev": (C.c_int, [_P, _P, C.c_long, _P, _P]),
    "gprc_gpr_predict_precomputed": (C.c_int, [_P, c_double_p, c_double_p, C.c_long, c_double_p, c_double_p]),
    "gprc_gpr_predict_cov": (C.c_int, [_P, c_double_p, C.c_long, c_double_p, c_double_p]),
    "gprc_grid_points": (C.c_int, [_P, c_double_p, C.c_int, C.c_int, c_double_p]),
    "gprc_gpr_predict_grid": (C.c_int, [_P, c_double_p, C.c_int, c_double_p, c_double_p]),
    "gprc_gpr_get": (C.c_int, [_P, C.c_int, c_double_p]),
    "gprc_gpr_n": (C.c_long, [_P]),
    "gprc_gpr_free": (None, [_P]),
    "gprc_logml": (C.c_int, [_P, _K, c_double_p, C.c_int, C.c_long, c_double_p, C.c_double, c_double_p, c_double_p,
                             c_long_p]),
    "gprc_logml_grad": (C.c_int, [_P, _K, c_double_p, C.c_int, C.c_long, c_double_p, C.c_double, C.c_int, c_double_p,
                                  C.c_int, c_long_p]),
    "gprc_logml_batch": (C.c_int, [_P, _K, C.c_int, c_double_p, C.c_int, C.c_long, c_double_p, C.c_double,
                                   c_double_p, c_double_p, c_long_p]),
    "gprc_optim_brent": (C.c_int, [OBJECTIVE_FN, _P, C.c_double, C.c_double, C.c_double, c_double_p]),
    "gprc_optim_vmmin": (C.c_int, [OBJECTIVE_FN, OBJECTIVE_FN, _P, c_double_p, C.c_int, C.c_int, C.c_double,
                                   C.c_double, c_double_p, c_int_p, c_int_p]),
    "gprc_optim_until_error": (C.c_int, [OBJECTIVE_FN, OBJECTIVE_FN, _P, c_double_p, C.c_int, C.c_int, C.c_double,
                                         C.c_double, c_double_p, c_double_p]),
    "gprc_fit_family": (C.c_int, [_P, C.c_int, c_double_p, C.c_int, C.c_long, c_double_p, C.c_double, C.c_int,
                                  c_double_p, c_int_p, c_double_p, c_long_p]),
    "gprc_gpc_fit": (C.c_int, [_P, _K, c_double_p, C.c_int, C.c_long, c_double_p, C.c_double, C.c_int, C.c_int,
                               C.POINTER(_P), c_int_p, c_double_p, C.c_int, c_double_p, c_double_p, c_int_p]),
    "gprc_gpc_fit_precomputed": (C.c_int, [_P, c_double_p, C.c_long, c_double_p, C.c_double, C.c_int, C.c_int,
                                           C.POINTER(_P), c_int_p, c_double_p, C.c_int, c_double_p, c_double_p,
                                           c_int_p]),
    "gprc_gpc_predict_latent": (C.c_int, [_P, c_double_p, C.c_long, c_double_p, c_double_p]),
    "gprc_gpc_predict_latent_precomputed": (C.c_int, [_P, c_double_p, c_double_p, C.c_long, c_double_p, c_double_p]),
    "gprc_gpc_predict_class": (C.c_int, [_P, c_double_p, C.c_long, c_double_p, c_int_p]),
    "gprc_logistic_gaussian": (C.c_int, [_P, c_double_p, c_double_p, C.c_long, c_double_p, c_int_p]),
    "gprc_gpc_get": (C.c_int, [_P, C.c_int, c_double_p]),
    "gprc_gpc_n": (C.c_long, [_P]),
    "gprc_gpc_dim": (C.c_int, [_P]),
    "gprc_gpr_dim": (C.c_int, [_P]),
    "gprc_gpc_free": (None, [_P]),
    "gprc_mvn_sample": (C.c_int, [_P, c_double_p, c_double_p, C.c_long, c_double_p, C.c_long, c_double_p, c_long_p]),
    "gprc_dist_unique_id": (C.c_int, [C.c_char_p, C.c_char_p]),
    "gprc_dist_create": (C.c_int, [_P, C.c_char_p, C.c_int, C.c_int, C.c_char_p, C.POINTER(_P)]),
    "gprc_dist_free": (None, [_P]),
    "gprc_dist_set_timeline": (C.c_int, [_P, C.c_int]),
    "gprc_dist_get_timeline": (C.c_int, [_P, c_double_p, C.c_int, C.POINTER(C.c_int)]),
    "gprc_dist_gpr_fit": (C.c_int, [_P, _K, c_double_p, C.c_int, C.c_long, c_double_p, C.c_double, c_double_p,
                                    c_double_p, c_long_p, c_double_p]),
    "gprc_dist_gpr_fit_replicated": (C.c_int, [_P, _K, c_double_p, C.c_int, C.c_long, c_double_p, C.c_double,
                                               C.POINTER(_P), c_double_p, c_long_p, c_double_p]),
    "gprc_dev_potrf": (C.c_int, [_P, _P, C.c_long, C.c_long, _P, c_long_p]),
    "gprc_dev_dgemm": (C.c_int, [_P, C.c_int, C.c_long, C.c_long, C.c_long, C.c_double, _P, C.c_long, _P, C.c_long,
                                 C.c_double, _P, C.c_long]),
    "gprc_dev_trtri": (C.c_int, [_P, _P, C.c_long, C.c_long, _P, _P, _P]),
    "gprc_dev_int8_rate": (C.c_int, [_P, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
}

_lib = None
_lock = threading.Lock()


def load():
    """dlopen libgprc.so and bind every declared symbol.  Needs no GPU (used by the CPU test tier)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise GprcError("libgprc.so is not built (%s); run `python -c 'import __graft_entry__ as g; g.build()'` "
                                "or `make -C gaussian-process-regression_b200/csrc`: there is no CPU fallback" % LIB_PATH)
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        raise GprcError("libgprc error %d: %s" % (rc, load().gprc_last_error().decode()))


def dptr(a: np.ndarray):
    return a.ctypes.data_as(c_double_p)


def f64(a, order="C"):
    return np.require(a, dtype=np.float64, requirements=["C_CONTIGUOUS" if order == "C" else "F_CONTIGUOUS", "ALIGNED"])


def points(X: np.ndarray) -> np.ndarray:
    """D x n array (columns are points, the reference's layout) -> the ABI's column-major D x n buffer, i.e. the
    points contiguous one after another."""
    return np.ascontiguousarray(np.asarray(X, dtype=np.float64).T)


class Context:
    """One device, one stream.  Created lazily; fails loudly without a GPU."""

    def __init__(self, device: int = 0):
        self.lib = load()
        h = _P()
        check(self.lib.gprc_ctx_create(C.byref(h), device))
        self.handle = h
        self.device = device

    def close(self):
        if getattr(self, "handle", None):
            self.lib.gprc_ctx_free(self.handle)
            self.handle = None

    # no __del__: at interpreter shutdown a context could be collected before the models that still point into it;
    # contexts live until close() is called explicitly or the process ends

    def set_option(self, option, value):
        check(self.lib.gprc_ctx_set_option(self.handle, option, int(value)))

    def sync(self):
        check(self.lib.gprc_ctx_sync(self.handle))

    def reset_timers(self):
        self.lib.gprc_ctx_reset_timers(self.handle)

    def timers(self):
        ms = (C.c_double * 8)()
        launches = C.c_long(0)
        check(self.lib.gprc_ctx_get_timers(self.handle, ms, C.byref(launches)))
        return {n: ms[i] for i, n in enumerate(T_NAMES)}, launches.value

    def trim(self):
        """release the context's cached device blocks; returns the number of bytes handed back to the driver"""
        n = C.c_ulonglong(0)
        check(self.lib.gprc_ctx_trim(self.handle, C.byref(n)))
        return int(n.value)

    def last_predict_path(self):
        return int(self.lib.gprc_ctx_last_predict_path(self.handle))

    def last_predict_chunks(self):
        return int(self.lib.gprc_ctx_last_predict_chunks(self.handle))

    def mark(self, slot):
        check(self.lib.gprc_ctx_mark(self.handle, slot))

    def elapsed_ms(self, a, b):
        ms = C.c_double(0.0)
        check(self.lib.gprc_ctx_elapsed_ms(self.handle, a, b, C.byref(ms)))
        return ms.value

    # device buffers (bench "value" leg: inputs resident in HBM)
    def malloc(self, nbytes):
        p = _P()
        check(self.lib.gprc_dev_malloc(self.handle, C.byref(p), nbytes))
        return p

    def free(self, p):
        check(self.lib.gprc_dev_free(self.handle, p))

    def h2d(self, p, arr: np.ndarray):
        check(self.lib.gprc_dev_h2d(self.handle, p, arr.ctypes.data_as(_P), arr.nbytes))

    def d2h(self, arr: np.ndarray, p):
        check(self.lib.gprc_dev_d2h(self.handle, arr.ctypes.data_as(_P), p, arr.nbytes))

    def upload(self, arr: np.ndarray):
        """Copy the array's buffer as it lies in memory (C- or Fortran-contiguous) to a new device buffer."""
        if not (arr.flags.c_contiguous or arr.flags.f_contiguous):
            arr = np.ascontiguousarray(arr)
        p = self.malloc(arr.nbytes)
        self.h2d(p, arr)
        return p


_default_ctx = {}


def default_context() -> Context:
    dev = int(os.environ.get("GPRC_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    if dev not in _default_ctx:
        _default_ctx[dev] = Context(dev)
    return _default_ctx[dev]
