"""The reference-side binding of INTEGRATION.md section 3, as a maintainer of jhamrick/bayesian-quadrature would add it:
a ctypes stub over the C-ABI of include/bq_b200.h and the three scoring loops of the reference's ``BQ`` class
(bayesian_quadrature/bq.py:399-402, :420-422, :442-444) replaced by ONE library call each.

``patch_reference(BQ)`` applies it to a class with the reference ``BQ`` object's attributes (the reference's own class, or
the state holder of tests/test_gpu_reference_binding.py, which runs the reference's scoring tests through libbq_b200.so).
Nothing of bayesian_quadrature_b200's Python layer is used here: this file talks to the shared library only."""
import ctypes
import logging
import os

import numpy as np

LIB = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bayesian_quadrature_b200", "libbq_b200.so")
_lib = None
_dp, _ip, _vp = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int), ctypes.c_void_p
ST_SHORTCUT, ST_NOTPD, ST_ESM_INF, ST_EM_INF, ST_ESM_BAD, ST_EM_BAD, ST_XA_BAD = 1, 2, 4, 8, 16, 32, 64
logger = logging.getLogger("bayesian_quadrature")


def lib():
    global _lib
    if _lib is None:
        L = ctypes.CDLL(LIB)
        L.bqb_batch_create.argtypes = [ctypes.POINTER(_vp), ctypes.c_int, ctypes.c_int, ctypes.c_int]
        L.bqb_batch_destroy.argtypes = [_vp]
        L.bqb_batch_setup.argtypes = [_vp, _ip, _ip, _dp, _dp, ctypes.c_int, _dp, _dp, _dp, ctypes.c_int, _vp]
        L.bqb_batch_info.argtypes = [_vp, _dp, _dp, _dp, _ip, _dp]
        L.bqb_batch_set_approx.argtypes = [_vp, ctypes.c_int, _dp, _dp, _dp, ctypes.c_int, ctypes.c_longlong, ctypes.c_int]
        L.bqb_score_host.argtypes = [_vp, _dp, ctypes.c_longlong, ctypes.c_int, _dp, _dp, _ip]
        L.bqb_last_error.restype = ctypes.c_char_p
        _lib = L
    return _lib


def _p(a, t=_dp):
    return a.ctypes.data_as(t)


class DeviceModel(object):
    """Factors of the current (x_s, l_s, x_c, hyper-parameters) state of a reference BQ object on the GPU."""

    def __init__(self, bq, device=0):
        L = lib()
        self.h = _vp()
        if L.bqb_batch_create(ctypes.byref(self.h), device, 1, bq.ns) != 0:
            raise RuntimeError(L.bqb_last_error())
        ns, nc = np.array([bq.ns], np.int32), np.array([bq.nc], np.int32)
        x_s, l_s = np.ascontiguousarray(bq.x_s, dtype=np.float64), np.ascontiguousarray(bq.l_s, dtype=np.float64)
        x_c = np.zeros(16)
        x_c[:bq.nc] = bq.x_c
        ptl, pl = np.asarray(bq.gp_log_l.params, dtype=np.float64), np.asarray(bq.gp_l.params, dtype=np.float64)
        hyp = np.array([ptl[0], ptl[1], ptl[-1], pl[0], pl[1], pl[-1]])                     # h_tl, w_tl, s_tl, h_l, w_l, s_l
        periodic = type(bq.gp_l.K).__name__ == "PeriodicKernel"
        if periodic or bq.options['use_approx']:
            # non-Gaussian kernel / trapezoid integrals (bq.py:498-510): kernel kind, the two periods, the grid of bq.py:167-171
            period = np.array([ptl[2], pl[2]]) if periodic else None
            xo = np.ascontiguousarray(bq._approx_x, dtype=np.float64) if bq.options['use_approx'] else None
            p_xo = np.ascontiguousarray(bq._approx_px, dtype=np.float64) if bq.options['use_approx'] else None
            if L.bqb_batch_set_approx(self.h, int(periodic), _p(period) if periodic else None, _p(xo) if xo is not None else None,
                                      _p(p_xo) if xo is not None else None, 0 if xo is None else xo.size, 0, 0) != 0:
                raise RuntimeError(L.bqb_last_error())
        prior = np.array([bq.options['x_mean'][0], bq.options['x_cov'][0, 0], bq.options['candidate_thresh']], dtype=np.float64)
        rc = L.bqb_batch_setup(self.h, _p(ns, _ip), _p(nc, _ip), _p(x_s), _p(l_s), bq.ns, _p(x_c), _p(hyp), _p(prior), 0, None)
        if rc != 0:
            msg = L.bqb_last_error()
            L.bqb_batch_destroy(self.h)
            raise RuntimeError(msg)
        st = np.zeros(1, np.int32)
        L.bqb_batch_info(self.h, None, None, None, _p(st, _ip), None)
        if st[0]:
            L.bqb_batch_destroy(self.h)
            raise np.linalg.LinAlgError("device setup status %d" % st[0])

    def esm_and_em(self, x_a):
        x_a = np.ascontiguousarray(x_a, dtype=np.float64)
        esm, em = np.empty(x_a.size), np.empty(x_a.size)
        st = np.empty(x_a.size, np.int32)
        if lib().bqb_score_host(self.h, _p(x_a), 0, x_a.size, _p(esm), _p(em), _p(st, _ip)) != 0:
            raise RuntimeError(lib().bqb_last_error())
        return esm, em, st

    def __del__(self):
        if getattr(self, "h", None):
            lib().bqb_batch_destroy(self.h)
            self.h = None


def _device_model(self):
    """Memoised like the gp package's Kxx / Lxx: rebuilt when data, candidates or parameters changed."""
    key = (self.x_s.tobytes(), self.l_s.tobytes(), self.x_c.tobytes(), tuple(self.gp_log_l.params), tuple(self.gp_l.params),
           bool(self.options['use_approx']))
    cached = getattr(self, "_b200", None)
    if cached is None or cached[0] != key:
        self._b200 = (key, DeviceModel(self))
    return self._b200[1]


def _raise_like_esm_and_em(x_a, esm, em, st):
    """bq.py:451-452 and :514-525 on the per-point status bits."""
    if (st & ST_XA_BAD).any():
        raise ValueError("invalid value for x_a: %s", x_a[np.argmax(st & ST_XA_BAD != 0)])
    if (st & ST_ESM_BAD).any():
        i = int(np.argmax(st & ST_ESM_BAD != 0))
        raise RuntimeError("invalid expected squared mean for x_a=%s: %s" % (x_a[[i]], esm[i]))
    if (st & ST_EM_BAD).any():
        i = int(np.argmax(st & ST_EM_BAD != 0))
        raise RuntimeError("invalid expected mean for x_a=%s: %s" % (x_a[[i]], em[i]))
    for i in np.nonzero(st & ST_ESM_INF)[0]:
        logger.warn("expected squared mean for x_a=%s is infinity!", x_a[[i]])
    for i in np.nonzero(st & ST_EM_INF)[0]:
        logger.warn("expected mean for x_a=%s is infinity!", x_a[[i]])


def expected_squared_mean_and_mean(self, x_a):
    esm, em, st = self._device_model().esm_and_em(x_a)      # replaces: for i in xrange(x_a.shape[0]): self._esm_and_em(x_a[[i]])
    _raise_like_esm_and_em(np.asarray(x_a), esm, em, st)
    return np.stack([esm, em], axis=1)


def expected_squared_mean(self, x_a):
    return expected_squared_mean_and_mean(self, x_a)[:, 0]


def expected_mean(self, x_a):
    return expected_squared_mean_and_mean(self, x_a)[:, 1]


def patch_reference(BQ):
    """Returns a subclass of the reference's BQ whose three scoring loops go through libbq_b200.so; everything else -- Z_mean
    and Z_var (Cython bq_c), the gp objects, sample_hypers, marginalize, choose_next -- is the reference's own code."""
    return type("BQ_b200", (BQ,), {
        "_device_model": _device_model,
        "expected_squared_mean_and_mean": expected_squared_mean_and_mean,
        "expected_squared_mean": expected_squared_mean,
        "expected_mean": expected_mean,
    })
