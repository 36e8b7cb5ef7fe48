"""ctypes binding of libbq_b200.so (C-ABI in include/bq_b200.h).

There is no CPU fallback: if the CUDA library cannot be loaded, or no sm_100 device is
present, every entry point raises.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BQB200_LIB") or os.path.join(HERE, "libbq_b200.so")     # override: A/B of kernel variants
NC_MAX = 16

ST_OK, ST_SHORTCUT, ST_NOTPD, ST_ESM_INF, ST_EM_INF, ST_ESM_BAD, ST_EM_BAD, ST_XA_BAD = 0, 1, 2, 4, 8, 16, 32, 64
SETUP_OK, SETUP_KTL_NOTPD, SETUP_KL_NOTPD, SETUP_MEAN_TOO_LARGE, SETUP_BAD_INPUT = 0, 1, 2, 3, 4
EINVAL, EUNSUPPORTED, ESTATE, ENUMERIC = -1, -2, -3, -4

_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)
_vp = ctypes.c_void_p
_ll = ctypes.c_longlong

#: every symbol include/bq_b200.h declares (checked by tests/test_capi_symbols.py)
SYMBOLS = {
    "bqb_last_error": (ctypes.c_char_p, []),
    "bqb_version": (ctypes.c_int, []),
    "bqb_device_count": (ctypes.c_int, [_ip]),
    "bqb_ns_capacity": (ctypes.c_int, [ctypes.c_int]),
    "bqb_batch_create": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "bqb_batch_destroy": (None, [_vp]),
    "bqb_batch_setup": (ctypes.c_int, [_vp, _ip, _ip, _dp, _dp, ctypes.c_int, _dp, _dp, _dp, ctypes.c_int, _vp]),
    "bqb_batch_stage": (ctypes.c_int, [_vp, _ip, _dp, _dp, ctypes.c_int, _dp, _dp, _vp]),
    "bqb_batch_set_hypers": (ctypes.c_int, [_vp, _dp, _vp]),
    "bqb_batch_log_lh_grad": (ctypes.c_int, [_vp, _dp, _ip, ctypes.c_int, ctypes.c_int, _dp, _dp, _ip, _vp]),
    "bqb_batch_log_lh_grad_periodic": (ctypes.c_int, [_vp, _dp, _dp, _ip, ctypes.c_int, ctypes.c_int, _dp, _dp, _ip, _vp]),
    "bqb_batch_set_periods": (ctypes.c_int, [_vp, _dp, _vp]),
    "bqb_batch_set_approx": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp, _dp, ctypes.c_int, _ll, ctypes.c_int]),
    "bqb_batch_setup_device": (ctypes.c_int, [_vp, ctypes.c_int, _vp]),
    "bqb_batch_seed_candidates": (ctypes.c_int, [_vp, ctypes.POINTER(ctypes.c_uint), _vp]),
    "bqb_batch_rng_get": (ctypes.c_int, [_vp, ctypes.POINTER(ctypes.c_uint), _ip]),
    "bqb_batch_rng_set": (ctypes.c_int, [_vp, ctypes.POINTER(ctypes.c_uint), _ip]),
    "bqb_batch_draw_candidates": (ctypes.c_int, [_vp, ctypes.c_int, _vp]),
    "bqb_batch_draw_candidates_wrapped": (ctypes.c_int, [_vp, ctypes.c_int, _vp]),
    "bqb_batch_add_observations": (ctypes.c_int, [_vp, _vp, _vp, _vp]),
    "bqb_batch_get_staged": (ctypes.c_int, [_vp, _ip, _ip, _dp, _dp, _dp]),
    "bqb_batch_capacity": (ctypes.c_int, [_vp]),
    "bqb_batch_info": (ctypes.c_int, [_vp, _dp, _dp, _dp, _ip, _dp]),
    "bqb_score_device": (ctypes.c_int, [_vp, _vp, _ll, ctypes.c_int, _vp, _vp, _vp, _ll, _vp, _vp]),
    "bqb_score_device_range": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp, _ll, ctypes.c_int, _vp, _vp, _vp, _ll, _vp, _vp]),
    "bqb_score_device_grouped": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp, _ll, ctypes.c_int, ctypes.c_int, _vp, _vp, _vp, _ll,
                                                _vp, _vp]),
    "bqb_sum_neg_accum_device": (ctypes.c_int, [_vp, _vp, _ll, ctypes.c_int, _ll, _vp, _vp]),
    "bqb_sum_neg_accum_groups_device": (ctypes.c_int, [_vp, _vp, _ll, ctypes.c_int, ctypes.c_int, _ll, _vp, _ll, _vp]),
    "bqb_predict_device": (ctypes.c_int, [_vp, _vp, _ll, ctypes.c_int, _vp, _vp, _ll, _vp]),
    "bqb_predict_host": (ctypes.c_int, [_vp, _dp, _ll, ctypes.c_int, _dp, _dp]),
    "bqb_predict_rows_device": (ctypes.c_int, [_vp, _ip, ctypes.c_int, _vp, _ll, ctypes.c_int, _vp, _vp, _ll, _vp]),
    "bqb_predict_rows_host": (ctypes.c_int, [_vp, _ip, ctypes.c_int, _dp, _ll, ctypes.c_int, _dp, _dp]),
    "bqb_alpha_read": (ctypes.c_int, [_vp, ctypes.c_int, _dp]),
    "bqb_expected_var_host": (ctypes.c_int, [_vp, ctypes.c_int, _dp, ctypes.c_int, _dp, _ip]),
    "bqb_score_host": (ctypes.c_int, [_vp, _dp, _ll, ctypes.c_int, _dp, _dp, _ip]),
    "bqb_expected_var_device": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _ll, _vp, _vp]),
    "bqb_expected_var_rows_device": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp, _ll, _ll, _vp, _ll, _vp]),
    "bqb_mean_neg_device": (ctypes.c_int, [_vp, _vp, _ll, _ll, _vp, _vp]),
    "bqb_argmin_device": (ctypes.c_int, [_vp, _vp, _ll, _dp, ctypes.POINTER(_ll), _vp]),
    "bqb_argmin_pair_device": (ctypes.c_int, [_vp, _vp, _ll, _ll, _vp, _vp]),
    "bqb_choose_step_device": (ctypes.c_int, [_vp, ctypes.c_int, _vp, ctypes.c_int, _vp, _vp, _ll, _vp, _vp]),
    "bqb_choose_step_exchange": (ctypes.c_int, [_vp, ctypes.c_int, _vp, ctypes.c_int, _vp, _vp, _ll, _ll, ctypes.POINTER(_vp), ctypes.c_int,
                                                ctypes.c_int, ctypes.c_ulonglong, _vp, _vp]),
    "bqb_argmin_rows_device": (ctypes.c_int, [_vp, _vp, _ll, _ll, _vp, _vp, _vp]),
    "bqb_argmin_ties_rows_device": (ctypes.c_int, [_vp, _vp, _ll, _ll, _vp, _vp, _vp, _vp, _vp]),
    "bqb_batch_set_cutoff": (ctypes.c_int, [_vp, ctypes.c_double]),
    "bqb_batch_set_presort": (ctypes.c_int, [_vp, ctypes.c_int]),
    "bqb_batch_set_zero_copy": (ctypes.c_int, [_vp, ctypes.c_int]),
    "bqb_batch_work_counter": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.POINTER(ctypes.c_ulonglong)]),
    "bqb_launch_count": (ctypes.c_ulonglong, [_vp]),
    "bqb_model_doubles": (ctypes.c_int, [_vp]),
    "bqb_model_read": (ctypes.c_int, [_vp, ctypes.c_int, _dp]),
}

_lib = None


class BQB200Error(RuntimeError):
    pass


def load():
    """Loads the CUDA library; raises ImportError when it is missing (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "bayesian_quadrature_b200: %s is missing — build it with "
                "`python -m bayesian_quadrature_b200.build` (needs nvcc, sm_100a). "
                "There is no CPU fallback." % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def _check(rc, what):
    if rc != 0:
        msg = load().bqb_last_error().decode("utf-8", "replace")
        if rc == EINVAL:
            raise ValueError("%s: %s" % (what, msg))
        if rc == EUNSUPPORTED:
            raise NotImplementedError("%s: %s" % (what, msg))
        if rc == ENUMERIC:
            raise np.linalg.LinAlgError("%s: %s" % (what, msg))
        raise BQB200Error("%s failed (code %d): %s" % (what, rc, msg))


def device_count():
    n = ctypes.c_int(0)
    _check(load().bqb_device_count(ctypes.byref(n)), "bqb_device_count")
    return n.value


def ns_capacity(ns):
    """Padded observation capacity class the library uses for `ns` observations; NotImplementedError beyond the device limit."""
    cap = load().bqb_ns_capacity(int(ns))
    if cap == EUNSUPPORTED:
        raise NotImplementedError("%d observations per instance exceed the device limit" % ns)
    if cap < 0:
        raise ValueError("invalid number of observations: %s" % ns)
    return cap


def _d(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _pd(a):
    return a.ctypes.data_as(_dp)


def _ptr(t):
    """Device pointer of a torch tensor (or None)."""
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


def _stream(stream):
    """A CUDA stream handle as the C-ABI takes it (None: the legacy default stream)."""
    return _vp(stream) if stream else None


def _query(x, n_inst=None, name="x_a"):
    """(row stride, na) of query points x: [na] shared by every instance (stride 0) or [B, na], a numpy array or a torch
    tensor.  With ``n_inst`` a 2-D x must have that many rows."""
    if x.ndim == 1:
        return 0, x.shape[0]
    if n_inst is not None and x.shape[0] != n_inst:
        raise ValueError("%s must be [na] or [n_inst, na]" % name)
    return (x.shape[1] if isinstance(x, np.ndarray) else x.stride(0)), x.shape[1]


class Batch(object):
    """B model instances (one BQ problem under one hyper-parameter set each) resident on one GPU."""

    def __init__(self, n_inst, ns_max, device=0):
        self._h = _vp()
        self.n_inst, self.ns_max, self.device = int(n_inst), int(ns_max), int(device)
        _check(load().bqb_batch_create(ctypes.byref(self._h), self.device, self.n_inst, self.ns_max), "bqb_batch_create")

    def close(self):
        if getattr(self, "_h", None):
            try:
                load().bqb_batch_destroy(self._h)
            except Exception:          # interpreter shutdown: module globals may already be gone
                pass
            self._h = None

    __del__ = close

    def setup(self, ns, nc, x_s, l_s, x_c, hyp, prior, check_max=False, stream=None):
        """x_s, l_s: [B, in_stride]; x_c: [B, <=16]; hyp: [B, 6]; prior: [B, 3] (host arrays)."""
        B = self.n_inst
        ns = np.ascontiguousarray(np.broadcast_to(np.asarray(ns, dtype=np.int32), (B,)))
        nc = np.ascontiguousarray(np.broadcast_to(np.asarray(nc, dtype=np.int32), (B,)))
        x_s, l_s = _d(x_s).reshape(B, -1), _d(l_s).reshape(B, -1)
        xc = np.zeros((B, NC_MAX))
        x_c = _d(x_c).reshape(B, -1)
        if x_c.shape[1] > NC_MAX:
            raise NotImplementedError("more than %d candidates per instance" % NC_MAX)
        xc[:, :x_c.shape[1]] = x_c
        hyp, prior = _d(hyp).reshape(B, 6), _d(prior).reshape(B, 3)
        _check(load().bqb_batch_setup(self._h, ns.ctypes.data_as(_ip), nc.ctypes.data_as(_ip), _pd(x_s), _pd(l_s),
                                      x_s.shape[1], _pd(xc), _pd(hyp), _pd(prior), int(check_max),
                                      _stream(stream)), "bqb_batch_setup")
        self.ns, self.nc = ns, nc
        return self.info()

    def info(self):
        B = self.n_inst
        Zm, Zv, llh = np.empty(B), np.empty(B), np.empty(B)
        st = np.empty(B, dtype=np.int32)
        l_c = np.empty((B, NC_MAX))
        _check(load().bqb_batch_info(self._h, _pd(Zm), _pd(Zv), _pd(llh), st.ctypes.data_as(_ip), _pd(l_c)), "bqb_batch_info")
        return {"Z_mean": Zm, "Z_var": Zv, "log_lh": llh, "status": st, "l_c": l_c}

    # ---- device-resident active sampling (include/bq_b200.h, "device-resident active sampling")
    @property
    def capacity(self):
        return int(load().bqb_batch_capacity(self._h))

    def stage(self, ns, x_s, l_s, hyp, prior, stream=None):
        B = self.n_inst
        ns = np.ascontiguousarray(np.broadcast_to(np.asarray(ns, dtype=np.int32), (B,)))
        x_s, l_s = _d(x_s).reshape(B, -1), _d(l_s).reshape(B, -1)
        hyp, prior = _d(hyp).reshape(B, 6), _d(prior).reshape(B, 3)
        _check(load().bqb_batch_stage(self._h, ns.ctypes.data_as(_ip), _pd(x_s), _pd(l_s), x_s.shape[1], _pd(hyp), _pd(prior),
                                      _stream(stream)), "bqb_batch_stage")

    def set_hypers(self, hyp, stream=None):
        """Replace the hyper-parameters [n_inst, 6] of the staged instances (the next setup_device uses them)."""
        hyp = _d(hyp).reshape(self.n_inst, 6)
        _check(load().bqb_batch_set_hypers(self._h, _pd(hyp), _stream(stream)), "bqb_batch_set_hypers")

    def log_lh_grad(self, hyp, inst=None, check_max=True, stream=None, period=None):
        """Joint log marginal likelihood and its gradient for rows of hyper-parameters hyp [n, 6] (h, w, s of gp_log_l,
        then of gp_l); row r is instance inst[r] (default: instance r).  Evaluated on the staged observations and
        candidates; the set-up model is left untouched.  Returns (log_lh [n], grad [n, 6], status [n]); a row whose status
        is not SETUP_OK has log_lh -inf and a NaN gradient.  A batch of the periodic kernel takes the periods of every row,
        period [n, 2] = (p of gp_log_l, p of gp_l), and returns grad [n, 8] in the order h_tl, w_tl, s_tl, h_l, w_l, s_l,
        p_tl, p_l."""
        hyp = _d(hyp).reshape(-1, 6)
        n = hyp.shape[0]
        if period is not None:
            period = _d(period).reshape(-1, 2)
            if period.shape[0] != n:
                raise ValueError("period must have one row per row of hyp")
        if inst is not None:
            inst = np.ascontiguousarray(inst, dtype=np.int32).reshape(-1)
            if inst.shape[0] != n:
                raise ValueError("inst must have one entry per row of hyp")
        llh, grad, st = np.empty(n), np.empty((n, 6 if period is None else 8)), np.empty(n, dtype=np.int32)
        rows = (inst.ctypes.data_as(_ip) if inst is not None else None, n, int(check_max), _pd(llh), _pd(grad),
                st.ctypes.data_as(_ip), _stream(stream))
        if period is None:
            _check(load().bqb_batch_log_lh_grad(self._h, _pd(hyp), *rows), "bqb_batch_log_lh_grad")
        else:
            _check(load().bqb_batch_log_lh_grad_periodic(self._h, _pd(hyp), _pd(period), *rows), "bqb_batch_log_lh_grad_periodic")
        return llh, grad, st

    def log_lh_grad_periodic(self, hyp, period, inst=None, check_max=True, stream=None):
        """log_lh_grad(hyp, inst, check_max, stream, period=period): the periodic kernel's form under its own name."""
        return self.log_lh_grad(hyp, inst, check_max, stream, period=period)

    def set_periods(self, period, stream=None):
        """Replace the periods [n_inst, 2] of a batch of the periodic kernel (the next setup_device uses them)."""
        period = _d(period).reshape(self.n_inst, 2)
        _check(load().bqb_batch_set_periods(self._h, _pd(period), _stream(stream)), "bqb_batch_set_periods")

    def set_approx(self, kernel_kind=0, period=None, xo=None, p_xo=None, force_generic=False):
        """Kernel kind (0 Gaussian, 1 periodic with period [n_inst, 2] = p of gp_log_l / gp_l) and, when ``xo`` / ``p_xo``
        are given ([n_xo] shared or [n_inst, n_xo]), the trapezoid approximation of the integrals over that grid
        (``use_approx`` of the reference).  Takes effect at the next setup."""
        n_xo, stride = 0, 0
        if period is not None:
            period = _d(period).reshape(self.n_inst, 2)
        if xo is not None:
            xo, p_xo = _d(xo), _d(p_xo)
            if xo.shape != p_xo.shape:
                raise ValueError("xo and p_xo must have the same shape")
            n_xo = xo.shape[-1]
            if xo.ndim == 2:
                if xo.shape[0] != self.n_inst:
                    raise ValueError("per-instance grids must be [n_inst, n_xo]")
                stride = n_xo
        self._approx_keep = (period, xo, p_xo)
        _check(load().bqb_batch_set_approx(self._h, int(kernel_kind), _pd(period) if period is not None else None,
                                           _pd(xo) if xo is not None else None, _pd(p_xo) if p_xo is not None else None,
                                           int(n_xo), int(stride), int(bool(force_generic))), "bqb_batch_set_approx")

    def setup_device(self, check_max=False, stream=None):
        _check(load().bqb_batch_setup_device(self._h, int(check_max), _stream(stream)), "bqb_batch_setup_device")
        return self.info()

    def seed_candidates(self, seeds, stream=None):
        seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
        if seeds.shape != (self.n_inst,):
            raise ValueError("one 32-bit seed per instance")
        _check(load().bqb_batch_seed_candidates(self._h, seeds.ctypes.data_as(ctypes.POINTER(ctypes.c_uint)),
                                                _stream(stream)), "bqb_batch_seed_candidates")

    def rng_get(self):
        """(words [624, n_inst] uint32, positions [n_inst] int32) of the per-instance MT19937 generators."""
        mt = np.empty((624, self.n_inst), dtype=np.uint32)
        pos = np.empty(self.n_inst, dtype=np.int32)
        _check(load().bqb_batch_rng_get(self._h, mt.ctypes.data_as(ctypes.POINTER(ctypes.c_uint)), pos.ctypes.data_as(_ip)),
               "bqb_batch_rng_get")
        return mt, pos

    def rng_set(self, mt, pos):
        mt = np.ascontiguousarray(mt, dtype=np.uint32)
        pos = np.ascontiguousarray(pos, dtype=np.int32)
        if mt.shape != (624, self.n_inst) or pos.shape != (self.n_inst,):
            raise ValueError("mt must be [624, n_inst], pos [n_inst]")
        _check(load().bqb_batch_rng_set(self._h, mt.ctypes.data_as(ctypes.POINTER(ctypes.c_uint)), pos.ctypes.data_as(_ip)),
               "bqb_batch_rng_set")

    def draw_candidates(self, n_candidate, stream=None):
        _check(load().bqb_batch_draw_candidates(self._h, int(n_candidate), _stream(stream)),
               "bqb_batch_draw_candidates")

    def draw_candidates_wrapped(self, n_candidate, stream=None):
        """draw_candidates on [-pi p_tl, pi p_tl] (periodic kernel)."""
        _check(load().bqb_batch_draw_candidates_wrapped(self._h, int(n_candidate), _stream(stream)),
               "bqb_batch_draw_candidates_wrapped")

    def add_observations(self, x_new, l_new, stream=None):
        """x_new, l_new: float64 CUDA tensors [n_inst]."""
        _check(load().bqb_batch_add_observations(self._h, _ptr(x_new), _ptr(l_new), _stream(stream)),
               "bqb_batch_add_observations")

    def get_staged(self):
        B, cap = self.n_inst, self.capacity
        ns, nc = np.empty(B, dtype=np.int32), np.empty(B, dtype=np.int32)
        x_s, l_s, x_c = np.empty((B, cap)), np.empty((B, cap)), np.empty((B, NC_MAX))
        _check(load().bqb_batch_get_staged(self._h, ns.ctypes.data_as(_ip), nc.ctypes.data_as(_ip), _pd(x_s), _pd(l_s), _pd(x_c)),
               "bqb_batch_get_staged")
        return {"ns": ns, "nc": nc, "x_s": x_s, "l_s": l_s, "x_c": x_c}

    def score_host(self, x_a, want_em=True, want_status=True):
        """x_a: [na] shared by all instances, or [B, na].  Returns (esm, em, status) as [B, na] numpy arrays."""
        x_a = _d(x_a)
        B = self.n_inst
        stride, na = _query(x_a, B)
        esm = np.empty((B, na))
        em = np.empty((B, na)) if want_em else None
        st = np.empty((B, na), dtype=np.int32) if want_status else None
        _check(load().bqb_score_host(self._h, _pd(x_a), stride, na, _pd(esm), _pd(em) if want_em else None,
                                     st.ctypes.data_as(_ip) if want_status else None), "bqb_score_host")
        return esm, em, st

    def predict_host(self, x):
        """(l_mean, v_log_l) as [B, na] numpy arrays for x [na] (shared) or [B, na]: gp_l.mean(x), diag gp_log_l.cov(x)."""
        x = _d(x)
        B = self.n_inst
        stride, na = _query(x, B, "x")
        m, v = np.empty((B, na)), np.empty((B, na))
        _check(load().bqb_predict_host(self._h, _pd(x), stride, na, _pd(m), _pd(v)), "bqb_predict_host")
        return m, v

    def predict_device(self, x, l_mean, v_log_l, stream=None):
        """torch CUDA tensors: x float64 [na] or [B, na]; outputs float64 [B, na]."""
        stride, na = _query(x)
        _check(load().bqb_predict_device(self._h, _ptr(x), stride, na, _ptr(l_mean), _ptr(v_log_l), l_mean.stride(0),
                                         _stream(stream)), "bqb_predict_device")

    @staticmethod
    def _rows(rows):
        """(int32 array or None, its ctypes pointer or None, its length) of an instance list (None: every instance)."""
        if rows is None:
            return None, None, 0
        rows = np.ascontiguousarray(rows, dtype=np.int32).reshape(-1)
        return rows, rows.ctypes.data_as(_ip), rows.shape[0]

    def predict_rows_host(self, x, rows=None):
        """(l_mean, v_log_l) [B, na] numpy arrays for x [na] (shared) or [B, na]: gp_l.mean(x), diag gp_log_l.cov(x) of the
        instances in ``rows`` (default: all), for any batch and any s_l; the rows of other instances are NaN."""
        x = _d(x)
        B = self.n_inst
        stride, na = _query(x, B, "x")
        m, v = np.full((B, na), np.nan), np.full((B, na), np.nan)
        rows, rp, n = self._rows(rows)
        _check(load().bqb_predict_rows_host(self._h, rp, n, _pd(x), stride, na, _pd(m), _pd(v)), "bqb_predict_rows_host")
        return m, v

    def predict_rows_device(self, x, l_mean, v_log_l, rows=None, stream=None):
        """predict_rows_host on torch CUDA tensors: x float64 [na] or [B, na]; l_mean / v_log_l float64 [B, na] with unit
        column stride.  Only the rows of the listed instances (default: all) are written; no host synchronisation."""
        stride, na = _query(x)
        rows, rp, n = self._rows(rows)
        _check(load().bqb_predict_rows_device(self._h, rp, n, _ptr(x), stride, na, _ptr(l_mean), _ptr(v_log_l),
                                              l_mean.stride(0), _stream(stream)), "bqb_predict_rows_device")

    def read_alpha(self, inst=0):
        """alpha_l = (K_l + s_l^2 I)^-1 l_sc of instance ``inst`` (ns + nc entries): observations in ascending order, then the
        candidates, as in the model block."""
        hdr = self.read_model(inst)                   # H_NS, H_NC: the counts of the last setup
        out = np.empty(int(hdr[0]) + int(hdr[1]))
        _check(load().bqb_alpha_read(self._h, int(inst), _pd(out)), "bqb_alpha_read")
        return out

    def expected_var_host(self, x_a, inst=0, out=None):
        """BQ.expected_Z_var for one instance: numpy in, numpy out, plus the OR of the status bits.
        `out` may be a preallocated (ideally page-locked) float64 array."""
        x_a = _d(x_a)
        if out is None:
            out = np.empty(x_a.shape[0])
        fl = ctypes.c_int(0)
        _check(load().bqb_expected_var_host(self._h, int(inst), _pd(x_a), x_a.shape[0], _pd(out), ctypes.byref(fl)),
               "bqb_expected_var_host")
        return out, fl.value

    def score_device(self, x_a, esm, em=None, status=None, flags=None, stream=None):
        """torch CUDA tensors: x_a float64 [na] or [B, na]; esm/em float64 [B, na]; status int32 [B, na]."""
        stride, na = _query(x_a)
        out_stride = esm.stride(0) if esm.dim() == 2 else esm.shape[0]
        _check(load().bqb_score_device(self._h, _ptr(x_a), stride, na, _ptr(esm), _ptr(em), _ptr(status), out_stride,
                                       _ptr(flags), _stream(stream)), "bqb_score_device")

    def score_device_range(self, inst0, n_inst, x_a, esm, em=None, status=None, flags=None, stream=None):
        """score_device for instances [inst0, inst0 + n_inst); row 0 of esm / em / status / flags belongs to inst0."""
        stride, na = _query(x_a)
        out_stride = esm.stride(0) if esm.dim() == 2 else esm.shape[0]
        _check(load().bqb_score_device_range(self._h, int(inst0), int(n_inst), _ptr(x_a), stride, na, _ptr(esm), _ptr(em),
                                             _ptr(status), out_stride, _ptr(flags), _stream(stream)),
               "bqb_score_device_range")

    def score_device_grouped(self, inst0, n_inst, x_a, xa_group, esm, em=None, status=None, flags=None, stream=None):
        """score_device_range where instance inst0 + i reads row i // xa_group of x_a [n_inst / xa_group, na] (or the shared
        [na]); inst0 must be a multiple of xa_group."""
        stride, na = _query(x_a)
        if x_a.dim() != 1 and xa_group >= 1 and x_a.shape[0] < -(-int(n_inst) // int(xa_group)):
            raise ValueError("x_a has %d rows; %d instances in groups of %d read %d" % (
                x_a.shape[0], n_inst, xa_group, -(-int(n_inst) // int(xa_group))))
        out_stride = esm.stride(0) if esm.dim() == 2 else esm.shape[0]
        _check(load().bqb_score_device_grouped(self._h, int(inst0), int(n_inst), _ptr(x_a), stride, int(xa_group), na, _ptr(esm),
                                               _ptr(em), _ptr(status), out_stride, _ptr(flags), _stream(stream)),
               "bqb_score_device_grouped")

    def sum_neg_accum_groups_device(self, esm, n_groups, group_size, acc, stream=None):
        """acc[g] += sum over rows g*group_size ... (g+1)*group_size - 1 of -esm, in row order, for g < n_groups."""
        acc_stride = acc.stride(0) if acc.dim() == 2 else acc.shape[0]
        _check(load().bqb_sum_neg_accum_groups_device(self._h, _ptr(esm), esm.stride(0), int(n_groups), int(group_size), esm.shape[1],
                                                      _ptr(acc), acc_stride, _stream(stream)),
               "bqb_sum_neg_accum_groups_device")

    def sum_neg_accum_device(self, esm, n_rows, acc, stream=None):
        """acc[p] += sum over the first n_rows rows of -esm[:, p], in row order (running form of mean_neg_device)."""
        _check(load().bqb_sum_neg_accum_device(self._h, _ptr(esm), esm.stride(0), int(n_rows), esm.shape[1], _ptr(acc),
                                               _stream(stream)), "bqb_sum_neg_accum_device")

    def expected_var_device(self, inst, esm, out, stream=None):
        _check(load().bqb_expected_var_device(self._h, int(inst), _ptr(esm), esm.numel(), _ptr(out),
                                              _stream(stream)), "bqb_expected_var_device")

    def expected_var_rows_device(self, inst0, n_inst, esm, out, stream=None):
        """out[r] = Z_mean^2 + Z_var - esm[r] for instances inst0 + r, r < n_inst: float64 CUDA tensors [>= n_inst, na] with
        unit column stride (strided rows are fine; esm and out may be the same tensor)."""
        if esm.dim() != 2 or out.dim() != 2 or esm.shape[1] != out.shape[1] or min(esm.shape[0], out.shape[0]) < int(n_inst):
            raise ValueError("esm and out must be [>= n_inst, na] tensors with the same na")
        if (esm.shape[1] > 1 and esm.stride(1) != 1) or (out.shape[1] > 1 and out.stride(1) != 1):
            raise ValueError("esm and out must have contiguous rows")
        _check(load().bqb_expected_var_rows_device(self._h, int(inst0), int(n_inst), _ptr(esm), esm.stride(0), esm.shape[1],
                                                   _ptr(out), out.stride(0), _stream(stream)),
               "bqb_expected_var_rows_device")

    def mean_neg_device(self, esm, loss, stream=None):
        _check(load().bqb_mean_neg_device(self._h, _ptr(esm), esm.stride(0), esm.shape[1], _ptr(loss),
                                          _stream(stream)), "bqb_mean_neg_device")

    def argmin_device(self, v, stream=None):
        mn, idx = ctypes.c_double(0), _ll(0)
        _check(load().bqb_argmin_device(self._h, _ptr(v), v.numel(), ctypes.byref(mn), ctypes.byref(idx),
                                        _stream(stream)), "bqb_argmin_device")
        return mn.value, idx.value

    def argmin_pair_device(self, v, offset, pair, stream=None):
        """(min, first index + offset) of `v` written to the 2-element float64 CUDA tensor `pair`; no host sync."""
        _check(load().bqb_argmin_pair_device(self._h, _ptr(v), v.numel(), int(offset), _ptr(pair),
                                             _stream(stream)), "bqb_argmin_pair_device")

    def choose_step_device(self, x_a, esm, ev, pair, offset=0, inst=0, stream=None):
        """Fused esm + expected variance + (min, first index + offset) for one instance; CUDA tensors, no host sync."""
        _check(load().bqb_choose_step_device(self._h, int(inst), _ptr(x_a), x_a.numel(), _ptr(esm), _ptr(ev), int(offset),
                                             _ptr(pair), _stream(stream)), "bqb_choose_step_device")

    def choose_step_exchange(self, x_a, esm, ev, offset, peer_ptrs, world, rank, seq, out_ptr, inst=0, stream=None, cyclic_block=0):
        """choose_step_device + cross-rank exchange in the reduction kernel (see dist.PairExchange); no host sync."""
        _check(load().bqb_choose_step_exchange(self._h, int(inst), _ptr(x_a), x_a.numel(), _ptr(esm), _ptr(ev), int(offset),
                                               int(cyclic_block), peer_ptrs, int(world), int(rank), int(seq), _vp(out_ptr),
                                               _stream(stream)), "bqb_choose_step_exchange")

    def argmin_rows_device(self, v, mins, idxs, stream=None):
        """Per-instance (min, first index) of the CUDA tensor v [n_inst, n] into mins (float64) / idxs (int64)."""
        _check(load().bqb_argmin_rows_device(self._h, _ptr(v), v.stride(0), v.shape[1], _ptr(mins), _ptr(idxs),
                                             _stream(stream)), "bqb_argmin_rows_device")

    def argmin_ties_rows_device(self, v, mins, u, idxs, counts=None, stream=None):
        """Per-instance random pick among the points of v [n_inst, n] within np.isclose of mins [n_inst] (bq.py:664-665):
        the k-th close point, k = min(floor(u * c), c - 1) of c close points, for uniforms u [n_inst] in [0, 1), into
        idxs (int64); counts (int64, optional) receives c.  CUDA tensors, no host synchronisation."""
        _check(load().bqb_argmin_ties_rows_device(self._h, _ptr(v), v.stride(0), v.shape[1], _ptr(mins), _ptr(u), _ptr(idxs),
                                                  _ptr(counts), _stream(stream)), "bqb_argmin_ties_rows_device")

    def set_cutoff(self, cut_arg):
        """Relevance cut-off of the band skipping (default 72; float('inf') = dense algorithm)."""
        _check(load().bqb_batch_set_cutoff(self._h, float(cut_arg)), "bqb_batch_set_cutoff")

    def set_presort(self, mode):
        """Pre-sort of unsorted query vectors in the host entry points: 0 never, 1 automatic (default), 2 always."""
        _check(load().bqb_batch_set_presort(self._h, int(mode)), "bqb_batch_set_presort")

    def set_zero_copy(self, enable):
        """Host entry points with page-locked arrays: in-place PCIe access by the kernel (True, default) or staged copies."""
        _check(load().bqb_batch_set_zero_copy(self._h, int(bool(enable))), "bqb_batch_set_zero_copy")

    def work_counter(self, enable=True):
        """DMMA instructions executed since the last call (0 if the counter was off); (re)arms or disarms the counter."""
        n = ctypes.c_ulonglong(0)
        _check(load().bqb_batch_work_counter(self._h, int(bool(enable)), ctypes.byref(n)), "bqb_batch_work_counter")
        return int(n.value)

    @property
    def launch_count(self):
        return int(load().bqb_launch_count(self._h))

    def read_model(self, inst=0):
        n = load().bqb_model_doubles(self._h)
        out = np.empty(n)
        _check(load().bqb_model_read(self._h, int(inst), _pd(out)), "bqb_model_read")
        return out
