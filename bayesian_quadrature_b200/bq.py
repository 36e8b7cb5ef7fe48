"""``BQ`` — drop-in for ``bayesian_quadrature.BQ`` (reference: bayesian_quadrature/bq.py) whose
expected-variance active-sampling path runs on a B200 through libbq_b200.so.

Same constructor, options, methods, return types and exceptions as the reference class.  What
differs is *where the work happens*:

* ``expected_squared_mean`` / ``expected_mean`` / ``expected_squared_mean_and_mean`` /
  ``expected_Z_var`` make ONE device call for the whole vector ``x_a`` (the reference loops in
  Python and refactorises a bordered Gram matrix per point, bq.py:399-402 / :447-527);
* ``Z_mean`` / ``Z_var`` / ``l_c`` come from the device setup kernel, once per (data, hyper set);
* ``choose_next`` scores all sampled hyper-parameter sets as one device batch and reduces the
  marginal loss on device (bq.py:659-666); ``marginalize`` stays a generic host loop because it
  accepts arbitrary callables (bq.py:604-657).

Host-only pieces (candidate draw with the numpy RNG, hyper-parameter fitting/sampling, plotting,
pickling) stay host Python.  There is no CPU fallback for the device pieces: without the CUDA
library or a GPU they raise.
"""
import logging
import os
import warnings
from copy import copy, deepcopy

import numpy as np

from . import _lib
from . import util
from .gp import GP, GaussianKernel, PeriodicKernel

logger = logging.getLogger("bayesian_quadrature")
DTYPE = np.dtype("float64")
MIN = np.log(np.exp2(np.float64(np.finfo(np.float64).minexp + 4)))   # bq.py:15
MAX = np.log(np.exp2(np.float64(np.finfo(np.float64).maxexp - 4)))   # bq.py:16

_SETUP_ERRORS = {
    _lib.SETUP_KTL_NOTPD: (np.linalg.LinAlgError, "Matrix is not positive definite (gp_log_l.Kxx)"),
    _lib.SETUP_KL_NOTPD: (np.linalg.LinAlgError, "Matrix is not positive definite (gp_l.Kxx)"),
    _lib.SETUP_MEAN_TOO_LARGE: (np.linalg.LinAlgError, "GP mean is too large"),      # bq.py:947
    _lib.SETUP_BAD_INPUT: (ValueError, "invalid (non-finite or non-positive) model inputs"),
}


def _looks_sorted(x):
    """Sampled test (about 2000 points) for an ascending vector; only the speed of the device pass depends on it."""
    n = x.shape[0]
    stride = max(n // 2048, 1)
    i = np.arange(0, n - stride, stride)
    return bool((x[i] <= x[i + 1]).all() and (x[i] <= x[i + stride]).all())


def _raise_setup(status):
    exc, msg = _SETUP_ERRORS.get(int(status), (RuntimeError, "device setup failed with status %s" % status))
    raise exc(msg)


def _vonmises_px(x, mu, var):
    """Prior density of the wrapped (periodic) mode on the grid x: bq_c.p_x_vonmises / vonmises_logpdf (bq_c.pyx:31-60)
    with kappa = 1 / var.  The reference normalises with libc's j0 (the Bessel function of the FIRST kind), not I0: kept,
    so that results stay identical."""
    from scipy.special import j0
    kappa = 1.0 / var
    return np.exp(-np.log(2 * np.pi * j0(kappa)) + kappa * np.cos(np.asarray(x, dtype=DTYPE) - mu))


class _DeviceModel(object):
    """The device-resident factors of ONE BQ object: a single-instance batch handle that lives as long as the
    observation capacity class does.  ``refresh`` re-stages the data only when observations / candidates / prior
    changed and otherwise just replaces the six hyper-parameters and re-runs the setup kernel on the same buffers
    (what one evaluation of the hyper-parameter log-density costs, bq.py:533-552)."""

    def __init__(self, device):
        self.device = device
        self.batch = None
        self.cap = None
        self.data_key = None
        self.key = None          # (data_key, hyper-parameters) the factors on the device belong to
        self.guarded = False     # the bq.py:942-947 guard was evaluated for `key`
        self.status = None
        self.Z_mean = self.Z_var = self.log_lh = None
        self.l_c = None

    def close(self):
        if self.batch is not None:
            self.batch.close()
        self.batch, self.key, self.data_key = None, None, None

    def refresh(self, data_key, x_s, l_s, x_c, hyp, prior, check_max, approx=None):
        """``approx``: None (Gaussian kernel, closed-form integrals) or (kind, (p_tl, p_l), xo, p_xo) for the generic
        path (periodic kernel and / or the trapezoid approximation over the grid ``xo``; ``xo`` may be None)."""
        akey = None if approx is None else (approx[0], tuple(approx[1]), None if approx[2] is None else
                                            (approx[2].tobytes(), approx[3].tobytes()))
        key = (data_key, tuple(float(v) for v in hyp), akey)
        if key == self.key and (self.guarded or not check_max):
            return self
        ns, nc = x_s.shape[0], x_c.shape[0]
        cap = _lib.ns_capacity(ns)
        if self.batch is None or cap != self.cap:
            self.close()
            self.batch, self.cap = _lib.Batch(1, cap, device=self.device), cap
            self.approx_key = None
        hyp = np.asarray(hyp, dtype=DTYPE).reshape(1, 6)
        self.key = None
        if akey != getattr(self, "approx_key", None):
            if approx is None:
                self.batch.set_approx(0)
            else:
                self.batch.set_approx(approx[0], period=np.array([approx[1]], dtype=DTYPE) if approx[0] else None,
                                      xo=approx[2], p_xo=approx[3])
            self.approx_key = akey
        if data_key != self.data_key:
            info = self.batch.setup([ns], [nc], x_s[None], l_s[None], x_c[None] if nc else np.zeros((1, 0)), hyp,
                                    np.asarray(prior, dtype=DTYPE).reshape(1, 3), check_max=check_max)
            self.data_key = data_key
        else:
            self.batch.set_hypers(hyp)
            info = self.batch.setup_device(check_max=check_max)
        self.key, self.guarded = key, bool(check_max)
        self.status = int(info["status"][0])
        self.Z_mean = float(info["Z_mean"][0])
        self.Z_var = float(info["Z_var"][0])
        self.log_lh = float(info["log_lh"][0])
        self.l_c = np.array(info["l_c"][0, :nc])
        return self


class _PinnedPool(object):
    """Page-locked result buffers for the host API.  A device->host copy into pageable memory is
    staged by the driver at a fraction of PCIe speed, so results are written into pinned arrays;
    a buffer is handed out again only after the caller has dropped every reference to the array
    it was given (so two results never alias)."""

    def __init__(self, keep=6):
        self._bufs, self._keep = [], keep

    def take(self, n):
        import sys
        import torch
        for t, arr in self._bufs:
            if arr.shape[0] >= n and sys.getrefcount(arr) <= 3:      # only the pool (tuple + loop var) holds it
                return arr[:n]
        t = torch.empty(max(n, 1), dtype=torch.float64).pin_memory()
        arr = t.numpy()
        self._bufs.append((t, arr))
        if len(self._bufs) > self._keep:
            self._bufs.pop(0)
        return arr[:n]


_POOL = _PinnedPool()


class BQ(object):
    r"""Bayesian quadrature estimate of :math:`Z = \int \ell(x) N(x | \mu, \sigma^2) dx` with a GP
    over :math:`\log\ell` and a second GP over :math:`\exp(\log\ell)` (reference class docstring,
    bq.py:19-49).

    Parameters
    ----------
    x, l : 1-D arrays of sample locations and (strictly positive) likelihood values
    options : the six mandatory keyword options of :meth:`load_options`
    """

    def __init__(self, x, l, **options):
        self.x_s = np.array(x, dtype=DTYPE)
        self.l_s = np.array(l, dtype=DTYPE)
        # same validation order and messages as bq.py:63-70
        if (self.l_s <= 0).any():
            raise ValueError("l_s contains zero or negative values")
        if self.x_s.ndim > 1:
            raise ValueError("invalid number of dimensions for x")
        if self.l_s.ndim > 1:
            raise ValueError("invalid number of dimensions for l")
        if self.x_s.shape != self.l_s.shape:
            raise ValueError("shape mismatch for x and l")
        self.tl_s = np.log(self.l_s)
        self.ns = self.x_s.shape[0]

        self.load_options(**options)
        self.initialized = False
        self.gp_log_l = self.gp_l = None
        self.x_c = self.l_c = self.nc = None
        self.x_sc = self.l_sc = self.nsc = None
        self._approx_cache = None
        self._reset_device_state()

    def _reset_device_state(self):
        self._dev_model = None
        self._last_d2h_bytes = 0
        #: CUDA device index of this object's kernels (one process per GPU: LOCAL_RANK)
        self.device = int(os.environ.get("LOCAL_RANK", "0"))

    def load_options(self, kernel, n_candidate, candidate_thresh, x_mean, x_var, optim_method):
        """Same six mandatory options as the reference (bq.py:94-127)."""
        self.options = {
            "kernel": kernel,
            "n_candidate": int(n_candidate),
            "candidate_thresh": float(candidate_thresh),
            "x_mean": np.array([x_mean], dtype=DTYPE, order="F"),
            "x_cov": np.array([[x_var]], dtype=DTYPE, order="F"),
            "use_approx": not (kernel is GaussianKernel),
            "wrapped": kernel is PeriodicKernel,
            "optim_method": optim_method,
        }
        if self.options["use_approx"]:
            logger.debug("Using approximate solutions for non-Gaussian kernel")

    # ------------------------------------------------------------------ initialisation
    def init(self, params_tl, params_l):
        """Build the two GPs and draw the candidate points (bq.py:132-171)."""
        kernel = self.options["kernel"]
        self.gp_log_l = GP(kernel(*params_tl[:-1]), self.x_s, self.tl_s, s=params_tl[-1])
        self.gp_log_l.jitter = np.zeros(self.ns, dtype=DTYPE)
        self._choose_candidates(params_l)
        self.gp_l = GP(kernel(*params_l[:-1]), self.x_sc, self.l_sc, s=params_l[-1])
        self.gp_l.jitter = np.zeros(self.nsc, dtype=DTYPE)
        # the 1000-point approximation grid (bq.py:170-171) is only read by the trapezoid path and by pickling:
        # built on first access (properties below), so that init / add_observation do not pay for it every round
        self._approx_cache = None
        self._approx_spec = (self._approx_bound(-1), self._approx_bound(+1))     # as of init, like the reference's grid
        self.initialized = True

    def _choose_candidates(self, params_l=None):
        """Candidate draw and filtering on the host with the global numpy RNG, exactly the calls of
        bq.py:967-991; their values l_c = exp(gp_log_l.mean(x_c)) come from the device."""
        logger.debug("Choosing candidate points")
        if self.options["wrapped"]:
            xmin, xmax = -np.pi * self.gp_log_l.K.p, np.pi * self.gp_log_l.K.p
        else:
            xmin = self.x_s.min() - self.gp_log_l.K.w
            xmax = self.x_s.max() + self.gp_log_l.K.w
        xc = np.random.uniform(xmin, xmax, self.options["n_candidate"])
        util.filter_candidates(xc, self.x_s, self.options["candidate_thresh"])
        self.x_c = np.sort(xc[~np.isnan(xc)])
        self.nc = self.x_c.shape[0]
        if params_l is None:
            params_l = self.gp_l.params
        self.l_c = self._log_l_values(self.gp_log_l.params, np.asarray(params_l, dtype=DTYPE), check_max=False)
        self.x_sc = np.array(np.concatenate([self.x_s, self.x_c]))
        self.l_sc = np.array(np.concatenate([self.l_s, self.l_c]))
        self.nsc = self.ns + self.nc

    # ------------------------------------------------------------------ device model cache
    def _data_key(self):
        return (self.x_s.tobytes(), self.l_s.tobytes(), self.x_c.tobytes(), float(self.options["x_mean"][0]),
                float(self.options["x_cov"][0, 0]), self.options["candidate_thresh"], self.device)

    def _refresh_device(self, params_tl, params_l, check_max):
        """Device factors for (current data, the given parameters); returns the model whatever its setup status."""
        if self._dev_model is None or self._dev_model.device != self.device:
            if self._dev_model is not None:
                self._dev_model.close()
            self._dev_model = _DeviceModel(self.device)
        ptl, pl = np.asarray(params_tl, dtype=DTYPE), np.asarray(params_l, dtype=DTYPE)
        hyp = np.array([ptl[0], ptl[1], ptl[-1], pl[0], pl[1], pl[-1]], dtype=DTYPE)      # (h, w, s) of both GPs
        prior = (float(self.options["x_mean"][0]), float(self.options["x_cov"][0, 0]), self.options["candidate_thresh"])
        approx = None
        periodic = self.options["kernel"] is PeriodicKernel
        if periodic or self.options["use_approx"]:
            # generic device path (csrc/bq_score_generic.cu): periodic kernel and / or trapezoid integrals over the grid of
            # bq.py:167-171.  During init the candidates' values are needed before the grid exists (bq.py:985 comes
            # before :168): l_c only involves gp_log_l, so that pass runs with closed forms / without a grid.
            xo = p_xo = None
            if self.options["use_approx"] and (self.initialized or self.gp_l is not None):
                xo, p_xo = self._approx()
            approx = (1 if periodic else 0, (ptl[2], pl[2]) if periodic else (1.0, 1.0), xo, p_xo)
        return self._dev_model.refresh(self._data_key(), self.x_s, self.l_s, self.x_c, hyp, prior, check_max, approx)

    def _log_l_values(self, params_tl, params_l, check_max):
        """l_c = exp(gp_log_l.mean(x_c)) from the device (bq.py:985 / :942-950).  Only gp_log_l is involved, as in the
        reference: a gp_l Gram matrix that is not positive definite under the *current* gp_l parameters is not an
        error here (l_c is computed before K_l is factorised) -- it surfaces when the gp_l factors are used."""
        model = self._refresh_device(params_tl, params_l, check_max)
        if model.status not in (_lib.SETUP_OK, _lib.SETUP_KL_NOTPD):
            _raise_setup(model.status)
        return model.l_c

    def _device_model(self):
        """Device factors for the *current* state; rebuilt only when data or parameters changed
        (the counterpart of the `gp` package's memoised Kxx / Lxx / inv_Kxx_y)."""
        if not self.initialized and self.gp_l is None:
            raise RuntimeError("BQ object is not initialized: call init() first")
        model = self._refresh_device(self.gp_log_l.params, self.gp_l.params, check_max=False)
        if model.status != _lib.SETUP_OK:
            _raise_setup(model.status)
        return model

    def _invalidate_device(self):
        if self._dev_model is not None:
            self._dev_model.close()
        self._dev_model = None

    # ------------------------------------------------------------------ mean / variance of l
    def _predict(self, x):
        """(gp_l.mean(x), diag gp_log_l.cov(x)) for a vector of finite points in one device pass; None for other input, which
        the host GPs answer.  The Gaussian kernel with s_l = 0 in a tensor-core capacity class (ns <= 256) takes the
        scoring kernel's prediction mode; every other problem (the trapezoid path, the periodic kernel, a noisy gp_l, the
        512 class) takes the prediction kernel, which reads alpha_l = (K_l + s_l^2 I)^-1 l_sc from the setup."""
        x = np.ascontiguousarray(x, dtype=DTYPE)
        if x.ndim != 1 or not np.isfinite(x).all():
            return None
        batch = self._device_model().batch
        if self.options["use_approx"] or self.gp_l.get_param("s") != 0 or self.ns > 256:
            m, v = batch.predict_rows_host(x)
        else:
            m, v = batch.predict_host(x)
        return m[0], v[0]

    def l_mean(self, x):
        """Mean of the final approximation to l: the mean of the GP over exp(log l) (bq.py:177-200).  One device pass for a
        1-D vector of finite points whatever the kernel, s_l or number of observations (``_predict``); the host GPs answer
        other input."""
        pred = self._predict(x)
        return self.gp_l.mean(x) if pred is None else pred[0]

    def l_var(self, x):
        """Marginal variance of the final approximation (bq.py:202-231): v_log_l * m_l^2, negative values set to 0, with both
        factors from one device pass for a 1-D vector of finite points (``_predict``), from the host GPs otherwise."""
        pred = self._predict(x)
        if pred is None:
            v_log_l = np.diag(self.gp_log_l.cov(x)).copy()
            m_l = self.gp_l.mean(x)
        else:
            m_l, v_log_l = pred
        l_var = v_log_l * m_l ** 2
        l_var[l_var < 0] = 0
        return l_var

    # ------------------------------------------------------------------ Z
    def Z_mean(self):
        """E[Z] (bq.py:237-291; bq_c.Z_mean bq_c.pyx:157-213), computed by the setup kernel."""
        m_Z = self._device_model().Z_mean
        if m_Z <= 0:
            warnings.warn("m_Z = %s" % m_Z)          # bq_c.pyx:210-211
        return m_Z

    def Z_var(self):
        """V[Z] (bq.py:297-348; bq_c.Z_var bq_c.pyx:264-355), computed by the setup kernel."""
        V_Z = self._device_model().Z_var
        if V_Z <= 0:
            warnings.warn("V_Z = %s" % V_Z)          # bq_c.pyx:352-353
        return V_Z

    # ------------------------------------------------------------------ expected variance (the hot path)
    @staticmethod
    def _check_x_a(x_a, scan=True):
        """Input validation of bq.py:451-452.  With ``scan=False`` the NaN/inf scan is left to the
        device (status bit ST_XA_BAD), which costs nothing; the caller then raises the same
        ValueError from the flags."""
        if x_a is None:
            raise ValueError("invalid value for x_a: %s", x_a)       # bq.py:451-452
        x_a = np.ascontiguousarray(x_a, dtype=DTYPE)
        if x_a.ndim != 1:
            raise ValueError("x_a must be a 1-D array")
        if scan:
            BQ._raise_bad_x_a(x_a)
        return x_a

    @staticmethod
    def _raise_bad_x_a(x_a):
        bad = ~np.isfinite(x_a)
        if bad.any():
            raise ValueError("invalid value for x_a: %s", x_a[np.argmax(bad)])

    @staticmethod
    def _report(x_a, esm, em, status, where=""):
        """The reference's post-checks (bq.py:514-525) on a vector of results; ``where`` is appended to every message
        (BatchBQ names the problem there)."""
        if status is None:
            return
        bad = (status & _lib.ST_ESM_BAD) != 0
        if bad.any():
            i = int(np.argmax(bad))
            raise RuntimeError("invalid expected squared mean for x_a=%s: %s%s" % (x_a[[i]], esm[i], where))
        bad = (status & _lib.ST_EM_BAD) != 0
        if bad.any():
            i = int(np.argmax(bad))
            raise RuntimeError("invalid expected mean for x_a=%s: %s%s" % (x_a[[i]], None if em is None else em[i], where))
        for bit, name in ((_lib.ST_ESM_INF, "expected squared mean"), (_lib.ST_EM_INF, "expected mean")):
            idx = np.nonzero(status & bit)[0]
            for i in idx[:5]:
                logger.warning("%s for x_a=%s is infinity!%s", name, x_a[[i]], where)
            if idx.size > 5:
                logger.warning("%s is infinity for %d more points%s", name, idx.size - 5, where)

    def _score(self, x_a, want_em=True):
        x_a = self._check_x_a(x_a)
        model = self._device_model()
        esm, em, st = model.batch.score_host(x_a, want_em=want_em, want_status=True)
        esm, st = esm[0], st[0]
        em = em[0] if want_em else None
        self._last_d2h_bytes = esm.nbytes + st.nbytes + (em.nbytes if want_em else 0)
        self._report(x_a, esm, em, st)
        return esm, em, st

    def expected_Z_var(self, x_a):
        r"""E[V(Z) | l_s, l_a] = E[Z|l_s]^2 + V(Z|l_s) - E[ E[Z|l_s,l_a]^2 ] for every point of `x_a`
        (bq.py:354-377).  One fused device pass; only the result vector crosses PCIe."""
        x_a = self._check_x_a(x_a, scan=False)
        model = self._device_model()
        if model.Z_mean <= 0:
            warnings.warn("m_Z = %s" % model.Z_mean)
        if model.Z_var <= 0:
            warnings.warn("V_Z = %s" % model.Z_var)
        ev, flags = model.batch.expected_var_host(x_a, out=_POOL.take(x_a.shape[0]))
        self._last_d2h_bytes = ev.nbytes + 4
        if flags & _lib.ST_XA_BAD:
            self._raise_bad_x_a(x_a)            # bq.py:451-452
        if flags & ~(_lib.ST_SHORTCUT | _lib.ST_NOTPD):
            self._score(x_a, want_em=True)      # slow path: fetch per-point status, raise / warn like bq.py:514-525
        return ev

    def expected_squared_mean(self, x_a):
        """E[ E[Z|l_s,l_a]^2 ] for every point of `x_a` (bq.py:379-402)."""
        return self._score(x_a, want_em=False)[0]

    def expected_mean(self, x_a):
        """E[ E[Z|l_s,l_a] ] for every point of `x_a` (bq.py:404-423)."""
        return self._score(x_a)[1]

    def expected_squared_mean_and_mean(self, x_a):
        """[na, 2] array of (expected squared mean, expected mean) (bq.py:425-445)."""
        esm, em, _ = self._score(x_a)
        return np.stack([esm, em], axis=1)

    def _esm_and_em(self, x_a):
        """Single-point form kept for callers of the reference's private helper (bq.py:447-527)."""
        if x_a is None or np.isnan(x_a) or np.isinf(x_a):
            raise ValueError("invalid value for x_a: %s", x_a)
        esm, em, _ = self._score(np.asarray(x_a, dtype=DTYPE).reshape(1))
        return esm[0], em[0]

    # ------------------------------------------------------------------ hyper-parameters (host)
    def _make_llh_params(self, params):
        """Joint log marginal likelihood of both GPs as a function of the parameter vector
        (bq.py:533-552); invalid parameters map to -inf.

        The reference evaluates it as _set_gp_log_l_params (l_c refreshed, "GP mean is too large" guard) ->
        _set_gp_l_params -> gp_log_l.log_lh + gp_l.log_lh.  Here ONE run of the setup kernel on the object's
        resident device buffers (only the six hyper-parameters are uploaded) yields l_c, the guard and both log
        likelihoods; the host GP objects are left in exactly the state the reference's sequence leaves them in."""
        nparam = len(params)

        def f(x):
            if x is None or np.isnan(x).any():
                return -np.inf
            new_tl = dict(zip(params, x[:nparam]))
            new_l = dict(zip(params, x[nparam:]))
            try:
                for p, v in new_tl.items():                  # bq.py:934-936 (ValueError from the first invalid value)
                    self.gp_log_l.set_param(p, v)
            except ValueError:
                return -np.inf
            self.gp_log_l.jitter.fill(0)
            names = list(self.gp_l.K.names) + ["s"]
            trial_l, l_ok = self.gp_l.params, True
            for p, v in new_l.items():                       # would gp_l.set_param accept every value?  (gp.py setters)
                l_ok = l_ok and p in names and ((v >= 0) if p == "s" else (v > 0))
                if l_ok:
                    trial_l[names.index(p)] = v
            # one device pass under (new gp_log_l parameters, the gp_l parameters the reference would have at log_lh time)
            model = self._refresh_device(self.gp_log_l.params, trial_l if l_ok else self.gp_l.params, check_max=True)
            if model.status not in (_lib.SETUP_OK, _lib.SETUP_KL_NOTPD):
                return -np.inf                               # LinAlgError of bq.py:945-947 / gp_log_l.Kxx: gp_l untouched
            self._retarget_gp_l(model.l_c)                   # bq.py:949-957
            try:
                self._set_gp_l_params(new_l)                 # bq.py:959-965
            except ValueError:
                return -np.inf
            if model.status != _lib.SETUP_OK:
                return -np.inf                               # gp_l.Kxx not positive definite: gp_l.log_lh is -inf
            return model.log_lh
        return f

    def _current_params(self, params):
        p0_tl = [self.gp_log_l.get_param(p) for p in params]
        p0_l = [self.gp_l.get_param(p) for p in params]
        return np.array(p0_tl + p0_l)

    def fit_hypers(self, params):
        """Maximise the joint marginal likelihood over the named parameters (bq.py:554-562)."""
        f = self._make_llh_params(params)
        p0 = util.find_good_parameters(f, self._current_params(params), self.options["optim_method"])
        if p0 is None:
            raise RuntimeError("couldn't find good parameters")

    def sample_hypers(self, params, n=1, nburn=10):
        """Slice-sample hyper-parameters of both GPs (bq.py:565-598)."""
        nparam = len(params)
        window = 2 * nparam
        p0 = self._current_params(params)
        f = self._make_llh_params(params)
        if f(p0) < MIN:
            pn = util.find_good_parameters(f, p0, self.options["optim_method"])
            if pn is None:
                raise RuntimeError("couldn't find good starting parameters")
            p0 = pn
        hypers = util.slice_sample(f, nburn + n, window, p0, nburn=nburn, freq=1)
        return hypers[:, :nparam], hypers[:, nparam:]

    # ------------------------------------------------------------------ active sampling
    def marginalize(self, funs, n, params):
        """Approximate marginals of arbitrary callables over sampled hyper-parameters
        (bq.py:604-657): generic host loop, one device setup per sample."""
        state = deepcopy(self.__getstate__())
        values = []
        for fun in funs:
            value = fun()                     # evaluated once just for the output shape (bq.py:626-633)
            try:
                m = value.shape
            except AttributeError:
                values.append(np.empty(n))
            else:
                values.append(np.empty((n,) + m))
        hypers_tl, hypers_l = self.sample_hypers(params, n=n, nburn=1)
        for i in range(n):
            params_tl = dict(zip(params, hypers_tl[i]))
            params_l = dict(zip(params, hypers_l[i]))
            self._set_gp_log_l_params(params_tl)
            self._set_gp_l_params(params_l)
            for j, fun in enumerate(funs):
                try:
                    values[j][i] = fun()
                except:
                    logger.error("error with parameters %s and %s", params_tl, params_l)
                    raise
        self.__setstate__(state)
        return values

    #: score buffer of the chunked marginal loss: [chunk, na] doubles of at most this many bytes (stays L2-resident on a B200)
    LOSS_CHUNK_BYTES = 64 << 20

    def marginal_loss(self, x_a, hypers_tl, hypers_l, params, reduce="mean"):
        """Marginal loss of choose_next — the mean over hyper-parameter samples of
        ``-expected_squared_mean(x_a)`` (bq.py:660-662) — for ALL samples in one device batch.
        Each sample goes through the semantics of ``_set_gp_log_l_params`` / ``_set_gp_l_params``
        (bq.py:933-965: l_c recomputed, "GP mean is too large" guard).

        The samples are scored chunk by chunk through one [chunk, na] buffer and accumulated in sample order
        (``bqb_sum_neg_accum_device``): the additions of ``values[0].mean(axis=0)`` in the same order, without the
        [n, na] matrix (819 MB at 1024 samples x 10^5 points).  ``reduce="sum"`` returns the sum over the samples
        instead of the mean (what a rank contributes when the samples are sharded across GPUs)."""
        import torch
        x_a = self._check_x_a(x_a)
        n = len(hypers_tl)
        base_tl, base_l = self.gp_log_l.params, self.gp_l.params
        names = list(self.gp_log_l.K.names) + ["s"]
        hyp = np.empty((n, 6))
        periodic = self.options["kernel"] is PeriodicKernel
        period = np.ones((n, 2))
        for i in range(n):
            ptl, pl = base_tl.copy(), base_l.copy()
            for name, v in zip(params, hypers_tl[i]):
                ptl[names.index(name)] = v
            for name, v in zip(params, hypers_l[i]):
                pl[names.index(name)] = v
            hyp[i] = [ptl[0], ptl[1], ptl[-1], pl[0], pl[1], pl[-1]]
            if periodic:
                period[i] = [ptl[2], pl[2]]
        batch = _lib.Batch(n, self.ns, device=self.device)
        try:
            if periodic or self.options["use_approx"]:       # generic device path, the grid of bq.py:167-171 for every sample
                xo, p_xo = self._approx() if self.options["use_approx"] else (None, None)
                batch.set_approx(1 if periodic else 0, period=period if periodic else None, xo=xo, p_xo=p_xo)
            prior = np.tile([float(self.options["x_mean"][0]), float(self.options["x_cov"][0, 0]),
                             self.options["candidate_thresh"]], (n, 1))
            info = batch.setup(np.full(n, self.ns), np.full(n, self.nc), np.tile(self.x_s, (n, 1)),
                               np.tile(self.l_s, (n, 1)), np.tile(self.x_c, (n, 1)), hyp, prior, check_max=True)
            bad = np.nonzero(info["status"])[0]
            if bad.size:
                logger.error("error with parameters %s", hyp[bad[0]])
                _raise_setup(info["status"][bad[0]])
            dev = torch.device("cuda", self.device)
            x_d = torch.from_numpy(x_a).to(dev)
            na = x_a.shape[0]
            # points in arbitrary order defeat the kernels' band skipping (DESIGN.md 4.1): score them in ascending order
            perm = None
            if na >= 8192 and self.ns > 64 and not _looks_sorted(x_a):      # (pays from the ns <= 128 class up)
                x_d, perm = torch.sort(x_d)
            loss = torch.zeros(na, dtype=torch.float64, device=dev)
            chunk = int(max(1, min(n, self.LOSS_CHUNK_BYTES // max(8 * na, 1))))
            for c in (148, 74, 37):           # whole shares of the 148 SMs per instance: the launches fill exactly one wave
                if n > c and chunk >= c:
                    chunk = c
                    break
            esm = torch.empty(chunk, max(na, 1), dtype=torch.float64, device=dev)
            flags = torch.zeros(chunk, dtype=torch.int32, device=dev)
            seen = torch.zeros(chunk, dtype=torch.int32, device=dev)          # OR of the status bits, slot-wise over the chunks
            for i0 in range(0, n, chunk):
                cnt = min(chunk, n - i0)
                batch.score_device_range(i0, cnt, x_d, esm, None, None, flags)
                batch.sum_neg_accum_device(esm, cnt, loss)
                seen[:cnt] |= flags[:cnt]
            if reduce == "mean":
                loss = loss / n                                                # bq.py:662
            elif reduce != "sum":
                raise ValueError("reduce must be 'mean' or 'sum'")
            if perm is not None:
                loss = torch.empty_like(loss).scatter_(0, perm, loss)         # back to the caller's order
            if int(np.bitwise_or.reduce(seen.cpu().numpy())) & (_lib.ST_ESM_BAD | _lib.ST_EM_BAD):
                raise RuntimeError("invalid expected squared mean under a sampled hyper-parameter set")
            return loss, batch
        except Exception:
            batch.close()
            raise

    def log_lh_batch(self, hypers_tl, hypers_l, params):
        """Joint log marginal likelihood ``gp_log_l.log_lh + gp_l.log_lh`` (bq.py:546) of MANY hyper-parameter
        proposals in one device batch (SURVEY §8(f).1): entry i is what ``_make_llh_params(params)`` would return
        for ``concatenate([hypers_tl[i], hypers_l[i]])`` — including -inf for invalid values, a non-PD Gram matrix
        or the "GP mean is too large" guard (bq.py:536-548) — without touching this object's state."""
        hypers_tl, hypers_l = np.atleast_2d(hypers_tl), np.atleast_2d(hypers_l)
        n = hypers_tl.shape[0]
        names = list(self.gp_log_l.K.names) + ["s"]
        hyp = np.empty((n, 6))
        hyp[:, :3], hyp[:, 3:] = self.gp_log_l.params, self.gp_l.params
        for j, name in enumerate(params):
            hyp[:, names.index(name)] = hypers_tl[:, j]
            hyp[:, 3 + names.index(name)] = hypers_l[:, j]
        ok = np.isfinite(hyp).all(axis=1) & (hyp[:, [0, 1, 3, 4]] > 0).all(axis=1) & (hyp[:, [2, 5]] >= 0).all(axis=1)
        out = np.full(n, -np.inf)
        if ok.any():
            m = int(ok.sum())
            batch = _lib.Batch(m, self.ns, device=self.device)
            try:
                prior = np.tile([float(self.options["x_mean"][0]), float(self.options["x_cov"][0, 0]),
                                 self.options["candidate_thresh"]], (m, 1))
                info = batch.setup(np.full(m, self.ns), np.full(m, self.nc), np.tile(self.x_s, (m, 1)),
                                   np.tile(self.l_s, (m, 1)), np.tile(self.x_c, (m, 1)), hyp[ok], prior, check_max=True)
            finally:
                batch.close()
            out[ok] = np.where(info["status"] == _lib.SETUP_OK, info["log_lh"], -np.inf)
        return out

    def choose_next(self, x_a, n, params, plot=False, deterministic=False):
        """Pick the next query location: argmin over `x_a` of the marginal negative expected squared
        mean (bq.py:659-681).  Like the reference, ties within ``np.isclose`` of the minimum are
        broken with ``np.random.choice``; ``deterministic=True`` returns the first minimiser instead."""
        x_a = self._check_x_a(x_a)
        # the reference deep-copies the whole pickled state around the sampling (bq.py:622, :655); all that the sampler
        # can change are the two parameter vectors, the candidate values they imply and the jitter records
        saved = (self.gp_log_l.params, self.gp_l.params, self.l_c, self.gp_log_l.jitter.copy(), self.gp_l.jitter.copy())
        try:
            hypers_tl, hypers_l = self.sample_hypers(params, n=n, nburn=1)
        finally:
            self.gp_log_l.params, self.gp_l.params = saved[0], saved[1]
            self._retarget_gp_l(saved[2])
            self.gp_log_l.jitter[:], self.gp_l.jitter[:] = saved[3], saved[4]
        loss_d, batch = self.marginal_loss(x_a, hypers_tl, hypers_l, params)
        try:
            if deterministic:
                _, choice = batch.argmin_device(loss_d)
                loss = None
            else:
                loss = loss_d.cpu().numpy()
                best = np.min(loss)
                close = np.nonzero(np.isclose(loss, best))[0]
                choice = np.random.choice(close)
        finally:
            batch.close()
        best = x_a[choice]
        if plot:
            self._plot_choice(x_a, loss if loss is not None else loss_d.cpu().numpy(), best)
        return best

    def add_observation(self, x_a, l_a):
        """Add (or average in) an observation and re-initialise (bq.py:683-701)."""
        diffs = np.abs(x_a - self.x_s)
        if diffs.min() < self.options["candidate_thresh"]:
            c = diffs.argmin()
            logger.debug("x_a=%s is close to x_s=%s, averaging them", x_a, self.x_s[c])
            self.x_s[c] = (self.x_s[c] + x_a) / 2.
            self.l_s[c] = (self.l_s[c] + l_a) / 2.
            self.tl_s[c] = np.log(float(self.l_s[c]))
        else:
            self.x_s = np.append(self.x_s, float(x_a))
            self.l_s = np.append(self.l_s, float(l_a))
            self.tl_s = np.append(self.tl_s, np.log(float(l_a)))
            self.ns += 1
        self.init(self.gp_log_l.params, self.gp_l.params)

    # ------------------------------------------------------------------ parameter setters
    def _retarget_gp_l(self, l_c):
        """bq.py:949-957: new candidate values, gp_l retargeted at (x_sc, l_sc), jitter cleared."""
        self.l_c = l_c
        self.l_sc = np.array(np.concatenate([self.l_s, self.l_c]))
        self.gp_l.x = self.x_sc
        self.gp_l.y = self.l_sc
        self.gp_l.jitter.fill(0)

    def _set_gp_log_l_params(self, params):
        """bq.py:933-957: set parameters of the GP over log l, recompute the candidate values
        l_c = exp(mean(x_c)) (on device, with the "GP mean is too large" guard) and retarget gp_l."""
        for p, v in params.items():
            self.gp_log_l.set_param(p, v)
        self.gp_log_l.jitter.fill(0)
        self._retarget_gp_l(self._log_l_values(self.gp_log_l.params, self.gp_l.params, check_max=True))

    def _set_gp_l_params(self, params):
        """bq.py:959-965."""
        for p, v in params.items():
            self.gp_l.set_param(p, v)
        self.gp_l.jitter.fill(0)

    # ------------------------------------------------------------------ approximation grid (state only)
    def _approx(self):
        if not self.initialized and self.gp_l is None:
            return None, None
        if self._approx_cache is None:
            x = np.linspace(self._approx_spec[0], self._approx_spec[1], 1000)
            self._approx_cache = (x, self._make_approx_px(x))
        return self._approx_cache

    def _approx_bound(self, side):
        if self.options["wrapped"]:
            return side * np.pi * self.gp_log_l.K.p
        return (self.x_sc.min() - self.gp_log_l.K.w) if side < 0 else (self.x_sc.max() + self.gp_log_l.K.w)

    _approx_x = property(lambda self: self._approx()[0])
    _approx_px = property(lambda self: self._approx()[1])

    def _make_approx_x(self, xmin=None, xmax=None, n=1000):
        """bq.py:993-1006 (kept because the grid is part of the pickled state)."""
        if xmin is None:
            xmin = self._approx_bound(-1)
        if xmax is None:
            xmax = self._approx_bound(+1)
        return np.linspace(xmin, xmax, n)

    def _make_approx_px(self, x=None):
        """Prior density on the approximation grid (bq.py:1008-1026, bq_c.p_x_gaussian)."""
        if x is None:
            x = self._approx_x
        mu = float(self.options["x_mean"][0])
        var = float(self.options["x_cov"][0, 0])
        if self.options["wrapped"]:
            return _vonmises_px(x, mu, var)
        return np.exp(-0.5 * (np.log(2 * np.pi) + np.log(var) + (x - mu) ** 2 / var))

    # ------------------------------------------------------------------ plotting (host, optional matplotlib)
    @staticmethod
    def _plt():
        import matplotlib.pyplot as plt
        return plt

    def plot_gp_log_l(self, ax, f_l=None, xmin=None, xmax=None):
        x = self._make_approx_x(xmin=xmin, xmax=xmax, n=1000)
        if f_l is not None:
            ax.plot(x, np.log(f_l(x)), "k-", lw=2)
        self.gp_log_l.plot(ax, xlim=[x.min(), x.max()], color="r")
        ax.plot(self.x_c, np.log(self.l_c), "bs", markersize=4, label=r"$m_{\log\ell}(x_c)$")
        ax.set_title(r"GP over $\log\ell$")
        util.set_scientific(ax, -5, 4)

    def plot_gp_l(self, ax, f_l=None, xmin=None, xmax=None):
        x = self._make_approx_x(xmin=xmin, xmax=xmax, n=1000)
        if f_l is not None:
            ax.plot(x, f_l(x), "k-", lw=2)
        self.gp_l.plot(ax, xlim=[x.min(), x.max()], color="r")
        ax.plot(self.x_c, self.l_c, "bs", markersize=4, label=r"$\exp(m_{\log\ell}(x_c))$")
        ax.set_title(r"GP over $\exp(\log\ell)$")
        util.set_scientific(ax, -5, 4)

    def plot_l(self, ax, f_l=None, xmin=None, xmax=None, legend=True):
        x = self._make_approx_x(xmin=xmin, xmax=xmax, n=1000)
        if f_l is not None:
            ax.plot(x, f_l(x), "k-", lw=2, label=r"$\ell(x)$")
        l_mean = self.l_mean(x)
        l_sd = np.sqrt(self.l_var(x))
        ax.fill_between(x, l_mean - l_sd, l_mean + l_sd, color="r", alpha=0.2)
        ax.plot(x, l_mean, "r-", lw=2, label="final approx")
        ax.plot(self.x_s, self.l_s, "ro", markersize=5, label=r"$\ell(x_s)$")
        ax.plot(self.x_c, self.l_c, "bs", markersize=4, label=r"$\exp(m_{\log\ell}(x_c))$")
        ax.set_title("Final Approximation")
        ax.set_xlim(x.min(), x.max())
        util.set_scientific(ax, -5, 4)
        if legend:
            ax.legend(loc=0, fontsize=10)

    def plot_expected_squared_mean(self, ax, xmin=None, xmax=None):
        x_a = self._make_approx_x(xmin=xmin, xmax=xmax, n=1000)
        ax.plot(x_a, self.expected_squared_mean(x_a), label=r"$E[\mathrm{m}(Z)^2]$", color="k", lw=2)
        ax.set_xlim(x_a.min(), x_a.max())
        util.hlines(ax, self.Z_mean() ** 2, color="#00FF00", lw=2, label=r"$\mathrm{m}(Z)^2$")
        util.vlines(ax, self.x_sc, color="k", linestyle="--", alpha=0.5)
        util.set_scientific(ax, -5, 4)
        ax.legend(loc=0, fontsize=10)
        ax.set_title(r"Expected squared mean of $Z$")

    def plot_expected_variance(self, ax, xmin=None, xmax=None):
        x_a = self._make_approx_x(xmin=xmin, xmax=xmax, n=1000)
        ax.plot(x_a, self.expected_Z_var(x_a), label=r"$E[\mathrm{Var}(Z)]$", color="k", lw=2)
        ax.set_xlim(x_a.min(), x_a.max())
        util.hlines(ax, self.Z_var(), color="#00FF00", lw=2, label=r"$\mathrm{Var}(Z)$")
        util.vlines(ax, self.x_sc, color="k", linestyle="--", alpha=0.5)
        util.set_scientific(ax, -5, 4)
        ax.legend(loc=0, fontsize=10)
        ax.set_title(r"Expected variance of $Z$")

    def plot(self, f_l=None, xmin=None, xmax=None):
        fig, axes = self._plt().subplots(1, 3)
        self.plot_gp_log_l(axes[0], f_l=f_l, xmin=xmin, xmax=xmax)
        self.plot_gp_l(axes[1], f_l=f_l, xmin=xmin, xmax=xmax)
        self.plot_l(axes[2], f_l=f_l, xmin=xmin, xmax=xmax)
        ymins, ymaxs = zip(*[ax.get_ylim() for ax in axes[1:]])
        for ax in axes[1:]:
            ax.set_ylim(min(ymins), max(ymaxs))
        fig.set_figwidth(14)
        fig.set_figheight(3.5)
        return fig, axes

    def _plot_choice(self, x_a, loss, best):
        fig, (ax1, ax2) = self._plt().subplots(1, 2, sharex=True)
        self.plot_l(ax1, xmin=x_a.min(), xmax=x_a.max())
        util.vlines(ax1, best, color="g", linestyle="--", lw=2)
        ax2.plot(x_a, loss, "k-", lw=2)
        util.vlines(ax2, best, color="g", linestyle="--", lw=2)
        ax2.set_title("Negative expected sq. mean")
        fig.set_figwidth(10)
        fig.set_figheight(3.5)

    # ------------------------------------------------------------------ pickling / copying
    _STATE_KEYS = ("gp_log_l", "gp_log_l_jitter", "gp_l", "gp_l_jitter", "_approx_x", "_approx_px")

    def __getstate__(self):
        """Same keys as the reference (bq.py:840-860, pinned by its test_getstate); device buffers
        are caches rebuilt from this state and are never pickled."""
        state = {"x_s": self.x_s, "l_s": self.l_s, "tl_s": self.tl_s, "options": self.options,
                 "initialized": self.initialized}
        if self.initialized:
            state.update(gp_log_l=self.gp_log_l, gp_log_l_jitter=self.gp_log_l.jitter, gp_l=self.gp_l,
                         gp_l_jitter=self.gp_l.jitter, _approx_x=self._approx_x, _approx_px=self._approx_px)
        return state

    def __setstate__(self, state):
        """bq.py:862-902."""
        self.x_s, self.l_s, self.tl_s = state["x_s"], state["l_s"], state["tl_s"]
        self.ns = self.x_s.shape[0]
        self.options = state["options"]
        self.initialized = state["initialized"]
        if not hasattr(self, "_dev_model"):
            self._reset_device_state()
        if self.initialized:
            self.gp_log_l = state["gp_log_l"]
            self.gp_log_l.jitter = state["gp_log_l_jitter"]
            self.gp_l = state["gp_l"]
            self.gp_l.jitter = state["gp_l_jitter"]
            self.x_sc, self.l_sc = self.gp_l._x, self.gp_l._y
            self.nsc = self.x_sc.shape[0]
            self.x_c, self.l_c = self.x_sc[self.ns:], self.l_sc[self.ns:]
            self.nc = self.nsc - self.ns
            self._approx_cache = (state["_approx_x"], state["_approx_px"])
        else:
            self.gp_log_l = self.gp_l = None
            self.x_c = self.l_c = self.nc = None
            self.x_sc = self.l_sc = self.nsc = None
            self._approx_cache = None

    def __copy__(self):
        new = type(self).__new__(type(self))
        new.__setstate__(self.__getstate__())
        return new

    def __deepcopy__(self, memo):
        new = type(self).__new__(type(self))
        new.__setstate__(deepcopy(self.__getstate__(), memo))
        return new

    def copy(self, deep=True):
        return deepcopy(self) if deep else copy(self)
