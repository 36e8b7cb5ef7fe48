"""``BatchBQ`` — P independent 1-D BQ problems advanced in lock-step on one GPU (BASELINE config C5:
a batch of problems doing rounds of expected-variance active sampling, problems sharded across
GPUs with no collective; SURVEY.md §8(e), §8(f).2).

Per problem the semantics are those of the reference's ``BQ`` object under the batch's hyper-parameters:
``init`` draws and filters candidates (bq.py:967-991), a round scores a query grid with
``expected_squared_mean`` (bq.py:379-402), picks the first minimiser of ``-esm`` (bq.py:660-663,
deterministic mode), and ``add_observation`` merges or appends the new point and re-initialises
(bq.py:683-701).  Differences forced by batching, both documented in SURVEY appendix A.4: every
problem has its own ``RandomState(seed + p)`` candidate stream (the reference uses one global
RNG), and device arrays are padded to the batch's largest ``ns`` / ``nc``.

``choose_next(x_a, n=...)`` marginalises over hyper-parameter samples like the reference's ``BQ.choose_next``
(bq.py:659-681): ``sample_hypers`` slice-samples every problem's chain with one batched log-density evaluation per
step (``log_lh``), and ``marginal_loss`` scores the P x S (problem, sample) instances in chunks of whole problems.  Chain p
draws from its own counter-based stream keyed by the pair (seed, p) (the reference's single global libc ``rand`` stream
cannot be split per problem; SURVEY appendix A.4 documents the same choice for the candidate streams).

``kernel=PeriodicKernel`` runs every problem with the periodic kernel, as ``BQ(kernel=PeriodicKernel)`` does: the
parameters of a GP are (h, w, p, s), candidates are drawn on [-pi p_tl, pi p_tl] (bq.py:217-218), and the integrals are
trapezoid sums over the 1000-point grid of that range with the von Mises prior density (``BQ._approx``), built at
``init`` from the p_tl of that moment.

All per-problem bookkeeping is numpy-vectorised over the batch; scoring, the per-problem argmin
and the model setup run on the device through the C-ABI.
"""
import logging
import time

import numpy as np

from . import _lib
from . import util
from .bq import _SETUP_ERRORS, _vonmises_px
from .gp import GaussianKernel, PeriodicKernel

logger = logging.getLogger("bayesian_quadrature")
_NAMES = ("h", "w", "s")                     # GaussianKernel parameters, then the noise: columns of one GP's (h, w, s)
_NAMES_PERIODIC = ("h", "w", "p", "s")       # PeriodicKernel parameters, then the noise (BQ.init's params_tl / params_l)
# columns (of gp_log_l, of gp_l) of a parameter in a row of hyper-parameters: hyp [6], then for the periodic kernel period [2]
_COLS = {"h": (0, 3), "w": (1, 4), "s": (2, 5), "p": (6, 7)}
N_GRID = 1000                                # points of the approximation grid (bq.py:167-171)


def filter_candidates_batch(x_c, x_s, ns, thresh):
    """Vectorised ``bq_c.filter_candidates`` (bq_c.pyx:601-650) over a batch: x_c [P, m] is modified
    in place (NaN = removed), x_s [P, cap] holds ns[p] valid observations per row."""
    P, m = x_c.shape
    xt = np.ascontiguousarray(x_c.T)         # [m, P]: contiguous per-candidate vectors
    changed = True
    with np.errstate(invalid="ignore"):
        while changed:                       # the reference repeats the pair sweep while anything merged
            changed = False
            for i in range(m):
                for j in range(i + 1, m):
                    hit = np.abs(xt[i] - xt[j]) < thresh          # NaN (removed) compares False
                    if hit.any():
                        xt[i] = np.where(hit, (xt[i] + xt[j]) / 2.0, xt[i])
                        xt[j] = np.where(hit, np.nan, xt[j])
                        changed = True
    x_c[:] = xt.T
    # drop candidates closer than thresh to an observation: the nearest observation is one of the two
    # neighbours in sorted order, found with a vectorised binary search (same |x_c - x_s| < thresh test)
    cap = x_s.shape[1]
    valid = np.arange(cap)[None, :] < ns[:, None]
    xs = np.sort(np.where(valid, x_s, np.inf), axis=1)
    xs = np.concatenate([np.full((P, 1), -np.inf), xs, np.full((P, 1), np.inf)], axis=1)    # sentinels at both ends
    rows = np.arange(P)
    steps = int(np.ceil(np.log2(cap + 2))) + 1
    for i in range(m):
        q = x_c[:, i]
        lo = np.zeros(P, dtype=np.int64)                 # invariant: xs[lo] < q <= xs[hi] (NaN q: comparisons False)
        hi = np.full(P, cap + 1, dtype=np.int64)
        for _ in range(steps):
            mid = (lo + hi) >> 1
            go = xs[rows, mid] < q
            lo = np.where(go, mid, lo)
            hi = np.where(go, hi, mid)
        with np.errstate(invalid="ignore"):
            close = (np.abs(q - xs[rows, lo]) < thresh) | (np.abs(q - xs[rows, hi]) < thresh)
        x_c[close, i] = np.nan


class BatchBQ(object):
    def __init__(self, x_s, l_s, params_tl, params_l, n_candidate, candidate_thresh, x_mean, x_var, seed=0,
                 device=0, ns_reserve=0, device_resident=False, kernel=GaussianKernel):
        """x_s, l_s: [P, ns0] initial observations; params_*: (h, w, s) shared by all problems or [P, 3];
        x_mean / x_var scalars or [P].  ``ns_reserve`` extra observation slots are pre-allocated.

        ``kernel`` is GaussianKernel or PeriodicKernel; with PeriodicKernel params_* are (h, w, p, s) or [P, 4], the
        periods are kept in ``self.period`` [P, 2] (p of gp_log_l, of gp_l) next to ``self.hyp`` [P, 6], and x_mean /
        x_var are the mean and the inverse concentration of the von Mises prior.

        ``device_resident=True`` keeps the observations, the candidate generators (one MT19937 stream per problem,
        bit-identical to ``np.random.RandomState(seed + p)``) and the candidate filter on the GPU: a round then moves
        only the chosen points and their likelihood values across PCIe (SURVEY.md §8(f).2).  Both modes produce the
        same candidates, choices and Z estimates (tests/test_gpu_bq_api.py)."""
        x_s, l_s = np.asarray(x_s, dtype=np.float64), np.asarray(l_s, dtype=np.float64)
        if x_s.ndim != 2 or x_s.shape != l_s.shape:
            raise ValueError("x_s and l_s must be [P, ns] arrays of the same shape")
        if (l_s <= 0).any():
            raise ValueError("l_s contains zero or negative values")
        self.P, ns0 = x_s.shape
        self.cap = ns0 + int(ns_reserve)
        self.x_s = np.zeros((self.P, self.cap)); self.x_s[:, :ns0] = x_s
        self.l_s = np.ones((self.P, self.cap)); self.l_s[:, :ns0] = l_s
        self.ns = np.full(self.P, ns0, dtype=np.int32)
        bc = lambda v, k: np.ascontiguousarray(np.broadcast_to(np.asarray(v, dtype=np.float64), (self.P, k)))
        if kernel not in (GaussianKernel, PeriodicKernel):
            raise ValueError("kernel must be GaussianKernel or PeriodicKernel")
        self.periodic = kernel is PeriodicKernel
        self._names = _NAMES_PERIODIC if self.periodic else _NAMES
        if self.periodic:
            ptl, pl = bc(params_tl, 4), bc(params_l, 4)
            self.hyp = np.ascontiguousarray(np.concatenate([ptl[:, [0, 1, 3]], pl[:, [0, 1, 3]]], axis=1))
            self.period = np.ascontiguousarray(np.stack([ptl[:, 2], pl[:, 2]], axis=1))
        else:
            self.hyp = np.concatenate([bc(params_tl, 3), bc(params_l, 3)], axis=1)
        self.prior = np.stack([bc(x_mean, 1)[:, 0], bc(x_var, 1)[:, 0], np.full(self.P, float(candidate_thresh))], axis=1)
        self.n_candidate, self.thresh = int(n_candidate), float(candidate_thresh)
        if self.n_candidate > _lib.NC_MAX:
            raise NotImplementedError("n_candidate > %d" % _lib.NC_MAX)
        self.device_resident = bool(device_resident)
        self.seed = int(seed)
        self.rngs = None if self.device_resident else [np.random.RandomState(seed + p) for p in range(self.P)]
        self._ns_max = ns0                                 # upper bound of ns over the problems (device mode)
        # capacity class chosen for ns0 + ns_reserve from the start (both modes, so that they run the same kernels): a
        # batch that is known to grow does not migrate to the next class after the first appended observation
        self._class_hint = min(self.cap, 512)
        self.device = int(device)
        self.batch = None
        self.x_c = np.zeros((self.P, _lib.NC_MAX))
        self.nc = np.zeros(self.P, dtype=np.int32)
        self.init()

    def close(self):
        if self.batch is not None:
            self.batch.close()
            self.batch = None
        for b in getattr(self, "_sample_batches", {}).values():
            b.close()
        self._sample_batches = {}

    # ---------------------------------------------------------------- bq.py:132-171 / :967-991 per problem
    def _check_info(self, info):
        bad = np.nonzero(info["status"])[0]
        if bad.size:
            raise np.linalg.LinAlgError("problem %d failed device setup with status %d" % (bad[0], info["status"][bad[0]]))
        self.info = info
        return info

    def _init_device(self):
        """Device-resident (re-)initialisation: candidates are drawn, filtered and sorted on the GPU."""
        if self.batch is None:                             # first call: upload the observations, seed the generators
            cap_class = _lib.load().bqb_ns_capacity(max(int(self._ns_max), self._class_hint))
            if cap_class < 0:
                raise NotImplementedError("more than 512 observations per problem")
            self.batch = _lib.Batch(self.P, cap_class, device=self.device)
            self._cap_class = cap_class
            stride = min(self.cap, cap_class)
            self.batch.stage(self.ns, self.x_s[:, :stride], self.l_s[:, :stride], self.hyp, self.prior)
            self.batch.seed_candidates((self.seed + np.arange(self.P)) & 0xffffffff)
        if self.periodic:
            self._apply_approx()
            self.batch.draw_candidates_wrapped(self.n_candidate)
        else:
            self.batch.draw_candidates(self.n_candidate)
        info = self._check_info(self.batch.setup_device())
        self._host_stale = True
        return info

    def sync_host(self):
        """Device mode: refresh the host mirrors x_s, l_s, ns, x_c, nc from the GPU."""
        if self.device_resident and getattr(self, "_host_stale", False):
            st = self.batch.get_staged()
            cap = st["x_s"].shape[1]
            if cap > self.cap:
                self.x_s = np.concatenate([self.x_s, np.zeros((self.P, cap - self.cap))], axis=1)
                self.l_s = np.concatenate([self.l_s, np.ones((self.P, cap - self.cap))], axis=1)
                self.cap = cap
            self.x_s[:, :cap], self.l_s[:, :cap] = st["x_s"], st["l_s"]
            self.ns, self.nc, self.x_c = st["ns"], st["nc"], st["x_c"]
            self._host_stale = False

    def _grow_device(self):
        """Move the device batch to the next capacity class (observations and generator states are carried over)."""
        st = self.batch.get_staged()
        mt, pos = self.batch.rng_get()
        old_cap = self.batch.capacity
        cap_class = _lib.load().bqb_ns_capacity(old_cap + 1)
        if cap_class < 0:
            raise NotImplementedError("more than 512 observations per problem")
        self.batch.close()
        self.batch = _lib.Batch(self.P, cap_class, device=self.device)
        self._cap_class = cap_class
        self.batch.stage(st["ns"], st["x_s"], st["l_s"], self.hyp, self.prior)
        self.batch.rng_set(mt, pos)
        if self.periodic:
            self.batch.set_approx(1, period=self.period, xo=self.xo, p_xo=self.p_xo)

    def _apply_approx(self):
        """Periodic kernel: the grid of every problem from its current p_tl (``BQ._approx`` as of init: np.linspace of
        [-pi p_tl, pi p_tl], the von Mises density on it) and its upload, with the periods, to the device batch."""
        mu, var = self.prior[:, 0], self.prior[:, 1]
        self.xo = np.empty((self.P, N_GRID))
        self.p_xo = np.empty((self.P, N_GRID))
        for p in range(self.P):                            # BQ's scalar expressions, so that the grids are the same bits
            p_tl = float(self.period[p, 0])
            self.xo[p] = np.linspace(-1 * np.pi * p_tl, +1 * np.pi * p_tl, N_GRID)
            self.p_xo[p] = _vonmises_px(self.xo[p], float(mu[p]), float(var[p]))
        self.batch.set_approx(1, period=self.period, xo=self.xo, p_xo=self.p_xo)

    def init(self):
        if self.device_resident:
            return self._init_device()
        if self.periodic:
            lo, hi = -np.pi * self.period[:, 0], np.pi * self.period[:, 0]      # bq.py:217-218
        else:
            w_tl = self.hyp[:, 1]
            idx = np.arange(self.cap)[None, :] < self.ns[:, None]
            lo = np.where(idx, self.x_s, np.inf).min(axis=1) - w_tl
            hi = np.where(idx, self.x_s, -np.inf).max(axis=1) + w_tl
        xc = np.stack([self.rngs[p].uniform(lo[p], hi[p], self.n_candidate) for p in range(self.P)])
        filter_candidates_batch(xc, self.x_s, self.ns, self.thresh)
        xc.sort(axis=1)                                   # NaNs sort last
        self.nc = (~np.isnan(xc)).sum(axis=1).astype(np.int32)
        self.x_c[:] = 0.0
        self.x_c[:, :self.n_candidate] = np.nan_to_num(xc, nan=0.0)
        cap_class = _lib.load().bqb_ns_capacity(max(int(self.ns.max()), self._class_hint))
        if cap_class < 0:
            raise NotImplementedError("more than 512 observations per problem")
        if self.batch is None or self._cap_class != cap_class:       # crossed a kernel capacity class: new device batch
            self.close()
            self.batch = _lib.Batch(self.P, cap_class, device=self.device)
            self._cap_class = cap_class
        if self.periodic:
            self._apply_approx()
        stride = min(self.cap, cap_class)
        info = self.batch.setup(self.ns, self.nc, self.x_s[:, :stride], self.l_s[:, :stride], self.x_c, self.hyp, self.prior)
        return self._check_info(info)

    def Z_mean(self):
        return self.info["Z_mean"]

    def Z_var(self):
        return self.info["Z_var"]

    # ---------------------------------------------------------------- hyper-parameter samples (bq.py:533-598)
    def _rows(self):
        """The batch's hyper-parameter rows: hyp [P, 6], with the periodic kernel [P, 8] = (hyp, period)."""
        return np.concatenate([self.hyp, self.period], axis=1) if self.periodic else self.hyp

    def _set_rows(self, rows):
        self.hyp[:] = rows[:, :6]
        if self.periodic:
            self.period[:] = rows[:, 6:]

    def _upload_rows(self, rows):
        """Hyper-parameter rows [P, 6 | 8] to the device batch (the next setup_device uses them)."""
        self.batch.set_hypers(rows[:, :6])
        if self.periodic:
            self.batch.set_periods(rows[:, 6:])

    def _cols(self, params):
        """(columns of gp_log_l, columns of gp_l) of the named parameters in a hyper-parameter row."""
        bad = [p for p in params if p not in self._names]
        if not params or bad:
            raise ValueError("unknown hyper-parameter in %s (BatchBQ has %s)" % (list(params), ", ".join(self._names)))
        return [_COLS[p][0] for p in params], [_COLS[p][1] for p in params]

    def _hyp_rows(self, hypers_tl, hypers_l, params):
        """[..., 6] hyper-parameter rows (h, w, s of gp_log_l, then of gp_l; with the periodic kernel [..., 8], the periods
        p_tl, p_l last): the batch's own with the named entries replaced by hypers_tl / hypers_l [P, ..., len(params)]."""
        hypers_tl, hypers_l = np.asarray(hypers_tl, dtype=np.float64), np.asarray(hypers_l, dtype=np.float64)
        k = len(params)
        if hypers_tl.shape != hypers_l.shape or hypers_tl.shape[0] != self.P or hypers_tl.shape[-1] != k:
            raise ValueError("hypers_tl and hypers_l must be [P, ..., %d] arrays of the same shape" % k)
        mid = hypers_tl.shape[1:-1]
        base = self._rows()
        w = base.shape[1]
        hyp = np.array(np.broadcast_to(base.reshape((self.P,) + (1,) * len(mid) + (w,)), (self.P,) + mid + (w,)))
        for j, name in enumerate(params):
            if name not in self._names:
                raise ValueError("unknown hyper-parameter %r (BatchBQ has %s)" % (name, ", ".join(self._names)))
            ct, cl = _COLS[name]
            hyp[..., ct], hyp[..., cl] = hypers_tl[..., j], hypers_l[..., j]
        return hyp

    @staticmethod
    def _valid_hyp(hyp):
        """The values GP.set_param accepts: finite, h and w positive, s non-negative (and the periods of [..., 8] rows
        positive)."""
        ok = (np.isfinite(hyp).all(axis=-1) & (hyp[..., [0, 1, 3, 4]] > 0).all(axis=-1)
              & (hyp[..., [2, 5]] >= 0).all(axis=-1))
        if hyp.shape[-1] == 8:
            ok &= (hyp[..., 6:] > 0).all(axis=-1)
        return ok

    def log_lh(self, hypers_tl, hypers_l, params):
        """Joint log marginal likelihood ``gp_log_l.log_lh + gp_l.log_lh`` of every problem under its own proposal
        hypers_tl[p] / hypers_l[p] ([P, len(params)]): entry p is what the reference's ``_make_llh_params(params)``
        (bq.py:533-552) returns for problem p -- l_c recomputed from the candidates, -inf for an invalid value, a Gram
        matrix that is not positive definite or the "GP mean is too large" guard (bq.py:942-947); a log likelihood that
        does not come out finite (a numerically singular Gram matrix) is -inf too, so that no chain of sample_hypers can
        settle on it.

        One setup of all P problems on the batch itself; the batch's own hyper-parameters are set up again afterwards
        (the setup is deterministic, so the scoring model, Z_mean and Z_var are exactly what they were)."""
        hyp = self._hyp_rows(hypers_tl, hypers_l, params)
        ok = self._valid_hyp(hyp)
        hyp[~ok] = self._rows()[~ok]                      # rows the device must not see; their result is -inf
        try:
            self._upload_rows(hyp)
            info = self.batch.setup_device(check_max=True)
        finally:
            self._upload_rows(self._rows())
            self._check_info(self.batch.setup_device())
        return np.where(ok & (info["status"] == _lib.SETUP_OK) & np.isfinite(info["log_lh"]), info["log_lh"], -np.inf)

    def _log_lh_grad_rows(self, rows, hyp):
        """(log_lh [r], grad [r, 6 | 8]) of the problems ``rows`` under the hyper-parameter rows hyp [r, 6 | 8], with the
        -inf semantics of log_lh (the gradient is NaN there).  Only the valid rows reach the device."""
        rows = np.asarray(rows, dtype=np.int64)
        ll, grad = np.full(rows.size, -np.inf), np.full((rows.size, hyp.shape[1]), np.nan)
        ok = self._valid_hyp(hyp)
        if ok.any():
            if self.periodic:
                l, g, st = self.batch.log_lh_grad_periodic(hyp[ok, :6], hyp[ok, 6:], inst=rows[ok], check_max=True)
            else:
                l, g, st = self.batch.log_lh_grad(hyp[ok], inst=rows[ok], check_max=True)
            good = (st == _lib.SETUP_OK) & np.isfinite(l)
            idx = np.nonzero(ok)[0][good]
            ll[idx], grad[idx] = l[good], g[good]
        return ll, grad

    def log_lh_grad(self, hypers_tl, hypers_l, params):
        """``log_lh`` with its gradient: the joint log marginal likelihood of every problem under hypers_tl[p] /
        hypers_l[p] ([P, len(params)]) and its derivatives with respect to those named parameters, from one launch of the
        gradient kernel (the closed-form derivative of both GPs' log likelihoods, including the dependence of l_c on the
        parameters of gp_log_l).  Returns (log_lh [P], grad_tl [P, k], grad_l [P, k]).  log_lh is -inf where ``log_lh``
        gives -inf, and the gradient is NaN there.  The batch's model is not touched."""
        hyp = self._hyp_rows(hypers_tl, hypers_l, params)
        if hyp.ndim != 2:
            raise ValueError("hypers_tl and hypers_l must be [P, %d]" % len(params))
        ll, g = self._log_lh_grad_rows(np.arange(self.P), hyp)
        ct, cl = self._cols(params)
        return ll, g[:, ct], g[:, cl]

    def fit_hypers(self, params, maxiter=200):
        """Maximise every problem's joint log marginal likelihood over the named parameters of both GPs
        (``BQ.fit_hypers``, bq.py:554-562), starting from the batch's hyper-parameters.  The optimiser is
        ``util.lbfgs_batch`` in the logarithms of the parameters, with the gradient from ``log_lh_grad``; each of its
        steps evaluates only the problems that are still running.  The fitted values are written into ``self.hyp`` and
        the model is set up again under them; the candidates stay as they are (the reference's fit only recomputes l_c).

        A problem whose start has zero probability raises RuntimeError naming it, before anything changes.  Fitting "s"
        needs s > 0 at the start for both GPs of every problem (ValueError otherwise).  Returns a dict: log_lh [P] at the
        fitted point, converged [P], iterations [P] and evaluations (problem evaluations in total)."""
        ct, cl = self._cols(params)
        cols6 = ct + cl
        start = self._rows()
        if not (start[:, cols6] > 0).all():
            raise ValueError("fitting %s needs positive starting values (it works with their logarithms)" % list(params))

        def fg(X, rows):
            hyp = start[rows].copy()
            hyp[:, cols6] = np.exp(X)
            ll, g = self._log_lh_grad_rows(rows, hyp)
            return ll, g[:, cols6] * hyp[:, cols6]           # d ll / d log(theta)
        try:
            res = util.lbfgs_batch(fg, np.log(start[:, cols6]), maxiter=maxiter)
        except RuntimeError as e:
            if getattr(e, "row", None) is None:
                raise
            raise RuntimeError("problem %d: zero probability at the starting hyper-parameters" % e.row) from e
        fitted = start.copy()
        fitted[:, cols6] = np.exp(res["x"])
        self._set_rows(fitted)
        self._upload_rows(self._rows())
        self._check_info(self.batch.setup_device())
        return {"log_lh": res["f"], "converged": res["converged"], "iterations": res["iterations"],
                "evaluations": res["evaluations"]}

    def sample_hypers(self, params, n, nburn=10, seed=0, first_problem=0, max_steps=None, stats=None):
        """Slice-sample the named hyper-parameters of both GPs of every problem (``BQ.sample_hypers``, bq.py:565-598):
        one chain per problem, started at the batch's hyper-parameters with window 2 * len(params), n samples after
        nburn.  Each sampler step is ONE ``log_lh`` evaluation of all problems.  Chain p draws from the counter stream
        keyed by the pair (seed, first_problem + p) (``util.stream_keys``, ``util.slice_sample_batch``), so its samples do
        not depend on the other problems of the batch; ``first_problem`` is the index of the batch's first problem in the
        caller's numbering (a shard or a sub-batch then draws the streams the whole batch would).  ``max_steps`` /
        ``stats``: see ``util.slice_sample_batch``.  Returns (hypers_tl, hypers_l), each [P, n, len(params)].  A problem
        whose start has zero probability raises RuntimeError (the reference would search for better starting parameters
        instead)."""
        k = len(params)
        ct, cl = self._cols(params) if k else ([], [])
        rows = self._rows()
        x0 = np.concatenate([rows[:, ct], rows[:, cl]], axis=1)
        f = lambda X: self.log_lh(X[:, :k], X[:, k:], params)
        keys = util.stream_keys(seed, int(first_problem) + np.arange(self.P))
        try:
            s = util.slice_sample_batch(f, x0, n, 2 * k, keys, nburn=nburn, max_steps=max_steps, stats=stats)
        except RuntimeError as e:
            if getattr(e, "chain", None) is None:
                raise
            raise RuntimeError("problem %d: zero probability at the starting hyper-parameters" % e.chain) from e
        return s[:, :, :k], s[:, :, k:]

    #: device memory of the model blocks of one marginal_loss chunk (whole problems x samples)
    MODEL_CHUNK_BYTES = 4 << 30
    #: the [problems x samples, na] score buffer of one scoring launch (64 MB stays L2-resident on a B200, as BQ.LOSS_CHUNK_BYTES)
    LOSS_CHUNK_BYTES = 64 << 20

    def _sample_batch(self, n_inst):
        """A device batch of n_inst (problem, sample) instances of the current capacity class, kept between calls."""
        cache = self.__dict__.setdefault("_sample_batches", {})
        for key in [k for k in cache if k[1] != self._cap_class]:
            cache.pop(key).close()
        key = (n_inst, self._cap_class)
        if key not in cache:                              # (at most two sizes: full chunks and the last one)
            cache[key] = _lib.Batch(n_inst, self._cap_class, device=self.device)
        return cache[key]

    def _chunks(self, S, na):
        """(problems per setup chunk, problems per scoring launch) under MODEL_CHUNK_BYTES / LOSS_CHUNK_BYTES."""
        model_bytes = 8 * _lib.load().bqb_model_doubles(self.batch._h)
        if self.periodic:
            model_bytes += 8 * (3 * N_GRID + 2)           # grid, prior density, trapezoid weights and periods per instance
        per_score = max(1, min(self.P, self.LOSS_CHUNK_BYTES // max(8 * S * max(na, 1), 1)))
        per_setup = max(1, min(self.P, self.MODEL_CHUNK_BYTES // (S * model_bytes)))
        if per_setup >= per_score:
            per_setup -= per_setup % per_score               # whole scoring launches per setup chunk
        return per_setup, min(per_score, per_setup)

    def _query(self, x_a):
        import torch
        dev = torch.device("cuda", self.device)
        if isinstance(x_a, torch.Tensor):
            return None, x_a.to(dev, torch.float64).contiguous()
        x_a = np.ascontiguousarray(x_a, dtype=np.float64)
        return x_a, torch.from_numpy(x_a).to(dev)

    def marginal_loss(self, x_a, hypers_tl, hypers_l, params, timings=None):
        """Marginal loss of choose_next for every problem: the mean over its S samples (hypers_tl / hypers_l
        [P, S, len(params)]) of ``-expected_squared_mean(x_a)`` (bq.py:640-663), as a [P, na] CUDA tensor; row p is
        ``BQ(problem p).marginal_loss(x_a, hypers_tl[p], hypers_l[p], params)``.  Each sample is set up with the semantics
        of ``_set_gp_log_l_params`` / ``_set_gp_l_params`` (bq.py:933-965: l_c recomputed, "GP mean is too large" guard).
        ``x_a`` is a shared grid [na] or per-problem grids [P, na] (numpy or a float64 CUDA tensor).

        The P x S instances are set up in chunks of whole problems (MODEL_CHUNK_BYTES of model blocks) and scored in
        launches of whole problems (LOSS_CHUNK_BYTES of scores): the S samples of a problem read its grid row
        (``score_device_grouped``) and a segmented reduction adds their -esm in sample order, the additions of
        ``values[0].mean(axis=0)``.
        ``timings``, when a dict, receives the seconds spent in the three phases ("setup", "score", "reduce"; CUDA events
        around each launch, which then synchronise after every scoring launch -- for measurements only)."""
        import torch
        hyp = self._hyp_rows(hypers_tl, hypers_l, params)
        if hyp.ndim != 3:
            raise ValueError("hypers_tl and hypers_l must be [P, S, %d]" % len(params))
        S = hyp.shape[1]
        if S < 1:
            raise ValueError("at least one hyper-parameter sample per problem")
        _, x_d = self._query(x_a)
        if x_d.dim() not in (1, 2) or (x_d.dim() == 2 and x_d.shape[0] != self.P):
            raise ValueError("x_a must be [na] or [P, na]")
        na = x_d.shape[-1]
        self.sync_host()
        ok = self._valid_hyp(hyp)
        if not ok.all():
            p, i = np.argwhere(~ok)[0]
            raise ValueError("invalid hyper-parameters %s in sample %d of problem %d" % (hyp[p, i], i, p))
        stride = min(self.cap, self._cap_class)
        per_setup, per_score = self._chunks(S, na)
        dev = x_d.device
        loss = torch.zeros(self.P, na, dtype=torch.float64, device=dev)
        if na == 0:
            return loss
        esm = torch.empty(per_score * S, na, dtype=torch.float64, device=dev)
        flags = torch.zeros(per_score * S, dtype=torch.int32, device=dev)
        bad_esm = torch.zeros(self.P, dtype=torch.bool, device=dev)
        bad_xa = torch.zeros(self.P, dtype=torch.bool, device=dev)
        for p0 in range(0, self.P, per_setup):
            cp = min(per_setup, self.P - p0)
            rep = lambda a: np.repeat(a[p0:p0 + cp], S, axis=0)
            batch = self._sample_batch(cp * S)
            t0 = time.perf_counter()
            hrows = hyp[p0:p0 + cp].reshape(cp * S, hyp.shape[-1])
            if self.periodic:                             # each sample's periods, its problem's grid
                batch.set_approx(1, period=hrows[:, 6:], xo=rep(self.xo), p_xo=rep(self.p_xo))
            info = batch.setup(rep(self.ns), rep(self.nc), rep(self.x_s[:, :stride]), rep(self.l_s[:, :stride]), rep(self.x_c),
                               hrows[:, :6], rep(self.prior), check_max=True)
            bad = np.nonzero(info["status"])[0]
            if bad.size:
                p, i = divmod(int(bad[0]), S)
                logger.error("error with parameters %s", hyp[p0 + p, i])
                exc, msg = _SETUP_ERRORS.get(int(info["status"][bad[0]]), (RuntimeError, "device setup failed"))
                raise exc("%s (problem %d, sample %d)" % (msg, p0 + p, i))
            if timings is not None:
                timings["setup"] = timings.get("setup", 0.0) + time.perf_counter() - t0     # setup synchronises
            for q0 in range(0, cp, per_score):
                cq = min(per_score, cp - q0)
                rows = x_d if x_d.dim() == 1 else x_d[p0 + q0:p0 + q0 + cq]
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)] if timings is not None else None
                if ev:
                    ev[0].record()
                batch.score_device_grouped(q0 * S, cq * S, rows, S, esm, None, None, flags)
                if ev:
                    ev[1].record()
                batch.sum_neg_accum_groups_device(esm, cq, S, loss[p0 + q0:p0 + q0 + cq])
                if ev:
                    ev[2].record()
                    ev[2].synchronize()
                    timings["score"] = timings.get("score", 0.0) + ev[0].elapsed_time(ev[1]) / 1e3
                    timings["reduce"] = timings.get("reduce", 0.0) + ev[1].elapsed_time(ev[2]) / 1e3
                fl = flags[:cq * S].view(cq, S)
                bad_esm[p0 + q0:p0 + q0 + cq] |= ((fl & (_lib.ST_ESM_BAD | _lib.ST_EM_BAD)) != 0).any(dim=1)
                bad_xa[p0 + q0:p0 + q0 + cq] |= ((fl & _lib.ST_XA_BAD) != 0).any(dim=1)
        loss /= S                                         # bq.py:662
        if bool(bad_xa.any().item()):
            raise ValueError("invalid value in x_a of problem %d" % int(torch.nonzero(bad_xa)[0, 0].item()))
        if bool(bad_esm.any().item()):
            raise RuntimeError("invalid expected squared mean under a sampled hyper-parameter set of problem %d"
                               % int(torch.nonzero(bad_esm)[0, 0].item()))
        return loss

    # ---------------------------------------------------------------- one active-sampling round
    def choose_next(self, x_a, on_device=False, n=None, params=None, hypers=None, seed=None, max_steps=None):
        """Deterministic choose_next of every problem over a shared grid ``x_a`` [na] or per-problem grids
        [P, na]: index and location of the first maximiser of expected_squared_mean.  ``x_a`` may be a float64
        CUDA tensor (it is then not uploaded again); with ``on_device=True`` the result is a pair of CUDA tensors.

        With ``n`` (and ``params``), the loss is marginalised over hyper-parameter samples like the reference's
        ``BQ.choose_next(x_a, n, params)`` (bq.py:659-681): ``sample_hypers(params, n, nburn=1, seed, max_steps)`` draws
        them, or ``hypers=(hypers_tl, hypers_l)`` ([P, S, len(params)]) gives them; the choice is the first minimiser of
        each problem's ``marginal_loss``.  Without ``seed``, the r-th sampling round of this batch uses the seed
        ``util.stream_keys(batch seed, r)``: every round draws fresh streams, as the reference's global stream advances."""
        if n is not None or hypers is not None:
            return self._choose_marginal(x_a, on_device, n, params, hypers, seed, max_steps)
        import torch
        dev = torch.device("cuda", self.device)
        if isinstance(x_a, torch.Tensor):
            x_d = x_a.to(dev, torch.float64).contiguous()
            x_a = None
        else:
            x_a = np.ascontiguousarray(x_a, dtype=np.float64)
            x_d = torch.from_numpy(x_a).to(dev)
        na = x_d.shape[-1]
        if getattr(self, "_esm", None) is None or self._esm.shape != (self.P, na):
            self._esm = torch.empty(self.P, na, dtype=torch.float64, device=dev)
            self._mins = torch.empty(self.P, dtype=torch.float64, device=dev)
            self._idxs = torch.empty(self.P, dtype=torch.int64, device=dev)
            self._flags = torch.zeros(self.P, dtype=torch.int32, device=dev)
        self.batch.score_device(x_d, self._esm, None, None, self._flags)
        self._esm.neg_()                                  # loss = -esm (bq.py:660)
        self.batch.argmin_rows_device(self._esm, self._mins, self._idxs)
        bad = int((self._flags & (_lib.ST_ESM_BAD | _lib.ST_EM_BAD | _lib.ST_XA_BAD)).ne(0).any().item())
        if bad:
            fl = self._flags.cpu().numpy()
            raise RuntimeError("invalid expected squared mean in problem %d" % int(np.argmax(fl & 112 != 0)))
        if on_device:
            x_next = x_d[self._idxs] if x_d.dim() == 1 else x_d.gather(1, self._idxs[:, None])[:, 0]
            return self._idxs, x_next
        idx = self._idxs.cpu().numpy()
        if x_a is None:
            x_a = x_d.cpu().numpy()
        x_next = x_a[idx] if x_a.ndim == 1 else x_a[np.arange(self.P), idx]
        return idx, x_next

    def _choose_marginal(self, x_a, on_device, n, params, hypers, seed, max_steps):
        import torch
        if params is None:
            raise ValueError("params names the sampled hyper-parameters")
        if hypers is None:
            if seed is None:
                r = self.__dict__.get("_sample_rounds", 0)
                self._sample_rounds = r + 1
                seed = int(util.stream_keys(self.seed, r))
            hypers = self.sample_hypers(params, n, nburn=1, seed=seed, max_steps=max_steps)
        x_a, x_d = self._query(x_a)
        loss = self.marginal_loss(x_d, hypers[0], hypers[1], params)
        mins = torch.empty(self.P, dtype=torch.float64, device=x_d.device)
        idxs = torch.empty(self.P, dtype=torch.int64, device=x_d.device)
        self.batch.argmin_rows_device(loss, mins, idxs)
        if on_device:
            x_next = x_d[idxs] if x_d.dim() == 1 else x_d.gather(1, idxs[:, None])[:, 0]
            return idxs, x_next
        idx = idxs.cpu().numpy()
        if x_a is None:
            x_a = x_d.cpu().numpy()
        x_next = x_a[idx] if x_a.ndim == 1 else x_a[np.arange(self.P), idx]
        return idx, x_next

    def add_observations(self, x_new, l_new):
        """Vectorised ``add_observation`` (bq.py:683-701): average into the nearest observation when it is
        closer than candidate_thresh, append otherwise; then re-initialise every problem.  In device-resident mode
        ``x_new`` / ``l_new`` may be CUDA tensors and nothing but they crosses PCIe."""
        if self.device_resident:
            import torch
            dev = torch.device("cuda", self.device)
            as_dev = lambda v: (v.to(dev, torch.float64).contiguous() if isinstance(v, torch.Tensor)
                                else torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64)).to(dev))
            x_d, l_d = as_dev(x_new), as_dev(l_new)
            if x_d.shape != (self.P,) or l_d.shape != (self.P,):
                raise ValueError("x_new and l_new must have one entry per problem")
            if not bool((l_d > 0).all().item()):
                raise ValueError("l_s contains zero or negative values")
            if self._ns_max + 1 > self.batch.capacity:
                self._grow_device()
            self.batch.add_observations(x_d, l_d)
            self._ns_max += 1
            return self._init_device()
        x_new, l_new = np.asarray(x_new, dtype=np.float64), np.asarray(l_new, dtype=np.float64)
        valid = np.arange(self.cap)[None, :] < self.ns[:, None]
        d = np.abs(x_new[:, None] - self.x_s)
        d[~valid] = np.inf
        c = d.argmin(axis=1)
        merge = d[np.arange(self.P), c] < self.thresh
        rows = np.nonzero(merge)[0]
        self.x_s[rows, c[rows]] = (self.x_s[rows, c[rows]] + x_new[rows]) / 2.0
        self.l_s[rows, c[rows]] = (self.l_s[rows, c[rows]] + l_new[rows]) / 2.0
        rows = np.nonzero(~merge)[0]
        if rows.size and self.ns[rows].max() >= self.cap:
            grow = max(16, self.cap // 4)
            self.x_s = np.concatenate([self.x_s, np.zeros((self.P, grow))], axis=1)
            self.l_s = np.concatenate([self.l_s, np.ones((self.P, grow))], axis=1)
            self.cap += grow
        self.x_s[rows, self.ns[rows]] = x_new[rows]
        self.l_s[rows, self.ns[rows]] = l_new[rows]
        self.ns[rows] += 1
        return self.init()
