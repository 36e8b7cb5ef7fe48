"""Host-side helpers of the BQ interface that are outside the CUDA hot path: candidate filtering,
the slice sampler, the optimiser wrapper and two plot helpers (reference:
bayesian_quadrature/util.py, util_c.pyx, and bq_c.filter_candidates)."""
import ctypes
import logging

import numpy as np

logger = logging.getLogger("bayesian_quadrature.util")
DTYPE = np.dtype("float64")
MIN = np.log(np.exp2(np.float64(np.finfo(np.float64).minexp + 4)))
RAND_MAX = 2147483647


def filter_candidates(x_c, x_s, thresh):
    """In-place candidate filter with the semantics of bq_c.filter_candidates (bq_c.pyx:601-650):
    repeatedly merge candidates closer than `thresh` into their midpoint (the second one becomes
    NaN), then drop candidates closer than `thresh` to an observation."""
    nc = x_c.shape[0]
    merged = True
    while merged:
        merged = False
        for i in range(nc):
            if np.isnan(x_c[i]):
                continue
            for j in range(i + 1, nc):
                if np.isnan(x_c[j]):
                    continue
                if abs(x_c[i] - x_c[j]) < thresh:
                    x_c[i] = (x_c[i] + x_c[j]) / 2.0
                    x_c[j] = np.nan
                    merged = True
    if x_s.size:
        for i in range(nc):
            if not np.isnan(x_c[i]) and (np.abs(x_c[i] - x_s) < thresh).any():
                x_c[i] = np.nan


class _LibcRand(object):
    """libc srand/rand, so that a run seeded through numpy consumes the same two random streams as
    the reference sampler (util_c.pyx:21-22, :33)."""

    def __init__(self):
        self._libc = ctypes.CDLL(None)
        self._libc.rand.restype = ctypes.c_int
        self._libc.srand.argtypes = [ctypes.c_uint]

    def seed(self, s):
        self._libc.srand(int(s))

    def uniform(self, lo, hi):
        return (self._libc.rand() / float(RAND_MAX)) * (hi - lo) + lo


def slice_sample(logpdf, niter, w, xval, nburn=1, freq=1):
    """Multivariate slice sampler along random directions with stepping-out and shrinkage
    (util.py:45-75 wrapper + util_c.pyx:25-148).  Returns samples[nburn:][::freq]."""
    xval = np.asarray(xval, dtype=DTYPE)
    d = xval.size
    samples = np.empty((niter, d))
    samples[0] = xval
    rng = _LibcRand()
    rng.seed(np.random.randint(0, RAND_MAX))
    i = 0
    while i < niter - 1:
        cur = samples[i]
        height = logpdf(cur)
        if height == -np.inf:
            raise RuntimeError("zero probability encountered")
        logy = np.log(rng.uniform(0, np.exp(height)))
        direction = np.random.rand(d) - 0.5
        direction /= np.linalg.norm(direction)
        left, right = -w, w
        j = 0
        while logpdf(cur + left * direction) >= logy:     # step out, at most 101 times per side
            left -= w
            j += 1
            if j > 100:
                break
        j = 0
        while logpdf(cur + right * direction) >= logy:
            right += w
            j += 1
            if j > 100:
                break
        while True:
            if (right - left) < 1e-9:             # window collapsed: retry this iteration
                break
            loc = rng.uniform(left, right)
            samples[i + 1] = cur + loc * direction
            if logpdf(samples[i + 1]) > logy:
                i += 1
                break
            if loc < 0:
                left = loc
            else:
                right = loc
    return samples[nburn:][::freq]


def _splitmix64(z):
    with np.errstate(over="ignore"):                     # arithmetic modulo 2^64 is the hash
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def counter_uniform(keys, counters):
    """Uniform doubles in [0, 1), one per (stream key, draw counter) pair (integer arrays of one shape): a splitmix64
    hash of the key, mixed with the counter and hashed again, keeps its top 53 bits.  A stream is a pure function of its
    key, so that many chains can draw from their own streams in any interleaving."""
    z = _splitmix64(_splitmix64(_u64(keys)) ^ _u64(counters))
    return (z >> np.uint64(11)).astype(DTYPE) * (1.0 / 9007199254740992.0)


def _u64(v):
    """Integers as uint64 words (negative values wrap modulo 2^64)."""
    v = np.asarray(v)
    return v.astype(np.uint64) if v.dtype.kind == "u" else v.astype(np.int64).astype(np.uint64)


def stream_keys(seed, problems):
    """Stream keys of problems ``problems`` under ``seed``: seed and problem index are hashed as separate words
    (splitmix64(splitmix64(seed) ^ p)), so that no (seed, p) pair shares the stream of another."""
    return _splitmix64(_splitmix64(_u64(np.full(np.shape(problems), seed))) ^ _u64(problems))


_START, _NEW, _LEFT, _RIGHT, _SHRINK, _DONE = range(6)


def slice_sample_batch(logpdf, x0, n, w, keys, nburn=1, max_steps=None, stats=None):
    """``slice_sample`` for many independent chains advanced in lock-step: chain p starts at x0[p] and returns
    ``samples[nburn:]`` of nburn + n iterations, i.e. an array [P, n, d].

    ``logpdf(X)`` takes the [P, d] points of all chains and returns their [P] log densities; it is called once per step,
    where every unfinished chain has exactly one point to evaluate (finished chains pass their last sample).  Per chain the
    algorithm is that of ``slice_sample``: a random unit direction, stepping-out of at most 101 steps per side, shrinkage,
    and a retry of the iteration when the window collapses below 1e-9.  The density of the current point is the one
    computed when it was accepted (``slice_sample`` evaluates it again, to the same value).  The slice height is
    drawn as ``height + log(u)``: ``slice_sample``'s ``log(u * exp(height))`` is infinite, and the chain stuck, once a
    joint log likelihood exceeds 709.

    Chain p draws from the counter stream ``counter_uniform(keys[p], 0, 1, 2, ...)``: per iteration one draw for the slice
    height, d for the direction (each minus 0.5, then normalised), one per shrinkage proposal.  Its samples therefore depend
    only on its key, its start and its own densities.  (``slice_sample`` shares the global libc and numpy streams instead.)
    A start of density -inf raises RuntimeError naming the chain.

    The chains advance in lock-step, so the slowest one sets the number of steps.  ``max_steps`` (default: no limit)
    caps the ``logpdf`` calls of this run: a chain that has not finished by then stays at its last accepted point for
    the samples it still owes (a shorter chain, not a different algorithm).  ``stats``, when a dict, receives "steps" (the
    ``logpdf`` calls made) and "unfinished" (the indices of the chains the cap stopped)."""
    x0 = np.array(x0, dtype=DTYPE, ndmin=2)
    P, d = x0.shape
    keys = _u64(keys).reshape(P)
    if max_steps is not None and max_steps < 1:
        raise ValueError("max_steps must be at least 1")
    n_calls = 0
    niter = nburn + int(n)
    samples = np.empty((P, niter, d))
    samples[:, 0] = x0
    rows = np.arange(P)
    it = np.zeros(P, dtype=np.int64)                     # index of the current point in samples
    ctr = np.zeros(P, dtype=np.uint64)
    phase = np.full(P, _START if niter > 1 else _DONE)
    height, logy, left, right, loc = (np.zeros(P) for _ in range(5))
    direction = np.zeros((P, d))
    steps = np.zeros(P, dtype=np.int64)

    def draw(sel, k):
        c = ctr[sel][:, None] + np.arange(k, dtype=np.uint64)[None, :]
        ctr[sel] += np.uint64(k)
        return counter_uniform(np.broadcast_to(keys[sel][:, None], c.shape), c)

    def begin(sel):                                      # a new iteration from the current point
        u = draw(sel, 1)[:, 0]
        with np.errstate(divide="ignore"):
            logy[sel] = height[sel] + np.log(u)           # log(u * exp(height)) without the overflow of exp above 709
        dv = draw(sel, d) - 0.5
        nrm = dv[:, 0] * dv[:, 0]
        for c in range(1, d):
            nrm += dv[:, c] * dv[:, c]
        direction[sel] = dv / np.sqrt(nrm)[:, None]
        left[sel], right[sel], steps[sel] = -w, w, 0
        phase[sel] = _LEFT

    while True:
        if (phase == _NEW).any():
            begin(phase == _NEW)
        collapsed = (phase == _SHRINK) & ((right - left) < 1e-9)
        if collapsed.any():
            begin(collapsed)
        shrink = phase == _SHRINK
        if shrink.any():
            loc[shrink] = draw(shrink, 1)[:, 0] * (right[shrink] - left[shrink]) + left[shrink]
        if (phase == _DONE).all():
            break
        if max_steps is not None and n_calls >= max_steps:
            for p in np.nonzero(phase != _DONE)[0]:
                samples[p, it[p] + 1:] = samples[p, it[p]]
            break
        cur = samples[rows, it]
        off = np.select([phase == _LEFT, phase == _RIGHT, phase == _SHRINK], [left, right, loc], 0.0)
        move = (phase == _LEFT) | (phase == _RIGHT) | (phase == _SHRINK)
        pts = np.where(move[:, None], cur + off[:, None] * direction, cur)
        f = np.asarray(logpdf(pts), dtype=DTYPE).reshape(P)
        n_calls += 1
        ph = phase.copy()

        sel = ph == _START
        if sel.any():
            bad = sel & (f == -np.inf)
            if bad.any():
                err = RuntimeError("zero probability encountered at the start of chain %d" % int(np.argmax(bad)))
                err.chain = int(np.argmax(bad))
                raise err
            height[sel] = f[sel]
            phase[sel] = _NEW
        for side, sign, nxt in ((_LEFT, -1.0, _RIGHT), (_RIGHT, 1.0, _SHRINK)):
            sel = ph == side
            if sel.any():
                up = sel & (f >= logy)
                bound = left if side == _LEFT else right
                bound[up] += sign * w
                steps[up] += 1
                out = sel & (~up | (steps > 100))
                phase[out], steps[out] = nxt, 0
        sel = ph == _SHRINK
        if sel.any():
            acc = sel & (f > logy)
            it[acc] += 1
            samples[rows[acc], it[acc]] = pts[acc]
            height[acc] = f[acc]
            phase[acc] = np.where(it[acc] == niter - 1, _DONE, _NEW)
            rej = sel & ~acc
            neg = rej & (loc < 0)
            left[neg] = loc[neg]
            pos = rej & ~(loc < 0)
            right[pos] = loc[pos]
    if stats is not None:
        stats["steps"], stats["unfinished"] = n_calls, np.nonzero(phase != _DONE)[0]
    return samples[:, nburn:]


def _rowdot(a, b):
    """Row-wise dot products of two [r, d] arrays, one column at a time (a row's arithmetic does not depend on r)."""
    s = a[:, 0] * b[:, 0]
    for c in range(1, a.shape[1]):
        s = s + a[:, c] * b[:, c]
    return s


def lbfgs_batch(fg, x0, maxiter=200, m=10, gtol=1e-5, ftol=2.2e-9, max_backtrack=20):
    """Maximise many independent smooth functions in lock-step with L-BFGS (memory ``m``) and a backtracking Armijo line
    search.  Row p starts at x0[p] ([P, d]).

    ``fg(X, rows)`` returns (f [r], g [r, d]), the values and gradients at the points X [r, d] of the rows ``rows`` (an
    index array); it is called once per step with the rows that are still running, each at its own trial point.  A trial
    whose value is -inf or NaN (or whose gradient is not finite) counts as a failed step: the step is halved.  The first
    step of a row (and the first after its history was reset) has length at most 1.  When ``max_backtrack`` trials of
    one step fail, the row forgets its history and searches once more along the steepest direction, as scipy's L-BFGS-B
    restarts; the default of 20 trials per line search is scipy's ``maxls``.

    A row stops, as scipy's L-BFGS-B does by default, when the largest gradient entry is at most ``gtol`` or when an
    accepted step changed f by at most ``ftol * max(|f_old|, |f_new|, 1)``: it has then converged.  It also stops, not
    converged, after ``maxiter`` iterations or when the line search fails along the steepest direction too.  Every row uses only its own values
    and row-wise arithmetic, so its result does not depend on the other rows.

    A start whose value is -inf or NaN raises RuntimeError with the attribute ``row``.  Returns a dict: x [P, d], f [P],
    converged [P] (bool), iterations [P], evaluations (points evaluated, all rows together) and calls (calls of fg)."""
    x = np.array(x0, dtype=DTYPE, ndmin=2)
    P, d = x.shape
    rows_all = np.arange(P)
    f, g = fg(x.copy(), rows_all)
    f, g = np.asarray(f, dtype=DTYPE).reshape(P), np.asarray(g, dtype=DTYPE).reshape(P, d)
    bad = ~np.isfinite(f)
    if bad.any():
        err = RuntimeError("zero probability at the start of row %d" % int(np.argmax(bad)))
        err.row = int(np.argmax(bad))
        raise err
    phi, G = -f, -g                                      # minimise phi = -f
    S, Y = np.zeros((P, m, d)), np.zeros((P, m, d))
    rho = np.zeros((P, m))
    nh = np.zeros(P, dtype=np.int64)                     # stored pairs
    head = np.zeros(P, dtype=np.int64)                   # slot of the next pair
    iters = np.zeros(P, dtype=np.int64)
    converged = np.abs(G).max(axis=1) <= gtol
    active = np.isfinite(G).all(axis=1) & ~converged
    p, t, slope, nbt = np.zeros((P, d)), np.zeros(P), np.zeros(P), np.zeros(P, dtype=np.int64)
    evaluations, calls = P, 1

    def direction(sel):
        """-H G for the rows sel (two-loop recursion over each row's own history), the step length and the slope."""
        r = sel.size
        q = G[sel].copy()
        al = np.zeros((r, m))
        for age in range(m):
            slot = (head[sel] - 1 - age) % m
            v = age < nh[sel]
            s_, y_ = S[sel, slot], Y[sel, slot]
            a = np.where(v, rho[sel, slot] * _rowdot(s_, q), 0.0)
            al[:, age] = a
            q = q - a[:, None] * y_
        newest = (head[sel] - 1) % m
        sy, yy = _rowdot(S[sel, newest], Y[sel, newest]), _rowdot(Y[sel, newest], Y[sel, newest])
        gam = np.where(nh[sel] > 0, sy / np.where(nh[sel] > 0, yy, 1.0), 1.0)
        z = gam[:, None] * q
        for age in reversed(range(m)):
            slot = (head[sel] - 1 - age) % m
            v = age < nh[sel]
            s_, y_ = S[sel, slot], Y[sel, slot]
            b = rho[sel, slot] * _rowdot(y_, z)
            z = z + np.where(v, al[:, age] - b, 0.0)[:, None] * s_
        pd_ = -z
        sl = _rowdot(G[sel], pd_)
        uphill = ~(sl < 0)                               # not a descent direction: forget the history
        if uphill.any():
            nh[sel[uphill]] = 0
            pd_[uphill] = -G[sel[uphill]]
            sl[uphill] = _rowdot(G[sel[uphill]], pd_[uphill])
        p[sel], slope[sel], nbt[sel] = pd_, sl, 0
        norm = np.sqrt(_rowdot(pd_, pd_))
        t[sel] = np.where(nh[sel] == 0, np.minimum(1.0, 1.0 / norm), 1.0)

    if active.any():
        direction(np.nonzero(active)[0])
    while active.any():
        sel = np.nonzero(active)[0]
        xt = x[sel] + t[sel, None] * p[sel]
        ft, gt = fg(xt.copy(), sel)
        ft, gt = np.asarray(ft, dtype=DTYPE).reshape(sel.size), np.asarray(gt, dtype=DTYPE).reshape(sel.size, d)
        evaluations += sel.size
        calls += 1
        pt = -ft
        with np.errstate(invalid="ignore"):
            ok = np.isfinite(pt) & np.isfinite(gt).all(axis=1) & (pt <= phi[sel] + 1e-4 * t[sel] * slope[sel])
        acc, rej = sel[ok], sel[~ok]
        if rej.size:
            t[rej] *= 0.5
            nbt[rej] += 1
            failed = rej[nbt[rej] >= max_backtrack]
            retry = failed[nh[failed] > 0]                   # forget the history, search along -G once more
            active[failed[nh[failed] == 0]] = False
            if retry.size:
                nh[retry] = 0
                direction(retry)
        if acc.size:
            s_ = xt[ok] - x[acc]
            y_ = -gt[ok] - G[acc]
            phi_old = phi[acc]
            x[acc], phi[acc], G[acc] = xt[ok], pt[ok], -gt[ok]
            iters[acc] += 1
            sy, yy = _rowdot(s_, y_), _rowdot(y_, y_)
            keep = sy > 2.2e-16 * yy                     # curvature condition; otherwise the pair is skipped
            ka = acc[keep]
            S[ka, head[ka]], Y[ka, head[ka]], rho[ka, head[ka]] = s_[keep], y_[keep], 1.0 / sy[keep]
            head[ka] = (head[ka] + 1) % m
            nh[ka] = np.minimum(nh[ka] + 1, m)
            done = ((np.abs(G[acc]).max(axis=1) <= gtol)
                    | (phi_old - phi[acc] <= ftol * np.maximum(np.maximum(np.abs(phi_old), np.abs(phi[acc])), 1.0)))
            converged[acc[done]] = True
            active[acc[done | (iters[acc] >= maxiter)]] = False
            nxt = acc[active[acc]]
            if nxt.size:
                direction(nxt)
    return {"x": x, "f": -phi, "converged": converged, "iterations": iters, "evaluations": int(evaluations),
            "calls": int(calls)}


def find_good_parameters(logpdf, x0, method, ntry=10):
    """Maximise `logpdf` with scipy (util.py:151-169): up to `ntry` restarts, returns None when no
    restart reaches a log-density above MIN."""
    import scipy.optimize as optim
    for i in range(ntry):
        logger.debug("Attempt #%d with %s", i + 1, method)
        res = optim.minimize(fun=lambda x: -logpdf(x), x0=x0, method=method)
        p = logpdf(res["x"])
        if p > MIN:
            return res["x"]
        if logpdf(x0) < p:
            x0 = res["x"]
    return None


def set_scientific(ax, low, high, axis=None):
    import matplotlib.pyplot as plt
    fmt = plt.ScalarFormatter()
    fmt.set_scientific(True)
    fmt.set_powerlimits((low, high))
    if axis is None or axis == "x":
        ax.get_xaxis().set_major_formatter(fmt)
    if axis is None or axis == "y":
        ax.get_yaxis().set_major_formatter(fmt)


def vlines(ax, x, **kwargs):
    ymin, ymax = ax.get_ylim()
    ax.vlines(x, ymin, ymax, **kwargs)


def hlines(ax, y, **kwargs):
    xmin, xmax = ax.get_xlim()
    ax.hlines(y, xmin, xmax, **kwargs)
