"""The batched slice sampler (util.slice_sample_batch) against a scalar per-chain run of the same algorithm on the same
counter-based streams; CPU only."""
import numpy as np
import pytest

from bayesian_quadrature_b200.util import counter_uniform, slice_sample_batch, stream_keys

D = 3
MU = np.array([[0.0, 1.0, -2.0], [3.0, 0.5, 0.0], [-1.0, -1.0, 4.0], [0.0, 0.0, 0.0], [2.0, -3.0, 1.0],
               [0.25, 0.0, -0.5], [-4.0, 2.0, 2.0]])
SD = np.array([[1.0, 2.0, 0.5], [0.3, 1.0, 1.0], [2.0, 2.0, 2.0], [1.0, 1.0, 1.0], [0.1, 0.7, 1.5],
               [1.0, 0.2, 3.0], [0.6, 0.6, 0.6]])
BOUNDED = 3                                          # chain 3 has the support |x_c| < 0.7 in every coordinate


def gauss(X, mu, sd, bounded):
    """Independent Gaussian log density per row (summed coordinate by coordinate, in order); -inf off a bounded support."""
    z = (X - mu) / sd
    out = -0.5 * (z[:, 0] * z[:, 0])
    for c in range(1, X.shape[1]):
        out = out - 0.5 * (z[:, c] * z[:, c])
    return np.where(bounded & ~(np.abs(X) < 0.7).all(axis=1), -np.inf, out)


def toy_batch(X):
    return gauss(X, MU[:len(X)], SD[:len(X)], np.arange(len(X)) == BOUNDED)


def toy_chain(p):
    return lambda x: gauss(x[None], MU[p:p + 1], SD[p:p + 1], np.array([p == BOUNDED]))[0]


class Stream(object):
    def __init__(self, key):
        self.key, self.ctr = key, 0

    def u(self):
        v = counter_uniform(np.array([self.key]), np.array([self.ctr], dtype=np.uint64))[0]
        self.ctr += 1
        return v

    def uniform(self, lo, hi):
        return self.u() * (hi - lo) + lo


def scalar_slice_sample(logpdf, niter, w, xval, key, nburn=1, stats=None):
    """util.slice_sample step for step, with the counter stream of `key` in place of libc rand / np.random.rand and the
    slice height drawn in log space."""
    xval = np.asarray(xval, dtype=np.float64)
    d = xval.size
    samples = np.empty((niter, d))
    samples[0] = xval
    rng = Stream(key)
    i = 0
    while i < niter - 1:
        cur = samples[i]
        height = logpdf(cur)
        if height == -np.inf:
            raise RuntimeError("zero probability encountered")
        with np.errstate(divide="ignore"):
            logy = height + np.log(rng.u())                 # log(uniform(0, exp(height))) without overflow
        direction = np.array([rng.u() for _ in range(d)]) - 0.5
        nrm = direction[0] * direction[0]
        for c in range(1, d):
            nrm += direction[c] * direction[c]
        direction = direction / np.sqrt(nrm)
        left, right = -w, w
        j = 0
        while logpdf(cur + left * direction) >= logy:
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
            if (right - left) < 1e-9:
                if stats is not None:
                    stats["retries"] = stats.get("retries", 0) + 1
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
    return samples[nburn:]


def counted(f):
    def g(x):
        g.calls += 1
        return f(x)
    g.calls = 0
    return g


def test_counter_stream_is_a_function_of_key_and_counter():
    a = counter_uniform(np.array([5, 5, 6]), np.array([0, 1, 0], dtype=np.uint64))
    b = counter_uniform(np.array([6, 5]), np.array([0, 1], dtype=np.uint64))
    assert a[2] == b[0] and a[1] == b[1] and a[0] != a[1]
    u = counter_uniform(np.full(100000, 11), np.arange(100000, dtype=np.uint64))
    assert (u >= 0).all() and (u < 1).all() and abs(u.mean() - 0.5) < 0.01


def test_batched_sampler_equals_scalar_chains():
    P, n, nburn, w = len(MU), 12, 4, 2.0
    x0 = MU + 0.1 * SD
    x0[BOUNDED] = 0.1
    keys = 1000 + np.arange(P)
    got = slice_sample_batch(toy_batch, x0, n, w, keys, nburn=nburn)
    assert got.shape == (P, n, D)
    for p in range(P):
        want = scalar_slice_sample(toy_chain(p), nburn + n, w, x0[p], keys[p], nburn=nburn)
        assert np.array_equal(got[p], want), "chain %d" % p
    assert (np.abs(got[BOUNDED]) < 0.7).all()


def test_chain_alone_equals_chain_in_batch():
    P, n, w = len(MU), 9, 1.5
    x0 = MU.copy()
    x0[BOUNDED] = -0.2
    keys = 77 + np.arange(P)
    batch = slice_sample_batch(toy_batch, x0, n, w, keys, nburn=2)
    for p in range(P):
        one = lambda X, p=p: gauss(X, MU[p:p + 1], SD[p:p + 1], np.array([p == BOUNDED]))
        alone = slice_sample_batch(one, x0[p:p + 1], n, w, keys[p:p + 1], nburn=2)
        assert np.array_equal(alone[0], batch[p]), "chain %d" % p


def test_step_out_is_capped_at_101_steps_per_side():
    """A flat density never stops the stepping-out: every iteration makes 101 + 101 evaluations, then one proposal
    (any point of the window is accepted); the batched run evaluates the start once and caches accepted densities."""
    n, w = 3, 0.5
    flat = counted(lambda X: np.zeros(len(X)))
    got = slice_sample_batch(flat, np.zeros((1, 2)), n, w, [9], nburn=0)
    assert flat.calls == 1 + (n - 1) * 203
    scalar = counted(lambda x: 0.0)
    want = scalar_slice_sample(scalar, n, w, np.zeros(2), 9, nburn=0)
    assert scalar.calls == (n - 1) * 204
    assert np.array_equal(got[0], want)
    steps = np.diff(got[0], axis=0)
    assert (np.sqrt((steps ** 2).sum(axis=1)) <= 102 * w).all()
    assert (np.sqrt((steps ** 2).sum(axis=1)) > w).any()         # only reachable by stepping out


def hole(x):
    """1-D density that is 0 at the origin, -0.1 on 0.5 <= |x| <= 3 and -inf elsewhere: from the origin every
    shrinkage proposal is rejected when the slice height is above -0.1, so the window collapses and the iteration is
    retried."""
    a = np.abs(x[..., 0])
    return np.where(a == 0, 0.0, np.where((a >= 0.5) & (a <= 3), -0.1, -np.inf))


def test_collapsed_window_retries_the_iteration():
    n, w = 6, 1.0
    keys = []
    for key in range(200):
        stats = {}
        want = scalar_slice_sample(lambda x: float(hole(x[None])[0]), n + 1, w, np.zeros(1), key, nburn=1, stats=stats)
        if stats.get("retries"):
            keys.append((key, want))
        if len(keys) == 3:
            break
    assert keys, "no key collapses a window"
    got = slice_sample_batch(hole, np.zeros((len(keys), 1)), n, w, [k for k, _ in keys], nburn=1)
    for r, (key, want) in enumerate(keys):
        assert np.array_equal(got[r], want), "key %d" % key
        assert (np.abs(got[r]) >= 0.5).all()


def test_zero_probability_start_names_the_chain():
    x0 = MU.copy()
    x0[BOUNDED] = 5.0                                        # outside chain 3's support
    with pytest.raises(RuntimeError, match="chain 3") as ei:
        slice_sample_batch(toy_batch, x0, 2, 1.0, np.arange(len(MU)))
    assert ei.value.chain == BOUNDED


def test_stream_keys_hash_seed_and_problem_as_separate_words():
    k = stream_keys(0, np.arange(4))
    assert len(set(k.tolist())) == 4
    assert stream_keys(1, np.array([0]))[0] != stream_keys(0, np.array([1]))[0]
    assert np.array_equal(stream_keys(7, np.arange(5))[2:], stream_keys(7, np.arange(2, 5)))     # a sub-batch's keys


def test_step_cap_stops_the_slow_chains_at_their_last_point():
    """With max_steps the run stops after that many logpdf calls; a chain that has not finished repeats its last
    accepted point, the finished ones are those of the uncapped run."""
    P, n, w = len(MU), 6, 2.0
    keys = 5 + np.arange(P)
    slow = np.zeros((P, D))
    slow[BOUNDED] = 0.1
    full_stats, cap_stats = {}, {}
    full = slice_sample_batch(toy_batch, slow, n, w, keys, nburn=1, stats=full_stats)
    cap = full_stats["steps"] // 2
    got = slice_sample_batch(toy_batch, slow, n, w, keys, nburn=1, max_steps=cap, stats=cap_stats)
    assert cap_stats["steps"] == cap and cap_stats["unfinished"].size > 0
    for p in range(P):
        if p not in cap_stats["unfinished"]:
            assert np.array_equal(got[p], full[p]), p
            continue
        k = 0                                                  # samples up to the last accepted one are the uncapped run's
        while k < n and np.array_equal(got[p, k], full[p, k]):
            k += 1
        assert k < n and (got[p, k:] == got[p, max(k - 1, 0)]).all(), p
    with pytest.raises(ValueError):
        slice_sample_batch(toy_batch, slow, n, w, keys, max_steps=0)
