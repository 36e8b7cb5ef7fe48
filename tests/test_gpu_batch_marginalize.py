"""BatchBQ.marginalize against BQ.marginalize on a loop of BQ objects (every quantity, every capacity class, the periodic
kernel, sampled s_l, shared and per-problem grids, a pre-sorted grid, a NaN point, small chunks), its modes, state,
sampling and errors; the tie-break kernel (bqb_argmin_ties_rows_device) against a numpy statement of the reference's rule;
and choose_next(deterministic=False)."""
import numpy as np
import pytest

from conftest import assert_close
from test_gpu_batch_readout import gaussian_case, periodic_case

pytestmark = pytest.mark.gpu

PARAMS = ["h", "w"]
NO_INDEX = 0x7fffffffffffffff
SCORED = ("expected_Z_var", "expected_squared_mean", "expected_mean", "expected_squared_mean_and_mean")
PREDICTED = ("l_mean", "l_var")


def sample_rows(bb, params, S, seed, spread=0.05):
    """[P, S, k] samples around each problem's own hyper-parameters (log-normal factors)."""
    rng = np.random.RandomState(seed)
    rows = bb._rows()
    cols = [{"h": (0, 3), "w": (1, 4), "s": (2, 5), "p": (6, 7)}[n] for n in params]
    htl = np.stack([rows[:, c[0]] for c in cols], axis=-1)[:, None, :] * np.exp(spread * rng.randn(bb.P, S, len(params)))
    hl = np.stack([rows[:, c[1]] for c in cols], axis=-1)[:, None, :] * np.exp(spread * rng.randn(bb.P, S, len(params)))
    return np.ascontiguousarray(htl), np.ascontiguousarray(hl)


def bq_marginalize(monkeypatch, bq, funs, htl, hl, params, x_of):
    """BQ.marginalize of the same quantities with sample_hypers returning the given samples."""
    monkeypatch.setattr(bq, "sample_hypers", lambda params, n=1, nburn=10: (htl, hl))
    calls = []
    for f in funs:
        if isinstance(f, str):
            calls.append(getattr(bq, f))
        else:
            calls.append((lambda name, x: (lambda: getattr(bq, name)(x)))(f[0], x_of(f[1])))
    return bq.marginalize(calls, htl.shape[0], params)


def check_parity(monkeypatch, bb, bqs, funs, htl, hl, params, x_rows, host_rounds, what, on_device=False):
    import torch
    got = bb.marginalize(funs, params=params, hypers=(htl, hl), on_device=on_device)
    assert len(got) == len(funs)
    for p, bq in enumerate(bqs):
        x_of = lambda x: x_rows[id(x)] if x_rows[id(x)].ndim == 1 else x_rows[id(x)][p]
        want = bq_marginalize(monkeypatch, bq, funs, htl[p], hl[p], params, x_of)
        for f, g, w in zip(funs, got, want):
            name = f if isinstance(f, str) else f[0]
            if isinstance(f, str):
                assert isinstance(g, np.ndarray) and g.shape == (bb.P, htl.shape[1])
            else:
                assert isinstance(g, torch.Tensor) == on_device
            g = g.cpu().numpy() if on_device and not isinstance(f, str) else g
            label = "%s %s problem %d" % (what, name, p)
            if name in PREDICTED and host_rounds:
                nan = np.isnan(w)
                assert np.array_equal(np.isnan(g[p]), nan), label
                assert_close(g[p][~nan], w[~nan], label)
            else:
                assert np.array_equal(g[p], w, equal_nan=True), label
    return got


CASES = [("gauss", 10), ("gauss", 40), ("gauss", 100), ("gauss", 200), ("gauss", 300), ("periodic", 5)]


@pytest.mark.parametrize("kind,ns0", CASES)
def test_marginalize_equals_a_loop_of_bq_marginalize(monkeypatch, kind, ns0):
    import torch
    bb, fl, bq_objects, grid = gaussian_case(ns0) if kind == "gauss" else periodic_case()
    bqs, states = bq_objects()
    params = PARAMS + (["p"] if kind == "periodic" else ["s"])
    per_problem = np.stack([grid + 0.01 * (p + 1) for p in range(bb.P)])
    nan_rows = per_problem.copy()
    nan_rows[2, 7] = np.nan                               # problem 2 alone goes to the host GPs
    x_t = torch.from_numpy(per_problem).cuda()
    x_rows = {id(grid): grid, id(x_t): per_problem, id(nan_rows): nan_rows}
    funs = ["Z_mean", "Z_var"] + [(n, grid) for n in SCORED + PREDICTED] + [(n, x_t) for n in SCORED + PREDICTED] + \
        [("l_mean", nan_rows)]
    if bb._cap_class == 128:                              # an unsorted shared grid that BQ's host entry points pre-sort
        big = np.random.RandomState(3).permutation(np.linspace(grid[0], grid[-1], 8192))
        x_rows[id(big)] = big
        funs += [("expected_Z_var", big), ("expected_squared_mean_and_mean", big)]
    for rnd in range(2):
        htl, hl = sample_rows(bb, params, 3, seed=rnd)
        if kind == "gauss":                               # sampled s: s_l = 0 except for one sample (prediction kernel)
            htl[..., 2] = 0.0
            hl[..., 2] = 0.0
            hl[0, 1, 2] = 1e-3
        before = [bb.batch.read_model(p) for p in range(bb.P)]
        with pytest.raises(ValueError, match="infs or NaNs"):            # gp_log_l.cov of BQ.l_var rejects the NaN too
            bb.marginalize([("l_var", nan_rows)], params=params, hypers=(htl, hl))
        check_parity(monkeypatch, bb, bqs, funs, htl, hl, params, x_rows, rnd > 0, "%s%d round %d" % (kind, ns0, rnd))
        assert all(np.array_equal(a, bb.batch.read_model(p)) for p, a in enumerate(before))
        if rnd == 1:
            break
        idx, x_next = bb.choose_next(grid)
        l_new = np.array([fl[p](x_next[p]) for p in range(bb.P)])
        bb.add_observations(x_next, l_new)
        for p, bq in enumerate(bqs):
            np.random.set_state(states[p])
            bq.add_observation(float(x_next[p]), float(l_new[p]))
            states[p] = np.random.get_state()
    bb.close()


def test_small_chunks_give_the_same_bits():
    import torch
    from bayesian_quadrature_b200 import _lib
    bb, _, _, grid = gaussian_case(40, P=5)
    S = 3
    htl, hl = sample_rows(bb, PARAMS, S, seed=4)
    x_t = torch.from_numpy(np.stack([grid + 0.02 * p for p in range(bb.P)])).cuda()
    funs = ["Z_mean", "Z_var"] + [(n, grid) for n in SCORED + PREDICTED] + [(n, x_t) for n in SCORED + PREDICTED]
    want = bb.marginalize(funs, params=PARAMS, hypers=(htl, hl))
    row_bytes = 8 * grid.size * (2 + 3)                   # the prediction rows of a shared and of a per-problem grid
    model_bytes = 8 * _lib.load().bqb_model_doubles(bb.batch._h) + row_bytes
    bb.MODEL_CHUNK_BYTES = 2 * S * model_bytes            # two problems per setup chunk ...
    bb.LOSS_CHUNK_BYTES = 8 * S * grid.size               # ... one per scoring launch
    assert bb._chunks(S, grid.size, row_bytes) == (2, 1)
    got = bb.marginalize(funs, params=PARAMS, hypers=(htl, hl))
    for f, g, w in zip(funs, got, want):
        assert np.array_equal(g, w), f
    bb.close()


@pytest.mark.parametrize("kind", ["gauss", "periodic"])
def test_modes_agree_and_state_is_untouched(kind):
    import torch
    make = (lambda dr: gaussian_case(40, P=4, device_resident=dr)) if kind == "gauss" else \
        (lambda dr: periodic_case(P=4, device_resident=dr))
    host, fl, _, grid = make(False)
    dev, _, _, _ = make(True)
    params = PARAMS + (["p"] if kind == "periodic" else [])
    g_d = torch.from_numpy(grid).cuda()
    funs_h = ["Z_mean", "Z_var"] + [(n, grid) for n in SCORED + PREDICTED]
    funs_d = ["Z_mean", "Z_var"] + [(n, g_d) for n in SCORED + PREDICTED]
    for rnd in range(2):
        htl, hl = sample_rows(host, params, 2, seed=10 + rnd)
        state = [(bb.hyp.copy(), bb.Z_mean().copy(), bb.Z_var().copy(), [bb.batch.read_model(p) for p in range(bb.P)])
                 for bb in (host, dev)]
        a = host.marginalize(funs_h, params=params, hypers=(htl, hl))
        b = dev.marginalize(funs_d, params=params, hypers=(htl, hl), on_device=True)
        c = host.marginalize(funs_h, params=params, hypers=(htl, hl), on_device=True)
        for f, x, y, z in zip(funs_h, a, b, c):
            y = y if isinstance(f, str) else y.cpu().numpy()
            z = z if isinstance(f, str) else z.cpu().numpy()
            assert np.array_equal(x, y, equal_nan=True) and np.array_equal(x, z, equal_nan=True), (f, rnd)
        for bb, (hyp, zm, zv, models) in zip((host, dev), state):
            assert np.array_equal(bb.hyp, hyp) and np.array_equal(bb.Z_mean(), zm) and np.array_equal(bb.Z_var(), zv)
            assert all(np.array_equal(m, bb.batch.read_model(p)) for p, m in enumerate(models))
        idx, x_h = host.choose_next(grid)
        idx_d, x_d = dev.choose_next(g_d, on_device=True)
        assert np.array_equal(idx_d.cpu().numpy(), idx)
        l_new = np.array([fl[p](x_h[p]) for p in range(host.P)])
        host.add_observations(x_h, l_new)
        dev.add_observations(x_d, torch.from_numpy(l_new).cuda())
    host.close()
    dev.close()


def test_sampling_uses_the_round_seed():
    from bayesian_quadrature_b200 import util
    bb, _, _, grid = gaussian_case(10, P=3)
    funs = ["Z_mean", ("expected_Z_var", grid)]
    got = bb.marginalize(funs, n=2, params=PARAMS, seed=77)
    want = bb.marginalize(funs, params=PARAMS, hypers=bb.sample_hypers(PARAMS, 2, nburn=1, seed=77))
    assert all(np.array_equal(g, w) for g, w in zip(got, want))
    r = bb.__dict__.get("_sample_rounds", 0)
    got = bb.marginalize(funs, n=2, params=PARAMS)        # no seed: the batch's next round seed
    assert bb._sample_rounds == r + 1
    want = bb.marginalize(funs, params=PARAMS, hypers=bb.sample_hypers(PARAMS, 2, nburn=1,
                                                                        seed=int(util.stream_keys(bb.seed, r))))
    assert all(np.array_equal(g, w) for g, w in zip(got, want))
    assert bb._sample_rounds == r + 1                     # given samples draw nothing
    bb.close()


def test_errors_name_the_problem_and_the_sample(monkeypatch):
    bb, _, _, grid = gaussian_case(10, P=3)
    htl, hl = sample_rows(bb, PARAMS, 3, seed=1)
    bad = htl.copy()
    bad[1, 2, 0] = 1e6                                    # "GP mean is too large" in sample 2 of problem 1
    with pytest.raises(np.linalg.LinAlgError, match=r"GP mean is too large \(problem 1, sample 2\)"):
        bb.marginalize(["Z_mean"], params=PARAMS, hypers=(bad, hl))
    bad = htl.copy()
    bad[2, 0, 1] = -1.0
    with pytest.raises(ValueError, match="sample 0 of problem 2"):
        bb.marginalize(["Z_mean"], params=PARAMS, hypers=(bad, hl))
    rows = np.tile(grid, (bb.P, 1))
    rows[2, 17] = np.nan
    for name in SCORED:
        with pytest.raises(ValueError, match="problem 2"):
            bb.marginalize([(name, rows)], params=PARAMS, hypers=(htl, hl))
    with pytest.raises(ValueError, match="expected_Z_var"):
        bb.marginalize(["Z_mean", ("expected_variance", grid)], params=PARAMS, hypers=(htl, hl))
    with pytest.raises(ValueError, match="expected_Z_var"):
        bb.marginalize(["l_mean"], params=PARAMS, hypers=(htl, hl))
    want = bb.marginalize(["Z_mean", ("expected_Z_var", grid)], params=PARAMS, hypers=(htl, hl))
    setup = bb._setup_samples

    def negative_z(hyp, per_setup):                       # what a setup reports for a non-positive Z_mean
        for p0, cp, batch, info in setup(hyp, per_setup):
            if p0 <= 1 < p0 + cp:
                info["Z_mean"][(1 - p0) * hyp.shape[1] + 2] = -1.0
            yield p0, cp, batch, info
    monkeypatch.setattr(bb, "_setup_samples", negative_z)
    with pytest.warns(UserWarning, match=r"m_Z .* \[\(1, 2\)\]") as rec:
        got = bb.marginalize(["Z_mean", ("expected_Z_var", grid)], params=PARAMS, hypers=(htl, hl))
    assert sum("m_Z" in str(w.message) for w in rec) == 1
    assert got[0][1, 2] == -1.0 and np.array_equal(got[1], want[1])   # the values come from the device headers
    bb.close()


# ---------------------------------------------------------------- the tie-break kernel
def ties_np(v, u):
    """The reference's rule (bq.py:664-665) with the uniform u in place of np.random.choice: the k-th point of
    isclose(loss, loss.min()), k = min(floor(u * c), c - 1); NaN never wins the minimum."""
    idx, cnt = [], []
    for row, ur in zip(v, u):
        finite = row[~np.isnan(row)]
        best = finite.min() if finite.size else np.inf
        close = np.nonzero(np.isclose(row, best))[0]
        c = close.size
        cnt.append(c)
        idx.append(close[min(int(np.floor(ur * c)), c - 1)] if c else NO_INDEX)
    return np.array(idx), np.array(cnt)


def run_ties(v, u):
    import torch
    from bayesian_quadrature_b200 import _lib
    rows = v.shape[0]
    b = _lib.Batch(rows, 16)
    mins = torch.empty(rows, dtype=torch.float64, device="cuda")
    idxs = torch.empty(rows, dtype=torch.int64, device="cuda")
    cnts = torch.empty(rows, dtype=torch.int64, device="cuda")
    b.argmin_rows_device(v, mins, idxs)
    first = idxs.clone()
    b.argmin_ties_rows_device(v, mins, torch.from_numpy(np.asarray(u, dtype=np.float64)).cuda(), idxs, cnts)
    b.close()
    return idxs.cpu().numpy(), cnts.cpu().numpy(), first.cpu().numpy()


def boundary_values(m):
    """(largest value np.isclose to m, the next double up) for a finite m."""
    v = m + (1e-8 + 1e-5 * abs(m))
    while not np.isclose(v, m):
        v = np.nextafter(v, -np.inf)
    while np.isclose(np.nextafter(v, np.inf), m):
        v = np.nextafter(v, np.inf)
    return v, np.nextafter(v, np.inf)


@pytest.mark.parametrize("na", [1, 7, 257, 10 ** 5])
def test_tie_kernel_follows_the_numpy_rule(na):
    import torch
    rng = np.random.RandomState(na)
    rows = []
    for m in (-3.7e-3, 0.0, 2.5, -1e12):
        row = m + np.abs(rng.randn(na)) * max(abs(m), 1e-6) + 1e-3
        if na > 1:
            pos = rng.choice(na, size=min(na, 5), replace=False)
            row[pos] = m                                  # exact ties
            if na > 7 and m != 0.0:
                inside, outside = boundary_values(m)
                row[rng.choice(na, 3, replace=False)] = inside
                row[rng.choice(na, 2, replace=False)] = outside
        else:
            row[0] = m
        rows.append(row)
    rows.append(np.full(na, 1.25))                        # all equal
    r = rng.randn(na)
    r[::3] = np.inf
    r[1::5] = np.nan
    rows.append(r)                                        # +inf and NaN entries around a finite minimum
    r = rng.randn(na)
    r[rng.choice(na, min(na, 3), replace=False)] = -np.inf
    rows.append(r)                                        # -inf is the minimum; its copies are the ties
    r = np.full(na, np.inf)
    r[::2] = np.nan
    rows.append(r)                                        # only +inf and NaN
    rows.append(np.full(na, np.nan))                      # no close point
    v = np.stack(rows)
    R = v.shape[0]
    pad = np.full((R, na + 5), -7.0)                      # strided rows: the padding must not be read
    pad[:, 2:na + 2] = v
    v_d = torch.from_numpy(pad).cuda()[:, 2:na + 2]
    for u in (np.zeros(R), np.full(R, 1.0 - 2.0 ** -53), np.random.RandomState(1).rand(R), np.full(R, 0.5)):
        got, cnt, _ = run_ties(v_d, u)
        want, wcnt = ties_np(v, u)
        assert np.array_equal(cnt, wcnt), (na, u)
        assert np.array_equal(got, want), (na, u, got, want)


def test_tie_kernel_choices_are_uniform_over_a_fixed_key_set():
    import torch
    from bayesian_quadrature_b200 import util
    R, c = 4096, 8
    row = np.linspace(1.0, 2.0, 257)
    ties = np.array([3, 40, 41, 100, 128, 200, 255, 256])
    row[ties] = 0.5
    u = util.counter_uniform(util.stream_keys(1234, np.arange(R)), np.uint64(2 ** 64 - 1))
    got, cnt, _ = run_ties(torch.from_numpy(np.tile(row, (R, 1))).cuda(), u)
    want, _ = ties_np(np.tile(row, (R, 1)), u)
    assert (cnt == c).all() and np.array_equal(got, want)
    hits = np.array([(got == t).sum() for t in ties])
    assert hits.sum() == R and (hits > 0).all()
    # counts of a uniform choice: mean 512, standard deviation sqrt(R p (1 - p)) = 21.2; the fixed set sits within 4 of them
    assert (np.abs(hits - R / c) < 4 * np.sqrt(R * (1 / c) * (1 - 1 / c))).all(), hits


def test_tie_kernel_argument_checks():
    import ctypes
    import torch
    from bayesian_quadrature_b200 import _lib
    L = _lib.load()
    b = _lib.Batch(2, 16)
    t = torch.zeros(2, 8, dtype=torch.float64, device="cuda")
    p = ctypes.c_void_p(t.data_ptr())
    f = L.bqb_argmin_ties_rows_device
    assert f(None, p, 8, 8, p, p, p, None, None) == _lib.EINVAL
    assert f(b._h, p, 7, 8, p, p, p, None, None) == _lib.EINVAL     # stride < n
    assert f(b._h, p, 8, 0, p, p, p, None, None) == _lib.EINVAL
    assert f(b._h, p, 8, 8, None, p, p, None, None) == _lib.EINVAL
    assert f(b._h, p, 8, 8, p, None, p, None, None) == _lib.EINVAL
    assert f(b._h, p, 8, 8, p, p, None, None, None) == _lib.EINVAL
    b.close()


# ---------------------------------------------------------------- choose_next(deterministic=False)
def _u(seed, P):
    from bayesian_quadrature_b200 import util
    return util.counter_uniform(util.stream_keys(seed, np.arange(P)), np.uint64(2 ** 64 - 1))


def test_random_choose_next_picks_within_the_isclose_set():
    from test_gpu_batch_marginal import make_batch, sample_sets
    bb, _, _ = make_batch()
    grid = np.linspace(-25, 25, 40001)                    # fine enough for neighbours within rtol of the maximum
    htl, hl = sample_sets(bb.P, 3, seed=3)
    loss = bb.marginal_loss(grid, htl, hl, PARAMS).cpu().numpy()
    idx, x_next = bb.choose_next(grid, hypers=(htl, hl), params=PARAMS, deterministic=False, seed=11)
    want, cnt = ties_np(loss, _u(11, bb.P))
    assert np.array_equal(idx, want) and np.array_equal(x_next, grid[idx]) and (cnt > 1).any(), cnt
    assert all(np.isclose(loss[p, idx[p]], loss[p].min()) for p in range(bb.P))
    again, _ = bb.choose_next(grid, hypers=(htl, hl), params=PARAMS, deterministic=False, seed=11)
    assert np.array_equal(again, idx)
    # another problem's samples change its own loss only
    other = htl.copy()
    other[1:] *= 1.05
    alone, _ = bb.choose_next(grid, hypers=(other, hl), params=PARAMS, deterministic=False, seed=11)
    assert alone[0] == idx[0]
    # the fixed hyper-parameters: the loss is -esm
    r = bb.__dict__.get("_sample_rounds", 0)
    first, _ = bb.choose_next(grid)
    assert bb.__dict__.get("_sample_rounds", 0) == r                 # deterministic calls draw nothing
    esm = bb.expected_squared_mean(grid)
    assert np.array_equal(first, (-esm).argmin(axis=1))              # the default is still the first minimiser
    idx, _ = bb.choose_next(grid, deterministic=False)
    assert bb._sample_rounds == r + 1
    from bayesian_quadrature_b200 import util
    want, cnt = ties_np(-esm, _u(int(util.stream_keys(bb.seed, r)), bb.P))
    assert np.array_equal(idx, want) and (cnt > 1).any(), cnt
    bb.close()


def test_random_choose_next_host_equals_device_resident():
    import torch
    from test_gpu_batch_marginal import make_batch
    host, fl, _ = make_batch(seed=123)
    dev, _, _ = make_batch(seed=123, device_resident=True)
    grid = np.linspace(-25, 25, 20001)
    g_d = torch.from_numpy(grid).cuda()
    for rnd in range(2):
        idx_h, x_h = host.choose_next(grid, n=2, params=PARAMS, deterministic=False)
        idx_d, x_d = dev.choose_next(g_d, on_device=True, n=2, params=PARAMS, deterministic=False)
        assert np.array_equal(idx_d.cpu().numpy(), idx_h) and np.array_equal(x_d.cpu().numpy(), x_h), rnd
        f_h, _ = host.choose_next(grid, deterministic=False)
        f_d, _ = dev.choose_next(g_d, on_device=True, deterministic=False)
        assert np.array_equal(f_d.cpu().numpy(), f_h), rnd
        l_new = np.array([fl[p](x_h[p]) for p in range(host.P)])
        host.add_observations(x_h, l_new)
        dev.add_observations(x_d, torch.from_numpy(l_new).cuda())
    host.close()
    dev.close()
