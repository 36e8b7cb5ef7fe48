"""BatchBQ with the periodic kernel: the periodic value-and-gradient kernel (bqb_batch_log_lh_grad_periodic) against the
float64 oracle of tests/test_periodic_llgrad_oracle.py and the setup kernel, against central differences of
BatchBQ.log_lh, the model it must leave alone; BatchBQ(kernel=PeriodicKernel) against a loop of BQ objects, host against
device-resident mode, fit_hypers and sample_hypers with the period among the parameters."""
import numpy as np
import pytest
from scipy.special import iv

from test_periodic_llgrad_oracle import oracle

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
CLASSES = [16, 64, 128, 160, 256, 512]
LOWER = {16: 4, 64: 17, 128: 65, 160: 129, 256: 161, 512: 257}
PARAMS_TL, PARAMS_L = (3.0, 1.2, 1.0, 0.0), (0.3, 0.8, 1.0, 0.0)     # (h, w, p, s), tests/test_gpu_generic.py
OPT = dict(n_candidate=10, candidate_thresh=0.5, x_mean=0.0, x_var=10.0)


def raw_case(cap, seed):
    """17 instances of class cap: ragged ns, nc = 0 .. 16 candidates between observations, s = 0 in even rows and s != 0
    in odd ones, per-row periods (at least 1, so that no two observations alias); the last three rows are the guard, a
    K_l that is not positive definite and an invalid value."""
    rng = np.random.RandomState(seed)
    B = 17
    ns = np.array([rng.randint(LOWER[cap], cap + 1) for _ in range(B)], dtype=np.int32)
    ns[0], ns[1], ns[B - 2], ns[B - 3] = cap, LOWER[cap], cap, cap
    nc = np.zeros(B, dtype=np.int32)
    x_s, l_s, x_c = np.zeros((B, cap)), np.ones((B, cap)), np.zeros((B, 16))
    hyp, period = np.zeros((B, 6)), np.zeros((B, 2))
    for i in range(B):
        n = int(ns[i])
        gap = 2 * np.pi / n
        x = np.linspace(-np.pi, np.pi, n + 1)[:-1] + rng.uniform(-0.05, 0.05, n) * gap
        perm = rng.permutation(n)                       # unsorted input: the kernel sorts
        x_s[i, :n] = x[perm]
        l_s[i, :n] = (np.exp(1.1 * np.cos(x - 0.1 * i)) * rng.uniform(0.8, 1.2, n) * 0.1)[perm]
        k = rng.choice(n - 1, size=min(i, 16, n - 1), replace=False)
        xc = np.sort(x[k] + 0.5 * gap + 0.1 * gap * rng.uniform(-1, 1, k.size))
        x_c[i, :xc.size], nc[i] = xc, xc.size
        hyp[i] = [3.0 * rng.uniform(0.8, 1.2), 1.2 * gap * rng.uniform(0.9, 1.1), 0.05 * (i % 2),
                  0.3 * rng.uniform(0.8, 1.2), 0.9 * gap * rng.uniform(0.9, 1.1), 1e-3 * (i % 2)]
        period[i] = rng.uniform(1.0, 1.1, 2)            # p >= 1: the observations span at most one period
    hyp[B - 3, 0] = 1e6                                 # "GP mean is too large"
    hyp[B - 2, 4:] = 1e4, 0.0                           # gp_l's kernel is numerically constant: K_l is not PD
    hyp[B - 1, 4] = -1.0                                # invalid value
    return ns, nc, x_s, l_s, x_c, hyp, period


def periodic_batch(B, cap, ns, nc, x_s, l_s, x_c, hyp, period):
    from bayesian_quadrature_b200 import _lib
    from bayesian_quadrature_b200.bq import _vonmises_px
    b = _lib.Batch(B, cap)
    xo = np.linspace(-np.pi, np.pi, 400)
    b.set_approx(1, period=period, xo=xo, p_xo=_vonmises_px(xo, 0.0, 10.0))
    base = np.tile([3.0, 0.3, 0.0, 0.3, 0.2, 0.0], (B, 1))
    b.setup(ns, nc, x_s, l_s, x_c, base, np.tile([0.0, 10.0, 0.5], (B, 1)))
    return b


@pytest.mark.parametrize("cap", CLASSES)
def test_periodic_gradient_vs_oracle_and_setup(cap):
    from bayesian_quadrature_b200 import _lib
    ns, nc, x_s, l_s, x_c, hyp, period = raw_case(cap, seed=cap + 1)
    B = ns.size
    b = periodic_batch(B, cap, ns, nc, x_s, l_s, x_c, hyp, period)
    ll, grad, st = b.log_lh_grad_periodic(hyp, period)
    assert grad.shape == (B, 8)
    b.set_hypers(hyp)
    b.set_periods(period)
    info = b.setup_device(check_max=True)
    assert np.array_equal(st, info["status"]), (st, info["status"])
    assert st[B - 3] == _lib.SETUP_MEAN_TOO_LARGE and st[B - 2] == _lib.SETUP_KL_NOTPD and st[B - 1] == _lib.SETUP_BAD_INPUT
    ok = st == _lib.SETUP_OK
    assert ok.sum() >= B - 3
    assert np.isneginf(ll[~ok]).all() and np.isnan(grad[~ok]).all()
    assert np.allclose(ll[ok], info["log_lh"][ok], rtol=1e-12, atol=0), np.abs(ll - info["log_lh"])[ok].max()
    for i in range(B - 1):
        want_st, want_ll, want_g, mag, cond = oracle(x_s[i, :ns[i]], l_s[i, :ns[i]], x_c[i, :nc[i]], hyp[i], period[i])
        assert st[i] == want_st, (i, st[i], want_st)
        if want_st != _lib.SETUP_OK:
            continue
        assert np.isclose(ll[i], want_ll, rtol=1e-9 + 16 * EPS * cond, atol=0), (i, ll[i], want_ll, cond)
        tol = 1e-9 * np.abs(want_g) + 16 * EPS * cond * mag
        assert (np.abs(grad[i] - want_g) <= tol).all(), (i, ns[i], nc[i], grad[i], want_g, tol, cond)
    # one instance gives the same bits whatever rows it is evaluated with
    sel = np.array([5, 0, 5, 9], dtype=np.int32)
    ll2, g2, _ = b.log_lh_grad_periodic(hyp[sel], period[sel], inst=sel)
    assert np.array_equal(ll2, ll[sel]) and np.array_equal(g2, grad[sel])
    bad = period.copy()
    bad[3, 1] = 0.0
    assert b.log_lh_grad_periodic(hyp, bad)[2][3] == _lib.SETUP_BAD_INPUT
    b.close()


def test_periodic_entry_points_refuse_the_gaussian_batch():
    from bayesian_quadrature_b200 import _lib
    ns, nc, x_s, l_s, x_c, hyp, period = raw_case(16, seed=3)
    B = ns.size
    b = _lib.Batch(B, 16)
    with pytest.raises(_lib.BQB200Error):
        b.log_lh_grad_periodic(hyp, period)                          # nothing staged
    b.setup(ns, nc, x_s, l_s, x_c, np.tile([3.0, 0.3, 0.0, 0.3, 0.2, 0.0], (B, 1)), np.tile([0.0, 10.0, 0.5], (B, 1)))
    with pytest.raises(NotImplementedError):
        b.log_lh_grad_periodic(hyp, period)
    with pytest.raises(_lib.BQB200Error):
        b.set_periods(period)
    b.seed_candidates(np.arange(B))
    with pytest.raises(_lib.BQB200Error):
        b.draw_candidates_wrapped(8)
    b.set_approx(1, period=period)
    with pytest.raises(NotImplementedError):
        b.log_lh_grad(hyp)                                            # the Gaussian entry point keeps refusing
    b.close()


def vonmises(mu, kappa):
    return lambda x: np.exp(-np.log(2 * np.pi * iv(0, kappa)) + kappa * np.cos(np.asarray(x) - mu))


def make_batch(P=4, seed=11, device_resident=False, params_tl=PARAMS_TL, params_l=PARAMS_L, ns_reserve=8):
    from bayesian_quadrature_b200 import BatchBQ, PeriodicKernel
    x0 = np.linspace(-np.pi, np.pi, 6)[:-1]
    fl = [vonmises(0.3 * p - 0.4, 1.1 + 0.2 * p) for p in range(P)]
    bb = BatchBQ(np.tile(x0, (P, 1)), np.stack([f(x0) for f in fl]), params_tl, params_l, seed=seed, ns_reserve=ns_reserve,
                 device_resident=device_resident, kernel=PeriodicKernel, **OPT)
    return bb, fl


def bq_objects(bb, fl, seed):
    """The single-problem BQ object of every problem, each initialised from the global RNG seeded with seed + p; returns
    them with the RNG state each one continues from."""
    from bayesian_quadrature_b200 import BQ, PeriodicKernel
    x0 = np.linspace(-np.pi, np.pi, 6)[:-1]
    bqs, states = [], []
    for p in range(bb.P):
        np.random.seed(seed + p)
        bq = BQ(x0, fl[p](x0), kernel=PeriodicKernel, optim_method="L-BFGS-B", **OPT)
        bq.init(params_tl=PARAMS_TL, params_l=PARAMS_L)
        bqs.append(bq)
        states.append(np.random.get_state())
    return bqs, states


def test_batch_rounds_equal_a_loop_of_bq_objects():
    seed, params = 11, ["h", "w", "p"]
    bb, fl = make_batch(seed=seed)
    bqs, states = bq_objects(bb, fl, seed)
    grid = np.linspace(-np.pi, np.pi, 301)[:-1]         # pi and -pi are one point of the circle
    for rnd in range(3):
        for p, bq in enumerate(bqs):
            n, c = int(bb.ns[p]), int(bb.nc[p])
            assert n == bq.ns and np.array_equal(bb.x_s[p, :n], bq.x_s), (rnd, p)
            assert c == bq.nc and np.array_equal(bb.x_c[p, :c], bq.x_c), (rnd, p)
            assert np.array_equal(bb.xo[p], bq._approx_x) and np.array_equal(bb.p_xo[p], bq._approx_px), (rnd, p)
            assert bb.Z_mean()[p] == bq.Z_mean() and bb.Z_var()[p] == bq.Z_var(), (rnd, p)
        esm, _, _ = bb.batch.score_host(grid)
        idx, x_next = bb.choose_next(grid)
        for p, bq in enumerate(bqs):
            e1, _, _ = bq._device_model().batch.score_host(grid)
            assert np.array_equal(e1[0], esm[p]), (rnd, p)
            assert int(np.argmax(bq.expected_squared_mean(grid))) == int(idx[p]), (rnd, p)
        l_new = np.array([fl[p](x_next[p]) for p in range(bb.P)])
        bb.add_observations(x_next, l_new)
        for p, bq in enumerate(bqs):
            np.random.set_state(states[p])
            bq.add_observation(float(x_next[p]), float(l_new[p]))
            states[p] = np.random.get_state()
    # log_lh with the period among the parameters (BQ._make_llh_params) and the marginal loss, problem by problem
    rs = np.random.RandomState(5)
    S = 3
    base_tl = np.array([PARAMS_TL[:3]] * bb.P)
    base_l = np.array([PARAMS_L[:3]] * bb.P)
    htl = base_tl[:, None, :] * rs.uniform(0.85, 1.15, (bb.P, S, 3))
    hl = base_l[:, None, :] * rs.uniform(0.85, 1.15, (bb.P, S, 3))
    loss = bb.marginal_loss(grid, htl, hl, params).cpu().numpy()
    for p, bq in enumerate(bqs):
        want, batch = bq.marginal_loss(grid, htl[p], hl[p], params)
        batch.close()
        assert np.array_equal(loss[p], want.cpu().numpy()), p
    got = bb.log_lh(htl[:, 0], hl[:, 0], params)
    for p, bq in enumerate(bqs):
        want = bq._make_llh_params(params)(np.concatenate([htl[p, 0], hl[p, 0]]))
        assert np.isclose(got[p], want, rtol=1e-12, atol=0), (p, got[p], want)
    bb.close()


def test_host_and_device_resident_rounds_agree():
    import torch
    host, fl = make_batch(seed=21)
    dev, _ = make_batch(seed=21, device_resident=True)
    grid = np.linspace(-np.pi, np.pi, 257)[:-1]         # pi and -pi are one point of the circle
    for rnd in range(4):
        dev.sync_host()
        assert np.array_equal(dev.ns, host.ns) and np.array_equal(dev.nc, host.nc), rnd
        for p in range(host.P):
            c = int(host.nc[p])
            assert np.array_equal(dev.x_c[p, :c], host.x_c[p, :c]), (rnd, p)
        assert np.array_equal(dev.Z_mean(), host.Z_mean()) and np.array_equal(dev.Z_var(), host.Z_var()), rnd
        if rnd == 3:                                    # one marginalised round: sample_hypers and marginal_loss in both modes
            idx_h, x_h = host.choose_next(grid, n=2, params=["h", "w", "p"], seed=7)
            idx_d, x_d = dev.choose_next(torch.from_numpy(grid).cuda(), on_device=True, n=2, params=["h", "w", "p"], seed=7)
        else:
            idx_h, x_h = host.choose_next(grid)
            idx_d, x_d = dev.choose_next(torch.from_numpy(grid).cuda(), on_device=True)
        assert np.array_equal(idx_d.cpu().numpy(), idx_h) and np.array_equal(x_d.cpu().numpy(), x_h), rnd
        l_new = np.array([fl[p](x_h[p]) for p in range(host.P)])
        host.add_observations(x_h, l_new)
        dev.add_observations(x_d, torch.from_numpy(l_new).cuda())
    host.close()
    dev.close()


def fd_log_grad(bb, params, X, delta=1e-4):
    k = len(params)
    out = np.empty_like(X)
    for c in range(2 * k):
        lo, hi = X.copy(), X.copy()
        lo[:, c] *= np.exp(-delta)
        hi[:, c] *= np.exp(delta)
        out[:, c] = (bb.log_lh(hi[:, :k], hi[:, k:], params) - bb.log_lh(lo[:, :k], lo[:, k:], params)) / (2 * delta)
    return out


def test_gradient_matches_central_differences_in_all_eight_directions():
    params = ["h", "w", "p", "s"]
    bb, _ = make_batch(params_tl=(3.0, 1.2, 1.0, 0.05), params_l=(0.3, 0.8, 1.0, 1e-3))
    assert (bb.nc > 0).all()                            # the l_c chain is exercised
    rows = bb._rows()
    X = np.concatenate([rows[:, [0, 1, 6, 2]], rows[:, [3, 4, 7, 5]]], axis=1)
    X[:, [0, 2, 5]] *= np.array([1.1, 0.95, 1.05])      # away from the start
    ll, gtl, gl = bb.log_lh_grad(X[:, :4], X[:, 4:], params)
    assert np.allclose(ll, bb.log_lh(X[:, :4], X[:, 4:], params), rtol=1e-12, atol=0)
    got = np.concatenate([gtl, gl], axis=1) * X
    fd = fd_log_grad(bb, params, X)
    tol = 1e-5 * np.abs(fd) + 1e-6 * np.maximum(1, np.abs(ll))[:, None]
    assert (np.abs(got - fd) <= tol).all(), (got, fd)
    bb.close()


def test_log_lh_grad_leaves_the_model_untouched():
    bb, _ = make_batch()
    grid = np.linspace(-np.pi, np.pi, 401)
    idx0, _ = bb.choose_next(grid)
    esm0 = bb._esm.clone()
    zm0, zv0 = bb.Z_mean().copy(), bb.Z_var().copy()
    m0 = [bb.batch.read_model(p) for p in range(bb.P)]
    rows = bb._rows()
    for scale in (0.9, 1.2, 1e6):
        bb.log_lh_grad(rows[:, [0, 1, 6]] * scale, rows[:, [3, 4, 7]] * scale, ["h", "w", "p"])
    for p in range(bb.P):
        assert np.array_equal(bb.batch.read_model(p), m0[p])
    assert np.array_equal(bb.Z_mean(), zm0) and np.array_equal(bb.Z_var(), zv0)
    idx1, _ = bb.choose_next(grid)
    assert np.array_equal(idx0, idx1) and np.array_equal(esm0.cpu().numpy(), bb._esm.cpu().numpy())
    bb.close()


def test_fit_hypers_with_the_period():
    from bayesian_quadrature_b200 import BatchBQ, PeriodicKernel
    params = ["h", "w", "p"]
    ptl, pl = (3.0, 1.2, 1.0, 0.1), (0.3, 0.8, 1.0, 1e-3)
    bb, _ = make_batch(params_tl=ptl, params_l=pl)
    bd, _ = make_batch(params_tl=ptl, params_l=pl, device_resident=True)
    bd.sync_host()
    assert np.array_equal(bd.x_c, bb.x_c)
    k = len(params)
    X0 = np.concatenate([bb._rows()[:, [0, 1, 6]], bb._rows()[:, [3, 4, 7]]], axis=1)
    ll0 = bb.log_lh(X0[:, :k], X0[:, k:], params)
    singles = []
    for p in range(bb.P):
        n, c = int(bb.ns[p]), int(bb.nc[p])
        one = BatchBQ(bb.x_s[p:p + 1, :n], bb.l_s[p:p + 1, :n], ptl, pl, ns_reserve=bb.cap - n, kernel=PeriodicKernel, **OPT)
        one.x_c[:], one.nc[:] = bb.x_c[p], c                 # the batch's candidates
        one._check_info(one.batch.setup(one.ns, one.nc, one.x_s, one.l_s, one.x_c, one.hyp, one.prior))
        singles.append(one)
    res = bb.fit_hypers(params, maxiter=60)
    rd = bd.fit_hypers(params, maxiter=60)
    assert np.array_equal(bb.hyp, bd.hyp) and np.array_equal(bb.period, bd.period)
    assert np.array_equal(res["log_lh"], rd["log_lh"])
    assert (res["log_lh"] >= ll0).all(), (res["log_lh"], ll0)
    assert not np.array_equal(bb.period[:, 0], np.full(bb.P, ptl[2]))         # the period moved
    X = np.concatenate([bb._rows()[:, [0, 1, 6]], bb._rows()[:, [3, 4, 7]]], axis=1)
    assert np.allclose(res["log_lh"], bb.log_lh(X[:, :k], X[:, k:], params), rtol=1e-12, atol=0)
    for p, one in enumerate(singles):
        r1 = one.fit_hypers(params, maxiter=60)
        assert np.array_equal(one.hyp[0], bb.hyp[p]) and np.array_equal(one.period[0], bb.period[p]), p
        assert r1["log_lh"][0] == res["log_lh"][p] and r1["iterations"][0] == res["iterations"][p]
        one.close()
    bb.close()
    bd.close()


def test_sampler_chains_are_independent_of_the_batch():
    from bayesian_quadrature_b200 import BatchBQ, PeriodicKernel
    params, seed = ["h", "w", "p"], 1000
    bb, fl = make_batch(seed=31)
    htl, hl = bb.sample_hypers(params, n=3, nburn=2, seed=seed)
    assert htl.shape == (bb.P, 3, 3)
    for i in range(3):
        assert np.isfinite(bb.log_lh(htl[:, i], hl[:, i], params)).all()
    x0 = np.linspace(-np.pi, np.pi, 6)[:-1]
    for p in (0, bb.P - 1):
        single = BatchBQ(x0[None], fl[p](x0)[None], PARAMS_TL, PARAMS_L, seed=31 + p, ns_reserve=8, kernel=PeriodicKernel, **OPT)
        assert np.array_equal(single.x_c[0], bb.x_c[p])
        s_tl, s_l = single.sample_hypers(params, n=3, nburn=2, seed=seed, first_problem=p)
        assert np.array_equal(s_tl[0], htl[p]) and np.array_equal(s_l[0], hl[p]), p
        single.close()
    bb.close()
