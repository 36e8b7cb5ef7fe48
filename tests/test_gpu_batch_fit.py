"""The batched hyper-parameter fit: the value-and-gradient kernel of the joint log likelihood (bqb_batch_log_lh_grad)
against a float64 numpy oracle and the setup kernel's log_lh, against central differences, the model it must leave alone,
and BatchBQ.fit_hypers against the single-problem BQ objective and scipy."""
import numpy as np
import pytest
import scipy.optimize as optim

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
MAX_EXPONENT = 707.0101241711442
SQRT_2PI = np.sqrt(2 * np.pi)


def _gram(xa, xb, h, w):
    d = xa[:, None] - xb[None, :]
    return (h * h / (SQRT_2PI * w)) * np.exp(-d * d / (2 * w * w)), d * d


def _gp_terms(K, G, D2, y, h, w, s):
    """log_lh of one GP and, per parameter (h, w, s), the pieces of its derivative: 1/2 a' Kd a - 1/2 tr(K^-1 Kd)."""
    n = K.shape[0]
    L = np.linalg.cholesky(K)
    Ki = np.linalg.inv(K)
    a = Ki @ y
    ll = -0.5 * y @ a - np.log(np.diag(L)).sum() - 0.5 * n * np.log(2 * np.pi)
    Kd = [2 * G / h, G * D2 / w ** 3 - G / w, 2 * s * np.eye(n)]
    terms = [(0.5 * a @ M @ a, -0.5 * np.trace(Ki @ M)) for M in Kd]
    return ll, a, Ki, Kd, terms, np.linalg.cond(K)


def oracle(x_s, l_s, x_c, hyp, check_max=True):
    """(status, log_lh, grad [6], magnitude [6], cond) of the joint log likelihood from the formulas, in float64."""
    from bayesian_quadrature_b200 import _lib
    h_t, w_t, s_t, h_l, w_l, s_l = hyp
    ns, nc = x_s.size, x_c.size
    G, D2 = _gram(x_s, x_s, h_t, w_t)
    y = np.log(l_s)
    try:
        ll_t, a, Ki, Kd, terms_t, cond_t = _gp_terms(G + s_t ** 2 * np.eye(ns), G, D2, y, h_t, w_t, s_t)
    except np.linalg.LinAlgError:
        return _lib.SETUP_KTL_NOTPD, -np.inf, None, None, None
    kc, dc2 = _gram(x_c, x_s, h_t, w_t)
    m = kc @ a
    if check_max and nc:
        V = np.maximum(h_t * h_t / (SQRT_2PI * w_t) - np.einsum("ij,jk,ik->i", kc, Ki, kc), 0)
        if (m + 2 * np.sqrt(V) > MAX_EXPONENT).any():
            return _lib.SETUP_MEAN_TOO_LARGE, -np.inf, None, None, None
    l_c = np.exp(m)
    x_sc, l_sc = np.concatenate([x_s, x_c]), np.concatenate([l_s, l_c])
    Gl, Dl2 = _gram(x_sc, x_sc, h_l, w_l)
    try:
        np.linalg.cholesky(Gl)
        ll_l, al, _, _, terms_l, cond_l = _gp_terms(Gl + s_l ** 2 * np.eye(ns + nc), Gl, Dl2, l_sc, h_l, w_l, s_l)
    except np.linalg.LinAlgError:
        return _lib.SETUP_KL_NOTPD, -np.inf, None, None, None
    gam = al[ns:] * l_c
    kd = [2 * kc / h_t, kc * dc2 / w_t ** 3 - kc / w_t, np.zeros_like(kc)]
    grad, mag = np.empty(6), np.empty(6)
    for i in range(3):
        u, v = kd[i] @ a, kc @ (Ki @ (Kd[i] @ a))
        grad[i] = sum(terms_t[i]) - (gam * (u - v)).sum()
        mag[i] = np.abs(terms_t[i]).sum() + (np.abs(gam) * (np.abs(u) + np.abs(v))).sum()
        grad[3 + i] = sum(terms_l[i])
        mag[3 + i] = np.abs(terms_l[i]).sum()
    return _lib.SETUP_OK, ll_t + ll_l, grad, mag, max(cond_t, cond_l)


CLASSES = [16, 64, 128, 160, 256, 512]
LOWER = {16: 2, 64: 17, 128: 65, 160: 129, 256: 161, 512: 257}     # (the synthetic likelihood needs ns >= 2)


def raw_case(cap, seed):
    """17 instances of class cap: ragged ns within the class, nc = 0 .. 16 candidates at midpoints between observations,
    s = 0 in even rows and s != 0 in odd ones; plus, in the last three rows, the guard, a K_l that is not positive definite
    and an invalid value."""
    from bayesian_quadrature_b200 import synthetic
    rng = np.random.RandomState(seed)
    B = 17
    lo = LOWER[cap]
    ns = np.array([rng.randint(lo, cap + 1) for _ in range(B)], dtype=np.int32)
    ns[0], ns[1], ns[B - 2] = cap, lo, cap
    nc = np.arange(B, dtype=np.int32)
    x_s, l_s, x_c = np.zeros((B, cap)), np.ones((B, cap)), np.zeros((B, 16))
    for i in range(B):
        x, l = synthetic.observations(int(ns[i]), synthetic.problem_shift(i))
        perm = rng.permutation(ns[i])                  # unsorted input: the kernel sorts
        x_s[i, :ns[i]], l_s[i, :ns[i]] = x[perm], l[perm]
        if nc[i]:
            k = rng.choice(max(int(ns[i]) - 1, 1), size=min(int(nc[i]), max(int(ns[i]) - 1, 1)), replace=False)
            xc = np.sort(np.sort(x)[k] + 0.625 + 0.2 * rng.uniform(-1, 1, k.size))
            x_c[i, :xc.size] = xc
            nc[i] = xc.size
    hs = synthetic.hyper_sets(B, seed=seed)
    hyp = np.stack([hs[:, 0], hs[:, 1], np.where(np.arange(B) % 2, 0.05, 0.0),
                    hs[:, 2], hs[:, 3], np.where(np.arange(B) % 2, 1e-3, 0.0)], axis=1)
    hyp[B - 3, 0] = 1e6                                # "GP mean is too large"
    hyp[B - 2, 4:] = 1e4, 0.0                          # length scale >> data span: K_l has numerical rank of a few, and
                                                       # dozens of its pivots are rounding noise, so it is not PD
    hyp[B - 1, 4] = -1.0                               # invalid value
    return ns, nc, x_s, l_s, x_c, hyp


@pytest.mark.parametrize("cap", CLASSES)
def test_value_and_gradient_vs_oracle_and_setup(cap):
    from bayesian_quadrature_b200 import _lib
    ns, nc, x_s, l_s, x_c, hyp = raw_case(cap, seed=cap)
    B = ns.size
    prior = np.tile([0.0, 100.0, 0.5], (B, 1))
    b = _lib.Batch(B, cap)
    base = np.tile([15.0, 2.0, 0.0, 0.2, 1.3, 0.0], (B, 1))
    b.setup(ns, nc, x_s, l_s, x_c, base, prior)
    ll, grad, st = b.log_lh_grad(hyp)
    # the setup kernel's log_lh under the same rows (BatchBQ.log_lh's path)
    b.set_hypers(hyp)
    info = b.setup_device(check_max=True)
    assert np.array_equal(st, info["status"]), (st, info["status"])
    assert st[B - 3] == _lib.SETUP_MEAN_TOO_LARGE and st[B - 2] == _lib.SETUP_KL_NOTPD and st[B - 1] == _lib.SETUP_BAD_INPUT
    ok = st == _lib.SETUP_OK
    assert np.isneginf(ll[~ok]).all() and np.isnan(grad[~ok]).all()
    assert np.allclose(ll[ok], info["log_lh"][ok], rtol=1e-12, atol=0), np.abs(ll - info["log_lh"])[ok].max()
    for i in range(B):
        want_st, want_ll, want_g, mag, cond = oracle(x_s[i, :ns[i]], l_s[i, :ns[i]], x_c[i, :nc[i]], hyp[i]) \
            if hyp[i, 4] > 0 else (_lib.SETUP_BAD_INPUT, -np.inf, None, None, None)
        assert st[i] == want_st, (i, st[i], want_st)
        if want_st != _lib.SETUP_OK:
            continue
        assert np.isclose(ll[i], want_ll, rtol=1e-9 + 4 * EPS * cond, atol=0), (i, ll[i], want_ll, cond)
        tol = 1e-9 * np.abs(want_g) + 16 * EPS * cond * mag
        assert (np.abs(grad[i] - want_g) <= tol).all(), (i, ns[i], nc[i], grad[i], want_g, tol, cond)
    # one instance gives the same bits whatever rows it is evaluated with
    sel = np.array([5, 0, 5, 9], dtype=np.int32)
    ll2, g2, _ = b.log_lh_grad(hyp[sel], inst=sel)
    assert np.array_equal(ll2, ll[sel]) and np.array_equal(g2, grad[sel])
    b.close()


def make_batch(P=4, ns0=20, device_resident=False, s=0.0, seed=31):
    """P problems with different ns (problem p gets P - 1 - p appended observations), as tests/test_gpu_batch_marginal."""
    from bayesian_quadrature_b200 import BatchBQ, synthetic
    x0, _ = synthetic.observations(ns0)
    fl = [synthetic.likelihood(ns0, synthetic.problem_shift(p)) for p in range(P)]
    opt = synthetic.options(ns0)
    ptl, pl = list(synthetic.PARAMS_TL), list(synthetic.PARAMS_L)
    ptl[2], pl[2] = s, s * 1e-2
    bb = BatchBQ(np.tile(x0, (P, 1)), np.stack([f(x0) for f in fl]), ptl, pl, opt["n_candidate"], opt["candidate_thresh"],
                 opt["x_mean"], opt["x_var"], seed=seed, ns_reserve=8, device_resident=device_resident)
    for r in range(P - 1):
        bb.sync_host()
        x_new = np.where(np.arange(P) <= r, x0.max() + 1.25 * (r + 1), bb.x_s[:, 0] + 0.1)
        bb.add_observations(x_new, np.array([fl[p](x_new[p]) for p in range(P)]))
    bb.sync_host()
    return bb, opt


def bq_of(bb, p, opt):
    """The single-problem BQ object of problem p under the batch's current hyper-parameters and candidates."""
    from bayesian_quadrature_b200 import BQ, GaussianKernel
    bb.sync_host()
    n, c = int(bb.ns[p]), int(bb.nc[p])
    bq = BQ(bb.x_s[p, :n].copy(), bb.l_s[p, :n].copy(), kernel=GaussianKernel, **opt)
    bq.init(params_tl=tuple(bb.hyp[p, :3]), params_l=tuple(bb.hyp[p, 3:]))
    bq.x_c, bq.nc = bb.x_c[p, :c].copy(), c
    return bq


def fd_log_grad(bb, params, X, delta=1e-4):
    """Central differences of BatchBQ.log_lh in the logarithms of the parameters at X = [P, 2k] (tl then l)."""
    k = len(params)
    out = np.empty_like(X)
    for c in range(2 * k):
        lo, hi = X.copy(), X.copy()
        lo[:, c] *= np.exp(-delta)
        hi[:, c] *= np.exp(delta)
        out[:, c] = (bb.log_lh(hi[:, :k], hi[:, k:], params) - bb.log_lh(lo[:, :k], lo[:, k:], params)) / (2 * delta)
    return out


def test_gradient_matches_central_differences_of_log_lh():
    params = ["h", "w", "s"]
    bb, _ = make_batch(P=4, s=0.3)
    k = len(params)
    X = np.concatenate([bb.hyp[:, :3], bb.hyp[:, 3:]], axis=1)
    X[:, [0, 3]] *= np.array([1.1, 1.5])               # away from the start, where l_c moves with the tl parameters
    ll, gtl, gl = bb.log_lh_grad(X[:, :k], X[:, k:], params)
    assert np.allclose(ll, bb.log_lh(X[:, :k], X[:, k:], params), rtol=1e-12, atol=0)
    assert (bb.nc > 0).any()                             # the l_c chain is exercised
    got = np.concatenate([gtl, gl], axis=1) * X
    fd = fd_log_grad(bb, params, X)
    tol = 1e-5 * np.abs(fd) + 1e-6 * np.maximum(1, np.abs(ll))[:, None]
    assert (np.abs(got - fd) <= tol).all(), (got, fd)
    bb.close()


def test_log_lh_grad_leaves_the_model_untouched():
    import torch
    bb, _ = make_batch(P=4)
    grid = torch.from_numpy(np.linspace(-25, 25, 2001)).cuda()
    idx0, _ = bb.choose_next(grid)
    esm0 = bb._esm.clone()
    zm0, zv0 = bb.Z_mean().copy(), bb.Z_var().copy()
    m0 = [bb.batch.read_model(p) for p in range(bb.P)]
    for scale in (0.9, 1.2, 1e6):
        bb.log_lh_grad(bb.hyp[:, :2] * scale, bb.hyp[:, 3:5] * scale, ["h", "w"])
    for p in range(bb.P):
        assert np.array_equal(bb.batch.read_model(p), m0[p])
    assert np.array_equal(bb.Z_mean(), zm0) and np.array_equal(bb.Z_var(), zv0)
    idx1, _ = bb.choose_next(grid)
    assert np.array_equal(idx0, idx1) and torch.equal(esm0, bb._esm)
    bb.close()


def test_fit_hypers_against_bq_objective_and_scipy():
    params = ["h", "w"]
    bb, opt = make_batch(P=4, s=0.1)                         # with s = 0 the likelihood grows without bound (DESIGN 8.2)
    start = [bq_of(bb, p, opt) for p in range(bb.P)]
    x0 = np.concatenate([bb.hyp[:, :2], bb.hyp[:, 3:5]], axis=1)
    res = bb.fit_hypers(params)
    assert res["evaluations"] >= bb.P and (res["iterations"] >= 1).all()
    X = np.concatenate([bb.hyp[:, :2], bb.hyp[:, 3:5]], axis=1)
    assert np.allclose(res["log_lh"], bb.log_lh(X[:, :2], X[:, 2:], params), rtol=1e-12, atol=0)
    for p in range(bb.P):
        f = start[p]._make_llh_params(params)
        assert np.isclose(f(X[p]), res["log_lh"][p], rtol=1e-9, atol=0)
        ref = optim.minimize(lambda x: -f(x), x0[p], method="L-BFGS-B")
        assert res["log_lh"][p] >= -ref.fun - 1e-7 * max(1.0, abs(ref.fun)), (p, res["log_lh"][p], -ref.fun)
    fd = fd_log_grad(bb, params, X)
    assert (np.abs(fd) <= 1e-3 * np.maximum(1, np.abs(res["log_lh"]))[:, None]).all(), (fd, res)
    bb.close()


def test_fit_hypers_rows_are_independent_and_modes_agree():
    from bayesian_quadrature_b200 import BatchBQ
    params = ["h", "w"]
    bb, opt = make_batch(P=4, s=0.1)
    bd, _ = make_batch(P=4, device_resident=True, s=0.1)
    singles = []
    for p in range(bb.P):
        n, c = int(bb.ns[p]), int(bb.nc[p])
        one = BatchBQ(bb.x_s[p:p + 1, :n], bb.l_s[p:p + 1, :n], bb.hyp[p, :3], bb.hyp[p, 3:], opt["n_candidate"],
                      opt["candidate_thresh"], opt["x_mean"], opt["x_var"], ns_reserve=bb.cap - n)
        one.x_c[:], one.nc[:] = bb.x_c[p], c                 # the batch's candidates
        one._check_info(one.batch.setup(one.ns, one.nc, one.x_s, one.l_s, one.x_c, one.hyp, one.prior))
        singles.append(one)
    res = bb.fit_hypers(params)
    rd = bd.fit_hypers(params)
    assert np.array_equal(bb.hyp, bd.hyp) and np.array_equal(res["log_lh"], rd["log_lh"])
    for p, one in enumerate(singles):
        r1 = one.fit_hypers(params)
        assert np.array_equal(one.hyp[0], bb.hyp[p]), (p, one.hyp[0], bb.hyp[p])
        assert r1["log_lh"][0] == res["log_lh"][p] and r1["iterations"][0] == res["iterations"][p]
        assert res["converged"][p]
        one.close()
    # the refreshed model is that of BQ objects set up under the fitted hyper-parameters, with the same candidates
    for p in range(bb.P):
        bq = bq_of(bb, p, opt)
        assert np.isclose(bb.Z_mean()[p], bq.Z_mean(), rtol=1e-9, atol=0)
        assert np.isclose(bb.Z_var()[p], bq.Z_var(), rtol=1e-7, atol=1e-13)
    bb.close()
    bd.close()


def test_fit_hypers_errors():
    from bayesian_quadrature_b200 import _lib
    bb, _ = make_batch(P=3)
    hyp0 = bb.hyp.copy()
    with pytest.raises(ValueError, match="positive"):
        bb.fit_hypers(["h", "s"])                            # s = 0 cannot be fitted in log-space
    bb.hyp[1, 0] = 1e6                                       # "GP mean is too large" at the start of problem 1
    with pytest.raises(RuntimeError, match="problem 1"):
        bb.fit_hypers(["w"])
    bb.hyp[1, 0] = hyp0[1, 0]
    assert np.array_equal(bb.hyp, hyp0)
    b = _lib.Batch(2, 16)
    with pytest.raises(_lib.BQB200Error):
        b.log_lh_grad(np.ones((2, 6)))                       # nothing staged
    b.close()
    bb.batch.set_approx(kernel_kind=1, period=np.ones((bb.P, 2)))
    with pytest.raises(NotImplementedError):
        bb.log_lh_grad(bb.hyp[:, :1], bb.hyp[:, 3:4], ["h"])
    bb.close()
