"""A float64 numpy oracle of the joint log likelihood gp_log_l.log_lh + gp_l.log_lh with the periodic kernel and its eight
derivatives (h, w, s of both GPs, then p_tl, p_l), including the dependence of l_c on the parameters of gp_log_l.  Held
here, without a GPU, to central differences of its own value and to the host GP objects; tests/test_gpu_batch_periodic.py
holds the device kernel to it."""
import numpy as np

MAX_EXPONENT = 707.0101241711442
SETUP_OK, SETUP_KTL_NOTPD, SETUP_KL_NOTPD, SETUP_MEAN_TOO_LARGE = 0, 1, 2, 3


def _gram(xa, xb, h, w, p):
    """G = h^2 exp(-2 sin^2(d / 2p) / w^2), D^2 = 4 sin^2(d / 2p) and F = d sin(d / p) / (w^2 p^2) (so dG/dp = G F)."""
    d = xa[:, None] - xb[None, :]
    D2 = (2 * np.sin(d / (2 * p))) ** 2
    return h * h * np.exp(-D2 / (2 * w * w)), D2, d * np.sin(d / p) / (w * w * p * p)


def _gp_terms(K, G, D2, F, y, h, w, s):
    """log_lh of one GP and, per parameter (h, w, s, p), the two terms 1/2 a' Kd a and -1/2 tr(K^-1 Kd)."""
    n = K.shape[0]
    L = np.linalg.cholesky(K)
    Ki = np.linalg.inv(K)
    a = Ki @ y
    ll = -0.5 * y @ a - np.log(np.diag(L)).sum() - 0.5 * n * np.log(2 * np.pi)
    Kd = [2 * G / h, G * D2 / w ** 3, 2 * s * np.eye(n), G * F]
    terms = [(0.5 * a @ M @ a, -0.5 * np.trace(Ki @ M)) for M in Kd]
    return ll, a, Ki, Kd, terms, np.linalg.cond(K)


def oracle(x_s, l_s, x_c, hyp, period, check_max=True):
    """(status, log_lh, grad [8], magnitude [8], cond) for hyp = (h, w, s of gp_log_l, then of gp_l) and period =
    (p_tl, p_l); the gradient is in the order h_tl, w_tl, s_tl, h_l, w_l, s_l, p_tl, p_l."""
    h_t, w_t, s_t, h_l, w_l, s_l = hyp
    p_t, p_l = period
    ns, nc = x_s.size, x_c.size
    G, D2, F = _gram(x_s, x_s, h_t, w_t, p_t)
    y = np.log(l_s)
    try:
        ll_t, a, Ki, Kd, terms_t, cond_t = _gp_terms(G + s_t ** 2 * np.eye(ns), G, D2, F, y, h_t, w_t, s_t)
    except np.linalg.LinAlgError:
        return SETUP_KTL_NOTPD, -np.inf, None, None, None
    kc, Dc2, Fc = _gram(x_c, x_s, h_t, w_t, p_t)
    m = kc @ a
    if check_max and nc:
        V = np.maximum(h_t * h_t - np.einsum("ij,jk,ik->i", kc, Ki, kc), 0)
        if (m + 2 * np.sqrt(V) > MAX_EXPONENT).any():
            return SETUP_MEAN_TOO_LARGE, -np.inf, None, None, None
    l_c = np.exp(m)
    x_sc, l_sc = np.concatenate([x_s, x_c]), np.concatenate([l_s, l_c])
    Gl, Dl2, Fl = _gram(x_sc, x_sc, h_l, w_l, p_l)
    try:
        np.linalg.cholesky(Gl)                          # the noise-free bordered matrix must be PD (the setup's order)
        ll_l, al, _, _, terms_l, cond_l = _gp_terms(Gl + s_l ** 2 * np.eye(ns + nc), Gl, Dl2, Fl, l_sc, h_l, w_l, s_l)
    except np.linalg.LinAlgError:
        return SETUP_KL_NOTPD, -np.inf, None, None, None
    gam = al[ns:] * l_c                                 # d ll_l / d l_c[j] = -(K_l^-1 l_sc)[ns + j], times d l_c / d m_j
    kd = [2 * kc / h_t, kc * Dc2 / w_t ** 3, np.zeros_like(kc), kc * Fc]
    grad, mag = np.empty(8), np.empty(8)
    for i, (ct, cl) in enumerate([(0, 3), (1, 4), (2, 5), (6, 7)]):
        u, v = kd[i] @ a, kc @ (Ki @ (Kd[i] @ a))       # d m_j = kd_j' a - k_j' K_t^-1 Kd a
        grad[ct] = sum(terms_t[i]) - (gam * (u - v)).sum()
        mag[ct] = np.abs(terms_t[i]).sum() + (np.abs(gam) * (np.abs(u) + np.abs(v))).sum()
        grad[cl] = sum(terms_l[i])
        mag[cl] = np.abs(terms_l[i]).sum()
    return SETUP_OK, ll_t + ll_l, grad, mag, max(cond_t, cond_l)


def problem(ns, nc, seed):
    """ns observations of a von Mises likelihood spread over [-pi, pi), nc candidates at midpoints, and hyper-parameters
    whose widths follow the spacing (well-conditioned Gram matrices)."""
    rs = np.random.RandomState(seed)
    gap = 2 * np.pi / ns
    x_s = np.linspace(-np.pi, np.pi, ns + 1)[:-1] + rs.uniform(-0.05, 0.05, ns) * gap
    l_s = np.exp(1.1 * np.cos(x_s - 0.1)) * rs.uniform(0.8, 1.2, ns) * 0.1
    k = rs.choice(ns - 1, size=min(nc, ns - 1), replace=False)
    x_c = np.sort(np.sort(x_s)[k] + 0.5 * gap + 0.1 * gap * rs.uniform(-1, 1, k.size))
    hyp = np.array([3.0 * rs.uniform(0.8, 1.2), 1.2 * gap * rs.uniform(0.9, 1.1), 0.05,
                    0.3 * rs.uniform(0.8, 1.2), 0.9 * gap * rs.uniform(0.9, 1.1), 1e-3])
    period = np.array([rs.uniform(1.0, 1.1), rs.uniform(1.0, 1.1)])     # p >= 1: the data span at most one period
    return x_s, l_s, x_c, hyp, period


def _ll(x_s, l_s, x_c, theta):
    return oracle(x_s, l_s, x_c, theta[:6], theta[6:])[1]


def test_oracle_gradient_matches_central_differences_of_its_value():
    for ns, nc, seed in [(6, 3, 0), (11, 4, 1), (20, 7, 2)]:
        x_s, l_s, x_c, hyp, period = problem(ns, nc, seed)
        st, ll, grad, _, _ = oracle(x_s, l_s, x_c, hyp, period)
        assert st == SETUP_OK and np.isfinite(ll)
        theta = np.concatenate([hyp, period])
        for c in range(8):
            dt = 1e-6 * theta[c]
            hi, lo = theta.copy(), theta.copy()
            hi[c] += dt
            lo[c] -= dt
            fd = (_ll(x_s, l_s, x_c, hi) - _ll(x_s, l_s, x_c, lo)) / (2 * dt)
            assert abs(grad[c] - fd) <= 1e-5 * abs(fd) + 1e-7 * max(1.0, abs(ll)) / theta[c], (ns, c, grad[c], fd)


def test_oracle_value_equals_the_host_gp_objects():
    from bayesian_quadrature_b200.gp import GP, PeriodicKernel
    for ns, nc, seed in [(6, 3, 3), (15, 5, 4)]:
        x_s, l_s, x_c, hyp, period = problem(ns, nc, seed)
        st, ll, _, _, cond = oracle(x_s, l_s, x_c, hyp, period)
        assert st == SETUP_OK
        gp_log_l = GP(PeriodicKernel(hyp[0], hyp[1], period[0]), x_s, np.log(l_s), s=hyp[2])
        l_c = np.exp(gp_log_l.mean(x_c))
        gp_l = GP(PeriodicKernel(hyp[3], hyp[4], period[1]), np.concatenate([x_s, x_c]), np.concatenate([l_s, l_c]), s=hyp[5])
        want = gp_log_l.log_lh + gp_l.log_lh
        assert abs(ll - want) <= 1e-12 * abs(want) + 1e-13 * cond, (ll, want, cond)


def test_oracle_statuses():
    x_s, l_s, x_c, hyp, period = problem(10, 4, 5)
    big = hyp.copy()
    big[0] = 1e6                                        # l_c = exp(m) with m + 2 sqrt(V) beyond MAX_EXPONENT
    assert oracle(x_s, l_s, x_c, big, period)[0] == SETUP_MEAN_TOO_LARGE
    assert oracle(x_s, l_s, x_c, big, period, check_max=False)[0] != SETUP_MEAN_TOO_LARGE
    flat = hyp.copy()
    flat[4], flat[5] = 1e4, 0.0                         # gp_l's kernel is a constant: the bordered K_l is singular
    assert oracle(x_s, l_s, x_c, flat, period)[0] == SETUP_KL_NOTPD
