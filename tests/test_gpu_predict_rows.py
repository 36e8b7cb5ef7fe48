"""The prediction kernel (csrc/bq_predict.cu) behind bqb_predict_rows_device / _host and the alpha_l the setup kernel keeps for
it (bqb_alpha_read): alpha_l against the reference's fixtures and the oracles, gp_l.mean / diag gp_log_l.cov against gp.GP,
oracle.approx.ApproxModel and the C oracle in every capacity class, with the periodic kernel and with a noisy gp_l; the
scoring kernels' prediction mode where both apply; launch independence; what a call must leave alone; the error semantics;
and the routing of BQ / BatchBQ.l_mean and l_var through it."""
import numpy as np
import pytest

from conftest import assert_close, load_golden
from oracle import approx

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps


@pytest.fixture(scope="module")
def lib():
    from bayesian_quadrature_b200 import _lib
    _lib.load()
    return _lib


def golden_batch(lib, g, approx):
    """A one-instance batch of a reference fixture: the generic kernel with its grid when ``approx``, else closed forms."""
    ns, nc = g["x_s"].size, g["x_c"].size
    ptl, pl = g["params_tl"], g["params_l"]
    kind = int(g.get("kind", 0))
    b = lib.Batch(1, ns)
    if approx:
        b.set_approx(kind, period=[[ptl[2], pl[2]]] if kind else None, xo=g["xo"], p_xo=g["p_xo"])
    hyp = np.array([ptl[0], ptl[1], ptl[-1], pl[0], pl[1], pl[-1]])
    prior = np.array([float(g["x_mean"]), float(g["x_var"]), float(g["candidate_thresh"])])
    info = b.setup([ns], [nc], g["x_s"][None], g["l_s"][None], g["x_c"][None] if nc else np.zeros((1, 0)), hyp[None], prior[None])
    assert info["status"][0] == lib.SETUP_OK
    return b


def model_order(alpha, x_s):
    """alpha over (x_s in the caller's order, x_c) -> the model's order (observations ascending, then the candidates)."""
    ns = x_s.size
    return np.concatenate([alpha[:ns][np.argsort(x_s, kind="stable")], alpha[ns:]])


def alpha_atol(x_s, x_c, params_l, kind, cond, dl_c, alpha):
    """Absolute tolerance of a stored alpha_l against a reference one: the scale max(1e-9, 0.1 cond eps) of a backward-stable
    solve, plus twice the first-order effect of the candidates' values l_c on which the two sides differ (each computes l_c
    from its own solve with K_tl; alpha_c is far more sensitive to it than the mean K_l(x, x_sc) alpha_l is)."""
    x_sc = np.concatenate([x_s, x_c])
    p_l = params_l[2] if kind else 1.0
    K = approx.kernel(kind, params_l[0], params_l[1], p_l, x_sc, x_sc) + params_l[-1] ** 2 * np.eye(x_sc.size)
    d = np.zeros(x_sc.size)
    d[x_s.size:] = dl_c
    return max(1e-9, 0.1 * cond * EPS) * np.abs(alpha).max() + 2 * np.abs(np.linalg.solve(K, d)).max()


def synthetic_problem(ns, nc, seed):
    from bayesian_quadrature_b200 import synthetic
    rs = np.random.RandomState(seed)
    x_s, l_s = synthetic.observations(ns, synthetic.problem_shift(seed))
    p = rs.permutation(ns)
    x_s, l_s = x_s[p], l_s[p]                                     # any order in
    xs = np.sort(x_s)
    x_c = np.sort(xs[rs.choice(ns - 1, size=nc, replace=False)] + 0.625)
    opt = synthetic.options(ns)
    return x_s, l_s, x_c, (opt["x_mean"], opt["x_var"], 0.5)


def gauss_batch(lib, problems, s_l=0.0, force_generic=False):
    """A Gaussian-kernel batch of synthetic problems [(ns, nc, seed)]; s_l one value or one per problem."""
    from bayesian_quadrature_b200 import synthetic
    P = len(problems)
    data = [synthetic_problem(*q) for q in problems]
    cap = max(q[0] for q in problems)
    x_s, l_s = np.zeros((P, cap)), np.ones((P, cap))
    x_c = np.zeros((P, 16))
    for p, (xs, ls, xc, _) in enumerate(data):
        x_s[p, :xs.size], l_s[p, :ls.size], x_c[p, :xc.size] = xs, ls, xc
    hyp = np.tile(np.array(synthetic.PARAMS_TL + synthetic.PARAMS_L), (P, 1))
    hyp[:, 5] = s_l
    prior = np.array([d[3] for d in data])
    b = lib.Batch(P, cap)
    if force_generic:
        b.set_approx(0, force_generic=True)
    info = b.setup([q[0] for q in problems], [q[1] for q in problems], x_s, l_s, x_c, hyp, prior)
    assert (info["status"] == lib.SETUP_OK).all()
    return b, data, hyp, info


def host_gps(data, hyp, l_c):
    from bayesian_quadrature_b200.gp import GP, GaussianKernel
    x_s, l_s, x_c, _ = data
    h = hyp
    gp_log_l = GP(GaussianKernel(h[0], h[1]), x_s, np.log(l_s), s=h[2])
    gp_l = GP(GaussianKernel(h[3], h[4]), np.concatenate([x_s, x_c]), np.concatenate([l_s, l_c[:x_c.size]]), s=h[5])
    return gp_log_l, gp_l


def check_mean(got, want, what):
    assert_close(got, want, what + " l_mean", rtol=1e-9, atol=1e-12 * np.abs(want).max())


def check_var(got, want, what):
    # a cancellation (k_tt - k' K^-1 k -> 0 at the observations): absolute tolerance on the scale of the variance
    assert_close(got, want, what + " v_log_l", rtol=1e-9, atol=1e-10 * np.abs(want).max())


# ---------------------------------------------------------------------------------------------------------------- alpha_l
@pytest.mark.parametrize("name,use_approx", [("periodic_a", True), ("periodic_b", True), ("approx_gauss", True),
                                         ("edge_noise", False), ("fixture", False), ("c1", False), ("c2", False),
                                         ("c3", False), ("c5", False)])
def test_stored_alpha_matches_the_reference_fixtures(lib, name, use_approx):
    g = load_golden(name)
    b = golden_batch(lib, g, use_approx)
    got = b.read_alpha(0)
    want = model_order(g["alpha_l"], g["x_s"])
    cond = float(g["cond_K_l"])
    nc = g["x_c"].size
    atol = alpha_atol(g["x_s"], g["x_c"], g["params_l"], int(g.get("kind", 0)), cond, b.info()["l_c"][0, :nc] - g["l_c"], want)
    assert_close(got, want, name + " alpha_l", rtol=max(1e-9, 0.1 * cond * EPS), atol=atol)
    b.close()


@pytest.mark.parametrize("ns,s_l", [(9, 0.0), (40, 0.0), (40, 1e-3), (100, 0.05), (300, 0.0)])
def test_stored_alpha_matches_the_c_oracle(lib, oracle, ns, s_l):
    from bayesian_quadrature_b200 import synthetic
    b, data, hyp, info = gauss_batch(lib, [(ns, 3, ns)], s_l)
    x_s, l_s, x_c, (mu, var, thr) = data[0]
    params_l = synthetic.PARAMS_L[:2] + (s_l,)
    om = oracle.OracleModel(x_s, l_s, x_c, synthetic.PARAMS_TL, params_l, mu, var, thr)
    assert_close(info["l_c"][0, :x_c.size], om.l_c, "l_c ns=%d" % ns)
    want = model_order(om.alpha_l, x_s)
    x_sc = np.concatenate([x_s, x_c])
    cond = np.linalg.cond(approx.kernel(0, params_l[0], params_l[1], 1.0, x_sc, x_sc) + s_l ** 2 * np.eye(x_sc.size))
    atol = alpha_atol(x_s, x_c, params_l, 0, cond, info["l_c"][0, :x_c.size] - om.l_c, want)
    assert_close(b.read_alpha(0), want, "alpha_l ns=%d s_l=%g" % (ns, s_l), rtol=max(1e-9, 0.1 * cond * EPS), atol=atol)
    b.close()


def test_stored_alpha_matches_the_approx_model(lib):
    for name in ("periodic_a", "periodic_b", "approx_gauss"):
        g = load_golden(name)
        b = golden_batch(lib, g, True)
        am = approx.ApproxModel(g["x_s"], g["l_s"], g["x_c"], g["params_tl"], g["params_l"], float(g["x_mean"]),
                                float(g["x_var"]), float(g["candidate_thresh"]), int(g["kind"]), g["xo"], g["p_xo"])
        want = model_order(am.alpha_l, g["x_s"])
        cond, nc = float(g["cond_K_l"]), g["x_c"].size
        atol = alpha_atol(g["x_s"], g["x_c"], g["params_l"], int(g["kind"]), cond, b.info()["l_c"][0, :nc] - am.l_c, want)
        assert_close(b.read_alpha(0), want, name + " alpha_l", rtol=max(1e-9, 0.1 * cond * EPS), atol=atol)
        b.close()


# ------------------------------------------------------------------------------------------------------ mean and variance
@pytest.mark.parametrize("ns,s_l", [(10, 0.0), (40, 0.0), (100, 0.0), (150, 0.0), (200, 0.0), (257, 0.0), (300, 0.0),
                                    (512, 0.0), (40, 1e-3), (100, 1e-3), (200, 0.05), (300, 1e-3)])
def test_mean_and_variance_match_the_oracles(lib, oracle, ns, s_l):
    """Every capacity class (16 ... 512) and a noisy gp_l: against gp.GP objects (the reference's route) and the C oracle's
    gp_log_l covariance; with s_l = 0 the mean interpolates the observations."""
    from bayesian_quadrature_b200 import synthetic
    b, data, hyp, info = gauss_batch(lib, [(ns, 4, ns + 1)], s_l)
    x_s, l_s, x_c, (mu, var, thr) = data[0]
    x = np.concatenate([np.linspace(x_s.min() - 8, x_s.max() + 8, 1001), x_s, x_c])
    m, v = b.predict_rows_host(x)
    gp_log_l, gp_l = host_gps(data[0], hyp[0], info["l_c"][0])
    what = "ns=%d s_l=%g" % (ns, s_l)
    check_mean(m[0], gp_l.mean(x), what)
    check_var(v[0], np.diag(gp_log_l.cov(x)), what)
    om = oracle.OracleModel(x_s, l_s, x_c, synthetic.PARAMS_TL, synthetic.PARAMS_L[:2] + (s_l,), mu, var, thr)
    check_var(v[0], om.gp_log_l_mean_cov(x)[1], what + " (C oracle)")
    if s_l == 0:
        assert np.allclose(m[0, 1001:1001 + ns], l_s, rtol=0, atol=1e-4 * l_s.max()), what
    b.close()


@pytest.mark.parametrize("name", ["periodic_a", "periodic_b", "approx_gauss"])
def test_mean_and_variance_match_the_approx_model(lib, name):
    """The generic path's fixtures (periodic kernel, trapezoid path): mean against ApproxModel.l_mean, variance against the
    same model's gp_log_l written out.  periodic_a's gp_log_l is nearly deterministic (cond K_tl 4.7e8): its variance is
    rounding noise on the scale cond eps k_tt, which bounds the comparison there."""
    g = load_golden(name)
    b = golden_batch(lib, g, True)
    am = approx.ApproxModel(g["x_s"], g["l_s"], g["x_c"], g["params_tl"], g["params_l"], float(g["x_mean"]),
                            float(g["x_var"]), float(g["candidate_thresh"]), int(g["kind"]), g["xo"], g["p_xo"])
    x = np.concatenate([g["x_a"], g["x_s"]])
    m, v = b.predict_rows_host(x)
    check_mean(m[0], am.l_mean(x), name)
    K = am.k_tl(x, g["x_s"])
    k_tt = np.diag(am.k_tl(x, x))
    want_v = k_tt - np.einsum("ij,jk,ik->i", K, am.inv_K_tl, K)
    atol = max(1e-10 * np.abs(want_v).max(), 10 * float(g["cond_K_tl"]) * EPS * k_tt.max())
    assert_close(v[0], want_v, name + " v_log_l", rtol=1e-9, atol=atol)
    b.close()


@pytest.mark.parametrize("ns", [10, 40, 100, 150, 200])
def test_agrees_with_the_prediction_mode_of_the_scoring_kernels(lib, ns):
    b, data, _, _ = gauss_batch(lib, [(ns, 4, ns), (ns - 3, 2, ns + 7), (ns, 0, ns + 9)])
    x = np.linspace(-1.2 * ns, 1.2 * ns, 777)
    m2, v2 = b.predict_host(x)
    m, v = b.predict_rows_host(x)
    for p in range(3):
        check_mean(m[p], m2[p], "ns=%d problem %d" % (ns, p))
        check_var(v[p], v2[p], "ns=%d problem %d" % (ns, p))
    b.close()


def test_non_finite_points_give_nan(lib):
    b, _, _, _ = gauss_batch(lib, [(40, 3, 1)], 1e-3)
    m, v = b.predict_rows_host(np.array([0.5, np.nan, np.inf, -np.inf, 1.5]))
    assert np.isnan(m[0, 1:4]).all() and np.isnan(v[0, 1:4]).all()
    assert np.isfinite(m[0, [0, 4]]).all() and np.isfinite(v[0, [0, 4]]).all()
    b.close()


# --------------------------------------------------------------------------------------------- launch independence, scope
def batches(lib):
    """A tensor-core batch with mixed s_l and ragged sizes, and a batch of the 512 class."""
    yield gauss_batch(lib, [(40, 3, 1), (33, 0, 2), (64, 16, 3), (17, 5, 4), (50, 2, 5)], s_l=[0.0, 1e-3, 0.0, 0.05, 0.0])[0]
    yield gauss_batch(lib, [(300, 3, 6), (257, 1, 7), (512, 4, 8)], s_l=[0.0, 1e-3, 0.0])[0]


def test_rows_are_independent_of_the_launch(lib):
    import torch
    for b in batches(lib):
        P = b.n_inst
        for na in (0, 1, 7, 33, 257):
            base = np.linspace(-30.0, 30.0, na)
            for shared in (True, False):
                x = base if shared else np.stack([base + 0.1 * p for p in range(P)])
                x_d = torch.from_numpy(np.ascontiguousarray(x)).cuda()

                def run(rows):
                    m = torch.full((P, na + 3), -7.0, dtype=torch.float64, device="cuda")
                    v = torch.full((P, na + 3), -7.0, dtype=torch.float64, device="cuda")
                    b.predict_rows_device(x_d, m[:, 1:na + 1], v[:, 1:na + 1], rows=rows)
                    return m.cpu().numpy(), v.cpu().numpy()
                m_all, v_all = run(None)
                m_list, v_list = run(list(range(P)))
                shuffled = np.random.RandomState(na).permutation(P)
                m_sh, v_sh = run(shuffled)
                assert np.array_equal(m_all, m_list) and np.array_equal(v_all, v_list)
                assert np.array_equal(m_all, m_sh) and np.array_equal(v_all, v_sh)
                assert (m_all[:, 0] == -7).all() and (m_all[:, na + 1:] == -7).all()   # nothing outside the rows
                for p in range(P):
                    m1, v1 = run([p])
                    assert np.array_equal(m1[p], m_all[p]) and np.array_equal(v1[p], v_all[p]), (na, shared, p)
                    others = np.arange(P) != p
                    assert (m1[others] == -7).all() and (v1[others] == -7).all()       # rows not listed are untouched
                mh, vh = b.predict_rows_host(x, rows=[P - 1])
                assert np.array_equal(mh[P - 1], m_all[P - 1, 1:na + 1]) and np.isnan(mh[:P - 1]).all()
        b.close()


def test_a_prediction_changes_no_model_and_no_score(lib):
    for b in batches(lib):
        x = np.linspace(-40.0, 40.0, 301)
        before = [b.read_model(p) for p in range(b.n_inst)]
        alpha = [b.read_alpha(p) for p in range(b.n_inst)]
        esm0, em0, st0 = b.score_host(x)
        b.predict_rows_host(x)
        b.predict_rows_host(x, rows=[0])
        for p in range(b.n_inst):
            assert np.array_equal(b.read_model(p), before[p]) and np.array_equal(b.read_alpha(p), alpha[p]), p
        esm1, em1, st1 = b.score_host(x)
        assert np.array_equal(esm0, esm1) and np.array_equal(em0, em1) and np.array_equal(st0, st1)
        b.close()


def test_generic_gaussian_batch_equals_the_tensor_core_batch(lib):
    """The kernel reads the same model and alpha_l whichever scoring kernel a batch uses."""
    probs = [(40, 3, 1), (64, 16, 3)]
    b0, _, _, _ = gauss_batch(lib, probs, 1e-3)
    b1, _, _, _ = gauss_batch(lib, probs, 1e-3, force_generic=True)
    x = np.linspace(-40.0, 40.0, 101)
    assert all(np.array_equal(a, c) for a, c in zip(b0.predict_rows_host(x), b1.predict_rows_host(x)))
    b0.close(); b1.close()


def test_errors(lib):
    import torch
    b, _, _, _ = gauss_batch(lib, [(40, 3, 1), (33, 0, 2)], 1e-3)
    x = np.linspace(-5, 5, 9)
    for rows in ([2], [-1], [0, 5]):
        with pytest.raises(ValueError, match="row out of range"):
            b.predict_rows_host(x, rows=rows)
    x_d = torch.from_numpy(x).cuda()
    m = torch.empty(2, 9, dtype=torch.float64, device="cuda")
    L = lib.load()
    rows = (lib.ctypes.c_int * 1)(0)
    assert L.bqb_predict_rows_device(b._h, rows, -1, lib._ptr(x_d), 0, 9, lib._ptr(m), lib._ptr(m), 9, None) == lib.EINVAL
    assert L.bqb_predict_rows_device(b._h, None, 0, lib._ptr(x_d), 0, 9, lib._ptr(m), lib._ptr(m), 8, None) == lib.EINVAL
    assert L.bqb_predict_rows_device(b._h, None, 0, None, 0, 9, lib._ptr(m), lib._ptr(m), 9, None) == lib.EINVAL
    assert L.bqb_predict_rows_device(b._h, None, 0, lib._ptr(x_d), 0, 0, lib._ptr(m), lib._ptr(m), 0, None) == 0    # na = 0
    b.close()
    fresh = lib.Batch(2, 40)
    with pytest.raises(lib.BQB200Error, match="not set up"):
        fresh.predict_rows_host(x)
    with pytest.raises(ValueError):
        fresh.read_alpha(0)
    fresh.close()
    g = load_golden("periodic_b")
    b = golden_batch(lib, g, True)
    with pytest.raises(NotImplementedError):
        b.predict_host(g["x_a"][:4])                     # the scoring kernels' prediction mode stays tensor-core only
    b.close()


# ------------------------------------------------------------------------------------------------------------- public API
def test_batch_routes_every_finite_problem_to_the_device(monkeypatch):
    """Periodic, noisy and 512-class batches: no host GP is built for a finite grid, rows equal a loop of BQ objects bit
    for bit at round 0 and within parity tolerance after a round, and BQ itself leaves its host GPs alone."""
    from test_gpu_batch_readout import gaussian_case, periodic_case
    from bayesian_quadrature_b200.gp import GP

    def no_host_gp(*args):
        raise AssertionError("a host GP answered")
    monkeypatch.setattr(GP, "mean", no_host_gp)          # neither BatchBQ nor BQ falls back to GP objects
    monkeypatch.setattr(GP, "cov", no_host_gp)
    for bb, fl, bq_objects, grid in (gaussian_case(40), gaussian_case(300), periodic_case()):
        bqs, states = bq_objects()
        for rnd in range(2):
            for name in ("l_mean", "l_var"):
                got = getattr(bb, name)(grid)
                for p, bq in enumerate(bqs):
                    want = getattr(bq, name)(grid)
                    if rnd == 0:
                        assert np.array_equal(got[p], want), (name, p)
                    else:
                        assert_close(got[p], want, "%s round %d problem %d" % (name, rnd, p))
            if rnd == 0:
                idx, x_next = bb.choose_next(grid)
                l_new = np.array([fl[p](x_next[p]) for p in range(bb.P)])
                bb.add_observations(x_next, l_new)
                for p, bq in enumerate(bqs):
                    np.random.set_state(states[p])
                    bq.add_observation(float(x_next[p]), float(l_new[p]))
        bb.close()


def test_device_resident_batch_moves_nothing_but_grid_and_result(monkeypatch):
    import torch
    from test_gpu_batch_readout import gaussian_case, periodic_case
    for make in (lambda dr: gaussian_case(300, device_resident=dr), lambda dr: periodic_case(device_resident=dr)):
        host, _, _, grid = make(False)
        dev, _, _, _ = make(True)
        dev._host_stale = True
        monkeypatch.setattr(dev, "sync_host", lambda: (_ for _ in ()).throw(AssertionError("sync_host")))
        g_d = torch.from_numpy(grid).cuda()
        for name in ("l_mean", "l_var"):
            assert np.array_equal(getattr(host, name)(grid), getattr(dev, name)(g_d, on_device=True).cpu().numpy()), name
        monkeypatch.undo()
        host.close(); dev.close()


def test_a_non_finite_grid_row_alone_goes_to_the_host_gps(monkeypatch):
    from test_gpu_batch_readout import gaussian_case
    from bayesian_quadrature_b200 import BatchBQ
    bb, _, _, grid = gaussian_case(40)
    rows = np.stack([grid + 0.01 * (p + 1) for p in range(bb.P)])
    clean_m, clean_v = bb.l_mean(rows), bb.l_var(rows)
    rows[2, 5] = np.nan
    seen = []
    real = BatchBQ._host_gps
    monkeypatch.setattr(BatchBQ, "_host_gps", lambda self, p: (seen.append(int(p)), real(self, p))[1])
    gp_log_l, gp_l = real(bb, 2)
    with pytest.raises(ValueError) as want:              # what the host GPs say about a NaN (gp_log_l.cov's finiteness check)
        gp_l.mean(rows[2])
        gp_log_l.cov(rows[2])
    with pytest.raises(ValueError) as got:
        bb.l_mean(rows)
    assert str(got.value) == str(want.value)
    assert seen == [2]                                   # the finite problems 0, 1 did not build host GPs
    rows[2, 5] = 0.0                                     # and a finite problem 2 gets the device route again
    seen.clear()
    assert np.array_equal(bb.l_var(rows)[:2], clean_v[:2]) and seen == []
    assert np.array_equal(bb.l_mean(rows)[:2], clean_m[:2])
    bb.close()
