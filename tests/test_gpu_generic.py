"""The generic device path (csrc/bq_score_generic.cu + the trapezoid / periodic modes of csrc/bq_setup2.cu): SURVEY 8(f).4,
the reference's `use_approx` branch (bq.py:251-252, :310-311, :498-510; bq_c.pyx:216-261, :358-422, :538-598) and
gp.PeriodicKernel.  Checked against fixtures produced by the unmodified reference (tests/golden/approx_gauss.npz,
periodic_a.npz, periodic_b.npz), against the numpy oracle (oracle/approx.py) on seeded ragged batches of every capacity
class and through BatchBQ.marginal_loss, against the C oracle (oracle/bq_oracle.c) with the Gaussian kernel's closed
forms, and -- with those closed forms -- against the tensor-core kernels, which compute the same thing.  The isclose
shortcut boundary of bq.py:456 is checked on every scoring kernel."""
import functools
from fractions import Fraction

import numpy as np
import pytest

from conftest import ATOL, RTOL, assert_close, load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    from bayesian_quadrature_b200 import _lib
    _lib.load()
    return _lib


def setup_generic(lib, g, kind=None, approx=True, force=False):
    ns, nc = g["x_s"].size, g["x_c"].size
    b = lib.Batch(1, ns)
    ptl, pl = g["params_tl"], g["params_l"]
    kind = int(g["kind"]) if kind is None else kind
    hyp = np.array([ptl[0], ptl[1], ptl[-1], pl[0], pl[1], pl[-1]])
    prior = np.array([float(g["x_mean"]), float(g["x_var"]), float(g["candidate_thresh"])])
    b.set_approx(kind, period=[[ptl[2], pl[2]]] if kind else None, xo=g["xo"] if approx else None,
                 p_xo=g["p_xo"] if approx else None, force_generic=force)
    info = b.setup([ns], [nc], g["x_s"][None], g["l_s"][None], g["x_c"][None] if nc else np.zeros((1, 0)), hyp[None], prior[None])
    assert info["status"][0] == lib.SETUP_OK
    return b, info


@pytest.mark.parametrize("name", ["fixture", "c1", "c2", "c5", "edge_noise"])
def test_generic_kernel_equals_the_tensor_core_kernels(lib, name):
    """Gaussian kernel, closed-form integrals: the plain-FP64 kernel against the DMMA kernels (dense cut-off) and the
    reference's fixture -- scores, expected variance (fused epilogue) and status bits."""
    g = dict(load_golden(name))
    g["kind"], g["xo"], g["p_xo"] = 0, None, None
    b0, _ = setup_generic(lib, g, approx=False, force=False)
    b0.set_cutoff(float("inf"))
    b1, _ = setup_generic(lib, g, approx=False, force=True)
    x_a = np.concatenate([g["x_a"], [np.nan, np.inf]])
    e0, m0, s0 = b0.score_host(x_a)
    e1, m1, s1 = b1.score_host(x_a)
    ok = np.isfinite(x_a)
    assert (s0 == s1).all()
    assert_close(e1[0][ok], e0[0][ok], name + " esm generic vs tensor-core", rtol=1e-9, atol=1e-300)
    assert_close(m1[0][ok], m0[0][ok], name + " em generic vs tensor-core", rtol=1e-9, atol=1e-300)
    assert_close(e1[0][:g["x_a"].size], g["esm"], name + " esm generic vs reference")
    ev0, f0 = b0.expected_var_host(g["x_a"])
    ev1, f1 = b1.expected_var_host(g["x_a"])
    assert f0 == f1
    assert_close(ev1, ev0, name + " expected variance", rtol=1e-9, atol=1e-9 * float(np.abs(g["esm"]).max()))
    with pytest.raises(NotImplementedError):
        b1.predict_host(g["x_a"][:4])
    b0.close(); b1.close()


@pytest.mark.parametrize("name", ["approx_gauss", "periodic_a", "periodic_b"])
def test_trapezoid_path_vs_reference_fixture(lib, name):
    g = load_golden(name)
    b, info = setup_generic(lib, g)
    nc = g["x_c"].size
    if nc:
        assert_close(info["l_c"][0, :nc], g["l_c"], name + " l_c")
    assert_close(info["Z_mean"][0], g["Z_mean"], name + " Z_mean")
    # Z_var = g' K_tl(xo, xo) g - r' K_tl^-1 r cancels to rounding noise when gp_log_l is nearly deterministic: the reference's
    # explicit-inverse route leaves cond * eps * (scale of the terms) there (-1.6e-9 at cond 4.7e8 in periodic_a)
    ptl = g["params_tl"]
    k0 = ptl[0] ** 2 if int(g["kind"]) else ptl[0] ** 2 / (np.sqrt(2 * np.pi) * ptl[1])
    tol = max(1e-13, 10 * float(g["cond_K_tl"]) * np.finfo(np.float64).eps * float(g["Z_mean"]) ** 2 * k0)
    assert abs(info["Z_var"][0] - float(g["Z_var"])) < tol, (info["Z_var"][0], float(g["Z_var"]), tol)
    assert abs(info["log_lh"][0] - float(g["log_lh"])) <= 1e-8 * abs(float(g["log_lh"]))
    esm, em, st = b.score_host(g["x_a"])
    assert ((st[0] & lib.ST_SHORTCUT) == g["shortcut"]).all()
    assert not (st[0] & (lib.ST_ESM_BAD | lib.ST_EM_BAD | lib.ST_XA_BAD)).any()
    assert_close(esm[0], g["esm"], name + " esm")
    assert_close(em[0], g["em"], name + " em")
    ev, _ = b.expected_var_host(g["x_a"])
    assert_close(ev, g["expected_Z_var"], name + " expected_Z_var", atol=max(ATOL, tol))
    b.close()


def test_bq_object_with_the_periodic_kernel():
    """The public class end to end (tests/util.py:76-91 of the reference: von Mises likelihood, wrapped domain, prior
    normalised as the reference does): same candidates, Z_mean, Z_var and scores as the reference's own run, and
    choose_next / add_observation keep working (tests/test_bq_object.py:303-350, :387-395)."""
    from scipy.special import iv
    from bayesian_quadrature_b200 import BQ, PeriodicKernel
    g = load_golden("periodic_b")
    np.random.seed(8728)
    x = np.linspace(-np.pi, np.pi, 6)[:-1]
    y = np.exp(-np.log(2 * np.pi * iv(0, 1.1)) + 1.1 * np.cos(x - 0.1))
    bq = BQ(x, y, n_candidate=10, x_mean=0.0, x_var=10.0, candidate_thresh=0.5, kernel=PeriodicKernel, optim_method="L-BFGS-B")
    bq.init(params_tl=(3, 1.2, 1, 0.), params_l=(0.3, 0.8, 1, 0.))
    assert bq.options["use_approx"] and bq.options["wrapped"]
    assert np.array_equal(bq.x_c, g["x_c"])
    assert_close(bq._approx_x, g["xo"], "approximation grid")
    assert_close(bq._approx_px, g["p_xo"], "prior on the grid")
    assert_close(bq.l_c, g["l_c"], "l_c")
    assert_close(bq.Z_mean(), g["Z_mean"], "Z_mean")
    assert abs(bq.Z_var() - float(g["Z_var"])) < 1e-12
    assert_close(bq.expected_squared_mean(g["x_a"]), g["esm"], "expected_squared_mean")
    assert_close(bq.expected_mean(g["x_a"]), g["em"], "expected_mean")
    assert_close(bq.expected_Z_var(g["x_a"]), g["expected_Z_var"], "expected_Z_var", atol=max(ATOL, 1e-13))
    assert_close(bq.l_mean(g["x_a"][:7]), bq.gp_l.mean(g["x_a"][:7]), "l_mean (host GPs)")
    grid = np.linspace(-np.pi, np.pi, 101)
    nxt = bq.choose_next(grid, n=2, params=["h", "w"])
    assert nxt in grid
    ns0 = bq.ns
    bq.add_observation(float(nxt), float(np.exp(-np.log(2 * np.pi * iv(0, 1.1)) + 1.1 * np.cos(nxt - 0.1))))
    assert bq.ns in (ns0, ns0 + 1) and np.isfinite(bq.Z_mean())


@pytest.mark.parametrize("ns,nc", [(257, 2), (300, 3), (512, 5)])
def test_more_than_256_observations_run_on_the_generic_kernel(lib, oracle, ns, nc):
    """The 512 capacity class (VERDICT r01 "missing" 5): setup by the second-generation kernel with its packed triangle in
    global scratch, scoring by the plain-FP64 kernel (the tensor-core kernels' k-step masks end at 256 observations).
    Gaussian kernel, closed-form integrals, against the C oracle (the reference algorithm) on a sample of points."""
    from bayesian_quadrature_b200 import synthetic
    rs = np.random.RandomState(ns)
    x_s, l_s = synthetic.observations(ns)
    p = rs.permutation(ns)
    x_s, l_s = x_s[p], l_s[p]                                    # any order in
    xs = np.sort(x_s)
    x_c = np.sort(xs[rs.choice(ns - 1, size=nc, replace=False)] + 0.625)
    opt = synthetic.options(ns)
    assert lib.ns_capacity(ns) == 512
    b = lib.Batch(1, ns)
    info = b.setup([ns], [nc], x_s[None], l_s[None], x_c[None], np.array([synthetic.PARAMS_TL + synthetic.PARAMS_L]),
                   np.array([[opt["x_mean"], opt["x_var"], 0.5]]), check_max=True)
    assert info["status"][0] == 0
    m = oracle.OracleModel(x_s, l_s, x_c, synthetic.PARAMS_TL, synthetic.PARAMS_L, opt["x_mean"], opt["x_var"], 0.5)
    assert_close(info["Z_mean"][0], m.Z_mean(), "Z_mean")
    assert_close(info["l_c"][0, :nc], m.l_c, "l_c")
    grid = synthetic.query_grid(ns, 4001)
    x_a = np.concatenate([grid[rs.choice(4001, 60, replace=False)], xs[:3], xs[:3] + 0.9e-4, x_c, x_c + 0.3, [xs[-1] + 40.0]])
    esm, em, st = b.score_host(x_a)
    o_esm, o_em, o_st = m.esm_and_em(x_a)
    assert ((st[0] & 3) == (o_st & 3)).all()
    assert_close(esm[0], o_esm, "esm ns=%d" % ns)
    assert_close(em[0], o_em, "em ns=%d" % ns)
    ev, _ = b.expected_var_host(grid)                                # fused epilogue, 4001 points
    assert np.isfinite(ev).all()
    m.close()
    b.close()


def test_per_instance_grids_and_periods(lib):
    """A batch whose instances carry their own approximation grid (xo_stride > 0), period and hyper-parameters gives,
    instance by instance, exactly what single-instance batches give."""
    g = load_golden("periodic_b")
    ns, nc = g["x_s"].size, g["x_c"].size
    ptl, pl = g["params_tl"], g["params_l"]
    B = 3
    hyp = np.array([[ptl[0] * (1 + 0.1 * i), ptl[1] * (1 + 0.05 * i), 0.0, pl[0], pl[1] * (1 - 0.05 * i), 0.0] for i in range(B)])
    period = np.array([[1.0 + 0.1 * i, 1.0 + 0.05 * i] for i in range(B)])
    xo = np.stack([np.linspace(-np.pi * (1 + 0.1 * i), np.pi * (1 + 0.1 * i), g["xo"].size) for i in range(B)])
    p_xo = np.stack([np.interp(xo[i], g["xo"], g["p_xo"]) for i in range(B)])
    prior = np.tile([float(g["x_mean"]), float(g["x_var"]), float(g["candidate_thresh"])], (B, 1))
    x_a = np.linspace(-3, 3, 257)
    b = lib.Batch(B, ns)
    b.set_approx(1, period=period, xo=xo, p_xo=p_xo)
    info = b.setup(np.full(B, ns), np.full(B, nc), np.tile(g["x_s"], (B, 1)), np.tile(g["l_s"], (B, 1)), np.tile(g["x_c"], (B, 1)),
                   hyp, prior)
    assert (info["status"] == 0).all()
    esm, em, st = b.score_host(x_a)
    for i in range(B):
        b1 = lib.Batch(1, ns)
        b1.set_approx(1, period=period[i:i + 1], xo=xo[i], p_xo=p_xo[i])
        i1 = b1.setup([ns], [nc], g["x_s"][None], g["l_s"][None], g["x_c"][None], hyp[i:i + 1], prior[i:i + 1])
        e1, m1, s1 = b1.score_host(x_a)
        assert i1["Z_mean"][0] == info["Z_mean"][i] and i1["Z_var"][0] == info["Z_var"][i]
        assert np.array_equal(e1[0], esm[i]) and np.array_equal(m1[0], em[i]) and np.array_equal(s1[0], st[i])
        b1.close()
    assert not np.array_equal(esm[0], esm[1])
    b.close()


# ---------------------------------------------------------------------------------------------------------------------
# Independent checks of the generic path against the numpy oracle (oracle/approx.py) and the C oracle (oracle/bq_oracle.c)
#
# Tolerances, fixed before any run: esm, em, Z_mean and l_c at the parity tolerance (RTOL / ATOL) -- every design below
# keeps cond(K_tl) and cond of the bordered K_l(x_sc, x_sc) under COND_MAX, which the case builders assert; Z_var to the
# absolute bound of tests/test_gpu_setup.zvar_bound, max(1e-13, 10 (cond_tl + cond_l) eps c_tl Z_mean^2); a point aliased
# to an observation by one period of gp_l's kernel duplicates that observation's row of K_l, so its Schur pivot is the
# jitter 1e-4 c_l alone and esm / em are held to max(RTOL, 1e4 cond_l eps) there (status bits exactly).  No query point
# comes near the overflow guard: every exponent of int_exp_norm stays below MAX_EXPONENT by far more than 1e-9 relative.

EPS = np.finfo(np.float64).eps
COND_MAX = 3e6
CLASSES = [16, 64, 128, 160, 256, 512]


def ulp_step(x, k):
    for _ in range(abs(k)):
        x = float(np.nextafter(x, np.inf if k > 0 else -np.inf))
    return x


def at_distance(c, t):
    """The doubles x nearest to c + t and c - t for which abs(c - x) == t exactly, as numpy evaluates it (None where
    no double within four ulps qualifies)."""
    out = []
    for x0 in (c + t, c - t):
        hit = [x for x in (ulp_step(x0, k) for k in (0, -1, 1, -2, 2, -3, 3, -4, 4)) if abs(c - x) == t]
        out.append(hit[0] if hit else None)
    return out


def fused_tol(xs):
    """1e-4 + 1e-5 |xs| rounded once, as a contracted fma computes it (exact rational arithmetic, one rounding)."""
    return float(Fraction(1e-5) * Fraction(abs(xs)) + Fraction(1e-4))


def shortcut_boundary(n, seed):
    """n observations x_s in (-1e-4, 1e-4) where numpy's isclose tolerance 1e-4 + 1e-5 |x_s| (product and sum rounded
    separately) and the fused one differ by an ulp -- alternately fused > numpy and fused < numpy -- each with the query
    points at exactly the larger of the two tolerances from it: isclose(x_a, x_s, atol=1e-4) is False there in the
    first case and True in the second, and the fused comparison says the opposite.  Returns [(x_s, [x_a, ...])]."""
    rs = np.random.RandomState(seed)
    out = []
    while len(out) < n:
        xs = float(rs.uniform(-1e-4, 1e-4))
        t_np, t_f = 1e-4 + 1e-5 * abs(xs), fused_tol(xs)
        if t_np == t_f or (t_f > t_np) != (len(out) % 2 == 0):
            continue
        pts = [x for x in at_distance(xs, max(t_np, t_f)) if x is not None]
        for x in pts:
            d = abs(x - xs)
            assert bool(np.isclose(x, xs, atol=1e-4)) == (d <= t_np) and (d <= t_np) != (d <= t_f)
        if pts:
            out.append((xs, pts))
    return out


def query_points(rs, x_s, x_c, thresh, lo, hi, n_uniform, pair=None, alias=None, extra=()):
    """Query points of one instance: a uniform sample of [lo, hi]; two observations exactly and at +-0.9e-4 / +-1.2e-4;
    up to four candidates exactly and at +-0.3 thresh; the points at exactly thresh from two candidates (|x_c - x| as
    numpy computes it) and an ulp either side; with a pair of candidates closer than 2 thresh, their mid-point and two
    points near it (close to both); with `alias` (the period 2 pi p_l of gp_l's kernel), the two observations moved by
    one period either way; then `extra`.  Returns (x_a, aliased mask)."""
    xs = np.sort(x_s)
    obs = xs[np.unique([0, xs.size // 2])]
    parts = [rs.uniform(lo, hi, n_uniform), obs, obs + 0.9e-4, obs - 0.9e-4, obs + 1.2e-4, obs - 1.2e-4]
    nc = x_c.size
    pick = sorted(set([0, nc - 1] + (list(pair) if pair is not None else []))) if nc else []
    for j in pick[:4]:
        parts.append(x_c[j] + np.array([0.0, 0.3 * thresh, -0.3 * thresh]))
    for j in [k for k in range(nc) if pair is None or k not in pair][:2]:
        for x in at_distance(x_c[j], thresh):
            if x is not None:
                parts.append(np.array([ulp_step(x, -1), x, ulp_step(x, 1)]))
    if pair is not None:
        m = 0.5 * (x_c[pair[0]] + x_c[pair[1]])
        assert abs(x_c[pair[1]] - x_c[pair[0]]) < 2 * thresh
        parts.append(m + np.array([0.0, 0.05, -0.05]) * thresh)
    parts.append(np.asarray(extra, dtype=np.float64))
    x_a = np.concatenate(parts)
    aliased = np.zeros(x_a.size, dtype=bool)
    if alias is not None:
        x_a = np.concatenate([x_a, obs + alias, obs - alias])
        aliased = np.concatenate([aliased, np.ones(2 * obs.size, dtype=bool)])
    return x_a, aliased


def place_candidates(rs, xs_sorted, gap, nc, pair):
    """nc candidates at the mid-points of random gaps; with `pair`, the first chosen gap holds two of them, at 0.3 and
    0.7 of the gap (0.4 gap apart).  Returns (sorted x_c, indices of the pair in x_c or None)."""
    ns = xs_sorted.size
    if nc == 0:
        return np.zeros(0), None
    k = rs.choice(ns - 1, size=nc - 1 if pair else nc, replace=False)
    x_c = xs_sorted[k] + gap / 2
    if pair:
        x_c = np.concatenate([x_c[1:], xs_sorted[k[:1]] + gap * np.array([0.25, 0.75])])
    x_c = np.sort(x_c)
    if not pair:
        return x_c, None
    i = int(np.argmin(np.diff(x_c)))
    return x_c, (i, i + 1)


def trapezoid_case(kind, ns, seed, nc=None, period=(1.0, 1.0), noise=(0.0, 0.0), nonuniform=False, shuffle=False,
                   origin=None, pair=False, legacy=False):
    """One instance of the trapezoid path, periodic (kind 1) or Gaussian (kind 0) kernel, with its own grid.

    Periodic: ns observations spread over [-pi, pi] at spacing gap = 2 pi / ns, widths 1.2 gap (gp_log_l) and 0.9 gap
    (gp_l) as in tests/test_gpu_batch_periodic.raw_case (1.6 and 1.2 gap for the first cases), von Mises prior, grid of 400 points over [-pi p_tl, pi p_tl].  Gaussian: observations 1.25 apart, widths 1.5
    and 1.1, a 700-point grid over the data +-3 under a normal prior.  `legacy` keeps the first seeded cases of this file
    as they were (jitter of +-0.05 / +-0.1 in absolute units, candidate_thresh 0.5, nc = 3 mid-gap candidates where the
    gap is wider than 1); otherwise jitter is 5 % of the spacing and candidate_thresh 0.4 of it.  `origin`: the
    observation nearest 0 is moved, with all others, so that it sits exactly at this value.  `nonuniform`: the grid
    points are spaced unevenly (a monotone warp of the uniform grid)."""
    from scipy.special import j0
    rs = np.random.RandomState(seed)
    s_tl, s_l = noise
    if kind:
        gap = 2 * np.pi / ns
        if legacy:
            rs.uniform(-np.pi, np.pi, ns)               # (a draw the first version made and discarded: same inputs)
        x_s = np.linspace(-np.pi, np.pi, ns + 1)[:-1] + rs.uniform(-0.05, 0.05, ns) * (1.0 if legacy else gap)
        l_s = np.exp(1.1 * np.cos(x_s - 0.1)) * rs.uniform(0.8, 1.2, ns) * 0.1
        w_tl, w_l = (1.6, 1.2) if legacy else (1.2, 0.9)
        ptl, pl = (3.0, w_tl * gap, period[0], s_tl), (0.3, w_l * gap, period[1], s_l)
        thresh = 0.5 if legacy else 0.4 * gap
        lo, hi = -np.pi * period[0], np.pi * period[0]
        n_xo = 400
    else:
        gap = 1.25
        x_s = gap * (np.arange(ns) - (ns - 1) / 2.0) + rs.uniform(-0.1, 0.1, ns) * (1.0 if legacy else 0.5 * gap)
        l_s = np.exp(-0.5 * (x_s / (0.2 * np.ptp(x_s))) ** 2) * rs.uniform(0.5, 1.5, ns) * 0.3 + 1e-3
        ptl, pl = (6.0, 1.5, s_tl), (0.4, 1.1, s_l)
        thresh = 0.5
        lo, hi = x_s.min() - 3, x_s.max() + 3
        n_xo = 700
    if origin is not None:
        k = int(np.argmin(np.abs(x_s)))
        x_s = x_s + (origin - x_s[k])
        x_s[k] = origin
        if not kind:
            lo, hi = x_s.min() - 3, x_s.max() + 3
    if legacy:
        nc = 3 if (kind == 0 or gap > 1.0) else 0
    x_c, pr = place_candidates(rs, np.sort(x_s), gap, nc, pair)
    t = np.linspace(0.0, 1.0, n_xo)
    if nonuniform:
        t = t + 0.12 * np.sin(2 * np.pi * t) / (2 * np.pi) + 0.03 * np.sin(6 * np.pi * t) / (2 * np.pi)
    xo = lo + (hi - lo) * t
    if kind:
        mu, var = 0.0, 10.0
        p_xo = np.exp(-np.log(2 * np.pi * j0(0.1)) + 0.1 * np.cos(xo))
    else:
        mu, var = 0.3, float(np.ptp(x_s) ** 2 / 9) if ns > 1 else 1.0
        p_xo = np.exp(-0.5 * (np.log(2 * np.pi * var) + (xo - mu) ** 2 / var))
    if shuffle:
        p = rs.permutation(ns)
        x_s, l_s = x_s[p], l_s[p]
    return dict(kind=kind, x_s=x_s, l_s=l_s, x_c=x_c, pair=pr, ptl=ptl, pl=pl, mu=mu, var=var, thresh=thresh, xo=xo,
                p_xo=p_xo, lo=lo, hi=hi, seed=seed)


@functools.lru_cache(maxsize=None)
def boundary_observations():
    return shortcut_boundary(8, seed=456)


# (ns, seed, options) of the instances of one ragged batch per capacity class.  `origin` = k puts an observation at the
# k-th shortcut-boundary observation and adds its constructed query points.  nc + 2 dense rows: nc <= 5 fit one 8-row
# block of the dense operand, 6 <= nc <= 13 need two and nc >= 14 three (the register bound NC_MAX = 16 is the last).
LEGACY = dict(legacy=True)
P1, P2 = (1.1, 1.05), (1.05, 1.1)
PERIODIC = {
    16: [(6, 0, LEGACY), (12, 1, LEGACY),
         (16, 16, dict(nc=14, pair=True, period=P1, noise=(0.05, 0.0), shuffle=True, origin=0)),
         (13, 17, dict(nc=7, pair=True, period=P2, noise=(0.0, 1e-3), nonuniform=True, origin=1))],
    64: [(40, 3, LEGACY),
         (64, 64, dict(nc=16, pair=True, period=P1, noise=(0.05, 0.0), shuffle=True, origin=2)),
         (17, 65, dict(nc=6, pair=True, period=P2, noise=(0.0, 1e-3), nonuniform=True, origin=3)),
         (37, 66, dict(nc=15, pair=True, period=P1, shuffle=True))],
    128: [(128, 128, dict(nc=15, pair=True, period=P1, noise=(0.05, 0.0), shuffle=True, origin=4)),
          (65, 129, dict(nc=7, pair=True, period=P2, noise=(0.0, 1e-3), nonuniform=True)),
          (101, 130, dict(nc=0, period=P1))],
    160: [(160, 160, dict(nc=16, pair=True, period=P2, noise=(0.0, 1e-3), shuffle=True, origin=5)),
          (129, 161, dict(nc=6, pair=True, period=P1, noise=(0.05, 0.0), nonuniform=True)),
          (150, 162, dict(nc=14, pair=True, period=P2))],
    256: [(256, 256, dict(nc=14, pair=True, period=P1, noise=(0.05, 0.0), shuffle=True, origin=6)),
          (161, 257, dict(nc=16, pair=True, period=P2, noise=(0.0, 1e-3), nonuniform=True)),
          (203, 258, dict(nc=7, pair=True, period=P1))],
    512: [(512, 512, dict(nc=15, pair=True, period=P2, noise=(0.0, 1e-3), shuffle=True, origin=7)),
          (257, 513, dict(nc=7, pair=True, period=P1, noise=(0.05, 0.0), nonuniform=True)),
          (301, 514, dict(nc=16, pair=True, period=P2))],
}
GAUSSIAN_TRAPEZOID = {
    16: [(11, 18, dict(nc=6, pair=True, noise=(0.0, 1e-3), shuffle=True, origin=1))],
    64: [(20, 2, LEGACY), (64, 67, dict(nc=16, pair=True, noise=(0.05, 0.0), nonuniform=True, origin=2))],
    128: [(70, 4, LEGACY), (128, 68, dict(nc=7, pair=True, noise=(0.0, 1e-3), shuffle=True, origin=3))],
    160: [(160, 69, dict(nc=15, pair=True, noise=(0.05, 0.0), nonuniform=True, origin=4))],
    256: [(256, 70, dict(nc=14, pair=True, noise=(0.0, 1e-3), shuffle=True, origin=5))],
    512: [(400, 71, dict(nc=16, pair=True, noise=(0.05, 0.0), nonuniform=True, origin=6))],
}


def build_trapezoid_cases(kind, specs, alias):
    out = []
    for ns, seed, opt in specs:
        opt = dict(opt)
        k = opt.pop("origin", None)
        c = trapezoid_case(kind, ns, seed, origin=None if k is None else boundary_observations()[k][0], **opt)
        rs = np.random.RandomState(seed + 1000)
        extra = [] if k is None else boundary_observations()[k][1]
        c["x_a"], c["aliased"] = query_points(rs, c["x_s"], c["x_c"], c["thresh"], c["lo"], c["hi"], 150 if ns <= 70 else 30,
                                              pair=c["pair"], alias=2 * np.pi * c["pl"][2] if (alias and kind) else None,
                                              extra=extra)
        out.append(c)
    return out


def conditioning(kind, x_s, x_c, ptl, pl):
    """(cond K_tl, cond of the bordered K_l(x_sc, x_sc) without noise, c_tl): what the error bounds scale with."""
    from oracle import approx
    p_tl, p_l = (ptl[2], pl[2]) if kind else (1.0, 1.0)
    K_tl = approx.kernel(kind, ptl[0], ptl[1], p_tl, x_s, x_s) + ptl[-1] ** 2 * np.eye(x_s.size)
    x_sc = np.concatenate([x_s, x_c])
    c_tl = ptl[0] ** 2 if kind else ptl[0] ** 2 / (np.sqrt(2 * np.pi) * ptl[1])
    return float(np.linalg.cond(K_tl)), float(np.linalg.cond(approx.kernel(kind, pl[0], pl[1], p_l, x_sc, x_sc))), c_tl


def expected_status(lib, esm, em, st):
    """The device's status bits for the oracle's outcome (bq.py:456-524): the branch taken, then the checks of the
    values the full computation produced."""
    want = np.array(st, dtype=np.int32)
    full = want == 0
    with np.errstate(invalid="ignore"):
        want[full & (np.isnan(esm) | (esm < 0))] |= lib.ST_ESM_BAD
    want[full & np.isnan(em)] |= lib.ST_EM_BAD
    want[full & np.isinf(esm)] |= lib.ST_ESM_INF
    want[full & np.isinf(em)] |= lib.ST_EM_INF
    return want


def worst(got, want, rtol, atol):
    """Largest |got - want| / (atol + rtol |want|): the share of the bound a result used."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    same = (got == want) | (np.isinf(got) & np.isinf(want) & (np.sign(got) == np.sign(want)))
    r = np.where(same, 0.0, np.abs(got - want) / (atol + rtol * np.abs(want)))
    return float(np.max(r)) if r.size else 0.0


def check_instance(lib, tag, info, i, b, x_a, esm, em, st, zm, zv, l_c, o, cond_tl, cond_l, c_tl, aliased, report):
    """One instance's device results against its oracle's: Z_mean, l_c, Z_var, status bits, esm, em, and the fused
    expected variance Zm^2 + Zv - esm of the choose_next epilogue.  `o` = (esm, em, status) of the oracle at x_a."""
    o_esm, o_em, o_st = o
    nc = l_c.size
    zv_tol = max(1e-13, 10 * (cond_tl + cond_l) * EPS * c_tl * zm ** 2)
    rel = np.where(aliased, max(RTOL, 1e4 * cond_l * EPS), RTOL)
    assert_close(info["Z_mean"][i], zm, "Z_mean " + tag)
    assert_close(info["l_c"][i, :nc], l_c, "l_c " + tag)
    assert abs(info["Z_var"][i] - zv) <= zv_tol, (tag, info["Z_var"][i], zv, zv_tol)
    want_st = expected_status(lib, o_esm, o_em, o_st)
    bad = np.nonzero(st != want_st)[0]
    assert bad.size == 0, (tag, "status", x_a[bad[:8]], st[bad[:8]], want_st[bad[:8]])
    for what, got, want in (("esm", esm, o_esm), ("em", em, o_em)):
        for sel, r in ((~aliased, RTOL), (aliased, float(rel.max()))):
            if sel.any():
                assert_close(got[sel], want[sel], "%s %s%s" % (what, tag, " (aliased)" if r != RTOL else ""), rtol=r, atol=ATOL)
    ev, _ = b.expected_var_host(x_a, inst=i)
    o_ev = zm ** 2 + zv - o_esm
    ev_tol = max(ATOL, zv_tol) + 2 * RTOL * zm ** 2 + rel * np.abs(o_esm)
    assert (np.abs(ev - o_ev) <= ev_tol).all(), (tag, "expected variance", float(np.max(np.abs(ev - o_ev) / ev_tol)))
    # the fused choose_next step of this instance alone: the batch launch's esm bit for bit, and (min, first index)
    import torch
    x_d = torch.from_numpy(x_a).cuda()
    esm_f, ev_f = torch.empty_like(x_d), torch.empty_like(x_d)
    pair = torch.empty(2, dtype=torch.float64, device=x_d.device)
    b.choose_step_device(x_d, esm_f, ev_f, pair, offset=3, inst=i)
    esm_f, ev_f, pair = esm_f.cpu().numpy(), ev_f.cpu().numpy(), pair.cpu().numpy()
    assert np.array_equal(esm_f, esm), (tag, "choose_step esm")
    assert (np.abs(ev_f - o_ev) <= ev_tol).all(), (tag, "choose_step expected variance")
    assert pair[0] == ev_f.min() and int(pair[1]) == 3 + int(np.argmin(ev_f)), (tag, pair)
    report.append("%s cond_tl %.2g cond_l %.2g | Z_mean %.2g l_c %.2g Z_var %.2g esm %.2g em %.2g ev %.2g%s" % (
        tag, cond_tl, cond_l, worst(info["Z_mean"][i], zm, RTOL, ATOL), worst(info["l_c"][i, :nc], l_c, RTOL, ATOL),
        abs(info["Z_var"][i] - zv) / zv_tol, worst(esm[~aliased], o_esm[~aliased], RTOL, ATOL),
        worst(em[~aliased], o_em[~aliased], RTOL, ATOL), float(np.max(np.abs(ev - o_ev) / ev_tol)),
        "" if not aliased.any() else " aliased esm %.2g em %.2g" % (worst(esm[aliased], o_esm[aliased], rel.max(), ATOL),
                                                                     worst(em[aliased], o_em[aliased], rel.max(), ATOL))))


def padded(rows):
    """Per-instance query vectors as one [B, na] array (short rows repeat their first point)."""
    na = max(r.size for r in rows)
    return np.stack([np.concatenate([r, np.full(na - r.size, r[0])]) for r in rows])


def assert_far_from_the_guard(tm, tC):
    """No exponent of int_exp_norm (bq_c.pyx:472-483) within 1e-9 relative of MAX_EXPONENT."""
    from oracle.approx import MAX_EXPONENT
    for a in (tm + 0.5 * tC, 2 * tm + 2 * tC):
        assert (np.abs(a - MAX_EXPONENT) > 1e-9 * MAX_EXPONENT).all()


def run_trapezoid_batch(lib, cap, kind, cases, report):
    from oracle import approx
    B = len(cases)
    ns = np.array([c["x_s"].size for c in cases], dtype=np.int32)
    nc = np.array([c["x_c"].size for c in cases], dtype=np.int32)
    assert max(lib.ns_capacity(int(n)) for n in ns) == cap
    X, L, XC = np.zeros((B, cap)), np.ones((B, cap)), np.zeros((B, 16))
    for i, c in enumerate(cases):
        X[i, :ns[i]], L[i, :ns[i]], XC[i, :nc[i]] = c["x_s"], c["l_s"], c["x_c"]
    hyp = np.array([[c["ptl"][0], c["ptl"][1], c["ptl"][-1], c["pl"][0], c["pl"][1], c["pl"][-1]] for c in cases])
    prior = np.array([[c["mu"], c["var"], c["thresh"]] for c in cases])
    b = lib.Batch(B, cap)
    b.set_approx(kind, period=np.array([[c["ptl"][2], c["pl"][2]] for c in cases]) if kind else None,
                 xo=np.stack([c["xo"] for c in cases]), p_xo=np.stack([c["p_xo"] for c in cases]))
    info = b.setup(ns, nc, X, L, XC, hyp, prior)
    assert (info["status"] == lib.SETUP_OK).all(), info["status"]
    esm, em, st = b.score_host(padded([c["x_a"] for c in cases]))
    for i, c in enumerate(cases):
        tag = "cap=%d kind=%d ns=%d nc=%d seed=%d" % (cap, kind, ns[i], nc[i], c["seed"])
        cond_tl, cond_l, c_tl = conditioning(kind, c["x_s"], c["x_c"], c["ptl"], c["pl"])
        assert cond_tl <= COND_MAX and cond_l <= COND_MAX, (tag, cond_tl, cond_l)
        m = approx.ApproxModel(c["x_s"], c["l_s"], c["x_c"], c["ptl"], c["pl"], c["mu"], c["var"], c["thresh"], kind,
                               c["xo"], c["p_xo"])
        x_a = c["x_a"]
        k_t = m.k_tl(x_a, m.x_s)
        assert_far_from_the_guard(k_t.dot(m.a_tl), m.k_tl([0.0], [0.0])[0, 0] - np.einsum("ij,jk,ik->i", k_t, m.inv_K_tl, k_t))
        na = x_a.size
        check_instance(lib, tag, info, i, b, x_a, esm[i, :na], em[i, :na], st[i, :na], m.Z_mean(), m.Z_var(), m.l_c,
                       m.esm_and_em(x_a), cond_tl, cond_l, c_tl, c["aliased"], report)
    b.close()


@pytest.mark.parametrize("cap", CLASSES)
def test_trapezoid_path_vs_numpy_oracle(lib, cap):
    """The periodic and the trapezoid path against the numpy restatement of the reference, one ragged batch per capacity
    class for each kernel (the periodic kernel, and the Gaussian kernel on a grid): ns at the class edges and off the
    multiples of 8, unsorted observations, widths tied to the spacing, periods p_tl != p_l (both != 1), 0 to 16
    candidates -- one, two and three blocks of dense rows -- with a pair closer than 2 candidate_thresh, observation
    noise on gp_log_l in some instances and on gp_l in others, a grid per instance (one of them non-uniform).  Query
    points at the shortcut and jitter boundaries, close to two candidates, aliased to an observation by one period
    (classes 16 and 64) and at the constructed isclose boundary."""
    report = []
    for kind, table in ((1, PERIODIC), (0, GAUSSIAN_TRAPEZOID)):
        run_trapezoid_batch(lib, cap, kind, build_trapezoid_cases(kind, table[cap], alias=cap <= 64), report)
    print("\n" + "\n".join(report))


def gaussian_case(ns, seed, nc, noise=(0.0, 0.0), origin=0.0, shuffle=False, pair=True):
    """Gaussian kernel with its closed-form integrals: observations 1.25 apart with the one nearest 0 exactly at
    `origin`, the likelihood and hyper-parameters of tests/test_gpu_setup.py, nc mid-gap candidates (with a pair 0.5
    apart), candidate_thresh 0.5."""
    from bayesian_quadrature_b200 import synthetic
    rs = np.random.RandomState(seed)
    x_s = 1.25 * (np.arange(ns, dtype=np.float64) - (ns - 1) // 2) + origin
    l_s = synthetic.likelihood(max(ns, 9))(x_s)
    x_c, pr = place_candidates(rs, x_s, 1.25, nc, pair and nc >= 2)
    opt = synthetic.options(max(ns, 9))
    if shuffle:
        p = rs.permutation(ns)
        x_s, l_s = x_s[p], l_s[p]
    return dict(x_s=x_s, l_s=l_s, x_c=x_c, pair=pr, hyp=np.array([15.0, 2.0, noise[0], 0.2, 1.3, noise[1]]),
                prior=np.array([opt["x_mean"], opt["x_var"], 0.5]), seed=seed)


def run_gaussian_batch(lib, oracle, cap, cases, x_rows, force_generic, check_max, report, tag0):
    B = len(cases)
    ns = np.array([c["x_s"].size for c in cases], dtype=np.int32)
    nc = np.array([c["x_c"].size for c in cases], dtype=np.int32)
    X, L, XC = np.zeros((B, cap)), np.ones((B, cap)), np.zeros((B, 16))
    for i, c in enumerate(cases):
        X[i, :ns[i]], L[i, :ns[i]], XC[i, :nc[i]] = c["x_s"], c["l_s"], c["x_c"]
    b = lib.Batch(B, cap)
    if force_generic:
        b.set_approx(0, force_generic=True)
    info = b.setup(ns, nc, X, L, XC, np.stack([c["hyp"] for c in cases]), np.stack([c["prior"] for c in cases]),
                   check_max=check_max)
    assert (info["status"] == lib.SETUP_OK).all(), info["status"]
    esm, em, st = b.score_host(padded(x_rows))
    for i, c in enumerate(cases):
        tag = "%s ns=%d nc=%d seed=%d" % (tag0, ns[i], nc[i], c["seed"])
        hyp, prior = c["hyp"], c["prior"]
        cond_tl, cond_l, c_tl = conditioning(0, c["x_s"], c["x_c"], hyp[:3], hyp[3:])
        assert cond_tl <= COND_MAX and cond_l <= COND_MAX, (tag, cond_tl, cond_l)
        m = oracle.OracleModel(c["x_s"], c["l_s"], c["x_c"], hyp[:3], hyp[3:], prior[0], prior[1], prior[2], check_max=check_max)
        x_a = x_rows[i]
        assert_far_from_the_guard(*m.gp_log_l_mean_cov(x_a))
        assert abs(info["log_lh"][i] - m.log_lh()) <= RTOL * abs(m.log_lh()), (tag, info["log_lh"][i], m.log_lh())
        na = x_a.size
        check_instance(lib, tag, info, i, b, x_a, esm[i, :na], em[i, :na], st[i, :na], m.Z_mean(), m.Z_var(), m.l_c,
                       m.esm_and_em(x_a), cond_tl, cond_l, c_tl, np.zeros(na, dtype=bool), report)
        m.close()
    b.close()


GAUSSIAN_GENERIC = {
    64: [(17, 2, 7, (0.0, 0.05), 0, True), (64, 3, 16, (1e-3, 0.0), 1, False), (37, 1, 0, (0.0, 0.05), 2, True)],
    256: [(161, 4, 15, (0.0, 0.05), 3, True), (256, 5, 6, (1e-3, 0.0), 4, False), (203, 6, 14, (0.0, 0.05), 5, True)],
    512: [(257, 7, 16, (0.0, 0.05), 6, True), (512, 8, 15, (1e-3, 0.0), 7, False), (301, 10, 7, (0.0, 0.05), 0, True)],
}


@pytest.mark.parametrize("cap", sorted(GAUSSIAN_GENERIC))
def test_gaussian_closed_forms_on_the_generic_kernel_vs_c_oracle(lib, oracle, cap):
    """The plain-FP64 kernel with the Gaussian kernel's closed-form integrals (forced below 257 observations, the only
    kernel of the 512 class) against the C restatement of the reference: 0 to 16 candidates, noise on gp_l (the s_l != 0
    re-factorisation of the setup kernel) or on gp_log_l, the guard of bq.py:942-947 on."""
    cases, rows, report = [], [], []
    for ns, seed, nc, noise, k, shuffle in GAUSSIAN_GENERIC[cap]:
        xs0, pts = boundary_observations()[k]
        c = gaussian_case(ns, seed, nc, noise, origin=xs0, shuffle=shuffle)
        rs = np.random.RandomState(seed + 2000)
        x_a, _ = query_points(rs, c["x_s"], c["x_c"], 0.5, c["x_s"].min() - 3, c["x_s"].max() + 3, 60, pair=c["pair"],
                              extra=list(pts) + [c["x_s"].min() - 100, c["x_s"].max() + 1e4])
        cases.append(c)
        rows.append(x_a)
    run_gaussian_batch(lib, oracle, cap, cases, rows, force_generic=True, check_max=True, report=report,
                       tag0="generic cap=%d" % cap)
    print("\n" + "\n".join(report))


@pytest.mark.parametrize("kernel", ["tc16", "tc64", "band128", "generic"])
def test_isclose_boundary_on_every_kernel(lib, oracle, kernel):
    """np.isclose(x_a, x_s, atol=1e-4) decides the shortcut of bq.py:456 with its tolerance rounded twice; points where a
    tolerance rounded once (fma) decides differently, next to observations near the origin, through the tensor-core
    kernels of the 16 and 64 classes, the band-relative kernel of the 128 class and the plain-FP64 kernel: the status
    bits are the reference's, and so are the scores."""
    cap, ns = {"tc16": (16, 9), "tc64": (64, 40), "band128": (128, 100), "generic": (64, 40)}[kernel]
    cases, rows, report = [], [], []
    for k, (xs0, pts) in enumerate(boundary_observations()[:4]):
        c = gaussian_case(ns, 10 + k, 2, origin=xs0, shuffle=bool(k & 1), pair=False)
        rs = np.random.RandomState(k)
        x_a = np.concatenate([pts, xs0 + np.array([0.0, 0.9e-4, -0.9e-4, 1.2e-4, -1.2e-4]),
                              rs.uniform(c["x_s"].min() - 3, c["x_s"].max() + 3, 40)])
        cases.append(c)
        rows.append(x_a)
    run_gaussian_batch(lib, oracle, cap, cases, rows, force_generic=kernel == "generic", check_max=False, report=report,
                       tag0=kernel)
    print("\n" + "\n".join(report))


def test_periodic_marginal_loss_vs_numpy_oracle():
    """BatchBQ(kernel=PeriodicKernel).marginal_loss -- P x S instances scored by the grouped launch (each sample's
    periods, its problem's own grid and candidates, per-problem query rows) and reduced in sample order -- against
    -mean_s esm of the numpy oracle under each sample."""
    from oracle import approx
    from bayesian_quadrature_b200 import BatchBQ, PeriodicKernel
    P, S, n = 3, 3, 9
    rs = np.random.RandomState(77)
    gap = 2 * np.pi / n
    x_s = np.stack([np.linspace(-np.pi, np.pi, n + 1)[:-1] + rs.uniform(-0.05, 0.05, n) * gap for _ in range(P)])
    l_s = np.stack([np.exp(-np.log(2 * np.pi) + (1.0 + 0.3 * p) * np.cos(x_s[p] - 0.4 * p)) for p in range(P)])
    ptl = np.array([[3.0, 1.2 * gap, 1.05 + 0.03 * p, 0.05] for p in range(P)])
    pl = np.array([[0.3, 0.7 * gap, 1.1 - 0.03 * p, 1e-3] for p in range(P)])
    bb = BatchBQ(x_s, l_s, ptl, pl, n_candidate=12, candidate_thresh=0.15, x_mean=0.0, x_var=10.0, seed=5, kernel=PeriodicKernel)
    assert (bb.nc >= 6).all() and (bb.nc >= 7).any()          # one and two blocks of dense rows
    params = ["h", "w", "p"]
    htl = ptl[:, None, :3] * rs.uniform(0.9, 1.1, (P, S, 3))
    hl = pl[:, None, :3] * rs.uniform(0.9, 1.1, (P, S, 3))
    x_a = np.stack([np.linspace(-np.pi * ptl[p, 2], np.pi * ptl[p, 2], 61)[:-1] + 0.01 * (p + 1) for p in range(P)])
    loss = bb.marginal_loss(x_a, htl, hl, params).cpu().numpy()
    for p in range(P):
        c = int(bb.nc[p])
        acc = np.zeros(x_a.shape[1])
        for s in range(S):
            t = (htl[p, s, 0], htl[p, s, 1], htl[p, s, 2], ptl[p, 3])
            l = (hl[p, s, 0], hl[p, s, 1], hl[p, s, 2], pl[p, 3])
            cond_tl, cond_l, _ = conditioning(1, x_s[p], bb.x_c[p, :c], t, l)
            assert cond_tl <= COND_MAX and cond_l <= COND_MAX, (p, s, cond_tl, cond_l)
            m = approx.ApproxModel(x_s[p], l_s[p], bb.x_c[p, :c], t, l, 0.0, 10.0, 0.15, 1, bb.xo[p], bb.p_xo[p])
            acc = acc - m.esm_and_em(x_a[p])[0]
        assert_close(loss[p], acc / S, "marginal loss of problem %d" % p)
    bb.close()
