"""GPU parity tests (run with -m gpu on the B200 box).  Every compute call goes through the
C-ABI (libbq_b200.so, via the ctypes binding) or the BQ class on top of it.

Checked against: (i) fixtures produced by the unmodified reference (tests/golden/*.npz),
(ii) the CPU oracle (oracle/bq_oracle.c) on seeded inputs, (iii) size-independent properties at
BASELINE.json's full sizes.  Tolerance: north_star's rtol 1e-9 / atol 1e-12 in float64 (conftest);
Z_var is a 6-10 digit cancellation and is judged by atol (SURVEY §7.2).
"""
import numpy as np
import pytest

from conftest import ATOL, RTOL, assert_close, load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    from bayesian_quadrature_b200 import _lib
    _lib.load()
    assert _lib.device_count() >= 1
    return _lib


def batch_of(lib, g, **kw):
    ns, nc = g["x_s"].size, g["x_c"].size
    b = lib.Batch(1, ns)
    hyp = np.concatenate([g["params_tl"], g["params_l"]])
    prior = np.array([float(g["x_mean"]), float(g["x_var"]), float(g["candidate_thresh"])])
    info = b.setup([ns], [nc], g["x_s"][None], g["l_s"][None], g["x_c"][None], hyp[None], prior[None], **kw)
    assert info["status"][0] == lib.SETUP_OK
    return b, info


@pytest.mark.parametrize("name", ["fixture", "c1", "c2", "c5", "c3"])
def test_capi_vs_reference_fixture(lib, name):
    g = load_golden(name)
    b, info = batch_of(lib, g)
    nc = g["x_c"].size
    assert_close(info["l_c"][0, :nc], g["l_c"], name + " l_c")
    assert_close(info["Z_mean"][0], g["Z_mean"], name + " Z_mean")
    assert abs(info["Z_var"][0] - float(g["Z_var"])) < 1e-13
    assert abs(info["log_lh"][0] - float(g["log_lh"])) <= RTOL * abs(float(g["log_lh"]))
    esm, em, st = b.score_host(g["x_a"])
    assert_close(esm[0], g["esm"], name + " esm")
    assert_close(em[0], g["em"], name + " em")
    assert ((st[0] & lib.ST_SHORTCUT) == g["shortcut"]).all()
    assert not (st[0] & (lib.ST_ESM_BAD | lib.ST_EM_BAD | lib.ST_XA_BAD)).any()
    ev = info["Z_mean"][0] ** 2 + info["Z_var"][0] - esm[0]
    assert_close(ev, g["expected_Z_var"], name + " expected_Z_var", atol=max(ATOL, 1e-13))
    ev2, flags = b.expected_var_host(g["x_a"])
    assert (ev2 == ev).all()
    if "grid_idx" in g and g["grid_idx"].size < g["x_a"].size:
        k = g["grid_idx"].size                       # the dense window around the peak is inside [:k]
        assert int(np.argmax(esm[0][:k])) == int(np.argmax(g["esm"][:k]))
    b.close()


@pytest.mark.parametrize("ns,seed", [(1, 0), (2, 1), (9, 2), (16, 3), (17, 4), (40, 5), (64, 6), (65, 7), (100, 8), (128, 9), (136, 12), (144, 13),
                                     (150, 10), (256, 11)])
def test_capi_vs_oracle_random(lib, oracle, ns, seed):
    """Seeded random problems of every capacity class, random + edge query points."""
    rs = np.random.RandomState(seed)
    x_s = np.sort(rs.uniform(-0.625 * ns, 0.625 * ns, ns)) if ns > 1 else np.array([0.3])
    if ns > 1:                                       # keep observations >= 0.6 apart (well conditioned)
        x_s = np.linspace(x_s.min(), x_s.max() + 0.6 * ns, ns) + rs.uniform(-0.2, 0.2, ns)
    l_s = np.exp(-0.5 * (x_s / (0.3 * max(np.ptp(x_s), 1.0))) ** 2) * rs.uniform(0.5, 1.5, ns) * 0.3 + 1e-3
    nc = int(rs.randint(0, 7))
    x_c = np.sort(rs.uniform(x_s.min() - 2, x_s.max() + 2, nc))
    if nc:
        keep = np.ones(nc, bool)
        for j in range(nc):
            if (np.abs(x_c[j] - x_s) < 0.5).any() or (j and keep[j - 1] and x_c[j] - x_c[j - 1] < 0.5):
                keep[j] = False
        x_c = x_c[keep]
        nc = x_c.size
    ptl, pl = (rs.uniform(3, 6), rs.uniform(1.0, 1.6), 0.0), (rs.uniform(0.2, 0.8), rs.uniform(0.8, 1.2), 0.0)
    mu, var, thresh = float(rs.uniform(-1, 1)), float(max(np.ptp(x_s), 2.0) ** 2 / 4), 0.5
    m = oracle.OracleModel(x_s, l_s, x_c, ptl, pl, mu, var, thresh)
    lo, hi = x_s.min() - 6, x_s.max() + 6
    x_a = np.concatenate([rs.uniform(lo, hi, 3000), x_s, x_s + 1.05e-4, x_s - 0.9e-4, x_c, x_c + 0.49, x_c - 0.5,
                          x_c + 0.25, [lo - 100, hi + 1e4]])
    b = lib.Batch(1, ns)
    info = b.setup([ns], [nc], x_s[None], l_s[None], x_c[None] if nc else np.zeros((1, 0)),
                   np.array([ptl + pl]), np.array([[mu, var, thresh]]))
    assert info["status"][0] == 0
    assert_close(info["Z_mean"][0], m.Z_mean(), "Z_mean")
    assert abs(info["Z_var"][0] - m.Z_var()) < 1e-12 * max(1.0, abs(m.Z_mean()) ** 2 * 1e3)
    esm, em, st = b.score_host(x_a)
    o_esm, o_em, o_st = m.esm_and_em(x_a)
    assert ((st[0] & 3) == (o_st & 3)).all()
    assert_close(esm[0], o_esm, "esm ns=%d" % ns)
    assert_close(em[0], o_em, "em ns=%d" % ns)
    b.close()


@pytest.mark.parametrize("ns,nc", [(64, 16), (100, 9), (128, 16), (150, 12), (200, 7), (256, 16)])
def test_many_candidates_vs_oracle(lib, oracle, ns, nc):
    """Up to NC_MAX = 16 candidates: two or three dense row blocks in the scoring kernels (and, in the resident classes,
    the fall-back to the streamed kernel when the scratch rows no longer fit).  A sorted grid (narrow bands: the fast
    path of the band-relative kernels) and unsorted scattered points (wide path) against the oracle."""
    rs = np.random.RandomState(77 + ns)
    x_s = np.linspace(-0.55 * ns, 0.55 * ns, ns) + rs.uniform(-0.2, 0.2, ns)
    l_s = np.exp(-0.5 * (x_s / (0.3 * np.ptp(x_s))) ** 2) * rs.uniform(0.5, 1.5, ns) * 0.3 + 1e-3
    left = x_s.min() - 1.1 * (1 + np.arange(nc // 2))
    right = x_s.max() + 1.1 * (1 + np.arange(nc - nc // 2))
    x_c = np.sort(np.concatenate([left, right]))
    ptl, pl = (4.0, 1.3, 0.0), (0.5, 1.0, 0.0)
    mu, var, thresh = 0.2, float(np.ptp(x_s) ** 2 / 4), 0.5
    m = oracle.OracleModel(x_s, l_s, x_c, ptl, pl, mu, var, thresh)
    b = lib.Batch(1, ns)
    info = b.setup([ns], [nc], x_s[None], l_s[None], x_c[None], np.array([ptl + pl]), np.array([[mu, var, thresh]]))
    assert info["status"][0] == 0
    assert_close(info["Z_mean"][0], m.Z_mean(), "Z_mean")
    lo, hi = x_c.min() - 4, x_c.max() + 4
    for name, x_a in (("grid", np.linspace(lo, hi, 4001)),
                      ("scattered", np.concatenate([rs.uniform(lo, hi, 1500), x_c, x_c + 0.49, x_c - 0.25, x_s[:5]]))):
        esm, em, st = b.score_host(x_a)
        o_esm, o_em, o_st = m.esm_and_em(x_a)
        assert ((st[0] & 3) == (o_st & 3)).all(), name
        assert_close(esm[0], o_esm, "%s esm ns=%d nc=%d" % (name, ns, nc))
        assert_close(em[0], o_em, "%s em ns=%d nc=%d" % (name, ns, nc))
    b.close()


@pytest.mark.parametrize("ns,shuffle", [(64, False), (64, True), (128, True), (150, False), (256, True), (256, False)])
def test_band_skipping_equals_the_dense_algorithm(lib, ns, shuffle):
    """The scoring kernels skip cross-kernel k-steps whose elements are below e^-72 of their point's leading element
    (DESIGN.md 4.1).  Against the same kernels with the cut-off at infinity (the dense algorithm): same scores to far
    below the parity tolerance on a sorted grid, on scattered points (where the hull criterion keeps more), on far-away
    points, and with observations in arbitrary order (appended observations are not sorted); and fewer DMMAs."""
    from bayesian_quadrature_b200 import synthetic
    rs = np.random.RandomState(ns)
    x_s, l_s = synthetic.observations(ns)
    perm = rs.permutation(ns) if shuffle else np.arange(ns)      # arbitrary observation order
    x_s, l_s = x_s[perm], l_s[perm]
    x_c = np.sort(rs.uniform(x_s.min(), x_s.max(), 3)) + 0.6
    x_c = x_c[(np.abs(x_c[:, None] - x_s[None, :]).min(axis=1) > 0.5)]
    opt = synthetic.options(ns)
    b = lib.Batch(1, ns)
    info = b.setup([ns], [x_c.size], x_s[None], l_s[None], x_c[None] if x_c.size else np.zeros((1, 0)),
                   np.array([synthetic.PARAMS_TL + synthetic.PARAMS_L]), np.array([[opt["x_mean"], opt["x_var"], 0.5]]))
    assert info["status"][0] == 0
    grid = synthetic.query_grid(ns, 20011)
    scattered = rs.uniform(grid[0], grid[-1], 20011)
    far = np.array([grid[0] - 1e3, grid[-1] + 1e6, 1e300, -1e300])
    for name, x_a in (("grid", grid), ("scattered", scattered), ("far", far)):
        b.set_cutoff(72.0)
        b.work_counter(True)
        esm, em, st = b.score_host(x_a)
        work_band = b.work_counter(True)
        b.set_cutoff(float("inf"))
        esm_d, em_d, st_d = b.score_host(x_a)
        work_dense = b.work_counter(False)
        assert (st == st_d).all()
        assert_close(esm[0], esm_d[0], "%s esm ns=%d" % (name, ns), rtol=1e-12, atol=1e-300)
        assert_close(em[0], em_d[0], "%s em ns=%d" % (name, ns), rtol=1e-12, atol=1e-300)
        assert 0 < work_band <= work_dense
        if name == "grid":                           # the setup kernel sorts the observations: whatever order they came in,
            assert work_band < 0.5 * work_dense, (work_band, work_dense)      # a tile's relevant k-steps are few and contiguous
    b.close()


@pytest.mark.parametrize("ns", [100, 128, 150, 200, 256])
def test_register_tile_variants_agree(lib, ns, monkeypatch):
    """The large capacity classes have two scoring kernels (bq_score.cu: BQB_REL = 0 absolute register tile, 1 the
    band-relative tile with 16 warps, the default) and, inside the band-relative one, a fast path (band fits the tile) and a
    wide path (windows regenerated per row block).  All of them compute the same sums over the same relevant k-steps in
    a different order: scores agree to ~1e-13, statuses exactly -- on a grid (narrow hulls: fast path), on unsorted
    scattered points without the pre-sort (hulls as wide as the domain: wide path), with every warp forced down the wide
    path, and with the dense cut-off."""
    from bayesian_quadrature_b200 import synthetic
    rs = np.random.RandomState(1000 + ns)
    x_s, l_s = synthetic.observations(ns)
    x_c = np.array([x_s.max() + 1.1, x_s.max() + 2.9])
    opt = synthetic.options(ns)
    b = lib.Batch(1, ns)
    info = b.setup([ns], [x_c.size], x_s[None], l_s[None], x_c[None],
                   np.array([synthetic.PARAMS_TL + synthetic.PARAMS_L]), np.array([[opt["x_mean"], opt["x_var"], 0.5]]))
    assert info["status"][0] == 0
    b.set_presort(0)
    grid = synthetic.query_grid(ns, 30011)
    scattered = rs.uniform(grid[0], grid[-1], 5003)
    ref = {}
    for rel, wide, cut in (("0", "0", 72.0), ("1", "0", 72.0), ("1", "1", 72.0), ("1", "0", float("inf"))):
        monkeypatch.setenv("BQB_REL", rel)
        monkeypatch.setenv("BQB_FORCE_WIDE", wide)
        b.set_cutoff(cut)
        for name, x_a in (("grid", grid), ("scattered", scattered)):
            esm, em, st = b.score_host(x_a)
            if name not in ref:
                ref[name] = (esm[0].copy(), em[0].copy(), st[0].copy())
                continue
            tag = "%s ns=%d rel=%s wide=%s cut=%g" % (name, ns, rel, wide, cut)
            assert (st[0] == ref[name][2]).all(), tag
            assert_close(esm[0], ref[name][0], "esm " + tag, rtol=1e-11, atol=1e-300)
            assert_close(em[0], ref[name][1], "em " + tag, rtol=1e-11, atol=1e-300)
    b.close()


@pytest.mark.parametrize("name,ns", [("c2", 64), ("c3", 256)])
def test_presort_of_scattered_query_points(lib, name, ns):
    """Query vectors in arbitrary order are sorted on the device by the host entry points, scored ascending and written
    back through the permutation: bit-identical results to scoring the sorted vector, whatever the pre-sort mode, for
    esm / em / status, for expected variance (pageable and page-locked arrays) and with invalid points in the vector."""
    import torch
    from bayesian_quadrature_b200 import synthetic
    g = load_golden(name)
    b, info = batch_of(lib, g)
    rs = np.random.RandomState(3)
    grid = synthetic.query_grid(ns, 50001)
    grid[77] = g["x_s"][3]                             # a shortcut point
    perm = rs.permutation(grid.size)
    x = grid[perm]
    esm_s, em_s, st_s = b.score_host(grid)             # sorted input: no sort
    ref = (esm_s[0][perm], em_s[0][perm], st_s[0][perm])
    for mode in (1, 0, 2):
        b.set_presort(mode)
        esm, em, st = b.score_host(x)
        assert np.array_equal(esm[0], ref[0]) and np.array_equal(em[0], ref[1]) and np.array_equal(st[0], ref[2]), mode
        ev, fl = b.expected_var_host(x)
        ev_pin, fl_pin = b.expected_var_host(torch.from_numpy(x).pin_memory().numpy(), out=torch.empty(x.size, dtype=torch.float64).pin_memory().numpy())
        want = info["Z_mean"][0] ** 2 + info["Z_var"][0] - ref[0]
        assert np.array_equal(ev, want) and np.array_equal(ev_pin, want), mode
        assert fl == fl_pin and (fl & lib.ST_SHORTCUT)
    b.set_presort(1)
    x_bad = x.copy()
    x_bad[[5, 40000]] = [np.nan, np.inf]
    esm, em, st = b.score_host(x_bad)
    assert (st[0][[5, 40000]] == lib.ST_XA_BAD).all() and np.isnan(esm[0][[5, 40000]]).all()
    ok = np.ones(x.size, bool); ok[[5, 40000]] = False
    assert np.array_equal(esm[0][ok], ref[0][ok])
    b.close()


def test_hyper_set_batch_vs_reference(lib):
    """C4 semantics: one instance per hyper-parameter set, shared x_a, marginal loss and argmin."""
    import torch
    g = load_golden("c4")
    H, ns, nc = g["hypers"].shape[0], g["x_s"].size, g["x_c"].size
    b = lib.Batch(H, ns)
    hyp = np.zeros((H, 6))
    hyp[:, 0], hyp[:, 1], hyp[:, 3], hyp[:, 4] = g["hypers"].T
    prior = np.tile([float(g["x_mean"]), float(g["x_var"]), float(g["candidate_thresh"])], (H, 1))
    info = b.setup(np.full(H, ns), np.full(H, nc), np.tile(g["x_s"], (H, 1)), np.tile(g["l_s"], (H, 1)),
                   np.tile(g["x_c"], (H, 1)), hyp, prior, check_max=True)
    assert (info["status"] == 0).all()
    assert_close(info["l_c"][:, :nc], g["l_c"], "c4 l_c")
    assert_close(info["Z_mean"], g["Z_mean"], "c4 Z_mean")
    esm, em, st = b.score_host(g["x_a"])
    assert_close(esm, g["esm"], "c4 esm")
    assert_close(em, g["em"], "c4 em")
    dev = torch.device("cuda", 0)
    x_d = torch.from_numpy(g["x_a"]).to(dev)
    esm_d = torch.empty(H, g["x_a"].size, dtype=torch.float64, device=dev)
    loss_d = torch.empty(g["x_a"].size, dtype=torch.float64, device=dev)
    b.score_device(x_d, esm_d)
    b.mean_neg_device(esm_d, loss_d)
    torch.cuda.synchronize()
    assert (esm_d.cpu().numpy() == esm).all()                      # host and device entry points agree bitwise
    assert_close(loss_d.cpu().numpy(), g["loss"], "c4 loss")
    mn, idx = b.argmin_device(loss_d)
    assert idx == int(g["argmin"]) and mn == loss_d.cpu().numpy().min()
    b.close()


@pytest.mark.parametrize("cap,lo", [(40, 20), (128, 70), (150, 10), (256, 100)])
def test_independent_problems_batch(lib, oracle, cap, lo):
    """C5 semantics: instances with different ns / nc / data in one batch, each with its own x_a -- in every kind of
    scoring kernel (resident, resident rolled, streamed), with observations in arbitrary order (the setup kernel sorts
    them) and instances far smaller than the batch's capacity class."""
    rs = np.random.RandomState(11 + cap)
    B = 6 if cap <= 128 else 4
    ns = rs.randint(lo, cap + 1, B)
    ns[0] = cap
    nc = rs.randint(0, 4, B)
    x_s, l_s, x_c = np.zeros((B, cap)), np.ones((B, cap)), np.zeros((B, 16))
    x_a = np.empty((B, 700))
    models = []
    for i in range(B):
        xs = 1.25 * (np.arange(ns[i]) - (ns[i] - 1) / 2.0) + rs.uniform(-0.1, 0.1, ns[i])
        ls = np.exp(-0.5 * ((xs - rs.uniform(-3, 3)) / 6.0) ** 2) * 0.2 + 1e-4
        xc = np.sort(rs.choice(xs[:-1], nc[i], replace=False) + 0.625)
        perm = rs.permutation(ns[i])
        xs, ls = xs[perm], ls[perm]
        x_s[i, :ns[i]], l_s[i, :ns[i]], x_c[i, :nc[i]] = xs, ls, xc
        x_a[i] = rs.uniform(xs.min() - 8, xs.max() + 8, 700)
        models.append(oracle.OracleModel(xs, ls, xc, (15, 2, 0), (0.2, 1.3, 0), 0.0, 10.0 * (ns[i] / 8.0) ** 2, 0.5))
    b = lib.Batch(B, cap)
    hyp = np.tile([15, 2, 0, 0.2, 1.3, 0], (B, 1)).astype(float)
    prior = np.stack([[0.0, 10.0 * (n / 8.0) ** 2, 0.5] for n in ns])
    info = b.setup(ns, nc, x_s, l_s, x_c, hyp, prior)
    assert (info["status"] == 0).all()
    esm, em, st = b.score_host(x_a)
    import torch
    dev = torch.device("cuda", 0)
    neg = torch.from_numpy(-esm).to(dev)
    mins = torch.empty(B, dtype=torch.float64, device=dev)
    idxs = torch.empty(B, dtype=torch.int64, device=dev)
    b.argmin_rows_device(neg, mins, idxs)                     # per-problem deterministic choose_next
    assert (idxs.cpu().numpy() == np.argmin(-esm, axis=1)).all() and (mins.cpu().numpy() == (-esm).min(axis=1)).all()
    for i in range(B):
        o_esm, o_em, o_st = models[i].esm_and_em(x_a[i])
        assert int(np.argmax(o_esm)) == int(idxs[i])          # same chosen point as the oracle
        assert_close(esm[i], o_esm, "problem %d esm" % i)
        assert_close(em[i], o_em, "problem %d em" % i)
        assert_close(info["Z_mean"][i], models[i].Z_mean(), "problem %d Z_mean" % i)
    b.close()


def test_status_codes_and_edge_sizes(lib):
    g = load_golden("fixture")
    b, info = batch_of(lib, g)
    Zm = info["Z_mean"][0]
    x = np.array([np.nan, np.inf, -np.inf, g["x_s"][2], g["x_s"][2] + 1e-8, g["x_s"][2] + 1e-10, 0.3])
    esm, em, st = b.score_host(x)
    assert (st[0][:3] == lib.ST_XA_BAD).all() and np.isnan(esm[0][:3]).all()
    assert (st[0][3:6] == lib.ST_SHORTCUT).all()
    assert (esm[0][3:6] == Zm * Zm).all() and (em[0][3:6] == Zm).all()      # exactly Z_mean^2 (bq.py:457-459)
    assert st[0][6] == lib.ST_OK
    # ragged sizes: empty, 1 point, sizes straddling warp / CTA tiles
    e0, _, _ = b.score_host(np.empty(0))
    assert e0.shape == (1, 0)
    xs = np.linspace(-9, 9, 1000)
    full, _, _ = b.score_host(xs)
    for n in (1, 7, 8, 9, 15, 16, 17, 127, 128, 129, 255, 257):
        part, _, _ = b.score_host(xs[:n])
        assert (part[0] == full[0][:n]).all()                                 # independent of tiling
    b.close()


def test_setup_failures_are_reported(lib):
    g = load_golden("fixture")
    b = lib.Batch(1, 9)
    hyp = np.array([[1000.0, 2.0, 0, 0.2, 1.3, 0]])
    prior = np.array([[0.0, 10.0, 0.5]])
    info = b.setup([9], [2], g["x_s"][None], g["l_s"][None], (g["x_c"] + 40.0)[None], hyp, prior, check_max=True)
    assert info["status"][0] == lib.SETUP_MEAN_TOO_LARGE                       # bq.py:945-947
    with pytest.raises(np.linalg.LinAlgError):
        b.score_host(np.zeros(3))
    # a numerically singular Gram matrix (length scale >> data range) fails the Cholesky like numpy's would
    info = b.setup([9], [2], g["x_s"][None], g["l_s"][None], g["x_c"][None], np.array([[15, 1e7, 0, 0.2, 1.3, 0]]), prior)
    assert info["status"][0] == lib.SETUP_KTL_NOTPD
    info = b.setup([9], [2], g["x_s"][None], -g["l_s"][None], g["x_c"][None], np.array([[15, 2.0, 0, 0.2, 1.3, 0]]), prior)
    assert info["status"][0] == lib.SETUP_BAD_INPUT
    b.close()
    with pytest.raises(NotImplementedError):
        lib.Batch(1, 10 ** 4)


def test_capi_misuse_is_reported_not_ignored(lib):
    """Argument / state errors come back as the reference's exception types (ValueError / NotImplementedError /
    RuntimeError), never as silent no-ops."""
    import torch
    g = load_golden("fixture")
    b = lib.Batch(2, 9)
    with pytest.raises(lib.BQB200Error):                       # nothing set up yet (BQB_ESTATE)
        b.score_host(np.zeros(3))
    with pytest.raises(lib.BQB200Error):
        b.draw_candidates(4)
    with pytest.raises(NotImplementedError):                   # more than 16 candidates
        b.setup([9, 9], [17, 2], np.tile(g["x_s"], (2, 1)), np.tile(g["l_s"], (2, 1)), np.zeros((2, 16)),
                np.tile([15, 2.0, 0, 0.2, 1.3, 0], (2, 1)), np.tile([0.0, 10.0, 0.5], (2, 1)))
    hyp, prior = np.tile([15, 2.0, 0, 0.2, 1.3, 0], (2, 1)), np.tile([0.0, 10.0, 0.5], (2, 1))
    b.stage([9, 9], np.tile(g["x_s"], (2, 1)), np.tile(g["l_s"], (2, 1)), hyp, prior)
    with pytest.raises(lib.BQB200Error):                       # generators not seeded
        b.draw_candidates(4)
    with pytest.raises(ValueError):
        b.seed_candidates([1, 2, 3])
    b.seed_candidates([1, 2])
    with pytest.raises(NotImplementedError):
        b.draw_candidates(17)
    b.draw_candidates(10)
    info = b.setup_device()
    assert (info["status"] == 0).all()
    with pytest.raises(ValueError):
        b.set_cutoff(-1.0)
    with pytest.raises(ValueError):
        b.set_presort(3)
    # appending beyond the batch's observation capacity (16 for ns <= 16) is refused, not dropped
    far = torch.tensor([100.0, 200.0], dtype=torch.float64, device="cuda")
    one = torch.ones(2, dtype=torch.float64, device="cuda")
    for k in range(b.capacity - 9):
        b.add_observations(far + 10.0 * k, one)
    with pytest.raises(NotImplementedError):
        b.add_observations(far + 1e4, one)
    assert (b.get_staged()["ns"] == b.capacity).all()
    b.close()


def test_full_size_properties_c2(lib, oracle):
    """BASELINE configs[1] at full size (ns=64, 10^6 points): determinism, tiling independence,
    non-negativity, device argmin == host argmin, and a 4000-point subsample against the oracle."""
    import torch
    from bayesian_quadrature_b200 import synthetic
    g = load_golden("c2")
    b, info = batch_of(lib, g)
    grid = synthetic.query_grid(64, 10 ** 6)
    dev = torch.device("cuda", 0)
    x_d = torch.from_numpy(grid).to(dev)
    esm = torch.empty(1, grid.size, dtype=torch.float64, device=dev)
    em = torch.empty_like(esm)
    st = torch.empty(1, grid.size, dtype=torch.int32, device=dev)
    flags = torch.zeros(1, dtype=torch.int32, device=dev)
    b.score_device(x_d, esm, em, st, flags)
    torch.cuda.synchronize()
    esm2 = torch.empty_like(esm)
    b.score_device(x_d, esm2)
    half = grid.size // 2 + 13
    esm3 = torch.empty_like(esm)
    b.score_device(x_d[:half], esm3[:, :half])
    b.score_device(x_d[half:], esm3[:, half:])
    torch.cuda.synchronize()
    assert torch.equal(esm, esm2) and torch.equal(esm, esm3)
    e = esm[0].cpu().numpy()
    s = st[0].cpu().numpy()
    assert (e >= 0).all() and np.isfinite(e).all()
    assert int(flags.item()) == int(np.bitwise_or.reduce(s))
    assert not (s & ~(lib.ST_SHORTCUT | lib.ST_NOTPD)).any()
    # the fixture's grid subset must reproduce the reference at the same grid points
    k = g["grid_idx"].size
    assert_close(e[g["grid_idx"]], g["esm"][:k], "c2 full-grid esm at fixture indices")
    ev = torch.empty(grid.size, dtype=torch.float64, device=dev)
    b.expected_var_device(0, esm, ev)
    mn, idx = b.argmin_device(ev)
    ev_h = ev.cpu().numpy()
    assert idx == int(np.argmin(ev_h)) and mn == ev_h.min()
    pair = torch.empty(2, dtype=torch.float64, device=dev)
    b.argmin_pair_device(ev[1000:], 1000, pair)                   # sharded form: offset = start of the shard
    pr = pair.cpu().numpy()
    assert pr[0] == ev_h[1000:].min() and int(pr[1]) == 1000 + int(np.argmin(ev_h[1000:]))
    # fused step: same esm / ev bit for bit, same (min, index)
    esm_f, ev_f = torch.empty(grid.size, dtype=torch.float64, device=dev), torch.empty(grid.size, dtype=torch.float64, device=dev)
    b.choose_step_device(x_d, esm_f, ev_f, pair, offset=7)
    pr = pair.cpu().numpy()
    assert torch.equal(esm_f, esm[0]) and torch.equal(ev_f, ev)
    assert pr[0] == ev_h.min() and int(pr[1]) == 7 + int(np.argmin(ev_h))
    assert idx == int(g["grid_idx"][int(np.argmax(g["esm"][:k]))])          # same chosen point as the reference
    sub = np.random.RandomState(5).choice(grid.size, 4000, replace=False)
    m = oracle.OracleModel(g["x_s"], g["l_s"], g["x_c"], g["params_tl"], g["params_l"], float(g["x_mean"]),
                           float(g["x_var"]), float(g["candidate_thresh"]))
    o_esm, o_em, o_st = m.esm_and_em(grid[sub])
    assert_close(e[sub], o_esm, "c2 subsample esm")
    assert_close(em[0].cpu().numpy()[sub], o_em, "c2 subsample em")
    assert ((s[sub] & 3) == (o_st & 3)).all()
    b.close()


def test_full_size_properties_c3(lib, oracle, monkeypatch):
    """BASELINE configs[2] at full size (ns=256, 10^7 points) on one GPU, through the band-relative streamed kernel:
    determinism, tiling independence, non-negativity, the reference at the fixture's grid points, device argmin == host
    argmin == the reference's choice, agreement with the absolute-tile kernel (BQB_REL=0) over all 10^7 points, and a
    300-point subsample against the oracle."""
    import torch
    from bayesian_quadrature_b200 import synthetic
    g = load_golden("c3")
    b, info = batch_of(lib, g)
    na = int(g["na_full"])
    grid = synthetic.query_grid(256, na)
    dev = torch.device("cuda", 0)
    x_d = torch.from_numpy(grid).to(dev)
    esm = torch.empty(1, na, dtype=torch.float64, device=dev)
    em = torch.empty_like(esm)
    st = torch.empty(1, na, dtype=torch.int32, device=dev)
    b.score_device(x_d, esm, em, st)
    esm2 = torch.empty_like(esm)
    b.score_device(x_d, esm2)
    cut = na // 3 + 5
    esm3 = torch.empty_like(esm)
    b.score_device(x_d[:cut], esm3[:, :cut])
    b.score_device(x_d[cut:], esm3[:, cut:])
    torch.cuda.synchronize()
    assert torch.equal(esm, esm2) and torch.equal(esm, esm3)
    monkeypatch.setenv("BQB_REL", "0")                           # the absolute-tile kernel: same sums, other order
    esm_abs = torch.empty_like(esm)
    b.score_device(x_d, esm_abs)
    torch.cuda.synchronize()
    monkeypatch.delenv("BQB_REL")
    e, e_abs = esm[0].cpu().numpy(), esm_abs[0].cpu().numpy()
    s = st[0].cpu().numpy()
    assert (e >= 0).all() and np.isfinite(e).all()
    assert not (s & ~(lib.ST_SHORTCUT | lib.ST_NOTPD)).any()
    assert_close(e, e_abs, "c3 band-relative vs absolute tile", rtol=1e-11, atol=1e-300)
    k = g["grid_idx"].size
    assert_close(e[g["grid_idx"]], g["esm"][:k], "c3 full-grid esm at fixture indices")
    assert_close(em[0].cpu().numpy()[g["grid_idx"]], g["em"][:k], "c3 full-grid em at fixture indices")
    ev, pair = torch.empty(na, dtype=torch.float64, device=dev), torch.empty(2, dtype=torch.float64, device=dev)
    esm_f = torch.empty(na, dtype=torch.float64, device=dev)
    b.choose_step_device(x_d, esm_f, ev, pair, offset=0)
    pr, ev_h = pair.cpu().numpy(), ev.cpu().numpy()
    assert torch.equal(esm_f, esm[0])
    assert pr[0] == ev_h.min() and int(pr[1]) == int(np.argmin(ev_h))
    gi = g["grid_idx"]                                           # among the fixture's points: the reference's choice
    assert int(gi[int(np.argmin(ev_h[gi]))]) == int(gi[int(np.argmax(g["esm"][:k]))])
    sub = np.random.RandomState(6).choice(na, 300, replace=False)
    m = oracle.OracleModel(g["x_s"], g["l_s"], g["x_c"], g["params_tl"], g["params_l"], float(g["x_mean"]),
                           float(g["x_var"]), float(g["candidate_thresh"]))
    o_esm, o_em, o_st = m.esm_and_em(grid[sub])
    assert_close(e[sub], o_esm, "c3 subsample esm")
    assert ((s[sub] & 3) == (o_st & 3)).all()
    b.close()


# ---------------------------------------------------------------------------------------------- round-2 edge fixtures
from conftest import truth_bound, truth_err  # noqa: E402


@pytest.mark.parametrize("name", ["edge_inf45", "edge_inf90"])
def test_overflow_guards_vs_reference(lib, name):
    """gauss_c.pyx:87-91 / bq_c.pyx:472-483 through the C-ABI: the same points are +inf as in the reference (esm only for
    h_tl = 45, esm and em for h_tl = 90), flagged ST_ESM_INF / ST_EM_INF; finite values agree with the reference and sit no
    further from the multi-precision truth than the envelope."""
    g = load_golden(name)
    b, info = batch_of(lib, g)
    esm, em, st = b.score_host(g["x_a"])
    esm, em, st = esm[0], em[0], st[0]
    assert (np.isinf(esm) == np.isinf(g["esm"])).all() and (np.isinf(em) == np.isinf(g["em"])).all()
    assert (esm[np.isinf(esm)] > 0).all() and (em[np.isinf(em)] > 0).all()
    assert (((st & lib.ST_ESM_INF) != 0) == np.isinf(g["esm"])).all()
    assert (((st & lib.ST_EM_INF) != 0) == np.isinf(g["em"])).all()
    assert not (st & (lib.ST_ESM_BAD | lib.ST_EM_BAD | lib.ST_NOTPD)).any()
    bound = truth_bound(g)
    assert truth_err(esm, g["truth_esm"]).max() <= bound
    assert truth_err(em, g["truth_em"]).max() <= bound
    assert_close(esm, g["esm"], name + " esm", rtol=bound)
    assert_close(em, g["em"], name + " em", rtol=bound)
    ev, flags = b.expected_var_host(g["x_a"])
    assert flags & lib.ST_ESM_INF and (np.isneginf(ev) == np.isinf(g["esm"])).all()
    b.close()


def test_observation_noise_vs_reference(lib):
    """s_tl = 0.3, s_l = 0.05 (SURVEY appendix A.2): K_tl + s_tl^2 I everywhere, alpha_l with s_l^2, bordered matrix without."""
    g = load_golden("edge_noise")
    b, info = batch_of(lib, g)
    assert_close(info["l_c"][0, :g["x_c"].size], g["l_c"], "l_c")
    assert_close(info["Z_mean"][0], g["Z_mean"], "Z_mean")
    assert abs(info["Z_var"][0] - float(g["Z_var"])) < 1e-13
    assert abs(info["log_lh"][0] - float(g["log_lh"])) <= RTOL * abs(float(g["log_lh"]))
    esm, em, st = b.score_host(g["x_a"])
    assert_close(esm[0], g["esm"], "esm")
    assert_close(em[0], g["em"], "em")
    assert ((st[0] & lib.ST_SHORTCUT) == g["shortcut"]).all()
    b.close()


@pytest.mark.parametrize("tag", ["a", "b", "c", "d"])
def test_conditioning_sweep_against_truth(lib, tag):
    """SURVEY 7.1 / VERDICT r01 weak #2: ns = 64 with (w_tl, w_l) = (2.0, 1.3) / (2.7, 1.66) / (3.5, 2.0) / (2.0, 2.5), i.e.
    cond(K_tl) = 1.4e5 / 3.5e9 / 7.8e15 / 1.4e5 and cond(K_l) up to 2.4e12.  The kernel uses explicit inverse factors
    (c L^-1 as DMMA operand); this measures where that stops being admissible: its error against the multi-precision
    truth must stay inside the envelope the reference's own error defines (conftest.truth_bound)."""
    g = load_golden("illcond_" + tag)
    b, info = batch_of(lib, g)
    esm, em, st = b.score_host(g["x_a"])
    ref = truth_err(g["esm"], g["truth_esm"])
    got = truth_err(esm[0], g["truth_esm"])
    got_em = truth_err(em[0], g["truth_em"])
    ref_em = truth_err(g["em"], g["truth_em"])
    print("illcond_%s cond_tl %.3g cond_l %.3g: esm err vs truth  cuda max %.3g median %.3g | reference max %.3g median %.3g ; "
          "em cuda max %.3g reference max %.3g" % (tag, float(g["cond_K_tl"]), float(g["cond_K_l"]), got.max(), np.median(got),
                                                    ref.max(), np.median(ref), got_em.max(), ref_em.max()))
    assert ((st[0] & lib.ST_SHORTCUT) == g["shortcut"]).all()
    assert not (st[0] & (lib.ST_ESM_BAD | lib.ST_EM_BAD | lib.ST_NOTPD)).any()
    if tag == "c":      # cond 7.8e15: rounding noise in any float64 implementation (reference: 170 % off); only sanity
        assert np.isfinite(esm[0]).all() and np.median(got) <= max(10 * np.median(ref), 1e-3)
        return
    bound = truth_bound(g)
    assert got.max() <= bound and got_em.max() <= bound
    assert abs(info["Z_mean"][0] - float(g["truth_Z_mean"])) <= bound * abs(float(g["truth_Z_mean"]))
    if tag == "a":      # well conditioned: plain parity with the reference as well
        assert_close(esm[0], g["esm"], "esm")
    b.close()


@pytest.mark.parametrize("ns,nc", [(64, 4), (40, 2), (17, 0), (64, 6)])
def test_64_class_kernel_vs_oracle(lib, oracle, ns, nc):
    """The scoring kernel of the 64-observation class against the oracle, with the relevance cut-off and dense: a grid,
    scattered points, shortcut / near-shortcut points, points on and near the candidates (jitter patterns) and invalid
    points."""
    from bayesian_quadrature_b200 import synthetic
    rs = np.random.RandomState(ns)
    x_s, l_s = synthetic.observations(ns)
    x_c = np.sort(np.concatenate([x_s.max() + 1.1 + 1.3 * np.arange(nc // 2), x_s.min() - 0.9 - 1.2 * np.arange(nc - nc // 2)]))
    opt = synthetic.options(ns)
    b = lib.Batch(1, ns)
    info = b.setup([ns], [nc], x_s[None], l_s[None], x_c[None] if nc else np.zeros((1, 0)),
                   np.array([synthetic.PARAMS_TL + synthetic.PARAMS_L]), np.array([[opt["x_mean"], opt["x_var"], 0.5]]))
    assert info["status"][0] == 0
    m = oracle.OracleModel(x_s, l_s, x_c, synthetic.PARAMS_TL, synthetic.PARAMS_L, opt["x_mean"], opt["x_var"], 0.5)
    grid = synthetic.query_grid(ns, 20011)
    pts = np.concatenate([rs.uniform(grid[0], grid[-1], 3001), x_s[:7], x_s[:7] + 0.9e-4, x_c, x_c + 0.3, [np.nan, 1e7, -np.inf]])
    for cut in (72.0, float("inf")):
        b.set_cutoff(cut)
        for name, x_a in (("grid", grid), ("points", pts)):
            tag = "%s ns=%d nc=%d cut=%g" % (name, ns, nc, cut)
            esm, em, st = b.score_host(x_a)
            o_esm, o_em, o_st = m.esm_and_em(x_a)
            assert ((st[0] & 3) == (o_st & 3)).all(), tag
            ok = np.isfinite(x_a)
            assert_close(esm[0][ok], o_esm[ok], "esm " + tag)
            assert_close(em[0][ok], o_em[ok], "em " + tag)
    b.close()


def test_full_size_properties_c4(lib, oracle):
    """BASELINE configs[3] at full size (1024 hyper-parameter sets x 10^5 points, ns = 64): every set through the semantics of
    _set_gp_log_l_params (guard on), the marginal loss accumulated chunk by chunk in sample order == the one-shot mean over
    the materialised [1024, 10^5] matrix bit for bit, independent of the chunk size, deterministic; device argmin == host
    argmin; 16 points of the loss against the oracle's mean over ALL 1024 sets, and three whole sets on a 500-point subsample."""
    import torch
    from bayesian_quadrature_b200 import synthetic
    g = load_golden("c2")
    ns, nc, n_hyper, na = 64, g["x_c"].size, 1024, 10 ** 5
    hyp4 = synthetic.hyper_sets(n_hyper)
    hyp = np.zeros((n_hyper, 6))
    hyp[:, 0], hyp[:, 1], hyp[:, 3], hyp[:, 4] = hyp4.T
    prior = np.tile([float(g["x_mean"]), float(g["x_var"]), float(g["candidate_thresh"])], (n_hyper, 1))
    b = lib.Batch(n_hyper, ns)
    info = b.setup(np.full(n_hyper, ns), np.full(n_hyper, nc), np.tile(g["x_s"], (n_hyper, 1)), np.tile(g["l_s"], (n_hyper, 1)),
                   np.tile(g["x_c"], (n_hyper, 1)), hyp, prior, check_max=True)
    assert (info["status"] == 0).all()
    dev = torch.device("cuda", 0)
    grid = synthetic.query_grid(ns, na)
    x_d = torch.from_numpy(grid).to(dev)

    def chunked(chunk):
        esm = torch.empty(chunk, na, dtype=torch.float64, device=dev)
        flags = torch.zeros(chunk, dtype=torch.int32, device=dev)
        acc = torch.zeros(na, dtype=torch.float64, device=dev)
        seen = 0
        for i0 in range(0, n_hyper, chunk):
            cnt = min(chunk, n_hyper - i0)
            b.score_device_range(i0, cnt, x_d, esm, None, None, flags)
            b.sum_neg_accum_device(esm, cnt, acc)
            seen |= int(np.bitwise_or.reduce(flags[:cnt].cpu().numpy()))
        return acc / n_hyper, seen
    loss74, fl = chunked(74)
    loss74b, _ = chunked(74)
    loss37, _ = chunked(37)
    assert not fl & ~(lib.ST_SHORTCUT | lib.ST_NOTPD)
    assert torch.equal(loss74, loss74b) and torch.equal(loss74, loss37)
    full = torch.empty(n_hyper, na, dtype=torch.float64, device=dev)            # 819 MB: what round 1 materialised
    b.score_device(x_d, full)
    loss_full = torch.empty(na, dtype=torch.float64, device=dev)
    b.mean_neg_device(full, loss_full)
    assert torch.equal(loss_full, loss74)
    lh = loss74.cpu().numpy()
    assert np.isfinite(lh).all() and (lh <= 0).all()
    mn, idx = b.argmin_device(loss74)
    assert idx == int(np.argmin(lh)) and mn == lh.min()
    # the oracle: the loss at 16 grid points over ALL 1024 sets, and three sets on 500 points
    pts = np.unique(np.concatenate([np.linspace(0, na - 1, 14).astype(np.int64), [idx, min(idx + 1, na - 1)]]))
    sub = np.random.RandomState(7).choice(na, 500, replace=False)
    acc = np.zeros(pts.size)
    for i in range(n_hyper):
        m = oracle.OracleModel(g["x_s"], g["l_s"], g["x_c"], (hyp[i, 0], hyp[i, 1], 0.0), (hyp[i, 3], hyp[i, 4], 0.0), float(g["x_mean"]),
                               float(g["x_var"]), float(g["candidate_thresh"]), check_max=True)
        o_esm, _, _ = m.esm_and_em(grid[pts])
        acc += -o_esm
        if i in (0, 511, 1023):
            o_sub, _, _ = m.esm_and_em(grid[sub])
            assert_close(full[i].cpu().numpy()[sub], o_sub, "c4 hyper set %d esm" % i)
            assert_close(info["Z_mean"][i], m.Z_mean(), "Z_mean[%d]" % i)
            assert_close(info["l_c"][i, :nc], m.l_c, "l_c[%d]" % i)
        m.close()
    assert_close(lh[pts], acc / n_hyper, "c4 marginal loss vs the oracle over all 1024 sets")
    b.close()


def test_full_size_properties_c5_round(lib, oracle):
    """One active-sampling round of BASELINE configs[4] at full size (16384 independent problems x 4096 points, ns = 128):
    device-resident and host-driven batches draw the same candidates (per-problem numpy-compatible MT19937 streams) and
    choose the same points; scores are deterministic; the per-problem device argmin equals the host argmin of the score
    rows; eight problems against the oracle on a 256-point subsample."""
    import torch
    from bayesian_quadrature_b200 import BatchBQ, synthetic
    P, ns, na = 16384, 128, 4096
    opt = synthetic.options(ns)
    x0, _ = synthetic.observations(ns)
    sp = synthetic.span(ns)
    shifts = np.array([synthetic.problem_shift(p) for p in range(P)])
    npdf = lambda x, m, s: np.exp(-0.5 * ((x - m) / s) ** 2) / (np.sqrt(2 * np.pi) * s)
    lik = lambda x: (0.5 * npdf(x, (-0.3 + shifts[:, 0]) * sp, 0.16 * sp) + 0.3 * npdf(x, (0.4 + shifts[:, 1]) * sp, 0.10 * sp)
                     + 0.2 * npdf(x, (0.1 + shifts[:, 2]) * sp, 0.3 * sp))
    l0 = np.stack([lik(np.full(P, x)) for x in x0], axis=1)
    args = (np.tile(x0, (P, 1)), l0, synthetic.PARAMS_TL, synthetic.PARAMS_L, opt["n_candidate"], opt["candidate_thresh"],
            opt["x_mean"], opt["x_var"])
    dev_b = BatchBQ(*args, seed=synthetic.SEED, device_resident=True)
    host_b = BatchBQ(*args, seed=synthetic.SEED)          # same ns_reserve -> same capacity class -> the same kernels
    dev_b.sync_host()
    assert np.array_equal(dev_b.nc, host_b.nc) and np.array_equal(dev_b.x_c, host_b.x_c)
    assert np.array_equal(dev_b.Z_mean(), host_b.Z_mean())
    grid = synthetic.query_grid(ns, na)
    grid_d = torch.from_numpy(grid).cuda()
    idx_d, x_d = dev_b.choose_next(grid_d, on_device=True)
    loss1 = dev_b._esm.clone()
    idx_d2, _ = dev_b.choose_next(grid_d, on_device=True)
    assert torch.equal(loss1, dev_b._esm) and torch.equal(idx_d, idx_d2)              # deterministic
    idx_h, x_h = host_b.choose_next(grid)
    assert np.array_equal(idx_d.cpu().numpy(), idx_h) and np.array_equal(x_d.cpu().numpy(), x_h)
    loss = loss1.cpu().numpy()                                                        # -esm
    assert np.isfinite(loss).all() and (loss <= 0).all()
    assert np.array_equal(loss.argmin(axis=1), idx_h)
    sub = np.random.RandomState(8).choice(na, 256, replace=False)
    for p in (0, 1, 777, 4095, 8192, 12345, 16000, 16383):
        c = host_b.nc[p]
        m = oracle.OracleModel(host_b.x_s[p, :ns], host_b.l_s[p, :ns], host_b.x_c[p, :c], synthetic.PARAMS_TL, synthetic.PARAMS_L,
                               opt["x_mean"], opt["x_var"], opt["candidate_thresh"])
        o_esm, _, _ = m.esm_and_em(grid[sub])
        assert_close(-loss[p, sub], o_esm, "c5 problem %d esm" % p)
        assert_close(host_b.Z_mean()[p], m.Z_mean(), "Z_mean[%d]" % p)
        m.close()
    # the round's update: same merged / appended observations on both sides
    l_new = lik(x_h)
    host_b.add_observations(x_h, l_new)
    dev_b.add_observations(x_d, torch.from_numpy(l_new).cuda())
    dev_b.sync_host()
    assert np.array_equal(dev_b.ns, host_b.ns)
    n1 = int(host_b.ns.max())
    assert np.array_equal(dev_b.x_s[:, :n1], host_b.x_s[:, :n1]) and np.array_equal(dev_b.x_c, host_b.x_c)
    assert np.array_equal(dev_b.Z_mean(), host_b.Z_mean())
    dev_b.close()
    host_b.close()
