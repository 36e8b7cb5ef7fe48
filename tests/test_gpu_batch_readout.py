"""BatchBQ's per-point read-outs (expected_Z_var, expected_squared_mean, expected_mean, expected_squared_mean_and_mean,
l_mean, l_var) against a loop of BQ objects in every capacity class and with the periodic kernel, host against
device-resident mode, on_device against host results; the row-wise expected-variance kernel
(bqb_expected_var_rows_device) against bqb_expected_var_host; the error semantics; and the model they must leave alone."""
import logging

import numpy as np
import pytest

from conftest import assert_close

pytestmark = pytest.mark.gpu

SEED = 8728
METHODS = ("expected_Z_var", "expected_squared_mean", "expected_mean", "expected_squared_mean_and_mean", "l_mean", "l_var")
PARAMS_TL, PARAMS_L = (3.0, 1.2, 1.0, 0.0), (0.3, 0.8, 1.0, 0.0)     # periodic (h, w, p, s), tests/test_gpu_batch_periodic.py
OPT_PERIODIC = dict(n_candidate=10, candidate_thresh=0.5, x_mean=0.0, x_var=10.0)


def gaussian_case(ns0, P=3, device_resident=False):
    """P synthetic problems of ns0 observations (per-problem mixture centres); problem 1 has a noisy gp_l (s_l = 1e-3), so
    that its l_mean / l_var come from the host GPs in every class.  ns_reserve = 0: the batch runs the capacity class of
    ns0, as each problem's BQ object does while two rounds keep ns in that class."""
    from bayesian_quadrature_b200 import BQ, BatchBQ, GaussianKernel, synthetic
    x0, _ = synthetic.observations(ns0)
    fl = [synthetic.likelihood(ns0, synthetic.problem_shift(p)) for p in range(P)]
    opt = synthetic.options(ns0)
    ptl = np.tile(synthetic.PARAMS_TL, (P, 1))
    pl = np.tile(synthetic.PARAMS_L, (P, 1))
    pl[1, 2] = 1e-3
    bb = BatchBQ(np.tile(x0, (P, 1)), np.stack([f(x0) for f in fl]), ptl, pl, opt["n_candidate"], opt["candidate_thresh"],
                 opt["x_mean"], opt["x_var"], seed=SEED, ns_reserve=0, device_resident=device_resident)

    def bq_objects():
        bqs, states = [], []
        for p in range(P):
            np.random.seed(SEED + p)                       # BatchBQ's candidate stream of problem p
            bq = BQ(x0, fl[p](x0), kernel=GaussianKernel, **opt)
            bq.init(params_tl=tuple(ptl[p]), params_l=tuple(pl[p]))
            bqs.append(bq)
            states.append(np.random.get_state())
        return bqs, states
    span = synthetic.span(ns0)
    return bb, fl, bq_objects, np.linspace(-2 * span, 2 * span, 301)


def periodic_case(P=3, device_resident=False):
    from bayesian_quadrature_b200 import BQ, BatchBQ, PeriodicKernel
    from scipy.special import iv
    x0 = np.linspace(-np.pi, np.pi, 6)[:-1]
    fl = [(lambda mu, k: (lambda x: np.exp(-np.log(2 * np.pi * iv(0, k)) + k * np.cos(np.asarray(x) - mu))))(0.3 * p - 0.4,
                                                                                                         1.1 + 0.2 * p)
          for p in range(P)]
    bb = BatchBQ(np.tile(x0, (P, 1)), np.stack([f(x0) for f in fl]), PARAMS_TL, PARAMS_L, seed=SEED, ns_reserve=0,
                 device_resident=device_resident, kernel=PeriodicKernel, **OPT_PERIODIC)

    def bq_objects():
        bqs, states = [], []
        for p in range(P):
            np.random.seed(SEED + p)
            bq = BQ(x0, fl[p](x0), kernel=PeriodicKernel, optim_method="L-BFGS-B", **OPT_PERIODIC)
            bq.init(params_tl=PARAMS_TL, params_l=PARAMS_L)
            bqs.append(bq)
            states.append(np.random.get_state())
        return bqs, states
    return bb, fl, bq_objects, np.linspace(-np.pi, np.pi, 301)[:-1]


def readout(obj, name, x, **kw):
    return getattr(obj, name)(x, **kw)


def models(bb):
    return [bb.batch.read_model(p) for p in range(bb.P)]


def on_host_route(bb, p):
    """True where BQ._predict leaves problem p to the host GPs (noisy gp_l, periodic kernel, more than 256 observations)."""
    return bb.periodic or bb.hyp[p, 5] != 0 or bb._cap_class > 256


CASES = [("gauss", 10), ("gauss", 40), ("gauss", 100), ("gauss", 200), ("gauss", 300), ("periodic", 5)]


@pytest.mark.parametrize("kind,ns0", CASES)
def test_readouts_equal_a_loop_of_bq_objects(kind, ns0):
    import torch
    bb, fl, bq_objects, grid = gaussian_case(ns0) if kind == "gauss" else periodic_case()
    bqs, states = bq_objects()
    want_class = {10: 16, 40: 64, 100: 128, 200: 256, 300: 512, 5: 16}[ns0]
    assert bb._cap_class == want_class
    per_problem = np.stack([grid + 0.01 * (p + 1) for p in range(bb.P)])
    grids = [("shared numpy", grid, grid), ("per-problem tensor", torch.from_numpy(per_problem).cuda(), per_problem)]
    if want_class == 128:                               # an unsorted shared grid that BQ's host entry points pre-sort
        big = np.random.RandomState(3).permutation(np.linspace(grid[0], grid[-1], 8192))
        grids.append(("unsorted 8192", big, big))
    for rnd in range(3):
        for p, bq in enumerate(bqs):
            n, c = int(bb.ns[p]), int(bb.nc[p])
            assert n == bq.ns and np.array_equal(bb.x_s[p, :n], bq.x_s) and np.array_equal(bb.x_c[p, :c], bq.x_c), (rnd, p)
            assert _lib_class(n) == want_class               # BQ runs the batch's kernels
        before = models(bb)
        for label, x, x_rows in grids:
            for name in METHODS:
                if label == "unsorted 8192" and name in ("l_mean", "l_var", "expected_mean"):
                    continue
                got = readout(bb, name, x)
                dev = readout(bb, name, x, on_device=True)
                assert isinstance(dev, torch.Tensor) and dev.is_cuda
                assert np.array_equal(dev.cpu().numpy(), got, equal_nan=True), (label, name, rnd)
                shape = (bb.P, x_rows.shape[-1]) + ((2,) if name == "expected_squared_mean_and_mean" else ())
                assert got.shape == shape, (label, name, got.shape)
                for p, bq in enumerate(bqs):
                    want = readout(bq, name, x_rows if x_rows.ndim == 1 else x_rows[p])
                    what = "%s %s round %d problem %d" % (label, name, rnd, p)
                    if name in ("l_mean", "l_var") and on_host_route(bb, p) and rnd > 0:
                        # host GPs over log l_s: BQ takes the log of appended values one scalar at a time, the batch of
                        # the whole vector (numpy's vector and scalar log may differ in the last bit)
                        assert_close(got[p], want, what)
                    else:
                        assert np.array_equal(got[p], want, equal_nan=True), what
        after = models(bb)
        for p in range(bb.P):
            assert np.array_equal(before[p], after[p]), (rnd, p)
        if rnd == 2:
            break
        idx, x_next = bb.choose_next(grid)
        l_new = np.array([fl[p](x_next[p]) for p in range(bb.P)])
        bb.add_observations(x_next, l_new)
        for p, bq in enumerate(bqs):
            np.random.set_state(states[p])
            bq.add_observation(float(x_next[p]), float(l_new[p]))
            states[p] = np.random.get_state()
    bb.close()


def _lib_class(n):
    from bayesian_quadrature_b200 import _lib
    return _lib.ns_capacity(n)


@pytest.mark.parametrize("kind", ["gauss", "periodic"])
def test_host_and_device_resident_modes_agree(kind):
    import torch
    make = (lambda dr: gaussian_case(40, P=4, device_resident=dr)) if kind == "gauss" else \
        (lambda dr: periodic_case(P=4, device_resident=dr))
    host, fl, _, grid = make(False)
    dev, _, _, _ = make(True)
    g_d = torch.from_numpy(grid).cuda()
    for rnd in range(3):
        for name in METHODS:
            a = readout(host, name, grid)
            b = readout(dev, name, g_d, on_device=True).cpu().numpy()
            assert np.array_equal(a, b, equal_nan=True), (name, rnd)
        idx, x_h = host.choose_next(grid)
        idx_d, x_d = dev.choose_next(g_d, on_device=True)
        assert np.array_equal(idx_d.cpu().numpy(), idx)
        l_new = np.array([fl[p](x_h[p]) for p in range(host.P)])
        host.add_observations(x_h, l_new)
        dev.add_observations(x_d, torch.from_numpy(l_new).cuda())
    host.close()
    dev.close()


@pytest.mark.parametrize("kind", ["gauss", "periodic"])
def test_rows_kernel_equals_the_single_instance_path(kind):
    """bqb_expected_var_rows_device: every row has the bits of bqb_expected_var_host of its instance (staged, and with a
    page-locked output through the scoring kernel's fused epilogue) and of (Zm * Zm + Zv) - esm in numpy, for strided rows
    of esm and out, a first instance > 0 and na = 0, 1, 7, 257; esm and out may be one buffer."""
    import torch
    bb, _, _, grid = gaussian_case(40, P=5) if kind == "gauss" else periodic_case(P=5)
    P = bb.P
    zm, zv = bb.info["Z_mean"], bb.info["Z_var"]
    for na in (0, 1, 7, 257):
        x = np.linspace(grid[0], grid[-1], na)
        x_d = torch.from_numpy(x).cuda()
        esm_buf = torch.full((P, na + 3), np.nan, dtype=torch.float64, device="cuda")
        esm = esm_buf[:, 1:na + 1]                      # strided rows
        if na:
            bb.batch.score_device(x_d, esm)
        out_buf = torch.full((P, na + 5), -1.0, dtype=torch.float64, device="cuda")
        inst0 = 2
        bb.batch.expected_var_rows_device(inst0, P - inst0, esm[inst0:], out_buf[inst0:, 2:na + 2])
        bb.batch.expected_var_rows_device(0, inst0, esm, out_buf[:, 2:na + 2])
        got = out_buf.cpu().numpy()
        assert (got[:, :2] == -1).all() and (got[:, na + 2:] == -1).all()     # nothing written outside the rows
        inplace = esm.clone()
        bb.batch.expected_var_rows_device(0, P, inplace, inplace)
        esm_h = esm.cpu().numpy()
        for p in range(P):
            want, _ = bb.batch.expected_var_host(x, inst=p)
            assert np.array_equal(got[p, 2:na + 2], want), (na, p)
            assert np.array_equal(inplace[p].cpu().numpy(), want), (na, p)
            assert np.array_equal(want, (zm[p] * zm[p] + zv[p]) - esm_h[p]), (na, p)
            if na:
                fused, _ = bb.batch.expected_var_host(x, inst=p, out=torch.empty(na, dtype=torch.float64).pin_memory().numpy())
                assert np.array_equal(fused, want), (na, p)
        assert np.array_equal(bb.expected_Z_var(x), got[:, 2:na + 2])
        assert np.array_equal(bb.expected_Z_var(x_d, on_device=True).cpu().numpy(), got[:, 2:na + 2])
        for name in METHODS[1:]:
            assert readout(bb, name, x).shape[:2] == (P, na), (name, na)
    bb.close()


def test_rows_kernel_argument_checks():
    import ctypes
    import torch
    from bayesian_quadrature_b200 import _lib
    L = _lib.load()
    bb, _, _, grid = gaussian_case(10, P=3)
    b = bb.batch
    esm = torch.zeros(3, 8, dtype=torch.float64, device="cuda")
    e, o = ctypes.c_void_p(esm.data_ptr()), ctypes.c_void_p(esm.data_ptr())
    f = L.bqb_expected_var_rows_device
    assert f(b._h, -1, 1, e, 8, 8, o, 8, None) == _lib.EINVAL
    assert f(b._h, 2, 2, e, 8, 8, o, 8, None) == _lib.EINVAL           # past the last instance
    assert f(b._h, 0, -1, e, 8, 8, o, 8, None) == _lib.EINVAL
    assert f(b._h, 0, 3, e, 7, 8, o, 8, None) == _lib.EINVAL           # esm stride < na
    assert f(b._h, 0, 3, e, 8, 8, o, 7, None) == _lib.EINVAL           # out stride < na
    assert f(b._h, 0, 3, e, 8, -1, o, 8, None) == _lib.EINVAL
    assert f(b._h, 0, 3, None, 8, 8, o, 8, None) == _lib.EINVAL
    assert f(None, 0, 1, e, 8, 8, o, 8, None) == _lib.EINVAL
    assert f(b._h, 1, 0, None, 8, 8, None, 8, None) == 0                # nothing to do
    assert f(b._h, 0, 3, None, 0, 0, None, 0, None) == 0
    with pytest.raises(ValueError):
        b.expected_var_rows_device(2, 2, esm, esm)
    fresh = _lib.Batch(3, 16)
    with pytest.raises(_lib.BQB200Error):                               # nothing set up
        fresh.expected_var_rows_device(0, 3, esm, esm)
    fresh.close()
    bb.close()


def test_invalid_point_raises_naming_the_problem():
    import torch
    bb, _, _, grid = gaussian_case(10, P=4)
    rows = np.tile(grid, (bb.P, 1))
    rows[2, 17] = np.nan
    for x in (rows, torch.from_numpy(rows).cuda()):
        for name in ("expected_Z_var", "expected_squared_mean", "expected_squared_mean_and_mean"):
            with pytest.raises(ValueError, match="problem 2"):
                readout(bb, name, x)
    bb.close()


def test_overflow_guards_warn_and_score_like_bq(caplog):
    """The edge_inf90 fixture (tests/test_gpu_bq_api.py::test_infinite_scores_warn_like_the_reference): infinite expected
    squared means are logged per problem, expected_Z_var is -inf there, and every value is BQ's."""
    from bayesian_quadrature_b200 import BQ, BatchBQ, GaussianKernel
    from conftest import load_golden
    g = load_golden("edge_inf90")
    P = 2
    opt = dict(n_candidate=10, x_mean=0.0, x_var=10.0, candidate_thresh=0.5)
    bb = BatchBQ(np.tile(g["x_s"], (P, 1)), np.tile(g["l_s"], (P, 1)), tuple(g["params_tl"]), tuple(g["params_l"]),
                 seed=SEED, **opt)
    with caplog.at_level(logging.WARNING, logger="bayesian_quadrature"):
        r = bb.expected_squared_mean_and_mean(g["x_a"])
        ev = bb.expected_Z_var(g["x_a"])
    for p in range(P):
        assert any("infinity" in rec.getMessage() and "(problem %d)" % p in rec.getMessage() for rec in caplog.records), p
        np.random.seed(SEED + p)
        bq = BQ(g["x_s"], g["l_s"], kernel=GaussianKernel, optim_method="L-BFGS-B", **opt)
        bq.init(params_tl=tuple(g["params_tl"]), params_l=tuple(g["params_l"]))
        assert np.array_equal(bb.x_c[p, :bb.nc[p]], bq.x_c)
        assert np.array_equal(r[p], bq.expected_squared_mean_and_mean(g["x_a"]), equal_nan=True), p
        assert np.array_equal(ev[p], bq.expected_Z_var(g["x_a"]), equal_nan=True), p
    assert np.isneginf(ev).any()
    bb.close()


def test_non_positive_Z_mean_warns_once_naming_the_problems():
    bb, _, _, grid = gaussian_case(10, P=4)
    want = bb.expected_Z_var(grid)
    bb.info["Z_mean"][[1, 3]] = -1.0                    # what the setup reports for a problem whose Z_mean is not positive
    with pytest.warns(UserWarning, match=r"m_Z .* in problems \[1, 3\]") as rec:
        ev = bb.expected_Z_var(grid)
    assert sum("m_Z" in str(w.message) for w in rec) == 1
    assert np.array_equal(ev, want)                     # the values come from the device headers, which are untouched
    bb.close()
