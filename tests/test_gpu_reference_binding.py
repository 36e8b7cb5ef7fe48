"""The drop-in boundary of INTEGRATION.md section 3: the ctypes stub a maintainer of the reference would add
(tests/ref_binding.py), which replaces the three scoring loops of the reference's ``BQ`` class (bq.py:399-402, :420-422,
:442-444) by one libbq_b200.so call each.  The stub reads nothing but the state of a reference ``BQ`` object (x_s, l_s, x_c,
the two GPs' kernels and parameters, the options, the approximation grid); here it is given the states of the reference's
own test problems as the unmodified reference held them, and what it returns is held to what the reference computed for them
(tests/golden/*.npz, written by tests/golden/make_golden.py): the reference's scoring tests
(bayesian_quadrature/tests/test_bq_object.py:145-170, :286-300) restated, the marginalisation of its ``choose_next`` loop
(bq.py:604-681) over the hyper-parameter sets its sampler drew, and its periodic problems, on B200."""
import numpy as np
import pytest
import scipy.stats

from conftest import assert_close, load_golden

pytestmark = pytest.mark.gpu


class _GP(object):
    """The two attributes of a reference ``gp.GP`` the stub reads: the kernel object (by class name) and ``params``."""

    def __init__(self, kernel, params):
        self.K = type(kernel, (object,), {})()
        self.params = np.array(params, dtype=np.float64)


class RefState(object):
    """A reference ``BQ`` object's state after ``BQ(x, l, **options).init(params_tl, params_l)`` (bq.py:132-171, :967-991),
    with the candidates that init drew."""

    def __init__(self, x_s, l_s, x_c, params_tl, params_l, x_mean=0.0, x_var=10.0, candidate_thresh=0.5,
                 kernel="GaussianKernel", xo=None, p_xo=None):
        self.x_s, self.l_s = np.array(x_s, dtype=np.float64), np.array(l_s, dtype=np.float64)
        self.x_c = np.array(x_c, dtype=np.float64)
        self.ns, self.nc = self.x_s.size, self.x_c.size
        self.gp_log_l, self.gp_l = _GP(kernel, params_tl), _GP(kernel, params_l)
        self.options = {"x_mean": np.array([float(x_mean)]), "x_cov": np.array([[float(x_var)]]),
                        "candidate_thresh": float(candidate_thresh), "use_approx": xo is not None}
        self._approx_x, self._approx_px = xo, p_xo

    @classmethod
    def from_golden(cls, g, kernel="GaussianKernel"):
        approx = int(g["use_approx"]) if "use_approx" in g else 0
        return cls(g["x_s"], g["l_s"], g["x_c"], g["params_tl"], g["params_l"], float(g["x_mean"]), float(g["x_var"]),
                   float(g["candidate_thresh"]), kernel, g["xo"] if approx else None, g["p_xo"] if approx else None)


@pytest.fixture(scope="module")
def BQ_b200():
    import ref_binding
    return ref_binding.patch_reference(RefState)


def test_reference_scoring_tests_through_the_library(BQ_b200, oracle):
    g = load_golden("fixture")
    bq = BQ_b200.from_golden(g)
    # expected_Z_var of the reference (bq.py:374-377) with its own Z_mean / Z_var
    ev = g["Z_mean"] ** 2 + g["Z_var"] - bq.expected_squared_mean(bq.x_s)
    assert np.allclose(ev, g["Z_var"], atol=1e-4)                                     # test_expected_Z_var_close (:145)
    x_a = np.random.RandomState(8728).uniform(-10, 10, 10)
    assert (bq.expected_squared_mean(x_a) >= 0).all()                                  # test_expected_squared_mean_valid (:153)
    for bad in (np.nan, np.inf, -np.inf):                                              # test_expected_squared_mean_params (:161)
        with pytest.raises(ValueError):
            bq.expected_squared_mean(np.array([bad]))
    for x in np.linspace(-5, 5, 20)[:, None]:                                          # test_expected_squared_mean_1 (:286)
        y = scipy.stats.norm.pdf(x, 0, 1)
        b1 = BQ_b200(x, y, [], (15, 2, 0), (0.2, 1.3, 0))                              # one observation, n_candidate=0
        m2 = oracle.OracleModel(x, y, [], (15, 2, 0), (0.2, 1.3, 0), 0.0, 10.0, 0.5).Z_mean() ** 2
        for dx in (0.0, 1e-10, 1e-8):
            assert np.allclose(m2, b1.expected_squared_mean(x - dx), atol=1e-4)


def test_patched_reference_equals_unpatched_reference(BQ_b200, oracle):
    """Same object state, scored by the reference's Cython loop (the fixture) and through the library: north-star
    tolerance."""
    g = load_golden("fixture")
    b = BQ_b200.from_golden(g)
    x_a = g["x_a"][:120]
    rb = b.expected_squared_mean_and_mean(x_a)
    assert_close(rb[:, 0], g["esm"][:120], "esm")
    assert_close(rb[:, 1], g["em"][:120], "em")
    assert_close(g["Z_mean"] ** 2 + g["Z_var"] - rb[:, 0], g["expected_Z_var"][:120], "expected_Z_var", atol=1e-12)
    assert_close(b.expected_mean(x_a), g["em"][:120], "em vs fixture")
    # parameters changed on the object (the reference's _set_gp_log_l_params / _set_gp_l_params): the device factors follow;
    # the same state in the C restatement of the reference
    b.gp_log_l.params = np.array([14.0, 1.9, 0.0])
    b.gp_l.params = np.array([0.25, 1.2, 0.0])
    m = oracle.OracleModel(g["x_s"], g["l_s"], g["x_c"], (14.0, 1.9, 0.0), (0.25, 1.2, 0.0), float(g["x_mean"]),
                           float(g["x_var"]), float(g["candidate_thresh"]), check_max=True)
    assert_close(b.expected_squared_mean(x_a), m.esm_and_em(x_a)[0], "esm after set_params")


def test_reference_choose_next_loop_runs_on_the_library(BQ_b200):
    """The marginalisation of the reference's own choose_next (bq.py:659-681: -esm averaged over the sampled
    hyper-parameter sets, the tie set of np.isclose to its minimum, np.random.choice in it) with every scoring call going
    through libbq_b200.so, over the sets the reference's sampler drew under the fixture's seed: the same loss, the same tie
    set and the point the unpatched reference chose (tests/golden/choose_fixture.npz)."""
    g = load_golden("choose_fixture")
    bq = BQ_b200(g["x_s"], g["l_s"], g["x_c"], (15, 2, 0), (0.2, 1.3, 0))
    x_a, n = g["x_a"], int(g["n"])
    esm = np.empty((n, x_a.size))
    for i in range(n):
        bq.gp_log_l.params = np.array([g["hypers_tl"][i, 0], g["hypers_tl"][i, 1], 0.0])
        bq.gp_l.params = np.array([g["hypers_l"][i, 0], g["hypers_l"][i, 1], 0.0])
        esm[i] = bq.expected_squared_mean(x_a)
    loss = (-esm).mean(axis=0)
    assert_close(loss, g["loss"], "marginal loss")
    close = np.nonzero(np.isclose(loss, loss.min()))[0]
    assert np.array_equal(close, g["tie_set"])
    assert close.size == 1 and x_a[close[0]] == float(g["chosen"])         # a tie set of one: np.random.choice has no choice


def test_patched_reference_with_the_periodic_kernel(BQ_b200):
    """The reference's own periodic problem (tests/util.py:76-91: PeriodicKernel, wrapped domain, `use_approx`) and a
    better-conditioned one, scored by the reference's Cython loop (the fixture) and, from the same object state, through
    the library (bqb_batch_set_approx: kernel kind, periods, the object's own approximation grid)."""
    for name in ("periodic_a", "periodic_b"):
        g = load_golden(name)
        b = BQ_b200.from_golden(g, kernel="PeriodicKernel")
        rb = b.expected_squared_mean_and_mean(g["x_a"])
        assert_close(rb[:, 0], g["esm"], "periodic esm, %d observations" % b.ns)
        assert_close(rb[:, 1], g["em"], "periodic em, %d observations" % b.ns)
