"""util.lbfgs_batch, the lock-step L-BFGS behind BatchBQ.fit_hypers: per-row optima against scipy's L-BFGS-B, rows that
stop at different iterations, -inf regions handled by backtracking, and rows independent of the batch they run in."""
import numpy as np
import pytest
import scipy.optimize as optim

from bayesian_quadrature_b200 import util


def quadratic(C, A):
    """Rows p: f(x) = -1/2 (x - C[p])' A[p] (x - C[p])."""
    def fg(X, rows):
        r = X - C[rows]
        Ar = np.einsum("pij,pj->pi", A[rows], r)
        return -0.5 * (r * Ar).sum(axis=1), -Ar
    return fg


def rosenbrock(a, b):
    """Rows p: f(x) = -((a_p - x0)^2 + b_p (x1 - x0^2)^2), maximum 0 at (a_p, a_p^2)."""
    def fg(X, rows):
        x0, x1 = X[:, 0], X[:, 1]
        ap, bp = a[rows], b[rows]
        f = (ap - x0) ** 2 + bp * (x1 - x0 ** 2) ** 2
        g0 = -2 * (ap - x0) - 4 * bp * x0 * (x1 - x0 ** 2)
        g1 = 2 * bp * (x1 - x0 ** 2)
        return -f, -np.stack([g0, g1], axis=1)
    return fg


def scipy_max(fg, x0, p):
    fun = lambda x: -fg(x[None], np.array([p]))[0][0]
    jac = lambda x: -fg(x[None], np.array([p]))[1][0]
    return optim.minimize(fun, x0, jac=jac, method="L-BFGS-B")


def test_quadratics_match_scipy_and_stop_at_different_iterations():
    rng = np.random.RandomState(3)
    P, d = 12, 4
    C = rng.uniform(-3, 3, (P, d))
    A = np.empty((P, d, d))
    for p in range(P):
        Q, _ = np.linalg.qr(rng.randn(d, d))
        A[p] = Q @ np.diag(np.logspace(0, p % 4, d)) @ Q.T          # condition 1 .. 1000
    x0 = rng.uniform(-1, 1, (P, d))
    fg = quadratic(C, A)
    res = util.lbfgs_batch(fg, x0)
    assert res["converged"].all()
    assert len(set(res["iterations"].tolist())) > 1                    # rows stop at different iterations
    for p in range(P):
        ref = scipy_max(fg, x0[p], p)
        assert res["f"][p] >= -ref.fun - 1e-9
        assert np.allclose(res["x"][p], C[p], atol=1e-4), (p, res["x"][p], C[p])
    assert res["evaluations"] < res["calls"] * P                       # finished rows are not evaluated again


def test_rosenbrock_rows_match_scipy():
    a = np.array([1.0, 0.5, -1.0, 2.0, 1.5])
    b = np.array([100.0, 10.0, 50.0, 5.0, 1.0])
    x0 = np.array([[-1.2, 1.0], [0.0, 0.0], [1.0, 1.0], [-0.5, 2.0], [3.0, -1.0]])
    fg = rosenbrock(a, b)
    res = util.lbfgs_batch(fg, x0)
    assert res["converged"].all()
    assert len(set(res["iterations"].tolist())) > 1
    for p in range(a.size):
        ref = scipy_max(fg, x0[p], p)
        assert res["f"][p] >= -ref.fun - 1e-9, (p, res["f"][p], -ref.fun)
        assert np.allclose(res["x"][p], [a[p], a[p] ** 2], atol=2e-3), (p, res["x"][p])


def test_minus_inf_region_is_backtracked():
    """f = -(x - 2)^2 left of a wall at 2.5 and -inf (or NaN) right of it: full steps that land behind the wall fail and
    are halved."""
    def fg(X, rows):
        x = X[:, 0]
        wall = np.where(rows % 2 == 0, -np.inf, np.nan)
        f = np.where(x < 2.5, -(x - 2.0) ** 2, wall)
        return f, (-2 * (x - 2.0))[:, None]
    x0 = np.array([[-40.0], [-40.0], [2.4], [1.0]])
    res = util.lbfgs_batch(fg, x0)
    assert res["converged"].all()
    assert np.allclose(res["x"][:, 0], 2.0, atol=1e-5)
    assert np.isfinite(res["f"]).all()


def test_rows_do_not_depend_on_the_batch():
    rng = np.random.RandomState(11)
    P = 7
    a, b = rng.uniform(-2, 2, P), rng.uniform(1, 100, P)
    x0 = rng.uniform(-2, 2, (P, 2))
    fg = rosenbrock(a, b)
    full = util.lbfgs_batch(fg, x0, maxiter=60)
    for p in range(P):
        one = util.lbfgs_batch(lambda X, rows: fg(X, np.full(rows.size, p)), x0[p:p + 1], maxiter=60)
        assert np.array_equal(one["x"][0], full["x"][p]) and one["f"][0] == full["f"][p]
        assert one["iterations"][0] == full["iterations"][p] and one["converged"][0] == full["converged"][p]
    assert (full["iterations"] <= 60).all()


def test_start_with_zero_probability_raises_naming_the_row():
    def fg(X, rows):
        f = np.where(X[:, 0] > 0, -X[:, 0] ** 2, -np.inf)
        return f, -2 * X
    with pytest.raises(RuntimeError) as ei:
        util.lbfgs_batch(fg, np.array([[1.0], [2.0], [-1.0]]))
    assert ei.value.row == 2
