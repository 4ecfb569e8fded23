"""Constant uncertainties on the CPU: the CPU reference of the Gram sweep against the exact
Jacobian, the covariance math against scipy.optimize.curve_fit, and the conventions of
``uncertainty.covariance_from_gram`` / ``covariances``."""
import numpy as np
import pytest
import scipy.optimize
import sympy as sp

from _gram_ref import VARS, curve_fit_pcov, exact, frob_rel, load_twin, twin_gram, winners
from src.visymre import uncertainty
from src.visymre.engine.compiler import compile_skeleton


@pytest.fixture(scope="module")
def twin():
    """The CPU reference of vsr_gram (tests/native/gram_twin.cpp)."""
    return load_twin()


@pytest.fixture(scope="module")
def cases():
    return winners()


def _finite(*arrays):
    return all(np.isfinite(np.asarray(a)).all() for a in arrays)


def _rss_bound(rss, y, n):
    # the residuals of a near-perfect fit cancel to the last digits of f, and the reference and numpy
    # round f differently: allow a few ulps of |y| per residual on top of the relative bound
    scale = 1e-15 * np.linalg.norm(y) + 1e-15 * n
    return 1e-10 * rss + 4 * np.sqrt(rss) * scale + scale ** 2


def test_twin_gram_matches_the_exact_jacobian(twin, cases):
    checked = 0
    for name, skel, c, X, y in cases:
        k = c.shape[0]
        prog = compile_skeleton(skel, k, VARS)
        rss, jtj = twin_gram(twin, prog, X, y, c)
        r, J = exact(skel, k, X, y, c)
        if not _finite(r, J):
            assert not (np.isfinite(rss) and np.isfinite(jtj).all()), name
            continue
        want = J.T @ J
        assert frob_rel(jtj, want) <= 1e-10, (name, jtj, want)
        assert np.array_equal(jtj, jtj.T), name
        assert abs(rss - r @ r) <= _rss_bound(r @ r, y, len(y)), (name, rss, r @ r)
        checked += 1
    assert checked >= 40, checked


def test_covariance_matches_curve_fit_formula(twin, cases):
    checked = 0
    for name, skel, c, X, y in cases:
        k = c.shape[0]
        free = c != 0.0
        if k == 0 or not free.any():
            continue
        r, J = exact(skel, k, X, y, c)
        if not _finite(r, J) or np.linalg.cond(J[:, free]) > 1e5:
            continue
        prog = compile_skeleton(skel, k, VARS)
        _, jtj = twin_gram(twin, prog, X, y, c)
        # the same rss on both sides: at an exact fit it is rounding, which the test above bounds
        cov, stderr, dof, rank = uncertainty.covariance_from_gram(r @ r, jtj, len(y), free)
        want = curve_fit_pcov(J[:, free], r @ r)
        assert rank == free.sum() and dof == len(y) - free.sum(), name
        assert frob_rel(cov[np.ix_(free, free)], want) <= 1e-8, (name, cov, want)
        assert np.isnan(stderr[~free]).all() and np.isnan(cov[~free]).all(), name
        np.testing.assert_allclose(stderr[free], np.sqrt(np.diag(want)), rtol=1e-8)
        checked += 1
    assert checked >= 25, checked


def test_pcov_of_scipy_curve_fit(twin, cases):
    """curve_fit itself, from the winning constants, on well-posed winners with noise in the data
    (at an exact fit rss is rounding and moves with any step curve_fit takes)."""
    done = []
    for name, skel, c, X, y in cases:
        k = c.shape[0]
        if k == 0 or (c == 0.0).any():
            continue
        r, J = exact(skel, k, X, y, c)
        if not _finite(r, J) or r @ r < 1e-6 * (y @ y) or np.linalg.cond(J) > 1e3:
            continue
        cs = [sp.Symbol(f"c{i}", real=True) for i in range(k)]
        xs = [sp.Symbol(v, real=True) for v in VARS]
        f = sp.lambdify(cs + xs, sp.sympify(skel, locals={str(s): s for s in cs + xs}), modules="numpy")

        def model(Xt, *p):
            return np.broadcast_to(f(*p, *Xt), (Xt.shape[1],))
        popt, pcov = scipy.optimize.curve_fit(model, X.T, y, p0=c)
        assert np.allclose(popt, c, rtol=1e-4, atol=1e-6), (name, popt, c)
        prog = compile_skeleton(skel, k, VARS)
        rss, jtj = twin_gram(twin, prog, X, y, c)
        cov, _, _, _ = uncertainty.covariance_from_gram(rss, jtj, len(y), np.ones(k, bool))
        assert frob_rel(cov, pcov) <= 1e-5, (name, cov, pcov)
        done.append(name)
        if len(done) == 3:
            break
    assert len(done) == 3, done


@pytest.mark.parametrize("skel", ["((c0)*((c1)*(x_1)))", "(((c0)*(x_1))+((c1)*(x_1)))", "(((c0)*(exp(c1)))*(x_1))"])
def test_degenerate_skeletons(twin, skel):
    rng = np.random.RandomState(3)
    X = np.zeros((200, 10))
    X[:, 0] = rng.uniform(-2, 2, 200)
    c = np.array([1.3, 0.7])
    y = 2.0 * X[:, 0] + rng.normal(0, 0.1, 200)
    prog = compile_skeleton(skel, 2, VARS)
    rss, jtj = twin_gram(twin, prog, X, y, c)
    cov, stderr, dof, rank = uncertainty.covariance_from_gram(rss, jtj, 200, np.ones(2, bool))
    assert rank == 1 and dof == 198
    assert np.isposinf(cov).all() and np.isposinf(stderr).all()


def test_conventions():
    jtj = np.array([[4.0, 1.0], [1.0, 3.0]])
    # full rank: s^2 (J^T J)^-1
    cov, stderr, dof, rank = uncertainty.covariance_from_gram(2.0, jtj, 10, np.ones(2, bool))
    np.testing.assert_allclose(cov, np.linalg.inv(jtj) * 2.0 / 8, rtol=1e-14)
    assert dof == 8 and rank == 2
    np.testing.assert_allclose(stderr, np.sqrt(np.diag(cov)))
    # dof <= 0
    cov, stderr, dof, rank = uncertainty.covariance_from_gram(2.0, jtj, 2, np.ones(2, bool))
    assert dof == 0 and rank == 2 and np.isposinf(cov).all() and np.isposinf(stderr).all()
    # nan in the Gram or the rss
    for r, g in ((2.0, np.array([[4.0, np.nan], [np.nan, 3.0]])), (np.nan, jtj), (np.inf, jtj)):
        cov, stderr, dof, rank = uncertainty.covariance_from_gram(r, g, 10, np.ones(2, bool))
        assert np.isposinf(cov).all() and rank == 0
    # k = 0
    cov, stderr, dof, rank = uncertainty.covariance_from_gram(2.0, np.zeros((0, 0)), 10, np.zeros(0, bool))
    assert cov.shape == (0, 0) and stderr.shape == (0,) and dof == 10 and rank == 0
    # a pruned constant: out of the matrix, nan rows / columns and stderr
    cov, stderr, dof, rank = uncertainty.covariance_from_gram(2.0, jtj, 10, np.array([True, False]))
    assert dof == 9 and rank == 1
    assert cov[0, 0] == pytest.approx(2.0 / 9 / 4.0, rel=1e-14)
    assert np.isnan(cov[1]).all() and np.isnan(cov[:, 1]).all() and np.isnan(stderr[1])
    # rank-deficient: the eigenvalue bound max(N, k) eps lambda_max
    eps = np.finfo(float).eps
    near = np.array([[1.0, 0.0], [0.0, 50 * eps]])
    assert uncertainty.covariance_from_gram(1.0, near, 100, np.ones(2, bool))[3] == 1
    assert uncertainty.covariance_from_gram(1.0, near, 10, np.ones(2, bool))[3] == 2


def test_failed_fits_give_none():
    """Exceptions and None in the list give None; a list with no fit touches no device."""
    assert uncertainty.covariances([None, ValueError("x")], np.zeros((5, 1)), np.zeros(5)) == [None, None]
