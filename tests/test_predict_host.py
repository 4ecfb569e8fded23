"""Prediction bands on the CPU: the host band assembly ``uncertainty.bands`` against the closed-form OLS
intervals of a linear skeleton, its conventions, and the delta-method variance built from sympy's exact
Jacobian against the OLS formula."""
import numpy as np
import pytest
import scipy.stats
import torch

from _gram_ref import exact
from src.visymre import uncertainty

LINEAR = "((c0)+((c1)*(x_1)))"


def _ols(seed=4, n=40):
    """A noisy straight line, its OLS fit and the covariance ``covariances`` would give for it."""
    rng = np.random.RandomState(seed)
    x = rng.uniform(-2, 3, n)
    y = 0.7 + 1.9 * x + rng.normal(0, 0.3, n)
    A = np.stack([np.ones(n), x], axis=1)
    beta = np.linalg.lstsq(A, y, rcond=None)[0]
    rss = float(np.sum((A @ beta - y) ** 2))
    cov, _, dof, _ = uncertainty.covariance_from_gram(rss, A.T @ A, n, np.ones(2, bool))
    return A, beta, rss, dof, cov


def _closed_form(A, beta, rss, dof, x0, level):
    """yhat -+ t s sqrt(x0^T (A^T A)^-1 x0) and yhat -+ t s sqrt(1 + x0^T (A^T A)^-1 x0)."""
    D = np.stack([np.ones_like(x0), x0], axis=1)
    h = np.einsum("ia,ab,ib->i", D, np.linalg.inv(A.T @ A), D)
    s = np.sqrt(rss / dof)
    t = scipy.stats.t.ppf((1 + level) / 2, dof)
    yhat = D @ beta
    return yhat, t * s * np.sqrt(h), t * s * np.sqrt(1 + h)


@pytest.mark.parametrize("level", [0.5, 0.9, 0.95, 0.99])
def test_bands_match_the_ols_intervals(level):
    A, beta, rss, dof, cov = _ols()
    x0 = np.linspace(-4, 5, 37)
    g = np.stack([np.ones_like(x0), x0], axis=1)    # d f / d c of c0 + c1 x_1
    value = g @ beta
    var = np.einsum("ia,ab,ib->i", g, cov, g)
    p = uncertainty.bands(torch.from_numpy(value), torch.from_numpy(var), cov, rss, dof, level)
    yhat, hw_ci, hw_pi = _closed_form(A, beta, rss, dof, x0, level)
    for got, want in ((p.value, yhat), (p.ci_low, yhat - hw_ci), (p.ci_high, yhat + hw_ci),
                      (p.pi_low, yhat - hw_pi), (p.pi_high, yhat + hw_pi)):
        np.testing.assert_allclose(got.numpy(), want, rtol=1e-12, atol=1e-12)
    assert p.dof == dof == 38 and p.level == level
    assert p.t == scipy.stats.t.ppf((1 + level) / 2, dof)
    assert p.se_fit.dtype == torch.float64


def test_delta_method_from_the_exact_jacobian_is_the_ols_formula():
    A, beta, rss, dof, cov = _ols(seed=5)
    Xn = np.zeros((25, 10))
    Xn[:, 0] = np.linspace(-3, 4, 25)
    value, J = exact(LINEAR, 2, Xn, np.zeros(25), beta)
    var = np.einsum("ia,ab,ib->i", J, cov, J)
    yhat, hw_ci, _ = _closed_form(A, beta, rss, dof, Xn[:, 0], 0.95)
    t = scipy.stats.t.ppf(0.975, dof)
    np.testing.assert_allclose(value, yhat, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(t * np.sqrt(var), hw_ci, rtol=1e-12)


def test_fixed_constants_carry_no_variance():
    # a pruned constant: nan row and column in cov, zeroed for the device
    cov, _, dof, _ = uncertainty.covariance_from_gram(2.0, np.array([[4.0, 1.0], [1.0, 3.0]]), 10,
                                                      np.array([True, False]))
    dc = uncertainty.device_cov(cov)
    assert np.isnan(cov[1]).all() and np.isfinite(dc).all()
    assert dc[0, 0] == cov[0, 0] and (dc[1] == 0).all() and (dc[:, 1] == 0).all()
    # the variance of a point is then that of the free constant alone, and the bands are finite
    g = np.array([[2.0, 5.0]])
    var = np.einsum("ia,ab,ib->i", g, dc, g)
    assert var[0] == 4.0 * cov[0, 0]
    p = uncertainty.bands(torch.tensor([1.0]), torch.from_numpy(var), cov, 2.0, dof)
    assert p.se_fit.item() == 2.0 * np.sqrt(cov[0, 0]) and torch.isfinite(p.pi_high).all()


def test_undeterminable_covariance_gives_infinite_bands():
    cov, _, dof, _ = uncertainty.covariance_from_gram(1.0, np.array([[1.0, 1.0], [1.0, 1.0]]), 50,
                                                      np.ones(2, bool))
    assert np.isposinf(cov).all()
    assert (uncertainty.device_cov(cov) == 0).all()
    value = torch.tensor([1.0, -2.0, float("nan")], dtype=torch.float64)
    p = uncertainty.bands(value, torch.zeros(3, dtype=torch.float64), cov, 1.0, dof)
    assert torch.isposinf(p.se_fit).all()
    assert torch.equal(p.value[:2], value[:2])
    assert torch.isneginf(p.ci_low[:2]).all() and torch.isposinf(p.ci_high[:2]).all()
    assert torch.isneginf(p.pi_low[:2]).all() and torch.isposinf(p.pi_high[:2]).all()
    for b in (p.ci_low, p.ci_high, p.pi_low, p.pi_high):
        assert torch.isnan(b[2])


def test_dof_at_most_zero_gives_infinite_bands():
    for dof in (0, -3):
        p = uncertainty.bands(torch.tensor([1.5]), torch.tensor([0.25]), np.eye(2), 1.0, dof)
        assert torch.isposinf(p.se_fit).all() and torch.isneginf(p.ci_low).all() and torch.isposinf(p.pi_high).all()
        assert p.value.item() == 1.5 and p.dof == dof and np.isnan(p.t)


def test_no_constants():
    # k == 0: cov is 0 x 0, the variance 0, the confidence band collapses onto the value and the
    # prediction band is value -+ t s
    value = torch.tensor([0.5, 2.0], dtype=torch.float64)
    p = uncertainty.bands(value, torch.zeros(2, dtype=torch.float64), np.zeros((0, 0)), 8.0, 20)
    t = scipy.stats.t.ppf(0.975, 20)
    assert torch.equal(p.se_fit, torch.zeros(2, dtype=torch.float64))
    assert torch.equal(p.ci_low, value) and torch.equal(p.ci_high, value)
    np.testing.assert_allclose(p.pi_high.numpy(), value.numpy() + t * np.sqrt(8.0 / 20), rtol=1e-15)
    assert uncertainty.device_cov(np.zeros((0, 0))).shape == (0, 0)


def test_negative_variance_is_clamped():
    value = torch.tensor([1.0, 1.0, 1.0], dtype=torch.float64)
    var = torch.tensor([-1e-18, 0.0, 4.0], dtype=torch.float64)
    p = uncertainty.bands(value, var, np.eye(1), 3.0, 3)
    assert p.se_fit.tolist() == [0.0, 0.0, 2.0]
    assert p.ci_low[0].item() == 1.0 and p.pi_high[0].item() == pytest.approx(1.0 + p.t, rel=1e-15)


def test_a_value_that_is_not_real_gives_nan_bands():
    value = torch.tensor([float("nan"), 3.0], dtype=torch.float64)
    var = torch.tensor([float("nan"), 1.0], dtype=torch.float64)
    p = uncertainty.bands(value, var, np.eye(1), 3.0, 3)
    for b in (p.ci_low, p.ci_high, p.pi_low, p.pi_high):
        assert torch.isnan(b[0]) and torch.isfinite(b[1])


def test_level_out_of_range():
    for level in (0.0, 1.0, 1.5, -0.1):
        with pytest.raises(ValueError):
            uncertainty.bands(torch.zeros(1), torch.zeros(1), np.eye(1), 1.0, 5, level)


def test_failed_fits_give_none_and_covs_must_match():
    """Exceptions and None in the list give None; a list with no fit touches no device."""
    assert uncertainty.predict([None, ValueError("x")], np.zeros((5, 1))) == [None, None]
    with pytest.raises(ValueError):
        uncertainty.predict([None, None], np.zeros((5, 1)), covs=[None])
    with pytest.raises(ValueError):
        uncertainty.predict([("", [1.0], 0.0, "((c0)*(x_1))")], np.zeros((5, 1)), covs=[None])
