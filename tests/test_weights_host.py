"""Weighted fits on the CPU: curve_fit's 1-D ``sigma`` conventions of ``covariance_from_gram`` and ``bands``
against scipy and the closed-form weighted OLS intervals, every ``ValueError`` of the ``sigma`` arguments,
and the weighted loss and gradient built from the host interpreter's per-point tangents against numpy and
sympy."""
import numpy as np
import pytest
import scipy.optimize
import scipy.stats
import sympy as sp
import torch

import _interp_ref as R
from conftest import make_cfg
from src.visymre import uncertainty
from src.visymre.architectures import bfgs as vbfgs
from src.visymre.architectures import refine
from src.visymre.engine import fitter
from src.visymre.engine.compiler import compile_skeleton

VARS = [f"x_{i}" for i in range(1, 11)]


def _wls(seed=3, n=50):
    """A straight line with heteroscedastic noise, its sigma and its weighted least-squares fit."""
    rng = np.random.RandomState(seed)
    x = rng.uniform(-2, 3, n)
    sigma = rng.uniform(0.1, 2.0, n)
    y = 0.7 + 1.9 * x + rng.normal(0, 1, n) * sigma
    A = np.stack([np.ones(n), x], axis=1)
    w = 1.0 / sigma ** 2
    G = A.T @ (w[:, None] * A)
    beta = np.linalg.solve(G, A.T @ (w * y))
    rss = float(np.sum(w * (A @ beta - y) ** 2))
    return x, y, sigma, A, w, G, beta, rss


@pytest.mark.parametrize("absolute", [False, True])
def test_weighted_covariance_matches_curve_fit(absolute):
    x, y, sigma, A, w, _, _, _ = _wls()
    # the analytic Jacobian: curve_fit's pcov is then exact up to rounding (MINPACK's own is a finite difference)
    popt, pcov = scipy.optimize.curve_fit(lambda x, a, b: a + b * x, x, y, p0=[0.0, 1.0], sigma=sigma,
                                          absolute_sigma=absolute,
                                          jac=lambda x, a, b: np.stack([np.ones_like(x), x], axis=1))
    rss = float(np.sum(w * (A @ popt - y) ** 2))
    cov, stderr, dof, rank = uncertainty.covariance_from_gram(rss, A.T @ (w[:, None] * A), len(x),
                                                              np.ones(2, bool), absolute_sigma=absolute)
    assert dof == len(x) - 2 and rank == 2
    np.testing.assert_allclose(cov, pcov, rtol=1e-10, atol=0)
    np.testing.assert_allclose(stderr, np.sqrt(np.diag(pcov)), rtol=1e-10)


def test_relative_covariance_does_not_depend_on_the_scale_of_sigma():
    _, _, _, A, w, G, _, rss = _wls()
    free = np.ones(2, bool)
    cov1, _, _, _ = uncertainty.covariance_from_gram(rss, G, A.shape[0], free)
    for f in (1e-3, 0.5, 7.0, 1e4):
        wf = w / f ** 2                      # sigma -> f sigma
        Gf = A.T @ (wf[:, None] * A)
        rf = rss / f ** 2                    # the same residuals, weighted by w / f^2
        cov_f, _, _, _ = uncertainty.covariance_from_gram(rf, Gf, A.shape[0], free)
        np.testing.assert_allclose(cov_f, cov1, rtol=1e-12)
        cov_abs, _, _, _ = uncertainty.covariance_from_gram(rf, Gf, A.shape[0], free, absolute_sigma=True)
        np.testing.assert_allclose(cov_abs, np.linalg.inv(G) * f ** 2, rtol=1e-12)


def test_absolute_covariance_keeps_the_inf_rules():
    G = np.array([[2.0, 1.0], [1.0, 3.0]])
    cov, _, dof, _ = uncertainty.covariance_from_gram(1.0, G, 2, np.ones(2, bool), absolute_sigma=True)
    assert dof == 0 and np.isinf(cov).all()
    sing = np.array([[1.0, 1.0], [1.0, 1.0]])
    cov, _, _, rank = uncertainty.covariance_from_gram(1.0, sing, 10, np.ones(2, bool), absolute_sigma=True)
    assert rank == 1 and np.isinf(cov).all()


@pytest.mark.parametrize("absolute", [False, True])
@pytest.mark.parametrize("level", [0.9, 0.95])
def test_bands_with_sigma_new_match_the_weighted_ols_intervals(absolute, level):
    _, _, _, A, w, G, beta, rss = _wls(seed=8)
    n = A.shape[0]
    cov, _, dof, _ = uncertainty.covariance_from_gram(rss, G, n, np.ones(2, bool), absolute_sigma=absolute)
    x0 = np.linspace(-4, 5, 29)
    D = np.stack([np.ones_like(x0), x0], axis=1)
    h = np.einsum("ia,ab,ib->i", D, np.linalg.inv(G), D)
    sig_new = np.linspace(0.2, 3.0, 29)
    value = D @ beta
    var = np.einsum("ia,ab,ib->i", D, cov, D)
    for sn in (sig_new, 1.7):
        p = uncertainty.bands(torch.from_numpy(value), torch.from_numpy(var), cov, rss, dof, level,
                              sigma_new=sn if np.ndim(sn) == 0 else torch.from_numpy(sn), absolute_sigma=absolute)
        if absolute:
            q = scipy.stats.norm.ppf((1 + level) / 2)
            hw_ci, hw_pi = q * np.sqrt(h), q * np.sqrt(h + np.square(sn))
        else:
            q = scipy.stats.t.ppf((1 + level) / 2, dof)
            s2 = rss / dof
            hw_ci, hw_pi = q * np.sqrt(s2 * h), q * np.sqrt(s2 * h + s2 * np.square(sn))
        assert p.t == q
        for got, want in ((p.ci_low, value - hw_ci), (p.ci_high, value + hw_ci),
                          (p.pi_low, value - hw_pi), (p.pi_high, value + hw_pi)):
            np.testing.assert_allclose(got.numpy(), want, rtol=1e-12, atol=1e-12)


def test_default_sigma_new_is_todays_band_bit_for_bit():
    _, _, _, A, w, G, beta, rss = _wls(seed=9)
    cov, _, dof, _ = uncertainty.covariance_from_gram(rss, G, A.shape[0], np.ones(2, bool))
    value = torch.linspace(-1, 1, 11, dtype=torch.float64)
    var = torch.linspace(0.0, 0.3, 11, dtype=torch.float64)
    a = uncertainty.bands(value, var, cov, rss, dof)
    b = uncertainty.bands(value, var, cov, rss, dof, sigma_new=1.0)
    assert torch.equal(a.pi_low, b.pi_low) and torch.equal(a.pi_high, b.pi_high)


# ---- every ValueError of the sigma arguments (raised before any device is touched) ----------------------
@pytest.mark.parametrize("sigma", [np.ones(9), np.ones((10, 1)), np.full(10, np.nan), np.full(10, np.inf),
                                   np.zeros(10), -np.ones(10)])
def test_bad_sigma_raises(sigma):
    with pytest.raises(ValueError):
        fitter.weights_from_sigma(sigma, 10, (fitter.F64,))


@pytest.mark.parametrize("s", [1e-20, 1e20])
def test_weights_outside_the_fp32_normal_range_raise_only_for_an_fp32_slot(s):
    sigma = np.full(10, s)
    w = fitter.weights_from_sigma(sigma, 10, (fitter.F64,))   # 1e40 and 1e-40 are normal fp64 numbers
    assert w.dtype == torch.float64
    with pytest.raises(ValueError):
        fitter.weights_from_sigma(sigma, 10, (fitter.F64, fitter.F32))


def _job(n=12, dtype=torch.float64):
    X = torch.zeros((1, n, 10), dtype=dtype)
    X[0, :, 0] = torch.linspace(0.5, 2.0, n, dtype=dtype)
    return X, 2.0 * X[0, :, 0]


def test_bfgs_batch_rejects_bad_sigma(golden, test_data):
    X, y = _job()
    toks = [[test_data.word2id[w] for w in ("S", "mul", "c", "x_1", "F")]]
    cfg = make_cfg(2)
    for bad in (np.ones(11), np.zeros(12), np.full(12, np.nan)):
        with pytest.raises(ValueError):
            vbfgs.bfgs_batch(toks, X, y, cfg, test_data, sigma=bad)
    with pytest.raises(ValueError):
        vbfgs.bfgs(toks[0], X, y, cfg, test_data, sigma=np.zeros(12))
    with pytest.raises(ValueError, match="idx_remove"):
        vbfgs.bfgs_batch(toks, X, y, make_cfg(2, idx_remove=True), test_data, sigma=np.ones(12))
    # fp32 points: the score slot is fp32, where 1/sigma^2 = 1e40 overflows
    Xf, yf = _job(dtype=torch.float32)
    with pytest.raises(ValueError):
        vbfgs.bfgs_batch(toks, Xf, yf, cfg, test_data, sigma=np.full(12, 1e-20))
    # precision fp32 sweeps: the eval slot is fp32 as well
    with pytest.raises(ValueError):
        vbfgs.bfgs_batch(toks, X, y, make_cfg(2, precision="fp32"), test_data, sigma=np.full(12, 1e20))


def test_refine_hypotheses_raises_for_bad_sigma_instead_of_failing_every_candidate(test_data):
    X, y = _job()
    hyp = [(0.0, [test_data.word2id[w] for w in ("S", "mul", "c", "x_1", "F")])]
    with pytest.raises(ValueError):
        refine.refine_hypotheses(hyp, X, y.reshape(1, -1, 1), make_cfg(2), test_data, sigma=np.ones(5))


def test_bands_and_predict_need_sigma_new_for_an_absolute_covariance():
    cov = np.eye(2)
    value, var = torch.zeros(4, dtype=torch.float64), torch.zeros(4, dtype=torch.float64)
    with pytest.raises(ValueError, match="sigma_new"):
        uncertainty.bands(value, var, cov, 1.0, 10, absolute_sigma=True)
    for bad in (np.ones(3), np.zeros(4), np.full(4, np.nan), np.ones((4, 1))):
        with pytest.raises(ValueError):
            uncertainty.bands(value, var, cov, 1.0, 10, sigma_new=bad)
    cv = uncertainty.ConstantCovariance(consts=np.ones(2), free=np.ones(2, bool), cov=cov, stderr=np.ones(2),
                                        rss=1.0, dof=10, rank=2, jtj=cov, absolute_sigma=True)
    with pytest.raises(ValueError, match="sigma_new"):
        uncertainty.predict([("", [1.0, 1.0], 0.0, "((c0)+((c1)*(x_1)))")], np.zeros((4, 1)), covs=[cv])


def test_covariances_rejects_bad_sigma():
    fits = [("", [1.0, 1.0], 0.0, "((c0)+((c1)*(x_1)))")]
    with pytest.raises(ValueError):
        uncertainty.covariances(fits, np.zeros((5, 1)), np.zeros(5), sigma=np.ones(4))
    with pytest.raises(ValueError):
        uncertainty.covariances(fits, np.zeros((5, 1)), np.zeros(5), sigma=np.zeros(5))


# ---- the weighted objective from the host interpreter's per-point tangents ------------------------------
@pytest.mark.parametrize("skel,k", [("((c0)*(sin(((c1)*(x_1))+(c2))))", 3), ("((c0)*(exp(((c1)*(x_1)))))", 2),
                                    ("(((c0)*(x_1))+((c1)/((x_2)+(c2))))", 3)])
def test_weighted_loss_and_gradient_from_host_tangents(hostsim, skel, k):
    rng = np.random.RandomState(k)
    n = 257
    X = np.zeros((n, 10))
    X[:, 0] = rng.uniform(-1.5, 1.5, n)
    X[:, 1] = rng.uniform(0.5, 2.0, n)
    y = rng.normal(size=n)
    w = np.exp(rng.uniform(np.log(1e-6), np.log(1e6), n))
    c = rng.uniform(0.5, 1.5, k)
    prog = compile_skeleton(skel, k, VARS)
    val, tan = R.host_duals(hostsim, prog.insns, prog.imms, c, X, k)
    r = val - y
    loss = np.mean(w * r * r)
    grad = 2.0 * np.mean((w * r)[:, None] * tan, axis=0)
    cs = sp.symbols(f"c0:{k}")
    xs = sp.symbols("x_1:11")
    expr = sp.sympify(skel, locals={f"c{i}": cs[i] for i in range(k)} | {f"x_{i + 1}": xs[i] for i in range(10)})
    f = sp.lambdify([cs, xs], expr, "numpy")
    dfs = [sp.lambdify([cs, xs], sp.diff(expr, ci), "numpy") for ci in cs]
    cols = [X[:, j] for j in range(10)]
    r_ref = f(c, cols) - y
    np.testing.assert_allclose(loss, np.mean(w * r_ref ** 2), rtol=1e-12)
    g_ref = np.array([2.0 * np.mean(w * r_ref * np.broadcast_to(df(c, cols), (n,))) for df in dfs])
    np.testing.assert_allclose(grad, g_ref, rtol=1e-10, atol=1e-12 * np.abs(g_ref).max())
    # w = 1 is the unweighted objective, bit for bit (a product with 1.0 is exact)
    ones = np.ones(n)
    assert np.mean(ones * r * r) == np.mean(r * r)
