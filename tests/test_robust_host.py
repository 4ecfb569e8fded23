"""Robust losses on the host: the numpy twin of the device's per-point factors against mpmath and scipy's
loss functions, ``covariance_from_gram`` on robust statistics against curve_fit's formula (least_squares'
scaled Jacobian, then its SVD ``pcov``), and every ``ValueError`` of the ``loss`` / ``f_scale`` arguments
(raised before any device is touched)."""
import mpmath as mp
import numpy as np
import pytest
import torch
from scipy.optimize._lsq.common import scale_for_robust_loss_function
from scipy.optimize._lsq.least_squares import arctan, cauchy, construct_loss_function, huber, soft_l1

import _robust_ref as RR
from conftest import make_cfg
from src.visymre import uncertainty
from src.visymre.architectures import bfgs as vbfgs
from src.visymre.architectures import refine
from src.visymre.engine import fitter

IMPL = {"soft_l1": soft_l1, "huber": huber, "cauchy": cauchy, "arctan": arctan}   # scipy's rho(z)
ZS = [0.0, 1e-300, 1e-20, 1e-8, 0.5, 1.0, np.nextafter(1.0, np.inf), np.nextafter(1.0, -np.inf), 2.0, 1e8, 1e300,
      np.inf]


def _mp_ref(loss, z):
    """(q, g, s) at z in 700-digit arithmetic (s unclamped): enough for 2 (sqrt(1 + z) - 1) at z = 1e-300."""
    mp.mp.dps = 700
    if z == np.inf:
        return 0.0, 0.0, 0.0
    Z = mp.mpf(float(z))
    if loss == "soft_l1":
        rho, g, s = 2 * (mp.sqrt(1 + Z) - 1), 1 / mp.sqrt(1 + Z), (1 + Z) ** mp.mpf(-1.5)
    elif loss == "huber":
        rho, g, s = (Z, 1, 1) if Z <= 1 else (2 * mp.sqrt(Z) - 1, 1 / mp.sqrt(Z), 0)
    elif loss == "cauchy":
        rho, g, s = mp.log1p(Z), 1 / (1 + Z), (1 - Z) / (1 + Z) ** 2
    else:
        rho, g, s = mp.atan(Z), 1 / (1 + Z * Z), (1 - 3 * Z * Z) / (1 + Z * Z) ** 2
    q = mp.mpf(1) if Z == 0 else rho / Z
    return float(q), float(g), float(s)


@pytest.mark.parametrize("loss", RR.ROBUST)
def test_twin_factors_match_mpmath(loss):
    q, g, sbar = RR.factors(loss, np.array(ZS))
    for i, z in enumerate(ZS):
        wq, wg, ws = _mp_ref(loss, z)
        np.testing.assert_allclose(q[i], wq, rtol=4e-16, atol=0, err_msg=f"q {loss} {z}")
        np.testing.assert_allclose(g[i], wg, rtol=4e-16, atol=0, err_msg=f"g {loss} {z}")
        np.testing.assert_allclose(sbar[i], max(ws, RR.EPS), rtol=1e-15, atol=0, err_msg=f"s {loss} {z}")


def test_twin_cost_at_infinity_is_scipys():
    for loss in RR.ROBUST:
        cost, gfac, _, ws = RR.terms(loss, 3.0, np.array([1e200]))
        assert cost[0] == 9.0 * (np.pi / 2 if loss == "arctan" else np.inf)
        assert gfac[0] == 0.0 and ws[0] == RR.EPS
    rho = construct_loss_function(1, "arctan", 3.0)(np.array([1e200]))   # scipy's C^2 rho at z = inf
    assert rho[0, 0] == 9.0 * np.pi / 2 and rho[1, 0] == 0.0


@pytest.mark.parametrize("loss", RR.ROBUST)
def test_twin_factors_match_scipys_loss_functions_where_they_are_accurate(loss):
    z = np.array([v for v in ZS if 1e-8 <= v < np.inf])
    rho = np.empty((3, len(z)))
    with np.errstate(all="ignore"):
        IMPL[loss](z.copy(), rho, cost_only=False)
    q, g, sbar = RR.factors(loss, z)
    eps = np.finfo(np.float64).eps
    # scipy's 2 (sqrt(1+z) - 1) cancels below z = 1, and its rho' + 2 z rho'' by up to eps rho'
    np.testing.assert_array_less(np.abs(q - rho[0] / z), (1e-14 + 4 * eps / np.minimum(z, 1.0)) * np.abs(q))
    np.testing.assert_allclose(g, rho[1], rtol=1e-14)
    with np.errstate(all="ignore"):
        s_scipy = rho[1] + 2 * rho[2] * z
    s_scipy = np.where(s_scipy > RR.EPS, s_scipy, RR.EPS)
    np.testing.assert_array_less(np.abs(sbar - s_scipy), 1e-14 * sbar + 4 * eps * g + 1e-300)


def test_huber_with_every_z_at_most_one_is_linear_bit_for_bit():
    r = np.random.RandomState(0).normal(size=1000) * 100.0
    w = np.exp(np.random.RandomState(1).uniform(-3, 3, 1000))
    for ww in (None, w):
        lin = RR.terms("linear", 1.0, r, ww)
        hub = RR.terms("huber", 2.0 ** 20, r, ww)
        for a, b in zip(lin, hub):
            assert a.tobytes() == b.tobytes()


# ---- covariance_from_gram on robust statistics is curve_fit's pcov -------------------------------------
def _curve_fit_pcov(J, r, w, loss, f_scale, absolute):
    """curve_fit's pcov after least_squares: the scaled Jacobian of sqrt(w)-weighted residuals, then SVD."""
    sw = np.sqrt(w)
    f = sw * r
    Jw = sw[:, None] * J
    rho = construct_loss_function(len(f), loss, f_scale)(f)
    cost = np.sum(rho[0])                        # = 2 * res.cost
    Js, _ = scale_for_robust_loss_function(Jw.copy(), f.copy(), rho)
    _, s, VT = np.linalg.svd(Js, full_matrices=False)
    pcov = (VT.T / s ** 2) @ VT
    if not absolute:
        pcov = pcov * cost / (len(f) - J.shape[1])
    return pcov, cost


@pytest.mark.parametrize("loss", RR.ROBUST)
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("absolute", [False, True])
def test_covariance_from_robust_gram_matches_curve_fit(loss, weighted, absolute):
    rng = np.random.RandomState(7)
    n = 200
    x = rng.uniform(0.2, 2.0, n)
    c = np.array([1.3, 0.8])
    J = np.stack([np.exp(c[1] * x), c[0] * x * np.exp(c[1] * x)], axis=1)
    r = rng.normal(size=n) * 0.2
    r[::10] += 5.0                              # outliers: z > 1 for every loss at f_scale 0.5
    w = np.exp(rng.uniform(-1, 1, n)) if weighted else np.ones(n)
    rss, jtj = RR.gram(loss, 0.5, r, J, w if weighted else None)
    cov, stderr, dof, rank = uncertainty.covariance_from_gram(rss, jtj, n, np.ones(2, bool), absolute)
    want, cost = _curve_fit_pcov(J, r, w, loss, 0.5, absolute)
    np.testing.assert_allclose(rss, cost, rtol=1e-12)
    np.testing.assert_allclose(cov, want, rtol=1e-9)
    assert rank == 2 and dof == n - 2


# ---- every ValueError of loss / f_scale ---------------------------------------------------------------
@pytest.mark.parametrize("loss,f_scale", [("bogus", 1.0), ("Huber", 1.0), (None, 1.0), (len, 1.0), ("huber", 0.0),
                                          ("huber", -1.0), ("huber", np.nan), ("huber", np.inf), ("huber", 1e160),
                                          ("huber", 1e-160), ("soft_l1", "x"), ("linear", 0.0)])
def test_robust_loss_rejects(loss, f_scale):
    with pytest.raises(ValueError):
        fitter.robust_loss(loss, f_scale)


def test_robust_loss_accepts():
    assert fitter.robust_loss() is None
    assert fitter.robust_loss("linear", 3.0) is None
    for name in RR.ROBUST:
        assert fitter.robust_loss(name, 2 ** 20) == (name, float(2 ** 20))
    assert fitter.robust_loss("cauchy", 1e150) == ("cauchy", 1e150)


def _job(n=12):
    X = torch.zeros((1, n, 10), dtype=torch.float64)
    X[0, :, 0] = torch.linspace(0.5, 2.0, n, dtype=torch.float64)
    return X, 2.0 * X[0, :, 0]


def test_bfgs_refine_and_covariances_reject_a_bad_loss(test_data):
    X, y = _job()
    toks = [[test_data.word2id[w] for w in ("S", "mul", "c", "x_1", "F")]]
    for loss, fs in (("bogus", 1.0), ("huber", 0.0), ("soft_l1", 1e-200)):
        with pytest.raises(ValueError):
            vbfgs.bfgs_batch(toks, X, y, make_cfg(2), test_data, loss=loss, f_scale=fs)
        with pytest.raises(ValueError):
            vbfgs.bfgs(toks[0], X, y, make_cfg(2), test_data, loss=loss, f_scale=fs)
        with pytest.raises(ValueError):
            refine.refine_hypotheses([(0.0, toks[0])], X, y.reshape(1, -1, 1), make_cfg(2), test_data, loss=loss,
                                     f_scale=fs)
        with pytest.raises(ValueError):
            uncertainty.covariances([("", [1.0], 0.0, "((c0)*(x_1))")], X, y, loss=loss, f_scale=fs)


def test_constant_covariance_defaults_to_the_linear_loss():
    cv = uncertainty.ConstantCovariance(consts=np.ones(1), free=np.ones(1, bool), cov=np.eye(1), stderr=np.ones(1),
                                        rss=1.0, dof=3, rank=1, jtj=np.eye(1))
    assert cv.loss == "linear" and cv.f_scale == 1.0
