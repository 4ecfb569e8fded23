"""vsr_predict and uncertainty.predict on the GPU: device values and variances against sympy's exact f
and Jacobian at every tangent width, consistency with vsr_gram, bit-for-bit independence of the batch,
the edge cases, int64 output offsets, the end-to-end path after bfgs_batch, and what the bands mean."""
import ctypes

import numpy as np
import pytest
import scipy.optimize
import scipy.stats
import torch

from _gram_ref import VARS, exact
from conftest import make_cfg
from src.visymre import uncertainty
from src.visymre.architectures import bfgs as vbfgs
from src.visymre.engine import fitter
from src.visymre.engine.compiler import compile_skeleton
from test_gpu_fit import _case_tensors
from test_gpu_uncertainty import WIDTHS, _BASIS, _points, _programs, _skeleton

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    return fitter.Engine("cuda:0")


def _spd(rng, k):
    A = rng.normal(size=(k, k))
    return A @ A.T / max(k, 1) + 0.1 * np.eye(k)


def _covs(rng, ks, kstride=16):
    cov = np.zeros((len(ks), kstride, kstride))
    for i, k in enumerate(ks):
        cov[i, :k, :k] = _spd(rng, k)
    return cov


def _reference(skel, k, X, c, cov):
    """(value [N], var [N]) from sympy's exact f and Jacobian, in fp64."""
    value, J = exact(skel, k, X, np.zeros(X.shape[0]), c)
    return value, np.einsum("ia,ab,ib->i", J, cov[:k, :k], J)


def _close(got, want, rtol, name):
    """Elementwise, relative to the row's scale (a sum of terms can cancel at single points)."""
    assert np.array_equal(np.isnan(got), np.isnan(want)), name
    inf = np.isinf(want)
    assert np.array_equal(got[inf], want[inf]), name
    ok = np.isfinite(want)
    if ok.any():
        np.testing.assert_allclose(got[ok], want[ok], rtol=rtol, atol=rtol * np.abs(want[ok]).max(), err_msg=name)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_values_and_variances_match_sympy_at_every_width(eng, dtype):
    ks, progs = _programs()
    X, _ = _points(5_003, 5, dtype)
    rng = np.random.RandomState(1)
    consts = rng.uniform(0.5, 1.5, size=(len(progs), 16)).astype(dtype).astype(np.float64)
    cov = _covs(rng, ks)
    dt = fitter.F64 if dtype == np.float64 else fitter.F32
    eng.set_points(torch.from_numpy(X), torch.zeros(X.shape[0]), dtypes=(dt,), n_vars=10)
    eng.set_programs(progs)
    value, var = eng.predict(np.arange(len(progs)), consts, cov=cov, dtype=dt)
    value, var = value.cpu().numpy(), var.cpu().numpy()
    rtol_v, rtol_s = (1e-12, 1e-10) if dtype == np.float64 else (1e-5, 1e-5)
    Xr = X.astype(np.float64)
    for i, (k, p) in enumerate(zip(ks, progs)):
        want_v, want_s = _reference(_skeleton(k), k, Xr, consts[i, :k], cov[i])
        _close(value[i], want_v, rtol_v, f"value k={k}")
        _close(var[i], want_s, rtol_s, f"var k={k}")


def test_consistent_with_vsr_gram(eng):
    ks, progs = _programs()
    X, y = _points(30_001, 8)
    eng.set_points(X, y, dtypes=(fitter.F64,), n_vars=10)
    eng.set_programs(progs)
    consts = np.random.RandomState(3).uniform(0.5, 1.5, size=(len(progs), 16))
    eye = np.broadcast_to(np.eye(16), (len(progs), 16, 16)).copy()
    value, var = eng.predict(np.arange(len(progs)), consts, cov=eye)
    rss, jtj = eng.gram(np.arange(len(progs)), consts)
    value, var, rss, jtj = (t.cpu().numpy() for t in (value, var, rss, jtj))
    for i, k in enumerate(ks):
        assert abs(var[i].sum() - np.trace(jtj[i, :k, :k])) <= 1e-12 * np.trace(jtj[i, :k, :k]), k
        assert abs(((value[i] - y) ** 2).sum() - rss[i]) <= 1e-12 * rss[i], k


def test_batch_independence_bit_for_bit(eng):
    ks, progs = _programs()
    X, _ = _points(20_000, 6)
    eng.set_points(X, np.zeros(20_000), dtypes=(fitter.F64,), n_vars=10)
    eng.set_programs(progs)
    rng = np.random.RandomState(2)
    consts = torch.from_numpy(rng.uniform(0.5, 1.5, size=(1024, 16)))
    prog_idx = np.arange(1024) % len(progs)
    cov = torch.from_numpy(_covs(rng, [ks[i] for i in prog_idx]))
    val_b, var_b = (t.cpu().numpy() for t in eng.predict(prog_idx, consts, cov=cov))
    perm = rng.permutation(1024)
    val_s, var_s = (t.cpu().numpy() for t in eng.predict(prog_idx[perm], consts, cov=cov, const_row=perm))
    assert np.array_equal(val_s, val_b[perm]) and np.array_equal(var_s, var_b[perm])
    for p in range(1024):
        v1, s1 = eng.predict([prog_idx[p]], consts[p:p + 1], cov=cov[p:p + 1])
        assert np.array_equal(v1.cpu().numpy()[0], val_b[p]) and np.array_equal(s1.cpu().numpy()[0], var_b[p]), p
    # values alone are the same values
    val_o, none = eng.predict(prog_idx, consts)
    assert none is None and np.array_equal(val_o.cpu().numpy(), val_b)


def _raw_predict(eng, prog_idx, consts, cov, ld_out, fill):
    """vsr_predict with an explicit row stride, outputs pre-filled with `fill`."""
    prog_idx = np.ascontiguousarray(prog_idx, dtype=np.int32)
    n = prog_idx.shape[0]
    consts = torch.as_tensor(consts, dtype=torch.float64).cuda().contiguous()
    cov = torch.as_tensor(cov, dtype=torch.float64).cuda().contiguous()
    value = torch.full((n, ld_out), fill, dtype=torch.float64, device="cuda:0")
    var = torch.full((n, ld_out), fill, dtype=torch.float64, device="cuda:0")
    eng._check(eng.lib.vsr_predict(eng._h, prog_idx.ctypes.data_as(ctypes.c_void_p), ctypes.c_void_p(0), n,
                                   ctypes.c_void_p(consts.data_ptr()), int(consts.shape[1]),
                                   ctypes.c_void_p(cov.data_ptr()), fitter.F64, ctypes.c_void_p(value.data_ptr()),
                                   ctypes.c_void_p(var.data_ptr()), ld_out, eng._stream()))
    return value.cpu().numpy(), var.cpu().numpy()


def test_edge_cases(eng):
    wide = "(" + "+".join(f"((c{j})*({_BASIS[j % len(_BASIS)]}))" for j in range(17)) + ")"
    domain = "((c0)*(sqrt((x_1)-(c1))))"
    skels = [(_skeleton(0), 0), (wide, 17), (domain, 2), (_skeleton(3), 3), (_skeleton(12), 12)]
    progs = [compile_skeleton(s, k, VARS) for s, k in skels]
    rng = np.random.RandomState(9)
    consts = np.zeros((len(skels), 17))
    consts[1] = np.linspace(0.5, 1.5, 17)
    consts[2, :2] = [1.5, 5.0]               # sqrt(x_1 - 5): not real for x_1 < 5
    consts[3, :3] = [0.7, 1.1, 0.9]
    consts[4, :12] = rng.uniform(0.5, 1.5, 12)
    cov = np.zeros((len(skels), 17, 17))
    for i, (_, k) in enumerate(skels):
        cov[i, :k, :k] = _spd(rng, k)
    for n in (1, 511, 512, 513, 3001):       # the tile is 512 points at widths <= 8, 256 above
        X = np.zeros((n, 10))
        X[:, :4] = rng.uniform(0.3, 9.0, size=(n, 4))
        eng.set_points(X, np.zeros(n), dtypes=(fitter.F64,), n_vars=10)
        eng.set_programs(progs)
        want = [_reference(s, k, X, consts[i, :k], cov[i]) for i, (s, k) in enumerate(skels)]
        for ld in (n, n + 37):
            value, var = _raw_predict(eng, np.arange(len(skels)), consts, cov, ld, -7.25)
            assert (value[:, n:] == -7.25).all() and (var[:, n:] == -7.25).all(), (n, ld)
            value, var = value[:, :n], var[:, :n]
            assert (var[0] == 0).all()                                         # k == 0
            assert np.isnan(var[1]).all()                                      # k > 16
            for i, (s, k) in enumerate(skels):
                want_v, want_s = want[i]
                _close(value[i], want_v, 1e-12, f"value {s} n={n}")
                if i not in (0, 1):
                    _close(var[i], want_s, 1e-10, f"var {s} n={n}")
            nan_at = X[:, 0] < 5.0
            assert np.array_equal(np.isnan(value[2]), nan_at) and np.array_equal(np.isnan(var[2]), nan_at)


def test_outputs_past_2_to_the_31(eng):
    """Values only, 2 200 pairs at N = 1e6: 2.2e9 pair-points (17.6 GB of output)."""
    n, pairs = 1_000_000, 2200
    need = pairs * n * 8 + (1 << 30)
    if torch.cuda.mem_get_info(0)[0] < need:
        pytest.skip(f"needs {need / 1e9:.1f} GB of free device memory")
    g = torch.Generator(device="cuda:0").manual_seed(11)
    X = torch.rand((n, 2), dtype=torch.float64, device="cuda:0", generator=g) * 2 + 0.5
    skels = [("(((c0)*(x_1))+(c1))", 2), ("((c0)*(sin((x_2)+(c1))))", 2), ("((c0)*(exp((x_1)*(c1))))", 2)]
    eng.set_points(X, torch.zeros(n, dtype=torch.float64), dtypes=(fitter.F64,), n_vars=2)
    eng.set_programs([compile_skeleton(s, k, VARS) for s, k in skels])
    prog_idx = np.arange(pairs) % len(skels)
    consts = np.random.RandomState(4).uniform(0.2, 1.2, size=(pairs, 2))
    value, var = eng.predict(prog_idx, consts)
    assert var is None
    Xh = np.zeros((n, 10))
    Xh[:, :2] = X.cpu().numpy()
    for p in (0, 1000, pairs - 3, pairs - 2, pairs - 1):
        s, k = skels[prog_idx[p]]
        want, _ = exact(s, k, Xh, np.zeros(n), consts[p])
        got = value[p].cpu().numpy()
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12 * np.abs(want).max(), err_msg=str(p))
    del value


def test_end_to_end_after_bfgs_batch(golden, test_data):
    checked = 0
    for case in golden["cases"]:
        X, y = _case_tensors(case)
        cfg = make_cfg(case["R"], case["norm"], case["idx_remove"], grad_mode="dual")
        calls = case["minimize_calls"][:case["R"]]
        x0 = [np.array([c["x0"] for c in calls])] if calls else None
        fits = vbfgs.bfgs_batch([case["tokens"]], X, y, cfg, test_data, x0=x0)
        if vbfgs._opt(cfg, "idx_remove", False):
            keep = (X < 200).all(dim=2).squeeze(0)
            Xf, yf = X[:, keep, :], y.reshape(-1)[:int(keep.sum())]
        else:
            Xf, yf = X, y
        covs = uncertainty.covariances(fits, Xf, yf)
        # held-out points: fresh draws within the range of the training points
        Xt = Xf[0].double().cpu().numpy()
        rng = np.random.RandomState(case["n"])
        lo, hi = Xt.min(axis=0), Xt.max(axis=0)
        Xn = rng.uniform(lo, hi, size=(997, Xt.shape[1]))
        preds = uncertainty.predict(fits, torch.from_numpy(Xn).cuda(), covs=covs, dtype=fitter.F64)
        Xn10 = np.concatenate([Xn, np.zeros((Xn.shape[0], 10 - Xn.shape[1]))], axis=1)
        for fit, cv, pr in zip(fits, covs, preds):
            if isinstance(fit, Exception):
                assert pr is None
                continue
            c = np.asarray(fit[1], dtype=np.float64)
            want_v, J = exact(str(fit[3]), c.size, Xn10, np.zeros(Xn.shape[0]), c)
            _close(pr.value.cpu().numpy(), want_v, 1e-12, str(fit[3]))
            assert pr.dof == cv.dof and pr.value.device.type == "cuda"
            if np.isfinite(cv.cov[np.ix_(cv.free, cv.free)]).all() and np.isfinite(J).all() and cv.dof > 0:
                dc = uncertainty.device_cov(cv.cov)
                want_se = np.sqrt(np.einsum("ia,ab,ib->i", J, dc, J))
                _close(pr.se_fit.cpu().numpy(), want_se, 1e-8, str(fit[3]))
            checked += 1
    assert checked >= 15, checked


def test_linear_fit_bands_match_the_ols_closed_form(eng):
    rng = np.random.RandomState(21)
    n = 300
    x = rng.uniform(-2, 3, n)
    y = 0.7 + 1.9 * x + rng.normal(0, 0.3, n)
    A = np.stack([np.ones(n), x], axis=1)
    beta = np.linalg.lstsq(A, y, rcond=None)[0]
    fit = ("", beta, 0.0, "((c0)+((c1)*(x_1)))")
    X = torch.from_numpy(x.reshape(n, 1))
    cv = uncertainty.covariances([fit], X, torch.from_numpy(y), engine=eng)
    x0 = np.linspace(-4, 5, 1001)
    pr = uncertainty.predict([fit], x0.reshape(-1, 1), covs=cv, level=0.9, engine=eng)[0]
    rss = float(np.sum((A @ beta - y) ** 2))
    D = np.stack([np.ones_like(x0), x0], axis=1)
    h = np.einsum("ia,ab,ib->i", D, np.linalg.inv(A.T @ A), D)
    s, t = np.sqrt(rss / (n - 2)), scipy.stats.t.ppf(0.95, n - 2)
    yhat = D @ beta
    for got, want in ((pr.value, yhat), (pr.ci_low, yhat - t * s * np.sqrt(h)), (pr.ci_high, yhat + t * s * np.sqrt(h)),
                      (pr.pi_low, yhat - t * s * np.sqrt(1 + h)), (pr.pi_high, yhat + t * s * np.sqrt(1 + h))):
        np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-9, atol=1e-9)
    assert pr.dof == n - 2 and pr.t == pytest.approx(t, rel=1e-15)


def test_bands_cover_at_their_level(eng):
    """200 seeded noisy data sets y = 2 sin(1.3 x_1) + 0.5 + N(0, 0.1^2), N = 200, fitted by curve_fit:
    at each of 5 fixed points the 95 % confidence band covers the true f and the 95 % prediction band
    a fresh noisy draw in a share of the data sets within the binomial 99 % bounds of 0.95."""
    skel = "(((c0)*(sin((c1)*(x_1))))+(c2))"
    truth = np.array([2.0, 1.3, 0.5])

    def f(x, c0, c1, c2):
        return c0 * np.sin(c1 * x) + c2
    x0 = np.array([-2.5, -1.0, 0.0, 1.2, 2.8])
    rng = np.random.RandomState(2024)
    fits, covs = [], []
    for _ in range(200):
        x = rng.uniform(-3, 3, 200)
        y = f(x, *truth) + rng.normal(0, 0.1, 200)
        c, _ = scipy.optimize.curve_fit(f, x, y, p0=truth)
        fit = ("", c, 0.0, skel)
        fits.append(fit)
        covs += uncertainty.covariances([fit], torch.from_numpy(x.reshape(-1, 1)), torch.from_numpy(y), engine=eng)
    preds = uncertainty.predict(fits, x0.reshape(-1, 1), covs=covs, engine=eng)
    f_true = f(x0, *truth)
    y_new = f_true + rng.normal(0, 0.1, size=(200, x0.size))
    ci = np.zeros(x0.size)
    pi = np.zeros(x0.size)
    for j, p in enumerate(preds):
        lo, hi = p.ci_low.cpu().numpy(), p.ci_high.cpu().numpy()
        ci += (lo <= f_true) & (f_true <= hi)
        lo, hi = p.pi_low.cpu().numpy(), p.pi_high.cpu().numpy()
        pi += (lo <= y_new[j]) & (y_new[j] <= hi)
    lo, hi = scipy.stats.binom.interval(0.99, 200, 0.95)
    assert ((ci >= lo) & (ci <= hi)).all(), ci
    assert ((pi >= lo) & (pi <= hi)).all(), pi


def test_argument_checks_and_overflow(eng):
    X = np.zeros((100, 10))
    X[:, 0] = np.linspace(0.0, 800.0, 100)
    eng.set_points(X, np.zeros(100), dtypes=(fitter.F64,), n_vars=1)
    eng.set_programs([compile_skeleton("((c0)*(exp(x_1)))", 1, VARS)])
    consts = np.ones((2, 1))
    with pytest.raises(ValueError):                 # fewer covariance rows than constant rows
        eng.predict([0, 0], consts, cov=np.ones((1, 1, 1)))
    with pytest.raises(ValueError):                 # const_row past the rows of consts / cov
        eng.predict([0, 0], consts, cov=np.ones((2, 1, 1)), const_row=[0, 2])
    with pytest.raises(ValueError):
        eng.predict([0, 0, 0], consts)
    value, var = eng.predict([0, 0], np.array([[1.0], [-1.0]]), cov=np.ones((2, 1, 1)))
    value, var = value.cpu().numpy(), var.cpu().numpy()
    with np.errstate(over="ignore"):
        want = np.exp(X[:, 0])
    assert np.isposinf(value[0, -1]) and np.isneginf(value[1, -1])             # +-inf past exp's range
    _close(value[0], want, 1e-13, "exp")
    _close(value[1], -want, 1e-13, "-exp")
    with np.errstate(over="ignore"):
        _close(var[0], want * want, 1e-13, "var exp")
