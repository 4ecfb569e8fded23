"""vsr_gram and uncertainty.covariances on the GPU: the device Gram against its CPU reference at
every tangent width, bit-for-bit independence of the batch, the edge cases, a config-5 size against
the closed form, the end-to-end path after bfgs_batch, and what the standard errors mean."""
import numpy as np
import pytest
import torch

import bench
from _gram_ref import VARS, exact, frob_rel, load_twin, twin_gram
from conftest import make_cfg
from src.visymre import uncertainty
from src.visymre.architectures import bfgs as vbfgs
from src.visymre.engine import fitter
from src.visymre.engine.compiler import compile_skeleton
from src.visymre.workloads import generator as wg
from test_gpu_fit import _case_tensors

pytestmark = pytest.mark.gpu
WIDTHS = [1, 2, 3, 4, 5, 6, 7, 8, 12, 16]
_BASIS = ["sin(x_1)", "x_2", "cos(x_3)", "exp((x_1)/(4))", "sqrt(x_2)", "(x_3)**(2)", "ln(x_1)", "x_4"]


@pytest.fixture(scope="module")
def eng():
    return fitter.Engine("cuda:0")


@pytest.fixture(scope="module")
def twin():
    """The CPU reference of vsr_gram (tests/native/gram_twin.cpp)."""
    return load_twin()


def _skeleton(k):
    """c0 * (c1 + sin(x_1 + c2) ...): every constant in a nonlinear place for k >= 2."""
    if k == 0:
        return "((sin(x_1))+(x_2))"
    terms = [f"((c{j})*({_BASIS[j % len(_BASIS)]}))" for j in range(1, k)]
    body = "((c0)+(x_1))" if not terms else "(" + "+".join(terms) + ")"
    return f"((c0)*{body})" if terms else body


def _points(n, seed, dtype=np.float64):
    rng = np.random.RandomState(seed)
    X = rng.uniform(0.3, 2.0, size=(n, 10)).astype(dtype)
    y = rng.normal(size=n).astype(dtype)
    return X, y


def _programs():
    ks = sorted({k for K in WIDTHS for k in (K, K - 1)})
    return ks, [compile_skeleton(_skeleton(k), k, VARS) for k in ks]


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_device_gram_matches_the_cpu_reference_at_every_width(eng, twin, dtype):
    ks, progs = _programs()
    X, y = _points(70_001, 5, dtype)
    eng.set_points(torch.from_numpy(X), torch.from_numpy(y), dtypes=(fitter.F64,), n_vars=10)
    eng.set_programs(progs)
    rng = np.random.RandomState(1)
    consts = rng.uniform(0.5, 1.5, size=(len(progs), 16))
    rss, jtj = eng.gram(np.arange(len(progs)), consts)
    rss, jtj = rss.cpu().numpy(), jtj.cpu().numpy()
    for i, (k, p) in enumerate(zip(ks, progs)):
        want_rss, want_jtj = twin_gram(twin, p, X, y, consts[i, :k])
        assert abs(rss[i] - want_rss) <= 1e-12 * want_rss, (k, rss[i], want_rss)
        assert frob_rel(jtj[i, :k, :k], want_jtj) <= 1e-12, k
        assert np.array_equal(jtj[i, :k, :k], jtj[i, :k, :k].T), k
        assert np.isnan(jtj[i, k:, :]).all() and np.isnan(jtj[i, :, k:]).all(), k


def test_batch_independence_bit_for_bit(eng):
    ks, progs = _programs()
    X, y = _points(20_000, 6)
    eng.set_points(X, y, dtypes=(fitter.F64,), n_vars=10)
    eng.set_programs(progs)
    rng = np.random.RandomState(2)
    consts = torch.from_numpy(rng.uniform(0.5, 1.5, size=(1024, 16)))
    prog_idx = np.arange(1024) % len(progs)
    rss_b, jtj_b = eng.gram(prog_idx, consts)
    rss_r, jtj_r = eng.gram(prog_idx[::-1].copy(), consts, const_row=np.arange(1024)[::-1].copy())
    rss_b, jtj_b = rss_b.cpu().numpy(), jtj_b.cpu().numpy()
    rss_r, jtj_r = rss_r.cpu().numpy()[::-1], jtj_r.cpu().numpy()[::-1]
    assert np.array_equal(rss_b, rss_r) and np.array_equal(jtj_b, jtj_r, equal_nan=True)
    for p in (0, 1, 7, len(progs) - 1, 500, 1023):
        rss_1, jtj_1 = eng.gram([prog_idx[p]], consts[p:p + 1])
        assert rss_1.item() == rss_b[p]
        assert np.array_equal(jtj_1.cpu().numpy()[0], jtj_b[p], equal_nan=True), p


def test_edge_cases(eng, twin):
    X, y = _points(3000, 7)
    wide = "(" + "+".join(f"((c{j})*({_BASIS[j % len(_BASIS)]}))" for j in range(17)) + ")"
    progs = [compile_skeleton(wide, 17, VARS), compile_skeleton(_skeleton(0), 0, VARS),
             compile_skeleton("((c0)*(sqrt((x_1)-(c1))))", 2, VARS)]
    eng.set_points(X, y, dtypes=(fitter.F64,), n_vars=10)
    eng.set_programs(progs)
    consts = np.zeros((3, 17))
    consts[0] = np.linspace(0.5, 1.5, 17)
    consts[2, :2] = [1.0, 1.0]               # x_1 - 1 < 0 for part of the points: not real there
    rss, jtj = eng.gram([0, 1, 2], consts)
    rss, jtj = rss.cpu().numpy(), jtj.cpu().numpy()
    want_wide, _ = twin_gram(twin, progs[0], X, y, consts[0])
    want_zero, _ = twin_gram(twin, progs[1], X, y, consts[1, :0])
    assert rss[0] == pytest.approx(want_wide, rel=1e-12) and np.isnan(jtj[0]).all()
    assert rss[1] == pytest.approx(want_zero, rel=1e-12) and np.isnan(jtj[1]).all()
    assert np.isnan(rss[2]) and np.isnan(jtj[2, :2, :2]).all()
    fits = [("", [1.0, 1.0], 0.0, "((c0)*(sqrt((x_1)-(c1))))"), ("", [], 0.0, _skeleton(0)), None]
    out = uncertainty.covariances(fits, X, y, engine=eng)
    assert np.isposinf(out[0].cov).all() and np.isposinf(out[0].stderr).all() and out[0].rank == 0
    assert out[1].cov.shape == (0, 0) and out[1].rss == pytest.approx(want_zero, rel=1e-12)
    assert out[2] is None


def test_config_5_size_against_the_closed_form(eng):
    n = 10_000_000
    g = torch.Generator(device="cuda:0").manual_seed(3)
    x = torch.rand(n, dtype=torch.float64, device="cuda:0", generator=g) * 4 - 2
    y = 1.5 * x - 0.25 + 0.1 * torch.randn(n, dtype=torch.float64, device="cuda:0", generator=g)
    eng.set_points(x.reshape(n, 1), y, dtypes=(fitter.F64,), n_vars=1)
    eng.set_programs([compile_skeleton("(((c0)*(x_1))+(c1))", 2, VARS)])
    c = torch.tensor([[1.4, -0.2]], dtype=torch.float64)
    rss, jtj = eng.gram([0], c)
    xn, yn = x.cpu().numpy(), y.cpu().numpy()
    r = 1.4 * xn - 0.2 - yn
    want = np.array([[np.sum(xn * xn), np.sum(xn)], [np.sum(xn), float(n)]])
    assert frob_rel(jtj.cpu().numpy()[0], want) <= 1e-10
    assert rss.item() == pytest.approx(float(np.sum(r * r)), rel=1e-10)


def _stderr_reference(fit, X, y):
    """(stderr, rss) from the exact Jacobian (sympy), or None when cond(J) > 1e5 or J is not finite."""
    c = np.asarray(fit[1], dtype=np.float64)
    free = c != 0.0
    if c.size == 0 or not free.any():
        return None
    r, J = exact(str(fit[3]), c.size, X, y, c)
    if not (np.isfinite(r).all() and np.isfinite(J).all()) or np.linalg.cond(J[:, free]) > 1e5:
        return None
    cov, stderr, _, rank = uncertainty.covariance_from_gram(r @ r, J.T @ J, len(y), free)
    return (stderr, r @ r) if rank == free.sum() and r @ r > 0 else None


def _canon(outs):
    return [repr(o) if isinstance(o, Exception) else (str(o[0]), np.asarray(o[1], np.float64).tobytes(),
                                                        np.asarray(o[2]).tobytes(), str(o[3])) for o in outs]


def test_end_to_end_after_bfgs_batch(golden, test_data):
    checked = 0
    jobs = []
    for case in golden["cases"]:
        X, y = _case_tensors(case)
        cfg = make_cfg(case["R"], case["norm"], case["idx_remove"], grad_mode="dual")
        calls = case["minimize_calls"][:case["R"]]
        x0 = [np.array([c["x0"] for c in calls])] if calls else None
        jobs.append(([case["tokens"]], X, y, cfg, test_data, x0))
    td = wg.make_test_data()
    for b in bench.make_workload(4, 10_000, 64, 10):
        X = torch.from_numpy(np.ascontiguousarray(b.X[None])).cuda()
        y = torch.from_numpy(np.ascontiguousarray(b.y)).cuda()
        jobs.append((list(b.tokens), X, y, wg.make_cfg(10, 64, grad_mode="dual"), td, b.x0))
    for toks, X, y, cfg, tdata, x0 in jobs:
        fits = vbfgs.bfgs_batch(toks, X, y, cfg, tdata, x0=x0)
        first = _canon(fits)
        if vbfgs._opt(cfg, "idx_remove", False):
            keep = (X < 200).all(dim=2).squeeze(0)
            Xf, yf = X[:, keep, :], y.reshape(-1)[:int(keep.sum())]
        else:
            Xf, yf = X, y
        out = uncertainty.covariances(fits, Xf, yf)
        again = _canon(vbfgs.bfgs_batch(toks, X, y, cfg, tdata, x0=x0))
        assert again == first
        Xn = Xf[0].double().cpu().numpy()
        Xn = np.concatenate([Xn, np.zeros((Xn.shape[0], 10 - Xn.shape[1]))], axis=1)
        yn = yf.reshape(-1).double().cpu().numpy()
        for fit, cv in zip(fits, out):
            if isinstance(fit, Exception):
                assert cv is None
                continue
            ref = _stderr_reference(fit, Xn, yn)
            if ref is None:
                continue
            want, rss = ref
            # at an exact fit rss is rounding of f - y: the device's and numpy's agree to a few ulps of
            # |y| per point, and the stderr is compared at the reference's rss
            scale = 1e-15 * np.linalg.norm(yn) + 1e-15 * len(yn)
            assert abs(cv.rss - rss) <= 1e-10 * rss + 4 * np.sqrt(rss) * scale + scale ** 2, (str(fit[3]), cv.rss, rss)
            free = cv.free
            np.testing.assert_allclose(cv.stderr[free] * np.sqrt(rss / cv.rss), want[free], rtol=1e-8,
                                       err_msg=str(fit[3]))
            checked += 1
    assert checked >= 20, checked


def test_affine_sin_and_a_degenerate_winner(golden):
    case = next(c for c in golden["cases"] if c["name"] == "affine_sin")
    X, y = _case_tensors(case)
    fit = (case["best_expr_str"], case["best_consts"], case["best_loss"], case["skeleton"])
    cv = uncertainty.covariances([fit, ("", [1.3, 0.7], 0.0, "((c0)*((c1)*(x_1)))")], X, y)
    assert np.isfinite(cv[0].stderr).all() and cv[0].rank == 2
    assert cv[1].rank == 1 and np.isposinf(cv[1].cov).all()


def test_standard_errors_cover_the_true_constants(golden, test_data):
    """200 seeded noisy data sets y = 2.5 sin(x_1) + 0.75 + N(0, 0.1^2), N = 1000: both true constants
    within 1.96 stderr in at least 88 % of them (95 % nominal; a loose binomial bound)."""
    case = next(c for c in golden["cases"] if c["name"] == "affine_sin")
    cfg = make_cfg(3, grad_mode="dual")
    rng = np.random.RandomState(12345)
    hits = np.zeros(2)
    for _ in range(200):
        X = np.zeros((1, 1000, 10))
        X[0, :, 0] = rng.uniform(-3, 3, 1000)
        y = 2.5 * np.sin(X[0, :, 0]) + 0.75 + rng.normal(0, 0.1, 1000)
        Xt, yt = torch.from_numpy(X).cuda(), torch.from_numpy(y).cuda()
        fit = vbfgs.bfgs_batch([case["tokens"]], Xt, yt, cfg, test_data, x0=[rng.randn(3, 2) * 10])[0]
        cv = uncertainty.covariances([fit], Xt, yt)[0]
        hits += np.abs(cv.consts - np.array([0.75, 2.5])) <= 1.96 * cv.stderr
    assert (hits >= 176).all(), hits
