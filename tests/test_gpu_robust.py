"""Robust losses on the GPU: huber with every z <= 1 reproduces the linear fit, evaluation and Gram bit for bit
on every kernel path; robust evaluation and Gram against the host interpreter's reference and the numpy twin;
FD fits against a robust scipy BFGS; outlier recovery against ``least_squares``; the ranking of a beam;
curve_fit's covariance; batch independence; the non-finite rules; and the loss carried to other engines."""
import ctypes

import numpy as np
import pytest
import scipy.optimize
import sympy as sp
import torch

import _interp_ref as R
import _robust_ref as RR
from _gram_ref import VARS, exact
from conftest import make_cfg
from oracle import vectorised
from src.visymre import uncertainty
from src.visymre.architectures import bfgs as vbfgs
from src.visymre.architectures.refine import refine_hypotheses
from src.visymre.engine import fitter, isa
from src.visymre.engine.compiler import compile_skeleton
from test_gpu_fit import _case_tensors
from test_gpu_uncertainty import _canon
from test_gpu_weights import DT, DUAL, FD, WIDTHS, _beam_jobs, _fit_all, _points, _programs, _set

pytestmark = pytest.mark.gpu
UNIT = 2.0 ** 20     # huber's f_scale with every z <= 1 on these data: the linear results, bit for bit
# Fits of beam candidates pass through residuals far above 2**20 (line searches from x0 = randn * 10), so
# the beam-level comparison keeps every finite z <= 1 with the largest scale whose C**2 is a normal double
WIDE = 2.0 ** 500


@pytest.fixture(scope="module")
def eng():
    return fitter.Engine("cuda:0")


def _set_loss(eng, loss, f_scale, dt):
    eng._check(eng.lib.vsr_set_loss(eng._h, isa.LOSS["VSR_LOSS_" + loss.upper()], float(f_scale), dt))


def _w(n, seed, lo=0.1, hi=10.0):
    return np.exp(np.random.RandomState(seed).uniform(np.log(lo), np.log(hi), n))


# ---- 1. the huber rule ---------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("n,offset", [(3001, 0), (3001, 1), (600_001, 0), (600_001, 1)])
@pytest.mark.parametrize("weighted", [False, True])
def test_huber_with_every_z_at_most_one_is_the_linear_eval_and_fit_bit_for_bit(eng, dtype, n, offset, weighted):
    """n = 3001: resident fit slices and eval_kernel; n = 600 001: streamed fp64 slices and the shared tiles
    of eval_tile_kernel.  offset 1: unaligned columns (coalesced loads instead of TMA)."""
    ks, progs = _programs()
    X, y = _points(n, 5, dtype)
    dt = DT[dtype]
    w = _w(n, 6) if weighted else None
    eng.set_programs(progs)
    consts = np.random.RandomState(3).uniform(0.5, 1.5, size=(len(ks), max(ks)))
    got = {}
    for loss in ("linear", "huber"):
        _set(eng, X, y, dt, w, offset)
        if loss == "huber":
            _set_loss(eng, "huber", UNIT, dt)
        lo, gr = eng.eval(np.arange(len(ks)), consts, dtype=dt, grad=True)
        out = [lo.cpu().numpy().tobytes(), gr.cpu().numpy().tobytes()]
        for mode in (DUAL, FD):
            out += _fit_all(eng, ks, mode, dtype, 8 if n > 10_000 else 40)
        got[loss] = out
    assert got["linear"] == got["huber"]


@pytest.mark.parametrize("weighted", [False, True])
def test_huber_with_every_z_at_most_one_is_the_linear_gram_bit_for_bit(eng, weighted):
    ks, progs = _programs()
    X, y = _points(70_001, 6)
    w = _w(70_001, 7) if weighted else None
    eng.set_programs(progs)
    consts = np.random.RandomState(4).uniform(0.5, 1.5, size=(len(ks), max(ks)))
    got = []
    for loss in (None, ("huber", UNIT)):
        eng.set_points(torch.from_numpy(X), torch.from_numpy(y), dtypes=(fitter.F64,), n_vars=10, w=w, loss=loss)
        rss, jtj = eng.gram(np.arange(len(ks)), consts)
        got.append((rss.cpu().numpy().tobytes(), jtj.cpu().numpy().tobytes()))
    assert got[0] == got[1]


# ---- 2. robust eval and Gram against the host reference -------------------------------------------------
@pytest.mark.parametrize("loss", RR.ROBUST)
@pytest.mark.parametrize("weighted", [False, True])
def test_robust_eval_and_gram_match_the_host_reference_at_every_width(eng, hostsim, loss, weighted):
    ks, progs = _programs()
    n = 20_001
    X, y = _points(n, 7)
    y[::13] += 30.0                                 # outliers: z far above 1
    w = _w(n, 8, 1e-3, 1e3) if weighted else None
    f_scale = 0.7
    consts = np.random.RandomState(9).uniform(0.5, 1.5, size=(len(ks), max(ks)))
    eng.set_points(torch.from_numpy(X), torch.from_numpy(y), dtypes=(fitter.F64,), n_vars=10, w=w,
                   loss=(loss, f_scale))
    eng.set_programs(progs)
    lo, gr = eng.eval(np.arange(len(ks)), consts, dtype=fitter.F64, grad=True)
    rss, jtj = eng.gram(np.arange(len(ks)), consts)
    lo, gr, rss, jtj = (t.cpu().numpy() for t in (lo, gr, rss, jtj))
    for j, (k, p) in enumerate(zip(ks, progs)):
        val, tan = R.host_duals(hostsim, p.insns, p.imms, consts[j, :k], X, next(K for K in WIDTHS if K >= k))
        tan = tan[:, :k]
        r = val - y
        want, g = RR.objective(loss, f_scale, r, tan, w)
        assert abs(lo[j] - want) <= 1e-12 * want, (k, lo[j], want)
        assert abs(rss[j] - n * want) <= 1e-12 * n * want
        if k == 0:
            continue
        _, gf, _, ws = RR.terms(loss, f_scale, r, w)
        bound = 2.0 * (np.abs(gf)[:, None] * np.abs(tan)).sum(axis=0) / n
        np.testing.assert_array_less(np.abs(gr[j, :k] - g), 1e-12 * bound + 1e-300, err_msg=str(k))
        _, G = RR.gram(loss, f_scale, r, tan, w)
        d = np.sqrt(np.diag(G))
        np.testing.assert_array_less(np.abs(jtj[j, :k, :k] - G), 1e-12 * np.outer(d, d) + 1e-300, err_msg=str(k))


# ---- 3. FD fits land where a robust scipy BFGS does -----------------------------------------------------
@pytest.mark.parametrize("loss", RR.ROBUST)
def test_robust_fit_lands_where_a_robust_scipy_bfgs_does(eng, golden, test_data, loss):
    checked = 0
    for case in golden["cases"]:
        calls = case["minimize_calls"][:case["R"]]
        if case["idx_remove"] or not calls or case["dtype"] != "float64":
            continue
        expr, k = vectorised.skeleton_string(case["tokens"], test_data.id2word)
        if k == 0:
            continue
        X, y = _case_tensors(case)
        Xn, yn = X[0].cpu().numpy(), y.cpu().numpy()
        f_scale = 0.1 * float(np.std(yn)) + 1e-3
        scale = 1.0 / float(yn.mean()) if case["norm"] == "NMSE" else 1.0
        eng.set_points(X[0], y, dtypes=(fitter.F64,), n_vars=10, loss=(loss, f_scale))
        eng.set_programs([compile_skeleton(expr, k, VARS)])
        x0 = np.array([c["x0"] for c in calls])
        res = eng.fit([0] * len(calls), list(range(len(calls))), x0, fitter.default_opts(grad_mode=FD, loss_scale=scale))
        dev = float(np.nanmin(res.loss.cpu().numpy()))
        cs = sp.symbols(f"c0:{k}")
        f = sp.lambdify([cs, sp.symbols("x_1:11")], sp.sympify(expr, locals={f"c{i}": cs[i] for i in range(k)}),
                        "numpy")

        def obj(c):
            with np.errstate(all="ignore"):
                r = f(c, [Xn[:, j] for j in range(10)]) - yn
                v = scale * np.mean(RR.terms(loss, f_scale, np.broadcast_to(r, yn.shape))[0])
            return v if np.isfinite(v) else 1e6

        ref = min(scipy.optimize.minimize(obj, s, method="BFGS").fun for s in x0)
        assert abs(dev - ref) <= 1e-6 * max(1.0, abs(ref)) + 1e-9, (case["name"], dev, ref)
        checked += 1
    assert checked >= 5, checked


# ---- 4. outliers ---------------------------------------------------------------------------------------
def _outlier_data(seed=3, n=400):
    rng = np.random.RandomState(seed)
    x = rng.uniform(0.2, 2.0, n)
    c_true = np.array([1.3, 0.8])
    y = c_true[0] * np.exp(c_true[1] * x) + rng.normal(size=n) * 0.05
    bad = rng.choice(n, n // 12, replace=False)       # 8 % of the points displaced by +10
    y[bad] += 10.0
    X = np.zeros((n, 10))
    X[:, 0] = x
    return X, y, c_true


def test_robust_bfgs_batch_recovers_the_constants_and_matches_least_squares(test_data):
    X, y, c_true = _outlier_data()
    toks = [test_data.word2id[t] for t in ("S", "mul", "c", "exp", "mul", "c", "x_1", "F")]
    cfg = make_cfg(4, grad_mode="dual")
    x0 = np.random.RandomState(1).uniform(0.5, 1.5, (4, 2))
    Xt, yt = torch.from_numpy(X[None]).cuda(), torch.from_numpy(y).cuda()
    lin = vbfgs.bfgs_batch([toks], Xt, yt, cfg, test_data, x0=[x0])[0]
    assert np.max(np.abs(np.asarray(lin[1]) / c_true - 1)) > 0.05          # linear is pulled off
    for loss in ("soft_l1", "huber", "cauchy"):
        fit = vbfgs.bfgs_batch([toks], Xt, yt, cfg, test_data, x0=[x0], loss=loss, f_scale=0.1)[0]
        c = np.asarray(fit[1], dtype=np.float64)
        assert np.max(np.abs(c / c_true - 1)) < 0.02, (loss, c)
        best = min((scipy.optimize.least_squares(lambda p: p[0] * np.exp(p[1] * X[:, 0]) - y, s, loss=loss,
                                                 f_scale=0.1, xtol=1e-15, ftol=1e-15, gtol=1e-15) for s in x0),
                   key=lambda r: r.cost)
        np.testing.assert_allclose(c, best.x, rtol=1e-4, err_msg=loss)
        assert abs(fit[2] - 2 * best.cost / len(y)) <= 1e-6 * 2 * best.cost / len(y)   # the robust mean cost


def test_refine_hypotheses_ranks_the_true_skeleton_first_under_a_robust_loss(test_data):
    rng = np.random.RandomState(3)
    n = 400
    x = rng.uniform(0.2, 2.0, n)
    y = 2.0 * x + 1.0 + rng.normal(size=n) * 0.05
    y[np.argsort(x)[-30:]] += 8.0                   # the largest x displaced upwards: a parabola fits better
    X = np.zeros((1, n, 10))
    X[0, :, 0] = x
    w2i = test_data.word2id
    true = [w2i[t] for t in ("S", "add", "mul", "c", "x_1", "c", "F")]
    quad = [w2i[t] for t in ("S", "add", "mul", "c", "mul", "x_1", "x_1", "c", "F")]
    hyps = [(-0.1, quad), (-0.2, true)]
    Xt, yt = torch.from_numpy(X).cuda(), torch.from_numpy(y).cuda().reshape(1, -1, 1)
    cfg = make_cfg(4, grad_mode="dual")
    x0 = [np.random.RandomState(2).uniform(0.5, 1.5, (4, 2))] * 2
    lin = refine_hypotheses(hyps, Xt, yt, cfg, test_data, x0=x0)
    assert list(lin["best_token"][0]) == quad
    for loss in ("soft_l1", "cauchy"):
        rob = refine_hypotheses(hyps, Xt, yt, cfg, test_data, x0=x0, loss=loss, f_scale=0.1)
        assert list(rob["best_token"][0]) == true, loss


# ---- 5. covariances: curve_fit's formula on the exact Jacobian ---------------------------------------------
SKEL = "((c0)*(exp(((c1)*(x_1)))))"


@pytest.mark.parametrize("loss", RR.ROBUST)
@pytest.mark.parametrize("absolute", [False, True])
@pytest.mark.parametrize("weighted", [False, True])
def test_robust_covariances_match_the_exact_jacobian_and_curve_fit(loss, absolute, weighted):
    X, y, c_true = _outlier_data(5, 200)
    sigma = np.random.RandomState(4).uniform(0.5, 2.0, len(y)) if weighted else None
    f = (lambda x, a, b: a * np.exp(b * x))
    popt, pcov = scipy.optimize.curve_fit(f, X[:, 0], y, p0=c_true, sigma=sigma, absolute_sigma=absolute, loss=loss,
                                          f_scale=0.1, method="trf")
    cv = uncertainty.covariances([("", list(popt), 0.0, SKEL)], torch.from_numpy(X), torch.from_numpy(y),
                                 sigma=sigma, absolute_sigma=absolute, loss=loss, f_scale=0.1)[0]
    assert cv.loss == loss and cv.f_scale == 0.1
    r, J = exact(SKEL, 2, X, y, popt)
    w = None if sigma is None else 1.0 / sigma ** 2
    rss, G = RR.gram(loss, 0.1, r, J, w)
    np.testing.assert_allclose(cv.rss, rss, rtol=1e-12)
    np.testing.assert_allclose(cv.jtj, G, rtol=1e-11)
    want = np.linalg.inv(G) * (1.0 if absolute else rss / (len(y) - 2))
    np.testing.assert_allclose(cv.cov, want, rtol=1e-9)
    np.testing.assert_allclose(cv.cov, pcov, rtol=1e-4)


# ---- 6. batch independence ----------------------------------------------------------------------------
def test_robust_eval_and_gram_do_not_depend_on_the_batch(eng):
    ks, progs = _programs()
    X, y = _points(50_001, 12)
    y[::17] += 20.0
    eng.set_points(torch.from_numpy(X), torch.from_numpy(y), dtypes=(fitter.F64,), n_vars=10, w=_w(50_001, 3),
                   loss=("cauchy", 0.5))
    eng.set_programs(progs)
    consts = np.random.RandomState(13).uniform(0.5, 1.5, size=(len(ks), max(ks)))
    rss_all, jtj_all = (t.cpu().numpy() for t in eng.gram(np.arange(len(ks)), consts))
    lo_all, gr_all = (t.cpu().numpy() for t in eng.eval(np.arange(len(ks)), consts, grad=True))
    for j in (0, 3, len(ks) - 1):
        rss1, jtj1 = (t.cpu().numpy() for t in eng.gram([j], consts[j:j + 1]))
        assert rss1[0].tobytes() == rss_all[j].tobytes() and jtj1[0].tobytes() == jtj_all[j].tobytes()
        lo1, gr1 = (t.cpu().numpy() for t in eng.eval([j], consts[j:j + 1], grad=True))
        assert lo1[0].tobytes() == lo_all[j].tobytes() and gr1[0].tobytes() == gr_all[j].tobytes()


# ---- 7. non-finite residuals ---------------------------------------------------------------------------
def test_a_candidate_that_is_not_real_gets_the_penalty_under_every_loss(eng):
    X, y = _points(5001, 14)
    X[:, 0] -= 1.0                                 # sqrt(x_1) is not real at about a third of the points
    p = compile_skeleton("((c0)*(sqrt(x_1)))", 1, VARS)
    want = None
    for loss in [None] + [(n, 0.5) for n in RR.ROBUST]:
        eng.set_points(torch.from_numpy(X), torch.from_numpy(y), dtypes=(fitter.F64,), n_vars=10, loss=loss)
        eng.set_programs([p])
        lo, _ = eng.eval([0], np.ones((1, 1)), grad=True)
        lo = float(lo.cpu().numpy()[0])
        assert not np.isfinite(lo) or lo >= 1e9, (loss, lo)
        want = lo if want is None else want
        assert (np.isnan(lo) and np.isnan(want)) or lo == want, (loss, lo, want)


def test_an_overflowing_z_gives_scipys_values(eng):
    X, y = _points(1000, 15)
    p = compile_skeleton("(c0)", 1, VARS)
    for loss in RR.ROBUST:
        eng.set_points(torch.from_numpy(X), torch.from_numpy(np.zeros(1000)), dtypes=(fitter.F64,), n_vars=10,
                       loss=(loss, 3.0))
        eng.set_programs([p])
        lo, gr = eng.eval([0], np.full((1, 1), 1e200), grad=True)      # r = 1e200: z = 1e400 / 9 = inf
        rss, jtj = eng.gram([0], np.full((1, 1), 1e200))
        lo, gr, rss, jtj = (float(t.cpu().numpy().reshape(-1)[0]) for t in (lo, gr, rss, jtj))
        want = 9.0 * (np.pi / 2 if loss == "arctan" else np.inf)
        assert lo == pytest.approx(want, rel=1e-12) and rss == pytest.approx(1000 * want, rel=1e-12), (loss, lo, rss)
        assert gr == 0.0, (loss, gr)
        assert jtj == 1000 * RR.EPS, (loss, jtj)


# ---- 8. other engines carry the loss -------------------------------------------------------------------
def test_two_engines_and_devices_carry_the_loss(golden, test_data):
    toks, X, y, cfg, td, x0 = _beam_jobs(golden, test_data, n_beams=1)[-1]
    hyps = [(-0.1 * i, t) for i, t in enumerate(toks)]
    devs = [[0, 0]] + ([[0, 1]] if torch.cuda.device_count() > 1 else [])
    outs = {}
    for loss in ("linear", "soft_l1"):
        for dv in [None] + devs:
            cfg.bfgs.devices = dv
            out = refine_hypotheses(hyps, X, y.reshape(1, -1, 1), cfg, td, x0=x0, loss=loss, f_scale=0.05)
            outs[(loss, str(dv))] = ([str(p) for p in out["all_bfgs_preds"]], np.asarray(out["all_bfgs_loss"]).tobytes())
    cfg.bfgs.devices = None
    for dv in devs:
        assert outs[("soft_l1", str(dv))] == outs[("soft_l1", "None")], dv
        assert outs[("linear", str(dv))] == outs[("linear", "None")], dv
    assert outs[("soft_l1", "None")] != outs[("linear", "None")]


def test_bfgs_batch_with_huber_at_a_wide_scale_is_the_linear_fit(golden, test_data):
    for toks, X, y, cfg, td, x0 in _beam_jobs(golden, test_data, n_beams=2):
        a = vbfgs.bfgs_batch(toks, X, y, cfg, td, x0=x0)
        b = vbfgs.bfgs_batch(toks, X, y, cfg, td, x0=x0, loss="huber", f_scale=WIDE)
        assert _canon(a) == _canon(b)
