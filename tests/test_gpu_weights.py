"""Weighted fits on the GPU: w = 1 reproduces the unweighted fit, evaluation and Gram bit for bit on every
kernel path; random weights against the host interpreter's reference and a weighted scipy BFGS; the
curve_fit sigma conventions of ``covariances`` and ``predict`` against the exact Jacobian, curve_fit and
their coverage."""
import ctypes

import numpy as np
import pytest
import scipy.optimize
import scipy.stats
import sympy as sp
import torch

import _interp_ref as R
import bench
from _gram_ref import VARS, exact
from conftest import make_cfg
from oracle import vectorised
from src.visymre import uncertainty
from src.visymre.architectures import bfgs as vbfgs
from src.visymre.architectures.refine import refine_hypotheses
from src.visymre.engine import fitter, isa
from src.visymre.engine.compiler import compile_skeleton
from src.visymre.workloads import generator as wg
from test_gpu_fit import _case_tensors
from test_gpu_uncertainty import _canon, _skeleton

pytestmark = pytest.mark.gpu
WIDTHS = [0, 1, 2, 3, 4, 5, 6, 7, 8, 12, 16]
FD, DUAL = isa.GRAD_MODE["VSR_GRAD_FD"], isa.GRAD_MODE["VSR_GRAD_DUAL"]
DT = {np.float64: fitter.F64, np.float32: fitter.F32}


@pytest.fixture(scope="module")
def eng():
    return fitter.Engine("cuda:0")


def _points(n, seed, dtype=np.float64):
    rng = np.random.RandomState(seed)
    X = rng.uniform(0.3, 2.0, size=(n, 10)).astype(dtype)
    y = rng.normal(size=n).astype(dtype)
    return X, y


def _programs():
    ks = sorted({k for K in WIDTHS for k in (K, max(K - 1, 0))})
    return ks, [compile_skeleton(_skeleton(k), k, VARS) for k in ks]


def _set(eng, X, y, dt, w=None, offset=0):
    """Points (and weights) of slot dt through vsr_set_points / vsr_set_weights; offset > 0 starts every
    column `offset` elements into its buffer, so that no column is 16-byte aligned (no TMA copies)."""
    td = torch.float64 if dt == fitter.F64 else torch.float32
    n = X.shape[0]
    ld = n + 4 + offset
    Xc = torch.zeros((10, ld), dtype=td, device=eng.device)
    Xc[:, offset:offset + n] = torch.from_numpy(X.T.copy()).to(td)
    yc = torch.zeros(n + offset, dtype=td, device=eng.device)
    yc[offset:] = torch.from_numpy(y).to(td)
    base = Xc.data_ptr() + offset * Xc.element_size()
    keep = [Xc, yc]
    eng._check(eng.lib.vsr_set_points(eng._h, ctypes.c_void_p(base), ctypes.c_void_p(yc[offset:].data_ptr()),
                                      n, ld, 10, dt))
    if w is not None:
        wc = torch.zeros(n + offset, dtype=td, device=eng.device)
        wc[offset:] = torch.from_numpy(np.asarray(w)).to(td)
        keep.append(wc)
        eng._check(eng.lib.vsr_set_weights(eng._h, ctypes.c_void_p(wc[offset:].data_ptr()), n, dt))
    eng._points[dt] = (Xc, yc)
    eng.n_vars = 10
    eng._keep = keep
    return keep


def _fit_all(eng, ks, mode, dtype, maxiter):
    rng = np.random.RandomState(11)
    R_ = 3
    x0 = rng.uniform(0.5, 1.5, size=(len(ks) * R_, max(ks)))
    dt = DT[dtype]
    opts = fitter.default_opts(grad_mode=mode, eval_dtype=dt, score_dtype=dt, maxiter_per_k=maxiter)
    res = eng.fit(np.repeat(np.arange(len(ks)), R_), np.arange(len(ks) * R_), x0, opts)
    torch.cuda.synchronize()
    return [t.cpu().numpy().tobytes() for t in (res.consts, res.lastx, res.loss, res.final_mse, res.info)]


# ---- w = 1 is the unweighted result, bit for bit ----------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("n,offset", [(3001, 0), (3001, 1), (600_001, 0), (600_001, 1)])
def test_unit_weights_give_the_unweighted_eval_and_fit_bit_for_bit(eng, dtype, n, offset):
    """n = 3001: resident fit slices and eval_kernel; n = 600 001: streamed fp64 slices and the shared
    tiles of eval_tile_kernel.  offset 1: unaligned columns (coalesced loads instead of TMA)."""
    ks, progs = _programs()
    X, y = _points(n, 5, dtype)
    dt = DT[dtype]
    eng.set_programs(progs)
    rng = np.random.RandomState(3)
    consts = rng.uniform(0.5, 1.5, size=(len(ks), max(ks)))
    got = {}
    for w in (None, np.ones(n)):
        _set(eng, X, y, dt, w, offset)
        loss, grad = eng.eval(np.arange(len(ks)), consts, dtype=dt, grad=True)
        out = [loss.cpu().numpy().tobytes(), grad.cpu().numpy().tobytes()]
        for mode in (DUAL, FD):
            out += _fit_all(eng, ks, mode, dtype, 8 if n > 10_000 else 40)
        got[w is None] = out
    assert got[True] == got[False]


def test_unit_weights_give_the_unweighted_gram_bit_for_bit(eng):
    ks, progs = _programs()
    X, y = _points(70_001, 6)
    eng.set_programs(progs)
    consts = np.random.RandomState(4).uniform(0.5, 1.5, size=(len(ks), max(ks)))
    got = []
    for w in (None, np.ones(70_001)):
        eng.set_points(torch.from_numpy(X), torch.from_numpy(y), dtypes=(fitter.F64,), n_vars=10, w=w)
        rss, jtj = eng.gram(np.arange(len(ks)), consts)
        got.append((rss.cpu().numpy().tobytes(), jtj.cpu().numpy().tobytes()))
    assert got[0] == got[1]


def _beam_jobs(golden, test_data, n_beams=4):
    jobs = []
    for case in golden["cases"]:
        if case["idx_remove"]:
            continue                      # sigma cannot be combined with idx_remove
        X, y = _case_tensors(case)
        cfg = make_cfg(case["R"], case["norm"], False, grad_mode="dual")
        calls = case["minimize_calls"][:case["R"]]
        x0 = [np.array([c["x0"] for c in calls])] if calls else None
        jobs.append(([case["tokens"]], X, y, cfg, test_data, x0))
    td = wg.make_test_data()
    for b in bench.make_workload(n_beams, 10_000, 64, 10):
        X = torch.from_numpy(np.ascontiguousarray(b.X[None])).cuda()
        y = torch.from_numpy(np.ascontiguousarray(b.y)).cuda()
        jobs.append((list(b.tokens), X, y, wg.make_cfg(10, 64, grad_mode="dual"), td, b.x0))
    return jobs


def test_bfgs_batch_with_unit_sigma_is_the_unweighted_fit(golden, test_data):
    refits = 0
    for toks, X, y, cfg, td, x0 in _beam_jobs(golden, test_data):
        a = vbfgs.bfgs_batch(toks, X, y, cfg, td, x0=x0)
        b = vbfgs.bfgs_batch(toks, X, y, cfg, td, x0=x0, sigma=torch.ones(X.shape[1], device=X.device))
        refits += "prune_fit" in vbfgs.LAST_TIMING
        assert _canon(a) == _canon(b)
    assert refits > 0                     # the prune re-fit ran


def test_two_engines_on_one_gpu_carry_the_weights(golden, test_data):
    hyps, cases = [], 0
    for toks, X, y, cfg, td, x0 in _beam_jobs(golden, test_data, n_beams=1)[-1:]:
        sigma = np.exp(np.random.RandomState(2).uniform(np.log(0.1), np.log(10.0), X.shape[1]))
        hyps = [(-0.1 * i, t) for i, t in enumerate(toks)]
        outs = []
        for dv, s in ((None, None), ([0, 0], np.ones(X.shape[1])), (None, sigma), ([0, 0], sigma)):
            cfg.bfgs.devices = dv
            out = refine_hypotheses(hyps, X, y.reshape(1, -1, 1), cfg, td, x0=x0, sigma=s)
            outs.append(([str(p) for p in out["all_bfgs_preds"]], np.asarray(out["all_bfgs_loss"]).tobytes()))
        cfg.bfgs.devices = None
        assert outs[0] == outs[1] and outs[2] == outs[3]
        assert outs[0] != outs[2]
        cases += 1
    assert cases == 1


# ---- random weights against the host reference -------------------------------------------------------
def _random_w(n, seed):
    return np.exp(np.random.RandomState(seed).uniform(np.log(1e-6), np.log(1e6), n))


def test_weighted_eval_and_gram_match_the_host_reference_at_every_width(eng, hostsim):
    ks, progs = _programs()
    n = 20_001
    X, y = _points(n, 7)
    w = _random_w(n, 8)
    consts = np.random.RandomState(9).uniform(0.5, 1.5, size=(len(ks), max(ks)))
    eng.set_points(torch.from_numpy(X), torch.from_numpy(y), dtypes=(fitter.F64,), n_vars=10, w=w)
    eng.set_programs(progs)
    loss, grad = eng.eval(np.arange(len(ks)), consts, dtype=fitter.F64, grad=True)
    rss, jtj = eng.gram(np.arange(len(ks)), consts)
    loss, grad, rss, jtj = (t.cpu().numpy() for t in (loss, grad, rss, jtj))
    for j, (k, p) in enumerate(zip(ks, progs)):
        val, tan = R.host_duals(hostsim, p.insns, p.imms, consts[j, :k], X, next(K for K in WIDTHS if K >= k))
        tan = tan[:, :k]
        r = val - y
        want_loss = np.sum(w * r * r) / n
        assert abs(loss[j] - want_loss) <= 1e-12 * want_loss, (k, loss[j], want_loss)
        assert abs(rss[j] - n * want_loss) <= 1e-12 * n * want_loss
        if k == 0:
            continue
        g = 2.0 * ((w * r) @ tan) / n
        scale = 2.0 * np.sqrt(want_loss * np.sum(w[:, None] * tan * tan, axis=0) / n)   # Cauchy-Schwarz bound
        np.testing.assert_array_less(np.abs(grad[j, :k] - g), 1e-12 * scale + 1e-300, err_msg=str(k))
        G = tan.T @ (w[:, None] * tan)
        d = np.sqrt(np.diag(G))
        np.testing.assert_array_less(np.abs(jtj[j, :k, :k] - G), 1e-12 * np.outer(d, d) + 1e-300, err_msg=str(k))


def test_weighted_gram_does_not_depend_on_the_batch(eng):
    ks, progs = _programs()
    X, y = _points(50_001, 12)
    eng.set_points(torch.from_numpy(X), torch.from_numpy(y), dtypes=(fitter.F64,), n_vars=10, w=_random_w(50_001, 3))
    eng.set_programs(progs)
    consts = np.random.RandomState(13).uniform(0.5, 1.5, size=(len(ks), max(ks)))
    rss_all, jtj_all = (t.cpu().numpy() for t in eng.gram(np.arange(len(ks)), consts))
    for j in (0, 3, len(ks) - 1):
        rss1, jtj1 = (t.cpu().numpy() for t in eng.gram([j], consts[j:j + 1]))
        assert rss1[0].tobytes() == rss_all[j].tobytes()
        assert jtj1[0].tobytes() == jtj_all[j].tobytes()


def test_weighted_fit_lands_where_a_weighted_scipy_bfgs_does(eng, golden, test_data):
    """FD mode restates scipy's default BFGS (2-point gradient): from the same x0 the best loss over the
    restarts agrees within the parity bound of the unweighted fit."""
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
        w = np.exp(np.random.RandomState(checked).uniform(np.log(1e-2), np.log(1e2), len(yn)))
        scale = 1.0 / float(yn.mean()) if case["norm"] == "NMSE" else 1.0
        eng.set_points(X[0], y, dtypes=(fitter.F64,), n_vars=10, w=w)
        eng.set_programs([compile_skeleton(expr, k, VARS)])
        x0 = np.array([c["x0"] for c in calls])
        res = eng.fit([0] * len(calls), list(range(len(calls))), x0, fitter.default_opts(grad_mode=FD, loss_scale=scale))
        dev = float(np.nanmin(res.loss.cpu().numpy()))
        cs = sp.symbols(f"c0:{k}")
        f = sp.lambdify([cs, sp.symbols("x_1:11")], sp.sympify(expr, locals={f"c{i}": cs[i] for i in range(k)}),
                        "numpy")

        def obj(c):
            with np.errstate(all="ignore"):
                v = scale * np.mean(w * (f(c, [Xn[:, j] for j in range(10)]) - yn) ** 2)
            return v if np.isfinite(v) else 1e6

        ref = min(scipy.optimize.minimize(obj, s, method="BFGS").fun for s in x0)
        assert abs(dev - ref) <= 1e-6 * max(1.0, abs(ref)) + 1e-9, (case["name"], dev, ref)
        checked += 1
    assert checked >= 5, checked


# ---- statistics ------------------------------------------------------------------------------------
def _hetero(seed, n=200):
    rng = np.random.RandomState(seed)
    x = rng.uniform(0.2, 2.0, n)
    sigma = rng.uniform(0.05, 0.5, n) * (1 + x)
    c_true = np.array([1.3, 0.8])
    y = c_true[0] * np.exp(c_true[1] * x) + rng.normal(size=n) * sigma
    X = np.zeros((n, 10))
    X[:, 0] = x
    return X, y, sigma, c_true


SKEL = "((c0)*(exp(((c1)*(x_1)))))"


def _wfit(X, y, sigma, c0):
    popt, pcov = scipy.optimize.curve_fit(lambda x, a, b: a * np.exp(b * x), X[:, 0], y, p0=c0, sigma=sigma,
                                          absolute_sigma=True)
    return popt, pcov


@pytest.mark.parametrize("absolute", [False, True])
def test_covariances_with_sigma_match_the_exact_jacobian_and_curve_fit(absolute):
    X, y, sigma, c_true = _hetero(1)
    popt, _ = _wfit(X, y, sigma, c_true)
    fit = ("", list(popt), 0.0, SKEL)
    cv = uncertainty.covariances([fit], torch.from_numpy(X), torch.from_numpy(y), sigma=sigma,
                                 absolute_sigma=absolute)[0]
    assert cv.absolute_sigma == absolute
    r, J = exact(SKEL, 2, X, y, popt)
    w = 1.0 / sigma ** 2
    G = J.T @ (w[:, None] * J)
    want = np.linalg.inv(G) * (1.0 if absolute else float(w @ (r * r)) / (len(y) - 2))
    np.testing.assert_allclose(cv.cov, want, rtol=1e-9)
    _, pcov = scipy.optimize.curve_fit(lambda x, a, b: a * np.exp(b * x), X[:, 0], y, p0=popt, sigma=sigma,
                                       absolute_sigma=absolute)
    np.testing.assert_allclose(cv.cov, pcov, rtol=1e-4)


def test_absolute_sigma_intervals_and_prediction_bands_cover_at_the_stated_rate(test_data):
    cfg = make_cfg(4, grad_mode="dual")
    toks = [test_data.word2id[t] for t in ("S", "mul", "c", "exp", "mul", "c", "x_1", "F")]
    hit_c, hit_pi, n_pi, runs = 0, 0, 0, 200
    for seed in range(runs):
        X, y, sigma, c_true = _hetero(100 + seed)
        Xt = torch.from_numpy(X[None]).cuda()
        yt = torch.from_numpy(y).cuda()
        x0 = [np.tile(c_true, (4, 1)) + np.random.RandomState(seed).normal(0, 0.05, (4, 2))]
        fit = vbfgs.bfgs_batch([toks], Xt, yt, cfg, test_data, x0=x0, sigma=torch.from_numpy(sigma).cuda())[0]
        cv = uncertainty.covariances([fit], Xt, yt, sigma=sigma, absolute_sigma=True)[0]
        c = np.asarray(fit[1], dtype=np.float64)
        hit_c += int(abs(c[1] - c_true[1]) <= scipy.stats.norm.ppf(0.975) * cv.stderr[1])
        rng = np.random.RandomState(10_000 + seed)
        Xn = np.zeros((20, 10))
        Xn[:, 0] = rng.uniform(0.2, 2.0, 20)
        sn = rng.uniform(0.05, 0.5, 20) * (1 + Xn[:, 0])
        y_new = c_true[0] * np.exp(c_true[1] * Xn[:, 0]) + rng.normal(size=20) * sn
        p = uncertainty.predict([fit], torch.from_numpy(Xn), covs=[cv], sigma_new=torch.from_numpy(sn))[0]
        lo, hi = p.pi_low.cpu().numpy(), p.pi_high.cpu().numpy()
        hit_pi += int(((y_new >= lo) & (y_new <= hi)).sum())
        n_pi += 20
    lo_c, hi_c = scipy.stats.binom.interval(0.999, runs, 0.95)
    assert lo_c <= hit_c <= hi_c, hit_c
    lo_p, hi_p = scipy.stats.binom.interval(0.999, n_pi, 0.95)
    # the points of one data set share its fitted curve: allow the spread of 200 clusters of 20
    assert lo_p - 40 <= hit_pi <= hi_p + 40, (hit_pi, n_pi)
