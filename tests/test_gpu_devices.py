"""cfg.bfgs.devices on the GPU: one process deals a beam's runs over several engines and returns the dict
of the one-engine fit, bit for bit.  ``devices=[0, 0]`` puts two engines on one GPU, which takes the whole
path -- dealing, points shared, programs on every engine, fits in flight together, records merged -- on a
single B200; ``devices="all"`` needs two GPUs."""
import numpy as np
import pytest
import torch

import bench
from conftest import make_cfg
from src.visymre.architectures import bfgs as vbfgs
from src.visymre.architectures.refine import refine_hypotheses
from src.visymre.engine import fitter, sharding
from src.visymre.workloads import generator as wg
from test_gpu_fit import _case_tensors

pytestmark = pytest.mark.gpu
SETTINGS = [("dual", "fp64"), ("fd", "fp64"), ("dual", "fp32")]


def _bits(v):
    a = np.asarray(v)
    return a.dtype.str, a.tobytes()


def _canon(out):
    """The dict with every string read and every loss as (dtype, bytes): equal means bit for bit."""
    return {"pred_target": [int(t) for t in out["pred_target"]],
            "all_bfgs_preds": [str(s) for s in out["all_bfgs_preds"]],
            "all_bfgs_loss": [_bits(v) for v in out["all_bfgs_loss"]],
            "best_bfgs_preds": [None if s is None else str(s) for s in out["best_bfgs_preds"]],
            "best_bfgs_loss": [_bits(v) for v in out["best_bfgs_loss"]],
            "best_token": [None if t is None else [int(x) for x in t] for t in out["best_token"]]}


def _both(hyps, X, y, cfg, td, x0, devices):
    """(one engine, ``devices``) outputs of refine_hypotheses on the same inputs and starting points."""
    outs = []
    for dv in (None, devices):
        cfg.bfgs.devices = dv
        np.random.seed(7)                  # candidates without given starting points draw them here
        outs.append(_canon(refine_hypotheses(hyps, X, y, cfg, td, x0=x0)))
    cfg.bfgs.devices = None
    return outs


def _diff(a, b):
    return {k: (a[k], b[k]) for k in a if a[k] != b[k]}


@pytest.mark.parametrize("mode,precision", SETTINGS)
def test_two_engines_on_one_gpu_equal_one_engine_on_the_golden_cases(golden, test_data, mode, precision):
    n = 0
    for case in golden["cases"]:
        X, y = _case_tensors(case)
        cfg = make_cfg(case["R"], case["norm"], case["idx_remove"], grad_mode=mode, precision=precision)
        calls = case["minimize_calls"][:case["R"]]
        x0 = [np.array([c["x0"] for c in calls])] if calls else None
        one, two = _both([(-0.1, case["tokens"])], X, y.reshape(1, -1, 1), cfg, test_data, x0, [0, 0])
        assert one == two, (case["name"], _diff(one, two))
        n += 1
    assert n == 17


@pytest.fixture(scope="module")
def bench_beams():
    return bench.make_workload(4, 10_000, 64, 10)


@pytest.mark.parametrize("mode,precision", SETTINGS)
def test_two_engines_on_one_gpu_equal_one_engine_on_bench_beams(bench_beams, mode, precision):
    td = wg.make_test_data()
    for b in bench_beams:
        X = torch.from_numpy(np.ascontiguousarray(b.X[None])).cuda()
        y = torch.from_numpy(np.ascontiguousarray(b.y)).reshape(1, -1, 1).cuda()
        hyps = [(-float(j), t) for j, t in enumerate(b.tokens)]
        cfg = wg.make_cfg(10, 64, grad_mode=mode, precision=precision)
        one, two = _both(hyps, X, y, cfg, td, b.x0, [0, 0])
        assert len(one["all_bfgs_loss"]) > 32
        assert one == two, (b.name, _diff(one, two))


def _tok(test_data, words):
    w2i = test_data.word2id
    return [w2i["S"]] + [w2i[w] for w in words.split()] + [w2i["F"]]


def test_prune_refit_and_the_empty_conventions_with_devices(test_data):
    rng = np.random.RandomState(11)
    X = torch.zeros((1, 300, 10), dtype=torch.float64)
    X[0, :, 0] = torch.tensor(rng.uniform(-2, 2, 300))
    y = (2.5 * X[0, :, 0]).reshape(1, -1, 1)
    cfg = make_cfg(4, grad_mode="dual")
    # c0 + c1*x_1 on y = 2.5 x_1: c0 fits to ~0, is pruned and the rest is fitted again on the home engine
    hyps = [(-0.1, _tok(test_data, "add c mul c x_1")), (-0.2, _tok(test_data, "mul c sin x_1")),
            (-0.3, _tok(test_data, "mul c x_1"))]
    x0 = [rng.randn(4, 2) * 3, rng.randn(4, 1) * 3, rng.randn(4, 1) * 3]
    cfg.bfgs.devices = [0, 0]
    out = refine_hypotheses(hyps, X.cuda(), y.cuda(), cfg, test_data, x0=x0)
    assert "prune_fit" in vbfgs.LAST_TIMING
    assert out["best_bfgs_loss"][0] < 1e-20
    one, two = _both(hyps, X.cuda(), y.cuda(), cfg, test_data, x0, [0, 0])
    assert one == two, _diff(one, two)
    # rows dropped by idx_remove: the fit stays on the home engine, every score is 1e9 (bfgs.py:130-131)
    Xr = X.clone()
    Xr[0, :9, 0] = 500.0
    cfg_r = make_cfg(2, idx_remove=True, grad_mode="fd")
    one, two = _both(hyps[:1], Xr.cuda(), y.cuda(), cfg_r, test_data, [x0[0][:2]], [0, 0])
    assert one == two and two["best_bfgs_loss"] == [_bits(1e9)], _diff(one, two)
    # nothing valid (the fallback fails too): [None] / [nan]
    cfg.bfgs.devices = [0, 0]
    out = refine_hypotheses([(-1.0, _tok(test_data, "add c"))], X.cuda(), y.cuda(), cfg, test_data)
    assert out["best_bfgs_preds"] == [None] and np.isnan(out["best_bfgs_loss"][0]) and out["all_bfgs_preds"] == []
    # every candidate scores nan (sqrt of negative points): [None] / [nan]
    Xn = X.clone()
    Xn[0, :, 0] = -1.0 - Xn[0, :, 0].abs()
    out = refine_hypotheses([(-0.1, _tok(test_data, "mul c sqrt x_1"))], Xn.cuda(), y.cuda(), cfg, test_data,
                            x0=[np.ones((4, 1))])
    assert out["best_bfgs_preds"] == [None] and np.isnan(out["best_bfgs_loss"][0])
    assert len(out["all_bfgs_preds"]) == 1


def test_devices_unset_or_none_is_the_one_engine_path(test_data, monkeypatch):
    """No engine beyond today's, no ``fit_devices``, the same launches: unset, None and one device."""
    beams, td = wg.feynman_beams(n_points=2000, n_cand=32, n_restarts=4, limit=1)
    b = beams[0]
    X = torch.from_numpy(np.ascontiguousarray(b.X[None])).cuda()
    y = torch.from_numpy(np.ascontiguousarray(b.y)).reshape(1, -1, 1).cuda()
    hyps = [(-float(j), t) for j, t in enumerate(b.tokens)]
    x0 = b.x0
    cfg = wg.make_cfg(4, 32)
    refine_hypotheses(hyps, X, y, cfg, td, x0=x0)        # compiles every skeleton: one stage from here on
    home = fitter.get_engine(0)

    def launches():
        return home.launches + sum(e.launches for k, e in fitter._SIDE.items() if k[0] == id(home))

    def refuse(*a, **k):
        raise AssertionError("fit_devices called")
    monkeypatch.setattr(sharding, "fit_devices", refuse)
    counts, outs = [], []
    for value in ("unset", None, [0]):
        if value != "unset":
            cfg.bfgs.devices = value
        n0 = launches()
        outs.append(_canon(refine_hypotheses(hyps, X, y, cfg, td, x0=x0)))
        counts.append(launches() - n0)
    assert counts[0] > 0 and counts[0] == counts[1] == counts[2], counts
    assert outs[0] == outs[1] == outs[2]


def test_all_devices_equal_one_engine(golden, test_data, bench_beams):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    td = wg.make_test_data()
    for b in bench_beams[:2]:
        X = torch.from_numpy(np.ascontiguousarray(b.X[None])).cuda()
        y = torch.from_numpy(np.ascontiguousarray(b.y)).reshape(1, -1, 1).cuda()
        hyps = [(-float(j), t) for j, t in enumerate(b.tokens)]
        for mode, precision in SETTINGS:
            cfg = wg.make_cfg(10, 64, grad_mode=mode, precision=precision)
            one, many = _both(hyps, X, y, cfg, td, b.x0, "all")
            assert one == many, (b.name, mode, precision, _diff(one, many))
    case = next(c for c in golden["cases"] if c["name"] == "prune_small")
    X, yc = _case_tensors(case)
    cfg = make_cfg(case["R"], case["norm"], case["idx_remove"])
    x0 = [np.array([c["x0"] for c in case["minimize_calls"][:case["R"]]])]
    one, many = _both([(-0.1, case["tokens"])], X, yc.reshape(1, -1, 1), cfg, test_data, x0, "all")
    assert one == many, _diff(one, many)
