"""One process, several engines (cfg.bfgs.devices): the dealing and the merge of ``fit_devices`` on the
CPU, with engines that fill their share of the runs from a fixed table (the fit itself needs a GPU), and
the refusal of several devices in a process that has a torch.distributed process group."""
import numpy as np
import pytest
import torch
import torch.distributed as dist

from conftest import make_cfg
from src.visymre.architectures import bfgs as vbfgs
from src.visymre.architectures import refine
from src.visymre.engine import sharding
from src.visymre.engine.native import VsrError


class TableEngine:
    """Stands in for ``Engine``: ``fit`` writes the table's rows of the runs it is handed."""

    def __init__(self, fm, loss, consts):
        self.device = torch.device("cpu")
        self.fm, self.loss, self.consts = (torch.as_tensor(a, dtype=torch.float64) for a in (fm, loss, consts))
        self.calls = []

    def fit(self, run_prog, run_slot, x0, opts):
        assert len(run_slot) > 0                       # vsr_fit rejects an empty run list
        self.calls.append((np.asarray(run_prog), np.asarray(run_slot)))
        res = sharding.empty_result(int(x0.shape[0]), int(x0.shape[1]), self.device)
        s = torch.as_tensor(np.asarray(run_slot), dtype=torch.long)
        res.final_mse[s] = self.fm[s]
        res.loss[s] = self.loss[s]
        res.lastx[s] = self.consts[s]
        return res


def _table(C=23, R=8, kmax=3):
    """The scores of the gloo test of test_sharding.py (nan, an all-nan candidate, nan and +inf only),
    plus a tie and an all-+inf candidate."""
    rng = np.random.RandomState(3)
    fm = rng.rand(C * R)
    fm[rng.rand(C * R) < 0.25] = np.nan
    fm[2 * R:3 * R] = np.nan
    fm[4 * R:5 * R] = np.nan
    fm[4 * R + 3] = fm[4 * R + 6] = np.inf
    loss, consts = rng.rand(C * R), rng.rand(C * R, kmax)
    cost = rng.rand(C * R)
    fm[7 * R + 1] = fm[7 * R + 5] = 0.0              # a tie
    fm[9 * R:10 * R] = np.inf                         # every restart +inf
    return fm, loss, consts, cost


def _nanargmin(fm, C, R):
    return np.asarray([0 if np.all(np.isnan(fm[c * R:(c + 1) * R])) else int(np.nanargmin(fm[c * R:(c + 1) * R]))
                       for c in range(C)])


def _same(a, b):
    return a.shape == b.shape and bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())


@pytest.mark.parametrize("n_dev", [1, 2, 3, 8])
def test_fit_devices_equals_merge_records_of_the_same_records(n_dev):
    C, R, kmax = 23, 8, 3
    fm, loss, consts, cost = _table(C, R, kmax)
    engines = [TableEngine(fm, loss, consts) for _ in range(n_dev)]
    win, results = sharding.fit_devices(engines, [kmax] * C, R, np.zeros((C * R, kmax)), None, cost=cost)
    # what the ranks of the gloo test exchange, from the same dealing
    parts = sharding.partition_runs(cost, n_dev)
    recs = []
    for p in parts:
        mine = torch.zeros(C * R, dtype=torch.bool)
        mine[torch.as_tensor(p)] = True
        f = torch.full((C * R,), float("nan"), dtype=torch.float64)
        f[mine] = torch.as_tensor(fm)[mine]
        recs.append(sharding.local_best_records(f, torch.as_tensor(loss), torch.as_tensor(consts), C, R, mine))
    assert _same(win, sharding.merge_records(torch.stack(recs), R))
    # every engine fitted exactly its share, once
    for eng, p in zip(engines, parts):
        assert len(eng.calls) == 1
        run_prog, run_slot = eng.calls[0]
        assert np.array_equal(run_slot, p) and np.array_equal(run_prog, p // R)
    assert len(results) == n_dev
    # and that is np.nanargmin over all restarts, as one engine would pick
    want = _nanargmin(fm, C, R)
    assert np.array_equal(win[:, 1].numpy().astype(int), want)
    rows = np.arange(C) * R + want
    np.testing.assert_array_equal(win[:, 3:3 + kmax].numpy(), consts[rows])
    np.testing.assert_array_equal(win[:, 2].numpy(), loss[rows])
    np.testing.assert_array_equal(win[:, -1].numpy(), fm[rows])


@pytest.mark.parametrize("C,R,n_dev", [(1, 1, 2), (2, 1, 3), (1, 2, 8)])
def test_more_devices_than_runs(C, R, n_dev):
    """The engines without a run are not called; they report ``empty_result`` and lose every merge."""
    kmax = 2
    fm = np.arange(C * R, dtype=np.float64)[::-1] * 0.25
    loss = fm + 1.0
    consts = np.arange(C * R * kmax, dtype=np.float64).reshape(C * R, kmax)
    engines = [TableEngine(fm, loss, consts) for _ in range(n_dev)]
    win, results = sharding.fit_devices(engines, [kmax] * C, R, np.zeros((C * R, kmax)), None)
    assert sum(len(e.calls) for e in engines) == C * R
    assert all(len(e.calls) == 0 for e in engines[C * R:])
    for res in results[C * R:]:
        assert torch.isnan(res.final_mse).all() and (res.info == -1).all()
    want = _nanargmin(fm, C, R)
    rows = np.arange(C) * R + want
    assert np.array_equal(win[:, 1].numpy().astype(int), want)
    np.testing.assert_array_equal(win[:, 3:3 + kmax].numpy(), consts[rows])
    np.testing.assert_array_equal(win[:, -1].numpy(), fm[rows])


def test_an_engine_error_names_the_device_after_the_others_ran():
    fm, loss, consts, cost = _table()
    good, bad, last = (TableEngine(fm, loss, consts) for _ in range(3))

    def fails(*a, **k):
        raise RuntimeError("boom")
    bad.fit = fails
    with pytest.raises(VsrError, match="cpu.*boom"):
        sharding.fit_devices([good, bad, last], [3] * 23, 8, np.zeros((23 * 8, 3)), None, cost=cost)
    assert len(good.calls) == 1 and len(last.calls) == 1      # every other engine's fit was still enqueued


def test_devices_knob_values_without_a_gpu():
    assert vbfgs.resolve_devices(make_cfg(2)) is None
    assert vbfgs.resolve_devices(make_cfg(2, devices=None)) is None
    for bad in ("cpu", [], [0, "cpu"], ["nonsense"]):
        with pytest.raises(ValueError):
            vbfgs.resolve_devices(make_cfg(2, devices=bad))


@pytest.fixture
def gloo_group(tmp_path):
    dist.init_process_group("gloo", init_method=f"file://{tmp_path / 'pg'}", rank=0, world_size=1)
    try:
        yield
    finally:
        dist.destroy_process_group()


def test_several_devices_with_a_process_group_raise(gloo_group, test_data):
    w = test_data.word2id
    toks = [w["S"], w["add"], w["c"], w["x_1"], w["F"]]
    X = torch.zeros((1, 16, 10), dtype=torch.float64)
    y = torch.zeros((1, 16, 1), dtype=torch.float64)
    for devices in ([0, 1], [torch.device("cuda", 0), torch.device("cuda", 1)], ["cuda:0", "cuda:0"]):
        cfg = make_cfg(2, devices=devices)
        with pytest.raises(ValueError, match="process group"):
            vbfgs.resolve_devices(cfg)
        with pytest.raises(ValueError, match="process group"):
            vbfgs.bfgs_batch([toks], X, y, cfg, test_data)
        with pytest.raises(ValueError, match="process group"):
            refine.refine_hypotheses([(-0.1, toks)], X, y, cfg, test_data)
