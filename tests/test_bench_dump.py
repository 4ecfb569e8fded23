"""bench.py --dump-outputs: the fit's outputs as finite float .npy files, sampled to stay under the limit."""
import os
import sys

import numpy as np
import torch

from conftest import ROOT

sys.path.insert(0, ROOT)
import bench  # noqa: E402
from src.visymre.engine.fitter import FitResult  # noqa: E402

FIELDS = ("consts", "lastx", "loss", "final_mse")


def _result(n_runs, kmax=3):
    """Shaped like a real fit: NaN past each run's number of constants (all of them for k = 0, status
    255), NaN / inf scores where the expression is not real at the fitted point."""
    rng = np.random.RandomState(1)
    k = rng.randint(0, kmax + 1, n_runs)
    consts, lastx = rng.randn(n_runs, kmax), rng.randn(n_runs, kmax)
    for a in (consts, lastx):
        a[np.arange(kmax)[None, :] >= k[:, None]] = np.nan
    final_mse = rng.rand(n_runs)
    final_mse[rng.rand(n_runs) < 0.3] = np.nan
    final_mse[rng.rand(n_runs) < 0.05] = np.inf
    info = rng.randint(0, 300, (n_runs, 4)).astype(np.int32)
    info[k == 0, 0] = 255
    return FitResult(consts=torch.from_numpy(consts), lastx=torch.from_numpy(lastx), loss=torch.from_numpy(rng.rand(n_runs)),
                     final_mse=torch.from_numpy(final_mse), info=torch.from_numpy(info))


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def _decode(got, name):
    """The field as the fit returned it, NaN where the entry was not finite."""
    mask = got[f"{name}_finite"].astype(bool)
    a = np.full(mask.shape, np.nan)
    a[mask] = got[name]
    return a


def test_every_field_is_written_finite_and_exactly(tmp_path):
    res = _result(40)
    bench.dump_outputs(str(tmp_path), None, res)
    got = _load(tmp_path)
    assert sorted(got) == sorted(["info"] + [n for f in FIELDS for n in (f, f + "_finite")])
    for name, a in got.items():
        assert a.dtype in (np.float32, np.float64) and np.isfinite(a).all(), name
    np.testing.assert_array_equal(got["info"], res.info.numpy())
    for f in FIELDS:
        want = getattr(res, f).numpy()
        np.testing.assert_array_equal(got[f"{f}_finite"], np.isfinite(want))
        np.testing.assert_array_equal(_decode(got, f), np.where(np.isfinite(want), want, np.nan))


def test_large_outputs_keep_the_same_seeded_sample_of_runs(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT", 8192)
    res = _result(1000)
    winners = torch.arange(12.0).reshape(3, 4)
    winners[1, 3] = float("nan")
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), winners, res)
    total = sum(os.path.getsize(tmp_path / "a" / f) - 128 for f in os.listdir(tmp_path / "a"))  # minus .npy headers
    assert total <= 8192
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sorted(a) == sorted(b)
    for name in a:
        assert np.isfinite(a[name]).all(), name
        np.testing.assert_array_equal(a[name], b[name])
    runs = a["runs"].astype(np.int64)
    assert 0 < len(runs) < 1000 and np.all(np.diff(runs) > 0)
    np.testing.assert_array_equal(a["info"], res.info.numpy()[runs])
    np.testing.assert_array_equal(_decode(a, "consts"), res.consts.numpy()[runs])
    np.testing.assert_array_equal(_decode(a, "final_mse"), np.where(np.isfinite(res.final_mse.numpy()[runs]),
                                                                    res.final_mse.numpy()[runs], np.nan))
    np.testing.assert_array_equal(_decode(a, "winners"), winners.numpy())
