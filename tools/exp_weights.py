#!/usr/bin/env python
"""GPU experiment: what per-point weights (``bfgs_batch(..., sigma=...)``, ``vsr_set_weights``) cost.

    python tools/exp_weights.py [--beams 24] [--out FILE]

Config 2 (bench.py's default workload, 64 candidates x 10 restarts, N = 10 000, dual gradients): every beam
is fitted with ``bfgs_batch`` in three settings, alternated beam by beam (the order rotates, so drift of
the card or the host falls on every setting alike): no weights, ``sigma = 1`` and a seeded random ``sigma``
in [0.1, 10] (log-uniform).  Per beam and setting: the fit's milliseconds (host clock around the call,
which ends in a device synchronisation) and fits/s (candidates x restarts per second).  The winners of
"no weights" and ``sigma = 1`` must be the same bit for bit (string, constants, loss): the tool counts the
candidates that differ and exits 1 unless the count is 0.  On the winners of each beam, ``vsr_gram`` with
the random weights against ``vsr_gram`` without (CUDA events, median of 5).

Config 5 shape (one black-box beam, N = 1e5 fp32 points, 1024 candidates x 10 restarts): the same three
settings, each fitted twice in rotation, the second pass timed: the weighted resident slices stage one
column more there than anywhere else in the benchmark.

The card's name, power limit and SM clocks are read in the same process.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "vision-sr_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from src.visymre import uncertainty  # noqa: E402
from src.visymre.architectures import bfgs as vbfgs  # noqa: E402
from src.visymre.engine import fitter, hostpool  # noqa: E402
from src.visymre.workloads import generator as wg  # noqa: E402

SETTINGS = ("none", "ones", "random")


def card():
    """Name, power limit and SM clocks of GPU 0 (nvidia-smi, read only)."""
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout
    f = [x.strip() for x in out.strip().split(",")]
    return {"name": f[0], "power_limit": f[1], "sm_clock": f[2], "sm_max_clock": f[3]}


def timed(fn, reps=5):
    """Median milliseconds of fn() between two CUDA events on the current stream."""
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms))


def sigma_of(setting, n, seed):
    if setting == "none":
        return None
    if setting == "ones":
        return torch.ones(n, dtype=torch.float64, device="cuda:0")
    s = np.exp(np.random.RandomState(seed).uniform(np.log(0.1), np.log(10.0), n))
    return torch.from_numpy(s).cuda()


def canon(fits):
    return [repr(o) if isinstance(o, Exception) else (str(o[0]), np.asarray(o[1], np.float64).tobytes(),
                                                        np.asarray(o[2]).tobytes()) for o in fits]


def fit(b, cfg, td, setting, seed):
    X = torch.from_numpy(np.ascontiguousarray(b.X)).cuda()
    y = torch.from_numpy(np.ascontiguousarray(b.y)).cuda()
    sigma = sigma_of(setting, X.shape[0], seed)
    torch.cuda.synchronize()
    t = time.perf_counter()
    fits = vbfgs.bfgs_batch(list(b.tokens), X, y, cfg, td, x0=b.x0, sigma=sigma)
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, fits, X, y, sigma


def dump(res, fh):
    """JSON with one top-level key, and one row of a list, per line."""
    items = []
    for key, val in res.items():
        if isinstance(val, list):
            body = "[\n" + ",\n".join("  " + json.dumps(r) for r in val) + "\n ]"
        else:
            body = json.dumps(val)
        items.append(f" {json.dumps(key)}: {body}")
    fh.write("{\n" + ",\n".join(items) + "\n}\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--beams", type=int, default=24)
    ap.add_argument("--c5-cand", type=int, default=1024)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "exp_weights_1gpu.json"))
    args = ap.parse_args()
    info = card()
    print(info, flush=True)
    beams = bench.make_workload(args.beams, 10_000, 64, 10)
    td = wg.make_test_data()
    cfg = wg.make_cfg(10, 64, grad_mode="dual")
    hostpool.warm()
    eng = fitter.get_engine(0)
    for s in SETTINGS:                                 # warm-up of every setting on beam 0, untimed
        fit(beams[0], cfg, td, s, 0)
    rows, differ = [], 0
    for bi, b in enumerate(beams):
        order = SETTINGS[bi % 3:] + SETTINGS[:bi % 3]
        row = dict(beam=b.name)
        out = {}
        for s in order:
            ms, fits, X, y, sigma = fit(b, cfg, td, s, bi)
            out[s] = (fits, X, y, sigma)
            row[f"{s}_ms"] = ms
            row[f"{s}_fits_per_s"] = len(b.tokens) * 10 / (ms * 1e-3)
        d = sum(1 for a, c in zip(canon(out["none"][0]), canon(out["ones"][0])) if a != c)
        row["winners_differ_none_vs_ones"] = d
        differ += d
        # vsr_gram on the random-sigma winners, with and without their weights
        fits, X, y, sigma = out["random"]
        good = [f for f in fits if not isinstance(f, Exception)]
        progs = uncertainty._compile([(str(f[3]), len(f[1])) for f in good])
        consts = np.zeros((len(good), max(1, max(len(f[1]) for f in good))))
        for j, f in enumerate(good):
            consts[j, :len(f[1])] = f[1]
        ct = torch.from_numpy(consts).cuda()
        idx = np.arange(len(good))
        eng.set_programs(progs)
        eng.set_points(X, y, dtypes=(fitter.F64,), n_vars=10)
        row["gram_ms"] = timed(lambda: eng.gram(idx, ct))
        eng.set_points(X, y, dtypes=(fitter.F64,), n_vars=10, w=1.0 / (sigma * sigma))
        row["gram_weighted_ms"] = timed(lambda: eng.gram(idx, ct))
        print(row, flush=True)
        rows.append(row)

    # ---- config 5 shape ----
    b5, _ = wg.blackbox_beam(100_000, args.c5_cand, 10, seed=0)
    wg.compile_beam(b5, td)
    cfg5 = wg.make_cfg(10, args.c5_cand, grad_mode="dual", precision="fp32")
    c5 = {}
    for rep in range(2):
        for s in (SETTINGS if rep == 0 else SETTINGS[1:] + SETTINGS[:1]):
            ms, fits, *_ = fit(b5, cfg5, td, s, 5)
            if rep == 1:
                c5[f"{s}_ms"] = ms
                c5[f"{s}_fits_per_s"] = args.c5_cand * 10 / (ms * 1e-3)
            if s == "none":
                c5_none = canon(fits)
            elif s == "ones":
                c5_ones = canon(fits)
    c5["winners_differ_none_vs_ones"] = sum(1 for a, c in zip(c5_none, c5_ones) if a != c)
    differ += c5["winners_differ_none_vs_ones"]
    print("config5", c5, flush=True)

    med = lambda key: float(np.median([r[key] for r in rows]))  # noqa: E731
    summary = {f"{s}_ms_median": med(f"{s}_ms") for s in SETTINGS}
    summary.update({f"{s}_fits_per_s_median": med(f"{s}_fits_per_s") for s in SETTINGS})
    summary["ones_over_none"] = float(np.median([r["ones_ms"] / r["none_ms"] for r in rows]))
    summary["random_over_none"] = float(np.median([r["random_ms"] / r["none_ms"] for r in rows]))
    summary["gram_ms_median"] = med("gram_ms")
    summary["gram_weighted_ms_median"] = med("gram_weighted_ms")
    summary["winners_differ_none_vs_ones"] = differ
    res = dict(tool="tools/exp_weights.py", card=info, host_workers=hostpool._POOL_N, config2=rows,
               config2_summary=summary, config5_shape=dict(points=100_000, cand=args.c5_cand, restarts=10, **c5))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        dump(res, fh)
    print(json.dumps(summary))
    return 1 if differ else 0


if __name__ == "__main__":
    sys.exit(main())
