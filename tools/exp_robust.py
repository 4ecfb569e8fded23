#!/usr/bin/env python
"""GPU experiment: what a robust loss (``bfgs_batch(..., loss=, f_scale=)``, ``vsr_set_loss``) costs.

    python tools/exp_robust.py [--beams 24] [--out FILE]

Config 2 (bench.py's default workload, 64 candidates x 10 restarts, N = 10 000, dual gradients): every beam
is fitted with ``bfgs_batch`` in three settings, alternated beam by beam (the order rotates, so drift of
the card or the host falls on every setting alike): ``linear``, ``huber`` with ``f_scale = 2**500`` (every
finite z <= 1: the linear trajectory through the robust kernels, so its ratio is the pure cost of the
robust sweep; ``2**20`` is not enough, the fits' line searches reach residuals above it) and ``soft_l1``
with ``f_scale = 1``.  Per beam and setting: the fit's milliseconds (host clock
around the call, which ends in a device synchronisation) and fits/s (candidates x restarts per second).
The winners of ``linear`` and ``huber`` must be the same bit for bit (string, constants, loss): the tool
counts the candidates that differ and exits 1 unless the count is 0.  On the winners of each beam,
``vsr_gram`` under soft_l1 against the linear ``vsr_gram`` (CUDA events, median of 5).

Config 5 shape (one black-box beam, N = 1e5 fp32 points, 1024 candidates x 10 restarts): the same three
settings, each fitted twice in rotation, the second pass timed.

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

SETTINGS = ("linear", "huber", "soft_l1")
LOSS = {"linear": ("linear", 1.0), "huber": ("huber", 2.0 ** 500), "soft_l1": ("soft_l1", 1.0)}


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


def canon(fits):
    return [repr(o) if isinstance(o, Exception) else (str(o[0]), np.asarray(o[1], np.float64).tobytes(),
                                                        np.asarray(o[2]).tobytes()) for o in fits]


def fit(b, cfg, td, setting):
    X = torch.from_numpy(np.ascontiguousarray(b.X)).cuda()
    y = torch.from_numpy(np.ascontiguousarray(b.y)).cuda()
    loss, f_scale = LOSS[setting]
    torch.cuda.synchronize()
    t = time.perf_counter()
    fits = vbfgs.bfgs_batch(list(b.tokens), X, y, cfg, td, x0=b.x0, loss=loss, f_scale=f_scale)
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, fits, X, y


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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "exp_robust_1gpu.json"))
    args = ap.parse_args()
    info = card()
    print(info, flush=True)
    beams = bench.make_workload(args.beams, 10_000, 64, 10)
    td = wg.make_test_data()
    cfg = wg.make_cfg(10, 64, grad_mode="dual")
    hostpool.warm()
    eng = fitter.get_engine(0)
    for s in SETTINGS:                                 # warm-up of every setting on beam 0, untimed
        fit(beams[0], cfg, td, s)
    rows, differ = [], 0
    for bi, b in enumerate(beams):
        order = SETTINGS[bi % 3:] + SETTINGS[:bi % 3]
        row = dict(beam=b.name)
        out = {}
        for s in order:
            ms, fits, X, y = fit(b, cfg, td, s)
            out[s] = (fits, X, y)
            row[f"{s}_ms"] = ms
            row[f"{s}_fits_per_s"] = len(b.tokens) * 10 / (ms * 1e-3)
        d = sum(1 for a, c in zip(canon(out["linear"][0]), canon(out["huber"][0])) if a != c)
        row["winners_differ_linear_vs_huber"] = d
        differ += d
        # vsr_gram on the soft_l1 winners, robust and linear
        fits, X, y = out["soft_l1"]
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
        eng.set_points(X, y, dtypes=(fitter.F64,), n_vars=10, loss=LOSS["soft_l1"])
        row["gram_robust_ms"] = timed(lambda: eng.gram(idx, ct))
        print(row, flush=True)
        rows.append(row)

    # ---- config 5 shape ----
    b5, _ = wg.blackbox_beam(100_000, args.c5_cand, 10, seed=0)
    wg.compile_beam(b5, td)
    cfg5 = wg.make_cfg(10, args.c5_cand, grad_mode="dual", precision="fp32")
    c5 = {}
    for rep in range(2):
        for s in (SETTINGS if rep == 0 else SETTINGS[1:] + SETTINGS[:1]):
            ms, fits, *_ = fit(b5, cfg5, td, s)
            if rep == 1:
                c5[f"{s}_ms"] = ms
                c5[f"{s}_fits_per_s"] = args.c5_cand * 10 / (ms * 1e-3)
            if s == "linear":
                c5_lin = canon(fits)
            elif s == "huber":
                c5_hub = canon(fits)
    c5["winners_differ_linear_vs_huber"] = sum(1 for a, c in zip(c5_lin, c5_hub) if a != c)
    differ += c5["winners_differ_linear_vs_huber"]
    print("config5", c5, flush=True)

    med = lambda key: float(np.median([r[key] for r in rows]))  # noqa: E731
    summary = {f"{s}_ms_median": med(f"{s}_ms") for s in SETTINGS}
    summary.update({f"{s}_fits_per_s_median": med(f"{s}_fits_per_s") for s in SETTINGS})
    for s in SETTINGS[1:]:
        ratio = [r[f"{s}_ms"] / r["linear_ms"] for r in rows]
        summary[f"{s}_over_linear"] = float(np.median(ratio))
        summary[f"{s}_over_linear_min_max"] = [float(np.min(ratio)), float(np.max(ratio))]
    summary["gram_ms_median"] = med("gram_ms")
    summary["gram_robust_ms_median"] = med("gram_robust_ms")
    summary["winners_differ_linear_vs_huber"] = differ
    res = dict(tool="tools/exp_robust.py", card=info, host_workers=hostpool._POOL_N, config2=rows,
               config2_summary=summary, config5_shape=dict(points=100_000, cand=args.c5_cand, restarts=10, **c5))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        dump(res, fh)
    print(json.dumps(summary))
    return 1 if differ else 0


if __name__ == "__main__":
    sys.exit(main())
