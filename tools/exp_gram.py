#!/usr/bin/env python
"""GPU experiment: what the covariance of fitted constants (uncertainty.covariances, vsr_gram) costs.

    python tools/exp_gram.py [--beams 24] [--out FILE]

Config 2 (bench.py's default workload): every beam is fitted with ``bfgs_batch`` (dual gradients), then
``covariances`` runs on its 64 winners.  Per beam: the fit (host clock around the call, which ends in a
device synchronisation), the skeleton compilation on the host in this process and in the host pool, the
whole ``covariances`` call, and -- with CUDA events, median of 5 -- the ``vsr_gram`` launch pair and
``vsr_eval`` with gradient on the same pairs (the same sweep over the points: the lower bound).

Config 5 shape: N = 1e5, 1e6, 1e7 random points and 1024 pairs (the winners' programs of the first beam,
cycled, at their fitted constants): ``vsr_gram`` time per call, per pair and per pair-point (events,
median of 5 after a warm-up call).  A sample of 32 of those pairs at N = 1e5 is checked against the CPU
reference of the sweep (``tests/native/gram_twin.cpp``); the tool exits 1 if any differs by more than 1e-12 (relative; Frobenius
for J^T J).  The card's name, power limit and SM clocks are read in the same process.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "vision-sr_b200"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from _gram_ref import frob_rel, load_twin, twin_gram  # noqa: E402
from src.visymre import uncertainty  # noqa: E402
from src.visymre.architectures import bfgs as vbfgs  # noqa: E402
from src.visymre.engine import fitter, hostpool  # noqa: E402
from src.visymre.workloads import generator as wg  # noqa: E402


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


def compile_ms(items, pool_min):
    saved = uncertainty.POOL_MIN
    uncertainty.POOL_MIN = pool_min
    t = time.perf_counter()
    progs = uncertainty._compile(items)
    uncertainty.POOL_MIN = saved
    return (time.perf_counter() - t) * 1e3, progs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--beams", type=int, default=24)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "exp_gram_1gpu.json"))
    args = ap.parse_args()
    twin = load_twin()
    info = card()
    print(info, flush=True)
    beams = bench.make_workload(args.beams, 10_000, 64, 10)
    td = wg.make_test_data()
    cfg = wg.make_cfg(10, 64, grad_mode="dual")
    hostpool.warm()
    eng = fitter.get_engine(0)
    rows = []
    for bi, b in enumerate([beams[0]] + beams):       # the first pass over beam 0 warms up, untimed
        X = torch.from_numpy(np.ascontiguousarray(b.X)).cuda()
        y = torch.from_numpy(np.ascontiguousarray(b.y)).cuda()
        torch.cuda.synchronize()
        t = time.perf_counter()
        fits = vbfgs.bfgs_batch(list(b.tokens), X, y, cfg, td, x0=b.x0)
        torch.cuda.synchronize()
        fit_ms = (time.perf_counter() - t) * 1e3
        items = [(str(f[3]), len(f[1])) for f in fits if not isinstance(f, Exception)]
        inline_ms, progs = compile_ms(items, 1 << 30)
        pool_ms, _ = compile_ms(items, 1)
        t = time.perf_counter()
        cov = uncertainty.covariances(fits, X, y)
        torch.cuda.synchronize()
        cov_ms = (time.perf_counter() - t) * 1e3
        consts = np.zeros((len(items), max(1, max(k for _, k in items))))
        j = 0
        for f in fits:
            if not isinstance(f, Exception):
                consts[j, :len(f[1])] = f[1]
                j += 1
        ct = torch.from_numpy(consts).cuda()
        idx = np.arange(len(items))
        gram_ms = timed(lambda: eng.gram(idx, ct))
        eval_ms = timed(lambda: eng.eval(idx, ct, dtype=fitter.F64, grad=True))
        if bi == 0:
            first_progs, first_consts = progs, consts
            continue
        row = dict(beam=b.name, winners=len(items), fit_ms=fit_ms, compile_inline_ms=inline_ms,
                   compile_pool_ms=pool_ms, covariances_ms=cov_ms, gram_ms=gram_ms, eval_grad_ms=eval_ms,
                   finite_stderr=int(sum(1 for c in cov if c is not None and np.isfinite(c.stderr[c.free]).all())))
        print(row, flush=True)
        rows.append(row)

    # ---- config 5 shape: 1024 pairs ----
    eng.set_programs(first_progs)
    pairs = np.arange(1024) % len(first_progs)
    ct = torch.from_numpy(first_consts[pairs]).cuda()
    scale = []
    bad = []
    for n in (100_000, 1_000_000, 10_000_000):
        g = torch.Generator(device="cuda:0").manual_seed(n)
        Xn = torch.rand((n, 10), dtype=torch.float64, device="cuda:0", generator=g) * 1.5 + 0.5
        yn = torch.randn(n, dtype=torch.float64, device="cuda:0", generator=g)
        eng.set_points(Xn, yn, dtypes=(fitter.F64,), n_vars=10)
        rss, jtj = eng.gram(pairs, ct)
        ms = timed(lambda: eng.gram(pairs, ct))
        scale.append(dict(n_points=n, pairs=1024, gram_ms=ms, us_per_pair=ms * 1e3 / 1024,
                          ns_per_pair_point=ms * 1e6 / (1024 * n)))
        print(scale[-1], flush=True)
        if n == 100_000:
            rss, jtj = rss.cpu().numpy(), jtj.cpu().numpy()
            Xh, yh = Xn.cpu().numpy(), yn.cpu().numpy()
            for p in np.random.RandomState(0).choice(1024, 32, replace=False):
                prog = first_progs[pairs[p]]
                k = prog.k
                want_rss, want_jtj = twin_gram(twin, prog, Xh, yh, first_consts[pairs[p], :k])
                got_j = jtj[p, :k, :k]
                if np.isnan(want_rss) or np.isnan(rss[p]):
                    ok = np.isnan(want_rss) and np.isnan(rss[p])
                else:
                    ok = abs(rss[p] - want_rss) <= 1e-12 * abs(want_rss) and (
                        k == 0 or np.array_equal(np.isfinite(got_j), np.isfinite(want_jtj)) and
                        frob_rel(np.nan_to_num(got_j), np.nan_to_num(want_jtj)) <= 1e-12)
                if not ok:
                    bad.append(dict(pair=int(p), k=k, rss=float(rss[p]), want=float(want_rss)))
    summary = dict(
        fit_ms_median=float(np.median([r["fit_ms"] for r in rows])),
        gram_ms_median=float(np.median([r["gram_ms"] for r in rows])),
        eval_grad_ms_median=float(np.median([r["eval_grad_ms"] for r in rows])),
        compile_inline_ms_median=float(np.median([r["compile_inline_ms"] for r in rows])),
        compile_pool_ms_median=float(np.median([r["compile_pool_ms"] for r in rows])),
        covariances_ms_median=float(np.median([r["covariances_ms"] for r in rows])),
        gram_share_of_fit=float(np.median([r["gram_ms"] / r["fit_ms"] for r in rows])))
    res = dict(tool="tools/exp_gram.py", card=info, host_workers=hostpool._POOL_N, config2=rows,
               config2_summary=summary, config5_shape=scale, reference_mismatches=bad)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(summary), "mismatches:", len(bad))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
