#!/usr/bin/env python
"""GPU experiment: what per-point predictions and their bands (uncertainty.predict, vsr_predict) cost.

    python tools/exp_predict.py [--beams 4] [--out FILE]

Config 2 (bench.py's default workload, N = 1e4): every beam is fitted with ``bfgs_batch`` (dual
gradients) and ``covariances`` runs on its 64 winners.  Then, on the same training points: one
``vsr_predict`` call with variances, one without, and ``vsr_eval`` value-only on the same pairs (the
same sweep with no per-point writes: the lower bound).

Config 5 (the black-box beam of BASELINE config 5 with 64 candidates): the beam is fitted on its 1e5
points, ``covariances`` runs on its 64 winners, and the same three calls run on N = 1e5, 1e6, 1e7 new
points of the config's distribution (X ~ N(0, 1) in 3 variables), in fp32 (the config's precision)
and fp64.

Per call: the median of 20 calls between two CUDA events (call time, host enqueue included), and the
kernel time from a separate torch.profiler run over 10 calls (sum of the launch's kernels).  Bytes
moved: the columns each pair's program reads (8 B per point each) plus 8 B (value) or 16 B (value and
variance) written per pair-point, over the kernel time, against the 7.7 TB/s HBM figure of the B200
data sheet.  The reference's way is timed for one winner: ``sp.lambdify`` with numpy at N = 1e6,
whose result is also the check of the device values there (the tool exits 1 on a mismatch above
1e-12 relative to the row's largest value).  The card's name, power limit and SM clocks are read in
the same process.
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
import sympy as sp  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from _gram_ref import VARS  # noqa: E402
from oracle import vectorised  # noqa: E402
from src.visymre import uncertainty  # noqa: E402
from src.visymre.architectures import bfgs as vbfgs  # noqa: E402
from src.visymre.engine import fitter, hostpool  # noqa: E402
from src.visymre.workloads import generator as wg  # noqa: E402

HBM_TBS = 7.7


def card():
    """Name, power limit and SM clocks of GPU 0 (nvidia-smi, read only)."""
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout
    f = [x.strip() for x in out.strip().split(",")]
    return {"name": f[0], "power_limit": f[1], "sm_clock": f[2], "sm_max_clock": f[3]}


def timed(fn, reps=20):
    """Median milliseconds of fn() between two CUDA events on the current stream."""
    fn()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms))


def kernel_ms(fn, reps=10):
    """Mean device milliseconds per call of the kernels fn() launches (torch.profiler, its own run)."""
    fn()
    torch.cuda.synchronize()
    acts = [torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    total, names = 0.0, set()
    for e in prof.key_averages():
        if "vsr::" in e.key:
            total += getattr(e, "device_time_total", None) or e.cuda_time_total
            names.add(e.key.split("(")[0])
    return total / reps / 1e3, sorted(names)


def bytes_moved(progs, pairs, n, elem, write_b):
    read = sum(bin(progs[p].var_mask).count("1") for p in pairs) * elem * n
    return read + len(pairs) * n * write_b


def pairs_of(fits, covs):
    """Device constants [n, kmax] and covariances [n, kmax, kmax] of the fits, as predict uploads them."""
    kmax = max(1, max(len(f[1]) for f in fits))
    consts = torch.zeros((len(fits), kmax), dtype=torch.float64)
    cov = torch.zeros((len(fits), kmax, kmax), dtype=torch.float64)
    for j, (f, cv) in enumerate(zip(fits, covs)):
        k = len(f[1])
        consts[j, :k] = torch.as_tensor(np.asarray(f[1], dtype=np.float64))
        cov[j, :k, :k] = torch.from_numpy(uncertainty.device_cov(cv.cov))
    return consts.cuda(), cov.cuda()


def measure(eng, progs, pairs, consts, cov, n, dt=fitter.F64):
    """The three calls on the engine's current points: call and kernel time, bytes, share of HBM."""
    idx = np.asarray(pairs)
    out = {}
    calls = {"predict_var": lambda: eng.predict(idx, consts, cov=cov, dtype=dt),
             "predict_value": lambda: eng.predict(idx, consts, dtype=dt),
             "eval_value": lambda: eng.eval(idx, consts, dtype=dt)}
    for name, fn in calls.items():
        call = timed(fn)
        kern, kernels = kernel_ms(fn)
        wb = {"predict_var": 16, "predict_value": 8, "eval_value": 0}[name]
        b = bytes_moved(progs, idx, n, 8 if dt == fitter.F64 else 4, wb)
        out[name] = dict(call_ms=call, kernel_ms=kern, kernels=kernels, bytes=b,
                         tb_per_s=b / (kern * 1e-3) / 1e12, share_of_hbm=b / (kern * 1e-3) / (HBM_TBS * 1e12),
                         ns_per_pair_point=kern * 1e6 / (len(idx) * n))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--beams", type=int, default=4)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "exp_predict_1gpu.json"))
    args = ap.parse_args()
    info = card()
    print(info, flush=True)
    beams = bench.make_workload(args.beams, 10_000, 64, 10)
    td = wg.make_test_data()
    cfg = wg.make_cfg(10, 64, grad_mode="dual")
    hostpool.warm()
    eng = fitter.get_engine(0)
    rows = []
    for b in beams:
        X = torch.from_numpy(np.ascontiguousarray(b.X)).cuda()
        y = torch.from_numpy(np.ascontiguousarray(b.y)).cuda()
        fits = [f for f in vbfgs.bfgs_batch(list(b.tokens), X, y, cfg, td, x0=b.x0) if not isinstance(f, Exception)]
        covs = uncertainty.covariances(fits, X, y)
        t = time.perf_counter()
        preds = uncertainty.predict(fits, X, covs=covs)
        torch.cuda.synchronize()
        predict_call_ms = (time.perf_counter() - t) * 1e3
        progs = eng.programs            # predict left the winners' programs and the points on the engine
        consts, cov = pairs_of(fits, covs)
        n = eng.n_points
        row = dict(beam=b.name, winners=len(fits), n_points=n, predict_call_ms=predict_call_ms,
                   finite_bands=int(sum(1 for p in preds if torch.isfinite(p.ci_high).all())),
                   **measure(eng, progs, range(len(fits)), consts, cov, n))
        print(json.dumps(row), flush=True)
        rows.append(row)

    # ---- config 5: 64 winners of a black-box beam, fitted on its 1e5 points ----
    b, td5 = wg.blackbox_beam(100_000, 64, 10, seed=0)
    X = torch.from_numpy(np.ascontiguousarray(b.X)).cuda()
    y = torch.from_numpy(np.ascontiguousarray(b.y)).cuda()
    fits = [f for f in vbfgs.bfgs_batch(list(b.tokens), X, y, cfg, td5, x0=b.x0) if not isinstance(f, Exception)]
    covs = uncertainty.covariances(fits, X, y)
    uncertainty.predict(fits, X, covs=covs)     # leaves the winners' programs on the engine
    progs = eng.programs
    consts, cov = pairs_of(fits, covs)
    scale = []
    mismatch = []
    host = None
    for n in (100_000, 1_000_000, 10_000_000):
        # new points of the config's distribution: X ~ N(0, 1) in 3 variables, fp32 and its fp64 copy
        g = torch.Generator(device="cuda:0").manual_seed(n)
        Xn = torch.zeros((n, 10), dtype=torch.float32, device="cuda:0")
        Xn[:, :3] = torch.randn((n, 3), dtype=torch.float32, device="cuda:0", generator=g)
        eng.set_points(Xn, torch.zeros(n, dtype=torch.float64, device="cuda:0"), dtypes=(fitter.F32, fitter.F64),
                       n_vars=3)
        for dt, name in ((fitter.F32, "fp32"), (fitter.F64, "fp64")):
            row = dict(n_points=n, pairs=len(progs), dtype=name,
                       **measure(eng, progs, range(len(progs)), consts, cov, n, dt))
            print(json.dumps(row), flush=True)
            scale.append(row)
        if n == 1_000_000:
            # the reference's way for one winner: sympy's lambdify with numpy on the host
            j = max(range(len(fits)), key=lambda i: len(fits[i][1]))
            skel, c = str(fits[j][3]), np.asarray(fits[j][1], dtype=np.float64)
            cs = [sp.Symbol(f"c{i}", real=True) for i in range(c.size)]
            xs = [sp.Symbol(v, real=True) for v in VARS]
            f = sp.lambdify(cs + xs, sp.sympify(skel, locals={str(s): s for s in cs + xs}),
                            modules=[{"re": np.real, "im": np.imag}, vectorised.MODULES, "numpy"])
            cols = list(Xn.double().cpu().numpy().T)
            ts = []
            with np.errstate(all="ignore"):
                for _ in range(3):
                    t = time.perf_counter()
                    want = np.asarray(f(*c, *cols))
                    if np.iscomplexobj(want):      # a value that is not real is nan, as on the device
                        want = np.where(want.imag == 0, want.real, np.nan)
                    want = np.broadcast_to(want.astype(np.float64), (n,))
                    ts.append((time.perf_counter() - t) * 1e3)
            t = time.perf_counter()
            got = eng.predict([j], consts[j:j + 1], dtype=fitter.F64)[0][0].cpu().numpy()
            one_ms = (time.perf_counter() - t) * 1e3
            ok = np.isfinite(want)
            scale_v = np.abs(want[ok]).max() if ok.any() else 1.0
            if not (np.array_equal(np.isfinite(got), ok) and np.all(np.abs(got[ok] - want[ok]) <= 1e-12 * scale_v)):
                mismatch.append(skel)
            host = dict(skeleton=skel, k=int(c.size), n_points=n, lambdify_numpy_ms=float(np.median(ts)),
                        device_predict_one_call_fp64_ms=one_ms)
            print(json.dumps(host), flush=True)
    summary = {name: dict(call_ms_median=float(np.median([r[name]["call_ms"] for r in rows])),
                          kernel_ms_median=float(np.median([r[name]["kernel_ms"] for r in rows])))
               for name in ("predict_var", "predict_value", "eval_value")}
    res = dict(tool="tools/exp_predict.py", card=info, hbm_tb_per_s=HBM_TBS, config2=rows, config2_summary=summary,
               config5=scale, host_reference=host, mismatches=mismatch)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(summary), "mismatches:", len(mismatch))
    return 1 if mismatch else 0


if __name__ == "__main__":
    sys.exit(main())
