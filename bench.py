#!/usr/bin/env python
"""Benchmark of the refinement hot path (BASELINE.json metric: candidate-fits/sec).

A STEP is the refinement of one beam -- what one ``fitfunc2`` call hands to its BFGS part: C
candidates x R restarts fitted over N points and scored.  ``--config`` selects the BASELINE.json
workload (default 2, the one the metric is quoted on):

  1  low_benchmarks.csv rows      C=16    R=10  N=500    fp64   (the only one the AS-IS reference runs)
  2  AI-Feynman table rows        C=64    R=10  N=1e4    fp64
  3  ODE-Strogatz (ode.xlsx)      C=128   R=32  N=1e4    fp64
  4  SRSD-shaped Feynman (log-uniform ranges)  C=256  R=64  N=1e5  fp32 sweeps, fp64 optimiser state
  5  black-box shaped, 3 variables, fp32 points  C=1024  R=10  N=--points (1e3 ... 1e7)

  value   whole-job candidate-fits/s with points, programs and starting points already resident in
          HBM when the timed region starts (device events, max over ranks)
  e2e     the same steps through the entry point a driver calls, ``refine_hypotheses`` (token ids and
          host tensors in, the reference's dict out): host->device copies, skeleton compilation
          (cold cache), fit, prune, winner formatting and the device->host read all inside the
          timed region.  ``e2e_abi`` is the C-ABI figure (vsr_upload_* + vsr_fit_host, host buffers,
          precompiled bytecode).
  roofline / cpu_baseline: see DESIGN.md section "Measurement".

N > 1 (torchrun): STRONG scaling of the north-star partition -- every step is ONE beam whose
(candidate, restart) runs are dealt over all ranks (engine/sharding.py), each rank fits its share, one
all-gather of per-candidate records inside the timed region, same argmin everywhere; the winners
are checked bit-for-bit against the one-GPU fit of the same beam in the run.  The throughput of N
independent replica beams (no collective, weak scaling) is kept as the extra key ``replicas``.

`--impl reference` times the reference's CPU implementation of the path on the host cores: the
as-is reference (oracle/_ref, built by oracle/build_ref.py) for config 1, the oracle port (scipy
BFGS over numpy columns -- the as-is reference cannot run at N >= ~1e4) for the others; one step =
all candidates of one beam on all cores, one pool for the whole run.

`--dump-outputs DIR` writes, after the timed steps, what the fit returned in the last timed step as
DIR/<name>.npy (see dump_outputs).  The workload is seeded, so two builds run with the same
arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "vision-sr_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

CONFIGS = {
    1: dict(table="low", points=500, cand=16, restarts=10, precision="fp64",
            what="low_benchmarks.csv rows (Nguyen-style, 1-2 variables)"),
    2: dict(table="feynman", points=10_000, cand=64, restarts=10, precision="fp64",
            what="AI-Feynman table rows (FeynmanEquations.xlsx)"),
    3: dict(table="ode", points=10_000, cand=128, restarts=32, precision="fp64",
            what="ODE-Strogatz rows (ode.xlsx), x_1, x_2 ~ U(0.1, 5)"),
    4: dict(table="srsd", points=100_000, cand=256, restarts=64, precision="fp32",
            what="SRSD-Feynman-shaped: Feynman rows, variables log-uniform over two decades"),
    5: dict(table="blackbox", points=100_000, cand=1024, restarts=10, precision="fp32",
            what="black-box shaped: X ~ N(0,1) in 3 variables (fp32), y = 1.5 x1 sin(0.7 x2) + 0.3 x3^2 + noise"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--points", type=int, default=0, help="override the config's number of points")
    ap.add_argument("--cand", type=int, default=0, help="override the config's beam size")
    ap.add_argument("--restarts", type=int, default=0, help="override the config's number of restarts")
    ap.add_argument("--grad-mode", default="dual", choices=["dual", "fd"])
    ap.add_argument("--precision", default="", choices=["", "fp64", "fp32"])
    ap.add_argument("--mode", default="auto", choices=["auto", "sharded", "replicas"],
                    help="N > 1: one beam sharded over the ranks (auto) or independent replica beams")
    ap.add_argument("--warps", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=25.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-api", action="store_true", help="skip the refine_hypotheses end-to-end loop")
    ap.add_argument("--rows", default="", help="comma separated table row names (default: table order)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the fit returned in the last timed step to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU fit (--impl b200)")
    c = CONFIGS[a.config]
    a.points = a.points or c["points"]
    a.cand = a.cand or c["cand"]
    a.restarts = a.restarts or c["restarts"]
    a.precision = a.precision or c["precision"]
    return a


# ---- workload (generated in parallel: sympy is slow) -----------------------------------------
def _gen_beam(job):
    import warnings
    warnings.filterwarnings("ignore")
    from src.visymre.workloads import generator as g
    table, e, row, n_points, n_cand, n_restarts = job
    td = g.make_test_data()
    if table in ("feynman", "srsd"):
        b = g.build_beam(e + (50_000 if table == "srsd" else 0), row["name"], row["replaced"] or row["formula"],
                         row["variables"], n_points, n_cand, n_restarts, td, log_uniform=(table == "srsd"))
    elif table == "low":
        b = g.low_beam(e, row, n_points, n_cand, n_restarts, td)
    elif table == "ode":
        b = g.build_beam(20_000 + e, row["name"], row["formula"], [dict(low=0.1, high=5.0)] * 2,
                         n_points, n_cand, n_restarts, td)
    else:
        b, _ = g.blackbox_beam(n_points, n_cand, n_restarts, seed=e)
    if b is None:
        return None
    g.compile_beam(b, td)
    return b


def table_rows(args):
    from src.visymre.workloads import generator as g
    t = g.load_tables()
    table = CONFIGS[args.config]["table"]
    if table in ("feynman", "srsd"):
        rows = [(e, r) for e, r in enumerate(t["feynman"]) if not r["name"].startswith("test_")]
    elif table == "low":
        rows = list(enumerate(t["low"]))
    elif table == "ode":
        rows = list(enumerate(t["ode"]))
    else:
        rows = [(0, dict(name="blackbox"))]
    if args.rows:
        want = args.rows.split(",")
        rows = [(e, r) for e, r in rows if r["name"] in want]
    return table, rows


def make_workload(n_beams, args, *legacy, rank=0, world=1, dist=None):
    """The first n_beams usable rows of the config's table, one beam each (cycled when the table is
    shorter).  With several ranks every rank generates rows rank, rank+world, ... with its share of the
    host cores and one all_gather_object puts the lists together: every rank holds the same beams."""
    from concurrent.futures import ProcessPoolExecutor
    if isinstance(args, int):   # make_workload(n, points, cand, restarts): config 2 at the given sizes
        args = argparse.Namespace(config=2, points=args, cand=legacy[0], restarts=legacy[1], rows="")
    table, rows = table_rows(args)
    rows = rows[: int(n_beams * 1.3) + 4]
    jobs = [(table, e, r, args.points, args.cand, args.restarts) for e, r in rows]
    workers = max(1, min(32, (os.cpu_count() or 2) // world, len(jobs)))
    mine = jobs[rank::world]
    with ProcessPoolExecutor(workers) as ex:
        got = list(ex.map(_gen_beam, mine))
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, got)
        got = [parts[i % world][i // world] for i in range(len(jobs))]
    beams = [b for b in got if b is not None]
    if not beams:
        raise RuntimeError("no beam could be generated")
    distinct = len(beams)
    while len(beams) < n_beams:      # fewer usable rows than steps: cycle
        beams.append(beams[len(beams) % distinct])
    return beams[:n_beams]


class Claims:
    """Replica mode: hands out the global step indices 0..n-1 to the ranks of ONE node: rank r takes its
    own stripe r, r+world, ... first and then what the others have not started yet.  A claim is an
    O_EXCL file creation in a directory all ranks see; with one rank it is a plain counter.  Beams
    are independent units: this is scheduling, not a data-path collective."""

    def __init__(self, n, rank, world, root, tag):
        self.n, self.rank, self.world, self.root, self.tag = n, rank, world, root, tag
        own = list(range(rank, n, world))
        others = [i for i in range(n - 1, -1, -1) if i % world != rank]
        self.order = own + others
        self.pos = 0

    def next(self):
        while self.pos < len(self.order):
            i = self.order[self.pos]
            self.pos += 1
            if self.world == 1:
                return i
            try:
                os.close(os.open(os.path.join(self.root, f"{self.tag}_{i}"), os.O_CREAT | os.O_EXCL | os.O_WRONLY))
                return i
            except FileExistsError:
                continue
        return None


# ---- clocks ---------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.2] or [r for _, r in self.rows]
        mhz = [float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(mhz)) if mhz else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(rows)}


# ---- CPU arm: the reference's path on the host cores ----------------------------------------------
def _cpu_fit(job):
    """One candidate through the CPU implementation.  kind 'port': oracle/vectorised.py; kind
    'reference': the unmodified reference's own bfgs_wrapper (oracle/_ref or $VISYMRE_REFERENCE), with
    its per-restart np.random.randn draws fed from the workload's starting points."""
    import warnings
    warnings.filterwarnings("ignore")
    kind, tokens, X, y, x0, R = job
    if kind == "port":
        from oracle import vectorised
        from src.visymre.workloads import generator as g
        rec = vectorised.Recorder()
        out = vectorised.bfgs_wrapper((tokens, X[None], y, g.make_cfg(R), g.make_test_data()), x0=x0, record=rec)
        return out[1], sum(r.get("nfev", 0) for r in rec.restarts)
    import torch
    from types import SimpleNamespace as NS
    from oracle import ref_harness
    # the reference's `src` is a namespace package and this repo's a regular one, which would win
    # whatever the order of sys.path: this worker process only ever runs the reference
    sys.path[:] = [p for p in sys.path if os.path.basename(p.rstrip("/")) != "vision-sr_b200"]
    ref_bfgs, ref_model, td = ref_harness.load()
    cfg = NS(bfgs=NS(n_restarts=R, add_coefficients_if_not_existing=False, idx_remove=False,
                     normalization_type="MSE", stop_time=1e9))
    nfev = [0]
    real_minimize, real_randn = ref_bfgs.minimize, np.random.randn
    draws = [np.asarray(r, dtype=np.float64) / 10.0 for r in x0]

    def counting(fun, start, **kw):
        res = real_minimize(fun, start, **kw)
        nfev[0] += int(res.nfev)
        return res

    def fed(*shape):
        return draws.pop(0).copy() if draws and len(draws[0]) == (shape[0] if shape else 1) else real_randn(*shape)
    ref_bfgs.minimize, ref_bfgs.np.random.randn = counting, fed
    try:
        out = ref_model.bfgs_wrapper((list(tokens), torch.tensor(X[None]), torch.tensor(y), cfg, td))
    finally:
        ref_bfgs.minimize, ref_bfgs.np.random.randn = real_minimize, real_randn
    return out[1], nfev[0]


def cpu_kind(args):
    """Which CPU implementation this config is timed on, and why."""
    if args.config == 1:
        sys.path.insert(0, ROOT)
        from oracle import ref_harness
        if ref_harness.available():
            return "reference"
    return "port"


class CpuArm:
    """One worker pool for a whole run; a step = all candidates of a beam."""

    def __init__(self, kind, R):
        from concurrent.futures import ProcessPoolExecutor
        import multiprocessing as mp
        self.kind, self.R = kind, R
        self.cores = min(os.cpu_count() or 1, 64)
        # spawn: the parent may hold a CUDA context, and the as-is reference must not meet this
        # repo's `src` package (same top-level name) in its process
        self.pool = ProcessPoolExecutor(self.cores, mp_context=mp.get_context("spawn"))
        list(self.pool.map(_noop, range(2 * self.cores)))   # start the workers before any timing

    def step(self, beam, limit=None):
        jobs = [(self.kind, beam.tokens[j], beam.X, beam.y, beam.x0[j], self.R)
                for j in range(len(beam.tokens) if limit is None else min(limit, len(beam.tokens)))]
        t0 = time.time()
        outs = list(self.pool.map(_cpu_fit, jobs))
        dt = time.time() - t0
        return len(jobs), dt, sum(o[1] for o in outs)

    def close(self):
        self.pool.shutdown(wait=False, cancel_futures=True)


def _noop(i):
    import numpy  # noqa: F401
    return i


def cpu_baseline(beams, args, budget_s):
    """candidate-fits/s of the CPU arm on the timed workload: whole beams while they fit the budget,
    else the first candidates of the first beam (the sample is sized from an untimed probe of one
    candidate per core)."""
    kind = cpu_kind(args)
    arm = CpuArm(kind, args.restarts)
    C = len(beams[0].tokens)
    arm.step(beams[0], limit=arm.cores)                        # imports / first-call costs, untimed
    _, t_probe, _ = arm.step(beams[0], limit=arm.cores)        # one candidate per core: sizes the sample
    rounds = max(1, int(budget_s / max(t_probe, 1e-3)))
    limit = None if rounds * arm.cores >= C else rounds * arm.cores
    n = dt = nfev = 0
    t_all = time.time()
    used = 0
    # whole beams spread EVENLY over the timed ones (a beam's CPU time varies 10x with its candidates;
    # the first few are not representative): as many as the budget is expected to cover
    seen, distinct = set(), []
    for b in beams:
        if id(b) not in seen:
            seen.add(id(b))
            distinct.append(b)
    # visiting order: first, last, middle, quarters, ... so that wherever the budget ends the sample is spread
    order, step = [0, len(distinct) - 1], len(distinct) - 1
    while step > 1:
        step = (step + 1) // 2
        order += [i for i in range(step, len(distinct) - 1, step) if i not in order]
    order = [i for i in dict.fromkeys(order) if 0 <= i < len(distinct)]
    for i in order:
        a, d, f = arm.step(distinct[i], limit=limit)
        n, dt, nfev, used = n + a, dt + d, nfev + f, used + 1
        if limit is not None or time.time() - t_all + d > budget_s:
            break
    arm.close()
    N = beams[0].X.shape[0]
    what = (f"all {C} candidates of {used} of the timed beams (evenly spread)" if limit is None
            else f"the first {limit} of the {C} candidates of the first timed beam")
    return {"value": n / dt, "unit": "candidate-fits/s", "cores": arm.cores, "kind": kind,
            "sample": f"{what} (R={args.restarts}, N={N}), "
                      + ("the unmodified reference's bfgs_wrapper (oracle/_ref)" if kind == "reference"
                         else "oracle/vectorised.py (scipy BFGS over numpy columns)")
                      + f" in {arm.cores} worker processes, {dt:.1f} s, nfev {nfev}",
            "seconds": dt, "nfev": nfev, "point_evals_per_s": nfev * N / dt}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    beams = make_workload(args.warmup + args.steps, args)
    kind = cpu_kind(args)
    arm = CpuArm(kind, args.restarts)
    n = dt = nfev = steps = 0
    # a step = all candidates of a beam while that takes under ~12 s, else a bounded sample of them
    arm.step(beams[0], limit=arm.cores)                        # imports / first-call costs
    _, t_probe, _ = arm.step(beams[0], limit=arm.cores)
    rounds = max(1, int(12.0 / max(t_probe, 1e-3)))
    limit = None if rounds * arm.cores >= args.cand else rounds * arm.cores
    for s in range(args.warmup + args.steps):
        a, d, f = arm.step(beams[s], limit=limit)
        if s >= args.warmup:
            n, dt, nfev, steps = n + a, dt + d, nfev + f, steps + 1
    arm.close()
    v = n / dt
    line = {"impl": "reference", "metric": "candidate_fits_per_sec", "value": v, "unit": "candidate-fits/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "strong" if args.gpus > 1 else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args),
            "cpu_baseline": {"value": v, "unit": "candidate-fits/s", "cores": arm.cores, "kind": kind,
                             "sample": f"{'all ' + str(args.cand) if limit is None else 'the first ' + str(limit) + ' of the ' + str(args.cand)} candidates of {steps} beams, one pool of {arm.cores} worker processes, "
                                       f"{dt:.1f} s, nfev {nfev}", "seconds": dt, "nfev": nfev},
            "e2e": {"value": v, "unit": "candidate-fits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, winners, res):
    """Writes what ``fit_step`` returned as ``.npy`` files: the per-run FitResult fields and, when
    sharded, the gathered per-candidate winners.  A non-finite entry is not a number to compare but
    the absence of one (NaN fills the columns past a run's number of constants and every column of a
    run with none; a score is NaN or inf where the expression is not real at the fitted point, and
    the refinement skips it), so each float field is written as its finite entries in row-major
    order, ``<name>.npy`` (float64), with ``<name>_finite.npy`` (float32, the field's shape, 1 where
    the entry is finite).  ``info``'s int32 status / nit / nfev are written as float64, exactly.
    Outputs over DUMP_LIMIT keep the same seeded sample of runs in every field, listed in ``runs.npy``."""
    runs = {f: getattr(res, f).cpu().numpy() for f in ("consts", "lastx", "loss", "final_mse", "info")}
    extra = {} if winners is None else {"winners": winners.cpu().numpy()}
    n_runs = len(runs["loss"])
    # at most 8 bytes per value and 4 per mask entry (info: 8 per entry, no mask)
    per_run = sum(a[0].size * (8 if f == "info" else 12) for f, a in runs.items())
    budget = DUMP_LIMIT - sum(a.size * 12 for a in extra.values())
    out = {}
    if n_runs * per_run > budget:
        keep = np.sort(np.random.RandomState(0).choice(n_runs, int(budget // (per_run + 8)), replace=False))
        runs = {f: a[keep] for f, a in runs.items()}
        out["runs"] = keep.astype(np.float64)
    out["info"] = runs.pop("info").astype(np.float64)
    for name, a in {**runs, **extra}.items():
        finite = np.isfinite(a)
        out[name] = a[finite].astype(np.float64)
        out[f"{name}_finite"] = finite.astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def workload_config(args):
    c = CONFIGS[args.config]
    return {"workload": f"BASELINE config {args.config}: {c['what']}, synthetic points, beam={args.cand}, "
                        f"restarts={args.restarts}, points={args.points}; one step = one beam",
            "baseline_config": args.config,
            "candidates_per_step": args.cand, "restarts": args.restarts, "points": args.points,
            "grad_mode": args.grad_mode, "precision": args.precision,
            "l2": "flushed between timed steps (256 MiB write)"}


def emit(line):
    """The ONE line of stdout: everything else a library prints there (NCCL's version banner ...) was
    sent to stderr by main()."""
    os.write(_STDOUT, (json.dumps(line) + "\n").encode())


_STDOUT = 1


def main():
    global _STDOUT
    args = parse()
    sys.stdout.flush()
    _STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from src.visymre.engine import fitter, hostpool, isa, sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    mode = args.mode if args.mode != "auto" else ("sharded" if world > 1 else "replicas")
    if world == 1:
        mode = "replicas"

    # ---- workload: warmup + steps distinct beams, the same on every rank ----
    beams = make_workload(args.warmup + args.steps, args, rank=rank, world=world, dist=dist if world > 1 else None)
    D = len(beams)
    timed = [(args.warmup + i) % D for i in range(args.steps)]   # beam index of timed step i
    warm = [s % D for s in range(args.warmup)]
    R, C = args.restarts, args.cand
    eval_dt = fitter.F32 if args.precision == "fp32" else fitter.F64
    x_is_f32 = beams[0].X.dtype == np.float32
    score_dt = fitter.F32 if x_is_f32 else fitter.F64
    opts = fitter.default_opts(grad_mode=isa.GRAD_MODE["VSR_GRAD_FD" if args.grad_mode == "fd" else "VSR_GRAD_DUAL"],
                               eval_dtype=eval_dt, score_dtype=score_dt, warps_per_run=args.warps)

    # ---- resident setup: one engine per distinct beam, everything uploaded before timing ----
    setups = {}
    for bi in sorted(set(timed + warm)):
        b = beams[bi]
        eng = fitter.Engine(dev)
        eng.set_points(b.X, b.y, dtypes=tuple({eval_dt, score_dt}))
        eng.set_programs(b.programs)
        kmax = max(1, max(p.k for p in b.programs))
        x0 = np.zeros((C * R, kmax))
        for j in range(C):
            x0[j * R:(j + 1) * R, :b.x0[j].shape[1]] = b.x0[j]
        cost = np.repeat([(p.k + 1.0) * p.n_insns for p in b.programs], R)
        setups[bi] = dict(eng=eng, x0d=torch.from_numpy(x0).to(dev), rp=np.repeat(np.arange(C), R),
                          rs=np.arange(C * R), x0h=x0, ks=[p.k for p in b.programs], cost=cost)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def fit_step(su):
        """One step on the device-resident data: the whole beam (one GPU / replica) or this rank's
        share of it plus the all-gather of the per-candidate records (sharded)."""
        if mode == "sharded":
            return sharding.fit_sharded(su["eng"], su["ks"], R, su["x0d"], opts, cost=su["cost"],
                                        key_dtype=torch.float32 if score_dt == fitter.F32 else None)
        return None, su["eng"].fit(su["rp"], su["rs"], su["x0d"], opts)

    import gc
    gc.collect()
    gc.disable()   # a generation-2 collection over sympy's object graph stalls the host for ~50-100 ms
    for bi in warm:
        fit_step(setups[bi])
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    t_wall0 = time.time()
    launches0 = sum(s["eng"].launches for s in setups.values())

    # ---- value: device-resident steps ----
    claim_root = None
    if world > 1 and mode == "replicas":
        claim_root = [None]
        if rank == 0:
            import tempfile
            claim_root[0] = tempfile.mkdtemp(prefix="vsr_bench_")
        dist.broadcast_object_list(claim_root, src=0)
        claim_root = claim_root[0]
    n_job = args.steps if mode == "sharded" else world * args.steps
    job = [timed[i % args.steps] for i in range(n_job)]
    prof = [0.0, 0.0, 0.0, 0.0]
    mine, ev, results, winners = [], [], [], []

    def timed_loop(tag):
        claims = Claims(n_job, rank, world, claim_root, tag) if mode == "replicas" else None
        i_seq = 0
        while True:
            if mode == "replicas":
                i = claims.next()
                if i is None:
                    break
            else:
                if i_seq >= n_job:
                    break
                i, i_seq = i_seq, i_seq + 1
            su = setups[job[i]]
            su["eng"].set_profiling(True)
            flush.fill_(i & 0xFF)          # evict the previous step's data from L2 (untimed)
            if mode == "sharded":
                barrier()                  # every rank starts the beam together (untimed)
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            win, res = fit_step(su)
            b_.record()
            # a driver needs the result of one beam before it decodes the next
            torch.cuda.synchronize()
            mine.append(job[i])
            ev.append((a, b_))
            results.append(res)
            winners.append(win)
            p = su["eng"].read_profile()
            su["eng"].set_profiling(False)
            for q in range(4):
                prof[q] += p[q]

    timed_loop("v")
    barrier()
    t_wall1 = time.time()
    step_ms = [a.elapsed_time(b_) for a, b_ in ev]
    total_ms = float(sum(step_ms))
    print(f"rank {rank} [{mode}]: {len(mine)} steps, {total_ms:.1f} ms: "
          + " ".join(f"{beams[bi].name}:{m:.1f}" for bi, m in zip(mine, step_ms)), file=sys.stderr)
    launches = sum(s["eng"].launches for s in setups.values()) - launches0
    fit_ms, fit_n, score_ms = prof[0], prof[1], prof[2]
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, winners[-1], results[-1])

    # ---- algorithmic work of the timed steps (from the runs' own evaluation counts) ----
    flops = pevals = abytes = 0.0
    es = 4 if args.precision == "fp32" else 8
    for i, bi in enumerate(mine):
        b = beams[bi]
        info = results[i].info.cpu().numpy().reshape(C, R, 4)
        N = b.X.shape[0]
        for j, p in enumerate(b.programs):
            nf = info[j, :, 2]
            nfev = float(nf[nf > 0].sum())       # slots other ranks fitted read -1 here
            per_pass = (1 + p.k) if args.grad_mode == "dual" else 1
            pevals += nfev * N * per_pass
            flops += nfev * N * per_pass * p.flops
            d_used = bin(p.var_mask).count("1")
            abytes += nfev * (N * (d_used + 1) * es + (1 + p.k) * 8)

    # ---- sharded: the winners equal the one-GPU answer, bit for bit (checked outside the timing) ----
    shard_check = None
    if mode == "sharded":
        bad = 0
        n_chk = min(len(mine), 4)
        for i in range(n_chk):
            su = setups[mine[i]]
            full = su["eng"].fit(su["rp"], su["rs"], su["x0d"], opts)
            fm = full.final_mse.cpu().numpy().reshape(C, R)
            if score_dt == fitter.F32:
                fm = fm.astype(np.float32)
            lx = full.lastx.cpu().numpy().reshape(C, R, -1)
            w = winners[i].cpu().numpy()
            for c in range(C):
                want = 0 if np.all(np.isnan(fm[c])) else int(np.nanargmin(fm[c]))
                if int(w[c, 1]) != want or not np.array_equal(w[c, 3:3 + lx.shape[2]], lx[c, want], equal_nan=True):
                    bad += 1
                    if rank == 0:
                        print(f"sharded != one GPU: beam {beams[mine[i]].name} candidate {c}: restart {int(w[c, 1])} vs {want}, "
                              f"score {w[c, -1]!r} vs {fm[c, want]!r}, scores of all restarts {fm[c].tolist()}, "
                              f"lastx {w[c, 3:3 + lx.shape[2]].tolist()} vs {lx[c, want].tolist()}", file=sys.stderr)
        t_bad = torch.tensor([bad], device=dev)
        dist.all_reduce(t_bad)
        shard_check = {"beams_checked": n_chk, "candidates_differing_from_one_gpu": int(t_bad.item())}

    # ---- replicas extra at N > 1 (weak scaling of independent beams, no collective) ----
    replicas = None
    if world > 1 and mode == "sharded":
        mode_saved, mode = mode, "replicas"
        claim_root = [None]
        if rank == 0:
            import tempfile
            claim_root[0] = tempfile.mkdtemp(prefix="vsr_bench_")
        dist.broadcast_object_list(claim_root, src=0)
        claim_root = claim_root[0]
        n_job_saved, job_saved = n_job, job
        n_job = world * args.steps
        job = [timed[i % args.steps] for i in range(n_job)]
        keep = (list(mine), list(ev), list(results), list(winners))
        mine.clear(); ev.clear(); results.clear(); winners.clear()
        barrier()
        timed_loop("r")
        barrier()
        rep_ms = float(sum(a.elapsed_time(b_) for a, b_ in ev))
        t_rep = torch.tensor([rep_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t_rep, op=dist.ReduceOp.MAX)
        replicas = {"value": world * args.steps * C / (t_rep.item() / 1e3), "unit": "candidate-fits/s", "scaling": "weak",
                    "what": f"{world} x {args.steps} independent beams claimed from one pool, no data-path collective"}
        mine[:], ev[:], results[:], winners[:] = keep
        mode, n_job, job = mode_saved, n_job_saved, job_saved

    # ---- e2e_abi: host buffers through the C ABI (uploads + fit + read-back), one GPU's view ----
    abi_ms, h2d_abi, d2h_abi = 0.0, 0, 0
    if rank == 0:
        e2e_eng = fitter.Engine(dev)
        seq = list(warm[-min(2, len(warm)):]) + [timed[i] for i in range(min(args.steps, 8))]
        n_warm = len(seq) - min(args.steps, 8)
        for pos, bi in enumerate(seq):
            su, b = setups[bi], beams[bi]
            n_vars_i = su["eng"].n_vars
            Xc = np.ascontiguousarray(b.X[:, :n_vars_i].T.astype(np.float64))  # column-major host copy
            yh = np.ascontiguousarray(b.y.astype(np.float64))
            insn_off = np.zeros(C + 1, dtype=np.int32)
            imm_off = np.zeros(C + 1, dtype=np.int32)
            for j, p in enumerate(b.programs):
                insn_off[j + 1] = insn_off[j] + p.insns.shape[0]
                imm_off[j + 1] = imm_off[j] + p.imms.shape[0]
            insns = np.concatenate([p.insns for p in b.programs]).astype(np.uint64)
            imms = np.concatenate([p.imms for p in b.programs]).astype(np.float64)
            ks = np.asarray([p.k for p in b.programs], dtype=np.int32)
            flush.fill_(1)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            st = e2e_eng._stream()
            vp = lambda a: a.ctypes.data_as(fitter.ctypes.c_void_p)  # noqa: E731
            e2e_eng._check(e2e_eng.lib.vsr_upload_points(e2e_eng._h, vp(Xc), vp(yh), Xc.shape[1], Xc.shape[1],
                                                         Xc.shape[0], fitter.F64, st))
            e2e_eng._check(e2e_eng.lib.vsr_upload_programs(e2e_eng._h, vp(insns), vp(insn_off), vp(imms), vp(imm_off),
                                                           vp(ks), C, st))
            e2e_eng._points = {fitter.F64: None}   # the points went in through the C ABI, not through set_points
            o64 = fitter.default_opts(grad_mode=opts.grad_mode, eval_dtype=fitter.F64, score_dtype=fitter.F64,
                                      warps_per_run=args.warps)
            out = e2e_eng.fit_host(su["rp"], su["rs"], su["x0h"], o64)
            dt = (time.perf_counter() - t0) * 1e3
            if pos >= n_warm:
                abi_ms += dt
                h2d_abi = (Xc.nbytes + yh.nbytes + insns.nbytes + imms.nbytes + insn_off.nbytes + imm_off.nbytes
                           + ks.nbytes + su["x0h"].nbytes + su["rp"].nbytes // 2 + su["rs"].nbytes // 2)
                d2h_abi = sum(v.nbytes for v in out.values())
        abi_n = min(args.steps, 8)
        e2e_eng.close()

    # ---- e2e: the Python entry point a driver calls (tokens + HOST tensors in, dict out) ----
    api_ms, api_n, h2d, d2h = 0.0, 0, 0, 0
    if not args.no_api:
        from src.visymre.architectures import bfgs as vbfgs
        from src.visymre.architectures.model import refine_hypotheses
        from src.visymre.workloads import generator as g
        td = g.make_test_data()
        cfg = g.make_cfg(R, C, grad_mode=args.grad_mode, precision=args.precision, shard=(mode == "sharded"))
        hostpool.warm()                       # the worker processes exist before the first call, as in a driver
        seq = list(warm) + list(timed)            # every warm-up step goes through the entry point too
        n_warm = len(seq) - len(timed)
        barrier()
        for pos, bi in enumerate(seq):
            b = beams[bi]
            Xh = torch.from_numpy(np.ascontiguousarray(b.X[None])).pin_memory()
            yh = torch.from_numpy(np.ascontiguousarray(b.y)).reshape(1, -1, 1).pin_memory()
            hyps = [(-float(j), t) for j, t in enumerate(b.tokens)]
            vbfgs._COMPILED.clear()           # cold compile cache: every step compiles its 64 skeletons
            flush.fill_(2)
            barrier()
            t0 = time.perf_counter()
            out = refine_hypotheses(hyps, Xh.to(dev, non_blocking=True), yh.to(dev, non_blocking=True), cfg, td, x0=b.x0)
            best = out["best_bfgs_preds"][0]  # the string a driver sympifies next (e.g. Feynman_test.py:78)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) * 1e3
            if rank == 0:
                print(f"e2e_ms {b.name}:{dt:.1f} " + " ".join(f"{k}={v:.1f}" for k, v in vbfgs.LAST_TIMING.items()), file=sys.stderr)
            if pos >= n_warm:
                api_ms += dt
                api_n += len(out["all_bfgs_loss"])
                h2d = Xh.numel() * Xh.element_size() + yh.numel() * yh.element_size() + sum(x.nbytes for x in b.x0)
                kmx = max(1, max(p.k for p in b.programs))   # scores + last points read back (records when sharded)
                d2h = C * 8 * (4 + kmx) if mode == "sharded" else C * R * 8 * (1 + kmx)
            del best

    gc.enable()   # (off since the first timed loop: this process holds every beam's sympy trees, and a
    #               generation-2 collection over them stalls a step for 50-100 ms; a driver holds one beam's)

    # ---- max over ranks ----
    t = torch.tensor([total_ms, api_ms], dtype=torch.float64, device=dev)
    agg = torch.tensor([float(launches), flops, pevals, abytes, fit_ms, fit_n, score_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(agg, op=dist.ReduceOp.SUM)
    total_ms_max, api_ms_max = t.tolist()
    launches_all, flops_all, pevals_all, abytes_all, fit_ms_all, fit_n_all, score_ms_all = agg.tolist()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:  # noqa: BLE001
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        fp = {}
        try:
            fp = json.load(open(os.path.join(ROOT, "profiles", "fp_peaks.json")))
        except Exception:  # noqa: BLE001
            pass
        key = "fp32_tflops" if args.precision == "fp32" else "fp64_tflops"
        sm_max = (clocks or {}).get("sm_max_mhz") or 1965.0
        derived = 148 * (128 if args.precision == "fp32" else 64) * 2 * sm_max * 1e6 / 1e12
        fp_peak = fp.get(key, derived)
        fp_src = "measured (profiles/fp_peaks.json)" if key in fp else f"derived: 148 SMs x lanes x 2 x {sm_max:.0f} MHz"
        cap = None
        for name in ("r02_ncu_capture.json", "r01_ncu_capture.json"):
            try:   # DRAM bytes of one launch of the dominant kernel, from the committed ncu capture
                cap = json.load(open(os.path.join(ROOT, "profiles", name)))
                break
            except Exception:  # noqa: BLE001
                pass
        traffic = (cap["dram_bytes_read"] + cap["dram_bytes_write"]) if cap else None
        fit_s = fit_ms_all / 1e3 / world      # per-rank average kernel time
        n_launch = max(1.0, fit_n_all)
        achieved_tf = flops_all / world / max(fit_s, 1e-9) / 1e12
        achieved_gbs = abytes_all / world / max(fit_s, 1e-9) / 1e9
        n_steps_job = args.steps if mode == "sharded" else world * args.steps
        value = n_steps_job * C / (total_ms_max / 1e3)
        line = {
            "metric": "candidate_fits_per_sec", "value": value, "unit": "candidate-fits/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms_max / args.steps, "higher_is_better": True,
            "scaling": "strong" if mode == "sharded" else "weak",
            "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "f64", "data": "synthetic",
            "config": workload_config(args),
            "partition": ("one beam's candidate x restart runs dealt over the ranks + one all-gather of per-candidate "
                          "records per step (engine/sharding.py)") if mode == "sharded" else "whole beams per GPU",
            "point_evals_per_sec": pevals_all / (total_ms_max / 1e3),
            "e2e": ({"value": n_steps_job * C / (api_ms_max / 1e3) if mode == "sharded" else world * api_n / (api_ms_max / 1e3),
                     "unit": "candidate-fits/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                     "path": "refine_hypotheses(token ids, pinned host X / y, cfg, test_data) -> dict: H2D copies, skeleton "
                             "compilation (cold cache, host worker pool), fit (sharded over the ranks when N > 1), prune, "
                             "winner formatting, D2H read", "host_workers": hostpool.default_workers()}
                    if api_ms_max else None),
            "e2e_abi": {"value": abi_n * C / (abi_ms / 1e3) if abi_ms else None, "unit": "candidate-fits/s",
                        "h2d_bytes_per_step": int(h2d_abi), "d2h_bytes_per_step": int(d2h_abi), "n_gpus": 1,
                        "path": "vsr_upload_points + vsr_upload_programs + vsr_fit_host (C ABI, host buffers, "
                                "precompiled bytecode)"},
            "gpu_launches": int(launches_all),
            "clocks": clocks,
            "roofline": {
                "kernel": "vsr::fit_kernel", "bound": "fp64" if args.precision == "fp64" else "fp32",
                "achieved": achieved_tf, "peak": fp_peak, "unit": "TFLOP/s", "frac": achieved_tf / fp_peak,
                "peak_source": fp_src,
                "launch_ms": fit_ms_all / n_launch, "share_of_step": fit_ms_all / world / (total_ms_max or 1),
                "traffic": traffic, "traffic_source": (cap or {}).get("source"),
                "ncu": {k: cap[k] for k in ("kernel", "issue_active_pct", "pipe_fp64_pct", "pipe_alu_pct",
                                            "pipe_lsu_pct", "duration_ms") if k in cap} if cap else None,
                "hbm": {"achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak,
                        "peak_source": hbm_src},
                "note": "algorithmic flops per SURVEY 8d (1 per arithmetic node, transcendental = 1); the kernel "
                        "is issue / FP-pipe bound, not HBM bound: see profiles/ for ncu pipe utilisation"},
        }
        if shard_check is not None:
            line["sharded_check"] = shard_check
        if replicas is not None:
            line["replicas"] = replicas
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline([beams[bi] for bi in timed], args, args.cpu_seconds)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
