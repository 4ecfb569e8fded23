"""Generate tests/golden/ref_low.json (+ ref_low_points.npz) from the UNMODIFIED reference on
BASELINE config 1: rows of scripts/low_benchmarks.csv, N = 500 points, R = 10 restarts -- the only
configuration the as-is reference can run at full size (SURVEY.md section 8d).

Run with VISYMRE_REFERENCE naming a reference checkout:  python oracle/make_golden_low.py [rows] [candidates per row]

Two processes, because the product package and the reference are both a top-level package
named ``src``:
  stage A (this repo's workload generator)  beams of config 1 -> a temporary pickle
  stage B (oracle/ref_harness.py)           the reference's own bfgs() on every case, every
                                            ``minimize`` call recorded (the reference source is
                                            not modified: the name is wrapped inside its module)
TEST INFRASTRUCTURE: nothing under vision-sr_b200/ imports this.
"""
import json
import os
import pickle
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT_JSON = os.path.join(ROOT, "tests", "golden", "ref_low.json")
OUT_NPZ = os.path.join(ROOT, "tests", "golden", "ref_low_points.npz")
N_POINTS, N_RESTARTS, BEAM = 500, 10, 16

STAGE_A = r"""
import pickle, sys, warnings
warnings.filterwarnings("ignore")
sys.path.insert(0, {pkg!r})
from src.visymre.workloads import generator as g
beams, td = g.low_beams(n_points={n}, n_cand={beam}, n_restarts={r})
out = [dict(name=b.name, truth=b.truth, X=b.X, y=b.y, tokens=b.tokens, x0=b.x0) for b in beams]
pickle.dump(out, open({dst!r}, "wb"))
"""


def _run_case(job):
    """Stage B worker: one candidate through the reference's bfgs() and bfgs_wrapper()."""
    import warnings
    warnings.filterwarnings("ignore")
    import numpy as np
    import torch
    from types import SimpleNamespace as NS
    sys.path.insert(0, ROOT)
    from oracle import ref_harness
    ref_bfgs, ref_model, td = ref_harness.load()
    name, cand, tokens, X, y, x0 = job
    cfg = NS(bfgs=NS(n_restarts=len(x0), add_coefficients_if_not_existing=False, idx_remove=False,
                     normalization_type="MSE", stop_time=1e9))
    log = []
    real_minimize = ref_bfgs.minimize

    def recording_minimize(fun, start, **kw):
        res = real_minimize(fun, start, **kw)
        log.append(dict(x0=np.asarray(start).tolist(), res_x=res.x.tolist(), fun=float(res.fun),
                        nit=int(res.nit), nfev=int(res.nfev), status=int(res.status)))
        return res

    # the reference draws x0 = np.random.randn(k) * 10 per restart (bfgs.py:103): feed it ours
    draws = [np.asarray(r, dtype=np.float64) / 10.0 for r in x0]
    real_randn = np.random.randn
    state = {"i": 0}

    def fed_randn(*shape):
        k = shape[0] if shape else 1
        i = state["i"]
        state["i"] += 1
        if i < len(draws):
            assert len(draws[i]) == k, (len(draws[i]), k)
            return draws[i].copy()
        return real_randn(*shape)

    rec = dict(row=name, cand=cand, tokens=[int(t) for t in tokens], x0=np.asarray(x0).tolist())
    ref_bfgs.minimize = recording_minimize
    ref_bfgs.np.random.randn = fed_randn
    t0 = time.time()
    try:
        expr_str, consts, loss, skel = ref_bfgs.bfgs(list(tokens), torch.tensor(X[None]), torch.tensor(y), cfg, td)
        rec.update(raised=None, best_expr_str=expr_str, best_consts=[float(c) for c in consts],
                   best_loss=float(loss), skeleton=skel)
    except Exception as exc:  # noqa: BLE001 -- the wrapper's contract: (None, nan, tokens)
        rec.update(raised=type(exc).__name__)
    finally:
        ref_bfgs.minimize = real_minimize
        ref_bfgs.np.random.randn = real_randn
    rec["minimize_calls"] = log
    rec["wall_s"] = round(time.time() - t0, 2)
    return rec


def main():
    import numpy as np
    n_rows = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    per_row = int(sys.argv[2]) if len(sys.argv) > 2 else 2
    with tempfile.TemporaryDirectory() as tmp:
        dst = os.path.join(tmp, "beams.pkl")
        code = STAGE_A.format(pkg=os.path.join(ROOT, "vision-sr_b200"), n=N_POINTS, beam=BEAM, r=N_RESTARTS, dst=dst)
        subprocess.check_call([sys.executable, "-c", code], cwd=tmp)
        beams = pickle.load(open(dst, "rb"))
    # a spread of rows over the table (1- and 2-variable rows both)
    pick = [beams[i] for i in np.linspace(0, len(beams) - 1, n_rows).astype(int)]
    jobs, points = [], {}
    for b in pick:
        points[b["name"] + "/X"] = b["X"][:, :2].copy()
        points[b["name"] + "/y"] = b["y"]
        for c in ([0, 3, 7, 11][:per_row]):
            jobs.append((b["name"], c, b["tokens"][c], b["X"], b["y"], b["x0"][c]))
    from concurrent.futures import ProcessPoolExecutor
    t0 = time.time()
    with ProcessPoolExecutor(min(os.cpu_count() or 2, 8)) as ex:
        cases = list(ex.map(_run_case, jobs))
    for c in cases:
        print(f"{c['row']:14s} cand {c['cand']:2d} {c['wall_s']:7.1f}s raised={c.get('raised')} "
              f"loss={c.get('best_loss')} expr={c.get('best_expr_str')}")
    import scipy
    import sympy
    import torch
    out = {"generator": "oracle/make_golden_low.py", "reference": "aidalee123/Vision-SR (unmodified)",
           "config": "BASELINE config 1: low_benchmarks.csv rows, N=500, R=10, fp64",
           "versions": {"numpy": np.__version__, "torch": torch.__version__, "sympy": sympy.__version__,
                        "scipy": scipy.__version__},
           "n_points": N_POINTS, "n_restarts": N_RESTARTS, "points": os.path.basename(OUT_NPZ),
           "cases": cases}
    with open(OUT_JSON, "w") as fh:
        # a loss / constant the reference produced as a complex number (sqrt/log of a negative
        # constant-free sub-tree folded by sympy) is kept as {"complex": [re, im]}
        json.dump(out, fh, default=lambda o: {"complex": [o.real, o.imag]} if isinstance(o, complex) else float(o))
    np.savez(OUT_NPZ, **points)
    print(f"wrote {OUT_JSON} ({os.path.getsize(OUT_JSON)} B), {OUT_NPZ} ({os.path.getsize(OUT_NPZ)} B), "
          f"{len(cases)} cases in {time.time() - t0:.0f} s")


if __name__ == "__main__":
    main()
