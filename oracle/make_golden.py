"""Generate tests/golden/ref_bfgs.json from the UNMODIFIED reference.

Run with VISYMRE_REFERENCE naming a reference checkout:  python oracle/make_golden.py
It imports the reference (VISYMRE_REFERENCE) through oracle/ref_harness.py, runs the reference's own
``bfgs()`` / ``bfgs_wrapper()`` on small seeded cases and records inputs, outputs and
per-restart optimiser facts (captured by wrapping the ``minimize`` name inside the
reference module; the reference source is not modified).
"""
import json
import os
import sys
import time
from types import SimpleNamespace as NS

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_harness  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                   "tests", "golden", "ref_bfgs.json")


def cfg_of(R, norm="MSE", idx_remove=False):
    return NS(bfgs=NS(n_restarts=R, add_coefficients_if_not_existing=False,
                      idx_remove=idx_remove, normalization_type=norm, stop_time=1e9))


def points(seed, n, ranges, fn, dtype=np.float64):
    rng = np.random.RandomState(seed)
    X = np.zeros((n, 10), dtype=np.float64)
    for j, (lo, hi) in enumerate(ranges):
        X[:, j] = rng.uniform(lo, hi, n)
    y = fn(*[X[:, j] for j in range(len(ranges))])
    return X.astype(dtype), y.astype(dtype)


# name, prefix words, ranges, ground truth, N, R, extra
CASES = [
    dict(name="affine_sin", words="add c mul c sin x_1", ranges=[(-3, 3)],
         fn=lambda a: 0.75 + 2.5 * np.sin(a), n=60, R=3),
    dict(name="nguyen1c", words="add mul c x_1 add mul c pow x_1 2 mul c pow x_1 3",
         ranges=[(-1, 1)], fn=lambda a: a + a**2 + a**3, n=80, R=4),
    dict(name="nguyen10c", words="mul cos mul c x_1 sin mul c x_1", ranges=[(0, 2)],
         fn=lambda a: np.cos(1.3 * a) * np.sin(0.7 * a), n=80, R=4),
    dict(name="korns12", words="add c mul mul c cos mul c pow x_1 3 sin mul c x_2",
         ranges=[(-1.5, 1.5), (-3, 3)],
         fn=lambda a, b: 2 - 2.1 * np.cos(0.9 * a**3) * np.sin(1.3 * b), n=100, R=4),
    dict(name="exp_log_sqrt", words="add mul c exp mul c x_1 ln add c sqrt x_2",
         ranges=[(0, 2), (0.5, 4)],
         fn=lambda a, b: 1.5 * np.exp(-0.8 * a) + np.log(2.0 + np.sqrt(b)), n=80, R=4),
    dict(name="pow_const_exponent", words="mul c pow x_1 c", ranges=[(0.5, 3)],
         fn=lambda a: 1.7 * a**2.5, n=60, R=4),
    dict(name="no_constants", words="add sin x_1 mul x_1 x_2", ranges=[(-2, 2), (-2, 2)],
         fn=lambda a, b: np.sin(a) + a * b + 0.01, n=40, R=2),
    dict(name="one_const_div_shift", words="div c x_2", ranges=[(0, 0), (1, 3)],
         fn=lambda a, b: 3.0 / b, n=50, R=3, note="x_2 is renamed x_1 (bfgs.py:11-21)"),
    dict(name="nmse", words="add c mul c x_1", ranges=[(-2, 2)], fn=lambda a: 4 + 3 * a,
         n=50, R=3, norm="NMSE"),
    dict(name="prune_small", words="add mul c x_1 c", ranges=[(-2, 2)], fn=lambda a: 2.0 * a,
         n=50, R=3),
    dict(name="fp32_points", words="add c mul c cos x_1", ranges=[(-3, 3)],
         fn=lambda a: 0.5 - 1.25 * np.cos(a), n=60, R=3, dtype="float32"),
    dict(name="tan_abs_asin", words="add mul c tan x_1 mul c asin mul c abs x_2",
         ranges=[(-1, 1), (-1, 1)],
         fn=lambda a, b: 0.4 * np.tan(a) + 1.2 * np.arcsin(0.8 * np.abs(b)), n=80, R=4),
    dict(name="exp_sqrt_ok", words="add mul c exp mul c x_1 mul c sqrt x_2",
         ranges=[(0, 2), (0.5, 4)],
         fn=lambda a, b: 1.5 * np.exp(-0.8 * a) + 0.6 * np.sqrt(b), n=80, R=4),
    dict(name="tan_asin_ok", words="add mul c tan x_1 mul c asin x_2",
         ranges=[(-1, 1), (-1, 1)],
         fn=lambda a, b: 0.4 * np.tan(a) + 1.2 * np.arcsin(b), n=80, R=3),
    dict(name="domain_violation", words="add c ln sub x_1 c", ranges=[(0.5, 3)],
         fn=lambda a: 0.3 + np.log(a + 0.25), n=60, R=4,
         note="ln of a negative argument for many c: 1e6 penalty plateau"),
    dict(name="invalid_prefix", words="add c", ranges=[(-1, 1)], fn=lambda a: a, n=20, R=2,
         note="incomplete tree: bfgs() raises, bfgs_wrapper returns (None, nan)"),
    dict(name="idx_remove_all_kept", words="add c mul c x_1", ranges=[(-2, 2)],
         fn=lambda a: 1 + 2 * a, n=40, R=2, idx_remove=True),
]


def main():
    ref_bfgs, ref_model, td = ref_harness.load()
    w2i = td.word2id
    out = {"generator": "oracle/make_golden.py", "reference": "aidalee123/Vision-SR (unmodified)",
           "versions": {"numpy": np.__version__, "torch": torch.__version__,
                        "sympy": __import__("sympy").__version__,
                        "scipy": __import__("scipy").__version__},
           "word2id": {k: int(v) for k, v in w2i.items()},
           "total_variables": list(td.total_variables), "cases": []}
    real_minimize = ref_bfgs.minimize
    for ci, case in enumerate(CASES):
        words = case["words"].split()
        tokens = [w2i["S"]] + [w2i[w] for w in words] + [w2i["F"]]
        dtype = np.dtype(case.get("dtype", "float64"))
        X, y = points(100 + ci, case["n"], case["ranges"], case["fn"], dtype)
        cfg = cfg_of(case["R"], case.get("norm", "MSE"), case.get("idx_remove", False))
        log = []

        def recording_minimize(fun, x0, **kw):
            res = real_minimize(fun, x0, **kw)
            log.append(dict(x0=np.asarray(x0).tolist(), res_x=res.x.tolist(), fun=float(res.fun),
                            nit=int(res.nit), nfev=int(res.nfev), status=int(res.status)))
            return res

        ref_bfgs.minimize = recording_minimize
        np.random.seed(1000 + ci)
        t0 = time.time()
        rec = dict(name=case["name"], words=words, tokens=tokens, dtype=str(dtype),
                   n=case["n"], R=case["R"], norm=case.get("norm", "MSE"),
                   idx_remove=case.get("idx_remove", False), note=case.get("note", ""),
                   seed=1000 + ci, X=X[:, :len(case["ranges"])].tolist(), y=y.tolist())
        try:
            expr_str, consts, loss, skel = ref_bfgs.bfgs(
                list(tokens), torch.tensor(X[None]), torch.tensor(y), cfg, td)
            rec.update(raised=None, best_expr_str=expr_str,
                       best_consts=[float(c) for c in consts], best_loss=float(loss),
                       skeleton=skel)
        except Exception as exc:  # the wrapper's contract: (None, nan, tokens)
            rec.update(raised=type(exc).__name__)
        finally:
            ref_bfgs.minimize = real_minimize
        rec["minimize_calls"] = log
        rec["wall_s"] = round(time.time() - t0, 3)
        if ref_model is not None:
            np.random.seed(1000 + ci)
            wr = ref_model.bfgs_wrapper((list(tokens), torch.tensor(X[None]), torch.tensor(y), cfg, td))
            rec["wrapper"] = [wr[0], None if wr[1] != wr[1] else float(wr[1])]
        print(f"{case['name']:24s} {rec['wall_s']:7.2f}s raised={rec.get('raised')} "
              f"loss={rec.get('best_loss')} expr={rec.get('best_expr_str')}")
        out["cases"].append(rec)
    with open(OUT, "w") as fh:
        json.dump(out, fh)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
