"""Worker processes for the sympy half of the refinement (host side).

What is left on the host once the fits run on the GPU is sympy: token ids -> infix -> ``sympify``
-> bytecode for every candidate (3-8 ms each) and ``str(expr with the fitted constants)`` for
every candidate (2-5 ms each, ``bfgs.py:120-124``).  The reference spends its 20 pool processes
(``model.py:490``) on whole ``bfgs()`` calls; here the same kind of pool does only this symbolic
work, in chunks, while the parent drives the GPU.

The pool is created on first use (``fork``, as the reference's pool is) and lives for the process.  ``VSR_HOST_WORKERS=0``
(or ``cfg.bfgs.host_workers = 0``) keeps everything in-process.
"""
import atexit
import os
import sys

_POOL = None
_POOL_N = 0


def default_workers():
    env = os.environ.get("VSR_HOST_WORKERS")
    if env is not None:
        return max(0, int(env))
    world = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1"))))
    return max(0, min(16, (os.cpu_count() or 2) // world - 1))


def _init_worker(paths):
    import warnings
    warnings.filterwarnings("ignore")
    for p in reversed(paths):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ["VSR_HOST_WORKERS"] = "0"          # workers never start pools of their own
    os.environ["CUDA_VISIBLE_DEVICES"] = ""       # ... and never touch the GPU
    from ..architectures import bfgs  # noqa: F401  (sympy and the compiler, imported once)
    # a full collection over sympy's caches stalls a task for 50-100 ms -- and the whole beam waits for
    # its slowest task: park what exists now in the permanent generation and collect the young
    # generation rarely (sympy's trees are acyclic; its caches are bounded)
    import gc
    gc.collect()
    gc.freeze()
    gc.set_threshold(50_000, 50, 1000)


def get_pool(n):
    """A process-wide pool of n workers (None when n <= 0)."""
    global _POOL, _POOL_N
    if n <= 0:
        return None
    if _POOL is None or _POOL_N != n:
        shutdown()
        import multiprocessing as mp
        from concurrent.futures import ProcessPoolExecutor
        pkg_root = os.path.dirname(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
        paths = [pkg_root] + [p for p in sys.path if p]
        # `fork` like the reference's own pool (model.py:490, created after the model sits on the
        # GPU): the workers only ever run sympy.  forkserver / spawn re-import the caller's
        # __main__, which breaks driver scripts without a __main__ guard; VSR_HOST_START selects them.
        ctx = mp.get_context(os.environ.get("VSR_HOST_START", "fork"))
        _POOL = ProcessPoolExecutor(n, mp_context=ctx, initializer=_init_worker, initargs=(paths,))
        _POOL_N = n
    return _POOL


def warm(n=None):
    """Start the workers and make them import sympy now (first call costs seconds)."""
    n = default_workers() if n is None else n
    pool = get_pool(n)
    if pool is not None:
        list(pool.map(_noop, range(2 * n)))
    # ... and this process prints one winner per call: sympy imports printers and evaluation rules of a
    # function class the first time it meets one (tens of ms each)
    try:
        import sympy as sp
        from ..architectures import bfgs as vb
        from .compiler import parse_skeleton
        expr = parse_skeleton("((c0)+((c1)*(sin((c2)*(x_1)))))+((cos(x_2))*(tan((c3)+(x_3))))+((exp((c4)*(x_1)))/(ln(Abs((c5)+(x_2)))))"
                              "+((sqrt(Abs(x_1)))*(asin((c6)/((10)+(Abs(x_1))))))+(((x_1)**(c7))*((pi)**(2)))")
        str(vb._substitute(expr, [sp.Symbol(f"c{i}") for i in range(8)], [0.5, -1.25, 3.0, 1e-3, 2.5e4, -7.0, 0.25, 1.5]))
    except Exception:  # noqa: BLE001 -- warming only
        pass
    return n


def _noop(i):
    return i


def shutdown():
    global _POOL, _POOL_N
    if _POOL is not None:
        _POOL.shutdown(wait=False, cancel_futures=True)
    _POOL, _POOL_N = None, 0


atexit.register(shutdown)


# ---- tasks (run in the workers) -------------------------------------------------------------------
def compile_chunk(job):
    """[(tokens, ...)] -> [(expr, k, Program) | Exception] for a chunk of candidates."""
    from ..architectures import bfgs as vb
    toks_list, cfg_bits, id2word, variables = job
    from types import SimpleNamespace as NS
    cfg = NS(bfgs=NS(add_coefficients_if_not_existing=cfg_bits[0]))
    td = NS(id2word=id2word, total_variables=variables)
    out = []
    for toks in toks_list:
        try:
            out.append(vb.compile_tokens(toks, cfg, td, variables))
        except Exception as exc:  # noqa: BLE001 -- per candidate, like bfgs_wrapper (model.py:15-19)
            out.append(_portable(exc))
    return out


def prune_task(job):
    """(Program, indices of its small constants, variables) -> architectures/bfgs.py:prepare_prune."""
    from ..architectures import bfgs as vb
    prog, small, variables = job
    return vb.prepare_prune(prog, small, variables)


def format_chunk(job):
    """[(skeleton string, [symbol order], [values])] -> [str(expression with the numbers in)]."""
    from ..architectures import bfgs as vb
    import sympy as sp
    out = []
    for expr, names, vals in job:
        try:
            out.append(str(vb._substitute(sp.sympify(expr), [sp.Symbol(n) for n in names], vals)))
        except Exception as exc:  # noqa: BLE001
            out.append(_portable(exc))
    return out


def compile_skeletons(job):
    """[(skeleton string, k)] -> [Program | Exception], variables x_1..x_10 (uncertainty.covariances)."""
    from .compiler import compile_skeleton
    variables = [f"x_{i}" for i in range(1, 11)]
    out = []
    for expr, k in job:
        try:
            out.append(compile_skeleton(expr, k, variables))
        except Exception as exc:  # noqa: BLE001 -- raised again in the parent
            out.append(_portable(exc))
    return out


def _portable(exc):
    """Exceptions cross the process boundary by pickle; some (sympy's) do not survive it."""
    import pickle
    try:
        pickle.loads(pickle.dumps(exc))
        return exc
    except Exception:  # noqa: BLE001
        return RuntimeError(f"{type(exc).__name__}: {exc}")
