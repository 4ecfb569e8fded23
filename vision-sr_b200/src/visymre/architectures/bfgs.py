"""Constant fitting of beam candidates on the B200 (drop-in for the reference module).

Same entry point, arguments, return value and quirks as reference
``src/visymre/architectures/bfgs.py`` (``bfgs`` :42-215; the step labels Q1..Q13 below
are SURVEY.md section 3.3), but nothing is evaluated on the CPU: the skeleton is
compiled to bytecode (``engine/compiler.py``) and every restart of every candidate is
optimised by one CUDA launch (``csrc/vsr_kernels.cuh``).  ``bfgs_batch`` is the native
shape of the work -- all candidates of a beam at once -- and ``bfgs`` is the
single-candidate view of it that ``hlsc.py:410`` and ``model.py:16`` call.

Extra, optional knobs read with ``getattr(cfg.bfgs, name, default)`` (the reference's
config.yaml does not have them, so drivers keep working unchanged):
  grad_mode   "dual" (default; exact forward-mode gradients) or "fd" (scipy's 2-point
              forward differences, reproduces the reference's trajectories)
  precision   "fp64" (default, what the reference's loss uses) or "fp32"
  prune_threshold / prune_tolerance   as in the reference (bfgs.py:143-144)
  devices     None (default: one engine on the current device), "all" (every visible CUDA device) or
              a list of device indices / torch.devices, the first one the home device: the beam's
              runs are dealt over one engine per entry in this process (``resolve_devices``)
"""
import re

import numpy as np
import sympy as sp
import torch

from ..dataset.generator import Generator
from ..engine import fitter, hostpool, isa, sharding
from ..engine.compiler import CompileError, compile_sympy, parse_skeleton
from . import data


def replace_illegal_variables(expr, max_var=5):
    """Q4 (bfgs.py:11-21): rename x_i to x_{i-1} when x_{i-1} does not occur, i = 2..5."""
    present = set(re.findall(r"x_\d+", expr))
    if "x_0" in present:
        raise ValueError(f"illegal variable x_0 in expression:\n{expr}")
    fixed = expr
    for i in range(2, max_var + 1):
        if f"x_{i}" in present and f"x_{i - 1}" not in present:
            fixed = re.sub(rf"\bx_{i}\b", f"x_{i - 1}", fixed)
    return fixed


def _opt(cfg, name, default=None):
    b = cfg.bfgs if hasattr(cfg, "bfgs") else cfg["bfgs"]
    try:
        return getattr(b, name)
    except (AttributeError, KeyError):
        pass
    try:
        return b[name]
    except (KeyError, TypeError, IndexError):
        return default


def resolve_devices(cfg):
    """``cfg.bfgs.devices`` as a list of CUDA ``torch.device``s (the first one is the home device, where
    the inputs and the fit's results live), or None when it is unset or None.

    ``"all"``: every visible CUDA device.  A list of device indices or devices: those, in that order; an
    entry may repeat, which puts a further engine on that device.  More than one device in a process that
    has a torch.distributed process group is a ``ValueError``: the runs are dealt over the ranks there
    (``bfgs.shard``), and dealing them over the ranks and the devices at once is not defined."""
    spec = _opt(cfg, "devices", None)
    if spec is None:
        return None
    if isinstance(spec, str) and spec.strip().lower() == "all":
        devs = [torch.device("cuda", i) for i in range(torch.cuda.device_count())]
    else:
        items = [spec] if isinstance(spec, (int, str, torch.device)) else list(spec)
        devs = []
        for d in items:
            try:
                d = torch.device(d) if isinstance(d, (str, torch.device)) else torch.device("cuda", int(d))
            except (RuntimeError, TypeError, ValueError) as exc:
                raise ValueError(f"cfg.bfgs.devices: {d!r} is not a CUDA device") from exc
            if d.type != "cuda":
                raise ValueError(f"cfg.bfgs.devices: {d} is not a CUDA device (the engine has no CPU path)")
            devs.append(d)
    if len(devs) > 1 and _process_group():
        raise ValueError("cfg.bfgs.devices names several devices in a process with a torch.distributed process "
                         "group: deal the runs over the ranks (bfgs.shard) or over the devices of one process, "
                         "not both")
    if not devs:
        raise ValueError(f"cfg.bfgs.devices = {spec!r}: no CUDA device")
    n = torch.cuda.device_count()
    devs = [torch.device("cuda", torch.cuda.current_device()) if d.index is None else d for d in devs]
    for d in devs:
        if d.index >= n:
            raise ValueError(f"cfg.bfgs.devices: {d} does not exist ({n} CUDA devices visible)")
    return devs


def _process_group():
    import torch.distributed as dist
    return dist.is_available() and dist.is_initialized()


def skeleton_string(pred_str, cfg, test_data):
    """Q1-Q5: token ids (leading S included) -> (c-named infix string, k)."""
    if isinstance(pred_str, list):
        pred_str = np.array(pred_str)
    if isinstance(pred_str, torch.Tensor):
        pred_str = pred_str.detach().cpu().numpy()
    ids = np.asarray(pred_str)[1:].tolist()
    raw = data.de_tokenize(ids, test_data.id2word)
    if _opt(cfg, "add_coefficients_if_not_existing", False) and "constant" not in raw:
        # The reference's branch (bfgs.py:52-64) hands the tuple returned by
        # constants_to_placeholder to sympy_to_prefix and always raises
        # UnknownSymPyOperator; its wrapper then drops the candidate.  Same outcome here.
        from ..dataset.generator import UnknownSymPyOperator
        raise UnknownSymPyOperator("add_coefficients_if_not_existing is broken in the reference")
    candidate = Generator.prefix_to_infix(raw, coefficients=["constant"],
                                          variables=test_data.total_variables)
    candidate = replace_illegal_variables(candidate.format(constant="constant"))
    k = candidate.count("constant")
    expr = candidate
    for i in range(k):
        expr = expr.replace("constant", f"c{i}", 1)
    return expr, k


class _Candidate:
    __slots__ = ("expr", "k", "prog", "error")

    def __init__(self):
        self.expr = self.prog = self.error = None
        self.k = 0


def _engine_opts(cfg, scale, eval_dtype, score_dtype):
    mode = str(_opt(cfg, "grad_mode", "dual")).lower()
    return fitter.default_opts(
        loss_scale=scale,
        stop_time=float(_opt(cfg, "stop_time", 1e9)),
        grad_mode=isa.GRAD_MODE["VSR_GRAD_FD" if mode == "fd" else "VSR_GRAD_DUAL"],
        eval_dtype=eval_dtype, score_dtype=score_dtype)


def _substitute(expr, symbols, values):
    """bfgs.py:120-124: put the numbers in.

    The reference re-sympifies its string and calls ``.replace(symbol, value)`` once per
    constant (~10 ms a time).  ``xreplace`` on the already-sympified skeleton, one constant
    after the other in the same order, rebuilds the same trees -- the values go through the
    same ``sympify`` conversion and the Floats combine in the same order -- and prints the
    same string (tests/test_host_path.py checks this on the workload's candidates)."""
    final = sp.sympify(expr)
    for s, v in zip(symbols, values):
        final = final.xreplace({s: sp.sympify(v)})
    return final


def _substitute_like_reference(expr_str, symbols, values):
    """The reference's own sequence, kept for the equivalence test."""
    final = expr_str
    for s, v in zip(symbols, values):
        final = sp.sympify(final).replace(s, v)
    return final


def prepare_prune(prog, small, variables):
    """Symbolic half of Q12 (bfgs.py:156-178) for one candidate whose best constants ``small`` are
    below the threshold: ``(zero_idx, rest, pruned Program | None, constant-free Program | Exception
    | None)``, or None when nothing is pruned (or the pruned skeleton cannot be lowered: the unpruned
    fit stays)."""
    csyms = [sp.Symbol(f"c{i}") for i in range(prog.k)]
    zero_idx = []
    for i in small:
        if prog.k == 1 and not _derivative_is_constant(prog.expr, csyms[i]):
            continue
        zero_idx.append(i)
    if not zero_idx:
        return None
    rest = [i for i in range(prog.k) if i not in zero_idx]
    if rest:
        # like the reference (bfgs.py:161-168): zeros substituted, the remaining symbols keep their
        # names and become arguments in their order (no renaming, so no re-canonicalisation)
        pruned = prog.expr.subs({csyms[i]: 0.0 for i in zero_idx})
        try:
            out = compile_sympy(pruned, len(rest), variables, slots={i: j for j, i in enumerate(rest)})
        except CompileError:
            return None
        out._expr = None           # nobody reads the pruned tree again
        return zero_idx, rest, out, None
    try:   # every constant pruned: the constant-free expression is scored as it is
        zprog = compile_sympy(prog.expr.subs({s: 0.0 for s in csyms}), 0, variables)
        zprog._expr = None
    except Exception as exc:  # noqa: BLE001 -- a singular tree (zoo*x_1 ...), scored 1e9 by the caller
        zprog = hostpool._portable(exc)
    return zero_idx, rest, None, zprog


def _prepare_prune_async(prog, small, variables, cfg, many=True):
    """``prepare_prune`` of one candidate: in the host pool when there is one and the caller has
    several candidates to prepare.  Returns a function that waits for the result."""
    pool = hostpool.get_pool(_host_workers(cfg)) if many else None
    fut = None
    if pool is not None:
        try:
            fut = pool.submit(hostpool.prune_task, (prog, small, list(variables)))
        except Exception:  # noqa: BLE001 -- broken pool: do it here
            hostpool.shutdown()
    if fut is None:
        got = prepare_prune(prog, small, variables)
        return lambda: got

    def wait():
        try:
            return fut.result()
        except Exception:  # noqa: BLE001 -- a worker died: do it here, the next call starts a fresh pool
            hostpool.shutdown()
            return prepare_prune(prog, small, variables)
    return wait


def _derivative_is_constant(expr, sym):
    """``sp.diff(expr, sym).is_constant()`` (bfgs.py:160), without its cost where the answer is plain.

    ``is_constant`` simplifies the derivative and then probes it numerically (25-160 ms on the
    workload's skeletons).  For a derivative that takes two clearly different finite values at two
    points it can only answer False: simplification keeps the function, so either its own numeric
    probes differ or some partial derivative is not identically zero, and both paths return False
    (sympy/core/expr.py:is_constant).  Everything else -- no free symbols, equal or non-finite
    probes -- is left to sympy itself."""
    d = sp.diff(expr, sym)
    free = sorted(d.free_symbols, key=lambda q: q.name)
    if free:
        try:
            vals = []
            for point in (0.3779, 1.6180, -0.7321):
                v = complex(d.evalf(17, subs={q: point + 0.0917 * j for j, q in enumerate(free)}))
                if v == v and abs(v) != float("inf"):
                    vals.append(v)
            for a in vals[1:]:
                if abs(a - vals[0]) > 1e-6 * max(1.0, abs(a), abs(vals[0])):
                    return False
        except Exception:  # noqa: BLE001 -- whatever went wrong, sympy decides
            pass
    return d.is_constant()


# compiled skeletons, keyed by the token sequence: beams of successive fitfunc calls on the
# same problem repeat most of their candidates (scripts/*_test.py loop 8x per equation)
_COMPILED = {}
_COMPILED_MAX = 8192
# milliseconds the stages of the last _bfgs_batch call took on the host (measurement aid)
LAST_TIMING = {}


def compile_tokens(toks, cfg, test_data, variables):
    """Q1-Q5 + lowering of ONE candidate: token ids -> (c-named infix string, k, Program)."""
    expr, k = skeleton_string(toks, cfg, test_data)
    prog = compile_sympy(parse_skeleton(expr), k, variables)
    prog.source = expr          # lets the program cross a process boundary without its sympy tree
    return expr, k, prog


def _cache_key(toks, cfg, test_data, variables):
    return (tuple(int(t) for t in (toks.tolist() if hasattr(toks, "tolist") else toks)),
            bool(_opt(cfg, "add_coefficients_if_not_existing", False)), tuple(variables),
            test_data.id2word.get(3))


def _remember(key, hit):
    if len(_COMPILED) >= _COMPILED_MAX:
        _COMPILED.pop(next(iter(_COMPILED)))
    _COMPILED[key] = hit
    return hit


def _compile_candidate(toks, cfg, test_data, variables):
    key = _cache_key(toks, cfg, test_data, variables)
    hit = _COMPILED.get(key)
    if hit is None:
        hit = _remember(key, compile_tokens(toks, cfg, test_data, variables))
    return hit


def _host_workers(cfg):
    n = _opt(cfg, "host_workers", None)
    return hostpool.default_workers() if n is None else int(n)


MAX_STAGES = 4     # the main engine and three side engines


def stage_goes(n_ready, n_remaining, stage_no, since_last_s, n_first):
    """Whether the next stage of a staged fit is launched now: ``n_ready`` of the ``n_remaining``
    candidates not yet launched are compiled, ``stage_no`` stages are out, the last one went
    ``since_last_s`` seconds ago.  Everything that is left always goes; the FIRST stage goes as soon as
    ``n_first`` candidates (enough to fill the GPU) are there; a later one when most of the rest is
    there and the stragglers have kept it waiting; the last engine only takes all that is left."""
    if n_ready == n_remaining:
        return True
    if stage_no >= MAX_STAGES - 1:
        return False
    if stage_no == 0:
        return n_ready >= n_first
    return n_ready >= max(8, (3 * n_remaining) // 4) and since_last_s > 4e-3


class _Compiling:
    """Skeleton compilation of a beam under way: cache hits are there at once, the misses are tasks in
    the host pool (heaviest skeletons first).  ``wait(indices)`` blocks until those candidates are
    compiled; ``out[i]`` is then ``(expr, k, Program)`` or the ``Exception`` candidate i raised."""

    def __init__(self, pred_strs, cfg, test_data, variables, share=None):
        """``share = (rank, world)``: the ranks of a process group were handed the same beam; each
        compiles every world-th missing skeleton and ``exchange()`` hands the programs round."""
        self._cfg, self._td, self._variables = cfg, test_data, variables
        self.keys = keys = [_cache_key(t, cfg, test_data, variables) for t in pred_strs]
        self.out = out = [_COMPILED.get(k) for k in keys]
        miss = [i for i, h in enumerate(out) if h is None]
        self.first = first = {}
        for i in miss:                        # a beam may hold the same token sequence twice
            first.setdefault(keys[i], i)
        todo = sorted(first.values())
        self.dup = [i for i in miss if first[keys[i]] != i]
        self.pending = []                     # (future, candidate indices), in submission order
        self.owner = {}                       # candidate -> position in pending
        c_id = next((i for i, w in test_data.id2word.items() if w in ("c", "constant")), 3)
        # weight: constants first (the iteration cap of a run is 200 k, bfgs.py:115), then length
        self.weight = [(sum(1 for t in k[0] if t == c_id), len(k[0])) for k in keys]
        todo.sort(key=lambda i: self.weight[i], reverse=True)
        self.shared = None
        if share is not None and share[1] > 1 and todo:
            self.shared = todo                        # what the ranks compile between them (same list everywhere)
            todo = todo[share[0]::share[1]]
        self.mine = list(todo)
        workers = _host_workers(cfg)
        pool = hostpool.get_pool(workers) if (len(todo) >= 8 and workers >= 2) else None
        if pool is not None:
            # small tasks, heaviest skeletons first: the workers stay evenly loaded to the end and the
            # candidates with the longest fits are ready first
            per = max(1, min(4, len(todo) // (3 * hostpool._POOL_N)))
            bits = (bool(_opt(cfg, "add_coefficients_if_not_existing", False)),)
            id2word = dict(test_data.id2word)
            for j in range(0, len(todo), per):
                ch = todo[j:j + per]
                try:
                    fut = pool.submit(hostpool.compile_chunk, ([list(keys[i][0]) for i in ch], bits, id2word, list(variables)))
                except Exception:  # noqa: BLE001 -- the pool is broken (a worker died earlier): a future that says so
                    from concurrent.futures import Future
                    fut = Future()
                    fut.set_exception(RuntimeError("host pool unavailable"))
                for i in ch:
                    self.owner[i] = len(self.pending)
                self.pending.append((fut, ch))
        else:
            for i in todo:
                try:
                    out[i] = _remember(keys[i], compile_tokens(pred_strs[i], cfg, test_data, variables))
                except Exception as exc:  # noqa: BLE001 -- the wrapper's contract (model.py:15-19)
                    out[i] = hostpool._portable(exc) if self.shared is not None else exc
            self._fill_dups()

    @property
    def staged(self):
        return bool(self.pending)

    def ready(self, indices):
        """The candidates of ``indices`` that are compiled by now (does not block)."""
        out = []
        for i in indices:
            if self.out[i] is not None:
                out.append(i)
                continue
            j = self.first.get(self.keys[i], i)
            pos = self.owner.get(j)
            if pos is None:
                if self.out[j] is not None:
                    out.append(i)
                continue
            fut = self.pending[pos][0]
            if fut is None or fut.done():
                out.append(i)
        return out

    def exchange(self):
        """Sharded compilation: one all_gather_object of what each rank compiled."""
        self.wait(self.mine)
        if self.shared is not None:
            import torch.distributed as dist
            parts = [None] * dist.get_world_size()
            dist.all_gather_object(parts, [(i, self.out[i]) for i in self.mine])
            for part in parts:
                for i, hit in part:
                    if self.out[i] is None:
                        self.out[i] = hit if isinstance(hit, Exception) else _remember(self.keys[i], hit)
            self.shared = None
        self._fill_dups()
        return self.out

    def _fill_dups(self):
        for i in self.dup:
            if self.out[i] is None and self.out[self.first[self.keys[i]]] is not None:
                self.out[i] = self.out[self.first[self.keys[i]]]

    def wait(self, indices=None):
        want = range(len(self.out)) if indices is None else indices
        need = sorted({self.owner[j] for i in want for j in [self.first.get(self.keys[i], i)]
                       if self.out[i] is None and j in self.owner})
        for pos in need:
            fut, ch = self.pending[pos]
            if fut is None:
                continue
            try:
                got = fut.result()
            except Exception:  # noqa: BLE001 -- a worker died (BrokenProcessPool ...): compile the task here
                hostpool.shutdown()               # the next call starts a fresh pool
                got = []
                for i in ch:
                    try:
                        got.append(compile_tokens(list(self.keys[i][0]), self._cfg, self._td, self._variables))
                    except Exception as exc:  # noqa: BLE001 -- per candidate (model.py:15-19)
                        got.append(exc)
            for i, r in zip(ch, got):
                self.out[i] = r if isinstance(r, Exception) else _remember(self.keys[i], r)
            self.pending[pos] = (None, ch)
        self._fill_dups()
        return self.out


def _compile_candidates(pred_strs, cfg, test_data, variables):
    """``(expr, k, Program)`` or the raised ``Exception`` for every candidate.  Cache misses are
    compiled in the host pool, in small tasks (sympy: 3-8 ms per candidate), when there are enough."""
    return _Compiling(pred_strs, cfg, test_data, variables).wait()


class LazyStr:
    """``str(skeleton with the fitted constants in)``, produced when somebody reads it.  Printing a
    fitted candidate through sympy costs 5-15 ms and every driver of the reference reads ONE string
    per ``fitfunc`` call (``best_bfgs_preds[0]``, e.g. Feynman_test.py:78)."""
    __slots__ = ("_job", "_text")

    def __init__(self, job):
        self._job, self._text = job, None

    def __str__(self):
        if self._text is None:
            prog, _, syms, vals = self._job
            self._text = str(_substitute(prog.expr, syms, vals))
            self._job = None
        return self._text

    __repr__ = __str__


class LazyStrings(list):
    """A list of strings some of which are still ``LazyStr``: every way of reading an element
    hands out (and keeps) the finished ``str``."""

    def _get(self, i):
        v = list.__getitem__(self, i)
        if isinstance(v, LazyStr):
            v = str(v)
            list.__setitem__(self, i, v)
        return v

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self._get(j) for j in range(*i.indices(len(self)))]
        return self._get(i if i >= 0 else i + len(self))

    def __iter__(self):
        return (self._get(i) for i in range(len(self)))

    def __eq__(self, other):
        return list(iter(self)) == list(other)

    __hash__ = None

    def __repr__(self):
        return repr(list(iter(self)))

    def __reduce__(self):
        return (list, (list(iter(self)),))


def _format_all(jobs, cfg):
    """``str(skeleton with the numbers in)`` for every job ``(Program, skeleton string, symbols,
    values)`` -- in the host pool when there are enough of them."""
    pool = hostpool.get_pool(_host_workers(cfg)) if len(jobs) >= 8 else None
    if pool is None:
        return [str(_substitute(prog.expr, syms, vals)) for prog, _, syms, vals in jobs]
    n = hostpool._POOL_N
    idx = [list(range(j, len(jobs), n)) for j in range(min(n, len(jobs)))]
    payload = [[(jobs[i][1], [sy.name for sy in jobs[i][2]], [float(v) for v in jobs[i][3]]) for i in ch] for ch in idx]
    out = [None] * len(jobs)
    for ch, res in zip(idx, pool.map(hostpool.format_chunk, payload)):
        for i, r in zip(ch, res):
            if isinstance(r, Exception):   # not expected: redo it here, where the error belongs
                r = str(_substitute(jobs[i][0].expr, jobs[i][2], jobs[i][3]))
            out[i] = r
    return out


def sigma_weights(sigma, X, cfg):
    """Weights ``1 / sigma**2`` of a fit of points ``X`` (``[1, N, d]`` or ``[N, d]``) under ``cfg``, checked
    in every point dtype the fit uses (``fitter.weights_from_sigma``); ``None`` without ``sigma``.  Raises
    ``ValueError`` for a bad ``sigma`` and for ``sigma`` with ``cfg.bfgs.idx_remove``: the reference pairs
    the kept rows with the first ``y``s (bfgs.py:78-82), so no pairing of the weights would mean anything."""
    if sigma is None:
        return None
    if _opt(cfg, "idx_remove", False):
        raise ValueError("sigma cannot be combined with cfg.bfgs.idx_remove")
    Xt = torch.as_tensor(X)
    n = int(Xt.shape[-2])
    score_dtype = fitter.F32 if Xt.dtype == torch.float32 else fitter.F64
    eval_dtype = fitter.F32 if str(_opt(cfg, "precision", "fp64")).lower() == "fp32" else fitter.F64
    return fitter.weights_from_sigma(sigma, n, {eval_dtype, score_dtype, fitter.F64})


def bfgs_batch(pred_strs, X, y, cfg, test_data, x0=None, engine=None, lazy_strings=False, sigma=None):
    """Fit every candidate of a beam in one go (see ``_bfgs_batch``).

    ``sigma``: optional 1-D array of N per-point standard deviations (any device), as
    ``scipy.optimize.curve_fit`` takes it: every fit then minimises ``loss_scale * mean(w r^2)`` with
    ``w = 1 / sigma**2``, and the returned loss, the per-restart score that picks the restart and the
    prune's acceptance are weighted.  ``ValueError`` for a wrong length, a sigma that is not finite and
    > 0, a ``1/sigma**2`` that is not a finite normal number in a point dtype of the fit, or ``sigma`` with
    ``cfg.bfgs.idx_remove``.  With a process group every rank passes its own ``sigma``, like ``X``, ``y``.

    With ``cfg.bfgs.collapse_duplicates`` (off by default; SURVEY 8f row 4) candidates that
    compile to the SAME bytecode -- beams that differ only in ways sympy canonicalises away,
    ``model.py:459-483`` keeps them all -- are fitted once, from the starting points of the first
    of them, and share the result; each keeps its own skeleton string.  The reference fits every
    duplicate again from fresh random starting points, so this changes which restarts a
    duplicate sees, not what a fit computes.
    """
    pred_strs = list(pred_strs)
    w = sigma_weights(sigma, X, cfg)
    if not _opt(cfg, "collapse_duplicates", False) or len(pred_strs) < 2:
        return _bfgs_batch(pred_strs, X, y, cfg, test_data, x0=x0, engine=engine, lazy_strings=lazy_strings, w=w)
    variables = list(test_data.total_variables)
    first, rep_of, own_expr = {}, [], []
    for i, toks in enumerate(pred_strs):
        try:
            expr, k, prog = _compile_candidate(toks, cfg, test_data, variables)
            key = (k, prog.insns.tobytes(), prog.imms.tobytes())
        except Exception:  # noqa: BLE001 -- fails again, on its own, in _bfgs_batch
            expr, key = None, ("error", i)
        rep_of.append(first.setdefault(key, i))
        own_expr.append(expr)
    reps = sorted(set(rep_of))
    pos = {r: j for j, r in enumerate(reps)}
    sub = _bfgs_batch([pred_strs[r] for r in reps], X, y, cfg, test_data,
                      x0=None if x0 is None else [x0[r] for r in reps], engine=engine, lazy_strings=lazy_strings,
                      w=w)
    out = []
    for i, r in enumerate(rep_of):
        res = sub[pos[r]]
        if i != r and not isinstance(res, Exception):
            res = (res[0], res[1], res[2], own_expr[i])
        out.append(res)
    return out


def _bfgs_batch(pred_strs, X, y, cfg, test_data, x0=None, engine=None, lazy_strings=False, w=None):
    """Fit every candidate of a beam in one go.

    Returns a list with one entry per candidate: the reference's 4-tuple
    ``(best_expr_str, best_consts, best_loss, expr)`` or the ``Exception`` that
    ``bfgs()`` would have raised for it.  ``x0``: optional list (one per candidate) of
    ``[R, k]`` starting points; default is the reference's ``np.random.randn(k) * 10``
    per restart (bfgs.py:103).  ``lazy_strings``: ``best_expr_str`` of every candidate is a
    ``LazyStr`` (printed through sympy when read) instead of a ``str``.  ``w``: per-point weights
    (``sigma_weights``) or ``None``.
    """
    import time as _time
    _t = [_time.perf_counter()]

    def _mark(name):
        now = _time.perf_counter()
        LAST_TIMING[name] = LAST_TIMING.get(name, 0.0) + (now - _t[0]) * 1e3
        _t[0] = now
    LAST_TIMING.clear()
    devices = resolve_devices(cfg)
    if devices and engine is not None and engine.device != devices[0]:
        raise ValueError(f"engine on {engine.device}, but the home device of cfg.bfgs.devices is {devices[0]}")
    y = y.squeeze()
    Xt = torch.as_tensor(X)
    if Xt.dim() == 2:
        Xt = Xt.unsqueeze(0)
    yt = torch.as_tensor(y).reshape(-1)
    variables = list(test_data.total_variables)
    R = int(_opt(cfg, "n_restarts"))

    # ---- Q1-Q5 + compilation, per candidate (failures stay per candidate): started here, collected
    # stage by stage below, while the GPU already fits the candidates that are ready ----
    world = sharding.world_size() if _opt(cfg, "shard", True) and not _opt(cfg, "idx_remove", False) else 1
    comp = _Compiling(pred_strs, cfg, test_data, variables,
                      share=(sharding.rank(), world) if world > 1 else None)
    if world > 1:
        comp.exchange()
    n_cand = len(pred_strs)
    cands = [None] * n_cand
    if not comp.staged and all(isinstance(h, Exception) for h in comp.out):
        return list(comp.out)     # nothing to fit: the engine is not touched

    # ---- Q6 outlier rows ----
    rows_removed = False
    if _opt(cfg, "idx_remove", False):
        keep = (Xt < 200).all(dim=2).squeeze(0)
        rows_removed = bool((~keep).any())
        Xt = Xt[:, keep, :]
        yt_fit = yt[:Xt.shape[1]]  # the reference pairs kept rows with the first y's (bfgs.py:78-82)
    else:
        yt_fit = yt

    # ---- Q7 normalisation ----
    norm = _opt(cfg, "normalization_type")
    if norm == "NMSE":
        # mean of the FULL y in y's own dtype, rows dropped by idx_remove included (bfgs.py:86-90)
        mean_y = float(np.mean(yt.detach().cpu().numpy()))
        scale = 1.0 / mean_y if abs(mean_y) > 1e-06 else 1.0
    elif norm == "MSE":
        scale = 1.0
    else:
        raise KeyError(norm)

    eng = engine if engine is not None else fitter.get_engine(
        devices[0] if devices else (Xt.device if Xt.is_cuda else None))
    score_dtype = fitter.F32 if Xt.dtype == torch.float32 else fitter.F64
    eval_dtype = fitter.F32 if str(_opt(cfg, "precision", "fp64")).lower() == "fp32" else fitter.F64
    eng.set_points(Xt[0], yt_fit, dtypes=tuple({eval_dtype, score_dtype, fitter.F64}), w=w)
    opts = _engine_opts(cfg, scale, eval_dtype, score_dtype)
    main_stream = torch.cuda.current_stream(eng.device)
    points_ready = torch.cuda.Event()
    points_ready.record(main_stream)      # side streams wait for the upload, not for the first stage's fit
    _mark("upload")

    world = sharding.world_size() if _opt(cfg, "shard", True) and not rows_removed else 1
    # cfg.bfgs.devices with several entries: the runs are dealt over one engine per entry, in this process
    # (like the ranks: one stage, one record per candidate back).  Rows dropped by idx_remove keep the fit
    # on the home device, as they keep it on one rank.
    spread = devices is not None and len(devices) > 1 and not rows_removed
    if spread:
        engines = fitter.device_engines(devices, home=eng)
        fitter.share_points(engines)
    # Stages: the skeletons are compiled heaviest first (most constants = longest fits); the fit of a
    # FIRST stage starts as soon as enough candidates to fill the GPU are compiled -- whichever they
    # are: sympy takes 3 ms for most skeletons and 30-60 ms for a few -- on the main engine; the rest
    # follows on side engines and streams that share the points, stragglers in a stage of their own.
    # One stage when there is nothing to overlap.
    def _stages():
        if not (comp.staged and world == 1 and not spread and n_cand >= 24 and _opt(cfg, "pipeline", True)):
            yield list(range(n_cand))
            return
        for j in (1, 2, 3):                    # the side engines exist before the first stage is launched
            fitter.get_side_engine(eng, j)     # (created once per process: a driver's first call pays)
        remaining = set(range(n_cand))
        n_first = max(8, min((n_cand + 2) // 3, hostpool._POOL_N or n_cand))
        stage_no, t_last = 0, _time.perf_counter()
        while remaining:
            ready = comp.ready(remaining)
            now = _time.perf_counter()
            go = stage_goes(len(ready), len(remaining), stage_no, now - t_last, n_first)
            if not go:
                _time.sleep(2e-4)
                continue
            stage = sorted(ready)
            remaining.difference_update(stage)
            stage_no, t_last = stage_no + 1, now
            yield stage

    def _collect(stage):
        comp.wait(stage)
        for i in stage:
            hit = comp.out[i]
            c = _Candidate()
            if isinstance(hit, Exception):
                c.error = hit
            else:
                c.expr, c.k, c.prog = hit
            cands[i] = c
        return [i for i in stage if cands[i].error is None]

    def _starts(live_s):
        # ---- Q8 restarts: one run per (candidate, restart) ----
        kmax = max(1, max(cands[i].k for i in live_s))
        start = np.zeros((len(live_s) * R, kmax), dtype=np.float64)
        for li, ci in enumerate(live_s):
            k = cands[ci].k
            for r in range(R):
                if x0 is not None and x0[ci] is not None:
                    v = np.asarray(x0[ci], dtype=np.float64)[r][:k]
                else:
                    v = np.random.randn(k) * 10
                start[li * R + r, :k] = v
        return start

    win_of = {}     # candidate -> record of the all-gather                (sharded, spread)
    launched = []
    for si, stage in enumerate(_stages()):
        live_s = _collect(stage)
        _mark("compile")
        if not live_s:
            continue
        start = _starts(live_s)
        if world > 1 or spread:
            cost = np.repeat([(cands[ci].k + 1.0) * cands[ci].prog.n_insns for ci in live_s], R)
            key_dtype = torch.float32 if score_dtype == fitter.F32 else None
            if spread:
                # the same dealing, per-part records and merge as the ranks', over the engines of this process
                for e in engines:
                    with torch.cuda.device(e.device):
                        e.set_programs([cands[i].prog for i in live_s])
                win, _ = sharding.fit_devices(engines, [cands[ci].k for ci in live_s], R,
                                              torch.from_numpy(start).to(eng.device), opts, cost=cost,
                                              key_dtype=key_dtype)
            else:
                # SURVEY 8e: the (candidate, restart) runs of the beam are dealt over the ranks of the default
                # process group, every rank fits its share, ONE all-gather brings back a record per candidate
                # (score, restart, constants) and every rank takes the same argmin.  Every rank must have
                # been called with the same candidates and points; the starting points are rank 0's.
                eng.set_programs([cands[i].prog for i in live_s])
                start_dev = sharding.broadcast_from_rank0(torch.from_numpy(start).to(eng.device))
                win, _ = sharding.fit_sharded(eng, [cands[ci].k for ci in live_s], R, start_dev, opts, cost=cost,
                                              key_dtype=key_dtype)
            win = win.cpu().numpy()
            for li, ci in enumerate(live_s):
                win_of[ci] = win[li]
            continue
        run_prog = np.repeat(np.arange(len(live_s), dtype=np.int32), R)
        run_slot = np.arange(len(live_s) * R, dtype=np.int32)
        if si == 0:
            eng.set_programs([cands[i].prog for i in live_s])
            res = eng.fit(run_prog, run_slot, torch.from_numpy(start), opts)
        else:
            side = fitter.get_side_engine(eng, si)
            side.adopt_points(eng)
            stream = fitter.side_stream(eng.device, si)
            stream.wait_event(points_ready)       # the points are uploaded on the caller's stream
            with torch.cuda.stream(stream):
                side.set_programs([cands[i].prog for i in live_s])
                res = side.fit(run_prog, run_slot, torch.from_numpy(start), opts)
            done = torch.cuda.Event()
            done.record(stream)
        if si == 0:
            stream = main_stream
            done = torch.cuda.Event()
            done.record(main_stream)
        launched.append((live_s, res, stream, done))
        _mark("launch")

    # ---- Q10/Q11 pick the restart, Q12 collect prune work: stage by stage as the fits finish, so
    # that the symbolic half of Q12 of an early stage runs in the host pool while a later one is
    # still on the GPU ----
    thr = _opt(cfg, "prune_threshold", 1e-3)
    tol = _opt(cfg, "prune_tolerance", 1.05)
    picked = {}
    prune_jobs, prune_waits = [], []

    def _pick(ci, best_consts, best_loss):
        c = cands[ci]
        csyms = [sp.Symbol(f"c{i}") for i in range(c.k)]
        picked[ci] = [best_consts, best_loss, csyms]
        return [i for i, v in enumerate(best_consts) if abs(v) < thr] if c.k > 0 else []

    if win_of:
        # sharded: every rank holds the same winners; the symbolic prune work is dealt over the ranks
        # and handed round with one all_gather_object
        todo = []
        for ci in sorted(win_of):
            rec, k = win_of[ci], cands[ci].k
            small = _pick(ci, rec[3:3 + k].copy(), np.float32(rec[-1]) if score_dtype == fitter.F32 else rec[-1])
            if small:
                todo.append((ci, small))
        mine = todo[sharding.rank()::world]
        waits = [(ci, _prepare_prune_async(cands[ci].prog, small, variables, cfg, many=len(mine) >= 4 and _host_workers(cfg) >= 2))
                 for ci, small in mine]
        done = [(ci, wait()) for ci, wait in waits]
        if world > 1 and todo:
            import torch.distributed as dist
            parts = [None] * world
            dist.all_gather_object(parts, done)
            done = [item for part in parts for item in part]
        for ci, got in done:
            prune_waits.append((ci, (lambda g=got: g)))
    waiting = list(launched)
    while waiting:
        pos = next((j for j, w in enumerate(waiting) if w[3].query()), None)
        if pos is None:
            if len(waiting) == 1:
                waiting[0][3].synchronize()
            else:
                _time.sleep(0.0002)
            continue
        live_s, res, stream, _ = waiting.pop(pos)
        with torch.cuda.stream(stream):
            lastx = res.lastx.cpu().numpy()
            final = res.final_mse.cpu().numpy()
        if score_dtype == fitter.F32:
            final = final.astype(np.float32)
        if rows_removed:
            final = np.full_like(final, 1e9)  # y_found - y raises on the shape mismatch (bfgs.py:130-131)
        todo = []
        for li, ci in enumerate(live_s):
            F_loss = final[li * R:(li + 1) * R]
            try:
                k_best = int(np.nanargmin(F_loss))
            except ValueError:
                k_best = 0
            small = _pick(ci, lastx[li * R + k_best, :cands[ci].k].copy(), F_loss[k_best])
            if small:
                todo.append((ci, small))
        for ci, small in todo:
            prune_waits.append((ci, _prepare_prune_async(cands[ci].prog, small, variables, cfg, many=len(todo) >= 4)))
    for _, _, stream, _ in launched:
        if stream is not main_stream:
            main_stream.wait_stream(stream)
    live = [i for i, c in enumerate(cands) if c is not None and c.error is None]
    results = [None if c is None else c.error for c in cands]
    if not live:
        return results
    _mark("fit")
    for ci, wait in prune_waits:
        got = wait()
        if got is not None:
            zero_idx, rest, prog, zprog = got
            prune_jobs.append(dict(ci=ci, zero=zero_idx, rest=rest, prog=prog, zprog=zprog))
    prune_jobs.sort(key=lambda j: j["ci"])

    _mark("prune_sym")
    # ---- Q12 re-fit the pruned skeletons (one more BFGS each, from the best point) ----
    fit_jobs = [j for j in prune_jobs if j["prog"] is not None]
    if fit_jobs:
        eng.set_programs([j["prog"] for j in fit_jobs])
        pk = max(len(j["rest"]) for j in fit_jobs)
        pstart = np.zeros((len(fit_jobs), pk), dtype=np.float64)
        for ji, j in enumerate(fit_jobs):
            pstart[ji, :len(j["rest"])] = picked[j["ci"]][0][j["rest"]]
        pres = eng.fit(list(range(len(fit_jobs))), list(range(len(fit_jobs))),
                       torch.from_numpy(pstart), opts)
        # the reference scores res_pruned.x, not the last evaluated point (bfgs.py:180)
        ploss, _ = eng.eval(list(range(len(fit_jobs))), pres.consts, dtype=score_dtype)
        pconsts = pres.consts.cpu().numpy()
        ploss = ploss.cpu().numpy()
        _mark("prune_fit")
        for ji, j in enumerate(fit_jobs):
            j["x"] = pconsts[ji, :len(j["rest"])]
            j["loss"] = ploss[ji]
    for j in prune_jobs:
        c = cands[j["ci"]]
        best_consts, best_loss, csyms = picked[j["ci"]]
        vals = np.zeros(c.k)
        if j["prog"] is not None:
            vals[j["rest"]] = j["x"]
            pruned_loss = j["loss"]
        else:  # every constant pruned: evaluate the constant-free expression
            try:
                if isinstance(j["zprog"], Exception):
                    raise j["zprog"]
                eng.set_programs([j["zprog"]])
                zl, _ = eng.eval([0], torch.zeros((1, 1)), dtype=score_dtype)
                pruned_loss = float(zl.cpu().numpy()[0])
            except Exception:  # noqa: BLE001 -- a singular tree (zoo*x_1 ...): bfgs.py:196-202 scores it 1e9,
                pruned_loss = 1e9  # the prune is rejected and the unpruned fit stays
        if score_dtype == fitter.F32:
            pruned_loss = np.float32(pruned_loss)
        if rows_removed:
            pruned_loss = 1e9
        ok = (pruned_loss < 1e-9) if best_loss == 0 else (pruned_loss <= best_loss * tol)
        if ok:
            picked[j["ci"]] = [vals, pruned_loss, csyms, True, j["zero"]]

    _mark("prune")
    # ---- Q13 strings ----
    fmt_jobs, fmt_meta = [], []
    for ci in live:
        c = cands[ci]
        entry = picked[ci]
        best_consts, best_loss, csyms = entry[0], entry[1], entry[2]
        if c.k == 0:
            results[ci] = (c.expr, [], best_loss, c.expr)
            continue
        if len(entry) > 3:  # pruned: zeros first, then the re-fitted ones (bfgs.py:184-196)
            order = list(entry[4]) + [i for i in range(c.k) if i not in entry[4]]
            vals = [0.0 if i in entry[4] else best_consts[i] for i in order]
            fmt_jobs.append((c.prog, c.expr, [csyms[i] for i in order], vals))
            consts_out = [0.0 if i in entry[4] else best_consts[i] for i in range(c.k)]
        else:
            fmt_jobs.append((c.prog, c.expr, csyms, list(best_consts)))
            consts_out = best_consts
        fmt_meta.append((ci, consts_out, best_loss))
    texts = [LazyStr(j) for j in fmt_jobs] if lazy_strings else _format_all(fmt_jobs, cfg)
    for (ci, consts_out, best_loss), text in zip(fmt_meta, texts):
        results[ci] = (text, consts_out, best_loss, cands[ci].expr)
    _mark("strings")
    return results


def bfgs(pred_str, X, y, cfg, test_data, x0=None, engine=None, sigma=None):
    """Reference signature (bfgs.py:42): one candidate, raises what the reference raises.  ``sigma``: see
    ``bfgs_batch``."""
    out = bfgs_batch([pred_str], X, y, cfg, test_data,
                     x0=None if x0 is None else [x0], engine=engine, sigma=sigma)[0]
    if isinstance(out, Exception):
        raise out
    return out
