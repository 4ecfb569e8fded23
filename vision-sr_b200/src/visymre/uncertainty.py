"""Covariance and standard errors of fitted constants, from statistics computed on the device.

``bfgs()`` returns ``(string, consts, loss, skeleton)`` and says nothing about how well the data
determine the constants.  ``covariances`` answers that for a list of such fits the way
``scipy.optimize.curve_fit`` does with its default ``absolute_sigma=False``::

    cov = s^2 (J^T J)^-1,   s^2 = rss / (N - k_free),   stderr = sqrt(diag(cov))

with ``J`` the N x k Jacobian of the skeleton in its constants at the fitted point.  The device
evaluates every point as a dual number whose tangents are a row of ``J``; one ``vsr_gram`` launch
reduces them to ``rss`` and ``J^T J`` for every fit of the list (``csrc/vsr_kernels.cuh``,
``gram_kernel``).  Only the k x k matrix comes back to the host, where this module inverts it.

Conventions:

* Free constants.  The reference's prune fixes constants at an exact ``0.0`` (bfgs.py:184-196); the
  4-tuple returns them as ``0.0`` and they are not fitted, so only the nonzero constants enter the
  matrix.  Rows and columns of a fixed constant are nan, so is its ``stderr``, and
  ``dof = N - k_free``.
* Undeterminable.  When ``dof <= 0``, when ``rss`` or ``J^T J`` holds a nan or inf (the expression
  is not real at some point), or when ``J^T J`` is numerically rank-deficient, the covariance of the
  free constants is ``inf``, as curve_fit reports "covariance of the parameters could not be
  estimated".  Rank-deficient means an eigenvalue ``lambda_i <= max(N, k) * eps * lambda_max``;
  ``rank`` is the number of eigenvalues above that bound (0 when the Gram holds a non-finite value).
* The one deviation from curve_fit.  The rank test is on ``J^T J``, which carries half the digits of
  ``J``: a direction of ``J`` whose singular value is below about ``sqrt(max(N, k) * eps)`` times the
  largest is called unidentifiable here.  curve_fit, working on ``J`` itself, would keep it, with a
  variance at least 1e12 times that of the best-determined direction.

The points are taken as given: pass the rows the fit saw (with ``idx_remove``, the kept rows).  A
skeleton's ``x_j`` reads column j-1 of ``X``, which is the fit's convention (not the drivers'
by-rank pairing of ``scoring.py``).

``predict`` evaluates fitted expressions at new points, and with the covariances gives the
delta-method confidence band of the mean and prediction band of a new observation at each point::

    se_fit(x)^2 = g(x)^T cov g(x),   g(x) = d f(x; c) / d c at the fitted c
    f(x) +- t se_fit(x),   f(x) +- t sqrt(se_fit(x)^2 + s^2),   t = t_{dof}((1 + level) / 2)

One ``vsr_predict`` launch writes ``f`` and ``g^T cov g`` of every point for every fit of the list
(``csrc/vsr_kernels.cuh``, ``predict_kernel``); ``bands`` assembles the rest on the device.

Per-point uncertainties (curve_fit's 1-D ``sigma``).  With ``sigma`` the weights are ``w = 1 / sigma^2``,
``rss`` is ``sum w r^2`` and ``J^T J`` becomes ``J^T W J``, both from one weighted ``vsr_gram`` launch::

    absolute_sigma=False:  cov = s^2 (J^T W J)^-1,  s^2 = sum w r^2 / dof
    absolute_sigma=True:   cov = (J^T W J)^-1        (sigma is the known scale of the noise)

The rank test and the ``inf`` rules above apply unchanged.  For the prediction band of a new observation
whose sigma is ``sigma_new``, the noise term is ``s^2 sigma_new^2`` for a relative covariance (the default
``sigma_new = 1`` gives ``s^2``) and ``sigma_new^2`` for an absolute one, whose bands use the normal
quantile instead of Student's t because the scale is known.
"""
from dataclasses import dataclass
from typing import Optional

import numpy as np
import scipy.stats
import torch

from .engine import fitter, hostpool
from .engine.compiler import compile_skeleton

_VARS = [f"x_{i}" for i in range(1, 11)]
# skeletons compiled in the host pool from this many on (below it the pool's round trip costs more
# than it saves; see DESIGN.md section 6c)
POOL_MIN = 16


@dataclass
class ConstantCovariance:
    """Uncertainty of the constants of one fit (host numpy arrays, k = number of constants)."""
    consts: np.ndarray   # [k] the fitted constants
    free: np.ndarray     # [k] bool: False for a constant the prune fixed at 0.0
    cov: np.ndarray      # [k, k] covariance; nan in rows / columns of fixed constants
    stderr: np.ndarray   # [k] sqrt(diag(cov))
    rss: float           # sum of squared residuals at consts
    dof: int             # N - number of free constants
    rank: int            # numerical rank of J^T J over the free constants
    jtj: np.ndarray      # [k, k] J^T J over all constants
    absolute_sigma: bool = False   # cov = (J^T W J)^-1 without the s^2 factor (see the module docstring)


def covariance_from_gram(rss, jtj, n, free, absolute_sigma=False):
    """``(cov, stderr, dof, rank)`` from the sum of squared residuals, ``J^T J`` ([k, k]), the number
    of points and the mask of free constants, with curve_fit's conventions (module docstring).  For a
    weighted fit pass ``sum w r^2`` and ``J^T W J``; ``absolute_sigma=True`` leaves out the factor
    ``s^2 = rss / dof``."""
    jtj = np.asarray(jtj, dtype=np.float64)
    free = np.asarray(free, dtype=bool)
    k = free.shape[0]
    kf = int(free.sum())
    dof = int(n) - kf
    cov = np.full((k, k), np.nan)
    rank = 0
    if kf > 0:
        sub = jtj[np.ix_(free, free)]
        cov_f = np.full((kf, kf), np.inf)
        if np.isfinite(rss) and np.isfinite(sub).all():
            w, V = np.linalg.eigh(sub)
            rank = int((w > max(int(n), kf) * np.finfo(np.float64).eps * w.max()).sum())
            if rank == kf and dof > 0:
                cov_f = (V / w) @ V.T
                if not absolute_sigma:
                    cov_f = cov_f * (float(rss) / dof)
                cov_f = 0.5 * (cov_f + cov_f.T)
        cov[np.ix_(free, free)] = cov_f
    with np.errstate(invalid="ignore"):
        stderr = np.sqrt(np.diag(cov))
    return cov, stderr, dof, rank


def _compile(items):
    """Programs of ``[(skeleton, k)]``, in the host pool when the list is long enough."""
    pool = hostpool.get_pool(hostpool.default_workers()) if len(items) >= POOL_MIN else None
    if pool is None:
        return [compile_skeleton(expr, k, _VARS) for expr, k in items]
    n = hostpool._POOL_N
    chunks = [list(range(j, len(items), n)) for j in range(min(n, len(items)))]
    out = [None] * len(items)
    for ch, res in zip(chunks, pool.map(hostpool.compile_skeletons, [[items[i] for i in ch] for ch in chunks])):
        for i, r in zip(ch, res):
            if isinstance(r, Exception):
                r = compile_skeleton(items[i][0], items[i][1], _VARS)   # raises here, where it belongs
            out[i] = r
    return out


def covariances(fits, X, y, engine=None, sigma=None, absolute_sigma=False):
    """Covariance of the constants of every fit of ``fits``.

    ``fits``: ``bfgs()`` / ``bfgs_batch()`` 4-tuples ``(string, consts, loss, skeleton)``; an
    ``Exception`` or ``None`` in the list gives ``None``.  ``X``: ``[1, N, d]`` or ``[N, d]`` on any
    device, fp32 or fp64; ``y``: squeezable to ``[N]``.  Returns one ``ConstantCovariance`` (or
    ``None``) per entry.  The whole list is evaluated with one ``vsr_gram`` call on ``engine`` (default:
    the process-wide engine of X's device, or of the current CUDA device); its points and programs are
    replaced.  ``sigma``: optional 1-D per-point standard deviations of ``y`` (N entries, any device), as
    curve_fit's ``sigma``; ``absolute_sigma``: curve_fit's flag (module docstring).  ``ValueError`` for a
    bad ``sigma`` (wrong length, not finite and > 0, ``1/sigma^2`` not a finite normal fp64 number).
    """
    X = torch.as_tensor(X)
    if X.dim() == 3:
        X = X[0]
    y = torch.as_tensor(y).reshape(-1)
    w = fitter.weights_from_sigma(sigma, X.shape[0], (fitter.F64,)) if sigma is not None else None
    out = [None] * len(fits)
    items = []
    for i, f in enumerate(fits):
        if f is None or isinstance(f, Exception):
            continue
        items.append((i, str(f[3]), np.asarray(f[1], dtype=np.float64).reshape(-1)))
    if not items:
        return out
    progs = _compile([(skel, c.shape[0]) for _, skel, c in items])
    eng = engine if engine is not None else fitter.get_engine(X.device if X.is_cuda else None)
    eng.set_points(X, y, dtypes=(fitter.F64,), n_vars=max(1, max(p.var_mask.bit_length() for p in progs)), w=w)
    eng.set_programs(progs)
    consts = np.zeros((len(items), max(1, max(c.shape[0] for _, _, c in items))))
    for j, (_, _, c) in enumerate(items):
        consts[j, :c.shape[0]] = c
    rss, jtj = eng.gram(np.arange(len(items)), torch.from_numpy(consts))
    rss, jtj = rss.cpu().numpy(), jtj.cpu().numpy()
    n = int(X.shape[0])
    for j, (i, _, c) in enumerate(items):
        k = c.shape[0]
        free = c != 0.0
        g = jtj[j, :k, :k].copy()
        cov, stderr, dof, rank = covariance_from_gram(rss[j], g, n, free, absolute_sigma)
        out[i] = ConstantCovariance(consts=c, free=free, cov=cov, stderr=stderr, rss=float(rss[j]),
                                    dof=dof, rank=rank, jtj=g, absolute_sigma=bool(absolute_sigma))
    return out


@dataclass
class Prediction:
    """A fitted expression at N points: device float64 tensors ``[N]``.  Without a covariance only
    ``value`` and ``level`` are set; the other fields are ``None``."""
    value: torch.Tensor                # f(x; c)
    se_fit: Optional[torch.Tensor]     # sqrt(max(g^T cov g, 0))
    ci_low: Optional[torch.Tensor]     # value -+ t se_fit: confidence band of the mean
    ci_high: Optional[torch.Tensor]
    pi_low: Optional[torch.Tensor]     # value -+ t sqrt(se_fit^2 + noise): prediction band of a new y
    pi_high: Optional[torch.Tensor]    # (noise = s^2 sigma_new^2, or sigma_new^2 for an absolute covariance)
    level: float
    t: Optional[float]                 # Student's t quantile at (1 + level) / 2 with dof degrees of freedom
                                       # (the normal quantile for an absolute covariance)
    dof: Optional[int]


def device_cov(cov):
    """The covariance ``vsr_predict`` reads: the nan rows and columns of constants the prune fixed at
    ``0.0`` become 0 (they carry no variance).  An ``inf`` (undeterminable) covariance becomes all 0:
    ``bands`` does not read the variance of such a fit."""
    cov = np.array(cov, dtype=np.float64)
    cov[np.isnan(cov)] = 0.0
    if np.isinf(cov).any():
        cov[:] = 0.0
    return cov


def bands(value, var, cov, rss, dof, level=0.95, sigma_new=None, absolute_sigma=False):
    """``Prediction`` from the values ``[N]`` and variances ``g^T cov g`` ``[N]`` of one fit (tensors
    on any device), its covariance (host, as ``covariances`` gives it), ``rss`` and ``dof``.

    ``s^2 = rss / dof`` and ``t = scipy.stats.t.ppf((1 + level) / 2, dof)``.  ``sigma_new`` (a scalar or
    ``[N]``): the sigma of a new observation at each point; the prediction band's noise term is
    ``s^2 sigma_new^2`` (default ``sigma_new = 1``: ``s^2``).  ``absolute_sigma=True`` (the covariance is
    ``(J^T W J)^-1``): the noise term is ``sigma_new^2``, which is then required (``ValueError``
    without it), and ``t`` is the normal quantile ``scipy.stats.norm.ppf((1 + level) / 2)``.  ``se_fit =
    sqrt(max(var, 0))``: from a positive semidefinite ``cov`` in fp64 ``var`` is below 0 only by
    rounding.  When the covariance could not be determined (an ``inf`` in ``cov``, or ``dof <= 0``)
    ``se_fit`` is ``inf`` and every band is infinite.  A nan value (``f`` not real at the point) gives
    nan bands.
    """
    if not 0.0 < level < 1.0:
        raise ValueError(f"level {level} is not in (0, 1)")
    if absolute_sigma and sigma_new is None:
        raise ValueError("an absolute covariance needs sigma_new for the prediction band")
    value = torch.as_tensor(value, dtype=torch.float64)
    var = torch.as_tensor(var, dtype=torch.float64, device=value.device)
    if sigma_new is not None:
        sigma_new = torch.as_tensor(sigma_new, dtype=torch.float64).to(value.device)
        if sigma_new.dim() > 1 or (sigma_new.dim() == 1 and sigma_new.shape != value.shape):
            raise ValueError(f"sigma_new must be a scalar or hold {value.shape[0]} entries")
        if not bool((torch.isfinite(sigma_new) & (sigma_new > 0)).all()):
            raise ValueError("every sigma_new must be finite and > 0")
    dof = int(dof)
    if absolute_sigma:
        t = float(scipy.stats.norm.ppf((1.0 + level) / 2.0))
    else:
        t = float(scipy.stats.t.ppf((1.0 + level) / 2.0, dof)) if dof > 0 else float("nan")
    if dof > 0 and not np.isinf(np.asarray(cov, dtype=np.float64)).any():
        se_fit = torch.sqrt(torch.clamp(var, min=0.0))
        half_ci = t * se_fit
        if absolute_sigma:
            noise = sigma_new * sigma_new
        elif sigma_new is None:
            noise = float(rss) / dof
        else:
            noise = (float(rss) / dof) * (sigma_new * sigma_new)
        half_pi = t * torch.sqrt(se_fit * se_fit + noise)
    else:
        se_fit = torch.full_like(value, float("inf"))
        half_ci = half_pi = se_fit
    return Prediction(value=value, se_fit=se_fit, ci_low=value - half_ci, ci_high=value + half_ci,
                      pi_low=value - half_pi, pi_high=value + half_pi, level=float(level), t=t, dof=dof)


def predict(fits, X_new, covs=None, level=0.95, engine=None, dtype=None, sigma_new=None):
    """Values of every fit of ``fits`` at the points ``X_new``, and with ``covs`` their confidence and
    prediction bands.

    ``fits``: ``bfgs()`` / ``bfgs_batch()`` 4-tuples ``(string, consts, loss, skeleton)``; an
    ``Exception`` or ``None`` in the list gives ``None``.  ``X_new``: ``[N, d]`` or ``[1, N, d]`` on any
    device; ``x_j`` reads column j-1, as in ``covariances``.  ``covs``: the list ``covariances(fits,
    X_train, y_train)`` returned (without it only ``value`` is computed).  ``dtype``: arithmetic of the
    sweep, ``fitter.F64`` or ``fitter.F32``; by default fp32 for fp32 points and fp64 otherwise, as the
    fit's final score.  ``sigma_new``: a scalar or ``[N]``, the sigma of a new observation at each point
    (see ``bands``); required when a covariance is absolute (``covariances(..., absolute_sigma=True)``),
    ``ValueError`` otherwise.  Returns one ``Prediction`` (or ``None``) per entry, with device float64
    tensors on the engine's device.

    The whole list is one ``vsr_predict`` call on ``engine`` (default: the process-wide engine of X's
    device, or of the current CUDA device); its points and programs are replaced.  Conventions (see
    ``bands`` for the rest): constants the prune fixed at ``0.0`` carry no variance; the variance is
    always fp64 arithmetic; a value is numpy's (nan where ``f`` is not real, +-inf on overflow); a fit
    with more than ``isa.MAX_DUAL`` constants gets nan variances.
    """
    X = torch.as_tensor(X_new)
    if X.dim() == 3:
        X = X[0]
    if covs is not None and len(covs) != len(fits):
        raise ValueError(f"{len(covs)} covariances for {len(fits)} fits")
    out = [None] * len(fits)
    items = []
    for i, f in enumerate(fits):
        if f is None or isinstance(f, Exception):
            continue
        if covs is not None and covs[i] is None:
            raise ValueError(f"fit {i} has no covariance")
        if covs is not None and covs[i].absolute_sigma and sigma_new is None:
            raise ValueError(f"fit {i} has an absolute covariance: its prediction band needs sigma_new")
        items.append((i, str(f[3]), np.asarray(f[1], dtype=np.float64).reshape(-1)))
    if not items:
        return out
    dt = dtype if dtype is not None else (fitter.F32 if X.dtype == torch.float32 else fitter.F64)
    progs = _compile([(skel, c.shape[0]) for _, skel, c in items])
    eng = engine if engine is not None else fitter.get_engine(X.device if X.is_cuda else None)
    eng.set_points(X, torch.zeros(X.shape[0], dtype=torch.float64), dtypes=(dt,),
                   n_vars=max(1, max(p.var_mask.bit_length() for p in progs)))
    eng.set_programs(progs)
    kmax = max(1, max(c.shape[0] for _, _, c in items))
    consts = np.zeros((len(items), kmax))
    cov = np.zeros((len(items), kmax, kmax)) if covs is not None else None
    for j, (i, _, c) in enumerate(items):
        k = c.shape[0]
        consts[j, :k] = c
        if cov is not None:
            cov[j, :k, :k] = device_cov(covs[i].cov)
    value, var = eng.predict(np.arange(len(items)), torch.from_numpy(consts),
                             cov=torch.from_numpy(cov) if cov is not None else None, dtype=dt)
    for j, (i, _, _) in enumerate(items):
        if cov is None:
            out[i] = Prediction(value=value[j], se_fit=None, ci_low=None, ci_high=None, pi_low=None,
                                pi_high=None, level=float(level), t=None, dof=None)
        else:
            cv = covs[i]
            out[i] = bands(value[j], var[j], cv.cov, cv.rss, cv.dof, level, sigma_new=sigma_new,
                           absolute_sigma=cv.absolute_sigma)
    return out
