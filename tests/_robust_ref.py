"""Host twin of the robust-loss factors of the device sweeps and Gram kernel (``vsr_kernels.cuh``,
``robust_factors`` / ``robust_step``), in numpy fp64 with the device's formation order.  The GPU tests use
it as the reference; ``test_robust_host.py`` checks it against mpmath and scipy.

``z = w r^2 / C^2``; ``q = rho(z) / z`` (1 at z = 0), ``g = rho'(z)``, ``sbar = max(rho' + 2 z rho'', 2^-52)``.
At ``z = inf`` (overflow from a finite residual) ``q = g = 0``, ``sbar = 2^-52`` and the cost is ``rho_inf``.
"""
import numpy as np

LOSSES = ("linear", "soft_l1", "huber", "cauchy", "arctan")
ROBUST = LOSSES[1:]
EPS = 2.0 ** -52
RHO_INF = {"soft_l1": np.inf, "huber": np.inf, "cauchy": np.inf, "arctan": np.pi / 2}


def factors(loss, z):
    """(q, g, sbar) of an array of z >= 0 (inf allowed)."""
    z = np.asarray(z, dtype=np.float64)
    one = np.ones_like(z)
    with np.errstate(all="ignore"):
        if loss == "linear":
            q, g, s = one, one.copy(), one.copy()
        elif loss == "soft_l1":
            t = 1.0 + z
            st = np.sqrt(t)
            q, g = 2.0 / (1.0 + st), 1.0 / st
            s = g / t
        elif loss == "huber":
            big = z > 1.0
            sz = np.sqrt(z)
            q = np.where(big, (2.0 * sz - 1.0) / z, 1.0)
            g = np.where(big, 1.0 / sz, 1.0)
            s = np.where(big, 0.0, 1.0)
        elif loss == "cauchy":
            q = np.where(z == 0.0, 1.0, np.log1p(z) / z)
            g = 1.0 / (1.0 + z)
            s = (1.0 - z) * g * g
        elif loss == "arctan":
            q = np.where(z == 0.0, 1.0, np.arctan(z) / z)
            g = 1.0 / (1.0 + z * z)
            s = (1.0 - 3.0 * z * z) * g * g
        else:
            raise ValueError(loss)
        inf = np.isinf(z)
        q = np.where(inf, 0.0, q)
        g = np.where(inf, 0.0, g)
        s = np.where(inf, 0.0, s)
    return q, g, np.where(s > EPS, s, EPS)


def terms(loss, f_scale, r, w=None):
    """Per-point (cost, gfac, wq, ws) of residuals r (weights w or None) as the device forms them: cost is
    C^2 rho(z) (``(rw q) r``), gfac multiplies df/dc in the gradient (``g rw``), and ``r wq r``, ``ws`` are
    the Gram factors.  A non-finite r gets the linear terms; an overflowing z scipy's rho(inf)."""
    r = np.asarray(r, dtype=np.float64)
    w = np.ones_like(r) if w is None else np.asarray(w, dtype=np.float64)
    c2 = float(f_scale) * float(f_scale)
    with np.errstate(all="ignore"):
        rw = w * r
        z = rw * r * (1.0 / c2)
        q, g, sbar = factors(loss, np.where(np.isfinite(z), z, np.inf))
        fin_r = np.isfinite(r)
        over = fin_r & ~np.isfinite(z)
        q = np.where(fin_r, q, 1.0)
        g = np.where(fin_r, g, 1.0)
        sbar = np.where(fin_r, sbar, 1.0)
        cost = np.where(over, c2 * RHO_INF.get(loss, np.inf), (rw * q) * r)
    return cost, g * rw, w * q, w * sbar


def objective(loss, f_scale, r, tan, w=None):
    """(mean cost, gradient 2/N sum g rw d_t with the sweep's finiteness guard) from residuals and tangents."""
    cost, gf, _, _ = terms(loss, f_scale, r, w)
    n = len(r)
    with np.errstate(all="ignore"):
        gt = gf[:, None] * tan
    gt = np.where(np.abs(gt) <= np.finfo(np.float64).max, gt, 0.0)
    return cost.sum() / n, 2.0 * gt.sum(axis=0) / n


def gram(loss, f_scale, r, J, w=None):
    """(rss = sum C^2 rho(z), J^T W S J) of finite residuals r and Jacobian J."""
    cost, _, _, ws = terms(loss, f_scale, r, w)
    return float(cost.sum()), J.T @ (ws[:, None] * J)
