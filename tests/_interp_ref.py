"""Arbitrary-precision reference for the interpreter's opcodes (shared by the CPU and GPU edge tests).

Values and derivatives come from mpmath at 60 digits, evaluated at the exact binary inputs the
interpreter sees; derivatives are closed forms, never a lambdified sympy derivative (which repeats the
kernel's own cancelling formulas).  The nan / +-inf pattern of values comes from numpy in the same
dtype, whose semantics the project promises.

Budgets are in ulps of the exact result (the ulp of its binade in the dtype, 2^-1074 / 2^-149 below
the normal range).  ``LIB`` holds the documented maximum ulp errors of the math libraries: the CUDA C
Programming Guide's table for the device build (``cuda``) and glibc's x86-64 figures for the g++ host
build (``host``).  The tangent budgets add up the roundings of each rule on top of them.
"""
import ctypes
import math

import mpmath as mpm
import numpy as np

from src.visymre.engine import isa

mp = mpm.mp
mp.dps = 60

OP = isa.OP
SRC = isa.SRC
VAR, CONST, IMM, STACK = SRC["VSR_SRC_VAR"], SRC["VSR_SRC_CONST"], SRC["VSR_SRC_IMM"], SRC["VSR_SRC_STACK"]

# documented max ulp errors: {build: {dtype: {function: ulps}}}
LIB = {
    "cuda": {
        np.float64: dict(exp=1, log=1, sin=2, cos=2, tan=2, asin=2, acos=2, atan=2, sinh=2, cosh=1, tanh=1, pow=2),
        np.float32: dict(exp=2, log=1, sin=2, cos=2, tan=4, asin=2, acos=2, atan=2, sinh=3, cosh=2, tanh=2, pow=4),
    },
    "host": {
        np.float64: dict(exp=1, log=1, sin=1, cos=1, tan=1, asin=1, acos=1, atan=1, sinh=2, cosh=2, tanh=2, pow=1),
        np.float32: dict(exp=1, log=1, sin=1, cos=1, tan=1, asin=1, acos=1, atan=1, sinh=2, cosh=2, tanh=2, pow=1),
    },
}
# sqrt and division are correctly rounded in both builds: 0.5 ulp


def _sech2(x):
    return 1 / mp.cosh(x) ** 2


def _datan(x):
    return 1 / (1 + x * x)


def _rsqrt1m(x):
    """1 / sqrt(1 - x^2): +inf at +-1, undefined outside."""
    s = 1 - x * x
    if s < 0:
        return None
    return mp.inf if s == 0 else 1 / mp.sqrt(s)


# name: (opcode, exact f, exact f', numpy f, budget(lib) -> (value ulps, tangent ulps)).
# A budget of n ulps bounds the relative error by n u (u = 2^-p): a library result within L ulp is
# within 2 L u, a correctly rounded operation within u, so the tangent budgets below count
# 2 L per library call and 1 per rounding of the rule.
UNARY = {
    "neg": ("VSR_NEG", lambda x: -x, lambda x: mp.mpf(-1), np.negative, lambda L: (0, 0)),
    "abs": ("VSR_ABS", abs, lambda x: mp.sign(x), np.abs, lambda L: (0, 0)),
    "sign": ("VSR_SIGN", mp.sign, lambda x: mp.mpf(0), np.sign, lambda L: (0, 0)),
    # -f*f: f, the square, the product
    "inv": ("VSR_INV", lambda x: 1 / x, lambda x: -1 / (x * x), np.reciprocal, lambda L: (0.5, 3)),
    # 0.5 / f: f, the division
    "sqrt": ("VSR_SQRT", mp.sqrt, lambda x: mp.inf if x == 0 else 1 / (2 * mp.sqrt(x)), np.sqrt, lambda L: (0.5, 2)),
    "exp": ("VSR_EXP", mp.exp, mp.exp, np.exp, lambda L: (L["exp"], L["exp"])),
    # 1 / a
    "log": ("VSR_LOG", mp.log, lambda x: 1 / x, np.log, lambda L: (L["log"], 0.5)),
    "sin": ("VSR_SIN", mp.sin, mp.cos, np.sin, lambda L: (L["sin"], L["cos"])),
    "cos": ("VSR_COS", mp.cos, lambda x: -mp.sin(x), np.cos, lambda L: (L["cos"], L["sin"])),
    # 1 + f*f: f twice, the product, the sum
    "tan": ("VSR_TAN", mp.tan, lambda x: 1 + mp.tan(x) ** 2, np.tan, lambda L: (L["tan"], 4 * L["tan"] + 2)),
    # 1 / sqrt((1 - a)(1 + a)): 1 - a exact from |a| = 1/2 on, 1 + a, the product, halved by sqrt,
    # sqrt, the division
    "asin": ("VSR_ASIN", mp.asin, _rsqrt1m, np.arcsin, lambda L: (L["asin"], 4)),
    "acos": ("VSR_ACOS", mp.acos, lambda x: None if _rsqrt1m(x) is None else -_rsqrt1m(x), np.arccos,
             lambda L: (L["acos"], 4)),
    # 1 / (1 + a*a): the square, the sum, the division
    "atan": ("VSR_ATAN", mp.atan, _datan, np.arctan, lambda L: (L["atan"], 3)),
    "sinh": ("VSR_SINH", mp.sinh, mp.cosh, np.sinh, lambda L: (L["sinh"], L["cosh"])),
    "cosh": ("VSR_COSH", mp.cosh, mp.sinh, np.cosh, lambda L: (L["cosh"], L["sinh"])),
    # 4e / (1 + e)^2, e = exp(-2|a|) (-2|a| exact): the result's sensitivity to e is at most 1, then
    # 1 + e (twice, squared), the product and the division
    "tanh": ("VSR_TANH", mp.tanh, _sech2, np.tanh, lambda L: (L["tanh"], 2 * L["exp"] + 4)),
}


def powi_budget(n):
    """x^|n| by binary powering: at most |n| - 1 roundings; a negative n adds the reciprocal; the
    tangent n f / a (or n a^(|n|-1)) two more."""
    m = abs(n)
    return (m - 1 + (1 if n < 0 else 0), m + 2)


POW_LIM = {np.float64: 708.0, np.float32: 87.0}


def pow_dual_budget(lib, blna, dtype):
    """The tangent-carrying path's a**b: exp(b ln a) while |b ln a| < 708 (87 in fp32).  ln a within
    L_log ulp and the rounding of b ln a put (2 L_log + 1) |b ln a| u into the exponent, exp adds
    2 L_exp u: 2.4e-13 of relative error at |b ln a| = 708 in fp64.  libm's pow elsewhere."""
    if not abs(blna) < POW_LIM[dtype]:
        return lib["pow"]
    return 2 * lib["exp"] + (2 * lib["log"] + 1) * abs(blna)


# ---- ulps ------------------------------------------------------------------------------------------
_FMT = {np.float64: (53, -1022, np.finfo(np.float64).max), np.float32: (24, -126, float(np.finfo(np.float32).max))}


def ulp_of(ref, dtype):
    p, emin, _ = _FMT[dtype]
    if ref == 0:
        return mp.ldexp(1, emin - p + 1)
    e = mp.frexp(ref)[1] - 1
    return mp.ldexp(1, max(e, emin) - p + 1)


def classify(ref, dtype):
    """'nan' | 'inf' | 'normal' | 'tiny' (below the normal range, not zero) | 'zero' of the exact result."""
    if ref is None or mp.isnan(ref):
        return "nan"
    if mp.isinf(ref):
        return "inf"
    p, emin, big = _FMT[dtype]
    if ref == 0:
        return "zero"
    if abs(ref) > big:
        return "inf"
    if abs(ref) < mp.ldexp(1, emin):
        return "tiny"
    return "normal"


def check_point(got, ref, budget, dtype, what):
    """One result against the exact one (None: undefined, i.e. nan).  Normal results: within `budget`
    ulps.  Exact results past the largest finite value: +-inf of the same sign.  Exact results below
    the normal range: a finite value no larger than the smallest normal, of the same sign or zero
    (where a formula underflows is a convention, not an accuracy).  Exact zero: exactly zero.  An
    exact value within the budget of the overflow threshold accepts either side of it."""
    p, emin, big = _FMT[dtype]
    cls = classify(ref, dtype)
    msg = f"{what}: got {got!r}, exact {'nan' if ref is None else mp.nstr(ref, 17)}"
    if cls == "nan":
        assert math.isnan(got), msg
        return
    w = (budget + 1) * mp.ldexp(1, 1 - p)
    edge = mp.mpf(big) * (1 - w) < abs(ref) < mp.mpf(big) * (1 + w)
    if cls == "inf" and not (edge and math.isfinite(got)):
        assert math.isinf(got) and (got > 0) == (ref > 0), msg
        return
    if cls == "zero":
        assert got == 0.0, msg
        return
    if cls == "tiny":
        assert math.isfinite(got) and abs(got) <= 2.0 ** emin and (got == 0 or (got > 0) == (ref > 0)), \
            msg + " (below the normal range)"
        return
    if edge and math.isinf(got) and (got > 0) == (ref > 0):
        return
    assert math.isfinite(got), msg
    err = abs(mp.mpf(got) - ref) / ulp_of(ref, dtype)
    assert err <= budget, f"{msg}: {float(err):.3g} ulp > {budget}"


def check_value(got, want_np, ref, budget, dtype, what):
    """A value: numpy (same dtype) decides nan and +-inf; a finite numpy value is checked against the
    exact one.  Next to the overflow threshold either side is accepted, as in check_point."""
    if math.isnan(want_np):
        assert math.isnan(got), f"{what}: got {got!r}, numpy nan"
    elif math.isinf(want_np) and (ref is None or classify(ref, dtype) in ("inf", "nan")):
        if ref is not None and not mp.isinf(ref) and math.isfinite(got):
            check_point(got, ref, budget, dtype, what)   # exact value finite: the threshold case
        else:
            assert got == want_np, f"{what}: got {got!r}, numpy {want_np!r}"
    else:
        check_point(got, ref, budget, dtype, what)


def sweep_bounds(v_ref, g_ref, y, bv, bg, dtype):
    """What the sweep must give on a grid: loss = mean r^2 and grad_j = mean of 2 r g_j with the
    non-finite terms dropped (r = f - y), from the exact per-point f and g, and the bound each may miss
    it by: the per-point budgets (`bv` ulps of f, `bg` ulps of g) carried through the terms, plus the
    fp64 summation.  v_ref [N] and g_ref [N, k] are mpf (None = nan)."""
    p, emin, _ = _FMT[dtype]
    N = len(v_ref)
    with mp.workdps(60):
        loss, lerr = mp.mpf(0), mp.mpf(0)
        k = len(g_ref[0])
        grad, gerr, gabs = [mp.mpf(0)] * k, [mp.mpf(0)] * k, [mp.mpf(0)] * k
        for i in range(N):
            f = v_ref[i]
            r = f - mp.mpf(float(y[i]))
            dv = bv * ulp_of(f, dtype) + mp.ldexp(1, emin - p + 1)
            loss += r * r
            lerr += 2 * abs(r) * dv + dv * dv
            for j in range(k):
                g = g_ref[i][j]
                if g is None or classify(g, dtype) in ("inf", "nan"):
                    continue  # the tangent is not finite: the sweep drops the term
                t = 2 * r * g
                grad[j] += t
                gabs[j] += abs(t)
                dg = bg * ulp_of(g, dtype) + mp.ldexp(1, emin)
                gerr[j] += 2 * (abs(r) * dg + abs(g) * dv + dv * dg)
        s = 4 * N * mp.mpf(2) ** -53
        loss_b = (lerr + s * loss) / N
        grad_b = [(gerr[j] + s * gabs[j]) / N for j in range(k)]
        return loss / N, loss_b, [g / N for g in grad], grad_b


def exact(fn, *args):
    """fn at the exact arguments (mpf), None where it is undefined (a domain error: nan in numpy).
    mpmath answers with complex numbers past the real domain, which counts as undefined."""
    try:
        with mp.workdps(60):
            r = fn(*[mp.mpf(float(a)) for a in args])
    except (ZeroDivisionError, ValueError):
        return None
    if isinstance(r, mpm.mpc):
        return r.real if r.imag == 0 else None
    return r


# ---- grids -------------------------------------------------------------------------------------------
def _sym(xs):
    return sorted(set(list(xs) + [-x for x in xs]))


def unary_grid(name, dtype):
    """Edge-of-domain points of one op in `dtype` (plus a few interior points), as dtype values."""
    f64 = dtype == np.float64
    big = float(np.finfo(dtype).max)
    tiny = float(np.finfo(dtype).tiny)
    sub = tiny / 8
    inter = [0.3, 0.7, 1.3, 2.9]
    base = [0.0, np.inf, np.nan]
    if name in ("tanh", "sinh", "cosh", "exp"):
        ov = 709.78 if f64 else 88.72
        ovh = 710.475 if f64 else 89.415
        pts = [1e-30, 1e-8, 0.5, 1, 2, 5, 9, 10, 15, 19, 19.1, 20, 22, 25, 30, 44, 45, 50, 88, 100,
               300, 354, 355, 360, 400, 700, 709, ov, ovh, 711, 1000, 1e30, big]
        if name == "exp":
            pts += [-745.2, -745.1, -744, -740, -720, -708.5, -708.3, -700, -103.9, -103.2, -87.4, -87.3, -80]
        xs = _sym(pts)
    elif name in ("asin", "acos"):
        kmax = 53 if f64 else 24
        eps = float(np.finfo(dtype).eps)
        pts = [1.0, 1 + eps, 1 + 2 * eps, 1.5, 2.0, sub, 0.5, 0.9] + [1 - 2.0 ** -k for k in range(1, kmax + 1)]
        xs = _sym(pts)
    elif name == "log":
        xs = [1.0 - 2.0 ** -k for k in (1, 10, 30, 52)] + [1.0 + 2.0 ** -k for k in (10, 30, 52)] + \
             [np.nextafter(dtype(1), dtype(2)), np.nextafter(dtype(1), dtype(0)), sub, tiny / 2 ** 20, tiny,
              -tiny, -1.0, -np.inf, big, 1e-300, 1e300]
    elif name == "sqrt":
        xs = [sub, tiny / 2 ** 20, tiny, 1e-300, 1e300, big, -0.0, -sub, -1.0, -np.inf, 2.0, 0.25]
    elif name == "tan":
        pi2 = np.pi / 2
        xs = [pi2, np.nextafter(pi2, 0), np.nextafter(pi2, 4), 3 * pi2, np.pi, 1e-300, 1e5, 1e22]
        if not f64:
            p32 = np.float32(pi2)
            xs += [float(p32), float(np.nextafter(p32, np.float32(0))), float(np.nextafter(p32, np.float32(4)))]
        xs = _sym(xs)
    elif name == "atan":
        xs = _sym([1e-300, 1e8, 1e16, 2.0 ** 511, 2.0 ** 511.5, 2.0 ** 512, 2.0 ** 520, 1e300, big, 2.0 ** 63.5,
                   2.0 ** 64, 2.0 ** 70, sub])
    elif name in ("inv", "abs", "sign", "neg"):
        xs = _sym([sub, tiny, 1 / big, 0.5 / big, 1e-300, 1e300, big]) + [-0.0]
    elif name == "sin" or name == "cos":
        xs = _sym([1e-300, np.pi / 2, np.pi, 1e5, 1e22, big, sub])
    else:
        raise KeyError(name)
    out = np.array(list(xs) + inter + [-v for v in inter] + base, dtype=np.float64)
    with np.errstate(over="ignore"):
        out = out.astype(dtype)
    return out


POWI_N = (2, 3, 7, 31, 100, -2, -3, -7, -31, -100)


def powi_grid(dtype):
    f64 = dtype == np.float64
    tiny = float(np.finfo(dtype).tiny)
    xs = _sym([0.5, 0.9, 1.0, 1.1, 1.5, 2.0, 3.0, 10.0, 1e-5, 1e5, 1e30, 1e-30, 1e100 if f64 else 1e10,
               1e-100 if f64 else 1e-10, tiny, tiny / 8, 1e300 if f64 else 1e38]) + [0.0, -0.0, np.inf, -np.inf, np.nan]
    with np.errstate(over="ignore"):
        return np.array(xs, dtype=np.float64).astype(dtype)


def pow_table(dtype):
    """(a, b) pairs: the IEEE / numpy special-case table and |b ln a| up to the overflow edge."""
    big = float(np.finfo(dtype).max)
    sub = float(np.finfo(dtype).tiny) / 8
    spec_a = [0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, np.nan, 0.5, -0.5, 2.0, -2.0, sub, big]
    spec_b = [0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, np.nan, 0.5, -0.5, 2.0, 3.0, -3.0, 2.5, 1e-30, 1e30]
    pairs = [(a, b) for a in spec_a for b in spec_b]
    lim = 709.0 if dtype == np.float64 else 88.0
    for a in (1.0 + 2.0 ** -20, 1.5, 2.0, 10.0, 0.25, 1e-3, 1e10, 1e-10, 2.0 ** -60):
        la = math.log(a)
        for L in (1e-6, 0.5, 3.0, 40.0, 0.5 * lim, 0.9 * lim, lim, 1.01 * lim, 1.05 * lim):
            for s in (1, -1):
                b = float(np.array(s * L / la, dtype=dtype))
                pairs.append((a, b))
    arr = np.array(pairs, dtype=np.float64)
    with np.errstate(over="ignore"):
        return arr.astype(dtype)


# ---- programs ------------------------------------------------------------------------------------------
def E(opname, src=0, idx=0, am=0, bm=0):
    return isa.encode(OP[opname], src, idx & 0xFFFF, am, bm)


def unary_program(opname, n=0, tail=True):
    """op(x_1 - c0) [+ c1]: at c0 = c1 = 0 the op's argument is x_1 exactly (signed zeros, inf and nan
    included), the tangent of c0 is -f'(x_1) and that of c1 is 1."""
    w = [E("VSR_LOAD", VAR, 0), E("VSR_SUB", CONST, 0, 0, 1), E(opname, 0, n, 1)]
    if tail:
        w.append(E("VSR_ADD", CONST, 1, 1, 2))
    w.append(E("VSR_END"))
    return np.array(w, dtype=np.uint64), np.zeros(1), 2 if tail else 1


def pow_programs():
    """(name, insns, k, roles) of the four places a power's operands can come from, each f = x_1 ** x_2 at
    c = 0 with a trailing + c_last: roles[j] = 'a' / 'b' says which operand c_j shifts (by -c_j)."""
    progs = []
    # POW VAR: acc (base, live) ** column
    progs.append(("pow_var", [E("VSR_LOAD", VAR, 0), E("VSR_SUB", CONST, 0, 0, 1), E("VSR_POW", VAR, 1, 1, 0),
                              E("VSR_ADD", CONST, 1, 1, 2), E("VSR_END")], 2, "a"))
    # RPOW VAR: column ** acc (exponent, live)
    progs.append(("rpow_var", [E("VSR_LOAD", VAR, 1), E("VSR_SUB", CONST, 0, 0, 1), E("VSR_RPOW", VAR, 0, 1, 0),
                               E("VSR_ADD", CONST, 1, 1, 2), E("VSR_END")], 2, "b"))
    # POW STACK: acc (base) ** popped (exponent), both live
    progs.append(("pow_stack", [E("VSR_LOAD", VAR, 1), E("VSR_SUB", CONST, 1, 0, 2), E("VSR_PUSH", 0, 0, 2),
                                E("VSR_LOAD", VAR, 0), E("VSR_SUB", CONST, 0, 0, 1), E("VSR_POW", STACK, 0, 1, 2),
                                E("VSR_ADD", CONST, 2, 3, 4), E("VSR_END")], 3, "ab"))
    # RPOW STACK: popped (base) ** acc (exponent), both live
    progs.append(("rpow_stack", [E("VSR_LOAD", VAR, 0), E("VSR_SUB", CONST, 0, 0, 1), E("VSR_PUSH", 0, 0, 1),
                                 E("VSR_LOAD", VAR, 1), E("VSR_SUB", CONST, 1, 0, 2), E("VSR_RPOW", STACK, 0, 2, 1),
                                 E("VSR_ADD", CONST, 2, 3, 4), E("VSR_END")], 3, "ab"))
    return [(n, np.array(w, dtype=np.uint64), k, r) for n, w, k, r in progs]


def pow_exact(a, b):
    """a ** b and its partials (exact), or None where numpy's real pow is nan."""
    a, b = float(a), float(b)
    if math.isnan(a) or math.isnan(b) or not (a > 0 and math.isfinite(a) and math.isfinite(b)):
        return None
    with mp.workdps(60):
        A, B = mp.mpf(a), mp.mpf(b)
        f = mp.power(A, B)
        return f, B * mp.power(A, B - 1), f * mp.log(A)


def validate(insns, k, n_imm):
    """The static checks vsr_upload_programs applies (operand indices, stack discipline, END)."""
    sp = 0
    assert 1 <= len(insns) <= isa.MAX_INSNS and int(insns[-1]) & 0xFF == OP["VSR_END"]
    for w in insns:
        op, src, idx, _, _ = isa.decode(w)
        assert op < OP["VSR_OP_COUNT"]
        if op == OP["VSR_PUSH"]:
            sp += 1
            assert sp <= isa.MAX_STACK
        elif OP["VSR_LOAD"] <= op <= OP["VSR_RPOW"]:
            if src == STACK:
                sp -= 1
                assert sp >= 0
            elif src == VAR:
                assert idx < isa.MAX_VARS
            elif src == CONST:
                assert idx < k
            else:
                assert src == IMM and idx < n_imm


# ---- the ISA in mpmath (forward mode with closed-form rules) -------------------------------------------
def mp_run(insns, imms, c, x, K):
    """Value and K tangents of a program at one point, exact (mpf), following the ISA's masks: an
    operand's tangents are the ones its bmask names (the interpreter carries no others)."""
    with mp.workdps(60):
        c = [mp.mpf(float(v)) for v in c]
        x = [mp.mpf(float(v)) for v in x]
        acc = (mp.mpf(0), [mp.mpf(0)] * K)
        stack = []
        for w in insns:
            op, src, idx, am, bm = isa.decode(w)
            name = isa.OP_NAME[op]
            if name == "VSR_END":
                return acc
            if name == "VSR_PUSH":
                stack.append((acc[0], [acc[1][i] if (am >> i) & 1 else mp.mpf(0) for i in range(K)]))
                continue
            if OP["VSR_LOAD"] <= op <= OP["VSR_RPOW"]:
                if src == STACK:
                    bv, bd = stack.pop()
                    bd = [bd[i] if (bm >> i) & 1 else mp.mpf(0) for i in range(K)]
                elif src == VAR:
                    bv, bd = x[idx], [mp.mpf(0)] * K
                elif src == CONST:
                    bv, bd = c[idx], [mp.mpf(1 if i == idx else 0) for i in range(K)]
                else:
                    bv, bd = mp.mpf(float(imms[idx])), [mp.mpf(0)] * K
                av, ad = acc
                if name == "VSR_LOAD":
                    acc = (bv, bd)
                elif name == "VSR_ADD":
                    acc = (av + bv, [p + q for p, q in zip(ad, bd)])
                elif name == "VSR_SUB":
                    acc = (av - bv, [p - q for p, q in zip(ad, bd)])
                elif name == "VSR_RSUB":
                    acc = (bv - av, [q - p for p, q in zip(ad, bd)])
                elif name == "VSR_MUL":
                    acc = (av * bv, [p * bv + av * q for p, q in zip(ad, bd)])
                elif name == "VSR_DIV":
                    acc = (av / bv, [(p * bv - av * q) / bv ** 2 for p, q in zip(ad, bd)])
                elif name == "VSR_RDIV":
                    acc = (bv / av, [(q * av - bv * p) / av ** 2 for p, q in zip(ad, bd)])
                else:
                    base, ex, dbase, dex = (av, bv, ad, bd) if name == "VSR_POW" else (bv, av, bd, ad)
                    f = mp.power(base, ex)
                    acc = (f, [ex * mp.power(base, ex - 1) * p + f * mp.log(base) * q for p, q in zip(dbase, dex)])
                continue
            av, ad = acc
            if name == "VSR_POWI":
                n = idx - 0x10000 if idx & 0x8000 else idx
                f, fp = mp.power(av, n), n * mp.power(av, n - 1)
            else:
                key = name[4:].lower()
                _, fn, dfn, _, _ = UNARY[key]
                f, fp = fn(av), dfn(av)
            acc = (f, [fp * p for p in ad])
    raise AssertionError("program without END")


# ---- host build --------------------------------------------------------------------------------------
def host_duals(hostsim, insns, imms, c, X, K):
    """(value [N], tangents [N, K]) of the g++ build; X [N, d] in the evaluation dtype."""
    N = X.shape[0]
    Xc = np.ascontiguousarray(X.T)
    cc = np.ascontiguousarray(np.asarray(c, dtype=np.float64).reshape(-1))
    if cc.size == 0:
        cc = np.zeros(1)
    ins = np.ascontiguousarray(insns, dtype=np.uint64)
    im = np.ascontiguousarray(imms, dtype=np.float64)
    val = np.empty(N)
    tan = np.zeros((N, max(K, 1)))
    dt = isa.DTYPE["VSR_F64"] if X.dtype == np.float64 else isa.DTYPE["VSR_F32"]
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    rc = hostsim.hostsim_duals(p(ins), p(im), p(cc), ctypes.c_int(int(cc.size)), p(Xc), ctypes.c_long(N),
                               ctypes.c_int(dt), ctypes.c_int(K), p(val), p(tan))
    assert rc == 0
    return val, tan[:, :K]


def predecode(hostsim, word):
    hostsim.hostsim_predecode.restype = ctypes.c_int
    hostsim.hostsim_predecode.argtypes = [ctypes.c_uint64]
    return hostsim.hostsim_predecode(int(word))
