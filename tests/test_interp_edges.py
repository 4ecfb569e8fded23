"""The interpreter's opcodes at the edges of their domains (g++ host build of csrc/vsr_interp.h).

Every opcode, for its value and its d/dc, in fp64 and fp32, against mpmath at 60 digits (closed-form
derivatives, exact binary inputs): saturation and overflow of tanh / sinh / cosh / exp, asin and acos at
and next to +-1, log and sqrt at 0 and subnormals, tan next to its poles, large POWI exponents and
negative bases, pow's special-case table in both operand roles and |b ln a| up to the overflow edge.
The value-only path (K = 0) and the tangent-carrying path must give the same nan / inf pattern and,
pow aside, the same finite values.  Every handler predecode() can produce runs with live tangents.
The budgets are the tables of tests/_interp_ref.py (ulps of the exact result)."""
import math

import numpy as np
import pytest

import _interp_ref as R
from _interp_ref import CONST, IMM, OP, STACK, VAR, E, mp
from src.visymre.engine import isa

DTYPES = [np.float64, np.float32]
BUILD = "host"


def _ids(d):
    return "f64" if d == np.float64 else "f32"


def _np(fn, x):
    with np.errstate(all="ignore"):
        return fn(x)


def _unary_case(hostsim, name, dtype, n=0):
    opname = "VSR_POWI" if name == "powi" else R.UNARY[name][0]
    if name == "powi":
        xs = R.powi_grid(dtype)
        want_np = _np(lambda v: np.power(v, dtype(n)), xs)
        fval = lambda x: mp.power(x, n)                      # noqa: E731
        fder = lambda x: n * mp.power(x, n - 1)              # noqa: E731
        bv, bt = R.powi_budget(n)
    else:
        _, fval, fder, npf, budget = R.UNARY[name]
        xs = R.unary_grid(name, dtype)
        want_np = _np(npf, xs)
        bv, bt = budget(R.LIB[BUILD][dtype])
    insns, imms, k = R.unary_program(opname, n)
    X = xs.reshape(-1, 1)
    v0, _ = R.host_duals(hostsim, insns, imms, np.zeros(k), X, 0)
    v2, t2 = R.host_duals(hostsim, insns, imms, np.zeros(k), X, 2)
    return xs, want_np, fval, fder, bv, bt, v0, v2, t2


@pytest.mark.parametrize("dtype", DTYPES, ids=_ids)
@pytest.mark.parametrize("name", sorted(R.UNARY) + [f"powi{n}" for n in R.POWI_N])
def test_unary_value_and_tangent_at_the_edges(hostsim, name, dtype):
    n = int(name[4:]) if name.startswith("powi") else 0
    xs, want_np, fval, fder, bv, bt, v0, v2, t2 = _unary_case(hostsim, name[:4] if n else name, dtype, n)
    for i, x in enumerate(xs):
        what = f"{name}({float(x)!r}) {_ids(dtype)}"
        ref = R.exact(fval, x) if not math.isnan(x) else None
        # value-only and tangent-carrying evaluation: the same value, bit for bit
        assert (math.isnan(v0[i]) and math.isnan(v2[i])) or v0[i] == v2[i], f"{what}: K=0 {v0[i]!r} K=2 {v2[i]!r}"
        R.check_value(v0[i], float(want_np[i]), ref, bv, dtype, what)
        if not math.isfinite(want_np[i]):
            continue
        # d/dc0 of op(x_1 - c0) + c1 is -f'(x_1); d/dc1 is 1
        assert t2[i, 1] == 1.0, what
        if name == "sqrt" and x == 0:
            assert -t2[i, 0] == math.copysign(math.inf, x), what   # 0.5 / +-0, IEEE's signed zero
            continue
        R.check_point(-t2[i, 0], R.exact(fder, x), bt, dtype, "d/dc " + what)


def test_the_corrected_rules_at_the_points_that_exposed_them(hostsim):
    """tanh in saturation, asin / acos next to +-1: the exact derivative, not the cancelled one."""
    for name, x, dtype in [("tanh", 19.5, np.float64), ("tanh", 25.0, np.float64), ("tanh", 10.0, np.float32),
                           ("asin", 1 - 2.0 ** -30, np.float64), ("acos", -(1 - 2.0 ** -40), np.float64),
                           ("asin", np.float32(0.999), np.float32)]:
        insns, imms, k = R.unary_program(R.UNARY[name][0])
        _, t = R.host_duals(hostsim, insns, imms, np.zeros(k), np.array([[x]], dtype=dtype), 2)
        ref = R.exact(R.UNARY[name][2], dtype(x))
        R.check_point(-t[0, 0], ref, R.UNARY[name][4](R.LIB[BUILD][dtype])[1], dtype, f"d {name}({x!r})")
        assert -t[0, 0] != 0.0


@pytest.mark.parametrize("dtype", DTYPES, ids=_ids)
@pytest.mark.parametrize("prog", [p[0] for p in R.pow_programs()])
def test_pow_both_roles_special_cases_and_overflow_edge(hostsim, prog, dtype):
    name, insns, k, roles = next(p for p in R.pow_programs() if p[0] == prog)
    AB = R.pow_table(dtype)
    want_np = _np(lambda ab: np.power(ab[:, 0], ab[:, 1]), AB)
    imms = np.zeros(1)
    v0, _ = R.host_duals(hostsim, insns, imms, np.zeros(k), AB, 0)
    vk, tk = R.host_duals(hostsim, insns, imms, np.zeros(k), AB, k)
    lib = R.LIB[BUILD][dtype]
    for i, (a, b) in enumerate(AB):
        what = f"{name} {float(a)!r}**{float(b)!r} {_ids(dtype)}"
        if not (math.isfinite(a) and math.isfinite(b)):
            ref = None if math.isnan(want_np[i]) else mp.mpf(float(want_np[i]))   # IEEE special cases
        else:
            ref = R.exact(mp.power, a, b)
        blna = abs(float(b) * math.log(float(a))) if 0 < a < np.inf and math.isfinite(b) else 0.0
        R.check_value(v0[i], float(want_np[i]), ref, lib["pow"], dtype, "K=0 " + what)
        R.check_value(vk[i], float(want_np[i]), ref, R.pow_dual_budget(lib, blna, dtype), dtype,
                      f"K={k} " + what)
        # the two paths: the same nan / inf pattern (inf ** 0 == 1 on both)
        assert math.isnan(v0[i]) == math.isnan(vk[i]) and (math.isfinite(v0[i]) == math.isfinite(vk[i])), what
        assert vk[i] == v0[i] or math.isfinite(v0[i]) or math.isnan(v0[i]), what
        assert tk[i, k - 1] == 1.0, what
        if a == np.inf and b == 0:
            # the existing rules at inf ** 0: d/da = b a^(b-1) = 0 * (1 / inf) = 0, d/db = f ln a = inf
            for j, role in enumerate(roles):
                assert (tk[i, j] == 0.0) if role == "a" else (tk[i, j] == -np.inf), (what, tk[i])
        ex = R.pow_exact(a, b)
        if ex is None or not math.isfinite(want_np[i]) or R.classify(ex[0], dtype) != "normal":
            continue
        bt = R.pow_dual_budget(lib, blna, dtype)
        for j, role in enumerate(roles):
            ref_d = ex[1] if role == "a" else ex[2]
            R.check_point(-tk[i, j], ref_d, bt + (1 if role == "a" else lib["log"] + 0.5), dtype,
                          f"d/d{role} " + what)


@pytest.mark.parametrize("dtype", DTYPES, ids=_ids)
def test_zero_tangent_stays_zero_at_infinite_derivatives(hostsim, dtype):
    """sqrt at 0, asin / acos at +-1: an exactly zero tangent times the infinite derivative stays 0."""
    for opname, xs in [("VSR_SQRT", [0.0]), ("VSR_ASIN", [1.0, -1.0]), ("VSR_ACOS", [1.0, -1.0])]:
        # op(x_1 + c0 * x_2) at x_2 = 0: the argument is x_1, its tangent an exact 0
        insns = np.array([E("VSR_LOAD", CONST, 0, 0, 1), E("VSR_MUL", VAR, 1, 1, 0), E("VSR_ADD", VAR, 0, 1, 0),
                          E(opname, 0, 0, 1), E("VSR_END")], dtype=np.uint64)
        X = np.array([[x, 0.0] for x in xs], dtype=dtype)
        v, t = R.host_duals(hostsim, insns, np.zeros(1), np.ones(1), X, 1)
        assert np.isfinite(v).all() and (t == 0.0).all(), (opname, v, t)


@pytest.mark.parametrize("dtype", DTYPES, ids=_ids)
@pytest.mark.parametrize("name", ["tanh", "asin", "acos", "sqrt", "log", "exp", "atan", "inv", "powi-7"])
def test_sweep_drops_non_finite_terms(hostsim, name, dtype):
    """hostsim_loss_grad (the sweep the fit runs) on an edge grid: mean r^2 and the mean of 2 r g over the
    exact per-point f and g, with the terms the sweep drops (non-finite r * g) dropped."""
    import ctypes
    n = -7 if name == "powi-7" else 0
    base = "powi" if n else name
    xs, want_np, fval, fder, bv, bt, v0, v2, t2 = _unary_case(hostsim, base, dtype, n)
    keep = np.isfinite(want_np)
    xs = xs[keep]
    y = np.full(xs.shape[0], 0.25, dtype=dtype)
    insns, imms, k = R.unary_program("VSR_POWI" if n else R.UNARY[name][0], n)
    # points whose terms the fp64 sum could overflow on say nothing about the rule: leave them out
    cap = np.finfo(np.float64).max / (8 * xs.shape[0])
    pts, v_ref, g_ref = [], [], []
    for x in xs:
        f, d = R.exact(fval, x), R.exact(fder, x)
        r = f - mp.mpf(float(y[0]))
        if r * r > cap or (d is not None and R.classify(d, dtype) == "normal" and abs(2 * r * d) > cap):
            continue
        pts.append(x)
        v_ref.append(f)
        g_ref.append([None if d is None else -d, mp.mpf(1)])
    xs = np.array(pts, dtype=dtype)
    y = y[:xs.shape[0]]
    want_l, bnd_l, want_g, bnd_g = R.sweep_bounds(v_ref, g_ref, y, bv, bt, dtype)
    loss = ctypes.c_double()
    grad = np.zeros(k)
    Xc = np.ascontiguousarray(xs.reshape(1, -1))
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    rc = hostsim.hostsim_loss_grad(p(np.ascontiguousarray(insns)), p(imms), p(np.zeros(k)), ctypes.c_int(k), p(Xc),
                                   p(y), ctypes.c_long(xs.shape[0]), ctypes.c_int(0 if dtype == np.float64 else 1),
                                   ctypes.c_int(1), ctypes.byref(loss), p(grad))
    assert rc == 0
    if mp.isinf(want_l) or want_l > np.finfo(np.float64).max:
        assert math.isinf(loss.value)
    else:
        assert abs(mp.mpf(loss.value) - want_l) <= bnd_l, (name, loss.value, want_l, bnd_l)
    for j in range(k):
        assert abs(mp.mpf(grad[j]) - want_g[j]) <= bnd_g[j], (name, j, grad[j], want_g[j], bnd_g[j])


# ---- handler coverage ---------------------------------------------------------------------------------
COV_K = 16
COV_C = [0.35 + 0.025 * j for j in range(COV_K)] + [0.6]          # c16: past the tangent slots


def _coverage_programs():
    """Hand-assembled programs that together reach every handler id predecode() produces (0..118), each
    binary form with live tangents in acc and, where the operand has them, in the operand too.  Every
    argument stays in (0.1, 1) so each op is in its domain.  Returns [(insns, imms, k)]."""
    progs = []
    imms = np.array([0.75, 1.25])
    binops = ["VSR_LOAD", "VSR_ADD", "VSR_SUB", "VSR_RSUB", "VSR_MUL", "VSR_DIV", "VSR_RDIV", "VSR_POW", "VSR_RPOW"]
    for op in binops:
        # VAR / IMM operands: acc = c0 * x_1 carries tangent 0
        for src, idx in ((VAR, 1), (IMM, 0)):
            progs.append([E("VSR_LOAD", CONST, 0, 0, 1), E("VSR_MUL", VAR, 0, 1, 0), E(op, src, idx, 1, 0),
                          E("VSR_ADD", CONST, 1, 1 if op != "VSR_LOAD" else 0, 2), E("VSR_END")])
        # CONST operand already live in acc (not fresh): (c0 * x_1) op c0
        progs.append([E("VSR_LOAD", CONST, 0, 0, 1), E("VSR_MUL", VAR, 0, 1, 0), E(op, CONST, 0, 1, 1), E("VSR_END")])
        # a constant past the tangent slots (no tangent): (c0 * x_1) op c16
        progs.append([E("VSR_LOAD", CONST, 0, 0, 1), E("VSR_MUL", VAR, 0, 1, 0),
                      E(op, CONST, 16, 0 if op == "VSR_LOAD" else 1, 0), E("VSR_END")])
        # STACK operand, tangents on both sides (c0, c2 below; c1, c2 in acc), at stack depth 1 and 2
        side_b = [E("VSR_LOAD", CONST, 0, 0, 1), E("VSR_MUL", VAR, 2, 1, 0), E("VSR_ADD", CONST, 2, 1, 4)]
        side_a = [E("VSR_LOAD", CONST, 1, 0, 2), E("VSR_MUL", VAR, 1, 2, 0), E("VSR_MUL", CONST, 2, 2, 4)]
        progs.append(side_b + [E("VSR_PUSH", 0, 0, 5)] + side_a + [E(op, STACK, 0, 6, 5), E("VSR_END")])
        outer = [E("VSR_LOAD", CONST, 3, 0, 8), E("VSR_MUL", VAR, 3, 8, 0), E("VSR_PUSH", 0, 0, 8)]
        progs.append(outer + side_b + [E("VSR_PUSH", 0, 0, 5)] + side_a + [E(op, STACK, 0, 6, 5),
                     E("VSR_MUL", IMM, 1, 5 if op == "VSR_LOAD" else 7, 0),
                     E("VSR_ADD", STACK, 0, 5 if op == "VSR_LOAD" else 7, 8), E("VSR_END")])
    # unary ops on c0 * x_1 + c1 * x_2 (in (0.1, 0.8)), POWI at two exponents
    for opn in range(OP["VSR_NEG"], OP["VSR_OP_COUNT"]):
        name = isa.OP_NAME[opn]
        for n in ((3, -2) if name == "VSR_POWI" else (0,)):
            progs.append([E("VSR_LOAD", CONST, 0, 0, 1), E("VSR_MUL", VAR, 0, 1, 0), E("VSR_PUSH", 0, 0, 1),
                          E("VSR_LOAD", CONST, 1, 0, 2), E("VSR_MUL", VAR, 1, 2, 0), E("VSR_ADD", STACK, 0, 2, 1),
                          E(name, 0, n, 3), E("VSR_END")])
    # fresh constants c_j for every tangent slot j: LOAD c_j, and acc (live in another slot) ADD / SUB / MUL c_j
    for j in range(COV_K):
        o = (j + 5) % COV_K
        progs.append([E("VSR_LOAD", CONST, j, 0, 1 << j), E("VSR_MUL", VAR, 0, 1 << j, 0), E("VSR_END")])
        for op in ("VSR_ADD", "VSR_SUB", "VSR_MUL"):
            progs.append([E("VSR_LOAD", CONST, o, 0, 1 << o), E("VSR_MUL", VAR, 1, 1 << o, 0),
                          E(op, CONST, j, 1 << o, 1 << j), E("VSR_END")])
    out = []
    for p in progs:
        wide = any(isa.decode(w)[1] == CONST and isa.decode(w)[2] == COV_K for w in p if isa.decode(w)[0] != OP["VSR_END"])
        out.append((np.array(p, dtype=np.uint64), imms, COV_K + 1 if wide else COV_K))
    return out


def _coverage_points(dtype):
    rng = np.random.RandomState(17)
    return rng.uniform(0.15, 0.9, size=(7, 4)).astype(dtype)


# handlers that run, but never with a live tangent: (id, reason)
NO_TANGENT_RULE = {
    0: "END has no operand",
    2 + (0 << 2) + CONST: "LOAD of a constant in a tangent slot is always a fresh-constant handler; this one is "
                          "reached only by constants past the 16 tangent slots, which carry no tangent",
}


def test_every_handler_runs_with_live_tangents(hostsim):
    seen, live = set(), set()
    for insns, imms, k in _coverage_programs():
        R.validate(insns, k, len(imms))
        for w in insns:
            h = R.predecode(hostsim, w)
            seen.add(h)
            _, _, _, am, bm = isa.decode(w)
            if am or bm:
                live.add(h)
    assert seen == set(range(119)), sorted(set(range(119)) - seen)
    assert set(range(119)) - live == set(NO_TANGENT_RULE), sorted(set(range(119)) - live)


@pytest.mark.parametrize("dtype", DTYPES, ids=_ids)
def test_coverage_programs_match_the_exact_isa(hostsim, dtype):
    """Each coverage program's value and 16 tangents against the ISA run in mpmath (closed-form rules),
    and its value-only run: the same values."""
    X = _coverage_points(dtype)
    eps = float(np.finfo(dtype).eps)
    for pi, (insns, imms, k) in enumerate(_coverage_programs()):
        c = np.array(COV_C[:k], dtype=dtype).astype(np.float64)
        v0, _ = R.host_duals(hostsim, insns, imms, c, X, 0)
        v, t = R.host_duals(hostsim, insns, imms, c, X, COV_K)
        if any(isa.decode(w)[0] in (OP["VSR_POW"], OP["VSR_RPOW"]) for w in insns):
            np.testing.assert_allclose(v0, v, rtol=16 * eps, atol=0)   # libm pow against exp(b ln a)
        else:
            assert np.array_equal(v0, v), (pi, isa.disassemble(insns))
        for i in range(X.shape[0]):
            rv, rd = R.mp_run(insns, imms, c, X[i], COV_K)
            scale = max([abs(rv)] + [abs(d) for d in rd])
            tol = 64 * eps * scale
            assert abs(mp.mpf(v[i]) - rv) <= tol, (pi, i, v[i], rv, isa.disassemble(insns))
            for j in range(COV_K):
                assert abs(mp.mpf(t[i, j]) - rd[j]) <= tol, (pi, i, j, t[i, j], rd[j], isa.disassemble(insns))
