"""The interpreter's opcodes at the edges of their domains, on the device: the grids and budgets of
tests/test_interp_edges.py (CUDA math library column) through vsr_predict and vsr_eval.

Values: ``Engine.predict`` without a covariance runs the value-only path (K = 0), with one the
tangent-carrying path; both return f64 per point.  Signed per-point tangents without a new entry:
each program ends in ``+ c_last`` (c = 0), so with the covariance 0.5 (e_j e_last^T + e_last e_j^T) the
kernel's fp64 form g^T C g is exactly g_j * g_last = g_j.  Where a tangent is infinite the cross form is
nan (0 * inf), and the unary ops read |g_0| through a program without the trailing constant and
cov = [[1]].  The optimiser's view: vsr_eval's loss and gradient on each grid equal the mean of r^2 and
of 2 r g over the exact per-point f and g, non-finite terms dropped, through the per-pair kernel and
through eval_tile_kernel."""
import math

import numpy as np
import pytest
import torch

import _interp_ref as R
from _interp_ref import OP, mp
from src.visymre.engine import fitter, isa
from src.visymre.engine.compiler import Program
from test_interp_edges import COV_C, COV_K, _coverage_points, _coverage_programs

pytestmark = pytest.mark.gpu
BUILD = "cuda"
DTYPES = [np.float64, np.float32]


def _ids(d):
    return "f64" if d == np.float64 else "f32"


@pytest.fixture(scope="module")
def eng():
    return fitter.Engine("cuda:0")


def _program(insns, imms, k):
    insns = np.asarray(insns, dtype=np.uint64)
    R.validate(insns, k, len(imms))
    vm = 0
    for w in insns:
        op, src, idx, _, _ = isa.decode(w)
        if OP["VSR_LOAD"] <= op <= OP["VSR_RPOW"] and op != OP["VSR_PUSH"] and src == R.VAR:
            vm |= 1 << idx
    return Program(insns=insns, imms=np.asarray(imms, dtype=np.float64), k=k, var_mask=vm,
                   stack_depth=isa.MAX_STACK, n_nodes=1, flops=1)


def _dt(dtype):
    return fitter.F64 if dtype == np.float64 else fitter.F32


def _cross(k):
    """cov rows j < k - 1: 0.5 (e_j e_last^T + e_last e_j^T)."""
    C = np.zeros((k - 1, k, k))
    for j in range(k - 1):
        C[j, j, k - 1] = C[j, k - 1, j] = 0.5
    return C


def _device(e, progs, X, dtype):
    """[(value K=0, value tangent path, g [N, k-1] signed or nan)] of programs whose last constant is
    added at the end, all constants 0."""
    N = X.shape[0]
    e.set_points(torch.from_numpy(np.ascontiguousarray(X)), torch.zeros(N, dtype=torch.float64),
                 dtypes=(_dt(dtype),), n_vars=X.shape[1])
    e.set_programs(progs)
    out = []
    for i, p in enumerate(progs):
        v0, none = e.predict([i], np.zeros((1, p.k)), dtype=_dt(dtype))
        assert none is None
        vk, g = e.predict([i] * (p.k - 1), np.zeros((p.k - 1, p.k)), cov=_cross(p.k), dtype=_dt(dtype))
        vk = vk.cpu().numpy()
        assert all(np.array_equal(vk[0], vk[j], equal_nan=True) for j in range(p.k - 1))
        out.append((v0.cpu().numpy()[0], vk[0], g.cpu().numpy().T))
    return out


def _unary(name):
    n = int(name[4:]) if name.startswith("powi") else 0
    if n:
        return "VSR_POWI", n, R.powi_grid, (lambda x: mp.power(x, n)), (lambda x: n * mp.power(x, n - 1)), \
            (lambda v, dtype: np.power(v, dtype(n))), lambda L: R.powi_budget(n)
    op, f, d, npf, budget = R.UNARY[name]
    return op, 0, (lambda dtype: R.unary_grid(name, dtype)), f, d, (lambda v, dtype: npf(v)), budget


@pytest.mark.parametrize("dtype", DTYPES, ids=_ids)
@pytest.mark.parametrize("name", sorted(R.UNARY) + [f"powi{n}" for n in R.POWI_N])
def test_unary_value_and_tangent_at_the_edges(eng, name, dtype):
    opname, n, grid, fval, fder, npf, budget = _unary(name)
    xs = grid(dtype)
    with np.errstate(all="ignore"):
        want_np = npf(xs, dtype)
    bv, bt = budget(R.LIB[BUILD][dtype])
    ins_a, imms, k = R.unary_program(opname, n)
    ins_b, _, _ = R.unary_program(opname, n, tail=False)
    [(v0, vk, g)] = _device(eng, [_program(ins_a, imms, k)], xs.reshape(-1, 1), dtype)
    eng.set_programs([_program(ins_b, imms, 1)])
    _, gabs2 = eng.predict([0], np.zeros((1, 1)), cov=np.ones((1, 1, 1)), dtype=_dt(dtype))
    gabs2 = gabs2.cpu().numpy()[0]
    for i, x in enumerate(xs):
        what = f"{name}({float(x)!r}) {_ids(dtype)} device"
        ref = R.exact(fval, x) if not math.isnan(x) else None
        assert (math.isnan(v0[i]) and math.isnan(vk[i])) or v0[i] == vk[i], f"{what}: K=0 {v0[i]!r} K=2 {vk[i]!r}"
        R.check_value(v0[i], float(want_np[i]), ref, bv, dtype, what)
        if not math.isfinite(want_np[i]):
            continue
        if name == "sqrt" and x == 0:
            assert math.isnan(g[i, 0]) and gabs2[i] == np.inf, what    # 0.5 / +-0
            continue
        dref = R.exact(fder, x)
        if math.isnan(g[i, 0]):
            # an infinite tangent turns the cross form nan: |g_0| must be infinite, as exactly
            assert R.classify(dref, dtype) == "inf" and gabs2[i] == np.inf, (what, dref, gabs2[i])
            continue
        R.check_point(-g[i, 0], dref, bt, dtype, "d/dc " + what)


@pytest.mark.parametrize("dtype", DTYPES, ids=_ids)
def test_pow_both_roles_special_cases_and_overflow_edge(eng, dtype):
    AB = R.pow_table(dtype)
    with np.errstate(all="ignore"):
        want_np = np.power(AB[:, 0], AB[:, 1])
    lib = R.LIB[BUILD][dtype]
    specs = R.pow_programs()
    res = _device(eng, [_program(ins, np.zeros(1), k) for _, ins, k, _ in specs], AB, dtype)
    for (name, _, k, roles), (v0, vk, g) in zip(specs, res):
        for i, (a, b) in enumerate(AB):
            what = f"{name} {float(a)!r}**{float(b)!r} {_ids(dtype)} device"
            if not (math.isfinite(a) and math.isfinite(b)):
                ref = None if math.isnan(want_np[i]) else mp.mpf(float(want_np[i]))
            else:
                ref = R.exact(mp.power, a, b)
            blna = abs(float(b) * math.log(float(a))) if 0 < a < np.inf and math.isfinite(b) else 0.0
            R.check_value(v0[i], float(want_np[i]), ref, lib["pow"], dtype, "K=0 " + what)
            R.check_value(vk[i], float(want_np[i]), ref, R.pow_dual_budget(lib, blna, dtype), dtype, "K>0 " + what)
            assert math.isnan(v0[i]) == math.isnan(vk[i]) and math.isfinite(v0[i]) == math.isfinite(vk[i]), what
            if not math.isfinite(v0[i]):
                assert v0[i] == vk[i] or math.isnan(v0[i]), what
            ex = R.pow_exact(a, b)
            if ex is None or not math.isfinite(want_np[i]) or R.classify(ex[0], dtype) != "normal":
                continue
            bt = R.pow_dual_budget(lib, blna, dtype)
            refs = [ex[1] if role == "a" else ex[2] for role in roles]
            for j, role in enumerate(roles):
                if math.isnan(g[i, j]):
                    assert any(R.classify(r, dtype) == "inf" for r in refs), (what, g[i])
                    continue
                R.check_point(-g[i, j], refs[j], bt + (1 if role == "a" else 2 * lib["log"] + 1), dtype,
                              f"d/d{role} " + what)


def _sweep_grid(name, dtype):
    """The unary grid's points with a finite value whose terms cannot overflow the fp64 sums."""
    opname, n, grid, fval, fder, npf, budget = _unary(name)
    xs = grid(dtype)
    with np.errstate(all="ignore"):
        xs = xs[np.isfinite(npf(xs, dtype))]
    cap = np.finfo(np.float64).max / (8 * xs.shape[0])
    pts, v_ref, g_ref = [], [], []
    for x in xs:
        f, d = R.exact(fval, x), R.exact(fder, x)
        r = f - mp.mpf(0.25)
        if r * r > cap or (d is not None and R.classify(d, dtype) == "normal" and abs(2 * r * d) > cap):
            continue
        pts.append(x)
        v_ref.append(f)
        g_ref.append([None if d is None else -d, mp.mpf(1)])
    return opname, n, np.array(pts, dtype=dtype), v_ref, g_ref, budget(R.LIB[BUILD][dtype])


@pytest.mark.parametrize("dtype", DTYPES, ids=_ids)
@pytest.mark.parametrize("tiled", [False, True], ids=["per_pair", "tile"])
def test_vsr_eval_drops_non_finite_terms(monkeypatch, tiled, dtype):
    """vsr_eval on each edge grid: loss = mean r^2, grad = mean 2 r g over the exact f and g with the
    non-finite terms dropped; eval_kernel, and eval_tile_kernel (forced for 8 pairs at any N)."""
    monkeypatch.setenv("VSR_TILE_MIN_POINTS", "1" if tiled else "1000000000")
    e = fitter.Engine("cuda:0")
    try:
        for name in ["tanh", "asin", "acos", "sqrt", "log", "exp", "atan", "inv", "sinh", "cosh", "tan", "powi-7"]:
            opname, n, xs, v_ref, g_ref, (bv, bt) = _sweep_grid(name, dtype)
            y = np.full(xs.shape[0], 0.25, dtype=dtype)
            want_l, bnd_l, want_g, bnd_g = R.sweep_bounds(v_ref, g_ref, y, bv, bt, dtype)
            ins, imms, k = R.unary_program(opname, n)
            e.set_points(torch.from_numpy(xs.reshape(-1, 1)), torch.from_numpy(y), dtypes=(_dt(dtype),), n_vars=1)
            e.set_programs([_program(ins, imms, k)])
            n0 = e.launches
            loss, grad = e.eval([0] * 8, np.zeros((8, k)), dtype=_dt(dtype), grad=True)
            assert e.launches > n0
            loss, grad = loss.cpu().numpy(), grad.cpu().numpy()
            assert (loss == loss[0]).all() and (grad == grad[0]).all(), name
            assert abs(mp.mpf(float(loss[0])) - want_l) <= bnd_l, (name, loss[0], want_l, bnd_l)
            for j in range(k):
                assert abs(mp.mpf(float(grad[0, j])) - want_g[j]) <= bnd_g[j], (name, j, grad[0, j], want_g[j])
    finally:
        e.close()


@pytest.mark.parametrize("dtype", DTYPES, ids=_ids)
def test_coverage_programs_upload_and_match_the_exact_isa(eng, dtype):
    """The hand-assembled coverage programs pass upload validation and give the exact ISA's values
    and, for the programs within the 16 tangent slots, |g|^2 through cov = I."""
    X = _coverage_points(dtype)
    eps = float(np.finfo(dtype).eps)
    cov = _coverage_programs()
    progs = [_program(ins, imms, k) for ins, imms, k in cov]
    eng.set_points(torch.from_numpy(X), torch.zeros(X.shape[0], dtype=torch.float64), dtypes=(_dt(dtype),), n_vars=4)
    eng.set_programs(progs)
    n = len(progs)
    consts = np.tile(np.array(COV_C, dtype=dtype).astype(np.float64), (n, 1))
    eye = np.broadcast_to(np.eye(COV_K + 1), (n, COV_K + 1, COV_K + 1)).copy()
    value, var = eng.predict(np.arange(n), consts, cov=eye, dtype=_dt(dtype))
    value, var = value.cpu().numpy(), var.cpu().numpy()
    for pi, (ins, imms, k) in enumerate(cov):
        for i in range(X.shape[0]):
            rv, rd = R.mp_run(ins, imms, consts[pi, :k], X[i], COV_K)
            scale = max([abs(rv)] + [abs(d) for d in rd])
            assert abs(mp.mpf(float(value[pi, i])) - rv) <= 64 * eps * scale, (pi, i, isa.disassemble(ins))
            if k > COV_K:
                assert math.isnan(var[pi, i])
            else:
                want = sum(d * d for d in rd)
                assert abs(mp.mpf(float(var[pi, i])) - want) <= 256 * eps * scale * scale, (pi, i, isa.disassemble(ins))
