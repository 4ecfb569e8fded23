"""Reference Gauss-Newton statistics for the uncertainty tests: a g++ build of the interpreter with a
serial loop over the points (``native/gram_twin.cpp``, ``twin_gram``) and the exact Jacobian from
``sympy.diff``, lambdified with the reference's modules."""
import ctypes
import json
import os
import subprocess
import tempfile

import numpy as np
import sympy as sp

from conftest import GOLDEN
from oracle import vectorised
from src.visymre.engine import isa

VARS = [f"x_{i}" for i in range(1, 11)]
_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(os.path.dirname(_HERE), "vision-sr_b200", "csrc")
_TWIN = None


def load_twin():
    """ctypes handle on ``native/gram_twin.cpp``, compiled once per process into a temporary
    directory (the tree is left as it is)."""
    global _TWIN
    if _TWIN is None:
        out = os.path.join(tempfile.mkdtemp(prefix="gram_twin_"), "libgram_twin.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-I" + _CSRC,
                               "-o", out, os.path.join(_HERE, "native", "gram_twin.cpp")])
        _TWIN = ctypes.CDLL(out)
    return _TWIN


def twin_gram(twin, prog, X, y, c):
    """(rss, jtj [k, k]) of ``prog`` at constants ``c`` over X [N, 10] / y [N] (fp64 or fp32)."""
    N = X.shape[0]
    Xc = np.ascontiguousarray(X.T)
    yc = np.ascontiguousarray(y, dtype=X.dtype)
    cc = np.ascontiguousarray(np.asarray(c, dtype=np.float64).reshape(-1))
    if cc.size == 0:
        cc = np.zeros(1)
    rss = ctypes.c_double()
    jtj = np.zeros((max(prog.k, 1), max(prog.k, 1)))
    rc = twin.gram_twin(
        prog.insns.ctypes.data_as(ctypes.c_void_p), prog.imms.ctypes.data_as(ctypes.c_void_p),
        cc.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(prog.k),
        Xc.ctypes.data_as(ctypes.c_void_p), yc.ctypes.data_as(ctypes.c_void_p), ctypes.c_long(N),
        ctypes.c_int(isa.DTYPE["VSR_F64"] if X.dtype == np.float64 else isa.DTYPE["VSR_F32"]),
        ctypes.byref(rss), jtj.ctypes.data_as(ctypes.c_void_p))
    assert rc == 0
    return rss.value, jtj[:prog.k, :prog.k]


def exact(skeleton, k, X, y, c):
    """(residuals r [N], Jacobian J [N, k]) from sympy: f and every d f / d c_j lambdified with the
    reference's modules, evaluated in fp64."""
    cs = [sp.Symbol(f"c{i}", real=True) for i in range(k)]
    xs = [sp.Symbol(v, real=True) for v in VARS]
    e = sp.sympify(skeleton, locals={str(s): s for s in cs + xs})
    cols = [X[:, j].astype(np.float64) for j in range(len(VARS))]
    N = X.shape[0]
    # sympy differentiates Abs of a power of x through re / im: real arguments here
    modules = [{"re": np.real, "im": np.imag}, vectorised.MODULES, "numpy"]

    def real(v):  # a value that is not real is nan, as on the device
        v = np.asarray(v)
        if np.iscomplexobj(v):
            v = np.where(v.imag == 0, v.real, np.nan)
        return np.broadcast_to(v.astype(np.float64), (N,))
    with np.errstate(all="ignore"):
        f = sp.lambdify(cs + xs, e, modules=modules)
        r = real(f(*c, *cols)) - y.astype(np.float64)
        J = np.zeros((N, k))
        for j in range(k):
            J[:, j] = real(sp.lambdify(cs + xs, sp.diff(e, cs[j]), modules=modules)(*c, *cols))
    return r, J


def winners():
    """Winning constants of the 17 golden cases (ref_bfgs.json) and the 40 config-1 candidates
    (ref_low.json): ``(name, skeleton, consts, X [N, 10] fp64, y [N] fp64)``."""
    out = []
    g = json.load(open(os.path.join(GOLDEN, "ref_bfgs.json")))
    for case in g["cases"]:
        if case.get("raised") or case.get("skeleton") is None:
            continue
        Xr = np.asarray(case["X"], dtype=np.float64).reshape(case["n"], -1)
        X = np.zeros((case["n"], 10))
        X[:, :Xr.shape[1]] = Xr
        out.append((case["name"], case["skeleton"], np.asarray(case["best_consts"], dtype=np.float64), X,
                    np.asarray(case["y"], dtype=np.float64).reshape(-1)))
    low = json.load(open(os.path.join(GOLDEN, "ref_low.json")))
    pts = np.load(os.path.join(GOLDEN, low["points"]))
    for case in low["cases"]:
        if case.get("raised") or case.get("skeleton") is None or not isinstance(case.get("best_consts"), list):
            continue
        if any(not isinstance(v, (int, float)) for v in case["best_consts"]):
            continue
        X = np.zeros((low["n_points"], 10))
        X[:, :2] = pts[case["row"] + "/X"]
        out.append((f"{case['row']}/{case['cand']}", case["skeleton"], np.asarray(case["best_consts"], dtype=np.float64),
                    X, np.asarray(pts[case["row"] + "/y"], dtype=np.float64)))
    return out


def frob_rel(a, b):
    nb = np.linalg.norm(b)
    return np.linalg.norm(a - b) / (nb if nb > 0 else 1.0)


def curve_fit_pcov(J, rss):
    """scipy.optimize.curve_fit's pcov (absolute_sigma=False) from the Jacobian: its own formula,
    on the SVD of J (scipy/optimize/_minpack_py.py)."""
    _, s, VT = np.linalg.svd(J, full_matrices=False)
    threshold = np.finfo(float).eps * max(J.shape) * s[0]
    s = s[s > threshold]
    VT = VT[:s.size]
    pcov = np.dot(VT.T / s ** 2, VT)
    return pcov * (rss / (J.shape[0] - J.shape[1]))
