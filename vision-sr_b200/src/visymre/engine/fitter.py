"""Host side of the refinement engine: device memory, uploads and batched calls.

``Engine`` owns one ``vsr_handle`` (``include/vsr.h``) on one CUDA device.  torch is
used for device memory and streams only; every number is produced by libvsr.so.
"""
import ctypes
from dataclasses import dataclass

import numpy as np
import torch

from . import isa, native
from .compiler import Program

F64, F32 = isa.DTYPE["VSR_F64"], isa.DTYPE["VSR_F32"]
_TORCH_DTYPE = {F64: torch.float64, F32: torch.float32}


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _np_ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


@dataclass
class FitResult:
    """Per-run outputs of ``Engine.fit`` (device tensors, rows = slots)."""
    consts: torch.Tensor     # [n_slots, kstride] res.x
    lastx: torch.Tensor      # [n_slots, kstride] last point the objective saw (bfgs.py:116)
    loss: torch.Tensor       # [n_slots] objective at consts
    final_mse: torch.Tensor  # [n_slots] plain MSE at lastx in the score dtype
    info: torch.Tensor       # [n_slots, 4] int32: status, nit, nfev, 0


def weights_from_sigma(sigma, n, dtypes):
    """Per-point weights ``w = 1 / sigma**2`` (fp64 tensor on sigma's device) of a 1-D ``sigma`` of length
    ``n``, as ``scipy.optimize.curve_fit`` takes it.  Raises ``ValueError`` when ``sigma`` has the wrong
    shape, holds a value that is not finite or not > 0, or when ``w`` is not a finite normal number in
    every point dtype of ``dtypes`` (an fp32 slot can overflow or underflow)."""
    s = torch.as_tensor(sigma, dtype=torch.float64)
    if s.dim() != 1 or int(s.shape[0]) != int(n):
        raise ValueError(f"sigma must be 1-D with {n} entries, got shape {tuple(s.shape)}")
    if not bool((torch.isfinite(s) & (s > 0)).all()):
        raise ValueError("every sigma must be finite and > 0")
    w = 1.0 / (s * s)
    _check_weights(w, dtypes)
    return w


def _check_weights(w, dtypes):
    for dt in dtypes:
        td = _TORCH_DTYPE[dt]
        wd = w.to(td)
        if not bool((torch.isfinite(wd) & (wd >= torch.finfo(td).tiny)).all()):
            raise ValueError(f"a weight 1/sigma^2 is not a finite normal {td} number at every point")


def default_opts(**over):
    lib = native.load()
    o = native.FitOpts()
    lib.vsr_fit_opts_default(ctypes.byref(o))
    for key, val in over.items():
        if not hasattr(o, key):
            raise AttributeError(f"vsr_fit_opts has no field {key!r}")
        setattr(o, key, val)
    return o


class Engine:
    def __init__(self, device=None):
        self.lib = native.load()
        if not torch.cuda.is_available():
            raise native.VsrError("no CUDA device: the refinement engine has no CPU fallback")
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise native.VsrError(f"device {self.device} is not a CUDA device (no CPU fallback)")
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", index)
        self._h = ctypes.c_void_p()
        rc = self.lib.vsr_create(index, ctypes.byref(self._h))
        if rc != 0:
            raise native.VsrError(f"vsr_create failed ({rc}): {self.lib.vsr_last_error(None).decode()}")
        self._points = {}      # dtype -> (Xc [d, ld], y [N]) tensors kept alive
        self._weights = {}     # dtype -> w [N] tensor kept alive (weighted points only)
        self._src = None       # (X2d, y1d) as given, for re-uploads with more columns
        self._w_src = None     # fp64 weights as given (None: unweighted)
        self.n_points = 0
        self.n_vars = 0
        self.programs = []
        self.kmax = 0

    # ---- lifetime ------------------------------------------------------------------
    def close(self):
        if self._h:
            self.lib.vsr_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        native.check(self.lib, self._h, rc)

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def launches(self):
        return int(self.lib.vsr_launch_count(self._h))

    def set_profiling(self, on):
        self._check(self.lib.vsr_set_profiling(self._h, int(bool(on))))

    def set_geometry(self, spec=None):
        """Measurement hook: "cluster:threads:seats[:optimiser warps]" overrides the launch geometry
        of ``fit`` (0 or a missing item keeps the built-in choice); None or "" restores it."""
        v = [int(x) for x in str(spec).split(":")] if spec else []
        v = (v + [0, 0, 0, 0])[:4]
        self._check(self.lib.vsr_set_geometry(self._h, *v))

    def set_phase_buffer(self, tensor):
        """int64 device tensor [n_slots, 8] (or None) for per-run phase cycle counts."""
        self._phase = tensor
        self._check(self.lib.vsr_set_phase_buffer(self._h, _ptr(tensor)))

    def read_profile(self):
        """(fit_ms, fit_launches, score_ms, score_launches) since the last read."""
        out = (ctypes.c_double * 4)()
        self._check(self.lib.vsr_read_profile(self._h, out))
        return tuple(out)

    # ---- points ----------------------------------------------------------------------
    def set_points(self, X, y, dtypes=(F64,), n_vars=None, w=None):
        """X: [N, d] (or [1, N, d]) tensor/array on any device; y: squeezable to [N].

        Columns are stored column-major on the device, one copy per requested dtype.
        Trailing all-zero columns are not stored unless a program reads them.
        ``w``: optional per-point weights [N] (``vsr_set_weights``), stored in every dtype slot; the fit,
        ``eval`` and ``gram`` then use ``sum w r^2``.  ``ValueError`` when a weight is not a finite normal
        number > 0 in a requested dtype.
        """
        X = torch.as_tensor(X)
        y = torch.as_tensor(y)
        if X.dim() == 3:
            X = X[0]
        y = y.reshape(-1)
        if X.dim() != 2 or X.shape[0] != y.shape[0] or X.shape[0] == 0:
            raise ValueError(f"points: X {tuple(X.shape)} / y {tuple(y.shape)}")
        if X.shape[1] > isa.MAX_VARS:
            X = X[:, :isa.MAX_VARS]
        X = X.to(self.device, non_blocking=True)
        y = y.to(self.device, non_blocking=True)
        if w is not None:
            w = torch.as_tensor(w, dtype=torch.float64).reshape(-1)
            if int(w.shape[0]) != int(X.shape[0]):
                raise ValueError(f"{int(w.shape[0])} weights for {int(X.shape[0])} points")
            w = w.to(self.device, non_blocking=True)
            _check_weights(w, dtypes)
        self._src = (X, y)
        self._w_src = w
        self.n_points = int(X.shape[0])
        if n_vars is None:
            nz = (X != 0).any(dim=0).nonzero()
            n_vars = int(nz.max().item()) + 1 if nz.numel() else 1
        self._want_dtypes = tuple(dtypes)
        self._upload_columns(max(1, min(int(n_vars), X.shape[1])))

    def _upload_columns(self, n_vars):
        X, y = self._src
        N = self.n_points
        ld = (N + 3) & ~3  # 16-byte aligned columns in either precision
        self._points = {}
        for dt in self._want_dtypes:
            td = _TORCH_DTYPE[dt]
            Xc = torch.zeros((n_vars, ld), dtype=td, device=self.device)
            Xc[:, :N] = X[:, :n_vars].t().to(td)
            yc = y.to(td).contiguous()
            self._check(self.lib.vsr_set_points(self._h, _ptr(Xc), _ptr(yc), N, ld, n_vars, dt))
            self._points[dt] = (Xc, yc)
        self._weights = {}
        if self._w_src is not None:
            for dt in self._want_dtypes:
                self._weights[dt] = self._w_src.to(_TORCH_DTYPE[dt]).contiguous()
                self._check(self.lib.vsr_set_weights(self._h, _ptr(self._weights[dt]), N, dt))
        self.n_vars = n_vars

    def adopt_points(self, other):
        """Use the points another engine of the same device holds (no copy: the same device tensors
        are registered with this handle): engines that fit parts of one beam concurrently."""
        self._src = other._src
        self._w_src = other._w_src
        self.n_points = other.n_points
        self.n_vars = other.n_vars
        self._want_dtypes = tuple(other._want_dtypes)
        self._points = dict(other._points)
        self._weights = dict(other._weights)
        for dt, (Xc, yc) in self._points.items():
            self._check(self.lib.vsr_set_points(self._h, _ptr(Xc), _ptr(yc), self.n_points, int(Xc.shape[1]),
                                                self.n_vars, dt))
            if dt in self._weights:
                self._check(self.lib.vsr_set_weights(self._h, _ptr(self._weights[dt]), self.n_points, dt))

    def ensure_dtype(self, dt):
        if dt not in self._points:
            if self._w_src is not None:
                _check_weights(self._w_src, (dt,))
            self._want_dtypes = tuple(self._want_dtypes) + (dt,)
            self._upload_columns(self.n_vars)

    # ---- programs --------------------------------------------------------------------
    def set_programs(self, programs):
        if not programs:
            raise ValueError("no programs")
        for p in programs:
            if not isinstance(p, Program):
                raise TypeError("set_programs expects compiled Program objects")
        insn_off = np.zeros(len(programs) + 1, dtype=np.int32)
        imm_off = np.zeros(len(programs) + 1, dtype=np.int32)
        for i, p in enumerate(programs):
            insn_off[i + 1] = insn_off[i] + p.insns.shape[0]
            imm_off[i + 1] = imm_off[i] + p.imms.shape[0]
        insns = np.ascontiguousarray(np.concatenate([p.insns for p in programs]).astype(np.uint64))
        imms = np.ascontiguousarray(np.concatenate([p.imms for p in programs]).astype(np.float64))
        ks = np.asarray([p.k for p in programs], dtype=np.int32)
        need_vars = max([p.var_mask.bit_length() for p in programs] + [1])
        if self._src is not None and need_vars > self.n_vars:
            if need_vars > self._src[0].shape[1]:
                raise ValueError(f"a program reads x_{need_vars} but X has {self._src[0].shape[1]} columns")
            self._upload_columns(need_vars)
        self._check(self.lib.vsr_upload_programs(self._h, _np_ptr(insns), _np_ptr(insn_off),
                                                 _np_ptr(imms), _np_ptr(imm_off), _np_ptr(ks),
                                                 len(programs), self._stream()))
        self.programs = list(programs)
        self.kmax = int(ks.max())

    # ---- batched evaluation ----------------------------------------------------------
    def eval(self, prog_idx, consts, dtype=F64, grad=False, const_row=None):
        """loss (and gradient) of pairs (program prog_idx[p], constants consts[row[p]]).

        Returns device tensors ``loss [n]`` and ``grad [n, kstride]`` (or None).
        """
        self.ensure_dtype(dtype)
        prog_idx = np.ascontiguousarray(np.asarray(prog_idx, dtype=np.int32))
        n = int(prog_idx.shape[0])
        consts = torch.as_tensor(consts, dtype=torch.float64, device=self.device)
        if consts.dim() == 1:
            consts = consts.reshape(n, -1) if consts.numel() else consts.reshape(n, 0)
        if consts.shape[1] == 0:
            consts = torch.zeros((consts.shape[0], 1), dtype=torch.float64, device=self.device)
        consts = consts.contiguous()
        kstride = int(consts.shape[1])
        rows = None
        if const_row is not None:
            rows = np.ascontiguousarray(np.asarray(const_row, dtype=np.int32))
        loss = torch.empty(n, dtype=torch.float64, device=self.device)
        g = torch.zeros((n, kstride), dtype=torch.float64, device=self.device) if grad else None
        self._check(self.lib.vsr_eval(self._h, _np_ptr(prog_idx),
                                      _np_ptr(rows) if rows is not None else ctypes.c_void_p(0),
                                      n, _ptr(consts), kstride, dtype, _ptr(loss), _ptr(g),
                                      self._stream()))
        return loss, g

    def gram(self, prog_idx, consts, const_row=None):
        """Gauss-Newton statistics (``vsr_gram``, fp64 points) of pairs (program prog_idx[p],
        constants consts[row[p]]).

        Returns device tensors ``rss [n]`` (sum of squared residuals) and ``jtj [n, kstride, kstride]``
        (J^T J over the program's k constants; entries past k stay nan, and so do all k x k entries of
        a program with more than ``isa.MAX_DUAL`` constants).
        """
        self.ensure_dtype(F64)
        prog_idx = np.ascontiguousarray(np.asarray(prog_idx, dtype=np.int32))
        n = int(prog_idx.shape[0])
        consts = torch.as_tensor(consts, dtype=torch.float64, device=self.device)
        if consts.dim() == 1:
            consts = consts.reshape(n, -1) if consts.numel() else consts.reshape(n, 0)
        if consts.shape[1] == 0:
            consts = torch.zeros((consts.shape[0], 1), dtype=torch.float64, device=self.device)
        consts = consts.contiguous()
        kstride = int(consts.shape[1])
        rows = None
        if const_row is not None:
            rows = np.ascontiguousarray(np.asarray(const_row, dtype=np.int32))
        rss = torch.empty(n, dtype=torch.float64, device=self.device)
        jtj = torch.full((n, kstride, kstride), float("nan"), dtype=torch.float64, device=self.device)
        self._check(self.lib.vsr_gram(self._h, _np_ptr(prog_idx),
                                      _np_ptr(rows) if rows is not None else ctypes.c_void_p(0),
                                      n, _ptr(consts), kstride, _ptr(rss), _ptr(jtj), self._stream()))
        return rss, jtj

    def predict(self, prog_idx, consts, cov=None, dtype=F64, const_row=None):
        """Per-point values (``vsr_predict``) of pairs (program prog_idx[p], constants consts[row[p]])
        over the points of ``dtype``, and with ``cov`` ([rows, k, k] f64, read for a, b < k of each
        program) the delta-method variance ``g^T cov[row[p]] g`` of every point, g = d f / d c.

        Returns device f64 tensors ``value [n, N]`` (nan / inf where numpy gives them) and ``var [n, N]``
        (None without ``cov``; 0 for programs without constants, nan for programs with more than
        ``isa.MAX_DUAL`` constants).
        """
        self.ensure_dtype(dtype)
        prog_idx = np.ascontiguousarray(np.asarray(prog_idx, dtype=np.int32))
        n = int(prog_idx.shape[0])
        consts = torch.as_tensor(consts, dtype=torch.float64, device=self.device)
        if consts.dim() == 1:
            consts = consts.reshape(n, -1) if consts.numel() else consts.reshape(n, 0)
        if consts.shape[1] == 0:
            consts = torch.zeros((consts.shape[0], 1), dtype=torch.float64, device=self.device)
        consts = consts.contiguous()
        kstride = int(consts.shape[1])
        n_rows = int(consts.shape[0])
        if cov is not None:
            cov = torch.as_tensor(cov, dtype=torch.float64, device=self.device)
            kc = int(cov.shape[-1]) if cov.dim() == 3 else -1
            # a pair reads row const_row[p] of consts and of cov alike
            if kc < 0 or kc > kstride or tuple(cov.shape) != (n_rows, kc, kc):
                raise ValueError(f"cov {tuple(cov.shape)} does not match consts {tuple(consts.shape)}")
            if kc < kstride:
                cov = torch.nn.functional.pad(cov, (0, kstride - kc, 0, kstride - kc))
            cov = cov.contiguous()
        rows = None
        if const_row is not None:
            rows = np.ascontiguousarray(np.asarray(const_row, dtype=np.int32))
            if rows.shape != (n,) or (n and (rows.min() < 0 or rows.max() >= n_rows)):
                raise ValueError(f"const_row must hold {n} rows in [0, {n_rows})")
        elif n_rows < n:
            raise ValueError(f"{n} pairs but {n_rows} rows of constants")
        N = self.n_points
        value = torch.empty((n, N), dtype=torch.float64, device=self.device)
        var = torch.empty((n, N), dtype=torch.float64, device=self.device) if cov is not None else None
        self._check(self.lib.vsr_predict(self._h, _np_ptr(prog_idx),
                                         _np_ptr(rows) if rows is not None else ctypes.c_void_p(0),
                                         n, _ptr(consts), kstride, _ptr(cov), dtype, _ptr(value), _ptr(var),
                                         N, self._stream()))
        return value, var

    def score(self, prog_idx, consts=None, dtype=F64, const_row=None):
        """Driver-side scoring (``vsr_score``): mean squared error of every pair with the
        prediction passed through numpy's ``nan_to_num`` first.  Returns a device tensor [n]."""
        self.ensure_dtype(dtype)
        prog_idx = np.ascontiguousarray(np.asarray(prog_idx, dtype=np.int32))
        n = int(prog_idx.shape[0])
        if consts is None:
            consts = torch.zeros((n, 1), dtype=torch.float64, device=self.device)
        consts = torch.as_tensor(consts, dtype=torch.float64, device=self.device)
        if consts.dim() == 1:
            consts = consts.reshape(n, -1)
        consts = consts.contiguous()
        rows = None
        if const_row is not None:
            rows = np.ascontiguousarray(np.asarray(const_row, dtype=np.int32))
        out = torch.empty(n, dtype=torch.float64, device=self.device)
        self._check(self.lib.vsr_score(self._h, _np_ptr(prog_idx),
                                       _np_ptr(rows) if rows is not None else ctypes.c_void_p(0),
                                       n, _ptr(consts), int(consts.shape[1]), dtype, _ptr(out),
                                       self._stream()))
        return out

    # ---- fitting ---------------------------------------------------------------------
    def fit(self, run_prog, run_slot, x0, opts=None, n_slots=None):
        """Multi-restart BFGS; ``x0`` is a device (or host) [n_slots, kstride] f64 tensor."""
        opts = opts if opts is not None else default_opts()
        self.ensure_dtype(opts.eval_dtype)
        self.ensure_dtype(opts.score_dtype)
        run_prog = np.ascontiguousarray(np.asarray(run_prog, dtype=np.int32))
        run_slot = np.ascontiguousarray(np.asarray(run_slot, dtype=np.int32))
        x0 = torch.as_tensor(x0, dtype=torch.float64).to(self.device).contiguous()
        if x0.dim() != 2:
            raise ValueError("x0 must be [n_slots, kstride]")
        n_slots = int(x0.shape[0]) if n_slots is None else n_slots
        kstride = int(x0.shape[1])
        nan = float("nan")
        res = FitResult(
            consts=torch.full((n_slots, kstride), nan, dtype=torch.float64, device=self.device),
            lastx=torch.full((n_slots, kstride), nan, dtype=torch.float64, device=self.device),
            loss=torch.full((n_slots,), nan, dtype=torch.float64, device=self.device),
            final_mse=torch.full((n_slots,), nan, dtype=torch.float64, device=self.device),
            info=torch.full((n_slots, 4), -1, dtype=torch.int32, device=self.device))
        self._check(self.lib.vsr_fit(self._h, _np_ptr(run_prog), _np_ptr(run_slot),
                                     int(run_prog.shape[0]), _ptr(x0), kstride,
                                     ctypes.byref(opts), _ptr(res.consts), _ptr(res.lastx),
                                     _ptr(res.loss), _ptr(res.final_mse), _ptr(res.info),
                                     self._stream()))
        return res

    def fit_host(self, run_prog, run_slot, x0, opts=None):
        """The same fit through ``vsr_fit_host``: numpy in, numpy out, synchronous."""
        opts = opts if opts is not None else default_opts()
        self.ensure_dtype(opts.eval_dtype)
        self.ensure_dtype(opts.score_dtype)
        run_prog = np.ascontiguousarray(np.asarray(run_prog, dtype=np.int32))
        run_slot = np.ascontiguousarray(np.asarray(run_slot, dtype=np.int32))
        x0 = np.ascontiguousarray(np.asarray(x0, dtype=np.float64))
        n_slots, kstride = x0.shape
        out = dict(consts=np.empty((n_slots, kstride)), lastx=np.empty((n_slots, kstride)),
                   loss=np.empty(n_slots), final_mse=np.empty(n_slots),
                   info=np.empty((n_slots, 4), dtype=np.int32))
        self._check(self.lib.vsr_fit_host(self._h, _np_ptr(run_prog), _np_ptr(run_slot),
                                          int(run_prog.shape[0]), n_slots, _np_ptr(x0), kstride,
                                          ctypes.byref(opts), _np_ptr(out["consts"]),
                                          _np_ptr(out["lastx"]), _np_ptr(out["loss"]),
                                          _np_ptr(out["final_mse"]), _np_ptr(out["info"]),
                                          self._stream()))
        return out


_ENGINES = {}


def get_engine(device=None):
    """Process-wide engine per CUDA device (created on first use)."""
    dev = torch.device(device if device is not None else "cuda")
    index = dev.index if dev.index is not None else (torch.cuda.current_device() if torch.cuda.is_available() else 0)
    if index not in _ENGINES:
        _ENGINES[index] = Engine(torch.device("cuda", index))
    return _ENGINES[index]


_SIDE = {}
_SIDE_STREAMS = {}


def get_side_engine(main, i):
    """i-th helper engine beside ``main`` (same device): fits another part of the same beam."""
    key = (id(main), i)
    if key not in _SIDE:
        _SIDE[key] = Engine(main.device)
        # first use of a stream costs: torch's allocator keeps a pool of blocks per stream and fills it
        # with cudaMalloc calls (which wait for the device).  Touch both pools of the side stream now.
        with torch.cuda.stream(side_stream(main.device, i)):
            for n in (1 << 10, 4 << 20):
                torch.empty(n, dtype=torch.uint8, device=main.device).zero_()
        torch.cuda.current_stream(main.device).wait_stream(side_stream(main.device, i))
    return _SIDE[key]


def side_stream(device, i):
    dev = torch.device(device)
    key = (dev.index, i)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=dev)
    return _SIDE_STREAMS[key]


def device_engines(devices, home=None):
    """One engine per entry of ``devices`` (CUDA devices, the first one the home device).  The first
    entry of a device gets that device's process-wide engine (``get_engine``; ``home`` for the first
    entry when given), every further entry of the same device another engine beside it
    (``get_side_engine``, the j-th repeat on side stream j), so that one GPU can hold several parts of
    a beam."""
    engines, first = [], {}
    for i, d in enumerate(devices):
        d = torch.device(d)
        with torch.cuda.device(d):          # creating a handle makes its device current: not the caller's
            if d not in first:
                first[d] = home if (i == 0 and home is not None) else get_engine(d)
                engines.append(first[d])
            else:
                engines.append(get_side_engine(first[d], sum(1 for e in engines if e.device == d)))
    return engines


def share_points(engines):
    """Give every engine the points (and weights) ``engines[0]`` holds (``set_points`` was called on it).  Each other
    device gets one copy, made from the home device's tensors: a peer copy on the home stream that torch
    orders before the device's own stream.  Further engines of a device adopt that device's copy."""
    home = engines[0]
    X, y = home._src
    holder = {home.device: home}
    for eng in engines[1:]:
        if eng.device in holder:
            eng.adopt_points(holder[eng.device])
            continue
        with torch.cuda.device(eng.device):
            eng.set_points(X, y, dtypes=home._want_dtypes, n_vars=home.n_vars, w=home._w_src)
        holder[eng.device] = eng
