"""ctypes binding of libvsr.so (the C ABI in ``include/vsr.h``).

The library is built in-tree from ``vision-sr_b200/csrc`` (``make -C csrc`` or
``__graft_entry__.build()``).  Importing this module never needs a GPU; creating an
``Engine`` does, and raises ``VsrError`` when the library or the device is missing --
there is no CPU fallback.
"""
import ctypes
import os
import subprocess

# vsr_fit launches one kernel per tangent width on its own stream.  With CUDA's default of 8
# hardware queues the streams of back-to-back fits alias and every fit runs ~10 % slower when
# the next one is already enqueued (tools/exp_valueloop.py); 32 queues remove that.  Only
# effective if set before the CUDA context exists, harmless otherwise.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

from . import isa

# VSR_LIB: A/B measurement hook (another build of the same ABI)
LIB_PATH = os.environ.get("VSR_LIB") or os.path.join(isa.CSRC_DIR, "libvsr.so")

c_i32p = ctypes.POINTER(ctypes.c_int32)
c_f64p = ctypes.POINTER(ctypes.c_double)
c_u64p = ctypes.POINTER(ctypes.c_uint64)
vp = ctypes.c_void_p


class VsrError(RuntimeError):
    pass


class FitOpts(ctypes.Structure):
    _fields_ = [("gtol", ctypes.c_double), ("c1", ctypes.c_double), ("c2", ctypes.c_double),
                ("xrtol", ctypes.c_double), ("fd_eps", ctypes.c_double),
                ("penalty", ctypes.c_double), ("loss_scale", ctypes.c_double),
                ("stop_time", ctypes.c_double), ("maxiter_per_k", ctypes.c_int32),
                ("grad_mode", ctypes.c_int32), ("eval_dtype", ctypes.c_int32),
                ("score_dtype", ctypes.c_int32), ("warps_per_run", ctypes.c_int32),
                ("reserved", ctypes.c_int32)]


class BeamRules(ctypes.Structure):
    _fields_ = [("arity1", ctypes.c_uint64), ("arity2", ctypes.c_uint64),
                ("transcendental", ctypes.c_uint64), ("all_ops", ctypes.c_uint64),
                ("masked_vars", ctypes.c_uint64), ("pow_id", ctypes.c_int32),
                ("c_id", ctypes.c_int32), ("start_id", ctypes.c_int32),
                ("finish_id", ctypes.c_int32), ("pad_id", ctypes.c_int32),
                ("length_eq", ctypes.c_int32)]


# name -> (restype, argtypes); mirrors include/vsr.h one to one
SIGNATURES = {
    "vsr_abi_version": (ctypes.c_int, []),
    "vsr_fit_opts_default": (None, [ctypes.POINTER(FitOpts)]),
    "vsr_create": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(vp)]),
    "vsr_destroy": (None, [vp]),
    "vsr_last_error": (ctypes.c_char_p, [vp]),
    "vsr_set_points": (ctypes.c_int, [vp, vp, vp, ctypes.c_int64, ctypes.c_int64,
                                      ctypes.c_int32, ctypes.c_int32]),
    "vsr_upload_points": (ctypes.c_int, [vp, vp, vp, ctypes.c_int64, ctypes.c_int64,
                                         ctypes.c_int32, ctypes.c_int32, vp]),
    "vsr_set_weights": (ctypes.c_int, [vp, vp, ctypes.c_int64, ctypes.c_int32]),
    "vsr_upload_programs": (ctypes.c_int, [vp, vp, vp, vp, vp, vp, ctypes.c_int32, vp]),
    "vsr_eval": (ctypes.c_int, [vp, vp, vp, ctypes.c_int32, vp, ctypes.c_int32, ctypes.c_int32,
                                vp, vp, vp]),
    "vsr_score": (ctypes.c_int, [vp, vp, vp, ctypes.c_int32, vp, ctypes.c_int32, ctypes.c_int32,
                                 vp, vp]),
    "vsr_gram": (ctypes.c_int, [vp, vp, vp, ctypes.c_int32, vp, ctypes.c_int32, vp, vp, vp]),
    "vsr_predict": (ctypes.c_int, [vp, vp, vp, ctypes.c_int32, vp, ctypes.c_int32, vp, ctypes.c_int32,
                                   vp, vp, ctypes.c_int64, vp]),
    "vsr_fit": (ctypes.c_int, [vp, vp, vp, ctypes.c_int32, vp, ctypes.c_int32,
                               ctypes.POINTER(FitOpts), vp, vp, vp, vp, vp, vp]),
    "vsr_fit_host": (ctypes.c_int, [vp, vp, vp, ctypes.c_int32, ctypes.c_int32, vp,
                                    ctypes.c_int32, ctypes.POINTER(FitOpts), vp, vp, vp, vp, vp,
                                    vp]),
    "vsr_beam_mask": (ctypes.c_int, [vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, vp,
                                     ctypes.POINTER(BeamRules), ctypes.c_int32, vp, vp]),
    "vsr_beam_mask_step": (ctypes.c_int, [vp, vp, vp, vp, vp, ctypes.c_int32, vp, ctypes.c_int32, vp,
                                          ctypes.POINTER(BeamRules), ctypes.c_int32, vp, vp]),
    "vsr_launch_count": (ctypes.c_int64, [vp]),
    "vsr_set_profiling": (ctypes.c_int, [vp, ctypes.c_int32]),
    "vsr_read_profile": (ctypes.c_int, [vp, c_f64p]),
    "vsr_set_phase_buffer": (ctypes.c_int, [vp, vp]),
    "vsr_set_geometry": (ctypes.c_int, [vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32]),
}

_lib = None


def build(force=False, verbose=False):
    """Compile libvsr.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    if force and os.path.exists(LIB_PATH):
        os.remove(LIB_PATH)
    cmd = ["make", "-j", str(os.cpu_count() or 4), "-C", isa.CSRC_DIR, "libvsr.so"]
    out = subprocess.run(cmd, capture_output=True, text=True)
    if verbose:
        print(out.stdout, out.stderr)
    if out.returncode != 0:
        raise VsrError(f"building libvsr.so failed:\n{out.stdout}\n{out.stderr}")
    return LIB_PATH


def load():
    """dlopen libvsr.so and attach the prototypes of include/vsr.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VsrError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; "
                       f"g.build()'` (there is no CPU fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError = ABI drift, fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.vsr_abi_version() != 1:
        raise VsrError("libvsr.so ABI version mismatch")
    _lib = lib
    return lib


def check(lib, handle, rc):
    if rc != 0:
        msg = lib.vsr_last_error(handle)
        raise VsrError(f"libvsr error {rc}: {msg.decode() if msg else '?'}")
