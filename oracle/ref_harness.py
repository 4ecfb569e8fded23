"""Import the UNMODIFIED reference hot path (TEST INFRASTRUCTURE, generation only).

A checkout of the reference (aidalee123/Vision-SR), named by the environment variable
``VISYMRE_REFERENCE``, is needed to regenerate the golden vectors under ``tests/golden/``; the tests
read those vectors, except ``tests/test_overlay.py``, which skips without the checkout.  The reference's
``src/visymre/architectures/bfgs.py`` imports cleanly once the packages that are
absent here -- none of which ``bfgs()`` touches -- are replaced by inert stubs
(SURVEY.md section 8c).  Run it in a process that does NOT have ``vision-sr_b200`` on
``sys.path``: both trees use the top-level package name ``src``.
"""
import importlib
import os
import pickle
import sys
import types

# a checkout of aidalee123/Vision-SR; unset: only oracle/_ref (oracle/build_ref.py) can serve the reference
REF_ROOT = os.environ.get("VISYMRE_REFERENCE", "")
_STUBS = ("numexpr", "hydra", "pytorch_lightning", "func_timeout", "h5py", "omegaconf")


class _Inert:
    """Stands in for anything an absent package would export: callable, usable as a
    decorator (with or without arguments), subclassable, attribute access never fails."""

    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        if len(a) == 1 and callable(a[0]) and not k:
            return a[0]          # bare decorator
        return _Inert()

    def __getattr__(self, name):
        return _Inert()


class _StubModule(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        if name and name[0].isupper():      # class-like: must be subclassable
            return type(name, (Exception,) if "Timed" in name or "Error" in name else (object,), {})
        return _Inert()


def _install_stubs():
    for name in _STUBS:
        try:
            importlib.import_module(name)
            continue
        except ImportError:
            pass
        sys.modules[name] = _StubModule(name)


VENDORED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")   # oracle/build_ref.py


def available():
    """Where the unmodified reference can be imported from: its checkout (VISYMRE_REFERENCE) or the
    byte-compiled copy oracle/build_ref.py made; None when neither is here."""
    if REF_ROOT and os.path.isdir(os.path.join(REF_ROOT, "src", "visymre")):
        return REF_ROOT
    tag = os.path.join(VENDORED, "PYTHON")
    if os.path.exists(tag) and open(tag).read().strip() == f"{sys.version_info.major}.{sys.version_info.minor}":
        return VENDORED
    return None


class _ArchiveFinder:
    """Serves the reference's modules from oracle/_ref/modules.bin (see oracle/build_ref.py)."""

    def __init__(self, path):
        import pickle as _p
        with open(path, "rb") as fh:
            self.mods = _p.load(fh)

    def find_spec(self, name, path=None, target=None):
        if name not in self.mods:
            return None
        from importlib.machinery import ModuleSpec
        is_pkg = self.mods[name][0]
        spec = ModuleSpec(name, self, is_package=is_pkg, origin="oracle/_ref/modules.bin:" + name)
        return spec

    def create_module(self, spec):
        return None

    def exec_module(self, module):
        import marshal
        exec(marshal.loads(self.mods[module.__name__][1]), module.__dict__)   # noqa: S102


def load(ref_root=None):
    """Returns (bfgs_module, model_module_or_None, test_data)."""
    ref_root = ref_root or available()
    if ref_root is None:
        raise ImportError("neither VISYMRE_REFERENCE nor oracle/_ref (python oracle/build_ref.py) is here")
    _install_stubs()
    archive = os.path.join(ref_root, "modules.bin")
    if os.path.exists(archive):
        if not any(isinstance(f, _ArchiveFinder) for f in sys.meta_path):
            for name in [m for m in sys.modules if m == "src" or m.startswith("src.")]:
                del sys.modules[name]          # this process only ever runs the reference from here on
            sys.meta_path.insert(0, _ArchiveFinder(archive))
    elif ref_root not in sys.path:
        sys.path.insert(0, ref_root)
    ref_bfgs = importlib.import_module("src.visymre.architectures.bfgs")
    importlib.import_module("src.visymre.dclasses")
    vendored = os.path.join(ref_root, "metadata.pkl")
    if os.path.exists(vendored):
        test_data = pickle.loads(open(vendored, "rb").read())
    else:
        raw = open(f"{ref_root}/scripts/weights/meta/metadata.h5", "rb").read()
        test_data = pickle.loads(raw[2048:2048 + 2926])
    test_data.id2word[3] = "constant"  # what fitfunc2 does before fitting (model.py:452)
    try:
        ref_model = importlib.import_module("src.visymre.architectures.model")
    except Exception:  # torchvision / lightning details: the wrapper is 6 lines, optional
        ref_model = None
    return ref_bfgs, ref_model, test_data
