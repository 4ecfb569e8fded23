"""Recipe for oracle/_ref: the UNMODIFIED reference hot path, byte-compiled where it lies.

The reference is pure Python (no build system).  This script compiles the few modules its
``bfgs()`` needs -- straight from ``$VISYMRE_REFERENCE/src/visymre`` -- to code objects in ONE
archive ``oracle/_ref/modules.bin`` (no reference source text is copied into the repo) and extracts the pickled vocabulary record from ``scripts/weights/meta/metadata.h5`` (bytes
2048..4974, SURVEY 8c).  ``oracle/_ref/`` is git-ignored; copied along with the tree to a machine without the
checkout, it lets ``bench.py --impl reference --config 1`` time this
as-is reference (``cpu_baseline.kind = "reference"``) and ``oracle/ref_harness.load()`` finds it.

Run:  python oracle/build_ref.py      (``__graft_entry__.build()`` does, when VISYMRE_REFERENCE names a checkout)
TEST INFRASTRUCTURE: nothing under vision-sr_b200/ imports oracle/.
"""
import os
import shutil
import sys

REF = os.environ.get("VISYMRE_REFERENCE", "")
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")
# what `import src.visymre.architectures.bfgs` / `.model` pull in (SURVEY 2.1), nothing else
MODULES = [
    "src/__init__.py", "src/visymre/__init__.py", "src/visymre/dclasses.py", "src/visymre/utils.py",
    "src/visymre/architectures/__init__.py", "src/visymre/architectures/bfgs.py",
    "src/visymre/architectures/data.py", "src/visymre/architectures/model.py",
    "src/visymre/architectures/beam_search.py", "src/visymre/architectures/MultimodalEncoder.py",
    "src/visymre/dataset/__init__.py", "src/visymre/dataset/generator.py",
    "src/visymre/dataset/sympy_utils.py", "src/visymre/dataset/data_utils.py",
]


def build(ref=REF, out=OUT):
    """One archive, ``oracle/_ref/modules.bin``: {dotted module name: (is_package, marshalled code
    object)} of the reference's own modules, compiled from where they lie (``compile()`` +
    ``marshal``: what a ``.pyc`` holds, without the file names a snapshot tool may filter)."""
    import marshal
    import pickle
    if not ref or not os.path.isdir(ref):
        raise FileNotFoundError("oracle/_ref is built from a checkout of the reference: set VISYMRE_REFERENCE")
    if os.path.isdir(out):
        shutil.rmtree(out)
    os.makedirs(out)
    mods = {}
    for rel in MODULES:
        src = os.path.join(ref, rel)
        is_pkg = rel.endswith("__init__.py")
        name = rel[:-3].replace("/", ".")
        if is_pkg:
            name = name[: -len(".__init__")]
        if os.path.exists(src):
            with open(src, "rb") as fh:
                code = compile(fh.read(), src, "exec", dont_inherit=True)
        elif is_pkg:                                # namespace package in the reference: an empty module
            code = compile("", rel, "exec")
        else:
            continue
        mods[name] = (is_pkg, marshal.dumps(code))
    with open(os.path.join(out, "modules.bin"), "wb") as fh:
        pickle.dump(mods, fh)
    raw = open(os.path.join(ref, "scripts/weights/meta/metadata.h5"), "rb").read()
    with open(os.path.join(out, "metadata.pkl"), "wb") as fh:
        fh.write(raw[2048:2048 + 2926])
    with open(os.path.join(out, "PYTHON"), "w") as fh:
        fh.write(f"{sys.version_info.major}.{sys.version_info.minor}\n")   # code objects are per minor version
    return len(mods)


if __name__ == "__main__":
    print(f"oracle/_ref: {build()} modules byte-compiled from {REF}")
