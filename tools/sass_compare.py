#!/usr/bin/env python
"""Compare the SASS of every kernel of two builds (no GPU needed).

    python tools/sass_compare.py OLD_BUILD_DIR NEW_BUILD_DIR

Both directories hold the instantiation objects ``inst_*.o`` (``inst_<type>_<K>.o`` and the robust
``inst_rb_<type>_<K>.o``) of ``vision-sr_b200/csrc/build`` (``make -C vision-sr_b200/csrc`` at two commits).
Every ``fit_kernel``, ``eval_kernel``, ``eval_tile_kernel``, ``gram_kernel`` and ``predict_kernel`` of an old
object is compared with the kernel of the new object of the same name that has the same kind, type, width,
points per thread and loss mode.  The mode is read from each naming scheme the kernels have had: no mode
argument (linear), ``..., W>``, ``..., W, RB>`` and ``..., (vsr::LossMode)n>``.  Only the instruction text
is compared: the function names (whose mangling carries the argument struct) and the column padding of the
listing, which cuobjdump sizes per object, are ignored.  Exits 1 if any kernel of the old build differs or
has no match.
"""
import glob
import os
import re
import subprocess
import sys

KINDS = ("fit_kernel", "eval_kernel", "eval_tile_kernel", "gram_kernel", "predict_kernel")
MODES = ("linear", "weighted", "robust")  # vsr::LossMode 0, 1, 2


def kernel_key(demangled):
    """(kind, T, K, P, mode) of a demangled kernel name, or None for other functions."""
    m = re.match(r"void vsr::(\w+)<([^>]*)>\(", demangled)
    if not m or m.group(1) not in KINDS:
        return None
    kind, args = m.group(1), [a.strip() for a in m.group(2).split(",")]
    if kind == "gram_kernel":  # fp64 only: no type argument
        args.insert(0, "double")
    t, k, p, rest = args[0], int(args[1]), int(args[2]), args[3:]
    if not rest:
        mode = 0
    elif len(rest) == 1 and rest[0] in ("false", "true"):  # <..., W>
        mode = 1 if rest[0] == "true" else 0
    elif len(rest) == 2:  # <..., W, RB>
        mode = 2 if rest[1] == "true" else (1 if rest[0] == "true" else 0)
    else:
        mm = re.fullmatch(r"\(vsr::LossMode\)(\d+)", rest[0])
        if len(rest) != 1 or not mm:
            raise ValueError(f"unknown kernel naming scheme: {demangled}")
        mode = int(mm.group(1))
    return kind, t, k, p, MODES[mode]


def kernels(obj):
    """{(kind, T, K, P, mode): [instruction lines]} of the kernels of one object."""
    out = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    parts = re.split(r"\n\s*Function : (\S+)\n", out)
    res = {}
    for name, body in zip(parts[1::2], parts[2::2]):
        dem = subprocess.run(["c++filt", name], capture_output=True, text=True, check=True).stdout.strip()
        key = kernel_key(dem)
        if key is None:
            continue
        body = body.split("\n\t\t..........")[0]
        res[key] = [" ".join(line.split()) for line in body.splitlines()]
    return res


def main():
    if len(sys.argv) != 3:
        print(__doc__)
        return 2
    old_dir, new_dir = sys.argv[1], sys.argv[2]
    n = same = 0
    for obj in sorted(glob.glob(os.path.join(old_dir, "inst_*.o"))):
        new_obj = os.path.join(new_dir, os.path.basename(obj))
        old, new = kernels(obj), (kernels(new_obj) if os.path.exists(new_obj) else {})
        for key, body in sorted(old.items()):
            n += 1
            if new.get(key) == body:
                same += 1
            else:
                print("differs:" if key in new else "missing:", os.path.basename(obj), *key)
    print(f"{same}/{n} kernels identical")
    return 0 if n and same == n else 1


if __name__ == "__main__":
    sys.exit(main())
