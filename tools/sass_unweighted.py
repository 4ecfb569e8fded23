#!/usr/bin/env python
"""Compare the SASS of the unweighted kernels of two builds (no GPU needed).

    python tools/sass_unweighted.py OLD_BUILD_DIR NEW_BUILD_DIR

Both directories hold the instantiation objects ``inst_<type>_<K>.o`` of ``vision-sr_b200/csrc/build``
(``make -C vision-sr_b200/csrc`` at two commits).  For every ``fit_kernel``, ``eval_kernel``,
``eval_tile_kernel``, ``gram_kernel`` and ``predict_kernel`` of the old build, the instructions of
``cuobjdump -sass`` are compared with those of the new build's ``W = false`` instantiation of the same
type, width and points per thread.  The function names are ignored (the new ones carry ``W`` and
``Weighted<...>`` in their mangling), so is the column padding of the listing, which cuobjdump sizes per
object.  Exits 1 if any kernel differs.
"""
import glob
import os
import re
import subprocess
import sys

KINDS = ("fit_kernel", "eval_kernel", "eval_tile_kernel", "gram_kernel", "predict_kernel")


def kernels(obj):
    """{(kind, template args without W): [instruction lines]} of the unweighted kernels of one object."""
    out = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    parts = re.split(r"\n\s*Function : (\S+)\n", out)
    res = {}
    for name, body in zip(parts[1::2], parts[2::2]):
        dem = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()
        m = re.match(r"void vsr::(\w+)<([^>]*?)(, (true|false))?>\(", dem)
        if not m or m.group(1) not in KINDS or m.group(4) == "true":
            continue
        body = body.split("\n\t\t..........")[0]
        res[(m.group(1), m.group(2))] = [" ".join(line.split()) for line in body.splitlines()]
    return res


def main():
    old_dir, new_dir = sys.argv[1], sys.argv[2]
    n = same = 0
    for obj in sorted(glob.glob(os.path.join(old_dir, "inst_*.o"))):
        old, new = kernels(obj), kernels(os.path.join(new_dir, os.path.basename(obj)))
        for key, body in sorted(old.items()):
            n += 1
            if new.get(key) == body:
                same += 1
            else:
                print("differs:", os.path.basename(obj), *key)
    print(f"{same}/{n} kernels identical")
    return 0 if n and same == n else 1


if __name__ == "__main__":
    sys.exit(main())
