#!/usr/bin/env python
"""Compare the SASS of every linear kernel of two builds (no GPU needed).

    python tools/sass_unchanged.py OLD_BUILD_DIR NEW_BUILD_DIR

Both directories hold the instantiation objects ``inst_<type>_<K>.o`` of ``vision-sr_b200/csrc/build``
(``make -C vision-sr_b200/csrc`` at two commits).  Every ``fit_kernel``, ``eval_kernel``,
``eval_tile_kernel``, ``gram_kernel`` and ``predict_kernel`` of the old build, weighted (``W = true``) or
not, is compared with the kernel of the new build that has the same template arguments and ``RB = false``
(the robust-loss kernels, ``RB = true``, live in the new build's ``inst_rb_*`` objects and have no
counterpart).  An old build without the ``RB`` argument is matched as well.  The function names are
ignored (their mangling carries the argument struct), so is the column padding of the listing, which
cuobjdump sizes per object.  Exits 1 if any kernel differs or is missing.
"""
import glob
import os
import re
import subprocess
import sys

KINDS = ("fit_kernel", "eval_kernel", "eval_tile_kernel", "gram_kernel", "predict_kernel")
RB_KINDS = ("fit_kernel", "eval_kernel", "eval_tile_kernel", "gram_kernel")
# template arguments without RB: <T, K, P, W> (gram: <K, P, W>)
N_ARGS = {"fit_kernel": 4, "eval_kernel": 4, "eval_tile_kernel": 4, "gram_kernel": 3}


def kernels(obj):
    """{(kind, template args without RB): [instruction lines]} of the linear kernels of one object."""
    out = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    parts = re.split(r"\n\s*Function : (\S+)\n", out)
    res = {}
    for name, body in zip(parts[1::2], parts[2::2]):
        dem = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()
        m = re.match(r"void vsr::(\w+)<([^>]*?)>\(", dem)
        if not m or m.group(1) not in KINDS:
            continue
        kind, args = m.group(1), [a.strip() for a in m.group(2).split(",")]
        if kind in RB_KINDS and len(args) == N_ARGS[kind] + 1:
            if args.pop() == "true":
                continue
        body = body.split("\n\t\t..........")[0]
        res[(kind, ", ".join(args))] = [" ".join(line.split()) for line in body.splitlines()]
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
