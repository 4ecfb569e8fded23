"""Python view of the bytecode ISA.

The opcodes, operand sources and limits are parsed out of ``csrc/vsr_isa.h`` at
import time, so the C header stays the single definition the kernels, the host
simulator and this compiler share.
"""
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))


def _find_csrc():
    """Where libvsr.so and vsr_isa.h live: $VSR_CSRC, the repo's csrc/ (three levels up), or the
    ``_native`` directory ``overlay.py`` puts beside this file in a reference checkout."""
    for d in (os.environ.get("VSR_CSRC"), os.path.join(_HERE, "..", "..", "..", "csrc"), os.path.join(_HERE, "_native")):
        if d and os.path.exists(os.path.join(d, "vsr_isa.h")):
            return os.path.normpath(d)
    return os.path.normpath(os.path.join(_HERE, "..", "..", "..", "csrc"))


CSRC_DIR = _find_csrc()
ISA_HEADER = os.path.join(CSRC_DIR, "vsr_isa.h")


def _parse(path):
    text = open(path).read()
    text = re.sub(r"//[^\n]*", "", text)
    enums, defines = {}, {}
    for m in re.finditer(r"enum\s+(\w+)\s*\{([^}]*)\}", text):
        nxt, members = 0, {}
        for item in m.group(2).split(","):
            item = item.strip()
            if not item:
                continue
            if "=" in item:
                name, val = [s.strip() for s in item.split("=")]
                nxt = int(val, 0)
            else:
                name = item
            members[name] = nxt
            nxt += 1
        enums[m.group(1)] = members
    for m in re.finditer(r"#define\s+(VSR_MAX_\w+)\s+(\d+)", text):
        defines[m.group(1)] = int(m.group(2))
    return enums, defines


_ENUMS, _DEFINES = _parse(ISA_HEADER)
OP = _ENUMS["VsrOp"]
SRC = _ENUMS["VsrSrc"]
FIT_STATUS = _ENUMS["VsrFitStatus"]
GRAD_MODE = _ENUMS["VsrGradMode"]
DTYPE = _ENUMS["VsrDtype"]
LOSS = _ENUMS["VsrLoss"]
OP_NAME = {v: k for k, v in OP.items()}
SRC_NAME = {v: k for k, v in SRC.items()}

MAX_VARS = _DEFINES["VSR_MAX_VARS"]
MAX_DUAL = _DEFINES["VSR_MAX_DUAL"]
MAX_CONSTS = _DEFINES["VSR_MAX_CONSTS"]
MAX_STACK = _DEFINES["VSR_MAX_STACK"]
MAX_INSNS = _DEFINES["VSR_MAX_INSNS"]
MAX_IMMS = _DEFINES["VSR_MAX_IMMS"]

# tangent widths the kernels are instantiated for (must match vsr_kernels.cu)
DUAL_WIDTHS = (0, 1, 2, 3, 4, 5, 6, 7, 8, 12, 16)


def pick_dual_width(k):
    """Smallest instantiated tangent width >= k, or None (-> FD-gradient mode)."""
    for w in DUAL_WIDTHS:
        if w >= k:
            return w
    return None


def encode(op, src=0, idx=0, amask=0, bmask=0):
    return ((op & 0xFF) | ((src & 0xFF) << 8) | ((idx & 0xFFFF) << 16)
            | ((amask & 0xFFFF) << 32) | ((bmask & 0xFFFF) << 48))


def decode(word):
    word = int(word)
    return (word & 0xFF, (word >> 8) & 0xFF, (word >> 16) & 0xFFFF,
            (word >> 32) & 0xFFFF, (word >> 48) & 0xFFFF)


def disassemble(insns, imms=()):
    lines = []
    for w in insns:
        op, src, idx, am, bm = decode(w)
        name = OP_NAME[op][4:]
        if OP["VSR_LOAD"] <= op <= OP["VSR_RPOW"] and op != OP["VSR_PUSH"]:
            s = SRC_NAME[src][8:]
            arg = f"{s}" if src == SRC["VSR_SRC_STACK"] else f"{s}[{idx}]"
            if src == SRC["VSR_SRC_IMM"] and idx < len(imms):
                arg += f"={imms[idx]!r}"
            lines.append(f"{name:5s} {arg:22s} a={am:#06x} b={bm:#06x}")
        elif op == OP["VSR_POWI"]:
            n = idx - 0x10000 if idx & 0x8000 else idx
            lines.append(f"{name:5s} {n:<22d} a={am:#06x}")
        else:
            lines.append(f"{name:5s} {'':22s} a={am:#06x}")
    return "\n".join(lines)
