#!/usr/bin/env python
"""Lay the B200 refinement path over a checkout of the reference (aidalee123/Vision-SR).

    python vision-sr_b200/overlay.py <reference checkout> [--out <copy to patch instead>]

What it does to ``<checkout>/src/visymre`` (nothing else is touched; with ``--out`` the checkout
is first copied there and the copy is patched):

  engine/                 added    compiler, native binding, fitter, sharding, host pool
  engine/_native/         added    libvsr.so + vsr_isa.h (the C ABI library, include/vsr.h)
  architectures/refine.py added    refine_hypotheses / bfgs_wrapper / beam_constraint_mask
  architectures/bfgs.py   REPLACED same ``bfgs(pred_str, X, y, cfg, test_data)`` signature and
                                   return (reference bfgs.py:42-215), fits on the GPU
  architectures/model.py  PATCHED  the "BFGS Parallel Part" of ``Model.fitfunc2``
                                   (reference model.py:444-520: 20 worker processes, one
                                   ``bfgs_wrapper`` task per candidate) becomes one call of
                                   ``refine_hypotheses``; the "Constraint Logic" block of the beam loop
                                   (model.py:382-411) gets a device branch (``beam_constraint_mask``,
                                   one launch per decode step) in front of its own host loop, which
                                   stays for CPU tensors; the network and the rest of the beam loop
                                   stay the reference's own code
  scoring.py, hlsc_batch.py added  driver-side scoring / batched HLSC evaluation (optional)
  uncertainty.py added            covariance / standard errors of fitted constants (optional)

The reference's drivers (``scripts/*_test.py`` through ``scripts/visymre_utils.py``) then run
unchanged: ``from src.visymre.architectures.model import Model`` still finds the reference's
``Model``, ``fitfunc = partial(model.fitfunc2, ...)`` now refines on the B200.
"""
import argparse
import os
import re
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(HERE, "src", "visymre")
MARK_BEGIN = "# ... (BFGS Parallel Part) ..."
PATCH = [
    "# --- refinement on the B200 (vision-sr_b200 overlay; replaces the process-pool BFGS part) ---",
    "from .refine import refine_hypotheses",
    "output = refine_hypotheses(generated_hyps.hyp, X, y, cfg_params, test_data)",
    "self.eq = output['best_bfgs_preds']",
    "return output",
]


def patch_model_source(text):
    """The reference's model.py with the BFGS part of fitfunc2 replaced.  Mechanical: from the
    marker comment the reference itself carries to the ``return output`` that ends the method."""
    lines = text.split("\n")
    try:
        a = next(i for i, l in enumerate(lines) if MARK_BEGIN in l)
    except StopIteration:
        raise ValueError("marker %r not found: not the reference's model.py (or already patched)" % MARK_BEGIN)
    b = next(i for i in range(a, len(lines)) if lines[i].strip() == "return output")
    indent = re.match(r"\s*", lines[a]).group(0)
    return "\n".join(lines[:a] + [indent + l for l in PATCH] + lines[b + 1:])


MASK_BEGIN = "# --- Constraint Logic ---"
MASK_END = "scores = scores + logit_mask"


def patch_constraint_block(text):
    """The "Constraint Logic" block of the beam loop (reference model.py:382-411: every beam copied to the
    host and walked in Python at every decode step) gets a device branch: one ``vsr_beam_mask`` launch
    when the beams live on the GPU.  The reference's own statements stay, unchanged, as the branch for
    CPU tensors.  Mechanical: from the block's marker comment to the line that applies the mask."""
    lines = text.split("\n")
    a = next((i for i, l in enumerate(lines) if MASK_BEGIN in l), None)
    if a is None:
        raise ValueError("marker %r not found" % MASK_BEGIN)
    b = next(i for i in range(a, len(lines)) if lines[i].strip() == MASK_END)
    ind = re.match(r"\s*", lines[a]).group(0)
    head = [
        ind + "# --- Constraint Logic --- (vision-sr_b200 overlay: one device launch when the beams are on the GPU)",
        ind + "if generated.is_cuda:",
        ind + "    from .refine import beam_constraint_mask",
        ind + "    logit_mask = beam_constraint_mask(",
        ind + "        generated, int(cur_len), beam_scores, n_words, arity_1_ids=arity_1_ids, arity_2_ids=arity_2_ids,",
        ind + "        transcendental_ids=transcendental_ids, all_op_ids=all_op_ids, masked_var_ids=masked_var_ids,",
        ind + "        pow_id=pow_id, c_id=c_id, start_id=start_id, finish_id=finish_id, pad_id=pad_id,",
        ind + "        length_eq=self.cfg.length_eq)",
        ind + "else:",
    ]
    body = ["    " + l if l.strip() else l for l in lines[a + 1:b]]
    return "\n".join(lines[:a] + head + body + lines[b:])


def install(checkout, out=None):
    src = os.path.join(checkout, "src", "visymre")
    if not os.path.isfile(os.path.join(src, "architectures", "model.py")):
        raise FileNotFoundError(f"{checkout} is not a checkout of the reference (src/visymre/architectures/model.py)")
    if out:
        shutil.copytree(checkout, out, dirs_exist_ok=True,
                        ignore=shutil.ignore_patterns("__pycache__", "*.ckpt", ".git"))
        src = os.path.join(out, "src", "visymre")
    # engine package + native library
    shutil.copytree(os.path.join(PKG, "engine"), os.path.join(src, "engine"), dirs_exist_ok=True,
                    ignore=shutil.ignore_patterns("__pycache__"))
    native = os.path.join(src, "engine", "_native")
    os.makedirs(native, exist_ok=True)
    shutil.copy(os.path.join(HERE, "csrc", "vsr_isa.h"), native)
    lib = os.path.join(HERE, "csrc", "libvsr.so")
    if os.path.exists(lib):
        shutil.copy(lib, native)
    # the refinement modules
    shutil.copy(os.path.join(PKG, "architectures", "refine.py"), os.path.join(src, "architectures", "refine.py"))
    shutil.copy(os.path.join(PKG, "architectures", "bfgs.py"), os.path.join(src, "architectures", "bfgs.py"))
    shutil.copy(os.path.join(PKG, "scoring.py"), os.path.join(src, "scoring.py"))
    shutil.copy(os.path.join(PKG, "hlsc.py"), os.path.join(src, "hlsc_batch.py"))
    shutil.copy(os.path.join(PKG, "uncertainty.py"), os.path.join(src, "uncertainty.py"))
    # Model.fitfunc2
    mp = os.path.join(src, "architectures", "model.py")
    with open(mp) as fh:
        patched = patch_constraint_block(patch_model_source(fh.read()))
    with open(mp, "w") as fh:
        fh.write(patched)
    return src


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("checkout")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    print("patched", install(a.checkout, a.out))
