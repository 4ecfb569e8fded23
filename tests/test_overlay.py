"""The drop-in at the level the reference's drivers use it (SURVEY 8b): ``vision-sr_b200/overlay.py`` lays
the package over a copy of the reference checkout, ``scripts/visymre_utils.py`` imports as the
drivers import it, and the checkout's own ``Model.fitfunc2`` -- beam loop and all -- ends in
``refine_hypotheses``.  Its output dict is compared with the UNPATCHED reference run on the same
scripted decoder.  Needs a checkout of the reference, named by VISYMRE_REFERENCE (oracle/ref_harness.py);
skips without one."""
import json
import os
import subprocess
import sys

import pytest

from conftest import PKG, ROOT
from oracle.ref_harness import REF_ROOT as REF

pytestmark = pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "src", "visymre")),
                                reason="needs a checkout of the reference: set VISYMRE_REFERENCE")


def _run(tree, patched, out):
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "_overlay_driver.py"), tree, "1" if patched else "0",
                        ROOT, out], capture_output=True, text=True, timeout=900, cwd=os.path.dirname(out), env=env)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    return json.load(open(out))


def test_overlay_patches_fitfunc2_and_the_drivers_module_imports(tmp_path):
    sys.path.insert(0, PKG)
    import overlay
    tree = str(tmp_path / "checkout")
    overlay.install(REF, out=tree)
    for rel in ("src/visymre/engine/native.py", "src/visymre/engine/_native/vsr_isa.h",
                "src/visymre/architectures/refine.py", "src/visymre/utils.py", "scripts/visymre_utils.py"):
        assert os.path.exists(os.path.join(tree, rel)), rel
    text = open(os.path.join(tree, "src/visymre/architectures/model.py")).read()
    assert "refine_hypotheses(generated_hyps.hyp, X, y, cfg_params, test_data)" in text
    assert "class Model(pl.LightningModule)" in text and "ProcessPoolExecutor(20)" not in text
    with pytest.raises(ValueError):
        overlay.patch_model_source(text)          # a second application finds no marker
    # the constraint block: a device branch in front of the reference's own (re-indented) statements
    assert "if generated.is_cuda:" in text and "beam_constraint_mask(" in text
    assert "hyp_seq = generated[i, :cur_len].cpu().tolist()" in text
    compile(text, "patched model.py", "exec")

    got = _run(tree, True, str(tmp_path / "patched.json"))
    ref = _run(REF, False, str(tmp_path / "reference.json"))
    assert got["has_refine_call"] and not got["has_process_pool"]
    assert ref["has_process_pool"] and not ref["has_refine_call"]
    assert got["refine_module"].startswith(tree)
    assert got["dict_keys"] == ref["dict_keys"] == sorted(
        ["pred_target", "all_bfgs_preds", "all_bfgs_loss", "best_bfgs_preds", "best_bfgs_loss", "best_token"])
    # the same candidates reach the fit, the same one wins, with the same loss (same basin)
    assert len(got["all_loss"]) == len(ref["all_loss"]) >= 2
    assert got["best_token"] == ref["best_token"]
    for a, b in zip(got["all_loss"], ref["all_loss"]):
        assert abs(a - b) <= 1e-6 * max(1.0, abs(b)) + 1e-9, (got["all_loss"], ref["all_loss"])
    assert abs(got["best_loss"][0] - ref["best_loss"][0]) <= 1e-9
    assert got["eq"] == got["best"]
