"""Subprocess body of tests/test_overlay.py (TEST INFRASTRUCTURE).

    python _overlay_driver.py <tree root> <patched: 0|1> <repo root> <out json>

Imports ``scripts/visymre_utils.py`` of the given tree (the reference, or the reference with
vision-sr_b200 laid over it) exactly as the drivers do, then runs the tree's own ``Model.fitfunc2``
on a SCRIPTED decoder: the network parts (``MultiModalEncoder``, ``decoder_transfomer``, ``fc_out``
...) are replaced by stand-ins that steer the reference's unmodified beam loop towards two known
skeletons, so everything from line 292 of model.py down to the returned dict is the tree's code.
In the patched tree the numeric fit inside ``refine_hypotheses`` is served by the CPU oracle
(the test needs no GPU); the reference tree runs its own process-pool BFGS.
"""
import json
import os
import sys
import types

tree, patched, repo, out_path = sys.argv[1], sys.argv[2] == "1", sys.argv[3], sys.argv[4]
sys.path.insert(0, repo)
from oracle import ref_harness  # noqa: E402

ref_harness._install_stubs()
sys.path.insert(0, os.path.join(tree, "scripts"))
sys.path.insert(0, tree)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import visymre_utils as vu  # noqa: E402  (scripts/visymre_utils.py: the module every driver imports)

Model = vu.Model                                   # visymre_utils.py:15
assert vu.BFGSParams and vu.FitParams              # visymre_utils.py:16
import inspect  # noqa: E402

src = inspect.getsource(Model.fitfunc2)
info = {"has_refine_call": "refine_hypotheses(" in src, "has_process_pool": "ProcessPoolExecutor(" in src}

import pickle  # noqa: E402

raw = open(os.path.join(tree, "scripts/weights/meta/metadata.h5"), "rb").read()   # overlay.install copies it
td = pickle.loads(raw[2048:2048 + 2926])
w = td.word2id
n_words = max(w.values()) + 1
SCRIPTS = [["add", "c", "mul", "c", "x_1"], ["mul", "c", "x_1"]]


class Scripted(types.SimpleNamespace):
    """What fitfunc2 touches on ``self`` (model.py:292-442)."""


def next_logits(prefix):
    """log-probabilities of the next token after ``prefix`` (ids, leading S)."""
    lo = torch.full((n_words,), -30.0)
    words = [td.id2word[i] for i in prefix[1:]]
    if not words:                                      # first step: open both scripts
        lo[w[SCRIPTS[0][0]]] = -0.1
        lo[w[SCRIPTS[1][0]]] = -2.5
        return lo
    for sc in SCRIPTS:
        if words == sc[:len(words)]:
            lo[w[sc[len(words)]] if len(words) < len(sc) else w["F"]] = -0.05
            return lo
    lo[w["x_2"]] = -5.0                                # off-script beams wander with a low score
    return lo


me = Scripted()
me.cfg = types.SimpleNamespace(dim_input=11, length_eq=9)
me.trg_pad_idx = w["P"]
me.ieee_tran = lambda t: t
me.MultiModalEncoder = types.SimpleNamespace(predict=lambda enc_in: torch.zeros(1, 4, 8))
me.make_trg_mask = lambda g: (torch.zeros_like(g, dtype=torch.bool), torch.zeros(g.shape[1], g.shape[1]))
me.pos_embedding = lambda pos: torch.zeros(pos.shape + (1,))
me.tok_embedding = lambda g: g.unsqueeze(-1).float()
me.decoder_transfomer = lambda trg, mem, mask, tgt_key_padding_mask=None: trg       # [len, beam, 1]: the ids
me.fc_out = lambda ids: torch.stack([torch.stack([next_logits([int(t) for t in ids[:, b, 0].tolist()])
                                                  for b in range(ids.shape[1])])] * ids.shape[0])
me._analyze_prefix_tree_context = types.MethodType(Model._analyze_prefix_tree_context, me)

rng = np.random.RandomState(11)
X = torch.tensor(rng.uniform(-2, 2, (40, 1)))
y = 0.5 + 1.5 * X[:, 0]
cfg = types.SimpleNamespace(beam_size=2, device="cpu", no_c_in_pow=False,
                            bfgs=types.SimpleNamespace(activated=True, n_restarts=2, add_coefficients_if_not_existing=False,
                                                       normalization_o=False, idx_remove=False, normalization_type="MSE",
                                                       stop_time=1e9))
np.random.seed(5)
if patched:
    # the GPU fit is not available here: serve refine_hypotheses' batch call from the CPU oracle,
    # every candidate from the RNG state a forked pool worker of the reference would start from
    import src.visymre.architectures.refine as refine
    from oracle import vectorised

    def oracle_batch(pred_strs, X_, y_, cfg_, td_, x0=None, engine=None, lazy_strings=False):
        outs = []
        for toks in pred_strs:
            np.random.seed(5)
            try:
                outs.append(vectorised.bfgs(toks, X_, y_, cfg_, td_))
            except Exception as exc:  # noqa: BLE001
                outs.append(exc)
        return outs
    refine.bfgs_batch = oracle_batch
    info["refine_module"] = refine.__file__
torch.manual_seed(0)
out = Model.fitfunc2(me, X, y, cfg_params=cfg, test_data=td)
info["dict_keys"] = sorted(out.keys())
info["best"] = [None if p is None else str(p) for p in out["best_bfgs_preds"]]
info["best_loss"] = [float(v) for v in out["best_bfgs_loss"]]
info["all_preds"] = sorted(str(p) for p in out["all_bfgs_preds"])
info["all_loss"] = sorted(float(v) for v in out["all_bfgs_loss"])
info["best_token"] = [None if t is None else [int(v) for v in t] for t in out["best_token"]]
info["eq"] = [None if p is None else str(p) for p in me.eq]
json.dump(info, open(out_path, "w"))
print("ok", info["best"], info["best_loss"])
