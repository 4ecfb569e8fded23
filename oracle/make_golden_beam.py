"""Generate tests/golden/ref_beam_mask.json from the UNMODIFIED reference (SURVEY 8f row 1).

Two things are recorded for seeded random beams of prefix sequences:
  * what ``Model._analyze_prefix_tree_context`` (model.py:522-560) returns for every beam, called as
    the plain function it is (it never touches ``self``);
  * the ``-inf`` mask of the "# --- Constraint Logic ---" block of ``Model.fitfunc2``
    (model.py:382-411).  The block is inline in a 230-line method, so its statements are read from
    the reference file AT GENERATION TIME (between its own two marker comments), dedented and
    executed unchanged with the names the method has in scope at that point.

Run with VISYMRE_REFERENCE naming a reference checkout:  python oracle/make_golden_beam.py
TEST INFRASTRUCTURE: nothing under vision-sr_b200/ imports this.
"""
import json
import os
import sys
import textwrap
from types import SimpleNamespace as NS

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_harness  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "ref_beam_mask.json")


def constraint_block():
    src = open(os.path.join(ref_harness.REF_ROOT, "src/visymre/architectures/model.py")).read().split("\n")
    a = next(i for i, l in enumerate(src) if "# --- Constraint Logic ---" in l)
    b = next(i for i, l in enumerate(src) if i > a and l.strip().startswith("# ------------------------"))
    return compile(textwrap.dedent("\n".join(src[a:b])), "reference model.py:%d-%d" % (a + 1, b), "exec"), (a + 1, b)


def main():
    _, ref_model, td = ref_harness.load()
    assert ref_model is not None, "the reference model module did not import"
    analyze = ref_model.Model._analyze_prefix_tree_context
    block, lines = constraint_block()
    w = td.word2id
    n_words = max(w.values()) + 1
    a1 = {w[k] for k in ("abs", "asin", "cos", "exp", "ln", "sin", "sqrt", "tan")}
    a2 = {w[k] for k in ("add", "div", "mul", "pow", "sub")}
    leaves = [w[f"x_{j}"] for j in range(1, 4)] + [w["c"], w["2"], w["pi"], w["-1"]]
    pool = sorted(a1) + sorted(a2) * 2 + leaves * 3 + [w["F"]]
    cases = []
    settings = [
        dict(name="as_shipped", trans=[], no_c_in_pow=False, masked=["x_4", "x_5", "x_6", "x_7", "x_8", "x_9", "x_10"]),
        dict(name="no_c_in_pow", trans=[], no_c_in_pow=True, masked=["x_3", "x_10"]),
        dict(name="nested_transcendentals", trans=["cos", "exp", "ln", "sin", "tan"], no_c_in_pow=True, masked=[]),
    ]
    for si, st in enumerate(settings):
        for cur_len in (1, 2, 3, 5, 9, 17, 33, 58, 61):
            rng = np.random.RandomState(1000 * si + cur_len)
            beam, length_eq = 40, 62
            gen = np.full((beam, length_eq), w["P"], dtype=np.int64)
            gen[:, 0] = w["S"]
            gen[:, 1:] = rng.choice(pool, size=(beam, length_eq - 1))
            gen[5, 0] = w["add"]                                   # a beam that does not start with S
            gen[6, 1:4] = [w["pow"], w["x_1"], w["x_2"]]           # pow: the exponent slot
            gen[7, 1:3] = [w["pow"], w["x_1"]]
            gen[8, 1:3] = [w["sin"], w["add"]]
            gen[9, 1:6] = [w["add"], w["x_1"], w["mul"], w["c"], w["x_2"]]   # complete tree
            scores = rng.normal(size=beam).astype(np.float32)
            scores[[3, 11]] = -1e9                                 # dead beams (model.py:387)
            trans_ids = {w[k] for k in st["trans"]}
            c_id = w.get("c", 3) if st["no_c_in_pow"] else None
            masked = {w[k] for k in st["masked"]}
            ctx = []
            for i in range(beam):
                v, f = analyze(None, gen[i, :cur_len].tolist(), a1, a2, trans_ids, w["pow"], c_id, w["S"])
                ctx.append([int(v), sorted(int(x) for x in f)])
            env = dict(torch=torch, scores=torch.zeros(beam, n_words), cfg_params=NS(beam_size=beam),
                       beam_scores=torch.tensor(scores), generated=torch.tensor(gen),
                       cur_len=torch.tensor(cur_len, dtype=torch.int64),
                       self=NS(cfg=NS(length_eq=length_eq),
                               _analyze_prefix_tree_context=lambda *a: analyze(None, *a)),
                       arity_1_ids=a1, arity_2_ids=a2, transcendental_ids=trans_ids, pow_id=w["pow"], c_id=c_id,
                       start_id=w["S"], all_op_ids=a1 | a2, finish_id=w["F"], pad_id=w["P"],
                       masked_var_ids=masked, n_words=n_words)
            exec(block, env)
            mask = env["logit_mask"].numpy()
            assert set(np.unique(mask)) <= {0.0, -np.inf}
            bits = [int(sum(1 << j for j in range(n_words) if mask[i, j] == -np.inf)) for i in range(beam)]
            cases.append(dict(setting=st["name"], cur_len=cur_len, length_eq=length_eq, beam=beam,
                              transcendental=sorted(trans_ids), c_id=c_id, masked_vars=sorted(masked),
                              generated=gen[:, :max(cur_len, 1)].tolist(), beam_scores=[float(s) for s in scores],
                              context=ctx, mask_bits=bits))
    out = dict(generator="oracle/make_golden_beam.py", reference="aidalee123/Vision-SR (unmodified)",
               block_lines=list(lines), n_words=n_words, word2id={k: int(v) for k, v in w.items()},
               arity_1=sorted(a1), arity_2=sorted(a2), cases=cases)
    with open(OUT, "w") as fh:
        json.dump(out, fh)
    print("wrote", OUT, os.path.getsize(OUT), "bytes,", len(cases), "cases; block = model.py:%d-%d" % lines)


if __name__ == "__main__":
    main()
