"""The refinement half of ``Model.fitfunc2`` on the B200.

Reference ``src/visymre/architectures/model.py``: ``bfgs_wrapper`` :13-19, the "BFGS
Parallel Part" of ``fitfunc2`` :444-520 and ``_analyze_prefix_tree_context`` :522-560.
The reference fans one ``bfgs_wrapper`` task per beam candidate out to a
``ProcessPoolExecutor(20)`` and pickles (X, y) into every task; here all candidates and
all their restarts go to the GPU as one batch (``bfgs.bfgs_batch``).  The encoder /
decoder forward and the beam loop above line 444 stay the reference's PyTorch code
(out of scope, SURVEY.md section 2.1).

This module has a name the reference does not use, so that it can be laid OVER a reference
checkout next to the reference's own ``model.py`` (``vision-sr_b200/overlay.py`` does that and
patches ``Model.fitfunc2`` to call ``refine_hypotheses``; see INTEGRATION.md).  In this
repo's own package ``architectures/model.py`` re-exports it under the reference's names.
"""
import numpy as np
import torch

from ..engine import fitter
from .bfgs import LazyStrings, bfgs, bfgs_batch, resolve_devices, sigma_weights

UNARY_NAMES = ("abs", "asin", "cos", "exp", "ln", "sin", "sqrt", "tan")   # model.py:295
BINARY_NAMES = ("add", "div", "mul", "pow", "sub")                        # model.py:296


def bfgs_wrapper(args):
    """model.py:13-19 -- one candidate; any exception drops it as (None, nan, tokens)."""
    ww, X_cpu, y_cpu, cfg_params, test_data = args
    try:
        pred_w_c, constants, loss_bfgs, exa = bfgs(ww, X_cpu, y_cpu, cfg_params, test_data)
        return (str(pred_w_c), loss_bfgs, ww)
    except Exception:  # noqa: BLE001
        return (None, float("nan"), ww)


def analyze_prefix_tree_context(seq, arity_1_ids, arity_2_ids, transcendental_ids, pow_id, c_id,
                                start_id=1):
    """model.py:522-560 -- open slots of a prefix sequence and the tokens forbidden next.

    Returns ``(valency, forbidden)``: valency 0 means the tree is complete.
    """
    frames = [[None, 1, frozenset()]]  # [operator, children still missing, constraints]
    tokens = seq[1:] if len(seq) > 0 and seq[0] == start_id else seq
    for tok in tokens:
        if not frames:
            break
        top = frames[-1]
        top[1] -= 1
        inherited = set(top[2])
        if c_id is not None and top[0] == pow_id and top[1] == 0:
            inherited.add(c_id)  # the exponent slot of a pow
        for_children = set(inherited)
        if tok in transcendental_ids:
            for_children |= set(transcendental_ids)
        if pow_id is not None and tok == pow_id:
            for_children.add(pow_id)
        if tok in arity_2_ids:
            frames.append([tok, 2, frozenset(for_children)])
        elif tok in arity_1_ids:
            frames.append([tok, 1, frozenset(for_children)])
        while frames and frames[-1][1] == 0:
            frames.pop()
    valency = sum(f[1] for f in frames)
    forbidden = set(frames[-1][2]) if frames else set()
    if c_id is not None and frames and frames[-1][0] == pow_id and frames[-1][1] == 1:
        forbidden.add(c_id)
    return valency, forbidden


def _as_list(ww):
    if isinstance(ww, torch.Tensor):
        return ww.cpu().tolist()
    if isinstance(ww, np.ndarray):
        return ww.tolist()
    return list(ww)


def refine_hypotheses(hyps, X, y, cfg_params, test_data, x0=None, engine=None, sigma=None, loss="linear",
                      f_scale=1.0):
    """The "BFGS Parallel Part" of fitfunc2 (model.py:444-520).

    ``hyps``: ``generated_hyps.hyp``, a list of ``(score, tokens)``; ``X`` ``[1, N, 10]``
    and ``y`` ``[1, N, 1]`` as fitfunc2 holds them (any device).  Returns the reference's
    output dict.  Candidates come back in beam order (the reference's order is process
    completion order, which is not reproducible).  ``cfg_params.bfgs.devices`` spreads the fit
    over several GPUs of this process (``bfgs.resolve_devices``); an invalid value raises
    ``ValueError`` here instead of failing every candidate.  ``sigma``: per-point standard deviations
    of ``y`` (1-D, N entries, any device) for weighted fits, see ``bfgs.bfgs_batch``; a bad ``sigma``
    raises ``ValueError`` here as well.  ``loss``, ``f_scale``: a robust loss (see ``bfgs.bfgs_batch``); the
    candidates are then fitted and ranked by the robust objective, and a bad value raises ``ValueError``.
    """
    w2i = test_data.word2id
    arity_1 = {w2i[n] for n in UNARY_NAMES if n in w2i}
    arity_2 = {w2i[n] for n in BINARY_NAMES if n in w2i}
    pow_id = w2i.get("pow")
    c_id = w2i.get("c", 3) if getattr(cfg_params, "no_c_in_pow", False) else None
    pad_id, start_id, finish_id = w2i.get("P", 0), w2i.get("S", 1), w2i.get("F", 2)

    if 3 in test_data.id2word:            # model.py:452-455 (mutates the shared metadata)
        test_data.id2word[3] = "constant"
    elif "c" in w2i:
        test_data.id2word[w2i["c"]] = "constant"

    sorted_hyps = sorted(hyps, key=lambda h: h[0], reverse=True)
    valid = []
    for score, ww in sorted_hyps:
        seq = _as_list(ww)
        if finish_id in seq:
            seq = seq[:seq.index(finish_id)]
        seq = [s for s in seq if s != pad_id]
        valency, _ = analyze_prefix_tree_context(seq, arity_1, arity_2, set(), pow_id, c_id, start_id)
        if valency == 0:
            valid.append(ww)
    if not valid and sorted_hyps:
        print("Warning: All beams were filtered out due to invalid structure. Fallback to top-1 raw.")
        valid = [sorted_hyps[0][1]]

    P_bfgs, L_bfgs, token = [], [], []
    if valid:
        resolve_devices(cfg_params)     # a wrong cfg.bfgs.devices is the caller's error, not every candidate's
        sigma_weights(sigma, X, cfg_params)   # so is a wrong sigma
        fitter.robust_loss(loss, f_scale)     # and a wrong loss
        try:
            outs = bfgs_batch(valid, X, y, cfg_params, test_data, x0=x0, engine=engine, lazy_strings=True,
                              sigma=sigma, loss=loss, f_scale=f_scale)
        except Exception as exc:  # noqa: BLE001 -- a batch-level failure fails every candidate
            outs = [exc] * len(valid)
        P_bfgs = LazyStrings()   # every string the reference returns; printed when read
        for ww, out in zip(valid, outs):
            if isinstance(out, Exception):
                continue
            P_bfgs.append(out[0])
            L_bfgs.append(out[2])
            token.append(ww)

    if len(L_bfgs) == 0 or all(np.isnan(np.array(L_bfgs, dtype=float))):
        L_bfgs = [float("nan")]
        best_L, best_P, best_tok = [float("nan")], [None], [None]
    else:
        b = int(np.nanargmin(np.array(L_bfgs, dtype=float)))
        best_P, best_L, best_tok = [P_bfgs[b]], [L_bfgs[b]], [token[b]]
    return {
        "pred_target": hyps[0][1] if hyps else [],
        "all_bfgs_preds": P_bfgs,
        "all_bfgs_loss": L_bfgs,
        "best_bfgs_preds": best_P,
        "best_bfgs_loss": best_L,
        "best_token": best_tok,
    }


def _bits(ids):
    m = 0
    for t in ids or ():
        t = int(t)
        if t < 0 or t >= 64:
            raise ValueError(f"token id {t} outside the 64-bit mask of vsr_beam_mask")
        m |= 1 << t
    return m


def _beam_rules(n_words, arity_1_ids, arity_2_ids, transcendental_ids, all_op_ids, masked_var_ids, pow_id, c_id,
                start_id, finish_id, pad_id, length_eq):
    from ..engine import native
    return native.BeamRules(arity1=_bits(arity_1_ids), arity2=_bits(arity_2_ids),
                            transcendental=_bits(transcendental_ids), all_ops=_bits(all_op_ids),
                            masked_vars=_bits([v for v in (masked_var_ids or ()) if int(v) < n_words]),
                            pow_id=-1 if pow_id is None else int(pow_id),
                            c_id=-1 if c_id is None else int(c_id), start_id=int(start_id),
                            finish_id=-1 if finish_id is None else int(finish_id),
                            pad_id=-1 if pad_id is None else int(pad_id), length_eq=int(length_eq))


class BeamMaskState:
    """The constraint mask of the beam search kept INCREMENTALLY on the device (``vsr_beam_mask_step``).

    The decode loop of ``fitfunc2`` appends one token per beam per step and re-orders the beams
    (model.py:412-440); the reference re-walks every prefix from its first token at every step
    (model.py:385-411).  Here the open frames of every beam's prefix tree live in device tensors:
    ``step(tokens, beam_scores)`` consumes the step's tokens and returns the ``-inf`` mask for the
    next one, ``reorder(beam_idx)`` follows the search's re-ordering.  No host synchronisation."""

    MAX_DEPTH = 128      # open frames (the stateless kernel walks with the same cap); prefixes are capped at length_eq <= 100 tokens

    def __init__(self, beam, n_words, device="cuda", **rules):
        from ..engine import native
        self.lib = native.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise native.VsrError("BeamMaskState needs a CUDA device (there is no CPU path)")
        self.beam, self.n_words = int(beam), int(n_words)
        self.rules = _beam_rules(n_words, **rules)
        D = self.MAX_DEPTH
        self.op = torch.full((beam, D), -1, dtype=torch.int8, device=self.device)
        self.missing = torch.zeros((beam, D), dtype=torch.int8, device=self.device)
        self.missing[:, 0] = 1
        self.cons = torch.zeros((beam, D), dtype=torch.int64, device=self.device)
        self.depth = torch.ones(beam, dtype=torch.int32, device=self.device)
        self.pos = torch.zeros(beam, dtype=torch.int32, device=self.device)

    def reorder(self, beam_idx):
        idx = torch.as_tensor(beam_idx, device=self.device, dtype=torch.long)
        self.op, self.missing, self.cons = self.op[idx].contiguous(), self.missing[idx].contiguous(), self.cons[idx].contiguous()
        self.depth, self.pos = self.depth[idx].contiguous(), self.pos[idx].contiguous()

    def step(self, tokens, beam_scores):
        import ctypes
        from ..engine import native
        tok = tokens.to(device=self.device, dtype=torch.int64).contiguous()
        sc = beam_scores.to(device=self.device, dtype=torch.float32).contiguous()
        out = torch.empty((self.beam, self.n_words), dtype=torch.float32, device=self.device)
        p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
        with torch.cuda.device(self.device):
            st = torch.cuda.current_stream().cuda_stream
            rc = self.lib.vsr_beam_mask_step(p(self.op), p(self.missing), p(self.cons), p(self.depth), p(self.pos),
                                             self.MAX_DEPTH, p(tok), self.beam, p(sc), ctypes.byref(self.rules),
                                             self.n_words, p(out), ctypes.c_void_p(st))
        if rc != 0:
            raise native.VsrError(f"vsr_beam_mask_step failed ({rc})")
        return out


def beam_constraint_mask(generated, cur_len, beam_scores, n_words, *, arity_1_ids, arity_2_ids,
                         transcendental_ids, all_op_ids, masked_var_ids, pow_id, c_id, start_id,
                         finish_id, pad_id, length_eq):
    """The "Constraint Logic" block of the beam search (model.py:382-411) as ONE device launch.

    ``generated``: [beam, L] int64 CUDA tensor of token ids, the first ``cur_len`` valid;
    ``beam_scores``: [beam] CUDA tensor.  Returns ``logit_mask`` [beam, n_words] float32 (0 or
    -inf) to be added to the log-probabilities, computed without a host synchronisation: the
    reference copies every beam to the host and walks it in Python at every decode step.
    """
    import ctypes
    from ..engine import native
    if not generated.is_cuda:
        raise native.VsrError("beam_constraint_mask needs CUDA tensors (there is no CPU path)")
    lib = native.load()
    gen = generated.to(torch.int64).contiguous()
    sc = beam_scores.to(torch.float32).contiguous()
    beam = int(gen.shape[0])
    out = torch.empty((beam, int(n_words)), dtype=torch.float32, device=gen.device)
    r = native.BeamRules(arity1=_bits(arity_1_ids), arity2=_bits(arity_2_ids),
                         transcendental=_bits(transcendental_ids), all_ops=_bits(all_op_ids),
                         masked_vars=_bits([v for v in (masked_var_ids or ()) if int(v) < n_words]),
                         pow_id=-1 if pow_id is None else int(pow_id),
                         c_id=-1 if c_id is None else int(c_id), start_id=int(start_id),
                         finish_id=-1 if finish_id is None else int(finish_id),
                         pad_id=-1 if pad_id is None else int(pad_id), length_eq=int(length_eq))
    with torch.cuda.device(gen.device):
        st = torch.cuda.current_stream().cuda_stream
        rc = lib.vsr_beam_mask(ctypes.c_void_p(gen.data_ptr()), int(gen.stride(0)), beam, int(cur_len),
                               ctypes.c_void_p(sc.data_ptr()), ctypes.byref(r), int(n_words),
                               ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(st))
    if rc != 0:
        raise native.VsrError(f"vsr_beam_mask failed ({rc})")
    return out
