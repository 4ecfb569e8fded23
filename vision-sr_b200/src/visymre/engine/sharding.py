"""Multi-GPU sharding of one beam's (candidate, restart) runs (SURVEY.md section 8e).

Every run is independent (reference bfgs.py:102, model.py:491), so the C*R runs of a beam
are dealt to the ranks longest-first round-robin; X and y are replicated (every rank is
handed the same tensors by the caller).  There is no collective on the data path.  The
only exchange is at the end: each rank reduces its own restarts to ONE record per
candidate, ``[final_mse, restart, loss, consts...]``, one all-gather moves the records
(C * (3 + kmax) * 8 bytes per rank: latency-bound), and every rank takes the same argmin.
Ties and all-nan candidates resolve to the lowest restart index -- what ``np.nanargmin``
over the restarts gives on a single GPU (bfgs.py:134-141).

torch.distributed is plumbing here (NCCL on GPUs, gloo in the CPU tests).

``fit_devices`` is the same dealing and merge inside ONE process that holds an engine per device:
device-to-device copies of the records take the place of the all-gather.
"""
import contextlib

import numpy as np
import torch
import torch.distributed as dist


def partition_runs(cost, world):
    """Deal run indices to ``world`` ranks: sort by cost (descending, stable), round-robin.

    Returns a list of ``world`` int64 arrays; every run appears exactly once.
    """
    order = np.argsort(-np.asarray(cost, dtype=np.float64), kind="stable")
    return [np.sort(order[r::world]) for r in range(world)]


def world_size(group=None):
    return dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1


def rank(group=None):
    return dist.get_rank(group) if dist.is_available() and dist.is_initialized() else 0


def broadcast_from_rank0(t, group=None):
    """Rank 0's copy of ``t`` on every rank (starting points drawn from an unseeded RNG differ
    per process, bfgs.py:103)."""
    if world_size(group) > 1:
        dist.broadcast(t, src=0, group=group)
    return t


def local_best_records(final_mse, loss, consts, n_cand, n_restarts, mine, key_dtype=None):
    """Per-candidate best of THIS rank's restarts.

    final_mse, loss: [C*R]; consts: [C*R, kmax]; mine: bool [C*R], runs this rank fitted.
    Returns a float64 tensor [C, 4 + kmax]: (score with nan counted as +inf, restart index (R when
    the rank holds no run of the candidate), loss, consts, raw score).
    """
    dev = final_mse.device
    C, R = n_cand, n_restarts
    kmax = consts.shape[1]
    fm = final_mse.reshape(C, R).to(torch.float64)
    if key_dtype is not None:   # the reference compares the scores in X's dtype (bfgs.py:126-141)
        fm = fm.to(key_dtype).to(torch.float64)
    own = mine.reshape(C, R)
    ridx = torch.arange(R, device=dev).expand(C, R)
    # np.nanargmin (bfgs.py:134-137) = first minimum with every nan counted as +inf (an all-nan list
    # falls back to restart 0, which is the same thing).  Here: the same rule over THIS rank's slots.
    inf = torch.full_like(fm, float("inf"))
    key = torch.where(torch.isnan(fm), inf, fm)
    best_val = torch.where(own, key, inf).min(dim=1).values
    hit = own & (key == best_val[:, None])
    best_own = torch.where(hit, ridx, torch.full_like(ridx, R)).min(dim=1).values   # R: holds no run of it
    best_r = best_own.clamp(max=R - 1)
    rec = torch.zeros((C, 3 + kmax), dtype=torch.float64, device=dev)
    rows = torch.arange(C, device=dev) * R + best_r
    rec[:, 0] = best_val
    rec[:, 1] = best_own.to(torch.float64)
    rec[:, 2] = loss.reshape(-1)[rows]
    rec[:, 3:] = consts[rows]
    # keep the raw score (nan stays nan) for the winner's report
    raw = final_mse.reshape(-1)[rows].to(torch.float64)
    rec = torch.cat([rec, raw[:, None]], dim=1)
    return rec


def merge_records(all_recs, n_restarts=None):
    """all_recs: [world, C, 4 + kmax] gathered records -> [C, 4 + kmax] winners.

    Order of preference: smaller finite score, then lower restart index.
    """
    val = all_recs[:, :, 0]
    rst = all_recs[:, :, 1]
    # lexicographic argmin over the rank axis on (val, rst)
    best_val = val.min(dim=0).values
    cand = val == best_val[None]
    rst_masked = torch.where(cand, rst, torch.full_like(rst, float("inf")))
    winner = rst_masked.argmin(dim=0)
    C = all_recs.shape[1]
    return all_recs[winner, torch.arange(C, device=all_recs.device)]


def allgather_best(rec, group=None, n_restarts=None):
    """One all-gather of the per-candidate records; every rank returns the same winners."""
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return merge_records(rec[None], n_restarts)
    world = dist.get_world_size(group)
    parts = [torch.empty_like(rec) for _ in range(world)]
    dist.all_gather(parts, rec.contiguous(), group=group)   # the path's only collective
    return merge_records(torch.stack(parts), n_restarts)


def empty_result(n_slots, kstride, device):
    """What a rank that holds no run reports: every slot nan / not run."""
    from .fitter import FitResult
    nan = float("nan")
    return FitResult(consts=torch.full((n_slots, kstride), nan, dtype=torch.float64, device=device),
                     lastx=torch.full((n_slots, kstride), nan, dtype=torch.float64, device=device),
                     loss=torch.full((n_slots,), nan, dtype=torch.float64, device=device),
                     final_mse=torch.full((n_slots,), nan, dtype=torch.float64, device=device),
                     info=torch.full((n_slots, 4), -1, dtype=torch.int32, device=device))


def fit_sharded(engine, programs_k, n_restarts, x0, opts, cost=None, group=None, key_dtype=None):
    """Fit a beam with its runs sharded over the ranks of ``group``.

    programs_k: constants per candidate (engine.set_programs was called with the same
    list on every rank); x0: [C*R, kmax] (identical on every rank).  Returns
    ``(winners [C, 4+kmax], local FitResult)`` where winners[:, 0] is the comparison
    key, [:, 1] the restart, [:, 2] the objective, [:, 3:3+kmax] the constants (lastx)
    and [:, -1] the raw final MSE.
    """
    C, R = len(programs_k), n_restarts
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if cost is None:
        cost = np.repeat(np.asarray(programs_k, dtype=np.float64) + 1.0, R)
    mine_idx = partition_runs(cost, world)[rank]
    run_prog = (mine_idx // R).astype(np.int32)
    if len(mine_idx):
        res = engine.fit(run_prog, mine_idx.astype(np.int32), x0, opts)
    else:
        # more ranks than runs: this rank fits nothing but must still take part in the all-gather
        # (vsr_fit rejects an empty run list; raising here would leave the others in the collective)
        res = empty_result(C * R, int(torch.as_tensor(x0).shape[1]), engine.device)
    mine = torch.zeros(C * R, dtype=torch.bool, device=res.loss.device)
    mine[torch.as_tensor(mine_idx, device=mine.device)] = True
    rec = local_best_records(res.final_mse, res.loss, res.lastx, C, R, mine, key_dtype)
    return allgather_best(rec, group, n_restarts=R), res


def _engine_streams(engines):
    """The stream each engine fits on: its device's current stream for the first engine of a device, side
    stream j for the j-th further one (``fitter.device_engines`` made it with that stream); None off CUDA."""
    from . import fitter
    seen, out = {}, []
    for eng in engines:
        dev = torch.device(eng.device)
        j = seen.get(dev, 0)
        seen[dev] = j + 1
        if dev.type != "cuda":
            out.append(None)
        else:
            out.append(torch.cuda.current_stream(dev) if j == 0 else fitter.side_stream(dev, j))
    return out


def _on(dev, stream):
    ctx = contextlib.ExitStack()
    if stream is not None:
        ctx.enter_context(torch.cuda.device(dev))
        ctx.enter_context(torch.cuda.stream(stream))
    return ctx


def fit_devices(engines, programs_k, n_restarts, x0, opts, cost=None, key_dtype=None):
    """Fit a beam with its runs dealt over the engines of ONE process, ``engines[0]``'s device being the
    home device: the single-process twin of ``fit_sharded``, with the same dealing (``partition_runs``),
    the same per-part reduction (``local_best_records``) and the same merge (``merge_records``), so that
    the winners are those of one engine that fits every run.

    Every engine holds the same points and the same program list (``fitter.share_points``,
    ``set_programs``); an engine may share its device with others.  x0: [C*R, kmax] on the home device
    (or the host); it is copied once to every other device on the home stream.  Every engine's fit is
    enqueued before the host waits on any of them, so that they run concurrently.  The records travel
    to the home device by device-to-device copies.  Returns ``(winners [C, 4+kmax] on the home device,
    [FitResult per engine])`` -- the layout of ``fit_sharded``.  When any device fails, ``VsrError``
    names it, raised once every device's work has finished.
    """
    from .native import VsrError
    C, R = len(programs_k), n_restarts
    if cost is None:
        cost = np.repeat(np.asarray(programs_k, dtype=np.float64) + 1.0, R)
    parts = partition_runs(cost, len(engines))
    home = torch.device(engines[0].device)
    x0 = torch.as_tensor(x0, dtype=torch.float64).to(home)
    kstride = int(x0.shape[1])
    x0_on = {}
    for eng in engines:        # peer copies on the home stream; torch makes the device's stream wait for them
        x0_on.setdefault(torch.device(eng.device), None)
    for dev in x0_on:
        x0_on[dev] = x0.to(dev, non_blocking=True)
    streams = _engine_streams(engines)
    results, recs, errors = [None] * len(engines), [None] * len(engines), []
    for i, (eng, mine_idx, stream) in enumerate(zip(engines, parts, streams)):
        dev = torch.device(eng.device)
        cur = torch.cuda.current_stream(dev) if stream is not None else None
        try:
            with _on(dev, stream):
                x0_d = x0_on[dev]
                if stream is not None and stream != cur:   # a further engine of the device: after the uploads
                    stream.wait_stream(cur)
                    x0_d.record_stream(stream)
                if len(mine_idx):
                    res = eng.fit((mine_idx // R).astype(np.int32), mine_idx.astype(np.int32), x0_d, opts)
                else:      # more engines than runs (vsr_fit rejects an empty run list)
                    res = empty_result(C * R, kstride, dev)
                mine = torch.zeros(C * R, dtype=torch.bool)
                mine[torch.as_tensor(mine_idx, dtype=torch.long)] = True
                # pageable host -> device without a stream synchronisation: the fit above stays in flight
                mine = mine.to(dev, non_blocking=True)
                rec = local_best_records(res.final_mse, res.loss, res.lastx, C, R, mine, key_dtype)
            if stream is not None and stream != cur:
                cur.wait_stream(stream)
                rec.record_stream(cur)          # read there by the copy or the merge
            with _on(dev, cur):
                recs[i] = rec.to(home, non_blocking=True)
            results[i] = res
        except Exception as exc:  # noqa: BLE001 -- raised below, once no device works any more
            errors.append((dev, exc))
    for dev in x0_on:
        if dev.type == "cuda":
            try:
                torch.cuda.synchronize(dev)
            except Exception as exc:  # noqa: BLE001 -- an asynchronous error of that device's work
                errors.append((dev, exc))
    if errors:
        dev, exc = errors[0]
        more = f" (and {len(errors) - 1} more: {', '.join(str(d) for d, _ in errors[1:])})" if len(errors) > 1 else ""
        raise VsrError(f"fit on {dev} failed: {exc}{more}") from exc
    return merge_records(torch.stack(recs), R), results
