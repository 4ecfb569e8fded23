#!/usr/bin/env python
"""GPU experiment: one beam's runs dealt over several GPUs of ONE process (cfg.bfgs.devices).

    python tools/exp_devices.py [--beams2 6] [--beams4 2] [--rounds 2] [--out FILE]

Config 2 and config 4 beams of bench.py go through ``refine_hypotheses`` with ``devices`` = the first
1, 2, 4 and 8 GPUs (as many as exist; with a single GPU the extra setting [0, 0] -- two engines on one
GPU -- runs the multi-device path there).  The settings alternate beam by beam within this process,
the compile cache is warm (every skeleton is compiled in an untimed first pass, as in a driver that
calls fitfunc2 on the same problem again) and the host's garbage collector is off in the timed loop.
Per setting: candidate-fits/s, ms per beam (host clock around the call, which ends in a device
synchronisation) and the number of candidates whose winner (string or loss bits) differs from the
one-device run of the same beam.  The card name and power limit are read in the same process.  Writes
JSON (default profiles/exp_devices_<n>gpu.json) and exits 1 when any winner differs.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "vision-sr_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from src.visymre.architectures.refine import refine_hypotheses  # noqa: E402
from src.visymre.workloads import generator as wg  # noqa: E402


def cards():
    """Name, power limit and max SM clock of every visible GPU (nvidia-smi, read only)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout
    except Exception as exc:  # noqa: BLE001
        return [{"error": str(exc)}]
    rows = []
    for line in out.strip().splitlines():
        f = [x.strip() for x in line.split(",")]
        if len(f) >= 4:
            rows.append({"index": int(f[0]), "name": f[1], "power_limit": f[2], "sm_max_clock": f[3]})
    return rows


def winners(out):
    """Per candidate: (string, loss dtype and bytes); the best one last."""
    def bits(v):
        a = np.asarray(v)
        return a.dtype.str, a.tobytes().hex()
    rows = [(str(s), bits(v)) for s, v in zip(out["all_bfgs_preds"], out["all_bfgs_loss"])]
    best = (None if out["best_bfgs_preds"][0] is None else str(out["best_bfgs_preds"][0]), bits(out["best_bfgs_loss"][0]))
    return rows + [best]


def settings(n_gpus):
    out = [list(range(n)) for n in (1, 2, 4, 8) if n <= n_gpus]
    if n_gpus == 1:
        out.append([0, 0])
    return out


def run_config(config, n_beams, rounds, sets):
    c = bench.CONFIGS[config]
    args = argparse.Namespace(config=config, points=c["points"], cand=c["cand"], restarts=c["restarts"], rows="")
    beams = bench.make_workload(n_beams, args)
    td = wg.make_test_data()
    cfg = wg.make_cfg(c["restarts"], c["cand"], grad_mode="dual", precision=c["precision"])
    data = []
    for b in beams:
        X = torch.from_numpy(np.ascontiguousarray(b.X[None])).pin_memory()
        y = torch.from_numpy(np.ascontiguousarray(b.y)).reshape(1, -1, 1).pin_memory()
        data.append((b, X, y, [(-float(j), t) for j, t in enumerate(b.tokens)]))

    def call(i, devs):
        b, X, y, hyps = data[i]
        cfg.bfgs.devices = devs
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = refine_hypotheses(hyps, X.to("cuda:0", non_blocking=True), y.to("cuda:0", non_blocking=True), cfg, td,
                                x0=b.x0)
        best = out["best_bfgs_preds"][0]    # the one string a driver reads (bench.py's e2e does the same)
        for d in set(devs):
            torch.cuda.synchronize(d)
        dt = (time.perf_counter() - t0) * 1e3
        del best
        return dt, winners(out)             # every other string is printed outside the timing

    for i in range(len(data)):              # untimed: compile cache, engines, side streams
        for devs in sets:
            call(i, devs)
    # the one-device answer, compile cache warm as in the timed calls: with a cold cache the one-engine
    # path fits a beam in stages as its skeletons get compiled, and on config 4 such a fit has been seen
    # to differ in the last bits from the one-stage fit (DESIGN.md section 5.1)
    ref = {i: call(i, [0])[1] for i in range(len(data))}
    ms = {str(d): [] for d in sets}
    differ = {str(d): 0 for d in sets}
    gc.collect()
    gc.disable()
    try:
        for r in range(rounds):
            for i in range(len(data)):
                k = (i + r) % len(sets)
                for devs in sets[k:] + sets[:k]:       # a different setting first on every beam
                    dt, w = call(i, devs)
                    ms[str(devs)].append(dt)
                    differ[str(devs)] += sum(1 for a, b_ in zip(w, ref[i]) if a != b_) + abs(len(w) - len(ref[i]))
    finally:
        gc.enable()
    out = {"config": config, "what": c["what"], "candidates": c["cand"], "restarts": c["restarts"],
           "points": c["points"], "precision": c["precision"], "beams": [d[0].name for d in data], "rounds": rounds,
           "settings": {}}
    for devs in sets:
        m = ms[str(devs)]
        out["settings"][str(devs)] = {
            "devices": devs, "engines": len(devs), "gpus": len(set(devs)),
            "fits_per_s": c["cand"] * len(m) / (sum(m) / 1e3),
            "ms_per_beam": float(np.mean(m)), "ms_per_beam_median": float(np.median(m)),
            "ms_per_beam_min": float(np.min(m)), "ms_per_beam_max": float(np.max(m)), "calls": len(m),
            "winners_differing_from_one_device": differ[str(devs)]}
        print(f"config {config} devices {devs}: {out['settings'][str(devs)]['fits_per_s']:.0f} fits/s, "
              f"{np.mean(m):.1f} ms/beam, {differ[str(devs)]} winners differ", flush=True)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--beams2", type=int, default=6, help="config-2 beams (0: skip)")
    ap.add_argument("--beams4", type=int, default=2, help="config-4 beams (0: skip)")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("exp_devices: no CUDA device (this is a GPU measurement)")
    n = torch.cuda.device_count()
    sets = settings(n)
    result = {"tool": "tools/exp_devices.py", "gpus_visible": n, "cards": cards(),
              "path": "refine_hypotheses(token ids, pinned host X / y, cfg with bfgs.devices) -> dict, strings read; "
                      "warm compile cache", "configs": []}
    for config, nb in ((2, a.beams2), (4, a.beams4)):
        if nb > 0:
            result["configs"].append(run_config(config, nb, a.rounds, sets))
    result["cards_after"] = cards()
    bad = sum(s["winners_differing_from_one_device"] for c in result["configs"] for s in c["settings"].values())
    result["winners_differing_from_one_device"] = bad
    path = a.out or os.path.join(ROOT, "profiles", f"exp_devices_{n}gpu.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as fh:
        json.dump(result, fh, indent=1)
    print("wrote", path, "winners differing:", bad, flush=True)
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
