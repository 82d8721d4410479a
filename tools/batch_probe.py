"""Batch of many sequence sets (gibbs_batch_*) against a loop of single-set handles: one JSON line per workload.

The loop creates its handles outside the timed window and times run_device + fetch_best per set, ending in a synchronise;
the batch times run_device + fetch_best over all sets. Both are timed with CUDA events after a warm-up of the same shapes,
and both compute the same per-set winners (checked before timing). Workloads:
  a  1024 sets of 20 x 100 bp, k = 8, R = 2, fixed background (the script's reps = 1 on C1-shaped sets)
  b  62 sets of 9-31 sequences of 45-1300 bp, k = 6, R = 2, data-derived background, alphabet size 5 without Gap
  c  64 sets of 100 x 500 bp, k = 12, R = 64, fixed background
MotifSampler (run_motif_device; pc = 1e-4, cutOff = 1.0; motifAmount 2 also fetches the winners' Positions lists):
  d  the sets of a, k = 8, R = 2, fixed background, motifAmount 1
  e  the sets of b, k = 6, R = 2, data-derived background, alphabet size 5, motifAmount 2 (fsx:407 per gene group)
  f  the same with motifAmount 1
  g  the sets of c, k = 12, R = 64, fixed background, motifAmount 1
Usage: python tools/batch_probe.py [--reps 5] [--only a,b,c,d,e,f,g]   (needs a GPU; prints the device name and power limit)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from gibbssampling_b200 import _abi  # noqa: E402
from gibbssampling_b200.engine import BatchEngine, GibbsEngine, make_params  # noqa: E402
from gibbssampling_b200.synthetic import background_of, planted_motif_set  # noqa: E402


def workload(name):
    """(sets, k, R, background, alphabet size, motifAmount: 0 = the SiteSampler)"""
    if name in "ad":
        seqs = planted_motif_set(1024 * 20, 100, 8, seed=11).sequences()
        return [seqs[20 * s: 20 * s + 20] for s in range(1024)], 8, 2, _abi.GIBBS_BG_FIXED, 4, 1 if name == "d" else 0
    if name in "bef":
        rng = np.random.default_rng(62)
        sets = [planted_motif_set(int(rng.integers(9, 32)), 1300, 6, seed=500 + s, min_length=45).sequences() for s in range(62)]
        return sets, 6, 2, _abi.GIBBS_BG_DATA, 5, {"b": 0, "e": 2, "f": 1}[name]
    seqs = planted_motif_set(64 * 100, 500, 12, seed=13).sequences()
    return [seqs[100 * s: 100 * s + 100] for s in range(64)], 12, 64, _abi.GIBBS_BG_FIXED, 4, 1 if name == "g" else 0


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        power = out.stdout.strip().splitlines()[0]
    except Exception:
        power = "unknown"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default="a,b,c,d,e,f,g")
    args = ap.parse_args()
    import torch
    dev_name, power = device_info()
    for name in args.only.split(","):
        sets, k, R, bgmode, alen, m = workload(name)
        bgs = [background_of(np.frombuffer(b"".join(s), dtype=np.uint8), 1e-4, alen) for s in sets]
        fixed = bgmode == _abi.GIBBS_BG_FIXED
        motif = {"cutoff": 1.0, "sampler": _abi.GIBBS_MOTIF_SAMPLER, "motif_amount": m} if m else {}
        params = [make_params(k, 1e-4, alen, bgs[s], background=bgmode, **motif) for s in range(len(sets))]
        batch = BatchEngine(sets)
        singles = [GibbsEngine(s) for s in sets]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

        def run_batch():
            (batch.run_motif_device if m else batch.run_device)(params[0], R, bg_per_set=bgs if fixed else None, chain_id_base=0, seed=1)
            best = batch.fetch_best(R - 1)
            return best, batch.fetch_best_positions(2) if m == 2 else [None] * len(sets)

        def run_loop():
            best, pos = [], []
            for s, eng in enumerate(singles):
                eng.run_device(params[s], R, chain_id_base=0, seed=1)
                best.append(eng.fetch_best(R - 1))
                pos.append(eng.fetch_best_positions(2) if m == 2 else None)
            torch.cuda.synchronize()
            return best, pos

        (got, got_pos), (want, want_pos) = run_batch(), run_loop()   # warm-up of every shape, and the results must agree
        same = all(g.sites.tolist() == w.sites.tolist() and g.scores.tobytes() == w.scores.tobytes() for g, w in zip(got, want))
        same = same and all(gp is None or np.array_equal(gp, wp) for gp, wp in zip(got_pos, want_pos))
        windows = sum(b.stats["window_scores"] for b in got[:1])   # (stats of a batch fetch are batch-wide)

        def timed(fn):
            ms = []
            for _ in range(args.reps):
                torch.cuda.synchronize()
                ev[0].record()
                fn()
                ev[1].record()
                ev[1].synchronize()
                ms.append(ev[0].elapsed_time(ev[1]))
            return float(np.median(ms)), float(np.min(ms)), float(np.max(ms))

        tb, tl = timed(run_batch), timed(run_loop)
        print(json.dumps({
            "workload": name, "sets": len(sets), "seqs": int(sum(len(s) for s in sets)), "k": k, "restarts_per_set": R,
            "background": "fixed" if fixed else "data", "sampler": f"MotifSampler m={m}" if m else "SiteSampler",
            "identical_to_single_handles": bool(same),
            "window_scores": int(windows),
            "batch_ms": round(tb[0], 3), "batch_ms_min_max": [round(tb[1], 3), round(tb[2], 3)],
            "loop_ms": round(tl[0], 3), "loop_ms_min_max": [round(tl[1], 3), round(tl[2], 3)],
            "batch_ms_per_set": round(tb[0] / len(sets), 5), "loop_ms_per_set": round(tl[0] / len(sets), 5),
            "batch_window_scores_per_s": windows / (tb[0] * 1e-3), "loop_window_scores_per_s": windows / (tl[0] * 1e-3),
            "speedup": round(tl[0] / tb[0], 2), "device": dev_name, "power_limit": power, "timing": "CUDA events, median of "
            f"{args.reps} after one warm-up",
        }), flush=True)
        batch.close()
        for e in singles:
            e.close()


if __name__ == "__main__":
    main()
