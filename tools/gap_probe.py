"""Cost of Gap as an alphabet member: one C2-shaped data-derived SiteSampler run (1000 x 500 bp, k = 12, pc = 1e-4) on
  gap5    gap-padded rows (runs of Gap at both ends and sparse Gaps, about 10 % of the symbols), alphabet size 5: Gap has its
          own PWM row (the masked path with the Gap slot)
  gap4    the same rows, alphabet size 4: Gap is a dead symbol like N (the masked path as before)
  nogap   the same set before the Gaps were written, alphabet size 5 (the A,C,G,T-only path)
Each run is run_device + fetch_best of R restarts, timed with CUDA events after a warm-up, median of --reps.
Usage: python tools/gap_probe.py [--chains 256] [--reps 5] [--only gap5,gap4,nogap]   (needs a GPU; prints the device name
and power limit)
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
from gibbssampling_b200.engine import GibbsEngine, make_params  # noqa: E402
from gibbssampling_b200.synthetic import planted_motif_set  # noqa: E402


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        power = out.stdout.strip().splitlines()[0]
    except Exception:
        power = "unknown"
    return name, power


def gapped(seqs, seed=3):
    """Runs of 0-40 Gaps at both ends of every row and 2 % sparse Gaps inside: about 10 % of the symbols."""
    rng = np.random.default_rng(seed)
    out = []
    for s in seqs:
        a = np.frombuffer(s, dtype=np.uint8).copy()
        a[rng.random(len(a)) < 0.02] = ord("-")
        lo, hi = int(rng.integers(0, 41)), int(rng.integers(0, 41))
        a[:lo] = ord("-")
        if hi:
            a[len(a) - hi:] = ord("-")
        out.append(a.tobytes())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chains", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default="gap5,gap4,nogap")
    args = ap.parse_args()
    import torch
    dev_name, power = device_info()
    base = planted_motif_set(1000, 500, 12, seed=2).sequences()
    gap = gapped(base)
    frac = sum(s.count(b"-") for s in gap) / sum(len(s) for s in gap)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for name, seqs, alen in (("gap5", gap, 5), ("gap4", gap, 4), ("nogap", base, 5)):
        if name not in args.only.split(","):
            continue
        params = make_params(12, 1e-4, alen, [0.25] * 4, background=_abi.GIBBS_BG_DATA)
        with GibbsEngine(seqs) as eng:
            def run():
                eng.run_device(params, args.chains, chain_id_base=0, seed=1)
                return eng.fetch_best(args.chains - 1)
            best = run()   # warm-up of the same shapes
            times = []
            for _ in range(args.reps):
                ev[0].record()
                run()
                ev[1].record()
                torch.cuda.synchronize()
                times.append(ev[0].elapsed_time(ev[1]))
            st = best.stats
        print(json.dumps({"workload": name, "alphabet_size": alen, "gap_fraction": round(frac if name != "nogap" else 0.0, 4),
                          "chains": args.chains, "ms": round(float(np.median(times)), 2), "ms_all": [round(t, 2) for t in times],
                          "site_updates": st["site_updates"], "exact_rescans": st["exact_rescans"], "sum": best.total,
                          "device": dev_name, "power_limit": power, "timing": f"CUDA events, median of {args.reps}"}), flush=True)


if __name__ == "__main__":
    main()
