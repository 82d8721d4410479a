"""Batches over several GPUs (gibbs_multi_batch_*): the workloads of tools/batch_probe.py split over 1, 2, 4 and 8 device
slots. Slot i runs on GPU i % device_count, so on a box with fewer GPUs than slots the slots share a GPU (the line's
"gpus" says how many distinct GPUs ran). One JSON line per (workload, slot count).

Timed: run + fetch_best over all slots (MotifSampler motifAmount 2 also fetches the winners' Positions), ending in a
synchronise on every device; host clock, median of --reps after one warm-up. The first run of a fresh object (which also
builds the per-set W / PPM-value tables and synchronises once per slot) is reported apart. The winners are checked against
one-device BatchEngine before timing. For the workloads of --balance, each slot's block is also timed alone as a
one-device batch on its GPU (the same run + fetch_best, median of --reps): how evenly the create-time split (cost of a set =
the sum of its sequence lengths) spreads the work, and, as the slowest block, what the slots would take on GPUs of their own.
Usage: python tools/multi_batch_probe.py [--reps 5] [--only a,...,g] [--slots 1,2,4,8] [--balance a,...,g]
(needs a GPU; prints the device names and power limits)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from batch_probe import workload  # noqa: E402
from gibbssampling_b200 import _abi  # noqa: E402
from gibbssampling_b200.engine import BatchEngine, MultiBatchEngine, device_count, make_params  # noqa: E402
from gibbssampling_b200.synthetic import background_of  # noqa: E402


def devices_info():
    import torch
    names = [torch.cuda.get_device_name(d) for d in range(torch.cuda.device_count())]
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        power = out.stdout.strip().splitlines()
    except Exception:
        power = ["unknown"]
    return names, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default="a,b,c,d,e,f,g")
    ap.add_argument("--slots", default="1,2,4,8")
    ap.add_argument("--balance", default="a,b,c,d,e,f,g")
    args = ap.parse_args()
    import torch
    names, power = devices_info()
    ndev = device_count()
    counts = [int(x) for x in args.slots.split(",")]
    print(json.dumps({"visible_devices": ndev, "device_names": names, "power_limits": power}), flush=True)

    def sync_all():
        for d in range(ndev):
            torch.cuda.synchronize(d)

    for name in args.only.split(","):
        sets, k, R, bgmode, alen, m = workload(name)
        bgs = [background_of(np.frombuffer(b"".join(s), dtype=np.uint8), 1e-4, alen) for s in sets]
        fixed = bgmode == _abi.GIBBS_BG_FIXED
        motif = {"cutoff": 1.0, "sampler": _abi.GIBBS_MOTIF_SAMPLER, "motif_amount": m} if m else {}
        params = make_params(k, 1e-4, alen, bgs[0], background=bgmode, **motif)

        def run(eng, first=0, n=None):
            n = len(sets) if n is None else n
            bg = bgs[first:first + n] if fixed else None
            (eng.run_motif_device if m else eng.run_device)(params, R, bg_per_set=bg, chain_id_base=0, seed=1)
            best = eng.fetch_best(R - 1)
            return best, eng.fetch_best_positions(2) if m == 2 else None

        def timed(fn):
            ms = []
            for _ in range(args.reps):
                sync_all()
                t0 = time.perf_counter()
                fn()
                sync_all()
                ms.append((time.perf_counter() - t0) * 1e3)
            return float(np.median(ms)), float(np.min(ms)), float(np.max(ms))

        with BatchEngine(sets) as one:
            want, want_pos = run(one)
        for n in counts:
            sync_all()
            t0 = time.perf_counter()
            mb = MultiBatchEngine(sets, devices=[i % ndev for i in range(n)])
            sync_all()
            create_ms = (time.perf_counter() - t0) * 1e3
            t0 = time.perf_counter()
            got, got_pos = run(mb)
            sync_all()
            first_ms = (time.perf_counter() - t0) * 1e3
            same = all(g.sites.tolist() == w.sites.tolist() and g.scores.tobytes() == w.scores.tobytes() and g.restart == w.restart
                       for g, w in zip(got, want))
            same = same and (got_pos is None or all(np.array_equal(a, b) for a, b in zip(got_pos, want_pos)))
            t = timed(lambda: run(mb))
            blocks = mb.slot_sets()
            cost = [int(sum(sum(len(q) for q in sets[s]) for s in range(f, f + c))) for f, c in blocks]
            row = {
                "workload": name, "slots": n, "gpus": min(n, ndev), "sets": len(sets), "k": k, "restarts_per_set": R,
                "sampler": f"MotifSampler m={m}" if m else "SiteSampler", "background": "fixed" if fixed else "data",
                "identical_to_one_device_batch": bool(same),
                "ms": round(t[0], 3), "ms_min_max": [round(t[1], 3), round(t[2], 3)],
                "first_run_ms": round(first_ms, 3), "create_ms": round(create_ms, 3),
                "slot_sets": [c for _, c in blocks], "slot_bases": cost,
                "timing": f"host clock around run + fetch_best, synchronise on every device, median of {args.reps} after warm-up",
            }
            if name in args.balance.split(",") and n > 1:
                slot_ms = []
                for d, (f, c) in enumerate(blocks):
                    if c == 0:
                        slot_ms.append(0.0)
                        continue
                    with BatchEngine(sets[f:f + c], device=d % ndev) as b:
                        run(b, f, c)
                        slot_ms.append(round(timed(lambda: run(b, f, c))[0], 3))
                row["slot_alone_ms"] = slot_ms
            print(json.dumps(row), flush=True)
            mb.close()


if __name__ == "__main__":
    main()
