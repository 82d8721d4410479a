#!/usr/bin/env python
"""bench.py -- Gibbs window-scores/s and site-updates/s on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C2] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one pass of the hot path over one batch: `chains` independent restarts of
SiteSampler.doSiteSamplingWithBPV (fs:691-695: random starts, greedy sweeps to convergence, left and
right phase-shift sweeps) on synthetic planted-motif DNA. At N = 1 the workload is BASELINE.json
configs[1] (C2: 1000 seqs x 500 bp, k = 12, 1024 chains). With N > 1 every rank runs `chains` more
chains (weak scaling; chain ids are global so results do not depend on N) and the step ends with the
single NCCL all_gather of each GPU's best (sum of scores, site vector).

One JSON line is printed by rank 0. `value` = window-scores/s over all ranks with the sequences
already resident in HBM (CUDA events on the launch stream, max over ranks); `e2e` = the same metric
through the public API with HOST buffers: per step the ASCII sequences are uploaded from pinned
memory and 2-bit packed, the chains run, and sites/scores/sums come back to the host.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (n_seqs, length, k, chains per GPU, phase shifts)
    "C1": (20, 100, 8, 1001, True),       # reference-scale: 20 x 100 bp, planted 8-mer, ONE sequential chain of 1000 iterations
                                          # = numberOfRepetitions 1000 of fs:434 (at most 1001 restarts, run here as parallel chains)
    "C2": (1000, 500, 12, 1024, True),    # the single-GPU configuration the metric is quoted on
    "C3": (10000, 1000, 16, 1024, True),  # 8192 restarts over 8 GPUs = 1024 per GPU
    "C4": (100000, 200, 20, 148, True),   # ChIP-seq-peak-sized set with phase-shift moves
}
# dram__bytes_read.sum + dram__bytes_write.sum of the seven kernels of one C2 step (ncu --set full, round 2, final build):
# init_smem_kernel, chain_kernel T = 1 / 4 / 8 / 16, chain_cluster_kernel 4 / 8 (read, write in MB each)
NCU_DRAM_BYTES_PER_STEP = int((0.224000 + 0.0 + 12.561920 + 0.000256 + 12.574208 + 1.253120 + 6.464000 + 0.000256 + 1.509120
                               + 0.000256 + 0.552192 + 0.0 + 0.465664 + 0.0) * 1e6)
NCU_DRAM_SOURCE = ("dram__bytes_read.sum + dram__bytes_write.sum of the seven kernels of one C2 step (init_smem_kernel, "
                   "chain_kernel T=1/4/8/16, chain_cluster_kernel 4/8), profiles/r02_ncu_c2_step_summary.txt")
# --family: which reference family the step runs (the default is the BASELINE.json workload)
FAMILIES = {
    "bpv": ("SiteSampler WithBPV restarts (fs:691)", "fixed (WithBPV), whole-set base counts",
            "gibbs::chain_kernel (a step = init_smem_kernel / init_tiled_kernel / init_kernel + chain_kernel<KP,1|4|8|16> + chain_cluster_kernel<KP,4|8>, "
            "timed together: kernel_ms)", "do_site_sampling_with_bpv"),
    "data": ("SiteSampler restarts with the data-derived drifting background (doSiteSampling, fs:697)",
             "data-derived, rebuilt per window (fs:470-473)", "gibbs::chain_kernel<KP, T, MASKED, DRIFT = true>", "do_site_sampling"),
    "motif": ("MotifSampler m = 1 restarts with a fixed background (doMotifSamplingWithPCV, fs:876), cutOff 0",
              "fixed pcv, whole-set base counts", "gibbs::motif_kernel<KP, T = 4>", None),
    "motif-data": ("MotifSampler m = 1 restarts with the data-derived background (doMotifSampling, fs:1034), cutOff 0",
                   "data-derived, rebuilt per held-out sequence (fs:896-905)", "gibbs::motif_kernel<KP, T = 4>", None),
}
PSEUDOCOUNT = 1e-4      # fsx:384
ALPHABET_SIZE = 5       # dnaBases = [A; T; G; C; Gap], fsx:368-369
SEED = 0xB200


def algorithmic_smem_bytes_per_window(k: int) -> float:
    """SURVEY.md section 8(d): k log-odds reads of 4 B + 2k bits of sequence per window score."""
    return 4.0 * k + k / 4.0


def algorithmic_hbm_bytes_per_site_update(length: int) -> float:
    """SURVEY.md section 8(d): ceil(L/4) packed row bytes + 8 B (old site read + new site write)."""
    return float((length + 3) // 4 + 8)


def workload_config(cfg_name: str, cfg, family: str, chains: int) -> dict:
    """The `config` object: identical for the GPU arm and the reference arm (the driver compares them)."""
    n, length, k, _, shifts = cfg
    fam_text, fam_bg, _, _ = FAMILIES[family]
    return {"workload": f"{cfg_name}: {n} seqs x {length} bp, k={k}, {chains} chains/GPU, {fam_text}"
                        + ("" if family.startswith("motif") else
                           f" (random starts + greedy sweeps + {'left/right shift sweeps' if shifts else 'no shifts'})"),
            "family": family, "chains_per_gpu": chains, "pseudocount": PSEUDOCOUNT, "alphabet_size": ALPHABET_SIZE,
            "background": fam_bg}


class ClockSampler:
    """nvidia-smi clocks and throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, indices):
        """indices: the GPUs of this job. ONE sampler process for all of them (rank 0 runs it): every extra nvidia-smi
        polling the driver at 10 Hz can stall kernel launches of every rank for a moment."""
        self.index = ",".join(str(i) for i in indices)
        self.proc = None
        self.lines: list[str] = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self) -> int:
        """index of the next sample: brackets the timed region inside a sampler that started earlier"""
        return len(self.lines)

    def stop(self, first: int = 0, last: int | None = None) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)   # let the sample that covers the end of the region arrive
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        ng = self.index.count(",") + 1      # one line per GPU per sample
        lines = self.lines[max(first - ng, 0): (last + 2 * ng) if last is not None else None] or self.lines[-2 * ng:]
        for line in lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks() -> dict:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        d["_source"] = "measured (MEASURED_PEAKS.json)"
        return d
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "_source": "fallback (B200_PROFILING.md)"}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the oracle (C restatement of the F# reference; the reference itself needs .NET, absent here)
# ---------------------------------------------------------------------------------------------------
def _oracle():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    oracle_lib.lib()
    return oracle_lib


def cpu_sample(ps, k, bg, *, threads: int, full_restart: bool, seed: int, chain_base: int,
               family: str = "bpv") -> tuple[float, int, int]:
    """Run `threads` chains concurrently on host threads (ctypes releases the GIL).
    Returns (wall seconds, window scores, site updates)."""
    O = _oracle()
    S = O.sources(ps.sequences())
    pcv = O.pcv_from_acgt(bg)
    if family == "data":
        name, pcv = ("do_site_sampling" if full_restart else "random_starts"), None
    else:
        name = "do_site_sampling_with_bpv" if full_restart else "random_starts_with_bpv"
    out = [None] * threads

    def work(t):
        rng, _ = O.make_rng(seed=seed, chain=chain_base + t)
        _, _, st = O.site_step(name, S, k, PSEUDOCOUNT, pcv=pcv, rng=rng)
        out[t] = (st.window_scores, st.site_updates)

    ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    t0 = time.perf_counter()
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    dt = time.perf_counter() - t0
    return dt, sum(o[0] for o in out), sum(o[1] for o in out)


def run_reference_arm(args, cfg_name, cfg) -> None:
    """`--impl reference`: the reference's CPU algorithm on the box's host cores. The F# cannot run here
    (no .NET runtime in the image or on the GPU box), so this times the oracle port -- its FAITHFUL mode: from-scratch
    leave-one-out rebuilds and a PWM per window like GibbsSampling.fs -- with all host threads. Same work as the GPU
    arm: whole restarts of the family's pipeline (random starts, greedy sweeps to convergence, left and right shift
    sweeps) on the same synthetic set, chain ids taken from the same range; one step = one restart per host thread
    (a bounded sample of the step's `chains` restarts)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from gibbssampling_b200.synthetic import background_of, planted_motif_set

    n, length, k, chains, shifts = cfg
    if args.chains:
        chains = args.chains
    if args.family.startswith("motif"):
        print(json.dumps({"impl": "reference", "unavailable": "the CPU port times the SiteSampler families only"}), flush=True)
        return
    ps = planted_motif_set(n, length, k, seed=SEED)
    bg = background_of(ps.ascii, PSEUDOCOUNT, ALPHABET_SIZE)
    cores = os.cpu_count() or 1
    # C3 / C4 restarts take hours in the faithful mode: there a step is one random-start sweep per thread
    full = n * n * length <= 2_000_000_000
    for w in range(args.warmup):
        cpu_sample(ps, k, bg, threads=cores, full_restart=full, seed=SEED, chain_base=(w * cores) % max(chains, 1), family=args.family)
    tot_t = tot_w = tot_u = 0.0
    for s in range(args.steps):
        dt, ws, us = cpu_sample(ps, k, bg, threads=cores, full_restart=full, seed=SEED,
                                chain_base=((args.warmup + s) * cores) % max(chains, 1), family=args.family)
        tot_t += dt
        tot_w += ws
        tot_u += us
    value = tot_w / tot_t
    what = (f"whole {FAMILIES[args.family][3]} restarts" if full else "one random-start sweep (fs:412) of a restart (whole restarts take hours at this size)")
    sample = (f"per step: {what}, one per host thread ({cores} threads, {int(tot_u / max(args.steps, 1))} site updates per step, "
              f"from-scratch PWM per site update and per window like the F#); oracle port (C, -O2, faithful mode)")
    line = {
        "impl": "reference", "metric": "gibbs_window_scores_per_sec", "value": value, "unit": "window-scores/s",
        "site_updates_per_sec": tot_u / tot_t, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot_t / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic planted-motif DNA (Philox key 0xB200, 10% planted-base mutation)",
        "config": workload_config(cfg_name, cfg, args.family, chains),
        "cpu_baseline": {"value": value, "unit": "window-scores/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "window-scores/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
DUMP_CHAIN_BYTES = 56 << 20   # per-chain arrays of --dump-outputs; with the winner's rows the dump stays under 64 MB


def last_step_outputs(eng, best) -> dict:
    """--dump-outputs: the results of the engine's last run_device, as float64 arrays (sites are exact in float64).
    best_*: the restart loop's winner as gibbs_fetch_best returns it (its scores and sites, their sum, which restart;
    restart -1 = the loop's initial value). chain_*: every restart's sites, scores and sum (gibbs_fetch), row i being
    restart chain_index[i]. When all restarts would exceed DUMP_CHAIN_BYTES, a fixed sample of them (seed SEED, rows in
    ascending order) is written instead, so two builds run with the same arguments write the same rows."""
    import numpy as np

    out = {"best_sites": best.sites, "best_scores": best.scores, "best_total": [best.total], "best_restart": [best.restart]}
    out = {name: np.array(v, dtype=np.float64) for name, v in out.items()}     # copies: `best` may be a reused pinned buffer
    res = eng.fetch(want_counts=False)
    chains, n = res.sites.shape
    rows = np.arange(chains)
    keep = DUMP_CHAIN_BYTES // (8 * (2 * n + 2))
    if chains > keep:
        rows = np.sort(np.random.default_rng(SEED).choice(chains, size=keep, replace=False))
    out.update({"chain_index": rows, "chain_sites": res.sites[rows], "chain_scores": res.scores[rows],
                "chain_sums": res.sums[rows]})
    return {name: np.asarray(v, dtype=np.float64) for name, v in out.items()}


def run_gpu_arm(args, cfg_name, cfg) -> None:
    import numpy as np
    import torch
    import torch.distributed as dist

    from gibbssampling_b200 import _abi
    from gibbssampling_b200.distributed import allgather_best
    from gibbssampling_b200.engine import GibbsEngine, make_params, measure_smem_bandwidth
    from gibbssampling_b200.synthetic import background_of, planted_motif_set

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: gibbssampling_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    n, length, k, chains, shifts = cfg
    if args.chains:
        chains = args.chains
    ps = planted_motif_set(n, length, k, seed=SEED)
    bg = background_of(ps.ascii, PSEUDOCOUNT, ALPHABET_SIZE)

    def params_of(family: str):
        return make_params(k, PSEUDOCOUNT, ALPHABET_SIZE, bg, phase_shifts=shifts,
                           background=_abi.GIBBS_BG_DATA if family in ("data", "motif-data") else _abi.GIBBS_BG_FIXED,
                           sampler=_abi.GIBBS_MOTIF_SAMPLER if family.startswith("motif") else _abi.GIBBS_SITE_SAMPLER,
                           cutoff=0.0)

    fam_text, fam_bg, fam_kernel, fam_oracle = FAMILIES[args.family]
    params = params_of(args.family)

    # pinned host copies of the inputs (e2e path uploads them every step)
    host_ascii = torch.empty(ps.ascii.size, dtype=torch.uint8, pin_memory=True)
    host_ascii.numpy()[:] = ps.ascii
    host_off = torch.empty(ps.offsets.size, dtype=torch.int64, pin_memory=True)
    host_off.numpy()[:] = ps.offsets

    eng = GibbsEngine(ps.sequences(), device=local_rank)
    for item in args.opt:                    # measurement switches (gibbs_set_option): none changes a result
        name, _, value = item.partition("=")
        eng.set_option(getattr(_abi, "GIBBS_OPT_" + name.upper()), int(value))
    stream = torch.cuda.Stream()            # a real (non-NULL) stream shared by torch events and the library
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.int32, device="cuda")  # > 126 MB L2
    chain_base = rank * chains
    reps = chains - 1                        # numberOfRepetitions of the restart loop the step's restarts feed (fs:434)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def finish_step(e):
        """the restart loop (fs:435-459) on the device; only the winner's rows come back; N > 1: one all_gather"""
        best = e.fetch_best(reps, pinned=True)
        if world > 1:
            allgather_best(best.total, chain_base + max(best.restart, 0), best.sites, best.scores)
        return best

    def timed_steps(e, prm, n_steps, seed0):
        """n_steps device-resident steps, each inside its own CUDA-event window on the launch stream (L2 flushed
        before the window opens). Returns (per-step windows in ms, per-step stats, the last step's winner)."""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_steps)]
        stats = []
        for s_ in range(n_steps):
            flush.fill_(s_)                     # L2 flush between steps, outside the per-step event window
            ev[s_][0].record(stream)
            e.run_device(prm, chains, chain_id_base=chain_base, seed=seed0 + s_)
            ev[s_][1].record(stream)
            best_ = finish_step(e)              # sync + D2H of the winner (not inside the event window)
            stats.append(best_.stats)
        return [a_.elapsed_time(b_) for a_, b_ in ev], stats, best_

    sampler = None
    if rank == 0:                            # ONE nvidia-smi for all GPUs of the job, started early (it needs a moment)
        sampler = ClockSampler(range(world))
        sampler.start()
    # ---- warm-up ----
    for w in range(args.warmup):
        eng.run_device(params, chains, chain_id_base=chain_base, seed=SEED - 1 - w)
        finish_step(eng)
    barrier()

    # ---- timed: device-resident ----
    barrier()
    clk_first = sampler.mark() if sampler else 0
    t_wall0 = time.perf_counter()
    win_ms, step_stats, last_best = timed_steps(eng, params, args.steps, SEED)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clk_last = sampler.mark() if sampler else 0
    outputs = last_step_outputs(eng, last_best) if (args.dump_outputs and rank == 0) else None
    dev_ms = sum(win_ms)
    tot_windows = sum(st["window_scores"] for st in step_stats)
    tot_updates = sum(st["site_updates"] for st in step_stats)
    tot_sweeps = sum(st["sweeps"] for st in step_stats)
    tot_rescans = sum(st["exact_rescans"] for st in step_stats)
    launches = sum(st["kernel_launches"] for st in step_stats)
    kernel_ms = [st["kernel_ms"] for st in step_stats]

    # ---- timed: end to end through the public API with host buffers ----
    h2d = int(ps.ascii.size + ps.offsets.size * 8)
    d2h = int(n * (4 + 8) + 8 + 4 + 8 * 8)      # the winner's (float*int)[] + its sum, restart index, run counters

    def e2e_step(s_: int):
        eng.upload_flat(host_ascii.numpy(), host_off.numpy())      # H2D + GPU 2-bit pack
        eng.run_device(params, chains, chain_id_base=chain_base, seed=SEED + s_)   # the same restarts as the device-timed step s_
        return finish_step(eng)                                     # what fs:434 / fs:615 / fs:856 returns

    for w in range(args.warmup):            # untimed: first use allocates the page-locked result buffers
        e2e_step(-1 - w)
    barrier()
    e2e_windows = 0
    t0 = time.perf_counter()
    for s_ in range(args.steps):
        best = e2e_step(s_)
        e2e_windows += best.stats["window_scores"]
        launches_e2e = best.stats["kernel_launches"]
    barrier()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop(clk_first, clk_last) if sampler else None
    assert len(best.sites) in (1, n)

    # ---- reduce over ranks: totals summed, times max; per-rank figures kept for attribution ----
    k_ms = sum(kernel_ms) / len(kernel_ms)
    mine = [dev_ms / args.steps, k_ms, 1e3 * e2e_s / args.steps, statistics.median(win_ms), max(win_ms), min(win_ms)]
    if world > 1:
        t = torch.tensor([dev_ms, e2e_s, t_wall], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        c = torch.tensor([tot_windows, tot_updates, e2e_windows, tot_sweeps, tot_rescans], dtype=torch.float64, device="cuda")
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        per = torch.zeros(world, len(mine), dtype=torch.float64, device="cuda")
        dist.all_gather_into_tensor(per, torch.tensor(mine, dtype=torch.float64, device="cuda"))
        per = per.tolist()
        dev_ms_max, e2e_s, t_wall = (float(x) for x in t.tolist())
        g_windows, g_updates, g_e2e_windows, g_sweeps, g_rescans = (float(x) for x in c.tolist())
    else:
        per = [mine]
        dev_ms_max = dev_ms
        g_windows, g_updates, g_e2e_windows, g_sweeps, g_rescans = tot_windows, tot_updates, e2e_windows, tot_sweeps, tot_rescans

    # ---- the other reference families on the same set (N = 1, default workload only): short runs, reported beside the headline ----
    peaks = measured_peaks()
    smem_gbs = None
    families = None
    if rank == 0:
        smem_gbs, _ = measure_smem_bandwidth(local_rank, 20000)
    if world == 1 and args.family == "bpv" and not args.no_families:
        families = {}
        for fam in ("data", "motif", "motif-data"):
            prm = params_of(fam)
            eng.run_device(prm, chains, chain_id_base=chain_base, seed=SEED - 7)     # warm-up (tables, allocations)
            finish_step(eng)
            ms, sts, _ = timed_steps(eng, prm, args.steps, SEED + 50)
            w_ = sum(st["window_scores"] for st in sts)
            kms = sum(st["kernel_ms"] for st in sts) / len(sts)
            rate = w_ / (sum(ms) * 1e-3)
            families[fam] = {"what": FAMILIES[fam][0], "kernel": FAMILIES[fam][2], "value": rate, "unit": "window-scores/s",
                             "ms_per_step": sum(ms) / len(ms), "kernel_ms": kms, "steps": len(ms),
                             "frac": rate * algorithmic_smem_bytes_per_window(k) / 1e9 / smem_gbs,
                             "site_updates_per_sec": sum(st["site_updates"] for st in sts) / (sum(ms) * 1e-3),
                             "gpu_launches": sum(st["kernel_launches"] for st in sts)}

    if rank == 0:
        sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count
        smem_theory = sm_count * 128.0 * float(peaks.get("sm_max_mhz", 1965.0)) * 1e6 / 1e9
        rank_windows_per_s = (tot_windows / args.steps) / (k_ms * 1e-3)
        rank_updates_per_s = (tot_updates / args.steps) / (k_ms * 1e-3)
        achieved = rank_windows_per_s * algorithmic_smem_bytes_per_window(k) / 1e9
        hbm_achieved = rank_updates_per_s * algorithmic_hbm_bytes_per_site_update(length) / 1e9
        value = g_windows / (dev_ms_max * 1e-3)
        cpu = None
        if world == 1 and not args.no_cpu and fam_oracle is not None:
            dt = ws = us = 0.0
            n_cpu_chains = 0
            if cfg_name == "C1":    # the reference-scale case runs in full: the restart loop of fs:434 with numberOfRepetitions = chains - 1
                O = _oracle()
                rng, _ = O.make_rng(seed=SEED, chain=0)
                t0 = time.perf_counter()
                _, _, st1 = O.best_information_content(0 if args.family == "bpv" else 1, chains - 1, O.sources(ps.sequences()), k,
                                                       PSEUDOCOUNT, rng, pcv=O.pcv_from_acgt(bg) if args.family == "bpv" else None)
                dt, ws, us, n_cpu_chains = time.perf_counter() - t0, st1.window_scores, st1.site_updates, int(st1.restarts)
            while cfg_name != "C1" and dt < 12.0 and n_cpu_chains < 64:          # about 10-30 s of CPU work
                d1, w1, u1 = cpu_sample(ps, k, bg, threads=1, full_restart=True, seed=SEED, chain_base=n_cpu_chains,
                                        family=args.family)
                dt, ws, us, n_cpu_chains = dt + d1, ws + w1, us + u1, n_cpu_chains + 1
            us = int(us)
            cpu = {"value": ws / dt, "unit": "window-scores/s", "site_updates_per_sec": us / dt, "cores": 1,
                   "kind": "port", "seconds": dt,
                   "sample": (f"chains 0..{n_cpu_chains - 1} of the same workload, full {fam_oracle} restarts ({us} site updates) "
                              "on 1 host core; C port of the F# reference (oracle/), reference-faithful from-scratch rebuilds; "
                              "the F# itself needs .NET, absent from this image")}
        config = workload_config(cfg_name, cfg, args.family, chains)
        line = {
            "metric": "gibbs_window_scores_per_sec", "value": value, "unit": "window-scores/s",
            "site_updates_per_sec": g_updates / (dev_ms_max * 1e-3),
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic planted-motif DNA (Philox key 0xB200, 10% planted-base mutation)",
            "config": config,
            "measurement": {"l2": "flushed between steps (256 MiB write) outside the per-step CUDA-event window; the packed "
                                  "sequences (144 KB at C2) are L2/SMEM-resident by design",
                            "timing": "CUDA events on the launch stream around each step, summed; max over ranks",
                            "init_path": {1: "chain kernel", 2: "grid-wide kernel, global gathers", 3: "grid-wide kernel, set in shared memory",
                                          4: "grid-wide kernel, set streamed through shared memory in tiles"}.get(step_stats[-1]["init_path"]),
                            "clock_sampler": "one nvidia-smi process on rank 0 for all GPUs of the job"},
            "window_scores_per_step": g_windows / args.steps, "site_updates_per_step": g_updates / args.steps,
            "sweeps_per_chain": g_sweeps / (args.steps * chains * world), "exact_rescans_per_step": g_rescans / args.steps,
            "wall_s_timed_region": t_wall,
            "per_rank": {"fields": ["event_window_ms_per_step", "kernel_ms_per_step", "e2e_ms_per_step", "window_ms_median",
                                    "window_ms_max", "window_ms_min"], "ranks": per},
            "roofline": {"bound": "smem", "achieved": achieved, "peak": smem_gbs, "unit": "GB/s", "frac": achieved / smem_gbs,
                         "traffic": NCU_DRAM_BYTES_PER_STEP if (cfg_name == "C2" and args.family == "bpv") else None,
                         "traffic_source": NCU_DRAM_SOURCE,
                         "peak_source": "measured live: LDS.128 streaming microbenchmark (gibbs_measure_smem_bandwidth)",
                         "peak_theoretical": smem_theory, "frac_of_theoretical": achieved / smem_theory,
                         "algorithmic_bytes_per_window_score": algorithmic_smem_bytes_per_window(k),
                         "kernel": fam_kernel, "kernel_ms": k_ms,
                         "hbm": {"achieved": hbm_achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                 "frac": hbm_achieved / peaks["hbm_gbs"], "peak_source": peaks["_source"],
                                 "algorithmic_bytes_per_site_update": algorithmic_hbm_bytes_per_site_update(length)}},
            "cpu_baseline": cpu,
            "e2e": {"value": g_e2e_windows / e2e_s, "unit": "window-scores/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * e2e_s / args.steps,
                    "api": "gibbs_upload + gibbs_run_device + gibbs_fetch_best (C ABI): ASCII in, the restart loop's "
                           "(float*int)[] out; the fs:434 loop is decided on the device; wall clock over the same "
                           "restarts (seeds) as the device-timed steps, each step uploading from pinned host memory"},
            "families": families,
            "gpu_launches": launches, "gpu_launches_e2e_per_step": launches_e2e,
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--config", choices=sorted(CONFIGS), default="C2")
    ap.add_argument("--family", choices=sorted(FAMILIES), default="bpv",
                    help="reference family of the step; bpv = the BASELINE.json workload (the only one the driver runs)")
    ap.add_argument("--chains", type=int, default=0, help="override chains per GPU")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--opt", action="append", default=[], metavar="NAME=VALUE",
                    help="gibbs_set_option switch for A/B measurements, e.g. --opt coop=0 (include/gibbs_b200.h, GIBBS_OPT_*)")
    ap.add_argument("--no-families", action="store_true", help="skip the short runs of the other reference families")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last device-timed step computed to DIR/<name>.npy (float64), see last_step_outputs")
    args = ap.parse_args()
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference_arm(args, args.config, cfg)
    else:
        run_gpu_arm(args, args.config, cfg)


if __name__ == "__main__":
    main()
