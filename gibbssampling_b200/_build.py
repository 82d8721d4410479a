"""Build recipe of libgibbs_b200.so (sm_100a only, in-tree so the .so travels with the repo).

The library is several translation units compiled in parallel and linked by nvcc:
  gibbs_api.cu        the extern "C" boundary, setup / primitive / init / MotifSampler kernels and
                      the winner-fetch kernels (gibbs_fetch.cuh, included by no other unit)
  gibbs_motif_tu.cu   the MotifSampler kernel, one team size per unit
  gibbs_motif2_tu.cu  the MotifSampler with motifAmount = 2
  gibbs_cluster_tu.cu one chain on a thread-block cluster of 4 / 8 CTAs (the last hand-over stages), one size per unit
  gibbs_init_tu.cu    the grid-wide random-start kernels, one kind per unit (same reason as the chain units)
  gibbs_batch_tu.cu   chain_batch_kernel (many sequence sets per launch), one group per unit like the chain units
  gibbs_motif_batch_tu.cu  the MotifSampler's batch kernels (motifAmount 1 and 2), one group per unit
  gibbs_chain_tu.cu   compiled once per GROUP of chain_kernel instantiations (warps per chain x masked symbols x
                      drifting background), without --split-compile: small modules give reproducible code for the
                      register-limited hot kernel (see the header of that file)
"""
from __future__ import annotations

import concurrent.futures
import os
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
OBJ_DIR = os.path.join(ROOT, "build", "obj")
LIB_PATH = os.path.join(PKG_DIR, "libgibbs_b200.so")
API_SOURCE = os.path.join(CSRC, "gibbs_api.cu")
CHAIN_SOURCE = os.path.join(CSRC, "gibbs_chain_tu.cu")
INIT_SOURCE = os.path.join(CSRC, "gibbs_init_tu.cu")
CLUSTER_SOURCE = os.path.join(CSRC, "gibbs_cluster_tu.cu")
MOTIF_SOURCE = os.path.join(CSRC, "gibbs_motif_tu.cu")
MOTIF2_SOURCE = os.path.join(CSRC, "gibbs_motif2_tu.cu")
BATCH_SOURCE = os.path.join(CSRC, "gibbs_batch_tu.cu")
MOTIF_BATCH_SOURCE = os.path.join(CSRC, "gibbs_motif_batch_tu.cu")
DEPS = [API_SOURCE, CHAIN_SOURCE, INIT_SOURCE, CLUSTER_SOURCE, MOTIF_SOURCE, MOTIF2_SOURCE, BATCH_SOURCE, MOTIF_BATCH_SOURCE] + [
    os.path.join(CSRC, f) for f in (
        "gibbs_device.cuh", "gibbs_kernels.cuh", "gibbs_motif.cuh", "gibbs_drift.cuh", "gibbs_drift_dev.cuh", "gibbs_cluster.cuh",
        "gibbs_motif2.cuh", "gibbs_batch.cuh", "gibbs_motif_batch.cuh", "gibbs_chain_body.inc", "gibbs_restart_select_body.inc",
        "gibbs_motif_body.inc", "gibbs_motif2_body.inc", "gibbs_fetch.cuh",
    )] + [os.path.join(ROOT, "include", "gibbs_b200.h"), os.path.abspath(__file__)]

# (entry point declared in gibbs_api.cu, warps per chain, masked symbols, drifting background)
CHAIN_GROUPS = [
    ("launch_chain_t4", 4, 0, 0),          # the benchmarked kernel
    ("launch_chain_drift_t4", 4, 0, 1),
    ("launch_chain_drift_t8", 8, 0, 1),
    ("launch_chain_t8", 8, 0, 0),
    ("launch_chain_t16", 16, 0, 0),
    ("launch_chain_t1", 1, 0, 0),
    ("launch_chain_drift_t1", 1, 0, 1),
    ("launch_chain_masked_t4", 4, 1, 0),
    ("launch_chain_masked_t1", 1, 1, 0),
    ("launch_chain_masked_drift_t4", 4, 1, 1),
    ("launch_chain_masked_drift_t1", 1, 1, 1),
]

# the random starts on the chain's own team (chain_kernel<.., INIT_ONLY = true>): 1 or 4 warps
CHAIN_INIT_GROUPS = [
    ("launch_chain_init_t4", 4, 0, 0), ("launch_chain_init_t1", 1, 0, 0),
    ("launch_chain_init_drift_t4", 4, 0, 1), ("launch_chain_init_drift_t1", 1, 0, 1),
    ("launch_chain_init_masked_t4", 4, 1, 0), ("launch_chain_init_masked_t1", 1, 1, 0),
    ("launch_chain_init_masked_drift_t4", 4, 1, 1), ("launch_chain_init_masked_drift_t1", 1, 1, 1),
]

# chain_batch_kernel (gibbs_batch_tu.cu): the sweeps and the random starts of every group a batch may launch -- 4 warps per
# chain for sets of >= 4 sequences, 1 warp for the rest, masked symbols, drifting background
BATCH_GROUPS = [
    (f"launch_batch{'_init' if init else ''}{'_masked' if masked else ''}{'_drift' if drift else ''}_t{team}", team, masked, drift, init)
    for init in (0, 1) for masked in (0, 1) for drift in (0, 1) for team in (4, 1)
]

# motif_batch_kernel / motif2_batch_kernel (gibbs_motif_batch_tu.cu): (entry point, motifAmount, warps per restart, masked
# symbols) -- motifAmount 1: 4 warps for sets of >= 4 sequences, 1 warp for the rest; motifAmount 2: one warp, A,C,G,T only
MOTIF_BATCH_GROUPS = [
    (f"launch_motif_batch{'_masked' if masked else ''}_t{team}", 1, team, masked) for masked in (0, 1) for team in (4, 1)
] + [("launch_motif2_batch", 2, 1, 0)]

COMMON_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-fmad=false",            # float64 products must round like the reference: no FMA contraction
    "-Xcompiler", "-fPIC",
    "-diag-suppress", "177",  # static kernels of the shared header that a given unit does not launch
    "-Xfatbin=-compress-all", # ~160 kernels with line info: 79 MB uncompressed, 23 MB compressed
]


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(p) > t for p in DEPS)


def _jobs(nvcc: str, verbose: bool) -> list[tuple[str, list[str]]]:
    extra = ["-Xptxas", "-v"] if verbose else []
    cores = os.cpu_count() or 1
    api_obj = os.path.join(OBJ_DIR, "gibbs_api.o")
    jobs = [(api_obj, [nvcc] + COMMON_FLAGS + extra + ["--split-compile", str(max(2, cores // 2)), "-c", "-o", api_obj,
                                                        API_SOURCE])]
    for name, team, masked, drift in CHAIN_GROUPS:
        obj = os.path.join(OBJ_DIR, name + ".o")
        jobs.append((obj, [nvcc] + COMMON_FLAGS + extra + [
            f"-DGIBBS_TU_NAME={name}", f"-DGIBBS_TU_T={team}", f"-DGIBBS_TU_MASKED={masked}", f"-DGIBBS_TU_DRIFT={drift}",
            "-c", "-o", obj, CHAIN_SOURCE]))
    for name, team, masked, drift in CHAIN_INIT_GROUPS:
        obj = os.path.join(OBJ_DIR, name + ".o")
        jobs.append((obj, [nvcc] + COMMON_FLAGS + extra + [
            f"-DGIBBS_TU_NAME={name}", f"-DGIBBS_TU_T={team}", f"-DGIBBS_TU_MASKED={masked}", f"-DGIBBS_TU_DRIFT={drift}",
            "-DGIBBS_TU_INIT_ONLY=1", "-c", "-o", obj, CHAIN_SOURCE]))
    for name, team, masked, drift, init in BATCH_GROUPS:
        obj = os.path.join(OBJ_DIR, name + ".o")
        jobs.append((obj, [nvcc] + COMMON_FLAGS + extra + [
            f"-DGIBBS_TU_NAME={name}", f"-DGIBBS_TU_T={team}", f"-DGIBBS_TU_MASKED={masked}", f"-DGIBBS_TU_DRIFT={drift}",
            f"-DGIBBS_TU_INIT_ONLY={init}", "-c", "-o", obj, BATCH_SOURCE]))
    for name, m, team, masked in MOTIF_BATCH_GROUPS:
        obj = os.path.join(OBJ_DIR, name + ".o")
        jobs.append((obj, [nvcc] + COMMON_FLAGS + extra + [
            f"-DGIBBS_TU_NAME={name}", f"-DGIBBS_TU_M={m}", f"-DGIBBS_TU_T={team}", f"-DGIBBS_TU_MASKED={masked}",
            "-c", "-o", obj, MOTIF_BATCH_SOURCE]))
    for kind, name in enumerate(("launch_init_wide", "launch_init_wide_drift", "launch_init_smem", "launch_init_tiled")):
        obj = os.path.join(OBJ_DIR, name + ".o")
        jobs.append((obj, [nvcc] + COMMON_FLAGS + extra + [f"-DGIBBS_INIT_TU_KIND={kind}", "-c", "-o", obj, INIT_SOURCE]))
    for t in (4, 1):
        obj = os.path.join(OBJ_DIR, f"launch_motif_t{t}.o")
        jobs.append((obj, [nvcc] + COMMON_FLAGS + extra + [f"-DGIBBS_MOTIF_TU_T={t}", "-c", "-o", obj, MOTIF_SOURCE]))
        obj = os.path.join(OBJ_DIR, f"launch_motif_masked_t{t}.o")   # sets with symbols outside A,C,G,T
        jobs.append((obj, [nvcc] + COMMON_FLAGS + extra + [f"-DGIBBS_MOTIF_TU_T={t}", "-DGIBBS_MOTIF_TU_MASKED=1", "-c", "-o", obj,
                                                            MOTIF_SOURCE]))
    for t in (8, 16):   # the hand-over stages of the MotifSampler (A,C,G,T-only sets)
        obj = os.path.join(OBJ_DIR, f"launch_motif_t{t}.o")
        jobs.append((obj, [nvcc] + COMMON_FLAGS + extra + [f"-DGIBBS_MOTIF_TU_T={t}", "-c", "-o", obj, MOTIF_SOURCE]))
    obj = os.path.join(OBJ_DIR, "launch_motif2.o")
    jobs.append((obj, [nvcc] + COMMON_FLAGS + extra + ["-c", "-o", obj, MOTIF2_SOURCE]))
    for c in (4, 8):
        obj = os.path.join(OBJ_DIR, f"launch_chain_cluster{c}.o")
        jobs.append((obj, [nvcc] + COMMON_FLAGS + extra + [f"-DGIBBS_CLUSTER_C={c}", "-c", "-o", obj, CLUSTER_SOURCE]))
    return jobs


def build(force: bool = False, verbose: bool = False, out: str | None = None, extra_flags: list[str] | None = None,
          only: list[str] | None = None) -> str:
    """Compile the CUDA library with nvcc (cross-compiles without a GPU).
    out / extra_flags: a variant build (tools/build_variant.sh) beside the in-tree library, e.g. other -D tuning macros.
    only: unit names (object basenames, e.g. launch_chain_t4) the flags apply to; the other units are linked from the
    in-tree build as they are (a variant that touches one kernel group compiles one unit)."""
    if out is None and not force and not is_stale():
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    obj_dir = OBJ_DIR if out is None else OBJ_DIR + "_" + os.path.splitext(os.path.basename(out))[0]
    os.makedirs(obj_dir, exist_ok=True)
    jobs = _jobs(nvcc, verbose)
    reused = []
    if out is not None or extra_flags:
        if only:
            reused = [o for o, _ in jobs if os.path.splitext(os.path.basename(o))[0] not in only]
            jobs = [(o, cmd) for o, cmd in jobs if os.path.splitext(os.path.basename(o))[0] in only]
        jobs = [(o.replace(OBJ_DIR, obj_dir, 1), [c.replace(OBJ_DIR, obj_dir, 1) for c in cmd[:1] + list(extra_flags or []) + cmd[1:]])
                for o, cmd in jobs]

    def run(job):
        return job, subprocess.run(job[1], capture_output=True, text=True)

    log = []
    with concurrent.futures.ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as pool:
        for job, res in pool.map(run, jobs):
            if res.returncode != 0:
                raise RuntimeError("nvcc failed: " + " ".join(job[1]) + "\n" + res.stdout + res.stderr)
            log.append(res.stderr)
    target = LIB_PATH if out is None else out
    link = [nvcc, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a", "-o", target]
    res = subprocess.run(link + [j[0] for j in jobs] + reused, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc link failed:\n" + res.stdout + res.stderr)
    if verbose:
        print("\n".join(log))
    return target


if __name__ == "__main__":
    print(build(force=True, verbose=True))
