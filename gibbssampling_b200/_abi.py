"""ctypes binding of libgibbs_b200.so -- the same symbols the F# shim binds with P/Invoke.

There is no CPU fallback: if the CUDA library is missing this module raises at load time, and
every compute call fails with GibbsCudaError when no B200/CUDA device is usable.
"""
from __future__ import annotations

import ctypes as C
import os

from . import _build

GIBBS_OK = 0
GIBBS_ERR_ARG = 1
GIBBS_ERR_SYMBOL = 2
GIBBS_ERR_SHORT_SEQ = 3
GIBBS_ERR_CUDA = 4
GIBBS_ERR_NCCL = 5
GIBBS_ERR_NOMEM = 6
GIBBS_ERR_ROULETTE = 7
GIBBS_ERR_UNSUPPORTED = 8

GIBBS_SITE_SAMPLER = 0
GIBBS_MOTIF_SAMPLER = 1
GIBBS_RNG_PHILOX = 0
GIBBS_RNG_INJECTED = 1
GIBBS_BG_FIXED = 0
GIBBS_BG_DATA = 1
GIBBS_MAX_K = 32
PHASE_INIT, PHASE_GREEDY, PHASE_LEFT, PHASE_RIGHT, PHASE_STOCHASTIC, PHASE_MOTIF_GREEDY = 1, 2, 4, 8, 16, 32

# every symbol include/gibbs_b200.h declares (tests check that the library exports all of them)
EXPORTS = [
    "gibbs_abi_version", "gibbs_last_error", "gibbs_device_count", "gibbs_create", "gibbs_upload",
    "gibbs_destroy", "gibbs_set_stream", "gibbs_num_sequences", "gibbs_set_team_warps", "gibbs_synchronize",
    "gibbs_loo_counts", "gibbs_window_scores", "gibbs_pick_argmax", "gibbs_pick_roulette",
    "gibbs_set_start_ppm", "gibbs_set_start_state", "gibbs_run_device", "gibbs_fetch", "gibbs_run", "gibbs_device_results",
    "gibbs_host_alloc", "gibbs_host_free", "gibbs_measure_smem_bandwidth",
    "gibbs_set_option", "gibbs_fetch_best", "gibbs_fetch_positions", "gibbs_fetch_best_positions",
    "gibbs_set_start_motif_state",
    "gibbs_multi_create", "gibbs_multi_destroy", "gibbs_multi_num_devices", "gibbs_multi_handle",
    "gibbs_multi_run_device", "gibbs_multi_fetch_best",
    "gibbs_batch_create", "gibbs_batch_destroy", "gibbs_batch_run_device", "gibbs_batch_fetch", "gibbs_batch_fetch_best",
]
GIBBS_OPT_INIT_PATH, GIBBS_OPT_EXACT_SCANS, GIBBS_OPT_STAGE2_AT, GIBBS_OPT_STAGE3_AT, GIBBS_OPT_CLUSTER, GIBBS_OPT_MIN_WIDTH = 1, 2, 3, 4, 5, 6
GIBBS_OPT_TILE_ROWS = 7
GIBBS_OPT_SEQ_SWEEPS = 8
GIBBS_INIT_AUTO, GIBBS_INIT_CHAIN, GIBBS_INIT_WIDE, GIBBS_INIT_SMEM, GIBBS_INIT_TILED = 0, 1, 2, 3, 4


class GibbsError(RuntimeError):
    """Base class; .code is the gibbs_status."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"[gibbs_status {code}] {msg}")
        self.code = code


class GibbsArgumentError(GibbsError, ValueError):
    """ArgumentNullException / ArgumentException of the reference (fs:24, fs:183)."""


class GibbsSymbolError(GibbsError, IndexError):
    """IndexOutOfRangeException analogue: a symbol the 2-bit tables cannot index (fs:17)."""


class GibbsShortSequenceError(GibbsError, ValueError):
    """InvalidOperationException from Array.take when a sequence is shorter than k (fs:152)."""


class GibbsCudaError(GibbsError):
    """CUDA failure or no device: there is no CPU fallback."""


class GibbsRouletteError(GibbsError, ValueError):
    """ArgumentException of fs:753 (pick beyond the accumulated mass)."""


class GibbsUnsupportedError(GibbsError, NotImplementedError):
    """A reference mode outside the built hot path."""


_ERRORS = {
    GIBBS_ERR_ARG: GibbsArgumentError,
    GIBBS_ERR_SYMBOL: GibbsSymbolError,
    GIBBS_ERR_SHORT_SEQ: GibbsShortSequenceError,
    GIBBS_ERR_CUDA: GibbsCudaError,
    GIBBS_ERR_NOMEM: GibbsCudaError,
    GIBBS_ERR_ROULETTE: GibbsRouletteError,
    GIBBS_ERR_UNSUPPORTED: GibbsUnsupportedError,
}


class Params(C.Structure):
    _fields_ = [
        ("k", C.c_int32),
        ("alphabet_size", C.c_int32),
        ("pseudocount", C.c_double),
        ("bg", C.c_double * 4),
        ("cutoff", C.c_double),
        ("sampler", C.c_int32),
        ("phase_shifts", C.c_int32),
        ("max_sweeps", C.c_int32),
        ("phase_mask", C.c_int32),
        ("background", C.c_int32),
        ("motif_amount", C.c_int32),
    ]


class RunStats(C.Structure):
    _fields_ = [
        ("site_updates", C.c_int64),
        ("window_scores", C.c_int64),
        ("sweeps", C.c_int64),
        ("exact_rescans", C.c_int64),
        ("capped_chains", C.c_int64),
        ("speculative_discards", C.c_int64),
        ("kernel_launches", C.c_int32),
        ("fast_path", C.c_int32),
        ("team_warps", C.c_int32),
        ("init_path", C.c_int32),
        ("kernel_ms", C.c_double),
    ]


_lib = None


def library_path() -> str:
    """GIBBS_B200_LIB selects another build of the same library (used to compare kernel variants)."""
    return os.environ.get("GIBBS_B200_LIB") or _build.LIB_PATH


def load() -> C.CDLL:
    """Load the CUDA library; raise loudly if it was never built (no fallback of any kind)."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is missing: build it with `python -m gibbssampling_b200._build` "
            "(nvcc, sm_100a). gibbssampling_b200 has no CPU fallback."
        )
    lib = C.CDLL(path)
    vp, i32, i64, u64, f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_double
    P = C.POINTER
    lib.gibbs_abi_version.restype = i32
    lib.gibbs_last_error.restype = C.c_char_p
    lib.gibbs_device_count.restype = i32
    lib.gibbs_create.argtypes = [P(C.c_uint8), P(i64), i32, i32, P(vp)]
    lib.gibbs_upload.argtypes = [vp, P(C.c_uint8), P(i64), i32]
    lib.gibbs_destroy.argtypes = [vp]
    lib.gibbs_set_stream.argtypes = [vp, vp]
    lib.gibbs_num_sequences.argtypes = [vp]
    lib.gibbs_synchronize.argtypes = [vp]
    lib.gibbs_set_team_warps.argtypes = [vp, i32]
    lib.gibbs_loo_counts.argtypes = [vp, P(i32), i32, i32, P(i32)]
    lib.gibbs_window_scores.argtypes = [vp, P(i32), i32, P(Params), P(f64), P(f64)]
    lib.gibbs_pick_argmax.argtypes = [vp, P(i32), i32, P(Params), P(f64), P(i32)]
    lib.gibbs_pick_roulette.argtypes = [vp, P(i32), i32, P(Params), f64, P(f64), P(i32)]
    lib.gibbs_set_start_state.argtypes = [vp, i32, P(i32), P(f64)]
    lib.gibbs_run_device.argtypes = [vp, P(Params), i32, i64, u64, i32, P(f64), i64]
    lib.gibbs_fetch.argtypes = [vp, P(i32), P(f64), P(f64), P(i32), P(i32), P(RunStats)]
    lib.gibbs_run.argtypes = [vp, P(Params), i32, i64, u64, i32, P(f64), i64, P(i32), P(f64), P(f64), P(i32),
                              P(i32), P(RunStats)]
    lib.gibbs_device_results.argtypes = [vp, P(vp), P(vp), P(vp)]
    lib.gibbs_measure_smem_bandwidth.argtypes = [i32, i32, P(f64), P(f64)]
    lib.gibbs_set_option.argtypes = [vp, i32, i32]
    lib.gibbs_fetch_best.argtypes = [vp, i32, P(i32), P(f64), P(i32), P(f64), P(i32), P(i32), P(RunStats)]
    lib.gibbs_fetch_positions.argtypes = [vp, i32, P(i32)]
    lib.gibbs_fetch_best_positions.argtypes = [vp, i32, P(i32)]
    lib.gibbs_set_start_motif_state.argtypes = [vp, i32, i32, P(i32), P(f64)]
    lib.gibbs_multi_create.argtypes = [P(C.c_uint8), P(i64), i32, P(i32), i32, P(vp)]
    lib.gibbs_multi_destroy.argtypes = [vp]
    lib.gibbs_multi_num_devices.argtypes = [vp]
    lib.gibbs_multi_handle.argtypes = [vp, i32]
    lib.gibbs_multi_run_device.argtypes = [vp, P(Params), i32, i64, u64, i32, P(f64), i64]
    lib.gibbs_multi_fetch_best.argtypes = [vp, i32, P(i32), P(f64), P(i32), P(f64), P(i32), P(i32), P(RunStats)]
    lib.gibbs_batch_create.argtypes = [P(C.c_uint8), P(i64), P(i32), i32, i32, P(vp)]
    lib.gibbs_batch_destroy.argtypes = [vp]
    lib.gibbs_batch_run_device.argtypes = [vp, P(Params), P(f64), i32, i64, u64]
    lib.gibbs_batch_fetch.argtypes = [vp, P(i32), P(f64), P(f64), P(RunStats)]
    lib.gibbs_batch_fetch_best.argtypes = [vp, i32, P(i32), P(f64), P(i32), P(f64), P(i32), P(i32), P(RunStats)]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name not in ("gibbs_last_error", "gibbs_multi_handle"):
            fn.restype = i32
    lib.gibbs_multi_handle.restype = vp
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc == GIBBS_OK:
        return
    msg = load().gibbs_last_error().decode(errors="replace")
    raise _ERRORS.get(rc, GibbsError)(rc, msg)
