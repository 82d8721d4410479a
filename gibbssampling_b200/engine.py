"""Host-side owner of one gibbs_handle: sequences resident in HBM + the CUDA entry points.

This is the Python twin of the F# shim (fsharp/GibbsSamplingB200.fs): it converts the reference's
argument shapes (BioArray[] of symbols, alphabet array, ProbabilityCompositeVector) into the flat
buffers of include/gibbs_b200.h and re-wraps the results. No arithmetic of the hot path happens
here; it all runs in libgibbs_b200.so on the GPU.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Iterable, Optional, Sequence

import numpy as np

from . import _abi
from ._abi import Params, RunStats

ACGT = "ACGT"


def _as_bytes(seq) -> bytes:
    """One BioArray: a str/bytes of symbols or an iterable of 1-char symbols / symbol codes."""
    if isinstance(seq, bytes):
        return seq
    if isinstance(seq, str):
        return seq.encode("ascii")
    if isinstance(seq, np.ndarray) and seq.dtype == np.uint8:
        return seq.tobytes()
    out = bytearray()
    for item in seq:
        out.append(symbol_code(item))
    return bytes(out)


def symbol_code(item) -> int:
    """BioItem.symbol (fs:17): the ASCII code of a symbol given as str, bytes, int or an object with .symbol."""
    if isinstance(item, (int, np.integer)):
        return int(item)
    if isinstance(item, str) and len(item) == 1:
        return ord(item)
    if isinstance(item, bytes) and len(item) == 1:
        return item[0]
    sym = getattr(item, "symbol", None)
    if sym is not None:
        return symbol_code(sym)
    raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, f"cannot interpret {item!r} as a sequence symbol")


def flatten_sources(sources: Sequence) -> tuple[np.ndarray, np.ndarray]:
    if sources is None:
        raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "sources is null (ArgumentNullException)")
    bs = [_as_bytes(s) for s in sources]
    off = np.zeros(len(bs) + 1, dtype=np.int64)
    if bs:
        off[1:] = np.cumsum([len(b) for b in bs])
    joined = b"".join(bs)
    buf = np.frombuffer(joined, dtype=np.uint8).copy() if joined else np.zeros(1, np.uint8)
    return buf, off


def _ptr(a: Optional[np.ndarray], t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


@dataclass
class BestResult:
    """What the reference's restart loops return (fs:434, fs:615, fs:856, fs:973): one (float*int)[] / MotifIndex[]."""
    sites: np.ndarray        # int32 [n] (or [1] when the loop's initial value survived)
    scores: np.ndarray       # float64, same length
    total: float             # Array.sum of the scores
    restart: int             # which restart it is, -1 = the initial value [|(0., 0)|]
    counts: Optional[np.ndarray]
    stats: dict


@dataclass
class RunResult:
    sites: np.ndarray        # int32 [chains, n]  (-1 = no site)
    scores: np.ndarray       # float64 [chains, n]
    sums: np.ndarray         # float64 [chains]
    best_chain: int
    counts: np.ndarray       # int32 [k, 4] PWM counts (A,C,G,T) of the best chain
    stats: dict


def make_params(k: int, pseudocount: float, alphabet_size: int, bg: Sequence[float], *, cutoff: float = 0.0,
                sampler: int = _abi.GIBBS_SITE_SAMPLER, phase_shifts: bool = True, max_sweeps: int = 0,
                phase_mask: int = 0, background: int = _abi.GIBBS_BG_FIXED, motif_amount: int = 1) -> Params:
    p = Params()
    p.k = int(k)
    p.alphabet_size = int(alphabet_size)
    p.pseudocount = float(pseudocount)
    for i in range(4):
        p.bg[i] = float(bg[i])
    p.cutoff = float(cutoff)
    p.sampler = int(sampler)
    p.phase_shifts = 1 if phase_shifts else 0
    p.max_sweeps = int(max_sweeps)
    p.phase_mask = int(phase_mask)
    p.background = int(background)
    p.motif_amount = int(motif_amount)
    return p


class GibbsEngine:
    """Sequences uploaded once, 2-bit packed on the GPU and kept resident in HBM."""

    def __init__(self, sources: Sequence, device: int = 0):
        self._lib = _abi.load()
        self._h = C.c_void_p()
        self._host: dict[str, tuple[int, int]] = {}   # pinned result buffers: name -> (address, bytes)
        buf, off = flatten_sources(sources)
        self.n = len(off) - 1
        self.lengths = np.diff(off).astype(np.int64)
        _abi.check(self._lib.gibbs_create(_ptr(buf, C.c_uint8), _ptr(off, C.c_int64), C.c_int32(self.n),
                                          C.c_int32(device), C.byref(self._h)))
        self.device = device

    # -- lifetime ---------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.gibbs_destroy(self._h)
            self._h = C.c_void_p()
        for ptr, _ in getattr(self, "_host", {}).values():
            self._lib.gibbs_host_free(C.c_void_p(ptr))
        self._host = {}

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def upload(self, sources: Sequence) -> None:
        buf, off = flatten_sources(sources)
        n = len(off) - 1
        _abi.check(self._lib.gibbs_upload(self._h, _ptr(buf, C.c_uint8), _ptr(off, C.c_int64), C.c_int32(n)))
        self.n = n
        self.lengths = np.diff(off).astype(np.int64)

    def upload_flat(self, buf: np.ndarray, off: np.ndarray) -> None:
        """Same as upload() for buffers that are already flat (pinned host memory in bench.py)."""
        n = len(off) - 1
        _abi.check(self._lib.gibbs_upload(self._h, _ptr(buf, C.c_uint8), _ptr(off, C.c_int64), C.c_int32(n)))
        self.n = n
        self.lengths = np.diff(off).astype(np.int64)

    def set_stream(self, cuda_stream: int) -> None:
        _abi.check(self._lib.gibbs_set_stream(self._h, C.c_void_p(cuda_stream)))

    def set_team_warps(self, warps: int) -> None:
        """Tuning knob: warps per chain (0 = automatic with hand-over stages; 1, 4, 8 or 16 = one launch of that size)."""
        _abi.check(self._lib.gibbs_set_team_warps(self._h, C.c_int32(warps)))

    def synchronize(self) -> None:
        _abi.check(self._lib.gibbs_synchronize(self._h))

    def set_option(self, option: int, value: int) -> None:
        """Explicit test / measurement switches (_abi.GIBBS_OPT_*); none changes a result."""
        _abi.check(self._lib.gibbs_set_option(self._h, C.c_int32(option), C.c_int32(value)))

    # -- primitives ---------------------------------------------------------------------------
    def _sites(self, sites) -> np.ndarray:
        a = np.ascontiguousarray(sites, dtype=np.int32)
        if a.shape != (self.n,):
            raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, f"sites must have {self.n} entries")
        return a

    def loo_counts(self, sites, heldout: int, k: int) -> np.ndarray:
        """Leave-one-out PWM counts [k,4] (A,C,G,T): getSegment |> createPFMOf |> fuse (fs:392-396)."""
        s = self._sites(sites)
        out = np.zeros((max(int(k), 1), 4), dtype=np.int32)
        _abi.check(self._lib.gibbs_loo_counts(self._h, _ptr(s, C.c_int32), C.c_int32(heldout), C.c_int32(k),
                                              _ptr(out, C.c_int32)))
        return out

    def window_scores(self, sites, heldout: int, params: Params) -> tuple[np.ndarray, np.ndarray]:
        """(raw float64 products, log2 scores) of every window of sources[heldout] (fs:301-314 loop body)."""
        s = self._sites(sites)
        if not (0 <= heldout < self.n):
            raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "heldout outside the sources")
        w = int(self.lengths[heldout]) - int(params.k) + 1
        raw = np.zeros(max(w, 1), dtype=np.float64)
        lg = np.zeros(max(w, 1), dtype=np.float64)
        _abi.check(self._lib.gibbs_window_scores(self._h, _ptr(s, C.c_int32), C.c_int32(heldout), C.byref(params),
                                                 _ptr(raw, C.c_double), _ptr(lg, C.c_double)))
        return raw[:w], lg[:w]

    def pick_argmax(self, sites, heldout: int, params: Params) -> tuple[float, int]:
        """getBestPWMSsWithBPV (fs:301-314): (log2 of the first strict maximum, its start position)."""
        s = self._sites(sites)
        score = C.c_double()
        site = C.c_int32()
        _abi.check(self._lib.gibbs_pick_argmax(self._h, _ptr(s, C.c_int32), C.c_int32(heldout), C.byref(params),
                                               C.byref(score), C.byref(site)))
        return score.value, site.value

    def pick_roulette(self, sites, heldout: int, params: Params, u: float) -> tuple[float, int]:
        """calculateNormalizedSegmentScores |> rouletteWheelSelection u (fs:759, fs:746), motifAmount = 1."""
        s = self._sites(sites)
        pwms = C.c_double()
        site = C.c_int32()
        _abi.check(self._lib.gibbs_pick_roulette(self._h, _ptr(s, C.c_int32), C.c_int32(heldout), C.byref(params),
                                                 C.c_double(u), C.byref(pwms), C.byref(site)))
        return pwms.value, site.value

    # -- chains ---------------------------------------------------------------------------------
    def run_device(self, params: Params, n_chains: int, *, chain_id_base: int = 0, seed: int = 0,
                   uniforms: Optional[np.ndarray] = None) -> None:
        """Launch n_chains restarts; results stay in HBM until fetch()."""
        if uniforms is not None:
            u = np.ascontiguousarray(uniforms, dtype=np.float64)
            if u.ndim == 1:
                u = u.reshape(1, -1)
            if u.shape[0] != n_chains:
                raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "uniforms must be [n_chains, draws]")
            _abi.check(self._lib.gibbs_run_device(self._h, C.byref(params), C.c_int32(n_chains),
                                                  C.c_int64(chain_id_base), C.c_uint64(seed),
                                                  C.c_int32(_abi.GIBBS_RNG_INJECTED), _ptr(u, C.c_double),
                                                  C.c_int64(u.shape[1])))
        else:
            _abi.check(self._lib.gibbs_run_device(self._h, C.byref(params), C.c_int32(n_chains),
                                                  C.c_int64(chain_id_base), C.c_uint64(seed),
                                                  C.c_int32(_abi.GIBBS_RNG_PHILOX), None, C.c_int64(0)))
        self._last = (int(n_chains), int(params.k))

    def set_start_ppm(self, ppm, k: Optional[int] = None) -> None:
        """`positionProbabilityMatrix` of the ...OfPPM / ...WithPPM functions (fs:644): the random starts of the
        following data-derived runs are scored against it. ppm = [k][4] (A,C,G,T per column) or the reference's
        [49][k] matrix (rows = symbol - 42); None clears it."""
        if ppm is None:
            _abi.check(self._lib.gibbs_set_start_ppm(self._h, None, C.c_int32(0)))
            return
        a = np.asarray(ppm, dtype=np.float64)
        if a.ndim == 2 and a.shape[0] == 49 and (k is None or a.shape[1] == k):
            a = a[[ord(c) - 42 for c in "ACGT"], :].T
        if a.ndim != 2 or a.shape[1] != 4 or (k is not None and a.shape[0] != k):
            raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "ppm must be [k][4] (A,C,G,T) or [49][k]")
        a = np.ascontiguousarray(a)
        _abi.check(self._lib.gibbs_set_start_ppm(self._h, _ptr(a, C.c_double), C.c_int32(a.shape[0])))

    def set_start_state(self, sites, scores) -> None:
        """startPositions : (float*int)[] of the sweep functions (fs:381 ...), per chain."""
        s = np.ascontiguousarray(sites, dtype=np.int32)
        v = np.ascontiguousarray(scores, dtype=np.float64)
        if s.ndim == 1:
            s, v = s.reshape(1, -1), v.reshape(1, -1)
        if s.shape != v.shape or s.shape[1] != self.n:
            raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "start state must be [n_chains, n_seqs]")
        _abi.check(self._lib.gibbs_set_start_state(self._h, C.c_int32(s.shape[0]), _ptr(s, C.c_int32),
                                                   _ptr(v, C.c_double)))

    def set_start_motif_state(self, positions, pwms) -> None:
        """motifMem : MotifIndex[] with up to m positions per sequence: positions [n_chains, n_seqs, m] (newest first,
        -1 = absent), pwms [n_chains, n_seqs]."""
        pos = np.ascontiguousarray(positions, dtype=np.int32)
        v = np.ascontiguousarray(pwms, dtype=np.float64)
        if pos.ndim == 2:
            pos, v = pos.reshape(1, *pos.shape), v.reshape(1, -1)
        if pos.ndim != 3 or pos.shape[:2] != v.shape or pos.shape[1] != self.n:
            raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "start state must be [n_chains, n_seqs, m]")
        _abi.check(self._lib.gibbs_set_start_motif_state(self._h, C.c_int32(pos.shape[0]), C.c_int32(pos.shape[2]),
                                                         _ptr(pos, C.c_int32), _ptr(v, C.c_double)))

    def fetch_positions(self, m: int) -> np.ndarray:
        """MotifIndex.Positions of every sequence of every chain of the last run: int32 [chains, n, m], newest first."""
        n_chains, _ = self._last
        out = np.zeros((n_chains, self.n, m), dtype=np.int32)
        _abi.check(self._lib.gibbs_fetch_positions(self._h, C.c_int32(m), _ptr(out, C.c_int32)))
        return out

    def fetch_best_positions(self, m: int) -> np.ndarray:
        """Positions lists of the array the last fetch_best returned: int32 [n, m]."""
        out = np.zeros((self.n, m), dtype=np.int32)
        _abi.check(self._lib.gibbs_fetch_best_positions(self._h, C.c_int32(m), _ptr(out, C.c_int32)))
        return out

    def _pinned(self, name: str, shape: tuple, dtype) -> np.ndarray:
        """Page-locked result buffer owned by this engine, grown on demand and reused by later fetches."""
        need = int(np.prod(shape)) * np.dtype(dtype).itemsize
        ptr, cap = self._host.get(name, (None, 0))
        if cap < need:
            if ptr:
                _abi.check(self._lib.gibbs_host_free(C.c_void_p(ptr)))
                self._host.pop(name)
            p = C.c_void_p()
            _abi.check(self._lib.gibbs_host_alloc(C.c_size_t(need), C.byref(p)))
            ptr, cap = p.value, need
            self._host[name] = (ptr, cap)
        buf = (C.c_uint8 * need).from_address(ptr)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def fetch(self, *, want_sites: bool = True, want_scores: bool = True, want_counts: bool = True,
              pinned: bool = False) -> RunResult:
        """Results of the last run_device. pinned=True returns views of page-locked buffers that the
        NEXT pinned fetch on this engine overwrites (and close() frees): copy what must outlive that."""
        n_chains, k = self._last
        if pinned:
            sites = self._pinned("sites", (n_chains, self.n), np.int32) if want_sites else None
            scores = self._pinned("scores", (n_chains, self.n), np.float64) if want_scores else None
            sums = self._pinned("sums", (n_chains,), np.float64)
        else:
            sites = np.zeros((n_chains, self.n), dtype=np.int32) if want_sites else None
            scores = np.zeros((n_chains, self.n), dtype=np.float64) if want_scores else None
            sums = np.zeros(n_chains, dtype=np.float64)
        counts = np.zeros((k, 4), dtype=np.int32) if want_counts else None
        best = C.c_int32()
        st = RunStats()
        _abi.check(self._lib.gibbs_fetch(self._h, _ptr(sites, C.c_int32), _ptr(scores, C.c_double),
                                         _ptr(sums, C.c_double), C.byref(best), _ptr(counts, C.c_int32),
                                         C.byref(st)))
        stats = {f: getattr(st, f) for f, _ in RunStats._fields_}
        return RunResult(sites, scores, sums, int(best.value), counts, stats)

    def fetch_best(self, repetitions: int, *, want_counts: bool = False, pinned: bool = False) -> BestResult:
        """The promote-or-restart loop of fs:435-459 over the restarts of the last run_device, decided on the GPU:
        only the winner's rows come back (gibbs_fetch_best)."""
        n_chains, k = self._last
        if pinned:
            sites = self._pinned("best_sites", (self.n,), np.int32)
            scores = self._pinned("best_scores", (self.n,), np.float64)
        else:
            sites = np.zeros(self.n, dtype=np.int32)
            scores = np.zeros(self.n, dtype=np.float64)
        counts = np.zeros((k, 4), dtype=np.int32) if want_counts else None
        n_out, restart, total, st = C.c_int32(), C.c_int32(), C.c_double(), RunStats()
        _abi.check(self._lib.gibbs_fetch_best(self._h, C.c_int32(repetitions), _ptr(sites, C.c_int32),
                                              _ptr(scores, C.c_double), C.byref(n_out), C.byref(total),
                                              C.byref(restart), _ptr(counts, C.c_int32), C.byref(st)))
        stats = {f: getattr(st, f) for f, _ in RunStats._fields_}
        return BestResult(sites[: n_out.value], scores[: n_out.value], total.value, int(restart.value), counts, stats)

    def run(self, params: Params, n_chains: int, *, chain_id_base: int = 0, seed: int = 0,
            uniforms: Optional[np.ndarray] = None, **fetch_kw) -> RunResult:
        self.run_device(params, n_chains, chain_id_base=chain_id_base, seed=seed, uniforms=uniforms)
        return self.fetch(**fetch_kw)

    def device_results(self) -> tuple[int, int, int]:
        """Device pointers (sites int32[chains,n], scores f64[chains,n], sums f64[chains]) of the last run."""
        a, b, c = C.c_void_p(), C.c_void_p(), C.c_void_p()
        _abi.check(self._lib.gibbs_device_results(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value


class MultiEngine:
    """One process, several GPUs (gibbs_multi_*): the sequences replicated on every device, the restarts of a run
    split into contiguous blocks over them. The F# shim uses the same calls for the restart loops."""

    def __init__(self, sources: Sequence, n_devices: int = 0, devices: Optional[Sequence[int]] = None):
        self._lib = _abi.load()
        self._m = C.c_void_p()
        buf, off = flatten_sources(sources)
        self.n = len(off) - 1
        dev = np.ascontiguousarray(devices, dtype=np.int32) if devices is not None else None
        if dev is not None:
            n_devices = len(dev)
        _abi.check(self._lib.gibbs_multi_create(_ptr(buf, C.c_uint8), _ptr(off, C.c_int64), C.c_int32(self.n),
                                                _ptr(dev, C.c_int32), C.c_int32(n_devices), C.byref(self._m)))
        self.n_devices = int(self._lib.gibbs_multi_num_devices(self._m))
        self._k = 0

    def close(self) -> None:
        if getattr(self, "_m", None) is not None and self._m.value:
            self._lib.gibbs_multi_destroy(self._m)
            self._m = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, option: int, value: int) -> None:
        for i in range(self.n_devices):
            h = self._lib.gibbs_multi_handle(self._m, C.c_int32(i))
            _abi.check(self._lib.gibbs_set_option(C.c_void_p(h), C.c_int32(option), C.c_int32(value)))

    def run_device(self, params: Params, n_chains: int, *, chain_id_base: int = 0, seed: int = 0,
                   uniforms: Optional[np.ndarray] = None) -> None:
        if uniforms is not None:
            u = np.ascontiguousarray(uniforms, dtype=np.float64).reshape(n_chains, -1)
            _abi.check(self._lib.gibbs_multi_run_device(self._m, C.byref(params), C.c_int32(n_chains), C.c_int64(chain_id_base),
                                                        C.c_uint64(seed), C.c_int32(_abi.GIBBS_RNG_INJECTED),
                                                        _ptr(u, C.c_double), C.c_int64(u.shape[1])))
        else:
            _abi.check(self._lib.gibbs_multi_run_device(self._m, C.byref(params), C.c_int32(n_chains), C.c_int64(chain_id_base),
                                                        C.c_uint64(seed), C.c_int32(_abi.GIBBS_RNG_PHILOX), None, C.c_int64(0)))
        self._k = int(params.k)

    def fetch_best(self, repetitions: int, *, want_counts: bool = False) -> BestResult:
        sites = np.zeros(self.n, dtype=np.int32)
        scores = np.zeros(self.n, dtype=np.float64)
        counts = np.zeros((self._k, 4), dtype=np.int32) if want_counts else None
        n_out, restart, total, st = C.c_int32(), C.c_int32(), C.c_double(), RunStats()
        _abi.check(self._lib.gibbs_multi_fetch_best(self._m, C.c_int32(repetitions), _ptr(sites, C.c_int32),
                                                    _ptr(scores, C.c_double), C.byref(n_out), C.byref(total),
                                                    C.byref(restart), _ptr(counts, C.c_int32), C.byref(st)))
        stats = {f: getattr(st, f) for f, _ in RunStats._fields_}
        return BestResult(sites[: n_out.value], scores[: n_out.value], total.value, int(restart.value), counts, stats)


def flatten_sets(sets: Sequence[Sequence]) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """S sets of sequences -> (symbols, int64 offsets[n_seqs + 1], int32 set_offsets[S + 1]) of gibbs_batch_create.
    Raises GibbsArgumentError for a null or empty list of sets and for an empty set."""
    if sets is None:
        raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "sets is null (ArgumentNullException)")
    sets = list(sets)
    if not sets:
        raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "a batch needs at least one set")
    set_off = np.zeros(len(sets) + 1, dtype=np.int32)
    flat = []
    for s, src in enumerate(sets):
        if src is None:
            raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, f"set {s} is null (ArgumentNullException)")
        src = list(src)
        if not src:
            raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, f"set {s} is empty")
        flat.extend(src)
        set_off[s + 1] = set_off[s] + len(src)
    buf, off = flatten_sources(flat)
    return buf, off, set_off


@dataclass
class BatchRunResult:
    """Every restart of every set: list entry s holds set s (sites / scores [R, N_s], sums [R])."""
    sites: list
    scores: list
    sums: list
    stats: dict


class BatchEngine:
    """Many independent sets of sequences (gibbs_batch_*): their restarts run together in a few launches; set s gives
    exactly what a GibbsEngine over sets[s] alone gives for the same parameters, seed and chain_id_base."""

    def __init__(self, sets: Sequence[Sequence], device: int = 0):
        self._lib = _abi.load()
        self._b = C.c_void_p()
        buf, off, set_off = flatten_sets(sets)
        self.n_sets = len(set_off) - 1
        self.set_offsets = set_off.astype(np.int64)
        self.sizes = np.diff(self.set_offsets)
        _abi.check(self._lib.gibbs_batch_create(_ptr(buf, C.c_uint8), _ptr(off, C.c_int64), _ptr(set_off, C.c_int32),
                                                C.c_int32(self.n_sets), C.c_int32(device), C.byref(self._b)))
        self.device = device
        self._last = None

    def close(self) -> None:
        if getattr(self, "_b", None) is not None and self._b.value:
            self._lib.gibbs_batch_destroy(self._b)
            self._b = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def run_device(self, params: Params, restarts_per_set: int, *, bg_per_set=None, chain_id_base: int = 0, seed: int = 0) -> None:
        """restarts_per_set restarts of every set; bg_per_set = [n_sets][4] backgrounds of the fixed-background family
        (None = params.bg for every set). Results stay in HBM until fetch() / fetch_best()."""
        bg = None
        if bg_per_set is not None:
            bg = np.ascontiguousarray(bg_per_set, dtype=np.float64)
            if bg.shape != (self.n_sets, 4):
                raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, f"bg_per_set must be [{self.n_sets}][4]")
        _abi.check(self._lib.gibbs_batch_run_device(self._b, C.byref(params), _ptr(bg, C.c_double), C.c_int32(restarts_per_set),
                                                    C.c_int64(chain_id_base), C.c_uint64(seed)))
        self._last = (int(restarts_per_set), int(params.k))

    def _need_run(self) -> tuple[int, int]:
        if self._last is None:
            raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "no run_device on this batch yet")
        return self._last

    def fetch(self) -> BatchRunResult:
        R, _ = self._need_run()
        total = int(self.set_offsets[-1])
        sites = np.zeros(R * total, dtype=np.int32)
        scores = np.zeros(R * total, dtype=np.float64)
        sums = np.zeros((self.n_sets, R), dtype=np.float64)
        st = RunStats()
        _abi.check(self._lib.gibbs_batch_fetch(self._b, _ptr(sites, C.c_int32), _ptr(scores, C.c_double), _ptr(sums, C.c_double),
                                               C.byref(st)))
        out_sites, out_scores = [], []
        for s in range(self.n_sets):
            a, n = R * int(self.set_offsets[s]), int(self.sizes[s])
            out_sites.append(sites[a: a + R * n].reshape(R, n))
            out_scores.append(scores[a: a + R * n].reshape(R, n))
        stats = {f: getattr(st, f) for f, _ in RunStats._fields_}
        return BatchRunResult(out_sites, out_scores, [sums[s] for s in range(self.n_sets)], stats)

    def fetch_best(self, repetitions: int, *, want_counts: bool = False) -> list[BestResult]:
        """The promote-or-restart loop of fs:435-459 of every set, decided on the GPU: one BestResult per set."""
        _, k = self._need_run()
        total = int(self.set_offsets[-1])
        sites = np.zeros(total, dtype=np.int32)
        scores = np.zeros(total, dtype=np.float64)
        n_out = np.zeros(self.n_sets, dtype=np.int32)
        sums = np.zeros(self.n_sets, dtype=np.float64)
        restart = np.zeros(self.n_sets, dtype=np.int32)
        counts = np.zeros((self.n_sets, k, 4), dtype=np.int32) if want_counts else None
        st = RunStats()
        _abi.check(self._lib.gibbs_batch_fetch_best(self._b, C.c_int32(repetitions), _ptr(sites, C.c_int32), _ptr(scores, C.c_double),
                                                    _ptr(n_out, C.c_int32), _ptr(sums, C.c_double), _ptr(restart, C.c_int32),
                                                    _ptr(counts, C.c_int32), C.byref(st)))
        stats = {f: getattr(st, f) for f, _ in RunStats._fields_}
        out = []
        for s in range(self.n_sets):
            a, n = int(self.set_offsets[s]), int(n_out[s])
            out.append(BestResult(sites[a: a + n].copy(), scores[a: a + n].copy(), float(sums[s]), int(restart[s]),
                                  counts[s] if counts is not None else None, stats))
        return out


def device_count() -> int:
    return int(_abi.load().gibbs_device_count())


def measure_smem_bandwidth(device: int = 0, iters: int = 20000) -> tuple[float, float]:
    g, ms = C.c_double(), C.c_double()
    _abi.check(_abi.load().gibbs_measure_smem_bandwidth(C.c_int32(device), C.c_int32(iters), C.byref(g), C.byref(ms)))
    return g.value, ms.value


def draws_per_chain(n_seqs: int, sampler: int = _abi.GIBBS_SITE_SAMPLER) -> int:
    """Uniform draws one restart consumes: N(N-1) initial sites (fs:595-598) + N roulette picks (fs:851)."""
    d = n_seqs * (n_seqs - 1)
    if sampler == _abi.GIBBS_MOTIF_SAMPLER:
        d += n_seqs
    return d
