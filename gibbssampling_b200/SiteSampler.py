"""SiteSampler -- the reference module's functions (fs:298-707) behind the CUDA library.

Same names, argument order and result shapes as /root/reference/GibbsSampling/GibbsSampling.fs:
every function returns `(float*int)[]` as a list of (log2 score, start position) tuples. The
keyword-only arguments are the documented ADDITIONS at the boundary (SURVEY.md section 0): the
reference seeds System.Random() from the clock, so reproducible runs need `seed` (Philox stream
`(seed, chain)`) or an injected stream of `uniforms`; `engine` lets callers keep the sequences
resident in HBM between calls.

All arithmetic runs in libgibbs_b200.so on the GPU. There is no CPU fallback.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np

from . import _abi
from .CompositeVector import ProbabilityCompositeVector
from .engine import BatchEngine, GibbsEngine, make_params, symbol_code

SiteArray = list  # (float*int)[]


def _bg_of(alphabet: Sequence, pcv: ProbabilityCompositeVector) -> list[float]:
    if alphabet is None or pcv is None:
        raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "alphabet / pcv is null (ArgumentNullException)")
    codes = {symbol_code(a) for a in alphabet}
    missing = [ch for ch in "ACGT" if ord(ch) not in codes]
    if missing:
        raise _abi.GibbsUnsupportedError(
            _abi.GIBBS_ERR_UNSUPPORTED,
            f"alphabet lacks {missing}: windows over those bases would score 0 (fs:283-287); "
            "the 2-bit GPU path needs A, C, G, T in the alphabet")
    extra = sorted(chr(c) for c in codes if chr(c) not in "ACGT-")
    if extra:   # the library takes a fifth alphabet member to be Gap (include/gibbs_b200.h, alphabet_size)
        raise _abi.GibbsUnsupportedError(
            _abi.GIBBS_ERR_UNSUPPORTED,
            f"alphabet members {extra} besides A, C, G, T and Gap would have PWM rows of their own (fs:283-287); not built")
    return [float(pcv[ch]) for ch in "ACGT"]


def _engine_for(sources, engine: Optional[GibbsEngine]) -> tuple[GibbsEngine, bool]:
    if engine is not None:
        return engine, False
    return GibbsEngine(sources), True


def _to_site_array(scores: np.ndarray, sites: np.ndarray) -> SiteArray:
    return [(float(s), int(p)) for s, p in zip(scores, sites)]


def _split_state(startPositions) -> tuple[np.ndarray, np.ndarray]:
    if startPositions is None:
        raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "startPositions is null (ArgumentNullException)")
    scores = np.array([float(s) for s, _ in startPositions], dtype=np.float64)
    sites = np.array([int(p) for _, p in startPositions], dtype=np.int32)
    return scores, sites


def _params(phase_mask: int, motifLength: int, pseudoCount: float, alphabet, pcv, max_sweeps: int = 0):
    """pcv given -> the WithBPV family (fixed background); pcv None -> the data-derived family (fs:462, fs:697)."""
    if pcv is None:
        _bg_of(alphabet, ProbabilityCompositeVector.ofACGT(1, 1, 1, 1))   # only checks that A,C,G,T are in the alphabet
        return make_params(motifLength, pseudoCount, len(alphabet), [0.25] * 4, phase_mask=phase_mask,
                           max_sweeps=max_sweeps, background=_abi.GIBBS_BG_DATA)
    return make_params(motifLength, pseudoCount, len(alphabet), _bg_of(alphabet, pcv), phase_mask=phase_mask,
                       max_sweeps=max_sweeps)


def _run_phases(phase_mask: int, motifLength: int, pseudoCount: float, alphabet, sources, pcv, *, start=None,
                seed: int = 0, chain: int = 0, uniforms=None, engine: Optional[GibbsEngine] = None,
                max_sweeps: int = 0, ppM=None) -> SiteArray:
    params = _params(phase_mask, motifLength, pseudoCount, alphabet, pcv, max_sweeps)
    eng, own = _engine_for(sources, engine)
    try:
        if start is not None:
            scores, sites = _split_state(start)
            eng.set_start_state(sites, scores)
        if ppM is not None:
            eng.set_start_ppm(ppM, motifLength)
        u = None if uniforms is None else np.asarray(uniforms, dtype=np.float64).reshape(1, -1)
        try:
            res = eng.run(params, 1, chain_id_base=chain, seed=seed, uniforms=u, want_counts=False)
        finally:
            if ppM is not None:
                eng.set_start_ppm(None)
        return _to_site_array(res.scores[0], res.sites[0])
    finally:
        if own:
            eng.close()


# ---------------------------------------------------------------------------------------------
# the reference's functions
# ---------------------------------------------------------------------------------------------
def bestPWMSOfHeldOutWithBPV(motifLength: int, pseudoCount: float, alphabet, sources, pcv, positions: Sequence[int],
                             heldOut: int, *, engine: Optional[GibbsEngine] = None) -> tuple[float, int]:
    """One site update: getBestPWMSsWithBPV (fs:301-314) applied to sources.[heldOut] with the leave-one-out PPM of
    `positions`, i.e. the body of the loop at fs:392-398.

    Not named after the reference function on purpose: getBestPWMSsWithBPV takes (motifLength, alphabet, source, pcv,
    positionProbabilityMatrix); at this boundary the PPM never leaves the GPU, so the caller passes what it is built
    from -- the other sequences' start positions -- and the argument list differs.
    """
    bg = _bg_of(alphabet, pcv)
    eng, own = _engine_for(sources, engine)
    try:
        return eng.pick_argmax(positions, heldOut, make_params(motifLength, pseudoCount, len(alphabet), bg))
    finally:
        if own:
            eng.close()


def getPWMOfRandomStartsWithBPV(motifLength, pseudoCount, alphabet, sources, pcv, **kw) -> SiteArray:
    """fs:412-430."""
    return _run_phases(_abi.PHASE_INIT, motifLength, pseudoCount, alphabet, sources, pcv, **kw)


def findBestMotifWithStartPosition(motifLength, pseudoCount, alphabet, sources, pcv, startPositions, **kw) -> SiteArray:
    """fs:381-408."""
    return _run_phases(_abi.PHASE_GREEDY, motifLength, pseudoCount, alphabet, sources, pcv, start=startPositions, **kw)


def getLeftShiftedBestPWMSsWithBPV(motifLength, pseudoCount, alphabet, sources, pcv, startPositions, **kw) -> SiteArray:
    """fs:350-377."""
    return _run_phases(_abi.PHASE_LEFT, motifLength, pseudoCount, alphabet, sources, pcv, start=startPositions, **kw)


def getRightShiftedBestPWMSsWithBPV(motifLength, pseudoCount, alphabet, sources, pcv, startPositions, **kw) -> SiteArray:
    """fs:318-346."""
    return _run_phases(_abi.PHASE_RIGHT, motifLength, pseudoCount, alphabet, sources, pcv, start=startPositions, **kw)


def doSiteSamplingWithBPV(motifLength, pseudoCount, alphabet, sources, pcv, **kw) -> SiteArray:
    """fs:691-695: random starts |> greedy sweeps |> left shifts |> right shifts."""
    mask = _abi.PHASE_INIT | _abi.PHASE_GREEDY | _abi.PHASE_LEFT | _abi.PHASE_RIGHT
    return _run_phases(mask, motifLength, pseudoCount, alphabet, sources, pcv, **kw)


def replay_restart_loop(numberOfRepetitions: int, restart_scores: np.ndarray, restart_sites: np.ndarray,
                        restart_sums: Optional[np.ndarray] = None) -> SiteArray:
    """The promote-or-restart loop of fs:435-459 (quirk A.6-8) over restarts that already ran -- the host-side model
    of what gibbs_fetch_best decides on the GPU (tests compare the two; multi-process runs use it on gathered results).

    The reference runs restarts one after another; here restart r is chain r of one kernel launch,
    and this function replays the loop's decisions over their results in the same order, so the
    returned array is the one the sequential loop would return. `restart_sums` = the left-to-right
    Array.sum of each restart's scores (computed on the GPU in that order); recomputed here if absent.
    State is kept as restart indices (None = [||], -1 = the initial [|(0., 0)|]).
    """
    if restart_sums is not None:
        sums = np.asarray(restart_sums, dtype=np.float64).tolist()
    else:
        sums = None

    def total(i) -> float:
        if i is None or i < 0:
            return 0.0
        if sums is not None:
            return sums[i]
        t = 0.0
        for v in restart_scores[i]:
            t = t + float(v)
        return t

    def same(a, b) -> bool:  # structural equality of two (float*int)[]
        if a is None or b is None:
            return a is None and b is None
        if a < 0 or b < 0:
            i = a if b < 0 else b
            if i < 0:
                return True
            return restart_scores.shape[1] == 1 and restart_scores[i][0] == 0.0 and restart_sites[i][0] == 0
        if sums is not None and sums[a] != sums[b]:
            return False   # equal score arrays have equal left-to-right sums (NaN sums are unequal either way)
        return bool(np.array_equal(restart_sites[a], restart_sites[b]) and
                    np.array_equal(restart_scores[a], restart_scores[b]))

    acc, best, r, n = None, -1, 0, 0
    while n <= numberOfRepetitions and not same(acc, best):
        if total(acc) > total(best):
            best = acc if acc is not None else best
            acc = None
        else:
            acc = r
            r += 1
        n += 1
    if best < 0:
        return [(0.0, 0)]
    return _to_site_array(restart_scores[best], restart_sites[best])


def _restart_loop(numberOfRepetitions, motifLength, pseudoCount, alphabet, sources, pcv, *, seed: int = 0, chain: int = 0,
                  uniforms=None, engine: Optional[GibbsEngine] = None, max_sweeps: int = 0, ppM=None) -> SiteArray:
    params = _params(0, motifLength, pseudoCount, alphabet, pcv, max_sweeps)
    eng, own = _engine_for(sources, engine)
    try:
        n_restarts = max(int(numberOfRepetitions) + 1, 1)
        u = None
        if uniforms is not None:
            u = np.asarray(uniforms, dtype=np.float64).reshape(n_restarts, -1)  # restart r consumes row r
        if ppM is not None:
            eng.set_start_ppm(ppM, motifLength)
        try:
            eng.run_device(params, n_restarts, chain_id_base=chain, seed=seed, uniforms=u)
        finally:
            if ppM is not None:
                eng.set_start_ppm(None)
        best = eng.fetch_best(int(numberOfRepetitions))   # the loop of fs:435-459 runs on the GPU; only the winner comes back
        return _to_site_array(best.scores, best.sites)
    finally:
        if own:
            eng.close()


def getMotifsWithBestInformationContentWithBPV(numberOfRepetitions, motifLength, pseudoCount, alphabet, sources, pcv,
                                               **kw) -> SiteArray:
    """fs:434-459. At most numberOfRepetitions + 1 restarts can run; they run as parallel chains."""
    if pcv is None:
        raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "pcv is null (ArgumentNullException)")
    return _restart_loop(numberOfRepetitions, motifLength, pseudoCount, alphabet, sources, pcv, **kw)


# ---- data-derived background (the background counts drift from window to window, fs:470-473) --------
def getPWMOfRandomStarts(motifLength, pseudoCount, alphabet, sources, **kw) -> SiteArray:
    """fs:589-611."""
    return _run_phases(_abi.PHASE_INIT, motifLength, pseudoCount, alphabet, sources, None, **kw)


def getBestPWMSsWithStartPositions(motifLength, pseudoCount, alphabet, sources, startPositions, **kw) -> SiteArray:
    """fs:554-585."""
    return _run_phases(_abi.PHASE_GREEDY, motifLength, pseudoCount, alphabet, sources, None, start=startPositions, **kw)


def getLeftShiftedBestPWMSs(motifLength, pseudoCount, alphabet, sources, startPositions, **kw) -> SiteArray:
    """fs:519-550."""
    return _run_phases(_abi.PHASE_LEFT, motifLength, pseudoCount, alphabet, sources, None, start=startPositions, **kw)


def getRightShiftedBestPWMSs(motifLength, pseudoCount, alphabet, sources, startPositions, **kw) -> SiteArray:
    """fs:483-515."""
    return _run_phases(_abi.PHASE_RIGHT, motifLength, pseudoCount, alphabet, sources, None, start=startPositions, **kw)


def doSiteSampling(motifLength, pseudoCount, alphabet, sources, **kw) -> SiteArray:
    """fs:697-701."""
    mask = _abi.PHASE_INIT | _abi.PHASE_GREEDY | _abi.PHASE_LEFT | _abi.PHASE_RIGHT
    return _run_phases(mask, motifLength, pseudoCount, alphabet, sources, None, **kw)


def getMotifsWithBestInformationContent(numberOfRepetitions, motifLength, pseudoCount, alphabet, sources, **kw) -> SiteArray:
    """fs:615-640 -- the call the reference script makes (fsx:384: reps 1, k 6, pc 1e-4, dnaBases)."""
    return _restart_loop(numberOfRepetitions, motifLength, pseudoCount, alphabet, sources, None, **kw)


# ---- start from a caller-supplied PositionProbabilityMatrix (fs:644-689, fs:703) --------------------------------
def getMotifsWithBestPWMSOfPPM(motifLength, pseudoCount, alphabet, sources, positionProbabilityMatrix, **kw) -> SiteArray:
    """fs:644-661: every sequence is scanned with the GIVEN PPM; the random sites of the other sequences only shape
    the drifting background. positionProbabilityMatrix: [49][k] like the reference's matrix, or [k][4] (A,C,G,T)."""
    if positionProbabilityMatrix is None:
        raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "positionProbabilityMatrix is null (ArgumentNullException)")
    return _run_phases(_abi.PHASE_INIT, motifLength, pseudoCount, alphabet, sources, None, ppM=positionProbabilityMatrix, **kw)


def doSiteSamplingWithPPM(motifLength, pseudoCount, alphabet, sources, ppM, **kw) -> SiteArray:
    """fs:703-707."""
    if ppM is None:
        raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "ppM is null (ArgumentNullException)")
    mask = _abi.PHASE_INIT | _abi.PHASE_GREEDY | _abi.PHASE_LEFT | _abi.PHASE_RIGHT
    return _run_phases(mask, motifLength, pseudoCount, alphabet, sources, None, ppM=ppM, **kw)


def getBestInformationContentOfPPM(numberOfRepetitions, motifLength, pseudoCount, alphabet, sources,
                                   positionProbabilityMatrix, **kw) -> SiteArray:
    """fs:664-689: the restart loop over doSiteSamplingWithPPM-shaped restarts."""
    if positionProbabilityMatrix is None:
        raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "positionProbabilityMatrix is null (ArgumentNullException)")
    return _restart_loop(numberOfRepetitions, motifLength, pseudoCount, alphabet, sources, None,
                         ppM=positionProbabilityMatrix, **kw)


# ---- many sets in one batch (gibbs_batch_*): one result per set, element s = the single-set function on sets[s] ------
# (engine=None: a BatchEngine on GPU 0; engine=MultiBatchEngine(sets, ...) spreads the sets over several GPUs)
def _restart_loop_of_sets(numberOfRepetitions, motifLength, pseudoCount, alphabet, sets, pcvs, *, seed: int = 0,
                          chain: int = 0, max_sweeps: int = 0, engine: Optional[BatchEngine] = None) -> list:
    if sets is not None:
        sets = list(sets)   # (a generator is read once)
    if pcvs is None:
        params = _params(0, motifLength, pseudoCount, alphabet, None, max_sweeps)
        bg = None
    else:
        pcvs = list(pcvs)
        if sets is not None and engine is None and len(pcvs) != len(sets):
            raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, f"{len(pcvs)} pcvs for {len(sets)} sets")
        bg = [_bg_of(alphabet, pcv) for pcv in pcvs]
        params = make_params(motifLength, pseudoCount, len(alphabet), bg[0] if bg else [0.25] * 4, max_sweeps=max_sweeps)
    eng = engine if engine is not None else BatchEngine(sets)
    try:
        eng.run_device(params, max(int(numberOfRepetitions) + 1, 1), bg_per_set=bg, chain_id_base=chain, seed=seed)
        return [_to_site_array(b.scores, b.sites) for b in eng.fetch_best(int(numberOfRepetitions))]
    finally:
        if engine is None:
            eng.close()


def getMotifsWithBestInformationContentWithBPVOfSets(numberOfRepetitions, motifLength, pseudoCount, alphabet, sets, pcvs,
                                                     **kw) -> list:
    """getMotifsWithBestInformationContentWithBPV (fs:434-459) of every set, pcvs[s] the background of sets[s]; the restarts
    of all sets run in one batch. Element s equals getMotifsWithBestInformationContentWithBPV(..., sets[s], pcvs[s]) with
    the same seed / chain."""
    if pcvs is None:
        raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "pcvs is null (ArgumentNullException)")
    return _restart_loop_of_sets(numberOfRepetitions, motifLength, pseudoCount, alphabet, sets, pcvs, **kw)


def getMotifsWithBestInformationContentOfSets(numberOfRepetitions, motifLength, pseudoCount, alphabet, sets, **kw) -> list:
    """getMotifsWithBestInformationContent (fs:615-640) of every set, in one batch; element s equals
    getMotifsWithBestInformationContent(..., sets[s]) with the same seed / chain."""
    return _restart_loop_of_sets(numberOfRepetitions, motifLength, pseudoCount, alphabet, sets, None, **kw)
