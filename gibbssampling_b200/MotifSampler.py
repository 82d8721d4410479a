"""MotifSampler -- the reference module's functions (fs:709-1038) behind the CUDA library.

`MotifIndex` = {PWMS: float; Positions: int list} (fs:712-716). motifAmount = 1 (one site per sequence or none) and
motifAmount = 2 (up to two non-overlapping sites, fs:727-742 -- the reference script's second live call, fsx:407) are
built; three and more sites per sequence raise GibbsUnsupportedError. Both the fixed-background (`...ByPCV` /
`...WithPCV`) family and the data-derived-background family (fs:885-1038) run on the GPU. The `...OfSets` functions run
the restart loops of many sets in one batch (gibbs_batch_run_motif_device); by default on one GPU, on several with
engine=MultiBatchEngine(sets, ...).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Optional

import numpy as np

from . import _abi
from .CompositeVector import ProbabilityCompositeVector
from .engine import BatchEngine, GibbsEngine, make_params
from .SiteSampler import _bg_of, _engine_for


@dataclass(frozen=True)
class MotifIndex:
    PWMS: float
    Positions: tuple = field(default_factory=tuple)


def createMotifIndex(pwms: float, pos) -> MotifIndex:
    """fs:719-723."""
    return MotifIndex(float(pwms), tuple(int(p) for p in pos))


def _check_m(motifAmount: int) -> int:
    m = int(motifAmount)
    if m not in (1, 2):
        raise _abi.GibbsUnsupportedError(
            _abi.GIBBS_ERR_UNSUPPORTED,
            f"motifAmount = {motifAmount}: one and two sites per sequence are built "
            "(calculatePWMsForSegmentCombinations, fs:727-742); three and more are not")
    return m


def _to_motif_array(scores: np.ndarray, sites: np.ndarray) -> list:
    """scores [n]; sites [n] (one position, -1 = none) or [n, m] Positions lists (newest first, -1 = absent)."""
    sites = np.asarray(sites)
    if sites.ndim == 1:
        return [MotifIndex(float(s), (int(p),) if p >= 0 else ()) for s, p in zip(scores, sites)]
    return [MotifIndex(float(s), tuple(int(p) for p in row if p >= 0)) for s, row in zip(scores, sites)]


def _split_motif_state(motifMem, m: int = 1) -> tuple[np.ndarray, np.ndarray]:
    """(PWMS [n], Positions [n, m] newest first / -1 = absent)"""
    if motifMem is None:
        raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "motifMem is null (ArgumentNullException)")
    scores = np.array([float(x.PWMS) for x in motifMem], dtype=np.float64)
    pos = np.full((len(motifMem), m), -1, dtype=np.int32)
    for i, x in enumerate(motifMem):
        if len(x.Positions) > m:
            raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, f"a MotifIndex holds {len(x.Positions)} positions, motifAmount = {m}")
        pos[i, :len(x.Positions)] = x.Positions
    return scores, pos


def _run(phase_mask: int, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, pcv, *, start=None,
         n_chains: int = 1, seed: int = 0, chain: int = 0, uniforms=None, engine: Optional[GibbsEngine] = None,
         max_sweeps: int = 0, ppM=None, best_of: Optional[int] = None) -> list:
    """pcv given -> the PCV family (fixed background); pcv None -> the data-derived family (fs:885-1038).
    Returns the MotifIndex[] of chain 0, or of the restart loop's winner when best_of (numberOfRepetitions) is given."""
    m = _check_m(motifAmount)
    if pcv is None:
        _bg_of(alphabet, ProbabilityCompositeVector.ofACGT(1, 1, 1, 1))   # only checks A,C,G,T are in the alphabet
        bg, background = [0.25] * 4, _abi.GIBBS_BG_DATA
    else:
        bg, background = _bg_of(alphabet, pcv), _abi.GIBBS_BG_FIXED
    eng, own = _engine_for(sources, engine)
    try:
        params = make_params(motifLength, pseudoCount, len(alphabet), bg, cutoff=cutOff, background=background,
                             sampler=_abi.GIBBS_MOTIF_SAMPLER, phase_mask=phase_mask, max_sweeps=max_sweeps, motif_amount=m)
        if start is not None:
            scores, pos = _split_motif_state(start, m)
            eng.set_start_motif_state(np.tile(pos, (n_chains, 1, 1)), np.tile(scores, (n_chains, 1)))
        u = None if uniforms is None else np.asarray(uniforms, dtype=np.float64).reshape(n_chains, -1)
        if ppM is not None:
            eng.set_start_ppm(ppM, motifLength)
        try:
            eng.run_device(params, n_chains, chain_id_base=chain, seed=seed, uniforms=u)
            if best_of is None:
                res = eng.fetch(want_counts=False)
                return _to_motif_array(res.scores[0], res.sites[0] if m == 1 else eng.fetch_positions(m)[0])
            best = eng.fetch_best(best_of)   # the restart loop (fs:857-881) runs on the GPU; only the winner comes back
            if m == 1 or best.restart < 0:
                return _to_motif_array(best.scores, best.sites)
            return _to_motif_array(best.scores, eng.fetch_best_positions(m))
        finally:
            if ppM is not None:
                eng.set_start_ppm(None)
    finally:
        if own:
            eng.close()


def rouletteWheelSelectionOfSites(motifLength, pseudoCount, cutOff, alphabet, sources, pcv, positions, heldOut: int,
                                  pick: float, *, engine: Optional[GibbsEngine] = None) -> MotifIndex:
    """calculateNormalizedSegmentScores (motifAmount 1) |> rouletteWheelSelection pick (fs:759-784, fs:746-754)
    for sources.[heldOut], with the leave-one-out PWM of `positions` (-1 = no site)."""
    bg = _bg_of(alphabet, pcv)
    eng, own = _engine_for(sources, engine)
    try:
        params = make_params(motifLength, pseudoCount, len(alphabet), bg, cutoff=cutOff, sampler=_abi.GIBBS_MOTIF_SAMPLER)
        pwms, site = eng.pick_roulette(positions, heldOut, params, pick)
        return MotifIndex(pwms, (site,) if site >= 0 else ())
    finally:
        if own:
            eng.close()


def findBestMotifPositionsWithStartPositionsByPCV(motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, pcv,
                                                  motifMem, **kw) -> list:
    """fs:828-853: the synchronous stochastic sweep (one roulette pick per sequence)."""
    return _run(_abi.PHASE_STOCHASTIC, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, pcv,
                start=motifMem, **kw)


def findBestMotifPositionsWithStartPositionByPCV(motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, pcv,
                                                 motifMem, **kw) -> list:
    """fs:788-822: greedy in-place sweeps until the positions stop changing."""
    return _run(_abi.PHASE_MOTIF_GREEDY, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, pcv,
                start=motifMem, **kw)


def doMotifSamplingWithPCV(motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, pcv, **kw) -> list:
    """One restart of fs:876-879: random starts |> stochastic sweep |> greedy sweeps (the reference inlines
    this pipeline in findBestInormationContentContainingMotifsWithPCV; there is no separate `do` function)."""
    return _run(0, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, pcv, **kw)


def replay_motif_restart_loop(numberOfRepetitions: int, scores: np.ndarray, sites: np.ndarray, sums: np.ndarray) -> list:
    """fs:857-881 over restarts that already ran (same loop as SiteSampler.replay_restart_loop, over MotifIndex[])."""
    sums = np.asarray(sums, dtype=np.float64).tolist()

    def total(i):
        return 0.0 if (i is None or i < 0) else sums[i]

    def same(a, b):
        if a is None or b is None:
            return a is None and b is None
        if a < 0 or b < 0:
            i = a if b < 0 else b
            if i < 0:
                return True
            return scores.shape[1] == 1 and scores[i][0] == 0.0 and sites[i][0] < 0   # [|{PWMS 0.; Positions []}|]
        if sums[a] != sums[b]:
            return False   # equal MotifIndex arrays have equal left-to-right sums
        return bool(np.array_equal(sites[a], sites[b]) and np.array_equal(scores[a], scores[b]))

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
        return [MotifIndex(0.0, ())]
    return _to_motif_array(scores[best], sites[best])


def findBestInormationContentContainingMotifsWithPCV(numberOfRepetitions, motifAmount, motifLength, pseudoCount, cutOff,
                                                     alphabet, sources, pcv, *, seed: int = 0, chain: int = 0,
                                                     uniforms=None, engine: Optional[GibbsEngine] = None,
                                                     max_sweeps: int = 0) -> list:
    """fs:856-881: restarts run as parallel chains, the promote-or-restart loop is replayed over their results."""
    n_restarts = max(int(numberOfRepetitions) + 1, 1)
    return _run(0, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, pcv, n_chains=n_restarts,
               seed=seed, chain=chain, uniforms=uniforms, engine=engine, max_sweeps=max_sweeps,
               best_of=int(numberOfRepetitions))


# ---- data-derived background (fs:885-1038): one background per held-out sequence (fs:896-905) -------------
def findBestMotifIndicesByWithStartPositions(motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, motifMem,
                                             **kw) -> list:
    """fs:935-970: the synchronous stochastic sweep."""
    return _run(_abi.PHASE_STOCHASTIC, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, None,
                start=motifMem, **kw)


def findBestMotifIndicesWithStartPositions(motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, motifMem,
                                           **kw) -> list:
    """fs:885-929: greedy in-place sweeps."""
    return _run(_abi.PHASE_MOTIF_GREEDY, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, None,
                start=motifMem, **kw)


def doMotifSampling(motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, **kw) -> list:
    """fs:1034-1038."""
    return _run(0, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, None, **kw)


def getMotifsWithBestInformationContents(numberOfRepetitions, motifAmount, motifLength, pseudoCount, cutOff, alphabet,
                                         sources, *, seed: int = 0, chain: int = 0, uniforms=None,
                                         engine: Optional[GibbsEngine] = None, max_sweeps: int = 0) -> list:
    """fs:973-998 -- the reference script's second live call (fsx:407: reps 1, motifAmount 2, k 6, pc 1e-4, cutOff 1.0)."""
    n_restarts = max(int(numberOfRepetitions) + 1, 1)
    return _run(0, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, None, n_chains=n_restarts,
               seed=seed, chain=chain, uniforms=uniforms, engine=engine, max_sweeps=max_sweeps,
               best_of=int(numberOfRepetitions))


def doMotifSamplingWithPPM(motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, ppM, **kw) -> list:
    """fs:1028-1032: SiteSampler.getMotifsWithBestPWMSOfPPM as the start, then the data-derived sweeps."""
    if ppM is None:
        raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "ppM is null (ArgumentNullException)")
    return _run(0, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, None, ppM=ppM, **kw)


def getBestPWMSsOfPPM(numberOfRepetitions, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, ppM, *,
                      seed: int = 0, chain: int = 0, uniforms=None, engine: Optional[GibbsEngine] = None,
                      max_sweeps: int = 0) -> list:
    """fs:1001-1026: the restart loop over doMotifSamplingWithPPM-shaped restarts."""
    if ppM is None:
        raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "ppM is null (ArgumentNullException)")
    n_restarts = max(int(numberOfRepetitions) + 1, 1)
    return _run(0, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sources, None, n_chains=n_restarts,
               seed=seed, chain=chain, uniforms=uniforms, engine=engine, max_sweeps=max_sweeps, ppM=ppM,
               best_of=int(numberOfRepetitions))


# ---- many sets in one batch (gibbs_batch_run_motif_device): one result per set, element s = the single-set function on sets[s]
def _motif_restart_loop_of_sets(numberOfRepetitions, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sets, pcvs, *,
                                seed: int = 0, chain: int = 0, max_sweeps: int = 0,
                                engine: Optional[BatchEngine] = None) -> list:
    m = _check_m(motifAmount)
    if sets is not None:
        sets = list(sets)   # (a generator is read once)
    if pcvs is None:
        _bg_of(alphabet, ProbabilityCompositeVector.ofACGT(1, 1, 1, 1))   # only checks A,C,G,T are in the alphabet
        bg, bg0, background = None, [0.25] * 4, _abi.GIBBS_BG_DATA
    else:
        pcvs = list(pcvs)
        if sets is not None and engine is None and len(pcvs) != len(sets):
            raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, f"{len(pcvs)} pcvs for {len(sets)} sets")
        bg = [_bg_of(alphabet, pcv) for pcv in pcvs]
        bg0, background = bg[0] if bg else [0.25] * 4, _abi.GIBBS_BG_FIXED
    params = make_params(motifLength, pseudoCount, len(alphabet), bg0, cutoff=cutOff, background=background,
                         sampler=_abi.GIBBS_MOTIF_SAMPLER, max_sweeps=max_sweeps, motif_amount=m)
    eng = engine if engine is not None else BatchEngine(sets)
    try:
        eng.run_motif_device(params, max(int(numberOfRepetitions) + 1, 1), bg_per_set=bg, chain_id_base=chain, seed=seed)
        best = eng.fetch_best(int(numberOfRepetitions))
        if m == 1:
            return [_to_motif_array(b.scores, b.sites) for b in best]
        pos = eng.fetch_best_positions(m)
        return [_to_motif_array(b.scores, b.sites if b.restart < 0 else pos[s]) for s, b in enumerate(best)]
    finally:
        if engine is None:
            eng.close()


def findBestInormationContentContainingMotifsWithPCVOfSets(numberOfRepetitions, motifAmount, motifLength, pseudoCount, cutOff,
                                                           alphabet, sets, pcvs, **kw) -> list:
    """findBestInormationContentContainingMotifsWithPCV (fs:856-881) of every set, pcvs[s] the background of sets[s]; the
    restarts of all sets run in one batch. Element s equals findBestInormationContentContainingMotifsWithPCV(...,
    sets[s], pcvs[s]) with the same seed / chain."""
    if pcvs is None:
        raise _abi.GibbsArgumentError(_abi.GIBBS_ERR_ARG, "pcvs is null (ArgumentNullException)")
    return _motif_restart_loop_of_sets(numberOfRepetitions, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sets, pcvs,
                                       **kw)


def getMotifsWithBestInformationContentsOfSets(numberOfRepetitions, motifAmount, motifLength, pseudoCount, cutOff, alphabet,
                                               sets, **kw) -> list:
    """getMotifsWithBestInformationContents (fs:973-998) of every set, in one batch -- e.g. the reference script's fsx:407
    call per gene group. Element s equals getMotifsWithBestInformationContents(..., sets[s]) with the same seed / chain."""
    return _motif_restart_loop_of_sets(numberOfRepetitions, motifAmount, motifLength, pseudoCount, cutOff, alphabet, sets, None,
                                       **kw)
