"""Host-side logic that needs no GPU: boundary types, the restart-loop replay, chain sharding."""
import numpy as np
import pytest

import oracle_lib as O
from gibbssampling_b200 import MotifSampler, PositionMatrix, SiteSampler, _abi
from gibbssampling_b200.CompositeVector import (ProbabilityCompositeVector, createFCVOf, createNormalizedPCVOfFCV,
                                                createPCVOfSources, fuseFrequencyVectors)
from gibbssampling_b200.distributed import select_best, shard_chains
from gibbssampling_b200.engine import draws_per_chain, flatten_sources, make_params, symbol_code
from gibbssampling_b200.synthetic import background_of, planted_motif_set

DNA = list("ATGC-")


def test_composite_vector_matches_oracle(golden):
    seqs = golden["sequences"]
    pcv = createPCVOfSources(DNA, golden["pc"], seqs)
    want = O.pcv_of_sources(O.sources(seqs), golden["pc"])
    assert pcv.Array.tobytes() == want.tobytes()
    assert pcv.acgt() == [golden["q"][c] for c in "ACGT"]
    fcv = createFCVOf("ACGT*Z")
    assert fcv["*"] == 1 and fcv["Z"] == 1 and fcv.Array.sum() == 6
    with pytest.raises(IndexError):
        createFCVOf("acgt")          # lower case is outside '*'..'Z' (fs:17); the parser folds case upstream
    fused = fuseFrequencyVectors(list("AC"), [createFCVOf("AACGT"), createFCVOf("CCT")])
    assert fused["A"] == 2 and fused["C"] == 3 and fused["G"] == 0 and fused["T"] == 0   # alphabet slots only
    norm = createNormalizedPCVOfFCV(list("AC"), 0.5, fused)
    assert norm["A"] == (2 + 0.5) / (5 + 2 * 0.5)


def test_background_helper_equals_reference_construction():
    ps = planted_motif_set(50, 80, 8, seed=3)
    bg = background_of(ps.ascii, 1e-4, 5)
    pcv = createPCVOfSources(DNA, 1e-4, ps.sequences())
    assert bg == pcv.acgt()


def test_flatten_sources_and_symbols():
    buf, off = flatten_sources(["ACG", b"T", list("GA"), [65, 67]])
    assert buf.tobytes() == b"ACGTGAAC" and off.tolist() == [0, 3, 4, 6, 8]
    assert symbol_code("A") == 65 and symbol_code(b"T") == 84 and symbol_code(71) == 71
    with pytest.raises(_abi.GibbsArgumentError):
        flatten_sources(None)
    with pytest.raises(_abi.GibbsArgumentError):
        symbol_code("AC")


def test_params_struct_roundtrip():
    p = make_params(12, 1e-4, 5, [0.1, 0.2, 0.3, 0.4], cutoff=1.0, sampler=1, phase_shifts=False, max_sweeps=7, phase_mask=6)
    assert (p.k, p.alphabet_size, p.pseudocount, list(p.bg), p.cutoff) == (12, 5, 1e-4, [0.1, 0.2, 0.3, 0.4], 1.0)
    assert (p.sampler, p.phase_shifts, p.max_sweeps, p.phase_mask, p.background) == (1, 0, 7, 6, 0)
    assert draws_per_chain(1000) == 999000 and draws_per_chain(10, _abi.GIBBS_MOTIF_SAMPLER) == 100


def _oracle_restarts(S, k, pc, pcv, seed, base, count):
    scores, sites = [], []
    for r in range(count):
        rng, _ = O.make_rng(seed=seed, chain=base + r)
        sc, pos, _ = O.site_step("do_site_sampling_with_bpv", S, k, pc, pcv=pcv, rng=rng)
        scores.append(sc)
        sites.append(pos)
    return np.array(scores), np.array(sites)


@pytest.mark.parametrize("reps", [0, 1, 2, 3, 6])
def test_restart_loop_replay_equals_oracle_loop(golden, reps):
    """fs:434-459 replayed over pre-computed restarts == the oracle running the loop sequentially."""
    S = O.sources(golden["sequences"])
    k, pc = golden["k"], golden["pc"]
    pcv = O.pcv_of_sources(S, pc)
    for seed in range(5):
        scores, sites = _oracle_restarts(S, k, pc, pcv, seed, 100, reps + 1)
        got = SiteSampler.replay_restart_loop(reps, scores, sites)
        rng, _ = O.make_rng(seed=seed, chain=100)
        want_s, want_p, st = O.best_information_content(0, reps, S, k, pc, rng, pcv=pcv)
        assert [p for _, p in got] == want_p.tolist()
        assert [s for s, _ in got] == want_s.tolist()
        assert st.restarts <= reps + 1


def test_restart_loop_quirks():
    # reps = 0: one restart runs at n = 0 and is never compared -> the initial [|(0., 0)|] comes back (A.6-8)
    s = np.array([[5.0, 6.0]])
    p = np.array([[1, 2]])
    assert SiteSampler.replay_restart_loop(0, s, p) == [(0.0, 0)]
    # reps = 1: R1 promoted iff its sum > 0
    assert SiteSampler.replay_restart_loop(1, s, p) == [(5.0, 1), (6.0, 2)]
    neg = np.array([[-5.0, 1.0], [9.0, 9.0]])
    assert SiteSampler.replay_restart_loop(1, neg, np.array([[1, 2], [3, 4]])) == [(0.0, 0)]   # R2 runs, is discarded
    # reps = 3: R1 promoted at n=1, R2 runs at n=2, compared at n=3 (promotion), loop ends
    two = np.array([[1.0, 1.0], [2.0, 2.0], [50.0, 50.0]])
    pos = np.array([[0, 0], [1, 1], [2, 2]])
    assert SiteSampler.replay_restart_loop(3, two, pos) == [(2.0, 1), (2.0, 1)]
    assert SiteSampler.replay_restart_loop(2, two, pos) == [(1.0, 0), (1.0, 0)]


def test_get_best_information_content(golden):
    items = [[(1.0, 0), (2.0, 1)], [(5.0, 2)], [(2.5, 3), (2.5, 4)], [(-1.0, 0)]]
    assert PositionMatrix.getBestInformationContent(items) == [(5.0, 2)]
    assert PositionMatrix.getBestInformationContent([[(-1.0, 0)]]) == []
    flat = np.array([1.0, 2.0, 5.0, 2.5, 2.5, -1.0])
    lens = np.array([2, 1, 2, 1], dtype=np.int32)
    import ctypes as C
    idx = C.c_int32()
    assert O.lib().or_get_best_information_content(flat.ctypes.data_as(C.POINTER(C.c_double)),
                                                   lens.ctypes.data_as(C.POINTER(C.c_int32)), 4, C.byref(idx)) == 0
    assert idx.value == 1
    assert PositionMatrix.getRandomNumberInSequence(6, 21, 0.4999) == 7


def test_shard_chains_partitions_exactly():
    for n_chains in (0, 1, 7, 8, 1024, 8192, 65536 + 3):
        for world in (1, 2, 4, 8):
            got = [shard_chains(n_chains, r, world) for r in range(world)]
            assert sum(c for _, c in got) == n_chains
            nxt = 0
            for first, count in got:
                assert first == nxt
                nxt += count
            assert max(c for _, c in got) - min(c for _, c in got) <= 1
    with pytest.raises(ValueError):
        shard_chains(8, 8, 8)


def test_select_best_is_strict_max_with_lowest_chain_id():
    sums = np.array([1.0, 7.0, 7.0, 3.0])
    assert select_best(sums, np.array([40, 30, 20, 10])) == 2
    assert select_best(sums, np.array([10, 20, 30, 40])) == 1
    assert select_best(np.array([-np.inf, -np.inf]), np.array([5, 4])) == 1


def test_unbuilt_reference_entry_points_say_so():
    with pytest.raises(_abi.GibbsArgumentError):      # a null PPM is the reference's ArgumentNullException
        SiteSampler.doSiteSamplingWithPPM(6, 1e-4, DNA, ["ACGTACGT"], None)
    with pytest.raises(_abi.GibbsArgumentError):
        MotifSampler.doMotifSamplingWithPPM(1, 6, 1e-4, 0.0, DNA, ["ACGTACGT"], None)
    with pytest.raises(_abi.GibbsUnsupportedError):
        SiteSampler.doSiteSampling(6, 1e-4, list("AT"), ["ACGTACGT"])
    with pytest.raises(_abi.GibbsUnsupportedError):
        SiteSampler.doSiteSamplingWithBPV(6, 1e-4, list("AT"), ["ACGTACGT"], ProbabilityCompositeVector())
    assert MotifSampler.createMotifIndex(1.5, [3]) == MotifSampler.MotifIndex(1.5, (3,))
    with pytest.raises(_abi.GibbsUnsupportedError):
        MotifSampler.doMotifSamplingWithPCV(3, 6, 1e-4, 1.0, DNA, ["ACGTACGT"], ProbabilityCompositeVector.ofACGT(.25, .25, .25, .25))


# ---------------------------------------------------------------------------------------------
# the event walk of restart_select_kernel (gibbs_fetch.cuh), modelled lane by lane
# ---------------------------------------------------------------------------------------------
def _event_walk(sums, scores, sites, reps, motif=False):
    """Python model of restart_select_kernel: 32 restarts per step, stopping only at events (iteration cap, a sum equal
    to the best one, a larger sum). Returns the restart index the loop returns (-1 = the initial value)."""
    import math
    n_chains, N = scores.shape
    best, bsum, r_next, n_next, done = -1, 0.0, 0, 1, False
    while not done and r_next < n_chains:
        ev = None
        for lane in range(32):
            r = r_next + lane
            if r >= n_chains:
                break
            s, nj = sums[r], n_next + lane
            if nj > reps or s == bsum or s > bsum:
                ev = (lane, r, nj, s)
                break
        if ev is None:
            cnt = min(32, n_chains - r_next)
            r_next += cnt
            n_next += cnt
            continue
        _, r_j, n_j, s_j = ev
        if n_j > reps:
            break
        if s_j == bsum:
            if best < 0:
                same = N == 1 and scores[r_j][0] == 0.0 and sites[r_j][0] == (-1 if motif else 0)
            else:
                same = bool(np.array_equal(sites[r_j], sites[best]) and np.array_equal(scores[r_j], scores[best]))
            if same:
                break
            r_next, n_next = r_j + 1, n_j + 1
            continue
        best, bsum = r_j, s_j
        if bsum < 0.0:
            done = True
        r_next, n_next = r_j + 1, n_j + 2
    return best


@pytest.mark.parametrize("seed", range(40))
def test_event_walk_equals_the_sequential_restart_loop(seed):
    from gibbssampling_b200 import MotifSampler, SiteSampler
    rng = np.random.default_rng(seed)
    n_chains = int(rng.integers(1, 150))
    N = int(rng.integers(1, 4))
    pool = rng.normal(size=(int(rng.integers(1, 6)), N)).round(1)         # few distinct rows: equal sums and equal arrays happen
    if seed % 5 == 0:
        pool = np.abs(pool)
    if seed % 7 == 0:
        pool[0, :] = 0.0
    rows = rng.integers(0, len(pool), size=n_chains)
    scores = pool[rows].copy()
    sites = (rows[:, None] % 2 + np.zeros((1, N), dtype=np.int64)).astype(np.int32)
    if seed % 7 == 0:
        sites[rows == 0] = 0
    if seed % 11 == 0:
        scores[rng.integers(0, n_chains)] = np.nan
    sums = np.array([sum([0.0] + [float(v) for v in row]) for row in scores])
    for reps in (0, 1, 2, n_chains - 1, n_chains + 5, 3 * n_chains):
        reps = max(reps, 0)
        if reps + 1 > n_chains and seed % 2:      # the library always runs reps + 1 restarts; model both anyway
            continue
        want = SiteSampler.replay_restart_loop(reps, scores, sites, sums) if reps + 1 <= n_chains else None
        if want is None:
            continue
        b = _event_walk(sums, scores, sites, reps)
        got = [(0.0, 0)] if b < 0 else [(float(s), int(p)) for s, p in zip(scores[b], sites[b])]
        assert str(got) == str(want), (seed, reps)
        msites = np.where(sites == 0, -1, sites)
        wantm = MotifSampler.replay_motif_restart_loop(reps, scores, msites, sums)
        b = _event_walk(sums, scores, msites, reps, motif=True)
        gotm = [MotifSampler.MotifIndex(0.0, ())] if b < 0 else MotifSampler._to_motif_array(scores[b], msites[b])
        assert str(gotm) == str(wantm), (seed, reps)


def test_alphabet_members_the_tables_cannot_hold_are_rejected():
    """A fifth alphabet member is taken to be Gap (the script's dnaBases, fsx:368-369); any other extra member would have a PWM
    row of its own in the reference (fs:283-287), so the host layer refuses it instead of scoring it as a dead symbol."""
    from gibbssampling_b200 import _abi
    from gibbssampling_b200.CompositeVector import ProbabilityCompositeVector
    from gibbssampling_b200.SiteSampler import _bg_of
    pcv = ProbabilityCompositeVector.ofACGT(0.1, 0.2, 0.3, 0.4)
    assert _bg_of(list("ATGC-"), pcv) == [0.1, 0.2, 0.3, 0.4]
    assert _bg_of(list("ACGT"), pcv) == [0.1, 0.2, 0.3, 0.4]
    with pytest.raises(_abi.GibbsUnsupportedError):
        _bg_of(list("ACGTN"), pcv)
    with pytest.raises(_abi.GibbsUnsupportedError):
        _bg_of(list("ACG"), pcv)
