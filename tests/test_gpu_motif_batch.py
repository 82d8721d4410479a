"""MotifSampler batches (gibbs_batch_run_motif_device, BatchEngine.run_motif_device, MotifSampler.…OfSets): every set must
give bit for bit what a MotifSampler handle over that set alone gives with the same parameters, seed and chain_id_base --
every restart, the Positions lists, the restart loop, the counters -- for motifAmount 1 and 2 and both backgrounds."""
import json
import os

import numpy as np
import pytest

import oracle_lib as O
from gibbssampling_b200 import MotifSampler, _abi
from gibbssampling_b200.CompositeVector import ProbabilityCompositeVector
from gibbssampling_b200.engine import BatchEngine, GibbsEngine, make_params
from gibbssampling_b200.synthetic import background_of, planted_motif_set

pytestmark = pytest.mark.gpu
DNA = list("ATGC-")
COUNTERS = ("site_updates", "window_scores", "sweeps")
FIXED, DATA = _abi.GIBBS_BG_FIXED, _abi.GIBBS_BG_DATA
MOTIF = _abi.GIBBS_MOTIF_SAMPLER


def _ragged_set(n, max_len, min_len, k, seed, other=None):
    """n sequences of min_len .. max_len bp with a planted k-mer; other = symbols outside A,C,G,T sprinkled in."""
    ps = planted_motif_set(n, max_len, min(k, min_len), seed=seed, min_length=min_len)
    seqs = ps.sequences()
    if other:
        rng = np.random.default_rng(seed)
        seqs = [bytearray(s) for s in seqs]
        for i in range(0, n, 2):
            for _ in range(3):
                seqs[i][int(rng.integers(0, len(seqs[i])))] = ord(other[int(rng.integers(0, len(other)))])
        seqs = [bytes(s) for s in seqs]
    return seqs


def _mixed_sets(k, masked=True):
    """N = 2 .. 200, ragged lengths; with masked, sets holding symbols outside A,C,G,T (1- and 4-warp, masked groups).
    Sequences are at least 4k + 3 long: under a fixed pcv a window over such a symbol has no background mass, and a
    sequence whose every window holds one makes the roulette run past the list (test_roulette_error_names_the_set)."""
    lo = max(4 * k + 3, 12)
    spec = [(2, 40, 0, None), (3, 60, 1, None), (4, 50, 2, None), (7, 90, 3, None), (33, 120, 4, None), (200, 80, 5, None),
            (12, 130, 11, None)]
    if masked:
        spec += [(2, 45, 6, "N*"), (3, 70, 7, "-"), (4, 64, 8, "N"), (7, 100, 9, "*-N"), (33, 75, 10, "N")]
    return [_ragged_set(n, max(L, lo + 8), lo, k, 100 + s, other) for n, L, s, other in spec]


def _acgt_sets(k):
    lo = max(k + 4, 16)
    spec = [(2, 30, 0), (3, 45, 1), (4, 40, 2), (6, 60, 3), (9, 50, 4), (17, 36, 5)]
    return [_ragged_set(n, max(L, lo + 6), lo, k, 300 + s) for n, L, s in spec]


def _bg(seqs):
    return background_of(np.frombuffer(b"".join(seqs), dtype=np.uint8), 1e-4, 4)


def _params(k, bg, background, cutoff, m=1, pc=1e-4, alen=4):
    return make_params(k, pc, alen, bg, cutoff=cutoff, background=background, sampler=MOTIF, motif_amount=m)


def _single(seqs, params, R, chain, seed):
    """every restart of a single-set handle: (RunResult, Positions lists [R, N, m])"""
    with GibbsEngine(seqs) as eng:
        res = eng.run(params, R, chain_id_base=chain, seed=seed, want_counts=False)
        return res, eng.fetch_positions(max(params.motif_amount, 1))


def _single_best(seqs, params, reps, chain, seed):
    with GibbsEngine(seqs) as eng:
        eng.run_device(params, reps + 1, chain_id_base=chain, seed=seed)
        best = eng.fetch_best(reps, want_counts=True)
        return best, eng.fetch_best_positions(max(params.motif_amount, 1))


def _same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float64).view(np.uint64), np.asarray(b, np.float64).view(np.uint64))


def _check_every_restart(sets, k, background, cutoff, m, R=3, chain=17, seed=2024):
    bgs = [_bg(s) for s in sets]
    with BatchEngine(sets) as b:
        b.run_motif_device(_params(k, bgs[0], background, cutoff, m), R, bg_per_set=bgs if background == FIXED else None,
                           chain_id_base=chain, seed=seed)
        got = b.fetch()
        pos = b.fetch_positions(m)
    total = {c: 0 for c in COUNTERS}
    no_site = 0
    for s, seqs in enumerate(sets):
        want, want_pos = _single(seqs, _params(k, bgs[s], background, cutoff, m), R, chain, seed)
        assert np.array_equal(got.sites[s], want.sites), f"set {s}"
        assert np.array_equal(pos[s], want_pos), f"set {s}"
        assert _same_bits(got.scores[s], want.scores), f"set {s}"
        assert _same_bits(got.sums[s], want.sums), f"set {s}"
        for c in COUNTERS:
            total[c] += want.stats[c]
        no_site += int((want.sites < 0).sum())
    for c in COUNTERS:
        assert got.stats[c] == total[c], c
    return no_site


@pytest.mark.parametrize("k", [1, 6, 12, 17, 32])
@pytest.mark.parametrize("background", [FIXED, DATA])
@pytest.mark.parametrize("high_cutoff", [False, True])
def test_every_restart_equals_a_single_set_handle(k, background, high_cutoff):
    """motifAmount 1 over mixed sets (1- and 4-warp groups, masked groups); a cut-off near the best windows' log2 score
    makes "no site" common."""
    cutoff = 1.5 * k if high_cutoff else 0.0
    no_site = _check_every_restart(_mixed_sets(k), k, background, cutoff, 1, seed=2024 + k)
    if high_cutoff:
        assert no_site > 0


@pytest.mark.parametrize("background", [FIXED, DATA])
@pytest.mark.parametrize("k,cutoff", [(4, 0.5), (6, 1.0), (9, 3.0)])
def test_every_restart_with_two_sites_equals_a_single_set_handle(background, k, cutoff):
    _check_every_restart(_acgt_sets(k), k, background, cutoff, 2, seed=77 + k)


@pytest.mark.parametrize("m", [1, 2])
@pytest.mark.parametrize("reps", [0, 1, 3, 7])
def test_restart_loop_of_every_set(m, reps):
    k, cutoff = 6, 1.0
    sets = _acgt_sets(k) if m == 2 else _mixed_sets(k)
    bgs = [_bg(s) for s in sets]
    with BatchEngine(sets) as b:
        b.run_motif_device(_params(k, bgs[0], FIXED, cutoff, m), reps + 1, bg_per_set=bgs, chain_id_base=5, seed=99)
        every = b.fetch()
        every_pos = b.fetch_positions(m)
        best = b.fetch_best(reps, want_counts=True)
        best_pos = b.fetch_best_positions(m)
    for s, seqs in enumerate(sets):
        lists = every_pos[s] if m == 2 else every.sites[s]
        replay = MotifSampler.replay_motif_restart_loop(reps, every.scores[s], lists, every.sums[s])
        got = MotifSampler._to_motif_array(best[s].scores, best[s].sites if best[s].restart < 0 or m == 1 else best_pos[s])
        assert got == replay, f"set {s}"
        want, want_pos = _single_best(seqs, _params(k, bgs[s], FIXED, cutoff, m), reps, 5, 99)
        assert best[s].sites.tolist() == want.sites.tolist(), f"set {s}"
        assert np.array_equal(best_pos[s], want_pos), f"set {s}"
        assert _same_bits(best[s].scores, want.scores)
        assert _same_bits(best[s].total, want.total)
        assert best[s].restart == want.restart
        assert best[s].counts.tolist() == want.counts.tolist(), f"set {s}"
        if reps == 0:   # one restart, one iteration: the loop returns its initial value [|{PWMS 0; Positions []}|]
            assert got == [MotifSampler.MotifIndex(0.0, ())] and best[s].restart == -1 and not best[s].counts.any()
            assert best[s].sites.tolist() == [-1] and (best_pos[s] == -1).all()


def _oracle_sets(k):
    from conftest import ROOT
    with open(os.path.join(ROOT, "tests", "golden", "appendix_b.json")) as f:
        g = json.load(f)
    sets = [g["sequences"], g["multi_sequences"]]
    sets += [planted_motif_set(n, 40, k, seed=200 + n, min_length=20).sequences() for n in (2, 5, 9)]
    return [[s.encode() if isinstance(s, str) else s for s in ss] for ss in sets]


@pytest.mark.parametrize("m", [1, 2])
def test_winners_equal_the_oracle(m):
    k, pc, cutoff, reps, seed, chain = 5, 1e-4, 1.0, 3, 41, 7
    sets = _oracle_sets(k)
    pcvs = [ProbabilityCompositeVector.ofACGT(*background_of(np.frombuffer(b"".join(ss), dtype=np.uint8), pc, 5)) for ss in sets]
    fixed = MotifSampler.findBestInormationContentContainingMotifsWithPCVOfSets(reps, m, k, pc, cutoff, DNA, sets, pcvs,
                                                                                 seed=seed, chain=chain)
    data = MotifSampler.getMotifsWithBestInformationContentsOfSets(reps, m, k, pc, cutoff, DNA, sets, seed=seed, chain=chain)
    for s, ss in enumerate(sets):
        S = O.sources(ss)
        bg = [pcvs[s][ch] for ch in "ACGT"]
        for variant, got in ((0, fixed[s]), (1, data[s])):
            rng, _ = O.make_rng(seed=seed, chain=chain)
            want, _ = O.best_motif_information_content(variant, reps, S, m, k, pc, cutoff, rng,
                                                       pcv=O.pcv_from_acgt(bg) if variant == 0 else None)
            assert [list(x.Positions) for x in got] == [list(p) for _, p in want], f"set {s}, variant {variant}"
            np.testing.assert_allclose([x.PWMS for x in got], [v for v, _ in want], rtol=1e-5)
        assert fixed[s] == MotifSampler.findBestInormationContentContainingMotifsWithPCV(reps, m, k, pc, cutoff, DNA, ss, pcvs[s],
                                                                                          seed=seed, chain=chain)
        assert data[s] == MotifSampler.getMotifsWithBestInformationContents(reps, m, k, pc, cutoff, DNA, ss, seed=seed, chain=chain)


@pytest.mark.parametrize("m,background", [(1, FIXED), (1, DATA), (2, FIXED), (2, DATA)])
def test_results_do_not_depend_on_set_order_or_batch_split(m, background):
    k, reps, cutoff = 6, 2, 1.0
    sets = _acgt_sets(k) if m == 2 else _mixed_sets(k)
    bgs = [_bg(s) for s in sets]
    fixed = background == FIXED

    def run(idx):
        with BatchEngine([sets[i] for i in idx]) as b:
            b.run_motif_device(_params(k, bgs[idx[0]], background, cutoff, m), reps + 1,
                               bg_per_set=[bgs[i] for i in idx] if fixed else None, chain_id_base=3, seed=8)
            every = b.fetch()
            pos = b.fetch_positions(m)
            best = b.fetch_best(reps, want_counts=True)
            best_pos = b.fetch_best_positions(m)
        return {i: (every.sites[j], every.scores[j], pos[j], best[j], best_pos[j]) for j, i in enumerate(idx)}

    base = run(list(range(len(sets))))
    perm = np.random.default_rng(1).permutation(len(sets)).tolist()
    split = run(perm[:3])
    split.update(run(perm[3:]))
    for other in (run(perm), split):
        for i in range(len(sets)):
            a, b = base[i], other[i]
            assert np.array_equal(a[0], b[0]) and _same_bits(a[1], b[1]) and np.array_equal(a[2], b[2]), i
            assert a[3].sites.tolist() == b[3].sites.tolist() and _same_bits(a[3].scores, b[3].scores), i
            assert a[3].restart == b[3].restart and a[3].counts.tolist() == b[3].counts.tolist(), i
            assert np.array_equal(a[4], b[4]), i


def _sample_against_handles(sets, got, pos, params_of, R, chain, seed, m, sample):
    for s in sample:
        want, want_pos = _single(sets[s], params_of(s), R, chain, seed)
        assert np.array_equal(got.sites[s], want.sites), f"set {s}"
        assert np.array_equal(pos[s], want_pos), f"set {s}"
        assert _same_bits(got.scores[s], want.scores) and _same_bits(got.sums[s], want.sums), f"set {s}"


def test_large_batch_of_one_site_runs():
    """4096 sets x 20 sequences x 100 bp, motifAmount 1: a sample of sets against single-set handles."""
    k, R, S = 8, 2, 4096
    sets = [planted_motif_set(20, 100, k, seed=5000 + s).sequences() for s in range(S)]
    bgs = [_bg(s) for s in sets]
    with BatchEngine(sets) as b:
        b.run_motif_device(_params(k, bgs[0], FIXED, 0.0), R, bg_per_set=bgs, chain_id_base=11, seed=3)
        got = b.fetch()
        pos = b.fetch_positions(1)
        best = b.fetch_best(R - 1)
    assert len(best) == S
    _sample_against_handles(sets, got, pos, lambda s: _params(k, bgs[s], FIXED, 0.0), R, 11, 3, 1, [0, 1, 777, 2048, S - 1])


def test_large_batch_of_two_site_runs():
    """A few hundred sets with motifAmount 2 and the data-derived background."""
    k, R, S = 6, 2, 300
    sets = [planted_motif_set(10, 60, k, seed=9000 + s).sequences() for s in range(S)]
    with BatchEngine(sets) as b:
        b.run_motif_device(_params(k, [0.25] * 4, DATA, 1.0, 2), R, chain_id_base=2, seed=12)
        got = b.fetch()
        pos = b.fetch_positions(2)
    _sample_against_handles(sets, got, pos, lambda s: _params(k, [0.25] * 4, DATA, 1.0, 2), R, 2, 12, 2, [0, 150, S - 1])


def test_one_batch_through_both_samplers_equals_fresh_batches():
    """SiteSampler -> MotifSampler m = 2 -> m = 1 -> SiteSampler on one BatchEngine: the per-set tables it caches are
    rebuilt whenever the sampler, motifAmount or background changes."""
    k, R = 6, 2
    sets = _acgt_sets(k)
    bgs = [_bg(s) for s in sets]
    site = make_params(k, 1e-4, 4, bgs[0])
    runs = [("site", site, bgs), ("motif", _params(k, bgs[0], FIXED, 1.0, 2), bgs), ("motif", _params(k, bgs[0], FIXED, 1.0, 1), bgs),
            ("motif", _params(k, bgs[0], DATA, 1.0, 2), None), ("site", site, bgs)]

    def go(b, kind, params, bg):
        (b.run_device if kind == "site" else b.run_motif_device)(params, R, bg_per_set=bg, chain_id_base=1, seed=21)
        every = b.fetch()
        m = max(params.motif_amount, 1)
        return every, b.fetch_positions(m), b.fetch_best(1, want_counts=True)

    with BatchEngine(sets) as shared:
        seen = [go(shared, *r) for r in runs]
    for r, (every, pos, best) in zip(runs, seen):
        with BatchEngine(sets) as fresh:
            w_every, w_pos, w_best = go(fresh, *r)
        for s in range(len(sets)):
            assert np.array_equal(every.sites[s], w_every.sites[s]) and _same_bits(every.scores[s], w_every.scores[s]), (r[0], s)
            assert np.array_equal(pos[s], w_pos[s]), (r[0], s)
            assert best[s].sites.tolist() == w_best[s].sites.tolist() and best[s].counts.tolist() == w_best[s].counts.tolist()


def test_errors_name_the_set_and_leave_the_batch_usable():
    k = 6
    good = [planted_motif_set(5, 40, k, seed=1).sequences(), planted_motif_set(3, 30, k, seed=2).sequences()]
    sets = good + [[b"ACGTACGTAC", b"ACG", b"ACGTACGTACGT"], [b"ACGT-ACGTACGT", b"TTTTACGTAGGA"]]
    with BatchEngine(sets) as b:
        with pytest.raises(_abi.GibbsShortSequenceError) as ei:
            b.run_motif_device(_params(k, [0.25] * 4, FIXED, 1.0), 2)
        assert "set 2, sequence 1" in str(ei.value)
    gap_sets = good + [sets[3]]
    bgs = [_bg(s) for s in gap_sets]
    with BatchEngine(gap_sets) as b:
        with pytest.raises(_abi.GibbsUnsupportedError) as ei:
            b.run_motif_device(_params(k, [0.25] * 4, FIXED, 1.0, alen=5), 2)
        assert "set 2" in str(ei.value)
        with pytest.raises(_abi.GibbsUnsupportedError) as ei:   # two sites per sequence need A,C,G,T-only sets
            b.run_motif_device(_params(k, [0.25] * 4, DATA, 1.0, 2), 2)
        assert "set 2" in str(ei.value)
        with pytest.raises(_abi.GibbsUnsupportedError):
            b.run_motif_device(_params(k, [0.25] * 4, FIXED, 1.0, 3), 2)
        with pytest.raises(_abi.GibbsUnsupportedError):         # the SiteSampler's entry point keeps refusing the MotifSampler
            b.run_device(_params(k, [0.25] * 4, FIXED, 1.0), 2)
        with pytest.raises(_abi.GibbsArgumentError):
            b.run_motif_device(make_params(k, 1e-4, 4, [0.25] * 4), 2)   # a SiteSampler params block
        with pytest.raises(_abi.GibbsArgumentError):
            b.run_motif_device(make_params(k, 1e-4, 4, [0.25] * 4, sampler=MOTIF, phase_mask=_abi.PHASE_STOCHASTIC), 2)
        with pytest.raises(_abi.GibbsArgumentError) as ei:
            b.run_motif_device(_params(k, [0.25] * 4, FIXED, 1.0), 2, bg_per_set=[[0.25] * 4, [0.25] * 4, [0.0, 0.5, 0.25, 0.25]])
        assert "set 2" in str(ei.value)
        with pytest.raises(_abi.GibbsArgumentError):             # no MotifSampler run yet
            b.fetch_positions(2)
        # still usable: a valid run equals the single-set handles
        b.run_motif_device(_params(k, bgs[0], FIXED, 1.0), 2, bg_per_set=bgs, chain_id_base=4, seed=6)
        got = b.fetch()
        with pytest.raises(_abi.GibbsArgumentError):             # positions of the motifAmount the run had
            b.fetch_positions(2)
    for s, seqs in enumerate(gap_sets):
        want, _ = _single(seqs, _params(k, bgs[s], FIXED, 1.0), 2, 4, 6)
        assert np.array_equal(got.sites[s], want.sites) and _same_bits(got.scores[s], want.scores)


def test_roulette_error_names_the_set():
    """A held-out sequence whose every window holds a symbol outside the alphabet has no background mass under a fixed
    pcv: the pick runs past the list (the reference throws, fs:753). Fetch names the set; the batch stays usable."""
    k = 4
    good = planted_motif_set(5, 40, k, seed=3).sequences()
    bad = good[:3] + [b"NNNNNNNNNNNN"]
    params = _params(k, [0.25] * 4, FIXED, 0.0)
    with GibbsEngine(bad) as eng:
        with pytest.raises(_abi.GibbsRouletteError):
            eng.run(params, 2, chain_id_base=0, seed=1, want_counts=False)
    with BatchEngine([good, bad]) as b:
        b.run_motif_device(params, 2, chain_id_base=0, seed=1)
        with pytest.raises(_abi.GibbsRouletteError) as ei:
            b.fetch()
        assert "set 1" in str(ei.value)
        with pytest.raises(_abi.GibbsRouletteError):
            b.fetch_best(1)
    with BatchEngine([good, good]) as b:
        b.run_motif_device(params, 2, chain_id_base=0, seed=1)
        got = b.fetch()
    want, _ = _single(good, params, 2, 0, 1)
    assert np.array_equal(got.sites[1], want.sites)
