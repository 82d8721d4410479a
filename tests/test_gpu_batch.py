"""Many sequence sets in one batch (gibbs_batch_*, engine.BatchEngine): every set must give bit for bit what a handle over
that set alone gives with the same parameters, seed and chain_id_base -- every restart, the restart loop, the counters."""
import numpy as np
import pytest

import oracle_lib as O
from gibbssampling_b200 import SiteSampler, _abi
from gibbssampling_b200.CompositeVector import ProbabilityCompositeVector
from gibbssampling_b200.engine import BatchEngine, GibbsEngine, make_params
from gibbssampling_b200.synthetic import background_of, planted_motif_set

pytestmark = pytest.mark.gpu
DNA = list("ATGC-")
COUNTERS = ("site_updates", "window_scores", "sweeps")


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


def _mixed_sets(k):
    lo = max(k, 12)
    spec = [(2, 40, 0, None), (3, 60, 1, None), (4, 50, 2, None), (7, 90, 3, None), (33, 120, 4, None), (200, 80, 5, None),
            (2, 45, 6, "N*"), (3, 70, 7, "-"), (4, 64, 8, "N"), (7, 100, 9, "*-N"), (33, 75, 10, "N"), (12, 130, 11, None)]
    return [_ragged_set(n, max(L, lo + 8), lo, k, 100 + s, other) for n, L, s, other in spec]


def _bg(seqs):
    return background_of(np.frombuffer(b"".join(seqs), dtype=np.uint8), 1e-4, 4)


def _single(seqs, params, R, chain, seed, team=None):
    with GibbsEngine(seqs) as eng:
        if team:
            eng.set_team_warps(team)
        return eng.run(params, R, chain_id_base=chain, seed=seed, want_counts=False)


def _same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float64).view(np.uint64), np.asarray(b, np.float64).view(np.uint64))


@pytest.mark.parametrize("k", [1, 6, 12, 17, 32])
@pytest.mark.parametrize("background", [_abi.GIBBS_BG_FIXED, _abi.GIBBS_BG_DATA])
@pytest.mark.parametrize("shifts", [True, False])
def test_every_restart_equals_a_single_set_handle(k, background, shifts):
    sets = _mixed_sets(k)
    R, chain, seed = 3, 17, 2024 + k
    bgs = [_bg(s) for s in sets]
    params = make_params(k, 1e-4, 4, bgs[0], phase_shifts=shifts, background=background)
    with BatchEngine(sets) as b:
        b.run_device(params, R, bg_per_set=bgs if background == _abi.GIBBS_BG_FIXED else None, chain_id_base=chain, seed=seed)
        got = b.fetch()
    total = {c: 0 for c in COUNTERS}
    for s, seqs in enumerate(sets):
        p = make_params(k, 1e-4, 4, bgs[s], phase_shifts=shifts, background=background)
        want = _single(seqs, p, R, chain, seed)
        assert np.array_equal(got.sites[s], want.sites), f"set {s}"
        assert _same_bits(got.scores[s], want.scores), f"set {s}"
        assert _same_bits(got.sums[s], want.sums), f"set {s}"
        for c in COUNTERS:
            total[c] += want.stats[c]
    for c in COUNTERS:
        assert got.stats[c] == total[c], c


@pytest.mark.parametrize("reps", [0, 1, 3, 7])
def test_restart_loop_of_every_set(reps):
    k = 6
    sets = _mixed_sets(k)
    bgs = [_bg(s) for s in sets]
    params = make_params(k, 1e-4, 4, bgs[0])
    with BatchEngine(sets) as b:
        b.run_device(params, reps + 1, bg_per_set=bgs, chain_id_base=5, seed=99)
        every = b.fetch()
        best = b.fetch_best(reps, want_counts=True)
    for s, seqs in enumerate(sets):
        replay = SiteSampler.replay_restart_loop(reps, every.scores[s], every.sites[s], every.sums[s])
        got = [(float(v), int(p)) for v, p in zip(best[s].scores, best[s].sites)]
        assert got == replay, f"set {s}"
        with GibbsEngine(seqs) as eng:
            eng.run_device(make_params(k, 1e-4, 4, bgs[s]), reps + 1, chain_id_base=5, seed=99)
            want = eng.fetch_best(reps, want_counts=True)
        assert best[s].sites.tolist() == want.sites.tolist()
        assert _same_bits(best[s].scores, want.scores)
        assert _same_bits(best[s].total, want.total)
        assert best[s].restart == want.restart
        assert best[s].counts.tolist() == want.counts.tolist(), f"set {s}"
        if reps == 0:   # one restart, one iteration: the loop returns its initial value (quirk A.6-8)
            assert got == [(0.0, 0)] and best[s].restart == -1 and not best[s].counts.any()


def test_winners_equal_the_oracle():
    from conftest import ROOT
    import json, os
    with open(os.path.join(ROOT, "tests", "golden", "appendix_b.json")) as f:
        g = json.load(f)
    k, pc, reps, seed, chain = 5, 1e-4, 3, 41, 7
    sets = [g["sequences"], g["multi_sequences"]]
    sets += [planted_motif_set(n, 40, k, seed=200 + n, min_length=20).sequences() for n in (2, 5, 9)]
    sets = [[s.encode() if isinstance(s, str) else s for s in ss] for ss in sets]
    pcvs = [ProbabilityCompositeVector.ofACGT(*background_of(np.frombuffer(b"".join(ss), dtype=np.uint8), pc, 5)) for ss in sets]
    fixed = SiteSampler.getMotifsWithBestInformationContentWithBPVOfSets(reps, k, pc, DNA, sets, pcvs, seed=seed, chain=chain)
    data = SiteSampler.getMotifsWithBestInformationContentOfSets(reps, k, pc, DNA, sets, seed=seed, chain=chain)
    for s, ss in enumerate(sets):
        S = O.sources(ss)
        bg = [pcvs[s][ch] for ch in "ACGT"]
        rng, _ = O.make_rng(seed=seed, chain=chain)
        score, pos, _ = O.best_information_content(0, reps, S, k, pc, rng, pcv=O.pcv_from_acgt(bg))
        assert [p for _, p in fixed[s]] == pos.tolist(), f"set {s}"
        np.testing.assert_allclose([v for v, _ in fixed[s]], score, rtol=1e-5)
        assert fixed[s] == SiteSampler.getMotifsWithBestInformationContentWithBPV(reps, k, pc, DNA, ss, pcvs[s], seed=seed, chain=chain)
        rng, _ = O.make_rng(seed=seed, chain=chain)
        score, pos, _ = O.best_information_content(1, reps, S, k, pc, rng)
        assert [p for _, p in data[s]] == pos.tolist(), f"set {s}"
        np.testing.assert_allclose([v for v, _ in data[s]], score, rtol=1e-5)
        assert data[s] == SiteSampler.getMotifsWithBestInformationContent(reps, k, pc, DNA, ss, seed=seed, chain=chain)


@pytest.mark.parametrize("background", [_abi.GIBBS_BG_FIXED, _abi.GIBBS_BG_DATA])
def test_results_do_not_depend_on_set_order_or_batch_split(background):
    k, reps = 8, 2
    sets = _mixed_sets(k)
    bgs = [_bg(s) for s in sets]
    params = make_params(k, 1e-4, 4, bgs[0], background=background)
    fixed = background == _abi.GIBBS_BG_FIXED

    def run(idx):
        with BatchEngine([sets[i] for i in idx]) as b:
            b.run_device(params, reps + 1, bg_per_set=[bgs[i] for i in idx] if fixed else None, chain_id_base=3, seed=8)
            every = b.fetch()
            best = b.fetch_best(reps, want_counts=True)
        return {i: (every.sites[j], every.scores[j], best[j]) for j, i in enumerate(idx)}

    base = run(list(range(len(sets))))
    perm = np.random.default_rng(1).permutation(len(sets)).tolist()
    split = run(perm[:5])
    split.update(run(perm[5:]))
    for other in (run(perm), split):
        for i in range(len(sets)):
            a, b = base[i], other[i]
            assert np.array_equal(a[0], b[0]) and _same_bits(a[1], b[1])
            assert a[2].sites.tolist() == b[2].sites.tolist() and _same_bits(a[2].scores, b[2].scores)
            assert a[2].restart == b[2].restart and a[2].counts.tolist() == b[2].counts.tolist()


def test_4096_sets_in_one_batch():
    k, R, n_sets = 8, 2, 4096
    ps = planted_motif_set(n_sets * 20, 100, k, seed=4096)
    seqs = ps.sequences()
    sets = [seqs[20 * s: 20 * s + 20] for s in range(n_sets)]
    bgs = [_bg(s) for s in sets]
    params = make_params(k, 1e-4, 5, bgs[0])
    with BatchEngine(sets) as b:
        b.run_device(params, R, bg_per_set=bgs, chain_id_base=0, seed=12)
        every = b.fetch()
        best = b.fetch_best(R - 1)
    for s in np.random.default_rng(4).choice(n_sets, 32, replace=False).tolist():
        p = make_params(k, 1e-4, 5, bgs[s])
        with GibbsEngine(sets[s]) as eng:
            eng.run_device(p, R, chain_id_base=0, seed=12)
            want = eng.fetch(want_counts=False)
            want_best = eng.fetch_best(R - 1)
        assert np.array_equal(every.sites[s], want.sites) and _same_bits(every.scores[s], want.scores), f"set {s}"
        assert best[s].sites.tolist() == want_best.sites.tolist() and _same_bits(best[s].scores, want_best.scores)


def test_errors_name_the_set_and_leave_the_batch_usable():
    k = 6
    good = [planted_motif_set(5, 40, k, seed=1).sequences(), planted_motif_set(3, 30, k, seed=2).sequences()]
    with pytest.raises(_abi.GibbsArgumentError):
        BatchEngine([good[0], []])
    with pytest.raises(_abi.GibbsSymbolError) as ei:
        BatchEngine([good[0], good[1][:2] + [b"ACGTacgt" * 4]])
    assert "set 1, sequence 2" in str(ei.value)
    sets = good + [[b"ACGTACGTAC", b"ACG", b"ACGTACGTACGT"], [b"ACGT-ACGTACGT", b"TTTTACGTAGGA"]]
    params = make_params(k, 1e-4, 4, [0.25] * 4)
    with BatchEngine(sets) as b:
        with pytest.raises(_abi.GibbsShortSequenceError) as ei:
            b.run_device(params, 2)
        assert "set 2, sequence 1" in str(ei.value)
    gap_sets = good + [sets[3]]
    with BatchEngine(gap_sets) as b:
        with pytest.raises(_abi.GibbsUnsupportedError) as ei:
            b.run_device(make_params(k, 1e-4, 5, [0.25] * 4), 2)
        assert "set 2" in str(ei.value)
        with pytest.raises(_abi.GibbsUnsupportedError):
            b.run_device(make_params(k, 1e-4, 4, [0.25] * 4, sampler=_abi.GIBBS_MOTIF_SAMPLER), 2)
        with pytest.raises(_abi.GibbsArgumentError):
            b.run_device(make_params(k, 1e-4, 4, [0.25] * 4, phase_mask=_abi.PHASE_INIT), 2)
        with pytest.raises(_abi.GibbsArgumentError):
            b.run_device(params, 2, bg_per_set=[[0.25] * 4, [0.25] * 4, [0.0, 0.5, 0.25, 0.25]])
        # still usable: a valid run equals the single-set handles
        bgs = [_bg(s) for s in gap_sets]
        b.run_device(params, 2, bg_per_set=bgs, chain_id_base=4, seed=6)
        got = b.fetch()
    for s, seqs in enumerate(gap_sets):
        want = _single(seqs, make_params(k, 1e-4, 4, bgs[s]), 2, 4, 6)
        assert np.array_equal(got.sites[s], want.sites) and _same_bits(got.scores[s], want.scores)


def test_sets_given_as_a_generator():
    k = 6
    sets = [planted_motif_set(n, 50, k, seed=30 + n).sequences() for n in (3, 6, 9)]
    pcvs = [ProbabilityCompositeVector.ofACGT(*background_of(np.frombuffer(b"".join(s), dtype=np.uint8), 1e-4, 5)) for s in sets]
    got = SiteSampler.getMotifsWithBestInformationContentWithBPVOfSets(1, k, 1e-4, DNA, (s for s in sets), pcvs, seed=3)
    assert len(got) == len(sets)
    for s, ss in enumerate(sets):
        assert got[s] == SiteSampler.getMotifsWithBestInformationContentWithBPV(1, k, 1e-4, DNA, ss, pcvs[s], seed=3)
