"""Many sequence sets over several devices (gibbs_multi_batch_*, engine.MultiBatchEngine): every output must be bit for bit
what one BatchEngine over the same sets returns, whatever the number of device slots. With fewer GPUs than slots the slots
share a device (slot i runs on GPU i % device_count), which exercises the same split, offsets and error numbering."""
import itertools

import numpy as np
import pytest

from gibbssampling_b200 import MotifSampler, SiteSampler, _abi
from gibbssampling_b200.engine import BatchEngine, GibbsEngine, MultiBatchEngine, device_count, make_params
from gibbssampling_b200.synthetic import background_of, planted_motif_set

pytestmark = pytest.mark.gpu
FIXED, DATA, MOTIF = _abi.GIBBS_BG_FIXED, _abi.GIBBS_BG_DATA, _abi.GIBBS_MOTIF_SAMPLER
COUNTERS = ("site_updates", "window_scores", "sweeps", "capped_chains")
K = 6


def _ragged_set(n, max_len, min_len, k, seed, other=None):
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


def _sets(masked):
    """ragged sets of 2 .. 200 sequences; masked: some hold symbols outside A,C,G,T"""
    lo = 4 * K + 3
    spec = [(2, 40, 0, None), (200, 60, 1, None), (3, 70, 2, None), (7, 90, 3, None), (33, 50, 4, None), (2, 35, 5, None),
            (12, 130, 6, None), (5, 45, 7, None), (4, 64, 8, None)]
    if masked:
        spec += [(2, 45, 9, "N*"), (3, 70, 10, "-"), (33, 75, 11, "N"), (7, 100, 12, "*-N")]
        spec = [spec[i] for i in (0, 9, 1, 10, 2, 3, 11, 4, 5, 12, 6, 7, 8)]   # masked sets spread over the slots
    return [_ragged_set(n, max(L, lo + 8), lo, K, 700 + s, other) for n, L, s, other in spec]


def _bg(seqs):
    return background_of(np.frombuffer(b"".join(seqs), dtype=np.uint8), 1e-4, 4)


def _devices(slots):
    ndev = device_count()
    return [i % ndev for i in range(slots)]


def _same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float64).view(np.uint64), np.asarray(b, np.float64).view(np.uint64))


# (sampler, background, motifAmount, masked sets)
KINDS = {
    "site_fixed": ("site", FIXED, 1, True),
    "site_data": ("site", DATA, 1, True),
    "motif1_fixed": ("motif", FIXED, 1, True),
    "motif1_data": ("motif", DATA, 1, True),
    "motif2_fixed": ("motif", FIXED, 2, False),
    "motif2_data": ("motif", DATA, 2, False),
}


def _run(eng, kind, sets, R, chain=5, seed=77):
    sampler, background, m, _ = KINDS[kind]
    bgs = [_bg(s) for s in sets]
    bg = bgs if background == FIXED else None
    if sampler == "site":
        eng.run_device(make_params(K, 1e-4, 4, bgs[0], background=background), R, bg_per_set=bg, chain_id_base=chain, seed=seed)
    else:
        params = make_params(K, 1e-4, 4, bgs[0], cutoff=1.0, background=background, sampler=MOTIF, motif_amount=m)
        eng.run_motif_device(params, R, bg_per_set=bg, chain_id_base=chain, seed=seed)
    return m


def _outputs(eng, m):
    """every output of the last run: fetch, fetch_positions, and fetch_best + fetch_best_positions for reps 0, 1, 2"""
    out = {"every": eng.fetch(), "pos": eng.fetch_positions(m)}
    for reps in (0, 1, 2):
        out[reps] = eng.fetch_best(reps, want_counts=True)
        out[(reps, "pos")] = eng.fetch_best_positions(m)
    return out


def _assert_equal(got, want, n_sets):
    for s in range(n_sets):
        assert np.array_equal(got["every"].sites[s], want["every"].sites[s]), f"set {s}"
        assert _same_bits(got["every"].scores[s], want["every"].scores[s]), f"set {s}"
        assert _same_bits(got["every"].sums[s], want["every"].sums[s]), f"set {s}"
        assert np.array_equal(got["pos"][s], want["pos"][s]), f"set {s}"
        for reps in (0, 1, 2):
            a, b = got[reps][s], want[reps][s]
            assert np.array_equal(a.sites, b.sites) and _same_bits(a.scores, b.scores), (reps, s)
            assert len(a.sites) == len(b.sites) and _same_bits(a.total, b.total) and a.restart == b.restart, (reps, s)
            assert np.array_equal(a.counts, b.counts), (reps, s)
            assert np.array_equal(got[(reps, "pos")][s], want[(reps, "pos")][s]), (reps, s)
    for c in COUNTERS:
        assert got["every"].stats[c] == want["every"].stats[c], c
        assert got[1][0].stats[c] == want[1][0].stats[c], c


def _check_identity(sets, kind, slots, R, devices=None):
    with BatchEngine(sets) as one:
        m = _run(one, kind, sets, R)
        want = _outputs(one, m)
    with MultiBatchEngine(sets, devices=devices if devices is not None else _devices(slots)) as mb:
        assert mb.n_devices == slots
        m = _run(mb, kind, sets, R)
        got = _outputs(mb, m)
    _assert_equal(got, want, len(sets))


@pytest.mark.parametrize("kind", list(KINDS))
@pytest.mark.parametrize("R", [1, 3])
@pytest.mark.parametrize("slots", [1, 2, 3, 8])
def test_every_output_equals_one_device_batch(kind, R, slots):
    _check_identity(_sets(KINDS[kind][3]), kind, slots, R)


def test_both_samplers_in_turn_on_one_object():
    """SiteSampler -> MotifSampler m = 2 -> m = 1 -> SiteSampler on one MultiBatchEngine, each against a fresh BatchEngine."""
    sets = _sets(False)
    with MultiBatchEngine(sets, devices=_devices(3)) as mb:
        for kind in ("site_fixed", "motif2_data", "motif1_fixed", "site_data"):
            m = _run(mb, kind, sets, 2)
            got = _outputs(mb, m)
            with BatchEngine(sets) as one:
                m = _run(one, kind, sets, 2)
                want = _outputs(one, m)
            _assert_equal(got, want, len(sets))


@pytest.mark.parametrize("kind", ["site_fixed", "motif1_data", "motif2_fixed"])
def test_more_slots_than_sets_and_a_single_set(kind):
    sets = _sets(False)[:3]
    with MultiBatchEngine(sets, devices=_devices(5)) as mb:
        assert mb.slot_sets() == [(0, 1), (1, 1), (2, 1), (3, 0), (3, 0)]
    _check_identity(sets, kind, 5, 2)
    _check_identity(sets[1:2], kind, 4, 3)


def test_sampler_wrappers_take_a_multi_device_engine():
    sets = _sets(True)
    with MultiBatchEngine(sets, devices=_devices(3)) as mb:
        got = SiteSampler.getMotifsWithBestInformationContentOfSets(2, K, 1e-4, list("ACGT"), sets, engine=mb, seed=9)
        got_m = MotifSampler.getMotifsWithBestInformationContentsOfSets(2, 1, K, 1e-4, 1.0, list("ACGT"), sets, engine=mb, seed=9)
    assert got == SiteSampler.getMotifsWithBestInformationContentOfSets(2, K, 1e-4, list("ACGT"), sets, seed=9)
    assert got_m == MotifSampler.getMotifsWithBestInformationContentsOfSets(2, 1, K, 1e-4, 1.0, list("ACGT"), sets, seed=9)
    acgt = _sets(False)
    with MultiBatchEngine(acgt, devices=_devices(2)) as mb:
        got2 = MotifSampler.getMotifsWithBestInformationContentsOfSets(1, 2, K, 1e-4, 1.0, list("ACGT"), acgt, engine=mb, seed=3)
    assert got2 == MotifSampler.getMotifsWithBestInformationContentsOfSets(1, 2, K, 1e-4, 1.0, list("ACGT"), acgt, seed=3)


def test_many_small_sets_on_eight_slots():
    """4096 sets x 20 sequences x 100 bp over 8 slots: a sample of sets against single-set handles."""
    k, R, S = 8, 2, 4096
    sets = [planted_motif_set(20, 100, k, seed=5000 + s).sequences() for s in range(S)]
    bgs = [_bg(s) for s in sets]
    with MultiBatchEngine(sets, devices=_devices(8)) as mb:
        assert [n for _, n in mb.slot_sets()] == [512] * 8   # equal shapes: equal blocks
        mb.run_device(make_params(k, 1e-4, 4, bgs[0]), R, bg_per_set=bgs, chain_id_base=11, seed=3)
        got = mb.fetch()
        best = mb.fetch_best(R - 1)
    assert len(best) == S
    for s in (0, 1, 511, 512, 2047, 2048, 3583, S - 1):
        with GibbsEngine(sets[s]) as eng:
            want = eng.run(make_params(k, 1e-4, 4, bgs[s]), R, chain_id_base=11, seed=3, want_counts=False)
        assert np.array_equal(got.sites[s], want.sites) and _same_bits(got.scores[s], want.scores), s
        assert _same_bits(got.sums[s], want.sums), s


def _optimum(cost, slots):
    """least largest block cost over all splits of cost into at most `slots` contiguous blocks (brute force)"""
    n, best = len(cost), None
    for cuts in range(min(slots, n)):
        for at in itertools.combinations(range(1, n), cuts):
            edges = (0,) + at + (n,)
            worst = max(sum(cost[a:b]) for a, b in zip(edges, edges[1:]))
            best = worst if best is None else min(best, worst)
    return best


def test_partition_is_contiguous_optimal_and_deterministic():
    rng = np.random.default_rng(42)
    for trial in range(24):
        n_sets = int(rng.integers(1, 10))
        slots = int(rng.integers(1, 6))
        sets = [[b"ACGT" * int(rng.integers(2, 30)) for _ in range(int(rng.integers(1, 4)))] for _ in range(n_sets)]
        cost = [sum(len(q) for q in s) for s in sets]
        seen = []
        for _ in range(2):
            with MultiBatchEngine(sets, devices=_devices(slots)) as mb:
                seen.append(mb.slot_sets())
        assert seen[0] == seen[1], trial
        blocks = seen[0]
        assert len(blocks) == slots
        nxt = 0
        for first, n in blocks:
            if n:
                assert first == nxt, (trial, blocks)
                nxt += n
        assert nxt == n_sets, (trial, blocks)
        assert sum(1 for _, n in blocks if n) == min(slots, n_sets), (trial, blocks)   # empty only for want of sets
        assert max(sum(cost[f:f + n]) for f, n in blocks if n) == _optimum(cost, slots), (trial, cost, blocks)


def _error(call):
    try:
        call()
    except _abi.GibbsError as e:
        return type(e), e.code, str(e)
    return None


def test_errors_name_the_global_set_and_leave_the_object_usable():
    good = [planted_motif_set(5, 40, K, seed=1).sequences(), planted_motif_set(3, 30, K, seed=2).sequences(),
            planted_motif_set(4, 50, K, seed=3).sequences()]
    short = [b"ACGTACGTAC", b"ACG", b"ACGTACGTACGT"]
    gapped = [b"ACGT-ACGTACGT", b"TTTTACGTAGGA"]
    motif = lambda bg, m=1, alen=4, background=FIXED: make_params(K, 1e-4, alen, bg, cutoff=1.0, sampler=MOTIF, motif_amount=m,
                                                                background=background)
    site = lambda alen=4, background=FIXED: make_params(K, 1e-4, alen, [0.25] * 4, background=background)
    cases = [  # (sets, the failing call on an engine)
        (good + [short], lambda e: e.run_device(site(), 2)),
        (good + [short], lambda e: e.run_motif_device(motif([0.25] * 4), 2)),
        (good + [gapped], lambda e: e.run_device(site(alen=5), 2)),
        (good + [gapped], lambda e: e.run_motif_device(motif([0.25] * 4, alen=5), 2)),
        (good + [gapped], lambda e: e.run_motif_device(motif([0.25] * 4, m=2, background=DATA), 2)),
        (good + [gapped], lambda e: e.run_motif_device(motif([0.25] * 4, m=3), 2)),
        (good + [gapped], lambda e: e.run_device(site(), 2, bg_per_set=[[0.25] * 4] * 3 + [[0.0, 0.5, 0.25, 0.25]])),
        (good + [gapped], lambda e: e.run_device(site(), 0)),
        (good + [gapped], lambda e: e.run_motif_device(site(), 2)),
    ]
    for sets, call in cases:
        with BatchEngine(sets) as one:
            want = _error(lambda: call(one))
        assert want is not None
        with MultiBatchEngine(sets, devices=_devices(3)) as mb:
            assert [f for f, n in mb.slot_sets() if f <= 3 < f + n][0] > 0   # the failing set lies on a later slot
            assert mb._lib.gibbs_multi_batch_fetch(mb._b, None, None, None, None) == _abi.GIBBS_ERR_ARG   # no run yet
            assert _error(lambda: call(mb)) == want
            # still usable: a valid run (k = 3 fits the short set too) equals the one-device batch
            bgs = [_bg(s) for s in sets]
            mb.run_device(make_params(3, 1e-4, 4, bgs[0]), 2, bg_per_set=bgs, chain_id_base=4, seed=6)
            got = mb.fetch()
            assert _error(lambda: call(mb)) == want
            with pytest.raises(_abi.GibbsArgumentError):
                mb.fetch()                       # the failed run left nothing to fetch
        with BatchEngine(sets) as one:
            one.run_device(make_params(3, 1e-4, 4, bgs[0]), 2, bg_per_set=bgs, chain_id_base=4, seed=6)
            ref = one.fetch()
        for s in range(len(sets)):
            assert np.array_equal(got.sites[s], ref.sites[s]) and _same_bits(got.scores[s], ref.scores[s])


def test_create_errors_name_the_global_set():
    good = [planted_motif_set(5, 40, K, seed=1).sequences(), planted_motif_set(3, 30, K, seed=2).sequences()]
    for bad in ([b"ACGTACGT", b"ACG#TT"], [b"ACGTACGT", b"acgt"]):
        sets = good + [good[0], bad]
        with pytest.raises(_abi.GibbsSymbolError) as one:
            BatchEngine(sets)
        with pytest.raises(_abi.GibbsSymbolError) as multi:
            MultiBatchEngine(sets, devices=_devices(3))
        assert str(multi.value) == str(one.value) and "set 3, sequence 1" in str(one.value)


def test_roulette_error_names_the_lowest_failing_global_set():
    """a held-out sequence whose every window holds a symbol outside the alphabet has no background mass under a fixed pcv:
    the pick runs past the list (fs:753); fetch names the lowest failing set, the object stays usable"""
    k = 4
    good = planted_motif_set(5, 40, k, seed=3).sequences()
    bad = good[:3] + [b"NNNNNNNNNNNN"]
    params = make_params(k, 1e-4, 4, [0.25] * 4, cutoff=0.0, sampler=MOTIF)
    sets = [good, good, good, bad, good, bad]
    with BatchEngine(sets) as one:
        one.run_motif_device(params, 2, chain_id_base=0, seed=1)
        want = _error(one.fetch)
    assert want is not None and "set 3" in want[2]
    with MultiBatchEngine(sets, devices=_devices(3)) as mb:
        assert [f for f, _ in mb.slot_sets()] == [0, 2, 4]
        mb.run_motif_device(params, 2, chain_id_base=0, seed=1)
        assert _error(mb.fetch) == want
        assert _error(lambda: mb.fetch_best(1)) == want
        with pytest.raises(_abi.GibbsArgumentError):
            mb.fetch_best_positions(1)       # no successful fetch_best
        mb.run_motif_device(params, 2, chain_id_base=0, seed=1)
        assert _error(lambda: mb.fetch_best(1)) == want
    with MultiBatchEngine([good] * 6, devices=_devices(3)) as mb:
        mb.run_motif_device(params, 2, chain_id_base=0, seed=1)
        got = mb.fetch()
    with GibbsEngine(good) as eng:
        ref = eng.run(params, 2, chain_id_base=0, seed=1, want_counts=False)
    for s in range(6):
        assert np.array_equal(got.sites[s], ref.sites)


def test_distinct_gpus():
    ndev = device_count()
    if ndev < 2:
        pytest.skip("needs at least two GPUs")
    sets = _sets(True)
    for kind in ("site_fixed", "motif1_data"):
        _check_identity(sets, kind, ndev, 3, devices=list(range(ndev)))
    _check_identity(_sets(False), "motif2_fixed", min(ndev, 8), 3, devices=list(range(min(ndev, 8))))
    with MultiBatchEngine(sets) as mb:   # n_devices = 0: every visible device
        assert mb.n_devices == ndev
