"""The run counters of the SiteSampler (gibbs_run_stats). Every sweep commits every sequence exactly once and a chain pauses
only at a sweep boundary, so over a whole run site_updates = sweeps * N and window_scores = sweeps * sum_n (len_n - k + 1),
whatever the team size, the hand-over stages, the cluster stages or the random-start path. exact_rescans counts the
committed updates that scored every window in float64: the committed updates are the reference's sequential sweep, so it
does not depend on how the chains were run either. speculative_discards depends on the team, not on which chains share a
launch."""
import numpy as np
import pytest

from gibbssampling_b200 import _abi
from gibbssampling_b200.engine import BatchEngine, GibbsEngine, make_params
from gibbssampling_b200.synthetic import background_of, planted_motif_set

pytestmark = pytest.mark.gpu


def _many_chains():
    """more than GIBBS_OPT_STAGE2_AT = 4 chains per SM of a B200 (148 SMs): the run starts on the 4-warp stage and hands
    its stragglers over to the 8-warp, 16-warp and cluster stages"""
    return 4 * 148 + 40


def _ragged(n, L, k, seed):
    """n sequences of k .. L bp; the first rows hold exactly one window (length k) or two"""
    ps = planted_motif_set(n, L, k, seed=seed, min_length=k)
    seqs = ps.sequences()
    seqs[0], seqs[3], seqs[7] = seqs[0][:k], seqs[3][:k + 1], seqs[7][:k]
    return seqs


def _check_per_sweep(seqs, k, stats):
    n = len(seqs)
    sum_w = sum(len(s) - k + 1 for s in seqs)
    assert stats["sweeps"] > 0
    assert stats["site_updates"] == stats["sweeps"] * n
    assert stats["window_scores"] == stats["sweeps"] * sum_w


SHAPES = [(70, 120, 9), (40, 300, 12), (33, 90, 20)]


@pytest.mark.parametrize("n,L,k", SHAPES, ids=lambda v: str(v))
def test_counters_per_sweep_for_every_team(n, L, k):
    seqs = _ragged(n, L, k, seed=500 + n)
    params = make_params(k, 1e-4, 5, background_of(np.frombuffer(b"".join(seqs), dtype=np.uint8), 1e-4, 5))
    chains = 96
    with GibbsEngine(seqs) as eng:
        eng.set_option(_abi.GIBBS_OPT_CLUSTER, 0)
        eng.set_team_warps(1)
        ref = eng.run(params, chains, chain_id_base=7, seed=31, want_counts=False)
        _check_per_sweep(seqs, k, ref.stats)
        assert ref.stats["speculative_discards"] == 0   # one warp never speculates
        for team in (4, 8, 16):
            eng.set_team_warps(team)
            got = eng.run(params, chains, chain_id_base=7, seed=31, want_counts=False)
            assert got.sites.tobytes() == ref.sites.tobytes(), team
            _check_per_sweep(seqs, k, got.stats)
            assert got.stats["sweeps"] == ref.stats["sweeps"], team
            assert got.stats["exact_rescans"] == ref.stats["exact_rescans"], team
            # a chain's discards depend on its team only: the same chains in two launches add up to one launch
            lo = eng.run(params, 40, chain_id_base=7, seed=31, want_counts=False).stats
            hi = eng.run(params, chains - 40, chain_id_base=47, seed=31, want_counts=False).stats
            assert lo["speculative_discards"] + hi["speculative_discards"] == got.stats["speculative_discards"], team
            assert lo["exact_rescans"] + hi["exact_rescans"] == ref.stats["exact_rescans"], team
        # every window in float64: each committed update is an exact rescan
        eng.set_option(_abi.GIBBS_OPT_EXACT_SCANS, 1)
        for team in (1, 4, 8, 16):
            eng.set_team_warps(team)
            got = eng.run(params, chains, chain_id_base=7, seed=31, want_counts=False)
            assert got.sites.tobytes() == ref.sites.tobytes(), team
            _check_per_sweep(seqs, k, got.stats)
            assert got.stats["exact_rescans"] == got.stats["site_updates"], team


@pytest.mark.parametrize("cluster", [0, 4, 8])
@pytest.mark.parametrize("seq_sweeps", [0, 2])
def test_counters_per_sweep_across_hand_overs(cluster, seq_sweeps):
    """automatic stages: chains pause at sweep boundaries and resume on wider teams, the one-warp first sweeps and the
    cluster stages included (which sweeps a chain runs on which team depends on when the others finish, so
    speculative_discards is not compared here)"""
    n, L, k = 130, 110, 12
    seqs = _ragged(n, L, k, seed=77)
    params = make_params(k, 1e-4, 5, background_of(np.frombuffer(b"".join(seqs), dtype=np.uint8), 1e-4, 5))
    chains = _many_chains()
    with GibbsEngine(seqs) as eng:
        eng.set_option(_abi.GIBBS_OPT_CLUSTER, 0)
        eng.set_team_warps(1)
        ref = eng.run(params, chains, seed=8, want_counts=False)
        eng.set_team_warps(0)
        eng.set_option(_abi.GIBBS_OPT_CLUSTER, cluster)
        eng.set_option(_abi.GIBBS_OPT_SEQ_SWEEPS, seq_sweeps)
        got = eng.run(params, chains, seed=8, want_counts=False)
    assert got.stats["kernel_launches"] > 2   # the chains were handed over at least once
    assert got.sites.tobytes() == ref.sites.tobytes()
    _check_per_sweep(seqs, k, got.stats)
    assert got.stats["sweeps"] == ref.stats["sweeps"]
    assert got.stats["exact_rescans"] == ref.stats["exact_rescans"]


@pytest.mark.parametrize("init_path", [_abi.GIBBS_INIT_CHAIN, _abi.GIBBS_INIT_WIDE, _abi.GIBBS_INIT_SMEM])
@pytest.mark.parametrize("background", [_abi.GIBBS_BG_FIXED, _abi.GIBBS_BG_DATA])
def test_counters_per_sweep_for_the_random_starts(init_path, background):
    """the random-start sweep counts one sweep per chain, on the chain's own team (INIT_ONLY) as on the grid-wide paths;
    a run without sweeps after it counts that sweep alone"""
    n, L, k = 60, 150, 10
    seqs = _ragged(n, L, k, seed=11)
    bg = background_of(np.frombuffer(b"".join(seqs), dtype=np.uint8), 1e-4, 5)
    chains = 200
    with GibbsEngine(seqs) as eng:
        eng.set_option(_abi.GIBBS_OPT_INIT_PATH, init_path)
        for mask, sweeps in ((_abi.PHASE_INIT, chains), (0, None)):
            got = eng.run(make_params(k, 1e-4, 5, bg, background=background, phase_mask=mask), chains, seed=3, want_counts=False)
            _check_per_sweep(seqs, k, got.stats)
            if init_path == _abi.GIBBS_INIT_CHAIN:
                assert got.stats["init_path"] == _abi.GIBBS_INIT_CHAIN
            if sweeps is not None:
                assert got.stats["sweeps"] == sweeps
                assert got.stats["speculative_discards"] == 0


def test_counters_per_sweep_for_a_batch_of_equal_sets():
    """every set of a batch runs the same sweeps body on its own rows: with sets of one shape the totals are per sweep too,
    and exact_rescans is the sum over single-set handles"""
    n, L, k, R = 24, 100, 8, 5
    base = _ragged(n, L, k, seed=900)
    sets = [[s[j % len(s):] + s[:j % len(s)] for s in base] for j in range(6)]   # rotated rows: one length profile
    bgs = [background_of(np.frombuffer(b"".join(x), dtype=np.uint8), 1e-4, 5) for x in sets]
    params = make_params(k, 1e-4, 5, bgs[0])
    with BatchEngine(sets) as b:
        b.run_device(params, R, bg_per_set=bgs, chain_id_base=2, seed=12)
        got = b.fetch()
    _check_per_sweep(sets[0], k, got.stats)
    rescans = 0
    for x, bg in zip(sets, bgs):
        with GibbsEngine(x) as eng:
            rescans += eng.run(make_params(k, 1e-4, 5, bg), R, chain_id_base=2, seed=12, want_counts=False).stats["exact_rescans"]
    assert got.stats["exact_rescans"] == rescans
