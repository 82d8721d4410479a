"""Gap '-' as a member of the alphabet (the script's dnaBases, fsx:368-369) under the SiteSampler with the data-derived
background (doSiteSampling fs:697, getBestPWMSs fs:462-479): Gap has its own PPM row (fs:255-261), a window over it
multiplies P[Gap, j] / q_w[Gap] in (fs:282-293), the other sequences' Gaps stay in the fused background (fs:67-69), and
every denominator of a gapped set -- gap-free rows included -- holds f0[Gap]. GPU vs the oracle with alphabet b"ATGC-"."""
import numpy as np
import pytest

import oracle_lib as O
from gibbssampling_b200 import SiteSampler, _abi
from gibbssampling_b200.engine import (BatchEngine, GibbsEngine, MultiBatchEngine, MultiEngine, device_count,
                                       draws_per_chain, make_params)
from gibbssampling_b200.synthetic import planted_motif_set

pytestmark = pytest.mark.gpu

RTOL = 1e-5
ALPHA = b"ATGC-"
DNA = list("ATGC-")
DATA = _abi.GIBBS_BG_DATA

# consensus rows of the reference script's gap-padded alignment (fsx:81-127), as in test_position_matrix.py
ALIGNED = [b"---ATGCATGCAAAAGTTGCA-AT--", b"--GATGCATGCAAAAGTTGCATAT--", b"----TGCATGCATAAGTTGCATATG-",
           b"-TGATGC-TGCAAAAGTTGCATAT--", b"---ATGCATGCAAAACTTGCATAT-A", b"--GATGCATGGAAAAGTTGCATATG-"]


def _gapped(seed, n, lo, hi, p_gap, extra="", p_extra=0.0, pad=0):
    """Random rows with Gaps (sparse, and runs of up to `pad` at both ends like an alignment) and other symbols."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        L = int(rng.integers(lo, hi + 1))
        s = rng.choice(list("ACGT"), size=L)
        s[rng.random(L) < p_gap] = "-"
        if extra:
            m = rng.random(L) < p_extra
            s[m] = rng.choice(list(extra), size=int(m.sum()))
        if pad:
            a, b = int(rng.integers(0, pad + 1)), int(rng.integers(0, pad + 1))
            s[:a] = "-"
            if b:
                s[L - b:] = "-"
        out.append("".join(s).encode())
    return out


def _same(got_sites, got_scores, want_scores, want_sites, msg=""):
    assert np.asarray(got_sites).tolist() == np.asarray(want_sites).tolist(), msg
    got, want = np.asarray(got_scores, dtype=np.float64), np.asarray(want_scores, dtype=np.float64)
    assert np.array_equal(np.isneginf(got), np.isneginf(want)), msg   # -inf only where the oracle has it
    np.testing.assert_allclose(got, want, rtol=RTOL, err_msg=msg)


def _params(k, pc, **kw):
    return make_params(k, pc, 5, [0.25] * 4, background=DATA, **kw)


def _restarts(seqs, k, pc, chains=3, seed=7, base=20, team=None, exact=False):
    S = O.sources(seqs)
    with GibbsEngine(seqs) as eng:
        if team is not None:
            eng.set_team_warps(team)
        if exact:
            eng.set_option(_abi.GIBBS_OPT_EXACT_SCANS, 1)
        res = eng.run(_params(k, pc), chains, chain_id_base=base, seed=seed, want_counts=False)
        u = np.random.default_rng(seed).random((1, draws_per_chain(len(seqs))))
        inj = eng.run(_params(k, pc), 1, uniforms=u, want_counts=False)
    for c in range(chains):
        rng, _ = O.make_rng(seed=seed, chain=base + c)
        score, pos, _ = O.site_step("do_site_sampling", S, k, pc, rng=rng, alphabet=ALPHA)
        _same(res.sites[c], res.scores[c], score, pos, f"chain {c}")
    rng, _ = O.make_rng(uniforms=u[0])
    score, pos, _ = O.site_step("do_site_sampling", S, k, pc, rng=rng, alphabet=ALPHA)
    _same(inj.sites[0], inj.scores[0], score, pos, "injected")
    return res


SHAPES = {
    "sparse": (_gapped(1, 7, 30, 60, 0.05), 6, 1e-4),
    "alignment": (ALIGNED, 8, 1e-4),
    "padded_rows": (_gapped(2, 9, 40, 80, 0.01, pad=12), 7, 1e-4),
    "every_window_gapped": (_gapped(3, 6, 30, 50, 0.03) + [b"ACG-TAC-GTA-CGT-ACG-TAC-GT"], 5, 1e-4),
    "all_gap_but_k": (_gapped(4, 6, 30, 50, 0.05) + [b"------ACGTAC-------"], 6, 1e-4),
    "gap_next_to_N_and_star": (_gapped(5, 8, 30, 60, 0.04, extra="N*", p_extra=0.04)
                               + [b"ACGTN-*-NACGTACGTAC-N*GTACG"], 6, 1e-4),
    "k1": (_gapped(6, 6, 12, 30, 0.1), 1, 1e-4),
    "k_odd": (_gapped(7, 8, 40, 70, 0.06, extra="N", p_extra=0.02), 11, 1e-2),
    "k32": (_gapped(8, 6, 60, 90, 0.04, pad=5), 32, 1.0),
    "ragged": (_gapped(9, 10, 15, 120, 0.05), 9, 1e-4),
    "pc0": (_gapped(10, 6, 30, 50, 0.08), 5, 0.0),
}


@pytest.mark.parametrize("shape", list(SHAPES))
def test_whole_restarts_match_oracle(shape):
    seqs, k, pc = SHAPES[shape]
    res = _restarts(seqs, k, pc)
    if pc == 0.0:
        assert res.stats["fast_path"] == 0


def test_gap_at_a_sites_first_and_last_column():
    """Start sites chosen so that a Gap sits at column 0 and at column k - 1: the own-site correction of the gap row."""
    k = 6
    seqs = [b"-CGTAC-GTACGT", b"ACGTA-ACGTAGC", b"TTGCA-CGTACCA", b"GGCAT-ACGT-AC", b"ACG-TACGTACGA"]
    start = np.array([0, 0, 5, 5, 3], dtype=np.int32)   # Gap at column 0 in rows 0, 2, 3, 4; at column 5 in rows 1, 3
    S = O.sources(seqs)
    scores0 = np.full(len(seqs), -50.0)
    with GibbsEngine(seqs) as eng:
        for mask, name in ((_abi.PHASE_GREEDY, "best_pwms_with_start_positions"), (_abi.PHASE_LEFT, "left_shifted"),
                           (_abi.PHASE_RIGHT, "right_shifted")):
            for team in (1, 4):
                eng.set_team_warps(team)
                eng.set_start_state(start, scores0)
                got = eng.run(_params(k, 1e-4, phase_mask=mask), 1, want_counts=False)
                score, pos, _ = O.site_step(name, S, k, 1e-4, state=(scores0, start), alphabet=ALPHA)
                _same(got.sites[0], got.scores[0], score, pos, f"{name} team {team}")


@pytest.mark.parametrize("shape", ["sparse", "alignment", "gap_next_to_N_and_star", "k_odd"])
def test_phases_alone_match_oracle(shape):
    seqs, k, pc = SHAPES[shape]
    n = len(seqs)
    S = O.sources(seqs)
    u = np.random.default_rng(11).random((1, draws_per_chain(n)))
    with GibbsEngine(seqs) as eng:
        got = eng.run(_params(k, pc, phase_mask=_abi.PHASE_INIT), 1, uniforms=u, want_counts=False)
        rng, _ = O.make_rng(uniforms=u[0])
        score, pos, _ = O.site_step("random_starts", S, k, pc, rng=rng, alphabet=ALPHA)
        _same(got.sites[0], got.scores[0], score, pos, "random_starts")
        state = (score, pos)
        for mask, name in ((_abi.PHASE_GREEDY, "best_pwms_with_start_positions"), (_abi.PHASE_LEFT, "left_shifted"),
                           (_abi.PHASE_RIGHT, "right_shifted")):
            eng.set_start_state(state[1], state[0])
            got = eng.run(_params(k, pc, phase_mask=mask), 1, want_counts=False)
            score, pos, _ = O.site_step(name, S, k, pc, state=state, alphabet=ALPHA)
            _same(got.sites[0], got.scores[0], score, pos, name)
            state = (score, pos)


def test_script_call_on_a_gap_padded_alignment():
    """doSiteSampling and getMotifsWithBestInformationContent with list("ATGC-") over the alignment rows (fsx:384)."""
    seqs, k, pc = SHAPES["alignment"]
    S = O.sources(seqs)
    got = SiteSampler.doSiteSampling(k, pc, DNA, seqs, seed=3, chain=1)
    rng, _ = O.make_rng(seed=3, chain=1)
    score, pos, _ = O.site_step("do_site_sampling", S, k, pc, rng=rng, alphabet=ALPHA)
    _same([p for _, p in got], [s for s, _ in got], score, pos)
    for reps in (1, 4):
        got = SiteSampler.getMotifsWithBestInformationContent(reps, k, pc, DNA, seqs, seed=2024, chain=3)
        rng, _ = O.make_rng(seed=2024, chain=3)
        ws, wp, _ = O.best_information_content(1, reps, S, k, pc, rng, alphabet=ALPHA)
        _same([p for _, p in got], [s for s, _ in got], ws, wp, f"reps {reps}")


def test_fast_path_agrees_with_the_exact_scan():
    """Team sizes and GIBBS_OPT_EXACT_SCANS give identical output. Most rows hold no Gap and take the ranking pass, so its
    float32 key and float64 re-scoring both see f0[Gap]."""
    ps = planted_motif_set(60, 200, 10, seed=5)
    seqs = list(ps.sequences())
    for i in range(0, 60, 7):   # one row in seven gapped
        s = bytearray(seqs[i])
        for j in range(3, len(s), 23):
            s[j] = ord("-")
        seqs[i] = bytes(s)
    params = _params(10, 1e-4)
    out = []
    with GibbsEngine(seqs) as eng:
        for team, exact in ((0, 0), (1, 0), (4, 0), (8, 0), (16, 0), (0, 1)):
            eng.set_team_warps(team)
            eng.set_option(_abi.GIBBS_OPT_EXACT_SCANS, exact)
            out.append(eng.run(params, 6, chain_id_base=3, seed=9, want_counts=False))
    assert out[0].stats["fast_path"] == 1 and out[-1].stats["fast_path"] == 0
    assert out[0].stats["exact_rescans"] < out[0].stats["site_updates"]
    for r in out[1:]:
        assert r.sites.tolist() == out[0].sites.tolist()
        assert r.scores.tobytes() == out[0].scores.tobytes() and r.sums.tobytes() == out[0].sums.tobytes()
    S = O.sources(seqs)
    rng, _ = O.make_rng(seed=9, chain=3)
    score, pos, _ = O.site_step("do_site_sampling", S, 10, 1e-4, rng=rng, alphabet=ALPHA)
    _same(out[0].sites[0], out[0].scores[0], score, pos)


def _batch_sets():
    return [SHAPES["sparse"][0], planted_motif_set(5, 40, 6, seed=1).sequences(), SHAPES["alignment"][0][:4] + [b"ACGTACGTACGT"],
            _gapped(21, 3, 20, 30, 0.1), _gapped(22, 12, 30, 60, 0.03, extra="N", p_extra=0.02)]


def test_batch_equals_single_handles():
    sets, k, R = _batch_sets(), 6, 3
    params = _params(k, 1e-4)
    with BatchEngine(sets) as b:
        b.run_device(params, R, chain_id_base=5, seed=13)
        got = b.fetch()
    for s, seqs in enumerate(sets):
        with GibbsEngine(seqs) as eng:
            want = eng.run(params, R, chain_id_base=5, seed=13, want_counts=False)
        assert got.sites[s].tolist() == want.sites.tolist(), s
        assert got.scores[s].tobytes() == want.scores.tobytes() and got.sums[s].tobytes() == want.sums.tobytes(), s


def test_multi_batch_and_multi_engine_equal_one_device():
    sets, k, R = _batch_sets(), 6, 3
    params = _params(k, 1e-4)
    with BatchEngine(sets) as b:
        b.run_device(params, R, chain_id_base=5, seed=13)
        want = b.fetch()
        want_best = b.fetch_best(R - 1, want_counts=True)
    with MultiBatchEngine(sets, devices=[0, 0]) as mb:
        mb.run_device(params, R, chain_id_base=5, seed=13)
        got = mb.fetch()
        got_best = mb.fetch_best(R - 1, want_counts=True)
    for s in range(len(sets)):
        assert got.sites[s].tolist() == want.sites[s].tolist(), s
        assert got.scores[s].tobytes() == want.scores[s].tobytes(), s
        assert got_best[s].sites.tolist() == want_best[s].sites.tolist() and got_best[s].restart == want_best[s].restart
        assert got_best[s].counts.tolist() == want_best[s].counts.tolist()
    seqs = sets[0]
    ndev = device_count()
    with GibbsEngine(seqs) as eng:
        res = eng.run(params, 7, chain_id_base=2, seed=4, want_counts=False)
        one = eng.fetch_best(6, want_counts=True)
    with MultiEngine(seqs, devices=[i % ndev for i in range(3)]) as m:
        m.run_device(params, 7, chain_id_base=2, seed=4)
        best = m.fetch_best(6, want_counts=True)
    assert best.sites.tolist() == one.sites.tolist() and best.scores.tobytes() == one.scores.tobytes()
    assert best.restart == one.restart and best.counts.tolist() == one.counts.tolist()
    assert best.stats["site_updates"] == res.stats["site_updates"]


def test_full_size_gapped_set():
    """C2's shape (1000 x 500, k 12) with gap-padded rows, a few chains against the oracle's fast pipeline."""
    ps = planted_motif_set(1000, 500, 12, seed=2)
    rng = np.random.default_rng(2)
    seqs = []
    for s in ps.sequences():
        s = bytearray(s)
        a, b = int(rng.integers(0, 40)), int(rng.integers(0, 40))
        s[:a] = b"-" * a
        if b:
            s[len(s) - b:] = b"-" * b
        seqs.append(bytes(s))
    S = O.sources(seqs)
    with GibbsEngine(seqs) as eng:
        res = eng.run(_params(12, 1e-4), 3, chain_id_base=0, seed=17, want_counts=False)
    scores, pos, sums, _ = O.fast_site_chains(1, S, 12, 1e-4, seed=17, chain_base=0, n_chains=3, threads=8, alphabet=ALPHA)
    for c in range(3):
        _same(res.sites[c], res.scores[c], scores[c], pos[c], f"chain {c}")


@pytest.mark.parametrize("case", range(40))
def test_fuzz_against_oracle(case):
    rng = np.random.default_rng(9000 + case)
    n, k = int(rng.integers(2, 10)), int(rng.integers(1, 14))
    pc = float(rng.choice([1e-4, 1e-2, 1.0]))
    seqs = _gapped(100 + case, n, k, k + int(rng.integers(0, 60)), float(rng.choice([0.02, 0.1, 0.3])),
                   extra=str(rng.choice(["", "N", "N*R"])), p_extra=0.03, pad=int(rng.integers(0, 6)))
    _restarts(seqs, k, pc, chains=2, seed=case, team=int(rng.choice([1, 4])))


def test_refusals_that_stay():
    seqs = SHAPES["sparse"][0]
    with GibbsEngine(seqs) as eng:
        with pytest.raises(_abi.GibbsUnsupportedError):   # the MotifSampler has no Gap row, under either background
            eng.run(make_params(6, 1e-4, 5, [0.25] * 4, background=DATA, sampler=_abi.GIBBS_MOTIF_SAMPLER, cutoff=1.0), 1)
        with pytest.raises(_abi.GibbsUnsupportedError):   # the fixed background has no pcv.[Gap]
            eng.run(make_params(6, 1e-4, 5, [0.25] * 4), 1)
        eng.set_start_ppm(np.full((6, 4), 0.25))           # a start PPM has rows A,C,G,T only
        with pytest.raises(_abi.GibbsUnsupportedError):
            eng.run(_params(6, 1e-4), 1)
        eng.run(make_params(6, 1e-4, 4, [0.25] * 4, background=DATA), 1)   # alphabet of 4: Gap is a dead symbol
        eng.set_start_ppm(None)
        eng.run(_params(6, 1e-4), 1)
    with BatchEngine([seqs, seqs]) as b:
        with pytest.raises(_abi.GibbsUnsupportedError):
            b.run_motif_device(make_params(6, 1e-4, 5, [0.25] * 4, background=DATA, sampler=_abi.GIBBS_MOTIF_SAMPLER,
                                           cutoff=1.0), 1)
