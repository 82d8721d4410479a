"""The MotifSampler's roulette pick (fs:746-754) at the edges where an approximate pick can go wrong.

The stochastic sweep (fs:828-853, fs:935-970) decides most picks from coarse logarithms (motif_stoch_fast,
gibbs_motif.cuh): each gated window's log2 score is estimated, the estimates decide `PWMS > cutOff` (fs:735) and a
warp prefix sum over them locates the bucket of the pick; the exact sequential walk runs only when an estimate lies
near the cut-off or the pick near a bucket edge. gibbs_pick_roulette goes through motif_roulette instead (a float64
scan with its own edge check, then the exact walk). Both are compared here with the oracle where those checks are
tightest:

- cut-offs at a window's own PWMS, one ulp and 1e-11 either side of it and 1e-9 below it, at scores up to 2^7
  where the rounding of a float logarithm is largest;
- picks on the edges of the exact walk's buckets and one ulp, 1e-12 and 1e-9 either side of them, on short, long and
  equal-weight lists and on scores in [128, 256), and past the end of the mass (the reference throws);
- the same edges for motifAmount = 2 (singles and pairs, motif2_kernel's sequential walk).

The tests without the gpu mark check the constructions with the oracle alone: that each window is in or out of the
list as intended, that each pick lands in the bucket it was built for, and that the chosen windows are the ones where
a float32 sum of exponent and logarithm misses log2 by more than the fast path's tolerance (an emulation: numpy's
float32 log2 stands in for the GPU's approximate one)."""
import math

import numpy as np
import pytest

import oracle_lib as O
from gibbssampling_b200 import _abi
from gibbssampling_b200.engine import GibbsEngine, make_params
from gibbssampling_b200.synthetic import background_of, planted_motif_set

RTOL = 1e-5
ALPHABET_SIZE = 5          # A,T,G,C,Gap
TEAMS = [1, 4, 8, 16]
TOL = 1e-6                 # motif_stoch_fast: an estimate within TOL of the cut-off is undecided
BIG_ERROR = 1.5e-6         # TOL + the GPU logarithm's own error (2^-21.4), which the emulation does not model
SKEWED = [0.05, 0.95 / 3, 0.95 / 3, 0.95 / 3]


# ---------------------------------------------------------------------------------------------------------------------
# helpers (CPU)
# ---------------------------------------------------------------------------------------------------------------------
def coarse_log2_float32(s: float) -> float:
    """Emulation of the float32 estimate `(float)e + log2f(m)` of log2(s): s = m * 2^e, m in [1, 2) rounded to float,
    the sum rounded to float. Correctly rounded float32 log2 stands in for the GPU's __log2f."""
    m, e = math.frexp(s)
    lg = np.log2(np.float32(m * 2.0))
    return float(np.float32(np.float32(e - 1) + lg))


def walk_edges(weights):
    """Bucket edges of the exact walk (fs:746-754): sum from 0.0 in list order, w = v / sum, bucket i = [acc, acc + w]
    with both bounds inclusive (the first bucket that holds the pick wins). Returns (lo, hi) lists."""
    total = 0.0
    for v in weights:
        total = total + v
    lo, hi, acc = [], [], 0.0
    for v in weights:
        nxt = acc + v / total
        lo.append(acc)
        hi.append(nxt)
        acc = nxt
    return lo, hi


def walk_pick(weights, u):
    """Index the exact walk picks, or None where the reference throws."""
    lo, hi = walk_edges(weights)
    for i, (a, b) in enumerate(zip(lo, hi)):
        if a <= u <= b:
            return i
    return None


def oracle_pick(weights, u):
    try:
        return O.roulette(weights, u)
    except O.OracleError as e:
        assert e.code == O.ERR_ROULETTE
        return None


def edge_picks(e):
    """Picks on and around an edge: the edge, one ulp either side, 1e-12 and 1e-9 either side."""
    return [e, math.nextafter(e, -1.0), math.nextafter(e, 2.0), e - 1e-12, e + 1e-12, e - 1e-9, e + 1e-9]


def loo_ppm(seqs, state, h, k, pc):
    """Leave-one-out PPM of MotifIndex state [(pwms, [positions])] without sequence h (fs:794-808)."""
    pfm = np.zeros((O.NSLOT, k), np.int32)
    for i, (_, pl) in enumerate(state):
        if i != h:
            for p0 in pl:
                for j in range(k):
                    pfm[seqs[i][p0 + j] - 42, j] += 1
    return O.ppm_of_pfm(pfm, len(seqs) - 1, pc)


def lists_of(seqs, state, k, pc, cutoff, pcv49, m=1):
    """The reference's list (background entries ++ candidates) of every held-out sequence."""
    return [O.candidates(seqs[h], k, m, cutoff, pcv49, loo_ppm(seqs, state, h, k, pc)) for h in range(len(seqs))]


def oracle_sweep(variant, seqs, m, k, pc, cutoff, pcv49, state, picks):
    """One synchronous stochastic sweep of the oracle per row of picks; None where the reference throws."""
    S = O.sources(seqs)
    out = []
    for row in picks:
        rng, _keep = O.make_rng(uniforms=row)
        try:
            want, _ = O.motif_step("stochastic", variant, S, m, k, pc, cutoff, pcv=pcv49, state=state, rng=rng)
        except O.OracleError as e:
            assert e.code == O.ERR_ROULETTE
            want = None
        out.append(want)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# a) cut-offs at a window's own PWMS, large scores
# ---------------------------------------------------------------------------------------------------------------------
CUT_SHAPES = [(k, bg) for k in (12, 16, 20, 24, 32) for bg in ("sample", "skewed")]


def _cut_set(k, bg):
    ps = planted_motif_set(12, 200, k, seed=5, mutation=0.02)
    seqs = ps.sequences()
    bg4 = background_of(ps.ascii, 1e-4, ALPHABET_SIZE) if bg == "sample" else SKEWED
    state = [(1.0, [int(t)]) for t in ps.truth]
    return seqs, bg4, state


def cut_windows(k, bg):
    """Windows X (held-out h, position w, PWMS) of the planted start state with the largest emulated error of either sign."""
    seqs, bg4, state = _cut_set(k, bg)
    pcv49 = O.pcv_from_acgt(bg4)
    pc = 1e-4
    found = []
    for h in range(len(seqs)):
        ppm = loo_ppm(seqs, state, h, k, pc)
        raw = O.window_scores_bpv(seqs[h], k, pcv49, ppm)
        for w, s in enumerate(raw):
            if s > 1.0:
                pw = math.log(s) / math.log(2.0)                       # log2 as the reference takes it (fs:303)
                found.append((coarse_log2_float32(float(s)) - pw, h, w, pw))
    found.sort()
    picked = [found[0], found[-1]]
    return [(h, w, pw, err) for err, h, w, pw in picked]


def cut_offs(pw):
    return [pw, math.nextafter(pw, -math.inf), math.nextafter(pw, math.inf), pw + 1e-11, pw - 1e-11, pw - 1e-9]


def cut_picks(lists, x):
    """Rows of picks, one per held-out sequence: midpoints of the bucket of X (or the first candidate), the bucket after
    it, the last bucket, and the buckets that hold 0.5 and 0.999."""
    h_x, w_x = x
    rows = [[], [], [], [], []]
    for h, lst in enumerate(lists):
        wts = [v for v, _ in lst]
        lo, hi = walk_edges(wts)
        n_bg = sum(1 for _, p in lst if not p)
        at = next((i for i, (_, p) in enumerate(lst) if p == [w_x]), None) if h == h_x else None
        if at is None:
            at = n_bg if n_bg < len(lst) else len(lst) - 1
        for r, i in enumerate((at, min(at + 1, len(lst) - 1), len(lst) - 1, walk_pick(wts, 0.5), walk_pick(wts, 0.999))):
            rows[r].append(0.5 * (lo[i] + hi[i]))
    return np.array(rows)


def _cut_case(k, bg):
    seqs, bg4, state = _cut_set(k, bg)
    pcv49 = O.pcv_from_acgt(bg4)
    for h, w, pw, err in cut_windows(k, bg):
        for cutoff in cut_offs(pw):
            lists = lists_of(seqs, state, k, 1e-4, cutoff, pcv49)
            yield seqs, bg4, state, (h, w, pw, err), cutoff, lists, cut_picks(lists, (h, w))


@pytest.mark.parametrize("k,bg", CUT_SHAPES, ids=[f"k{k}_{bg}" for k, bg in CUT_SHAPES])
def test_cut_off_constructions(k, bg):
    for seqs, bg4, state, (h, w, pw, err), cutoff, lists, picks in _cut_case(k, bg):
        kept = any(p == [w] for _, p in lists[h])
        assert kept == (pw > cutoff)                                    # strict > (fs:735)
        want = oracle_sweep(0, seqs, 1, k, 1e-4, cutoff, O.pcv_from_acgt(bg4), state, picks)
        for r, row in enumerate(picks):
            for hh, u in enumerate(row):
                wts = [v for v, _ in lists[hh]]
                i = walk_pick(wts, u)
                assert i is not None and i == oracle_pick(wts, u)
                lo, hi = walk_edges(wts)
                assert lo[i] < u < hi[i]                                # a midpoint, clear of both edges
                assert want[r][hh] == lists[hh][i]


def test_cut_off_windows_miss_the_float32_estimate_by_more_than_the_tolerance():
    """Above 32 a float32 sum of exponent and logarithm rounds to 2^-19 and coarser: the chosen windows include ones
    whose estimate misses log2 by more than the fast path's tolerance in each direction, the ones that can flip it."""
    errs = [err for k, bg in CUT_SHAPES for _, _, pw, err in cut_windows(k, bg)]
    assert min(errs) <= -BIG_ERROR and max(errs) >= BIG_ERROR, errs
    assert sum(abs(e) >= BIG_ERROR for e in errs) >= 4, errs


def _sweep(eng, params, state, picks, m=1):
    """The synchronous stochastic sweep on the GPU from `state`, one chain per row of picks (draw N(N-1) + n)."""
    rows, n = picks.shape
    pos = np.full((n, m), -1, np.int32)
    for i, (_, pl) in enumerate(state):
        pos[i, :len(pl)] = pl
    pw = np.array([v for v, _ in state])
    eng.set_start_motif_state(np.tile(pos, (rows, 1, 1)), np.tile(pw, (rows, 1)))
    u = np.zeros((rows, n * (n - 1) + n))
    u[:, n * (n - 1):] = picks
    res = eng.run(params, rows, uniforms=u, want_counts=False)
    if m == 1:
        return [[(float(res.scores[r][i]), [int(res.sites[r][i])] if res.sites[r][i] >= 0 else []) for i in range(n)]
                for r in range(rows)]
    got = eng.fetch_positions(m)
    return [[(float(res.scores[r][i]), [int(p) for p in got[r][i] if p >= 0]) for i in range(n)] for r in range(rows)]


def _same(got, want, what):
    assert [p for _, p in got] == [p for _, p in want], what
    np.testing.assert_allclose([v for v, _ in got], [v for v, _ in want], rtol=RTOL, err_msg=str(what))


@pytest.mark.gpu
@pytest.mark.parametrize("k,bg", CUT_SHAPES, ids=[f"k{k}_{bg}" for k, bg in CUT_SHAPES])
def test_stochastic_sweep_at_the_cut_off(k, bg):
    """fs:735 keeps a window only when its PWMS is strictly above cutOff: the sweep must agree at the window's own PWMS,
    one ulp either side, 1e-11 either side and 1e-9 below, for every team size."""
    seqs, bg4, state = _cut_set(k, bg)
    with GibbsEngine(seqs) as eng:
        sites = np.array([p[0] for _, p in state], np.int32)
        prm = make_params(k, 1e-4, ALPHABET_SIZE, bg4, sampler=_abi.GIBBS_MOTIF_SAMPLER)
        for h, w, pw, _ in cut_windows(k, bg):   # the one-ulp cut-offs need X's PWMS to the last bit on both sides
            assert eng.window_scores(sites, h, prm)[1][w] == pw, (h, w)
        for seqs, bg4, state, x, cutoff, lists, picks in _cut_case(k, bg):
            want = oracle_sweep(0, seqs, 1, k, 1e-4, cutoff, O.pcv_from_acgt(bg4), state, picks)
            params = make_params(k, 1e-4, ALPHABET_SIZE, bg4, cutoff=cutoff, sampler=_abi.GIBBS_MOTIF_SAMPLER,
                                 phase_mask=_abi.PHASE_STOCHASTIC)
            for team in TEAMS:
                eng.set_team_warps(team)
                got = _sweep(eng, params, state, picks)
                for r in range(len(picks)):
                    _same(got[r], want[r], (x, cutoff - x[2], team, r))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [20, 32])
def test_restart_with_a_cut_off_at_a_planted_window(k):
    """Whole doMotifSamplingWithPCV restarts (Philox) with the cut-off 1e-11 above and 1e-9 below a planted window."""
    seqs, bg4, _ = _cut_set(k, "sample")
    S = O.sources(seqs)
    pcv49 = O.pcv_from_acgt(bg4)
    for h, w, pw, err in cut_windows(k, "sample"):
        for cutoff in (pw + 1e-11, pw - 1e-9):
            params = make_params(k, 1e-4, ALPHABET_SIZE, bg4, cutoff=cutoff, sampler=_abi.GIBBS_MOTIF_SAMPLER)
            with GibbsEngine(seqs) as eng:
                res = eng.run(params, 4, chain_id_base=3, seed=41, want_counts=False)
            for c in range(4):
                rng, _ = O.make_rng(seed=41, chain=3 + c)
                want, _ = O.motif_step("do_motif_sampling", 0, S, 1, k, 1e-4, cutoff, pcv=pcv49, rng=rng)
                got = [(float(v), [int(s)] if s >= 0 else []) for v, s in zip(res.scores[c], res.sites[c])]
                _same(got, want, (k, cutoff - pw, c))


def _data_cases():
    """Data-derived background (fs:896-905): X's PWMS comes from the oracle's own stochastic picks (high picks of the
    planted start state), the cut-offs sit on it."""
    out = []
    for k in (20, 32):
        ps = planted_motif_set(10, 160, k, seed=7, mutation=0.02)
        seqs = ps.sequences()
        state = [(1.0, [int(t)]) for t in ps.truth]
        n = len(seqs)
        picks = np.array([np.full(n, 0.9999), np.full(n, 0.99), np.random.default_rng(k).random(n)])
        want = oracle_sweep(1, seqs, 1, k, 1e-4, 0.0, None, state, picks)
        scored = sorted({(coarse_log2_float32(2.0 ** v) - v, v) for row in want for v, p in row if p})
        out.append((k, seqs, state, picks, [scored[0], scored[-1]]))
    return out


@pytest.mark.gpu
def test_data_background_sweep_at_the_cut_off():
    for k, seqs, state, picks0, xs in _data_cases():
        n = len(seqs)
        picks = np.vstack([np.full(n, 0.5), np.full(n, 0.9999), np.random.default_rng(3).random((3, n))])
        with GibbsEngine(seqs) as eng:
            params = make_params(k, 1e-4, ALPHABET_SIZE, [0.25] * 4, cutoff=0.0, sampler=_abi.GIBBS_MOTIF_SAMPLER,
                                 phase_mask=_abi.PHASE_STOCHASTIC, background=_abi.GIBBS_BG_DATA)
            eng.set_team_warps(1)
            mine = {v for row in _sweep(eng, params, state, picks0) for v, p in row if p}
            assert all(pw in mine for _, pw in xs)   # the one-ulp cut-offs need X's PWMS to the last bit on both sides
            for err, pw in xs:
                for cutoff in cut_offs(pw):
                    want = oracle_sweep(1, seqs, 1, k, 1e-4, cutoff, None, state, picks)
                    params = make_params(k, 1e-4, ALPHABET_SIZE, [0.25] * 4, cutoff=cutoff, sampler=_abi.GIBBS_MOTIF_SAMPLER,
                                         phase_mask=_abi.PHASE_STOCHASTIC, background=_abi.GIBBS_BG_DATA)
                    for team in (1, 4, 16):
                        eng.set_team_warps(team)
                        got = _sweep(eng, params, state, picks)
                        for r in range(len(picks)):
                            _same(got[r], want[r], (k, cutoff - pw, team, r))


def test_data_background_constructions():
    errs = [err for _, _, _, _, xs in _data_cases() for err, _ in xs]
    assert min(errs) <= -BIG_ERROR or max(errs) >= BIG_ERROR, errs


def _masked_set():
    """A planted k = 24 set with an N in every sequence, away from the planted site: motif_kernel<..., MASKED = true>."""
    k = 24
    ps = planted_motif_set(8, 150, k, seed=9, mutation=0.02)
    seqs = []
    for s, t in zip(ps.sequences(), ps.truth):
        b = bytearray(s)
        b[int(t) + k + 7 if int(t) + k + 7 < len(b) else 3] = ord("N")
        seqs.append(bytes(b))
    state = [(1.0, [int(t)]) for t in ps.truth]
    return k, seqs, state, SKEWED


@pytest.mark.gpu
def test_masked_set_sweep_at_the_cut_off():
    k, seqs, state, bg4 = _masked_set()
    pcv49 = O.pcv_from_acgt(bg4)
    best, h_b, w_b = max((v, h, p[0]) for h, lst in enumerate(lists_of(seqs, state, k, 1e-4, 0.0, pcv49)) for v, p in lst if p)
    with GibbsEngine(seqs) as eng:
        sites = np.array([p[0] for _, p in state], np.int32)
        prm = make_params(k, 1e-4, ALPHABET_SIZE, bg4, sampler=_abi.GIBBS_MOTIF_SAMPLER)
        assert eng.window_scores(sites, h_b, prm)[1][w_b] == best
    for cutoff in cut_offs(best):
        lists = lists_of(seqs, state, k, 1e-4, cutoff, pcv49)
        h_x = next(h for h, lst in enumerate(lists) if any(v == best for v, p in lst if p)) if best > cutoff else 0
        picks = cut_picks(lists, (h_x, -1))
        want = oracle_sweep(0, seqs, 1, k, 1e-4, cutoff, pcv49, state, picks)
        params = make_params(k, 1e-4, ALPHABET_SIZE, bg4, cutoff=cutoff, sampler=_abi.GIBBS_MOTIF_SAMPLER,
                             phase_mask=_abi.PHASE_STOCHASTIC)
        with GibbsEngine(seqs) as eng:
            for team in (1, 4):
                eng.set_team_warps(team)
                got = _sweep(eng, params, state, picks)
                for r in range(len(picks)):
                    _same(got[r], want[r], (cutoff - best, team, r))


# ---------------------------------------------------------------------------------------------------------------------
# b) picks on bucket edges
# ---------------------------------------------------------------------------------------------------------------------
def _homopolymer(k, q_a, n=4, L=300):
    seqs = [b"A" * L for _ in range(n)]
    rest = (1.0 - q_a) / 3.0
    return seqs, [q_a, rest, rest, rest], [(1.0, [0]) for _ in range(n)], 1e-4, 0.0


def _planted(n, L, k, pc, cutoff, seed):
    ps = planted_motif_set(n, L, k, seed=seed)
    return ps.sequences(), background_of(ps.ascii, pc, ALPHABET_SIZE), [(1.0, [int(t)]) for t in ps.truth], pc, cutoff


EDGE_LISTS = {
    "short": lambda: _planted(6, 40, 8, 1e-4, 3.0, 61),                 # a few candidates
    "long": lambda: _planted(3, 5000, 8, 1.0, 0.0, 62),                 # hundreds of candidates, many lanes' blocks
    "equal": lambda: _homopolymer(24, 0.0525),                          # 277 equal candidates at PWMS ~ 102
    "above128": lambda: _homopolymer(32, 0.05),                         # scores in [128, 256)
}


def edge_rows(lists, k):
    """Rows of picks (one per held-out sequence) on the edges of every list: the end of the background mass, a middle
    edge, the last edge, each with edge_picks(), and u = 1.0."""
    per_h = []
    for lst in lists:
        wts = [v for v, _ in lst]
        lo, hi = walk_edges(wts)
        n_bg = sum(1 for _, p in lst if not p)
        mid = n_bg + (len(lst) - n_bg) // 2
        us = []
        for e in (lo[n_bg] if n_bg < len(lst) else hi[-1], lo[mid] if mid < len(lst) else hi[-1], hi[-1]):
            us += edge_picks(e)
        us.append(1.0)
        per_h.append(us)
    rows = np.array(per_h).T
    ok = np.array([all(walk_pick([v for v, _ in lst], u) is not None for lst, u in zip(lists, row)) for row in rows])
    return rows[ok], rows[~ok]


def _edge_case(name):
    seqs, bg4, state, pc, cutoff = EDGE_LISTS[name]()
    k = {"short": 8, "long": 8, "equal": 24, "above128": 32}[name]
    pcv49 = O.pcv_from_acgt(bg4)
    lists = lists_of(seqs, state, k, pc, cutoff, pcv49)
    good, bad = edge_rows(lists, k)
    past = np.array([[math.nextafter(walk_edges([v for v, _ in lst])[1][-1], 2.0) for lst in lists]])
    return seqs, bg4, state, pc, cutoff, k, pcv49, lists, good, np.vstack([bad, past])


@pytest.mark.parametrize("name", list(EDGE_LISTS))
def test_edge_constructions(name):
    seqs, bg4, state, pc, cutoff, k, pcv49, lists, good, bad = _edge_case(name)
    n_cand = [sum(1 for _, p in lst if p) for lst in lists]
    if name == "long":
        assert min(n_cand) >= 150
    if name == "equal":
        assert n_cand == [277] * len(seqs)
        v = lists[0][-1][0]
        assert 101 < v < 103 and all(x == v for x, p in lists[0] if p)
        assert coarse_log2_float32(2.0 ** v) - v >= BIG_ERROR
    if name == "above128":
        assert all(128 <= v < 256 for lst in lists for v, p in lst if p)
    for row in list(good) + list(bad):
        for lst, u in zip(lists, row):
            wts = [v for v, _ in lst]
            assert walk_pick(wts, u) == oracle_pick(wts, u)          # the helper is the oracle's walk
    # every edge is a real boundary: the pick on it and one ulp above land in neighbouring buckets
    for lst in lists:
        wts = [v for v, _ in lst]
        lo, hi = walk_edges(wts)
        n_bg = sum(1 for _, p in lst if not p)
        if n_bg < len(lst):
            e = lo[n_bg]
            assert walk_pick(wts, e) == n_bg - 1 and walk_pick(wts, math.nextafter(e, 2.0)) == n_bg
    assert len(bad) >= 1
    for row in bad:
        assert any(walk_pick([v for v, _ in lst], u) is None for lst, u in zip(lists, row))
    want = oracle_sweep(0, seqs, 1, k, pc, cutoff, pcv49, state, good)
    for r, row in enumerate(good):
        for h, u in enumerate(row):
            assert want[r][h] == lists[h][walk_pick([v for v, _ in lists[h]], u)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(EDGE_LISTS))
def test_pick_roulette_on_bucket_edges(name):
    """gibbs_pick_roulette: motif_roulette's scan, its edge check and the exact walk."""
    seqs, bg4, state, pc, cutoff, k, pcv49, lists, good, bad = _edge_case(name)
    sites = np.array([p[0] if p else -1 for _, p in state], np.int32)
    params = make_params(k, pc, ALPHABET_SIZE, bg4, cutoff=cutoff, sampler=_abi.GIBBS_MOTIF_SAMPLER)
    with GibbsEngine(seqs) as eng:
        for row in list(good) + list(bad):
            for h, u in enumerate(row):
                wts = [v for v, _ in lists[h]]
                i = oracle_pick(wts, u)
                if i is None:
                    with pytest.raises(_abi.GibbsRouletteError):
                        eng.pick_roulette(sites, h, params, u)
                    continue
                pwms, site = eng.pick_roulette(sites, h, params, u)
                assert ([site] if site >= 0 else []) == lists[h][i][1], (h, u)
                assert pwms == pytest.approx(lists[h][i][0], rel=RTOL)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(EDGE_LISTS))
def test_stochastic_sweep_on_bucket_edges(name):
    """The stochastic sweep (motif_stoch_fast, then the exact path): every edge pick of a list in one launch, one chain per
    row; a pick past the end of the mass fails the run like the reference's throw."""
    seqs, bg4, state, pc, cutoff, k, pcv49, lists, good, bad = _edge_case(name)
    want = oracle_sweep(0, seqs, 1, k, pc, cutoff, pcv49, state, good)
    params = make_params(k, pc, ALPHABET_SIZE, bg4, cutoff=cutoff, sampler=_abi.GIBBS_MOTIF_SAMPLER,
                         phase_mask=_abi.PHASE_STOCHASTIC)
    with GibbsEngine(seqs) as eng:
        for team in TEAMS:
            eng.set_team_warps(team)
            got = _sweep(eng, params, state, good)
            for r in range(len(good)):
                _same(got[r], want[r], (team, r, list(good[r])))
        assert all(w is None for w in oracle_sweep(0, seqs, 1, k, pc, cutoff, pcv49, state, bad))
        eng.set_team_warps(4)
        for row in bad:
            with pytest.raises(_abi.GibbsRouletteError):
                _sweep(eng, params, state, row[None, :])


# ---------------------------------------------------------------------------------------------------------------------
# c) motifAmount = 2
# ---------------------------------------------------------------------------------------------------------------------
def _pairs_case():
    n, L, k, pc, cutoff = 5, 40, 5, 1e-2, 1.0
    ps = planted_motif_set(n, L, k, seed=71)
    seqs = ps.sequences()
    bg4 = background_of(ps.ascii, pc, ALPHABET_SIZE)
    state = [(1.0, [int(t) + k + 3, int(t)] if int(t) + 2 * k + 3 <= L else [int(t)]) for t in ps.truth]
    pcv49 = O.pcv_from_acgt(bg4)
    lists = lists_of(seqs, state, k, pc, cutoff, pcv49, m=2)
    per_h = []
    for lst in lists:
        wts = [v for v, _ in lst]
        lo, hi = walk_edges(wts)
        first_single = next(i for i, (_, p) in enumerate(lst) if len(p) == 1)
        first_pair = next(i for i, (_, p) in enumerate(lst) if len(p) == 2)
        us = []
        for e in (lo[first_single], lo[first_pair], lo[(first_pair + len(lst)) // 2], hi[-1]):
            us += edge_picks(e)[:5]
        per_h.append(us)
    rows = np.array(per_h).T
    ok = np.array([all(walk_pick([v for v, _ in lst], u) is not None for lst, u in zip(lists, row)) for row in rows])
    return seqs, bg4, state, k, pc, cutoff, pcv49, lists, rows[ok]


def test_pairs_constructions():
    seqs, bg4, state, k, pc, cutoff, pcv49, lists, rows = _pairs_case()
    assert len(rows) >= 15 and any(len(p) == 2 for _, p in state)
    want = oracle_sweep(0, seqs, 2, k, pc, cutoff, pcv49, state, rows)
    for r, row in enumerate(rows):
        for h, u in enumerate(row):
            wts = [v for v, _ in lists[h]]
            i = walk_pick(wts, u)
            assert i == oracle_pick(wts, u) and want[r][h] == lists[h][i]


@pytest.mark.gpu
def test_two_site_sweep_on_bucket_edges():
    seqs, bg4, state, k, pc, cutoff, pcv49, lists, rows = _pairs_case()
    want = oracle_sweep(0, seqs, 2, k, pc, cutoff, pcv49, state, rows)
    params = make_params(k, pc, ALPHABET_SIZE, bg4, cutoff=cutoff, sampler=_abi.GIBBS_MOTIF_SAMPLER,
                         phase_mask=_abi.PHASE_STOCHASTIC, motif_amount=2)
    with GibbsEngine(seqs) as eng:
        got = _sweep(eng, params, state, rows, m=2)
    for r in range(len(rows)):
        _same(got[r], want[r], (r, list(rows[r])))
