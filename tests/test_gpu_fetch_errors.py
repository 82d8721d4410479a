"""The errors of the result fetches whose code a single-set handle and a batch share: the precondition texts of the
positions fetches (no run, no fetch_best, another motif_amount than the run's) and the roulette text of fetch_best, which
names the set in a batch and no set on a handle. Each is checked by its exact text through the C entry points."""
import ctypes as C

import numpy as np
import pytest

from gibbssampling_b200 import _abi
from gibbssampling_b200.engine import BatchEngine, GibbsEngine, make_params
from gibbssampling_b200.synthetic import planted_motif_set

pytestmark = pytest.mark.gpu
K = 4
MOTIF = make_params(K, 1e-4, 4, [0.25] * 4, cutoff=1.0, sampler=_abi.GIBBS_MOTIF_SAMPLER)  # motif_amount 1
ROULETTE = "a roulette pick lay beyond the accumulated mass (ArgumentException, fs:753)"


def _good():
    return planted_motif_set(5, 40, K, seed=3).sequences()


def _positions_error(lib, fn, obj, m, text):
    out = np.zeros(1024, dtype=np.int32)
    assert fn(obj, C.c_int32(m), out.ctypes.data_as(C.POINTER(C.c_int32))) == _abi.GIBBS_ERR_ARG
    assert lib.gibbs_last_error().decode() == text


def test_positions_preconditions_of_a_single_set_handle():
    lib = _abi.load()
    with GibbsEngine(_good()) as eng:
        _positions_error(lib, lib.gibbs_fetch_positions, eng._h, 1, "gibbs_fetch_positions without a preceding gibbs_run_device")
        eng.run_device(MOTIF, 2, seed=1)
        _positions_error(lib, lib.gibbs_fetch_best_positions, eng._h, 1,
                         "gibbs_fetch_best_positions without a preceding gibbs_fetch_best")
        _positions_error(lib, lib.gibbs_fetch_positions, eng._h, 2, "the last run had motif_amount = 1")
        eng.fetch_best(1)
        _positions_error(lib, lib.gibbs_fetch_best_positions, eng._h, 2, "the last run had motif_amount = 1")
        assert eng.fetch_best_positions(1).shape == (5, 1)


def test_positions_preconditions_of_a_batch():
    lib = _abi.load()
    with BatchEngine([_good(), planted_motif_set(7, 50, K, seed=4).sequences()]) as b:
        _positions_error(lib, lib.gibbs_batch_fetch_positions, b._b, 1, "gibbs_batch_fetch_positions without a preceding run")
        b.run_motif_device(MOTIF, 2, seed=1)
        _positions_error(lib, lib.gibbs_batch_fetch_best_positions, b._b, 1,
                         "gibbs_batch_fetch_best_positions without a preceding gibbs_batch_fetch_best")
        _positions_error(lib, lib.gibbs_batch_fetch_positions, b._b, 2, "the last run had motif_amount = 1")
        b.fetch_best(1)
        _positions_error(lib, lib.gibbs_batch_fetch_best_positions, b._b, 2, "the last run had motif_amount = 1")
        assert [p.shape for p in b.fetch_best_positions(1)] == [(5, 1), (7, 1)]


def test_fetch_best_roulette_error_text():
    """A held-out sequence whose every window holds a symbol outside the alphabet has no background mass under a fixed
    pcv, so its roulette pick runs past the list (fs:753)."""
    bad = _good()[:3] + [b"NNNNNNNNNNNN"]
    params = make_params(K, 1e-4, 4, [0.25] * 4, cutoff=0.0, sampler=_abi.GIBBS_MOTIF_SAMPLER)
    with GibbsEngine(bad) as eng:
        eng.run_device(params, 2, seed=1)
        with pytest.raises(_abi.GibbsRouletteError) as ei:
            eng.fetch_best(1)
        assert str(ei.value) == f"[gibbs_status {_abi.GIBBS_ERR_ROULETTE}] {ROULETTE}"
    with BatchEngine([_good(), bad]) as b:
        b.run_motif_device(params, 2, seed=1)
        with pytest.raises(_abi.GibbsRouletteError) as ei:
            b.fetch_best(1)
        assert str(ei.value) == f"[gibbs_status {_abi.GIBBS_ERR_ROULETTE}] set 1: {ROULETTE}"
