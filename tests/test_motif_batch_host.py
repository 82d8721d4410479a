"""Host side of the MotifSampler batch (gibbs_batch_run_motif_device, MotifSampler.…OfSets): what is checked before anything
reaches the GPU, and that a batch without a device fails loudly instead of computing on the CPU."""
import ctypes as C

import numpy as np
import pytest

from gibbssampling_b200 import MotifSampler, _abi
from gibbssampling_b200.CompositeVector import ProbabilityCompositeVector
from gibbssampling_b200.engine import make_params

DNA = list("ATGC-")
SETS = [["ACGTACGTACGT", "ACGTTTTTACGA"], ["GGGACGTAAACC", "TTACGTACCAAA", "CACGTGACGTTT"]]
PCV = ProbabilityCompositeVector.ofACGT(0.25, 0.25, 0.25, 0.25)


@pytest.mark.parametrize("call", [
    lambda: MotifSampler.getMotifsWithBestInformationContentsOfSets(1, 2, 6, 1e-4, 1.0, DNA, None),
    lambda: MotifSampler.findBestInormationContentContainingMotifsWithPCVOfSets(1, 1, 6, 1e-4, 1.0, DNA, None, [PCV]),
    lambda: MotifSampler.findBestInormationContentContainingMotifsWithPCVOfSets(1, 1, 6, 1e-4, 1.0, DNA, SETS, None),
    lambda: MotifSampler.findBestInormationContentContainingMotifsWithPCVOfSets(1, 1, 6, 1e-4, 1.0, DNA, SETS, [PCV]),
    lambda: MotifSampler.getMotifsWithBestInformationContentsOfSets(1, 1, 6, 1e-4, 1.0, DNA, [SETS[0], []]),
])
def test_wrappers_reject_null_sets_and_mismatched_pcvs(call):
    with pytest.raises(_abi.GibbsArgumentError):
        call()


def test_three_sites_per_sequence_are_unsupported_before_any_device_work():
    with pytest.raises(_abi.GibbsUnsupportedError):
        MotifSampler.getMotifsWithBestInformationContentsOfSets(1, 3, 6, 1e-4, 1.0, DNA, SETS)


def test_entry_points_reject_a_null_batch_or_params():
    lib = _abi.load()
    params = make_params(6, 1e-4, 4, [0.25] * 4, cutoff=1.0, sampler=_abi.GIBBS_MOTIF_SAMPLER, motif_amount=2)
    out = np.zeros(16, dtype=np.int32)
    assert lib.gibbs_batch_run_motif_device(None, C.byref(params), None, C.c_int32(2), C.c_int64(0), C.c_uint64(0)) == _abi.GIBBS_ERR_ARG
    assert "null batch" in lib.gibbs_last_error().decode()
    assert lib.gibbs_batch_run_motif_device(None, None, None, C.c_int32(2), C.c_int64(0), C.c_uint64(0)) == _abi.GIBBS_ERR_ARG
    for fn in (lib.gibbs_batch_fetch_positions, lib.gibbs_batch_fetch_best_positions):
        assert fn(None, C.c_int32(2), out.ctypes.data_as(C.POINTER(C.c_int32))) == _abi.GIBBS_ERR_ARG
        assert fn(None, C.c_int32(1), None) == _abi.GIBBS_ERR_ARG


def test_no_cpu_fallback_for_motif_batches_without_a_device():
    lib = _abi.load()
    if lib.gibbs_device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(_abi.GibbsCudaError) as ei:
        MotifSampler.getMotifsWithBestInformationContentsOfSets(1, 2, 6, 1e-4, 1.0, DNA, SETS, seed=1)
    assert ei.value.code == _abi.GIBBS_ERR_CUDA
    with pytest.raises(_abi.GibbsCudaError):
        MotifSampler.findBestInormationContentContainingMotifsWithPCVOfSets(1, 1, 6, 1e-4, 1.0, DNA, SETS, [PCV, PCV], seed=1)
