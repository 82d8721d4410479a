"""Host side of the batch API (gibbs_batch_*): how sets are flattened and validated before anything reaches the GPU,
and that a batch without a device fails loudly instead of computing on the CPU."""
import numpy as np
import pytest

from gibbssampling_b200 import _abi
from gibbssampling_b200.engine import BatchEngine, flatten_sets


def test_flatten_sets_concatenates_sets_and_records_their_boundaries():
    buf, off, set_off = flatten_sets([["ACGT", "AC"], ["GGG"], [b"TTTTA", "C", "NNA"]])
    assert buf.tobytes() == b"ACGTACGGGTTTTACNNA"
    assert off.tolist() == [0, 4, 6, 9, 14, 15, 18]
    assert set_off.dtype == np.int32 and set_off.tolist() == [0, 2, 3, 6]


@pytest.mark.parametrize("sets", [None, [], [["ACGT"], []], [["ACGT"], None]])
def test_flatten_sets_rejects_null_and_empty_sets(sets):
    with pytest.raises(_abi.GibbsArgumentError):
        flatten_sets(sets)


def test_batch_create_validates_set_offsets_before_any_device_work():
    """Bad set_offsets are GIBBS_ERR_ARG whether or not a device is present (checked before the device is touched)."""
    import ctypes as C
    lib = _abi.load()
    buf = np.frombuffer(b"ACGTACGTACGT", dtype=np.uint8).copy()
    off = np.array([0, 4, 8, 12], dtype=np.int64)
    b = C.c_void_p()
    for so in ([0, 2, 2, 3], [1, 2, 3], [0, 3, 2]):
        so = np.array(so, dtype=np.int32)
        rc = lib.gibbs_batch_create(buf.ctypes.data_as(C.POINTER(C.c_uint8)), off.ctypes.data_as(C.POINTER(C.c_int64)),
                                    so.ctypes.data_as(C.POINTER(C.c_int32)), C.c_int32(len(so) - 1), C.c_int32(0), C.byref(b))
        assert rc == _abi.GIBBS_ERR_ARG, so
        assert not b.value
    rc = lib.gibbs_batch_create(buf.ctypes.data_as(C.POINTER(C.c_uint8)), off.ctypes.data_as(C.POINTER(C.c_int64)), None,
                                C.c_int32(1), C.c_int32(0), C.byref(b))
    assert rc == _abi.GIBBS_ERR_ARG


def test_batch_symbol_errors_name_the_set_and_the_sequence():
    with pytest.raises(_abi.GibbsSymbolError) as ei:
        BatchEngine([["ACGT", "ACGT"], ["ACGT", "ACgT"]])
    assert "set 1, sequence 1" in str(ei.value)


def test_no_cpu_fallback_for_batches_without_a_device():
    lib = _abi.load()
    if lib.gibbs_device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(_abi.GibbsCudaError) as ei:
        BatchEngine([[b"ACGTACGT", b"ACGTACGT"], [b"ACGTAAAA", b"ACGTCCCC"]])
    assert ei.value.code == _abi.GIBBS_ERR_CUDA
    assert "no CPU fallback" in str(ei.value)
    from gibbssampling_b200 import SiteSampler
    with pytest.raises(_abi.GibbsCudaError):
        SiteSampler.getMotifsWithBestInformationContentOfSets(1, 4, 1e-4, list("ATGC-"), [["ACGTACGT", "ACGTTTTT"]], seed=1)
