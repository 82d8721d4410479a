"""Host side of the multi-device batch (gibbs_multi_batch_*, engine.MultiBatchEngine): the argument checks that run before
any device is touched, the error without a device, and the ctypes signatures."""
import ctypes as C

import numpy as np
import pytest

from gibbssampling_b200 import _abi
from gibbssampling_b200.engine import MultiBatchEngine, make_params

SEQS = [b"ACGTACGTACGT", b"ACGTTTTTACGA", b"GGGACGTAAACC", b"TTACGTACCAAA", b"CACGTGACGTTT"]
P = C.POINTER


def _flat():
    buf = np.frombuffer(b"".join(SEQS), dtype=np.uint8).copy()
    off = np.zeros(len(SEQS) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(s) for s in SEQS])
    return buf, off


def _create(lib, buf, off, set_off, n_sets, devices=None, n_devices=0, out=True):
    mb = C.c_void_p()
    rc = lib.gibbs_multi_batch_create(buf.ctypes.data_as(P(C.c_uint8)) if buf is not None else None,
                                      off.ctypes.data_as(P(C.c_int64)) if off is not None else None,
                                      set_off.ctypes.data_as(P(C.c_int32)) if set_off is not None else None, C.c_int32(n_sets),
                                      devices.ctypes.data_as(P(C.c_int32)) if devices is not None else None, C.c_int32(n_devices),
                                      C.byref(mb) if out else None)
    return rc, lib.gibbs_last_error().decode()


def _batch_create(lib, buf, off, set_off, n_sets, out=True):
    b = C.c_void_p()
    rc = lib.gibbs_batch_create(buf.ctypes.data_as(P(C.c_uint8)) if buf is not None else None,
                                off.ctypes.data_as(P(C.c_int64)) if off is not None else None,
                                set_off.ctypes.data_as(P(C.c_int32)) if set_off is not None else None, C.c_int32(n_sets),
                                C.c_int32(0), C.byref(b) if out else None)
    return rc, lib.gibbs_last_error().decode()


@pytest.mark.parametrize("case", ["null_out", "null_seqs", "null_offsets", "null_set_offsets", "no_sets", "first_not_zero",
                                  "empty_set", "decreasing"])
def test_argument_errors_come_before_any_device_work_and_match_the_one_device_batch(case):
    lib = _abi.load()
    buf, off = _flat()
    set_off = np.array([0, 2, 5], dtype=np.int32)
    n_sets, out = 2, True
    if case == "null_out":
        out = False
    elif case == "null_seqs":
        buf = None
    elif case == "null_offsets":
        off = None
    elif case == "null_set_offsets":
        set_off = None
    elif case == "no_sets":
        n_sets = 0
    elif case == "first_not_zero":
        set_off = np.array([1, 2, 5], dtype=np.int32)
    elif case == "empty_set":
        set_off = np.array([0, 2, 2], dtype=np.int32)
    elif case == "decreasing":
        set_off = np.array([0, 3, 2], dtype=np.int32)
    for n_devices in (0, 1, 3):
        rc, msg = _create(lib, buf, off, set_off, n_sets, n_devices=n_devices, out=out)
        assert rc == _abi.GIBBS_ERR_ARG
        assert (rc, msg) == _batch_create(lib, buf, off, set_off, n_sets, out=out)


def test_negative_device_count_is_an_argument_error():
    lib = _abi.load()
    buf, off = _flat()
    rc, msg = _create(lib, buf, off, np.array([0, 2, 5], dtype=np.int32), 2, n_devices=-1)
    assert rc == _abi.GIBBS_ERR_ARG and "n_devices" in msg


def test_engine_rejects_null_and_empty_sets_before_any_device_work():
    for sets in (None, [], [SEQS[:2], []]):
        with pytest.raises(_abi.GibbsArgumentError):
            MultiBatchEngine(sets, n_devices=2)


def test_entry_points_reject_a_null_object():
    lib = _abi.load()
    params = make_params(6, 1e-4, 4, [0.25] * 4)
    out = np.zeros(64, dtype=np.int32)
    o = out.ctypes.data_as(P(C.c_int32))
    first, n = C.c_int32(), C.c_int32()
    assert lib.gibbs_multi_batch_destroy(None) == _abi.GIBBS_OK
    assert lib.gibbs_multi_batch_num_devices(None) == 0
    assert lib.gibbs_multi_batch_slot_sets(None, 0, C.byref(first), C.byref(n)) == _abi.GIBBS_ERR_ARG
    for fn in (lib.gibbs_multi_batch_run_device, lib.gibbs_multi_batch_run_motif_device):
        assert fn(None, C.byref(params), None, C.c_int32(2), C.c_int64(0), C.c_uint64(0)) == _abi.GIBBS_ERR_ARG
        assert "null multi-device batch" in lib.gibbs_last_error().decode()
    assert lib.gibbs_multi_batch_fetch(None, o, None, None, None) == _abi.GIBBS_ERR_ARG
    assert lib.gibbs_multi_batch_fetch_best(None, 1, o, None, None, None, None, None, None) == _abi.GIBBS_ERR_ARG
    for fn in (lib.gibbs_multi_batch_fetch_positions, lib.gibbs_multi_batch_fetch_best_positions):
        assert fn(None, C.c_int32(1), o) == _abi.GIBBS_ERR_ARG


def test_no_cpu_fallback_without_a_device():
    lib = _abi.load()
    if lib.gibbs_device_count() > 0:
        pytest.skip("a CUDA device is present")
    buf, off = _flat()
    for devices, n_devices in ((None, 0), (None, 2), (np.array([0, 0], dtype=np.int32), 2)):
        rc, msg = _create(lib, buf, off, np.array([0, 2, 5], dtype=np.int32), 2, devices=devices, n_devices=n_devices)
        assert rc == _abi.GIBBS_ERR_CUDA and "no CUDA device" in msg
    with pytest.raises(_abi.GibbsCudaError):
        MultiBatchEngine([SEQS[:2], SEQS[2:]])


def test_ctypes_signatures():
    lib = _abi.load()
    vp, i32, i64, u64, f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_double
    want = {
        "gibbs_multi_batch_create": [P(C.c_uint8), P(i64), P(i32), i32, P(i32), i32, P(vp)],
        "gibbs_multi_batch_destroy": [vp],
        "gibbs_multi_batch_num_devices": [vp],
        "gibbs_multi_batch_slot_sets": [vp, i32, P(i32), P(i32)],
        "gibbs_multi_batch_run_device": [vp, P(_abi.Params), P(f64), i32, i64, u64],
        "gibbs_multi_batch_run_motif_device": [vp, P(_abi.Params), P(f64), i32, i64, u64],
        "gibbs_multi_batch_fetch": [vp, P(i32), P(f64), P(f64), P(_abi.RunStats)],
        "gibbs_multi_batch_fetch_best": [vp, i32, P(i32), P(f64), P(i32), P(f64), P(i32), P(i32), P(_abi.RunStats)],
        "gibbs_multi_batch_fetch_positions": [vp, i32, P(i32)],
        "gibbs_multi_batch_fetch_best_positions": [vp, i32, P(i32)],
    }
    for name, args in want.items():
        assert name in _abi.EXPORTS
        fn = getattr(lib, name)
        assert fn.argtypes == args, name
        assert fn.restype is i32, name
    # each mirrors its one-device twin
    for name in ("run_device", "run_motif_device", "fetch", "fetch_best", "fetch_positions", "fetch_best_positions"):
        assert getattr(lib, "gibbs_multi_batch_" + name).argtypes == getattr(lib, "gibbs_batch_" + name).argtypes
