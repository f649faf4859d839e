"""bbq_group_create's checks that need no GPU: an empty, duplicated or negative device list is refused with
BBQ_ERR_INVALID_ARG before any device is probed, and without a GPU the call fails with BBQ_ERR_NO_DEVICE, never falls
back, and leaves no thread behind."""
import ctypes as C
import os

import pytest

import bbq_b200


def _cfg(query_bits=4):
    return bbq_b200._native.BbqConfig(query_bits=query_bits, index_bits=1, similarity=1, iters=5, lambda_=0.1, device=-1)


def _create(devices, cfg=None):
    L = bbq_b200._native.load()
    g = C.c_void_p()
    arr = (C.c_int32 * max(1, len(devices)))(*devices)
    st = L.bbq_group_create(C.byref(cfg or _cfg()), arr, len(devices), C.byref(g))
    return st, L.bbq_last_error().decode(), g.value


def _tasks():
    return len(os.listdir("/proc/self/task"))


@pytest.mark.parametrize("devices,message", [([], "the device list is empty"),
                                             ([0, 0], "device 0 appears twice in the device list"),
                                             ([1, 0, 2, 1], "device 1 appears twice in the device list"),
                                             ([-1], "device list entry 0 is negative (-1)"),
                                             ([0, -3], "device list entry 1 is negative (-3)")])
def test_bad_device_lists_are_refused_before_any_probe(devices, message):
    # a config error would be reported by the probe's stage: the list is checked first
    assert _create(devices, _cfg(query_bits=9)) == (10, message, None)
    assert _create(devices) == (10, message, None)


def test_bad_config_gives_the_status_of_bbq_create():
    L = bbq_b200._native.load()
    st, msg, g = _create([0], _cfg(query_bits=0))
    ctx = C.c_void_p()
    assert (st, msg, g) == (L.bbq_create(C.byref(_cfg(query_bits=0)), C.byref(ctx)), L.bbq_last_error().decode(), None)
    assert st == 1


def test_no_gpu_no_fallback_no_thread_left():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    before = _tasks()
    for devices in ([0], [0, 1], [3, 1, 2]):
        assert _create(devices) == (100, "no CUDA device: libbbq_b200 has no CPU fallback", None)
    assert _tasks() == before
    with pytest.raises(bbq_b200.BbqError) as e:
        bbq_b200.BinaryQuantizationFormat({}, devices=[0, 1])
    assert e.value.status == 100
    assert _tasks() == before
