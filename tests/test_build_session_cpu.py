"""Build-session argument checks that fail before any CUDA call, and the loud failure without a GPU."""
import ctypes as C

import numpy as np
import pytest

from lphash_b200 import api


def test_begin_refuses_bad_arguments():
    L = api.lib()
    h = C.c_void_p()
    assert L.lphb_build_begin(0, 31, 20, 42, None) == api.E_ARG
    for k, m in [(31, 0), (40, 32), (19, 20), (64, 20)]:
        assert L.lphb_build_begin(0, k, m, 42, C.byref(h)) == api.E_ARG, (k, m)
        assert not h.value
    for device in (-1, 64):
        assert L.lphb_build_begin(device, 31, 20, 42, C.byref(h)) == api.E_ARG
    with pytest.raises(api.LphashError) as e:
        api.BuildSession(31, 32)
    assert e.value.code == api.E_ARG


def test_calls_without_a_session():
    L = api.lib()
    off = np.zeros(1, dtype=np.uint64)
    r = api.BuildReport()
    assert L.lphb_build_batch(None, None, off.ctypes.data, 0) == api.E_ARG
    assert L.lphb_build_batch_device(None, None, off.ctypes.data, off.ctypes.data, 0, None) == api.E_ARG
    assert L.lphb_build_end(None, None, 0, None, 0, C.byref(r)) == api.E_ARG
    assert L.lphb_build_free(None) == api.OK


def test_no_gpu_means_loud_failure():
    n = C.c_int(-1)
    if api.lib().lphb_device_count(C.byref(n)) == api.OK and n.value > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(api.LphashError) as e:
        api.BuildSession(31, 20)
    assert e.value.code == api.E_CUDA
