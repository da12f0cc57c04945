"""Argument validation of the real-time servers' C ABI (ntm_rt_* and ntm_rt_diffdel_*) without a GPU: no call here reaches
the device."""
import ctypes

from ntm_b200 import lib


def test_rt_rejects_bad_arguments():
    L = lib.load()
    rt = ctypes.c_void_p()
    # no handle, no output pointer
    assert L.ntm_rt_open(None, lib.MODE_F16, None, 1, 64, 0, 1000, ctypes.byref(rt)) == -1
    assert rt.value is None
    assert L.ntm_rt_open(None, lib.MODE_F16, None, 1, 64, 0, 1000, None) == -1
    assert L.ntm_rt_diffdel_open(None, lib.MODE_F16, None, None, 1, 64, 366, 0, 1, 1000, ctypes.byref(rt)) == -1
    assert rt.value is None
    assert L.ntm_rt_diffdel_open(None, lib.MODE_F16, None, None, 1, 64, 366, 0, 1, 1000, None) == -1
    # not a stream
    assert L.ntm_rt_process(None, None, None) == -1
    assert L.ntm_rt_close(None, None) == -1
    assert L.ntm_rt_diffdel_process(None, None, None, None, None) == -1
    assert L.ntm_rt_diffdel_close(None, None, None) == -1
