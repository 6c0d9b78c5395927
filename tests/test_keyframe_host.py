"""CPU tests of the keyframe entry points (include/icet_b200.h "keyframes"): without a device every entry point rejects
NULL or invalid arguments with a negative status and a message, and the Python class fails loudly."""
import ctypes as C

import numpy as np
import pytest


def _lib():
    import icet_b200
    icet_b200.build()
    return icet_b200.load_library()


def _no_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")


def test_keyframe_entry_points_reject_null_arguments():
    from icet_b200 import api
    L = _lib()
    p = api.make_params()
    pts = np.zeros((3, 16), np.float32)
    kf = C.c_void_p()
    res = api.Result()
    calls = [
        lambda: L.icet_b200_keyframe_create(None, C.byref(p), pts.ctypes.data, 16, 16, C.byref(kf)),
        lambda: L.icet_b200_keyframe_create_device(None, C.byref(p), pts.ctypes.data, 16, 16, C.byref(kf)),
        lambda: L.icet_b200_keyframe_gaussians(None),
        lambda: L.icet_b200_register_keyframe(None, C.byref(p), pts.ctypes.data, 16, 16, None, C.byref(res)),
        lambda: L.icet_b200_register_keyframe_batch_device(None, C.byref(p), 1, None, None, None, None),
    ]
    for call in calls:
        assert call() < 0
        assert L.icet_b200_last_error()
    assert L.icet_b200_keyframe_create(None, C.byref(p), pts.ctypes.data, 16, 16, C.byref(kf)) == -1
    assert b"ctx is NULL" in L.icet_b200_last_error()
    assert L.icet_b200_register_keyframe(None, C.byref(p), pts.ctypes.data, 16, 16, None, C.byref(res)) == -1
    assert b"keyframe is NULL" in L.icet_b200_last_error()
    assert L.icet_b200_keyframe_destroy(None) == 0  # like free(NULL)


def test_keyframe_create_without_device_fails_loudly():
    _no_device()
    import icet_b200
    with pytest.raises(icet_b200.IcetError) as e:
        icet_b200.Keyframe(np.zeros((100, 3), np.float32))
    assert "no CPU fallback" in str(e.value)
    with pytest.raises(icet_b200.IcetError) as e:
        icet_b200.Keyframe.from_device(0, 100)
    assert "no CPU fallback" in str(e.value)


def test_closed_keyframe_raises_without_calling_the_library():
    import icet_b200
    from icet_b200 import api

    class Trap:
        def __getattr__(self, name):
            raise AssertionError("library called: " + name)

    kf = object.__new__(api.Keyframe)  # a keyframe whose handle is gone
    kf._h, kf._L, kf._ctx = None, Trap(), None
    kf._p = api.make_params()
    with pytest.raises(icet_b200.IcetError, match="closed"):
        kf.register(np.zeros((3, 8), np.float32))
    with pytest.raises(icet_b200.IcetError, match="closed"):
        kf.register_batch_device([0], [8], 0)
    with pytest.raises(icet_b200.IcetError, match="closed"):
        kf.n_gauss1
    kf.close()
