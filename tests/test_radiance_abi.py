"""The radiance entry points of the C ABI (rtcuda_radiance / rtcuda_radiance_device) without a GPU: exported and bound, the ABI
unchanged (v4), every malformed call refused with INVALID_ARGUMENT before any device work, and the Python methods' ray checks."""
import ctypes as C

import numpy as np
import pytest

SYMBOLS = ["rtcuda_radiance", "rtcuda_radiance_device"]
INVALID_ARGUMENT = 1


@pytest.fixture(scope="module")
def lib(rc):
    return rc._ffi.load_library()


def test_radiance_symbols_are_exported_and_bound(rc, lib):
    assert set(SYMBOLS) <= set(rc._ffi.EXPORTED_SYMBOLS)
    assert lib.rtcuda_abi_version() == rc._ffi.ABI_VERSION == 4
    for name in SYMBOLS:
        fn = getattr(lib, name)
        assert fn.argtypes == [C.c_void_p, C.POINTER(rc._ffi.Settings), C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p], name
        assert fn.restype == C.c_int


@pytest.mark.parametrize("name", SYMBOLS)
def test_malformed_calls_are_refused_before_device_work(rc, lib, name):
    """No scene is needed to reach these checks (there is no GPU here): each refusal names what is wrong"""
    call = getattr(lib, name)
    rays = np.zeros((4, 8), np.float32)
    out = np.zeros((4, 3), np.float32)
    R, O = rays.ctypes.data, out.ctypes.data

    def settings(**kw):
        s = rc.RaytracerSettings(samples_per_pixel=4)
        for k, v in kw.items():
            setattr(s, k, v)
        return C.byref(s.to_c())

    def refused(status, text):
        assert status == INVALID_ARGUMENT and text in lib.rtcuda_last_error().decode(), lib.rtcuda_last_error()

    refused(call(None, settings(), R, 1 << 32, 0, O), "below 2^32")
    refused(call(None, settings(), R, 4, (1 << 32) - 3, O), "stream_base + count")
    refused(call(None, settings(), None, 4, 0, O), "rays is NULL")
    refused(call(None, settings(), R, 4, 0, None), "radiance is NULL")
    refused(call(None, None, R, 4, 0, O), "settings is NULL")
    refused(call(None, settings(samples_per_pixel=0), R, 4, 0, O), "samples_per_pixel")
    refused(call(None, settings(sampler=rc.Sampler.stratified(True, 0, 4)), R, 4, 0, O), "strata")
    refused(call(None, settings(), R, 4, (1 << 32) - 4, O), "scene is NULL")   # stream_base + count == 2^32 is allowed
    refused(call(None, settings(), None, 0, 0, O), "scene is NULL")


def test_radiance_methods_check_the_ray_array(rc):
    """dtype, shape and contiguity are checked in Python before the library is called (no scene is touched)"""
    r = rc.CudaRenderer.__new__(rc.CudaRenderer)
    st = rc.RaytracerSettings(samples_per_pixel=1)
    good = rc.make_rays(np.zeros((4, 3)), [0, 0, 1])
    for bad in (good.astype(np.float64), good[:, :7], good.reshape(-1), good[::2], np.asfortranarray(good), good.tolist()):
        with pytest.raises(ValueError):
            r.radiance(bad, st)
