"""The ray-query entry points of the C ABI (rtcuda_trace_rays / _device, rtcuda_occluded / _device) without a GPU: exported and
bound, the ABI unchanged (v4, same rtcuda_stats), malformed calls refused with INVALID_ARGUMENT before any device work, and
make_rays."""
import ctypes as C

import numpy as np
import pytest

QUERY_SYMBOLS = ["rtcuda_trace_rays", "rtcuda_trace_rays_device", "rtcuda_occluded", "rtcuda_occluded_device"]
INVALID_ARGUMENT = 1


@pytest.fixture(scope="module")
def lib(rc):
    return rc._ffi.load_library()


def test_query_symbols_are_exported_and_bound(rc, lib):
    assert set(QUERY_SYMBOLS) <= set(rc._ffi.EXPORTED_SYMBOLS)
    trace = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
    occl = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
    for name, args in zip(QUERY_SYMBOLS, (trace, trace, occl, occl)):
        fn = getattr(lib, name)
        assert fn.argtypes == args and fn.restype == C.c_int, name


def test_abi_is_unchanged(rc, lib):
    assert lib.rtcuda_abi_version() == rc._ffi.ABI_VERSION == 4
    assert [n for n, _ in rc._ffi.Stats._fields_][-3:] == ["update_ms", "bvh_sah_cost", "bvh_last_update"]
    sizes = (C.c_uint32 * 32)()
    assert lib.rtcuda_abi_struct_sizes(sizes, 32) == len(rc._ffi.ABI_STRUCTS)


def _calls(lib):
    rays = np.zeros((4, 8), np.float32)
    rays[:, 6] = -1.0
    t, ids, uv, occ = np.zeros(4, np.float32), np.zeros(8, np.uint32), np.zeros(8, np.float32), np.zeros(4, np.uint8)
    P = lambda a: a.ctypes.data
    return {
        "trace": lambda scene, r, n, no_out=False: lib.rtcuda_trace_rays(scene, r, n, *((None,) * 3 if no_out else (P(t), P(ids), P(uv)))),
        "trace_device": lambda scene, r, n, no_out=False: lib.rtcuda_trace_rays_device(scene, r, n, *((None,) * 3 if no_out else (P(t), None, None))),
        "occluded": lambda scene, r, n, no_out=False: lib.rtcuda_occluded(scene, r, n, None if no_out else P(occ)),
        "occluded_device": lambda scene, r, n, no_out=False: lib.rtcuda_occluded_device(scene, r, n, None if no_out else P(occ)),
    }, P(rays)


@pytest.mark.parametrize("which", ["trace", "trace_device", "occluded", "occluded_device"])
def test_malformed_calls_are_refused_before_device_work(lib, which):
    """No scene is needed to reach these checks (there is no GPU here): each refusal names what is wrong"""
    calls, rays = _calls(lib)
    call = calls[which]

    def refused(status, text):
        assert status == INVALID_ARGUMENT and text in lib.rtcuda_last_error().decode()

    refused(call(None, rays, 1 << 32), "below 2^32")
    refused(call(None, None, 4), "rays is NULL")
    refused(call(None, rays, 4, no_out=True), "every output is NULL")
    refused(call(None, rays, 4), "scene is NULL")
    refused(call(None, None, 0), "scene is NULL")


def test_make_rays_packs_and_validates(rc):
    r = rc.make_rays([[1, 2, 3], [4, 5, 6]], [0, 0, -1], t_min=[0.5, 0.25], t_max=10.0)
    assert r.dtype == np.float32 and r.shape == (2, 8) and r.flags.c_contiguous
    assert r.tolist() == [[1, 2, 3, 0.5, 0, 0, -1, 10], [4, 5, 6, 0.25, 0, 0, -1, 10]]
    assert rc.make_rays([0, 0, 0], [1, 0, 0])[0, 7] == np.inf
    with pytest.raises(ValueError):
        rc.make_rays([[0, 0]], [[1, 0, 0]])
    with pytest.raises(ValueError):
        rc.make_rays(np.zeros((3, 3)), np.ones((2, 3)))
    with pytest.raises(ValueError):
        rc.make_rays(np.zeros((3, 3)), np.ones((3, 3)), t_min=[0.0, 1.0])


def test_query_methods_check_the_ray_array(rc):
    """dtype, shape and contiguity are checked in Python before the library is called (no scene is touched)"""
    r = rc.CudaRenderer.__new__(rc.CudaRenderer)
    good = rc.make_rays(np.zeros((4, 3)), [0, 0, 1])
    for bad in (good.astype(np.float64), good[:, :7], good.reshape(-1), good[::2], np.asfortranarray(good), good.tolist()):
        with pytest.raises(ValueError):
            r.trace(bad)
        with pytest.raises(ValueError):
            r.occluded(bad)
