"""The surface-query entry points of the C ABI (rtcuda_trace_surfaces / rtcuda_trace_surfaces_device) without a GPU: exported and
bound, the ABI unchanged (v4, the same struct-size list), the 64-byte record's layout, every malformed call refused with
INVALID_ARGUMENT before any device work, and the Python methods' ray checks."""
import ctypes as C

import numpy as np
import pytest

SYMBOLS = ["rtcuda_trace_surfaces", "rtcuda_trace_surfaces_device"]
INVALID_ARGUMENT = 1
OFFSETS = {"point": 0, "t": 12, "normal": 16, "material": 28, "uv": 32, "geom_id": 40, "prim_id": 44, "albedo": 48, "light": 60}


@pytest.fixture(scope="module")
def lib(rc):
    return rc._ffi.load_library()


def test_surface_symbols_are_exported_and_bound(rc, lib):
    assert set(SYMBOLS) <= set(rc._ffi.EXPORTED_SYMBOLS)
    assert lib.rtcuda_abi_version() == rc._ffi.ABI_VERSION == 4
    for name in SYMBOLS:
        fn = getattr(lib, name)
        assert fn.argtypes == [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p], name
        assert fn.restype == C.c_int


def test_struct_size_list_is_unchanged(rc, lib):
    """the record is not part of rtcuda_abi_struct_sizes: the list still ends with rtcuda_stats"""
    buf = (C.c_uint32 * 64)()
    n = lib.rtcuda_abi_struct_sizes(buf, 64)
    assert n == len(rc._ffi.ABI_STRUCTS) == 13
    assert list(buf[:n]) == [C.sizeof(s) for s in rc._ffi.ABI_STRUCTS]
    assert rc._ffi.Surface not in rc._ffi.ABI_STRUCTS


def test_surface_record_layout(rc):
    S = rc._ffi.Surface
    assert C.sizeof(S) == 64
    assert {name: getattr(S, name).offset for name, _ in S._fields_} == OFFSETS
    dt = rc.backend.SURFACE_DTYPE
    assert dt.itemsize == 64 and {name: dt.fields[name][1] for name in dt.names} == OFFSETS


@pytest.mark.parametrize("name", SYMBOLS)
def test_malformed_calls_are_refused_before_device_work(rc, lib, name):
    """No scene is needed to reach these checks (there is no GPU here): each refusal names what is wrong"""
    call = getattr(lib, name)
    rays = np.zeros((4, 8), np.float32)
    out = np.zeros((4, 16), np.float32)
    R, O = rays.ctypes.data, out.ctypes.data

    def refused(status, text):
        assert status == INVALID_ARGUMENT and text in lib.rtcuda_last_error().decode(), lib.rtcuda_last_error()

    refused(call(None, R, 1 << 32, O), "below 2^32")
    refused(call(None, None, 4, O), "rays is NULL")
    refused(call(None, R, 4, None), "every output is NULL")
    refused(call(None, None, 0, None), "every output is NULL")
    refused(call(None, R, 4, O), "scene is NULL")
    refused(call(None, None, 0, O), "scene is NULL")


def test_surface_methods_check_the_ray_array(rc):
    """dtype, shape and contiguity are checked in Python before the library is called (no scene is touched)"""
    r = rc.CudaRenderer.__new__(rc.CudaRenderer)
    good = rc.make_rays(np.zeros((4, 3)), [0, 0, 1])
    for bad in (good.astype(np.float64), good[:, :7], good.reshape(-1), good[::2], np.asfortranarray(good), good.tolist()):
        with pytest.raises(ValueError):
            r.surfaces(bad)


def test_ray_surfaces_are_views_of_the_records(rc):
    rec = np.zeros(3, rc.backend.SURFACE_DTYPE)
    s = rc.RaySurfaces.from_records(rec)
    rec["normal"][1] = (0, 0, 1)
    rec["geom_id"][2] = 7
    assert s.normal.shape == (3, 3) and s.uv.shape == (3, 2) and s.albedo.shape == (3, 3) and s.t.shape == (3,)
    assert (s.normal[1] == (0, 0, 1)).all() and s.instance[2] == 7
    assert s.instance.dtype == s.primitive.dtype == s.material.dtype == s.light.dtype == np.uint32
