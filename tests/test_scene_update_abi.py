"""CPU-side checks of the scene-update ABI (v4): the entry point is exported and bound, the v4 stats fields sit at the end of
rtcuda_stats as compiled, and NULL arguments are refused before any device work."""
import ctypes as C

from conftest import load_scene


def test_scene_update_is_exported_and_bound(rc):
    lib = rc._ffi.load_library()
    assert "rtcuda_scene_update" in rc._ffi.EXPORTED_SYMBOLS
    assert lib.rtcuda_scene_update.argtypes == [C.c_void_p, C.POINTER(rc._ffi.SceneDesc)]
    assert lib.rtcuda_abi_version() == rc._ffi.ABI_VERSION == 4


def test_stats_v4_fields_match_the_library(rc):
    lib = rc._ffi.load_library()
    sizes = (C.c_uint32 * 32)()
    n = lib.rtcuda_abi_struct_sizes(sizes, 32)
    assert sizes[n - 1] == C.sizeof(rc._ffi.Stats)
    names = [f for f, _ in rc._ffi.Stats._fields_]
    assert names[-3:] == ["update_ms", "bvh_sah_cost", "bvh_last_update"]
    assert rc._ffi.Stats.bvh_last_update.offset + 8 == C.sizeof(rc._ffi.Stats)
    assert rc._ffi.Stats.update_ms.offset == rc._ffi.Stats.pixels_dropped.offset + 8


def test_null_scene_or_desc_is_an_invalid_argument(rc):
    lib = rc._ffi.load_library()
    holder = load_scene("cb", 64, 36).to_desc()
    assert lib.rtcuda_scene_update(None, C.byref(holder.desc)) == 1   # RTCUDA_ERR_INVALID_ARGUMENT
    assert b"null argument" in lib.rtcuda_last_error()
    assert lib.rtcuda_scene_update(C.c_void_p(0x1000), None) == 1
