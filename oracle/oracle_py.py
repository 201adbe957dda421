"""ctypes binding of oracle/liboracle.so — TEST INFRASTRUCTURE ONLY (see the header of oracle.cpp).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module. The product package never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(_HERE))
import raytracing_cuda as rc  # noqa: E402  (vocabulary types only: Scene, RaytracerSettings, RenderOutput)
from raytracing_cuda import _ffi  # noqa: E402

LIB_PATH = os.path.join(_HERE, "liboracle.so")
FLAG_BRUTE_FORCE = 1


class OracleStats(C.Structure):
    _fields_ = [("primary_rays", C.c_uint64), ("bounce_rays", C.c_uint64), ("shadow_rays", C.c_uint64),
                ("aov_rays", C.c_uint64), ("render_ms", C.c_double), ("build_ms", C.c_double), ("bvh_nodes", C.c_uint64)]


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "oracle.cpp")
    hdr = os.path.join(os.path.dirname(_HERE), "include", "rtcuda.h")
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.check_call(["make", "-C", _HERE, "-B", "liboracle.so"], stdout=subprocess.DEVNULL)
    return LIB_PATH


_lib = None
_lib_path = LIB_PATH


def use_native_build() -> str:
    """The CPU-baseline build (bench.py): the same oracle.cpp compiled `-O3 -march=native` ON THE HOST IT RUNS ON
    (BASELINE.md / SURVEY 8d), still -ffp-contract=off so its pixels are the portable build's. Kept apart from liboracle.so,
    which is built -O2 for any x86-64 host because the prebuilt file may be loaded on another host than the one that built it.
    The native library goes to a temporary directory of this process (removed at exit), so that the source tree may be read-only."""
    global _lib, _lib_path
    import atexit
    import shutil
    import tempfile
    if _lib_path != LIB_PATH:   # already built by this process
        return _lib_path
    tmp = tempfile.mkdtemp(prefix="raytracing_cuda_oracle_")
    atexit.register(shutil.rmtree, tmp, ignore_errors=True)
    path = os.path.join(tmp, "liboracle_native.so")
    src = os.path.join(_HERE, "oracle.cpp")
    subprocess.check_call(["g++", "-O3", "-march=native", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-pthread",
                           "-shared", "-o", path, src])
    _lib, _lib_path = None, path
    return path


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if _lib_path == LIB_PATH and not os.path.exists(LIB_PATH):
            build()
        l = C.CDLL(_lib_path)
        l.oracle_render.argtypes = [C.POINTER(_ffi.SceneDesc), C.POINTER(_ffi.Settings), C.POINTER(_ffi.Outputs), C.c_uint32,
                                    C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(OracleStats)]
        l.oracle_render.restype = C.c_int
        l.oracle_render_pixel.argtypes = [C.POINTER(_ffi.SceneDesc), C.POINTER(_ffi.Settings), C.c_uint32, C.c_uint32,
                                          C.c_uint32, C.c_uint32, C.POINTER(_ffi.PixelOutput), C.c_uint32]
        l.oracle_render_pixel.restype = C.c_int
        l.oracle_abi_struct_sizes.argtypes = [C.POINTER(C.c_uint32), C.c_uint32]
        l.oracle_abi_struct_sizes.restype = C.c_uint32
        l.oracle_fxhash_u32x3.argtypes = [C.c_uint32] * 3
        l.oracle_fxhash_u32x3.restype = C.c_uint64
        l.oracle_fxhash_u64.argtypes = [C.c_uint64]
        l.oracle_fxhash_u64.restype = C.c_uint64
        l.oracle_pcg32_stream.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint32)]
        l.oracle_pcg32_raw.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint32)]
        l.oracle_permute.argtypes = [C.c_uint32] * 3
        l.oracle_permute.restype = C.c_uint32
        l.oracle_range_u32.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32]
        l.oracle_range_u32.restype = C.c_uint32
        fp = C.POINTER(C.c_float)
        l.oracle_make_orthonormal_basis.argtypes = [fp, fp, fp]
        l.oracle_ray_sphere.argtypes = [fp, C.c_float, fp, fp, C.c_float, C.c_float, fp]
        l.oracle_ray_sphere.restype = C.c_int
        l.oracle_ray_triangle.argtypes = [fp, fp, fp, C.c_float, C.c_float, fp]
        l.oracle_ray_triangle.restype = C.c_int
        l.oracle_sampler_stream.argtypes = [C.POINTER(_ffi.Settings), C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, fp]
        l.oracle_sample_texture.argtypes = [C.POINTER(_ffi.SceneDesc), C.c_uint32, fp, fp]
        l.oracle_mip_level.argtypes = [C.POINTER(_ffi.SceneDesc), C.c_uint32, C.c_uint32, C.POINTER(C.c_uint8),
                                       C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        l.oracle_mip_level.restype = C.c_uint32
        l.oracle_bsdf.argtypes = [C.POINTER(_ffi.SceneDesc), C.POINTER(_ffi.Settings), C.c_uint32, C.c_int, fp, fp, C.c_uint32, fp]
        sizes = (C.c_uint32 * 32)()
        n = l.oracle_abi_struct_sizes(sizes, 32)
        mine = [C.sizeof(s) for s in _ffi.ABI_STRUCTS]
        if list(sizes[:n]) != mine:
            raise RuntimeError(f"oracle ABI struct size mismatch: {list(sizes[:n])} vs {mine}")
        _lib = l
    return _lib


def _fa(values):
    return (C.c_float * len(values))(*[float(v) for v in values])


def render(scene, settings, num_threads: int = 1, brute_force: bool = False, tile_rank: int = 0, tile_world: int = 1):
    """oracle_render -> (RenderOutput, stats dict)."""
    holder = scene.to_desc()
    out = rc.RenderOutput.allocate(scene.camera.raster_width, scene.camera.raster_height, rc.AovFlags(settings.outputs))
    s, o, st = settings.to_c(), out.to_c(), OracleStats()
    rcode = lib().oracle_render(C.byref(holder.desc), C.byref(s), C.byref(o), num_threads,
                                FLAG_BRUTE_FORCE if brute_force else 0, tile_rank, tile_world, C.byref(st))
    if rcode != 0:
        raise RuntimeError("oracle_render failed")
    return out, {n: getattr(st, n) for n, _ in OracleStats._fields_}


def render_pixel(scene, settings, x, y, lo, hi, brute_force: bool = False):
    holder = scene.to_desc()
    n = max(0, hi - lo)
    buf = (_ffi.PixelOutput * max(1, n))()
    s = settings.to_c()
    if lib().oracle_render_pixel(C.byref(holder.desc), C.byref(s), x, y, lo, hi, buf, FLAG_BRUTE_FORCE if brute_force else 0) != 0:
        raise RuntimeError("oracle_render_pixel failed")
    return [rc.SinglePixelOutput(b.sample_index, bool(b.hit), tuple(b.uv), tuple(b.normal), tuple(b.radiance)) for b in buf[:n]]
