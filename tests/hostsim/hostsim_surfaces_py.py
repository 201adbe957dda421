"""ctypes bindings of the surface-query test libraries — TEST INFRASTRUCTURE ONLY:
  tests/hostsim/libhostsim_surfaces.so (hostsim_surfaces.cpp): the surface-query body of the CUDA library (rt_query.h) on the CPU;
  tests/hostsim/liboracle_surfaces.so (oracle_surfaces.cpp): its reference, the CPU oracle's traverse_bvh HitInfo and get_albedo.
Both return one rtcuda_surface record per packed ray [N, 8] (raytracing_cuda.backend.SURFACE_DTYPE [N])."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from raytracing_cuda import _ffi  # noqa: E402
from raytracing_cuda.backend import SURFACE_DTYPE  # noqa: E402

HOSTSIM_LIB = os.path.join(HERE, "libhostsim_surfaces.so")
ORACLE_LIB = os.path.join(HERE, "liboracle_surfaces.so")
FLAG_BRUTE_FORCE = 1
_libs = {}


def _build(path, force=False):
    """make the library when it is missing or older than its sources (the Makefile rule holds the flags)"""
    csrc = os.path.join(ROOT, "opencl-raytracing_b200", "csrc")
    srcs = [os.path.join(HERE, f) for f in ("hostsim.cpp", "hostsim_surfaces.cpp", "oracle_surfaces.cpp")] + \
        [os.path.join(ROOT, "oracle", "oracle.cpp"), os.path.join(ROOT, "include", "rtcuda.h")] + \
        [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".h")]
    if force or not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["make", "-C", ROOT, "-B", os.path.relpath(path, ROOT)], stdout=subprocess.DEVNULL)
    return path


def build(force=False):
    _build(HOSTSIM_LIB, force)
    _build(ORACLE_LIB, force)


def _lib(path, symbol, extra):
    if path not in _libs:
        _build(path)
        fn = getattr(C.CDLL(path), symbol)
        fn.argtypes = [C.POINTER(_ffi.SceneDesc), C.c_void_p, C.c_uint64] + extra + [C.c_void_p]
        fn.restype = C.c_int
        _libs[path] = fn
    return _libs[path]


def _run(fn, scene, rays, *extra):
    rays = np.ascontiguousarray(rays, dtype=np.float32)
    n = rays.shape[0]
    holder = scene.to_desc()
    rec = np.empty(n, SURFACE_DTYPE)
    if fn(C.byref(holder.desc), rays.ctypes.data, n, *extra, rec.ctypes.data) != 0:
        raise RuntimeError("surface query harness failed")
    return rec


def trace_surfaces(scene, rays):
    """query_closest_ray + surface_finish_body (rt_query.h) on the CPU over the harness's build of `scene` (RTCUDA_BUILDER /
    HOSTSIM_WATERTIGHT apply)"""
    return _run(_lib(HOSTSIM_LIB, "hostsim_trace_surfaces", []), scene, rays)


def oracle_trace_surfaces(scene, rays, brute_force=False):
    """the reference: traverse_bvh's HitInfo per ray over the oracle's BVH2 (or every primitive in build order) and get_albedo
    with a zero footprint"""
    return _run(_lib(ORACLE_LIB, "oracle_trace_surfaces", [C.c_uint32]), scene, rays, FLAG_BRUTE_FORCE if brute_force else 0)
