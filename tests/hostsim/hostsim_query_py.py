"""ctypes bindings of the ray-query test libraries — TEST INFRASTRUCTURE ONLY:
  tests/hostsim/libhostsim_query.so (hostsim_query.cpp): the query bodies of the CUDA library (rt_query.h) run on the CPU;
  tests/hostsim/liboracle_query.so (oracle_query.cpp): their reference, the CPU oracle's traverse_bvh per ray.
Both return (t [N] float32, ids [N, 2] uint32, barycentrics [N, 2] float32, occluded [N] uint8) for packed rays [N, 8]."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from raytracing_cuda import _ffi  # noqa: E402

HOSTSIM_LIB = os.path.join(HERE, "libhostsim_query.so")
ORACLE_LIB = os.path.join(HERE, "liboracle_query.so")
FLAG_BRUTE_FORCE = 1
_libs = {}


def _build(path, force=False):
    """make the library when it is missing or older than its sources (the Makefile rule holds the flags)"""
    csrc = os.path.join(ROOT, "opencl-raytracing_b200", "csrc")
    srcs = [os.path.join(HERE, f) for f in ("hostsim.cpp", "hostsim_query.cpp", "oracle_query.cpp")] + \
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
        l = C.CDLL(path)
        fn = getattr(l, symbol)
        fn.argtypes = [C.POINTER(_ffi.SceneDesc), C.c_void_p, C.c_uint64] + extra + [C.c_void_p] * 4
        fn.restype = C.c_int
        _libs[path] = fn
    return _libs[path]


def _run(fn, scene, rays, *extra):
    rays = np.ascontiguousarray(rays, dtype=np.float32)
    n = rays.shape[0]
    holder = scene.to_desc()
    t, ids, uv, occ = np.empty(n, np.float32), np.empty((n, 2), np.uint32), np.empty((n, 2), np.float32), np.empty(n, np.uint8)
    if fn(C.byref(holder.desc), rays.ctypes.data, n, *extra, t.ctypes.data, ids.ctypes.data, uv.ctypes.data, occ.ctypes.data) != 0:
        raise RuntimeError("ray query harness failed")
    return t, ids, uv, occ


def trace_rays(scene, rays):
    """rt_query.h on the CPU over the harness's build of `scene` (RTCUDA_BUILDER / HOSTSIM_WATERTIGHT apply)"""
    return _run(_lib(HOSTSIM_LIB, "hostsim_trace_rays", []), scene, rays)


def oracle_trace_rays(scene, rays, brute_force=False):
    """the reference: traverse_bvh per ray over the oracle's BVH2 (or every primitive in build order)"""
    return _run(_lib(ORACLE_LIB, "oracle_trace_rays", [C.c_uint32]), scene, rays, FLAG_BRUTE_FORCE if brute_force else 0)
