"""ctypes bindings of the radiance test libraries — TEST INFRASTRUCTURE ONLY:
  tests/hostsim/libhostsim_radiance.so (hostsim_radiance.cpp): rtcuda_radiance's bodies (rt_query.h + the wavefront) on the CPU;
  tests/hostsim/liboracle_radiance.so (oracle_radiance.cpp): their reference, the CPU oracle's ray_radiance per ray and sample.
Both return (radiance [N, 3] float32, prepared rays [N, 8] float32) for packed rays [N, 8]."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from raytracing_cuda import _ffi  # noqa: E402

HOSTSIM_LIB = os.path.join(HERE, "libhostsim_radiance.so")
ORACLE_LIB = os.path.join(HERE, "liboracle_radiance.so")
_libs = {}


def _build(path, force=False):
    """make the library when it is missing or older than its sources (the Makefile rule holds the flags)"""
    csrc = os.path.join(ROOT, "opencl-raytracing_b200", "csrc")
    srcs = [os.path.join(HERE, f) for f in ("hostsim.cpp", "hostsim_radiance.cpp", "oracle_radiance.cpp")] + \
        [os.path.join(ROOT, "oracle", "oracle.cpp"), os.path.join(ROOT, "include", "rtcuda.h")] + \
        [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".h")]
    if force or not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["make", "-C", ROOT, "-B", os.path.relpath(path, ROOT)], stdout=subprocess.DEVNULL)
    return path


def build(force=False):
    _build(HOSTSIM_LIB, force)
    _build(ORACLE_LIB, force)


def _lib(path, symbol):
    if path not in _libs:
        _build(path)
        fn = getattr(C.CDLL(path), symbol)
        fn.argtypes = [C.POINTER(_ffi.SceneDesc), C.POINTER(_ffi.Settings), C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32,
                       C.c_void_p, C.c_void_p]
        fn.restype = C.c_int
        _libs[path] = fn
    return _libs[path]


def _run(fn, scene, settings, rays, stream_base, extra):
    rays = np.ascontiguousarray(rays, dtype=np.float32)
    n = rays.shape[0]
    holder = scene.to_desc()
    s = settings.to_c()
    out, prep = np.empty((n, 3), np.float32), np.empty((n, 8), np.float32)
    if fn(C.byref(holder.desc), C.byref(s), rays.ctypes.data, n, stream_base, extra, out.ctypes.data, prep.ctypes.data) != 0:
        raise RuntimeError("radiance harness failed")
    return out, prep


def radiance(scene, settings, rays, stream_base=0, capacity=0):
    """rtcuda_radiance's bodies on the CPU over the harness's build of `scene`, in batches of `capacity` path slots (0: 2^20)"""
    return _run(_lib(HOSTSIM_LIB, "hostsim_radiance"), scene, settings, rays, stream_base, capacity)


def oracle_radiance(scene, settings, rays, stream_base=0, num_threads=8):
    """the reference: the oracle's ray_radiance per ray and sample over the ray's normalised range"""
    return _run(_lib(ORACLE_LIB, "oracle_radiance"), scene, settings, rays, stream_base, num_threads)
