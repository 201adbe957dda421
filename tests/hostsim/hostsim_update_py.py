"""ctypes binding of tests/hostsim/libhostsim_update.so — TEST INFRASTRUCTURE ONLY (see hostsim_update.cpp): the scene-update
refit bodies of the CUDA library run on the CPU over the harness's scene build."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
import raytracing_cuda as rc  # noqa: E402
from raytracing_cuda import _ffi  # noqa: E402

LIB_PATH = os.path.join(HERE, "libhostsim_update.so")
_lib = None


def build(force=False):
    csrc = os.path.join(ROOT, "opencl-raytracing_b200", "csrc")
    srcs = [os.path.join(HERE, "hostsim_update.cpp"), os.path.join(HERE, "hostsim.cpp")] + \
        [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".h")]
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-o", LIB_PATH, srcs[0]])
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        l = C.CDLL(LIB_PATH)
        l.hostsim_refit_identity.argtypes = [C.POINTER(_ffi.SceneDesc), C.POINTER(C.c_uint32), C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.POINTER(C.c_double)]
        l.hostsim_refit_identity.restype = C.c_int
        l.hostsim_update_render.argtypes = [C.c_int, C.POINTER(_ffi.SceneDesc), C.POINTER(_ffi.SceneDesc), C.POINTER(_ffi.Settings),
                                            C.POINTER(_ffi.Outputs), C.c_double, C.POINTER(C.c_uint64), C.POINTER(C.c_double)]
        l.hostsim_update_render.restype = C.c_int
        _lib = l
    return _lib


def refit_identity(scene):
    """Build `scene`, then refit its tree with the same transforms. Returns the wide nodes and the primitive slots of the build
    and of the refit (float32 [N, 20] / [S, 12]) and the SAH costs (built, refitted)."""
    holder = scene.to_desc()
    counts, sah = (C.c_uint32 * 2)(), (C.c_double * 2)()
    lib().hostsim_refit_identity(C.byref(holder.desc), counts, None, None, None, None, sah)
    n, s = counts
    arrs = [np.zeros((n, 20), np.float32), np.zeros((n, 20), np.float32), np.zeros((s, 12), np.float32), np.zeros((s, 12), np.float32)]
    if lib().hostsim_refit_identity(C.byref(holder.desc), counts, *[a.ctypes.data for a in arrs], sah) != 0:
        raise RuntimeError("hostsim_refit_identity failed")
    return arrs[0], arrs[1], arrs[2], arrs[3], (sah[0], sah[1])


def _render(mode, scene_a, scene_b, settings, max_growth):
    ha, hb = scene_a.to_desc(), scene_b.to_desc()
    out = rc.RenderOutput.allocate(scene_b.camera.raster_width, scene_b.camera.raster_height, rc.AovFlags(settings.outputs))
    s, o = settings.to_c(), out.to_c()
    stats, info = (C.c_uint64 * 2)(), (C.c_double * 2)()
    if lib().hostsim_update_render(mode, C.byref(ha.desc), C.byref(hb.desc), C.byref(s), C.byref(o), max_growth, stats, info) != 0:
        raise RuntimeError("hostsim_update_render failed")
    return out, {"nodes_fetched": stats[0], "prims_fetched": stats[1]}, (int(info[0]), info[1])


def render(scene, settings):
    """build(scene) -> render, with the render loop the update path uses (same frame as hostsim_py.render)"""
    out, stats, _ = _render(0, scene, scene, settings, 0.0)
    return out, stats


def update_render(scene_a, scene_b, settings, max_growth=1e30):
    """build(scene_a) -> update to scene_b's camera / instance transforms / lights (the refit is replaced by a rebuild when its
    SAH cost exceeds max_growth x the built tree's: 0 forces the rebuild) -> render. Returns the frame, the fetch counts and
    (bvh_last_update, SAH cost after the update)."""
    return _render(1, scene_a, scene_b, settings, max_growth)
