"""ctypes binding of tests/hostsim/libhostsim.so — TEST INFRASTRUCTURE ONLY (see hostsim.cpp): the
per-thread kernel bodies of the CUDA library compiled for the CPU and run sequentially."""
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
from raytracing_cuda.backend import SURFACE_DTYPE  # noqa: E402

LIB_PATH = os.path.join(HERE, "libhostsim.so")
_lib = None

STATS = ["primary_rays", "bounce_rays", "shadow_rays", "aov_rays", "nodes_fetched", "prims_fetched", "bvh_node_count", "collapse_levels"]


def build(force=False):
    """make the library when it is missing or older than a source it compiles (the Makefile rule holds the flags)"""
    csrc = os.path.join(ROOT, "opencl-raytracing_b200", "csrc")
    srcs = [os.path.join(HERE, "hostsim.cpp"), os.path.join(ROOT, "include", "rtcuda.h")] + \
        [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".h")]
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["make", "-C", ROOT, "-B", os.path.relpath(LIB_PATH, ROOT)], stdout=subprocess.DEVNULL)
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        l = C.CDLL(LIB_PATH)
        scene, settings, outputs, vp = C.POINTER(_ffi.SceneDesc), C.POINTER(_ffi.Settings), C.POINTER(_ffi.Outputs), C.c_void_p
        l.hostsim_render.argtypes = [scene, settings, outputs, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint64)]
        l.hostsim_render_samples.argtypes = l.hostsim_render.argtypes + [C.c_uint32, C.c_uint32]
        fp = C.POINTER(C.c_float)
        l.hostsim_ray_triangle.argtypes = [C.c_int, fp, fp, fp, fp, fp, C.c_float, C.c_float, fp]
        l.hostsim_raster_rect.argtypes = [scene, C.POINTER(C.c_int)]
        l.hostsim_refit_identity.argtypes = [scene, C.POINTER(C.c_uint32), vp, vp, vp, vp, C.POINTER(C.c_double)]
        l.hostsim_update_render.argtypes = [scene, scene, settings, outputs, C.c_double, C.POINTER(C.c_uint64), C.POINTER(C.c_double)]
        l.hostsim_trace_rays.argtypes = [scene, vp, C.c_uint64, vp, vp, vp, vp]
        l.hostsim_trace_surfaces.argtypes = [scene, vp, C.c_uint64, vp]
        l.hostsim_radiance.argtypes = [scene, settings, vp, C.c_uint64, C.c_uint32, C.c_uint32, vp, vp]
        for f in (l.hostsim_render, l.hostsim_render_samples, l.hostsim_ray_triangle, l.hostsim_raster_rect, l.hostsim_refit_identity,
                  l.hostsim_update_render, l.hostsim_trace_rays, l.hostsim_trace_surfaces, l.hostsim_radiance):
            f.restype = C.c_int
        _lib = l
    return _lib


def render(scene, settings, tile_rank=0, tile_world=1, capacity=0, sample_range=None):
    """sample_range=(lo, hi): only those samples, the beauty plane holds their un-normalised sum (rtcuda_render_samples_device)"""
    holder = scene.to_desc()
    out = rc.RenderOutput.allocate(scene.camera.raster_width, scene.camera.raster_height, rc.AovFlags(settings.outputs))
    s, o = settings.to_c(), out.to_c()
    stats = (C.c_uint64 * 8)()
    lo, hi = sample_range if sample_range is not None else (0, 0)
    if lib().hostsim_render_samples(C.byref(holder.desc), C.byref(s), C.byref(o), tile_rank, tile_world, capacity, stats, lo, hi) != 0:
        raise RuntimeError("hostsim_render failed")
    return out, dict(zip(STATS, list(stats)))


def ray_triangle(mode, p0, p1, p2, o, d, t_min=0.0, t_max=float("inf")):
    """(hit, t, u, v) of the kernel-side triangle tests: mode 0 = Moller-Trumbore (reference), 1 = watertight"""
    fa = lambda v: (C.c_float * 3)(*[float(x) for x in v])
    out = (C.c_float * 3)()
    h = lib().hostsim_ray_triangle(mode, fa(p0), fa(p1), fa(p2), fa(o), fa(d), t_min, t_max, out)
    return bool(h), out[0], out[1], out[2]


def raster_rect(scene):
    """rt_cull.h scene_raster_rect: (x0, y0, x1, y1) inclusive, or None when every pixel is kept"""
    holder = scene.to_desc()
    rect = (C.c_int * 4)()
    return tuple(rect) if lib().hostsim_raster_rect(C.byref(holder.desc), rect) else None


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


def update_render(scene_a, scene_b, settings, max_growth=1e30):
    """build(scene_a) -> update to scene_b's camera / instance transforms / lights (the refit is replaced by a rebuild when its
    SAH cost exceeds max_growth x the built tree's: 0 forces the rebuild) -> render. Returns the frame, the stats of render()
    and (bvh_last_update, SAH cost after the update)."""
    ha, hb = scene_a.to_desc(), scene_b.to_desc()
    out = rc.RenderOutput.allocate(scene_b.camera.raster_width, scene_b.camera.raster_height, rc.AovFlags(settings.outputs))
    s, o = settings.to_c(), out.to_c()
    stats, info = (C.c_uint64 * 8)(), (C.c_double * 2)()
    if lib().hostsim_update_render(C.byref(ha.desc), C.byref(hb.desc), C.byref(s), C.byref(o), max_growth, stats, info) != 0:
        raise RuntimeError("hostsim_update_render failed")
    return out, dict(zip(STATS, list(stats))), (int(info[0]), info[1])


def trace_rays(scene, rays):
    """rt_query.h on the CPU over the harness's build of `scene` (RTCUDA_BUILDER / HOSTSIM_WATERTIGHT apply): (t [N] float32,
    ids [N, 2] uint32, barycentrics [N, 2] float32, occluded [N] uint8) for packed rays [N, 8]"""
    rays = np.ascontiguousarray(rays, dtype=np.float32)
    n = rays.shape[0]
    holder = scene.to_desc()
    t, ids, uv, occ = np.empty(n, np.float32), np.empty((n, 2), np.uint32), np.empty((n, 2), np.float32), np.empty(n, np.uint8)
    if lib().hostsim_trace_rays(C.byref(holder.desc), rays.ctypes.data, n, t.ctypes.data, ids.ctypes.data, uv.ctypes.data, occ.ctypes.data) != 0:
        raise RuntimeError("hostsim_trace_rays failed")
    return t, ids, uv, occ


def trace_surfaces(scene, rays):
    """query_closest_ray + surface_finish_body (rt_query.h) on the CPU over the harness's build of `scene` (RTCUDA_BUILDER /
    HOSTSIM_WATERTIGHT apply): one rtcuda_surface record per packed ray [N, 8] (raytracing_cuda.backend.SURFACE_DTYPE [N])"""
    rays = np.ascontiguousarray(rays, dtype=np.float32)
    holder = scene.to_desc()
    rec = np.empty(rays.shape[0], SURFACE_DTYPE)
    if lib().hostsim_trace_surfaces(C.byref(holder.desc), rays.ctypes.data, rays.shape[0], rec.ctypes.data) != 0:
        raise RuntimeError("hostsim_trace_surfaces failed")
    return rec


def radiance(scene, settings, rays, stream_base=0, capacity=0):
    """rtcuda_radiance's bodies on the CPU over the harness's build of `scene`, in batches of `capacity` path slots (0: 2^20):
    (radiance [N, 3] float32, prepared rays [N, 8] float32) for packed rays [N, 8]"""
    rays = np.ascontiguousarray(rays, dtype=np.float32)
    n = rays.shape[0]
    holder = scene.to_desc()
    s = settings.to_c()
    out, prep = np.empty((n, 3), np.float32), np.empty((n, 8), np.float32)
    if lib().hostsim_radiance(C.byref(holder.desc), C.byref(s), rays.ctypes.data, n, stream_base, capacity, out.ctypes.data, prep.ctypes.data) != 0:
        raise RuntimeError("hostsim_radiance failed")
    return out, prep
