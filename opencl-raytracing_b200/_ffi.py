"""ctypes mirror of include/rtcuda.h and loader of libraytracing_cuda.so.

This is the binding a `raytracing-cuda` crate would get from bindgen (the reference does the same for
its OptiX backend: crates/raytracing-optix/build.rs:3-55 over csrc/host/lib_api.h). The library is the
product path: if it is missing or fails to load this module raises — there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

NONE = 0xFFFFFFFF
ABI_VERSION = 4
MAX_DEVICES = 8

# enums (values must match rtcuda.h)
CAMERA_ORTHOGRAPHIC, CAMERA_PINHOLE, CAMERA_THIN_LENS = 0, 1, 2
SHAPE_TRIANGLE_MESH, SHAPE_SPHERE = 0, 1
LIGHT_POINT, LIGHT_DIRECTION, LIGHT_DIFFUSE_AREA = 0, 1, 2
(MATERIAL_DIFFUSE, MATERIAL_SMOOTH_DIELECTRIC, MATERIAL_SMOOTH_CONDUCTOR, MATERIAL_ROUGH_DIELECTRIC,
 MATERIAL_ROUGH_CONDUCTOR, MATERIAL_COATED_DIFFUSE) = range(6)
TEXTURE_IMAGE, TEXTURE_CONSTANT, TEXTURE_CHECKER, TEXTURE_SCALE, TEXTURE_MIX = range(5)
FILTER_NEAREST, FILTER_BILINEAR, FILTER_TRILINEAR = range(3)
WRAP_REPEAT, WRAP_MIRROR, WRAP_CLAMP = range(3)
IMAGE_U8, IMAGE_U16, IMAGE_F32 = range(3)
SAMPLER_INDEPENDENT, SAMPLER_STRATIFIED = 0, 1

STATUS_NAMES = {0: "OK", 1: "INVALID_ARGUMENT", 2: "CUDA", 3: "UNSUPPORTED", 4: "NO_DEVICE", 5: "OUT_OF_MEMORY"}


class Mat4(C.Structure):
    _fields_ = [("m", C.c_float * 16)]


class Transform(C.Structure):
    _fields_ = [("forward", Mat4), ("inverse", Mat4)]


class Camera(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("raster_width", C.c_uint32), ("raster_height", C.c_uint32),
                ("near_clip", C.c_float), ("far_clip", C.c_float), ("yfov", C.c_float),
                ("aperture_radius", C.c_float), ("focal_distance", C.c_float),
                ("screen_space_width", C.c_float), ("screen_space_height", C.c_float),
                ("world_to_raster", Transform), ("camera_to_world", Transform), ("raster_to_camera", Transform)]


class Shape(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("material", C.c_uint32), ("area_light", C.c_uint32),
                ("vertex_offset", C.c_uint32), ("vertex_count", C.c_uint32),
                ("tri_offset", C.c_uint32), ("tri_count", C.c_uint32),
                ("normal_offset", C.c_uint32), ("uv_offset", C.c_uint32),
                ("center", C.c_float * 3), ("radius", C.c_float),
                ("vertices", C.POINTER(C.c_float)), ("tris", C.POINTER(C.c_uint32)),
                ("normals", C.POINTER(C.c_float)), ("uvs", C.POINTER(C.c_float))]


class Instance(C.Structure):
    _fields_ = [("shape", C.c_uint32), ("_pad", C.c_uint32 * 3), ("object_to_world", Transform)]


class Light(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("shape", C.c_uint32),
                ("position_or_direction", C.c_float * 3), ("intensity_or_radiance", C.c_float * 3),
                ("light_to_world", Mat4)]


class Material(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("remap_roughness", C.c_uint32), ("albedo", C.c_uint32), ("eta", C.c_uint32),
                ("kappa", C.c_uint32), ("roughness", C.c_uint32), ("thickness", C.c_uint32), ("coat_albedo", C.c_uint32)]


class Texture(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("image", C.c_uint32), ("filter", C.c_uint32), ("wrap", C.c_uint32),
                ("a", C.c_uint32), ("b", C.c_uint32), ("c", C.c_uint32), ("_pad", C.c_uint32),
                ("value", C.c_float * 4), ("value2", C.c_float * 4)]


class Image(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("channels", C.c_uint32), ("format", C.c_uint32),
                ("byte_offset", C.c_uint64)]


class SceneDesc(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("_pad", C.c_uint32), ("camera", Camera),
                ("shapes", C.POINTER(Shape)), ("shape_count", C.c_uint32),
                ("instances", C.POINTER(Instance)), ("instance_count", C.c_uint32),
                ("lights", C.POINTER(Light)), ("light_count", C.c_uint32),
                ("materials", C.POINTER(Material)), ("material_count", C.c_uint32),
                ("textures", C.POINTER(Texture)), ("texture_count", C.c_uint32),
                ("images", C.POINTER(Image)), ("image_count", C.c_uint32),
                ("environment_light_texture", C.c_uint32), ("_pad2", C.c_uint32),
                ("vertices", C.POINTER(C.c_float)), ("vertex_count", C.c_uint64),
                ("tris", C.POINTER(C.c_uint32)), ("tri_count", C.c_uint64),
                ("normals", C.POINTER(C.c_float)), ("normal_count", C.c_uint64),
                ("uvs", C.POINTER(C.c_float)), ("uv_count", C.c_uint64),
                ("image_bytes", C.POINTER(C.c_uint8)), ("image_byte_count", C.c_uint64)]


class Settings(C.Structure):
    _fields_ = [("max_ray_depth", C.c_uint32), ("accumulate_bounces", C.c_uint32), ("light_sample_count", C.c_uint32),
                ("samples_per_pixel", C.c_uint32), ("has_seed", C.c_uint32), ("sampler_kind", C.c_uint32),
                ("seed", C.c_uint64), ("stratified_jitter", C.c_uint32), ("x_strata", C.c_uint32),
                ("y_strata", C.c_uint32), ("outputs", C.c_uint32), ("antialias_primary_rays", C.c_uint32),
                ("antialias_secondary_rays", C.c_uint32)]


class BackendSettings(C.Structure):
    _fields_ = [("device_id", C.c_int32), ("max_paths_in_flight", C.c_uint32), ("tile_rank", C.c_uint32),
                ("tile_world", C.c_uint32), ("collect_stats", C.c_uint32), ("flags", C.c_uint32),
                ("tile_size", C.c_uint32), ("num_devices", C.c_uint32), ("device_ids", C.c_int32 * 8)]


class Outputs(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32),
                ("beauty", C.c_void_p), ("normals", C.c_void_p), ("albedo", C.c_void_p), ("uv", C.c_void_p),
                ("mip_level", C.c_void_p), ("debug_ids", C.c_void_p), ("debug_depth", C.c_void_p)]


class PixelOutput(C.Structure):
    _fields_ = [("sample_index", C.c_uint32), ("hit", C.c_uint32), ("uv", C.c_float * 2),
                ("normal", C.c_float * 3), ("radiance", C.c_float * 3)]


class Stats(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("primary_rays", C.c_uint64), ("bounce_rays", C.c_uint64),
                ("shadow_rays", C.c_uint64), ("aov_rays", C.c_uint64), ("nodes_fetched", C.c_uint64),
                ("prims_fetched", C.c_uint64), ("extend_nodes", C.c_uint64), ("extend_prims", C.c_uint64),
                ("shadow_nodes", C.c_uint64), ("shadow_prims", C.c_uint64), ("shaded_vertices", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("extend_launches", C.c_uint64), ("shade_launches", C.c_uint64),
                ("shadow_launches", C.c_uint64), ("render_ms", C.c_double), ("bvh_build_ms", C.c_double),
                ("upload_ms", C.c_double), ("extend_ms", C.c_double), ("shade_ms", C.c_double),
                ("shadow_ms", C.c_double), ("other_ms", C.c_double), ("bvh_node_count", C.c_uint64),
                ("bvh_prim_count", C.c_uint64), ("nonfinite_values", C.c_uint64), ("primary_rays_culled", C.c_uint64), ("final_rays_skipped", C.c_uint64), ("bvh_fallback_lbvh", C.c_uint64),
                ("gather_ms", C.c_double), ("pixels_dropped", C.c_uint64),
                ("update_ms", C.c_double), ("bvh_sah_cost", C.c_double), ("bvh_last_update", C.c_uint64)]


STATS_COUNTERS, STATS_KERNEL_TIMES = 1, 2
BACKEND_WATERTIGHT = 1

ABI_STRUCTS = [Camera, Shape, Instance, Light, Material, Texture, Image, SceneDesc, Settings, BackendSettings,
               Outputs, PixelOutput, Stats]

# every symbol include/rtcuda.h declares
EXPORTED_SYMBOLS = ["rtcuda_init", "rtcuda_shutdown", "rtcuda_scene_upload", "rtcuda_scene_update", "rtcuda_scene_release", "rtcuda_release_cached_memory", "rtcuda_render",
                    "rtcuda_render_device", "rtcuda_render_samples_device", "rtcuda_render_samples_accumulate_device", "rtcuda_render_pixel", "rtcuda_get_stats", "rtcuda_last_error",
                    "rtcuda_abi_version", "rtcuda_abi_struct_sizes", "rtcuda_host_alloc", "rtcuda_host_free", "rtcuda_trace_rays",
                    "rtcuda_trace_rays_device", "rtcuda_occluded", "rtcuda_occluded_device", "rtcuda_radiance", "rtcuda_radiance_device"]

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libraytracing_cuda.so")

_lib = None


class RtCudaError(RuntimeError):
    pass


def load_library(path: str | None = None) -> C.CDLL:
    """dlopen libraytracing_cuda.so and declare its prototypes. Raises when the library is absent:
    the CUDA extension IS the backend, nothing else can serve render()."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise RtCudaError(f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback for the cuda backend)")
    lib = C.CDLL(path)
    lib.rtcuda_init.argtypes = [C.POINTER(BackendSettings), C.POINTER(C.c_void_p)]
    lib.rtcuda_init.restype = C.c_int
    lib.rtcuda_shutdown.argtypes = [C.c_void_p]
    lib.rtcuda_shutdown.restype = None
    lib.rtcuda_scene_upload.argtypes = [C.c_void_p, C.POINTER(SceneDesc), C.POINTER(C.c_void_p)]
    lib.rtcuda_scene_upload.restype = C.c_int
    lib.rtcuda_scene_update.argtypes = [C.c_void_p, C.POINTER(SceneDesc)]
    lib.rtcuda_scene_update.restype = C.c_int
    lib.rtcuda_scene_release.argtypes = [C.c_void_p]
    lib.rtcuda_scene_release.restype = None
    lib.rtcuda_host_alloc.argtypes = [C.c_size_t]
    lib.rtcuda_host_alloc.restype = C.c_void_p
    lib.rtcuda_host_free.argtypes = [C.c_void_p]
    lib.rtcuda_host_free.restype = None
    lib.rtcuda_release_cached_memory.argtypes = []
    lib.rtcuda_release_cached_memory.restype = None
    lib.rtcuda_render.argtypes = [C.c_void_p, C.POINTER(Settings), C.POINTER(Outputs)]
    lib.rtcuda_render.restype = C.c_int
    lib.rtcuda_render_device.argtypes = [C.c_void_p, C.POINTER(Settings), C.POINTER(Outputs)]
    lib.rtcuda_render_device.restype = C.c_int
    lib.rtcuda_render_samples_device.argtypes = [C.c_void_p, C.POINTER(Settings), C.c_uint32, C.c_uint32, C.c_void_p]
    lib.rtcuda_render_samples_device.restype = C.c_int
    lib.rtcuda_render_samples_accumulate_device.argtypes = [C.c_void_p, C.POINTER(Settings), C.c_uint32, C.c_uint32, C.c_void_p]
    lib.rtcuda_render_samples_accumulate_device.restype = C.c_int
    lib.rtcuda_render_pixel.argtypes = [C.c_void_p, C.POINTER(Settings), C.c_uint32, C.c_uint32, C.c_uint32,
                                        C.c_uint32, C.POINTER(PixelOutput)]
    lib.rtcuda_render_pixel.restype = C.c_int
    # ray queries: scene, rays (count x 8 floats), count, then the outputs (host or device addresses; None = skip)
    lib.rtcuda_trace_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rtcuda_trace_rays.restype = C.c_int
    lib.rtcuda_trace_rays_device.argtypes = lib.rtcuda_trace_rays.argtypes
    lib.rtcuda_trace_rays_device.restype = C.c_int
    lib.rtcuda_occluded.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
    lib.rtcuda_occluded.restype = C.c_int
    lib.rtcuda_occluded_device.argtypes = lib.rtcuda_occluded.argtypes
    lib.rtcuda_occluded_device.restype = C.c_int
    # radiance along rays: scene, settings, rays (count x 8 floats), count, stream_base, radiance (count x 3 floats)
    lib.rtcuda_radiance.argtypes = [C.c_void_p, C.POINTER(Settings), C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
    lib.rtcuda_radiance.restype = C.c_int
    lib.rtcuda_radiance_device.argtypes = lib.rtcuda_radiance.argtypes
    lib.rtcuda_radiance_device.restype = C.c_int
    lib.rtcuda_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
    lib.rtcuda_get_stats.restype = C.c_int
    lib.rtcuda_last_error.argtypes = []
    lib.rtcuda_last_error.restype = C.c_char_p
    lib.rtcuda_abi_version.argtypes = []
    lib.rtcuda_abi_version.restype = C.c_uint32
    lib.rtcuda_abi_struct_sizes.argtypes = [C.POINTER(C.c_uint32), C.c_uint32]
    lib.rtcuda_abi_struct_sizes.restype = C.c_uint32
    if lib.rtcuda_abi_version() != ABI_VERSION:
        raise RtCudaError("libraytracing_cuda.so ABI version mismatch")
    sizes = (C.c_uint32 * 32)()
    n = lib.rtcuda_abi_struct_sizes(sizes, 32)
    mine = [C.sizeof(s) for s in ABI_STRUCTS]
    if list(sizes[:n]) != mine:
        raise RtCudaError(f"ABI struct size mismatch: lib {list(sizes[:n])} vs ctypes {mine}")
    if path == LIB_PATH:
        _lib = lib
    return lib


def check(lib: C.CDLL, status: int, what: str) -> None:
    if status != 0:
        msg = lib.rtcuda_last_error()
        raise RtCudaError(f"{what} failed: {STATUS_NAMES.get(status, status)}: {msg.decode() if msg else ''}")


def host_array(lib: C.CDLL, shape, dtype):
    """A numpy array over page-locked memory from rtcuda_host_alloc (None when the library has none to give). The buffer returns
    to the library's cache when the last array that views it is collected."""
    import weakref
    import numpy as np
    dt = np.dtype(dtype)
    n = int(np.prod(shape))
    nbytes = n * dt.itemsize
    ptr = lib.rtcuda_host_alloc(nbytes)
    if not ptr:
        return None
    buf = (C.c_uint8 * nbytes).from_address(ptr)
    weakref.finalize(buf, lib.rtcuda_host_free, ptr)   # numpy keeps `buf` alive as the base of every view
    return np.frombuffer(buf, dtype=dt, count=n).reshape(shape)
