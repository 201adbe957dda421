"""The backend entry points — mirror of raytracing_cpu::{render, render_single_pixel,
CpuBackendSettings} (crates/raytracing-cpu/src/lib.rs:446-457, 645-858, 860-931) for `--backend cuda`.

Every call goes through libraytracing_cuda.so (include/rtcuda.h). There is no CPU path here: when the
library is missing `_ffi.load_library()` raises.
"""
from __future__ import annotations

import ctypes as C
import sys
import time
from dataclasses import dataclass
from typing import List, Optional

import numpy as np

from . import _ffi
from .renderer import AovFlags, RaytracerSettings, RenderOutput, SinglePixelOutput
from .scene import Scene


@dataclass
class CudaBackendSettings:
    """The analogue of CpuBackendSettings{num_threads} (lib.rs:446-457)."""
    device_id: int = 0
    max_paths_in_flight: int = 0       # 0 => backend default
    tile_rank: int = 0                 # this context renders the tiles i with i % tile_world == tile_rank
    tile_world: int = 1
    tile_size: int = 0                 # 0 => 64 (the reference's RenderTile grid); a power of two in [8, 64]
    collect_stats: int = 0             # _ffi.STATS_COUNTERS | _ffi.STATS_KERNEL_TIMES (True == counters)
    watertight: bool = False           # Woop's watertight triangle test instead of the reference's Moller-Trumbore
    # Multi-GPU inside one call (the analogue of CpuBackendSettings::num_threads, lib.rs:446-457): num_devices > 1 replicates the
    # scene on `device_ids` (default 0 .. num_devices-1), deals the tiles to them and returns the complete frame; every pixel
    # is the one a single GPU renders.
    num_devices: int = 0
    device_ids: Optional[List[int]] = None

    def to_c(self) -> _ffi.BackendSettings:
        b = _ffi.BackendSettings()
        b.device_id, b.max_paths_in_flight = self.device_id, self.max_paths_in_flight
        b.tile_rank, b.tile_world, b.collect_stats = self.tile_rank, self.tile_world, int(self.collect_stats)
        b.flags = _ffi.BACKEND_WATERTIGHT if self.watertight else 0
        b.tile_size = self.tile_size
        ids = list(self.device_ids) if self.device_ids is not None else list(range(max(0, self.num_devices)))
        n = self.num_devices or (len(ids) if self.device_ids is not None else 0)
        if n > _ffi.MAX_DEVICES or n > len(ids):
            raise ValueError(f"num_devices = {n} needs that many device_ids (at most {_ffi.MAX_DEVICES})")
        b.num_devices = n
        for i in range(n):
            b.device_ids[i] = ids[i]
        return b


def make_rays(origins, directions, t_min=0.0, t_max=np.inf) -> np.ndarray:
    """Pack rays for CudaRenderer.trace / occluded: float32 [N, 8] rows of origin.xyz, t_min, direction.xyz, t_max. `origins` and
    `directions` are [N, 3] (or one [3] row, broadcast); t_min / t_max are scalars or [N]. Directions are not normalised: hit
    t is in units of the direction's length."""
    o = np.asarray(origins, dtype=np.float32)
    d = np.asarray(directions, dtype=np.float32)
    if o.shape[-1:] != (3,) or d.shape[-1:] != (3,) or o.ndim > 2 or d.ndim > 2:
        raise ValueError(f"origins and directions must be [N, 3] or [3], got {o.shape} and {d.shape}")
    n = max(o.shape[0] if o.ndim == 2 else 1, d.shape[0] if d.ndim == 2 else 1)
    rays = np.empty((n, 8), dtype=np.float32)
    try:
        rays[:, 0:3] = o
        rays[:, 4:7] = d
        rays[:, 3] = np.asarray(t_min, dtype=np.float32)
        rays[:, 7] = np.asarray(t_max, dtype=np.float32)
    except ValueError as e:
        raise ValueError(f"ray fields do not broadcast to {n} rays: {e}") from None
    return rays


@dataclass
class RayHits:
    """Closest hits of CudaRenderer.trace, one row per ray: t (+inf on a miss), the instance index (geom_id) and the primitive
    index within its shape (prim_id, 0 for a sphere) as uint32 (_ffi.NONE on a miss), and the barycentrics (u, v) = the
    weights of the triangle's v1 and v2 (0 for spheres and misses)."""
    t: np.ndarray              # float32 [N]
    instance: np.ndarray       # uint32 [N]
    primitive: np.ndarray      # uint32 [N]
    barycentrics: np.ndarray   # float32 [N, 2]


# one rtcuda_surface record (include/rtcuda.h) as a numpy structured dtype: 64 bytes, the field offsets of _ffi.Surface
SURFACE_DTYPE = np.dtype([("point", np.float32, (3,)), ("t", np.float32), ("normal", np.float32, (3,)), ("material", np.uint32),
                          ("uv", np.float32, (2,)), ("geom_id", np.uint32), ("prim_id", np.uint32), ("albedo", np.float32, (3,)),
                          ("light", np.uint32)])


@dataclass
class RaySurfaces:
    """The surface at the closest hit of every ray of CudaRenderer.surfaces, one row per ray. t / instance / primitive are those
    of CudaRenderer.trace; point is the world-space hit point; normal the unit shading normal (interpolated vertex normal, or
    the geometric one, or the sphere's), not flipped toward the ray; uv the surface's texture coordinates; material and light
    the instance's material and area light (_ffi.NONE when it emits nothing); albedo the material's albedo at uv with a zero
    texture footprint. A miss (or an invalid ray) has t = +inf, zeros, and _ffi.NONE ids / material / light. The arrays are views
    of `records`, one SURFACE_DTYPE record per ray."""
    records: np.ndarray        # SURFACE_DTYPE [N]
    t: np.ndarray              # float32 [N]
    point: np.ndarray          # float32 [N, 3]
    normal: np.ndarray         # float32 [N, 3]
    uv: np.ndarray             # float32 [N, 2]
    instance: np.ndarray       # uint32 [N]
    primitive: np.ndarray      # uint32 [N]
    material: np.ndarray       # uint32 [N]
    light: np.ndarray          # uint32 [N]
    albedo: np.ndarray         # float32 [N, 3]

    @classmethod
    def from_records(cls, rec: np.ndarray) -> "RaySurfaces":
        return cls(rec, rec["t"], rec["point"], rec["normal"], rec["uv"], rec["geom_id"], rec["prim_id"], rec["material"], rec["light"],
                   rec["albedo"])


def _check_rays(rays) -> np.ndarray:
    if not isinstance(rays, np.ndarray) or rays.dtype != np.float32 or rays.ndim != 2 or rays.shape[1] != 8:
        raise ValueError("rays must be a float32 numpy array of shape [N, 8] (see make_rays)")
    if not rays.flags.c_contiguous:
        raise ValueError("rays must be C-contiguous")
    return rays


def warn_nonfinite(beauty: np.ndarray, log=None) -> int:
    """The tail of raytracing_cpu::render (lib.rs:813-854): every channel of the beauty plane is classified, the first 10
    NaN / infinite ones are reported in raster order, then the total. The count comes from the device (k_finalize); this
    only runs when it is non-zero. Returns the number of warnings."""
    log = log or (lambda m: print("warning: " + m, file=sys.stderr))
    bad = np.argwhere(~np.isfinite(beauty))          # row-major: (j, i, channel) in the reference's loop order
    for j, i, c in bad[:10]:
        kind = "NaN" if np.isnan(beauty[j, i, c]) else "infty"
        log(f"{'RGB'[c]} component of ({i}, {j}) is {kind}")
    if len(bad):
        log(f"encountered {len(bad)} NaN and infty values in radiance buffer")
    return len(bad)


class CudaRenderer:
    """A context + an uploaded scene (device BVH, textures). `render()` may be called repeatedly;
    the one-shot `render()` function below is the reference-shaped call."""

    def __init__(self, scene: Scene, backend_settings: Optional[CudaBackendSettings] = None):
        self.lib = _ffi.load_library()
        self.backend_settings = backend_settings or CudaBackendSettings()
        self.scene = scene
        self._ctx = C.c_void_p()
        self._scene = C.c_void_p()
        bs = self.backend_settings.to_c()
        t0 = time.perf_counter()
        _ffi.check(self.lib, self.lib.rtcuda_init(C.byref(bs), C.byref(self._ctx)), "rtcuda_init")
        t1 = time.perf_counter()
        holder = scene.to_desc(own_arrays=True)   # zero-copy: the library reads every mesh from its own arrays
        t2 = time.perf_counter()
        try:
            _ffi.check(self.lib, self.lib.rtcuda_scene_upload(self._ctx, C.byref(holder.desc), C.byref(self._scene)),
                       "rtcuda_scene_upload")
        except Exception:
            self.close()
            raise
        # host wall-clock of the three setup phases (reported by bench.py's end-to-end breakdown)
        self.setup_ms = {"init": 1e3 * (t1 - t0), "scene_to_desc": 1e3 * (t2 - t1), "upload_and_build": 1e3 * (time.perf_counter() - t2)}
        self.width, self.height = scene.camera.raster_width, scene.camera.raster_height

    def close(self) -> None:
        if getattr(self, "_scene", None) is not None and self._scene:
            self.lib.rtcuda_scene_release(self._scene)
            self._scene = C.c_void_p()
        if getattr(self, "_ctx", None) is not None and self._ctx:
            self.lib.rtcuda_shutdown(self._ctx)
            self._ctx = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def update(self, scene: Scene) -> None:
        """Move the camera, the instance transforms and the lights of the uploaded scene to those of `scene`, which must have
        the uploaded scene's topology (same shapes, instances -> shapes, light kinds, materials, textures, raster size and
        camera kind; rtcuda_scene_update). The BVH is refitted (or rebuilt) on the device; no geometry is copied again, and
        the next frame equals the frame of a fresh CudaRenderer(scene)."""
        holder = scene.to_desc(own_arrays=True)   # zero-copy: the library reads no mesh array
        _ffi.check(self.lib, self.lib.rtcuda_scene_update(self._scene, C.byref(holder.desc)), "rtcuda_scene_update")
        self.scene = scene

    def render(self, settings: RaytracerSettings) -> RenderOutput:
        """raytracing_cpu::render: host planes, row-major [H,W,C]."""
        out = RenderOutput.allocate(self.width, self.height, AovFlags(settings.outputs), lib=self.lib)
        self.render_into(settings, out)
        return out

    def render_into(self, settings: RaytracerSettings, out: RenderOutput) -> None:
        s, o = settings.to_c(), out.to_c()
        _ffi.check(self.lib, self.lib.rtcuda_render(self._scene, C.byref(s), C.byref(o)), "rtcuda_render")
        if out.beauty is not None:
            st = _ffi.Stats()
            self.lib.rtcuda_get_stats(self._scene, C.byref(st))
            if st.nonfinite_values:
                warn_nonfinite(out.beauty)

    def render_device(self, settings: RaytracerSettings, planes: dict) -> None:
        """Same render with DEVICE plane pointers ({'beauty': ptr, ...}); nothing is copied to the host."""
        o = _ffi.Outputs()
        o.width, o.height = self.width, self.height
        for k, v in planes.items():
            setattr(o, k, v)
        s = settings.to_c()
        _ffi.check(self.lib, self.lib.rtcuda_render_device(self._scene, C.byref(s), C.byref(o)), "rtcuda_render_device")

    def render_samples_device(self, settings: RaytracerSettings, sample_lo: int, sample_hi: int, beauty_sum_ptr: int) -> None:
        """Samples [sample_lo, sample_hi) of this context's pixels; the un-normalised radiance sum goes to the DEVICE
        plane at `beauty_sum_ptr` (3 floats / pixel). Sample-range partition across GPUs, progressive display."""
        s = settings.to_c()
        _ffi.check(self.lib, self.lib.rtcuda_render_samples_device(self._scene, C.byref(s), sample_lo, sample_hi, beauty_sum_ptr),
                   "rtcuda_render_samples_device")

    def render_samples_accumulate_device(self, settings: RaytracerSettings, sample_lo: int, sample_hi: int, beauty_sum_ptr: int) -> None:
        """Progressive rendering: ADD the un-normalised sum of samples [sample_lo, sample_hi) to the DEVICE plane in place
        (start from zeros; `plane / sample_hi` is the image so far). See examples/progressive_viewer.py."""
        s = settings.to_c()
        _ffi.check(self.lib, self.lib.rtcuda_render_samples_accumulate_device(self._scene, C.byref(s), sample_lo, sample_hi, beauty_sum_ptr),
                   "rtcuda_render_samples_accumulate_device")

    def render_pixel(self, settings: RaytracerSettings, x: int, y: int, sample_lo: int, sample_hi: int) -> List[SinglePixelOutput]:
        n = max(0, sample_hi - sample_lo)
        buf = (_ffi.PixelOutput * max(1, n))()
        s = settings.to_c()
        _ffi.check(self.lib, self.lib.rtcuda_render_pixel(self._scene, C.byref(s), x, y, sample_lo, sample_hi, buf),
                   "rtcuda_render_pixel")
        return [SinglePixelOutput(b.sample_index, bool(b.hit), tuple(b.uv), tuple(b.normal), tuple(b.radiance)) for b in buf[:n]]

    def trace(self, rays: np.ndarray) -> RayHits:
        """Closest hit of every ray of `rays` (float32 [N, 8], make_rays) in [t_min, t_max], both inclusive, no back-face
        culling; equal-t ties go to the larger (instance, primitive). Host arrays; blocks until the results are here. Queries
        leave the render state and stats() alone."""
        rays = _check_rays(rays)
        n = rays.shape[0]
        t = np.empty(n, np.float32)
        ids = np.empty((n, 2), np.uint32)
        uv = np.empty((n, 2), np.float32)
        _ffi.check(self.lib, self.lib.rtcuda_trace_rays(self._scene, rays.ctypes.data, n, t.ctypes.data, ids.ctypes.data, uv.ctypes.data),
                   "rtcuda_trace_rays")
        return RayHits(t, ids[:, 0].copy(), ids[:, 1].copy(), uv)

    def occluded(self, rays: np.ndarray) -> np.ndarray:
        """bool [N]: whether anything is hit in [t_min, t_max] (the any-hit walk of shadow rays)."""
        rays = _check_rays(rays)
        occ = np.empty(rays.shape[0], np.uint8)
        _ffi.check(self.lib, self.lib.rtcuda_occluded(self._scene, rays.ctypes.data, rays.shape[0], occ.ctypes.data), "rtcuda_occluded")
        return occ.view(np.bool_)

    def trace_device(self, rays_ptr: int, count: int, t_ptr: Optional[int] = None, ids_ptr: Optional[int] = None,
                     barycentrics_ptr: Optional[int] = None) -> None:
        """trace() on DEVICE arrays of the context's first GPU (e.g. torch tensors' data_ptr()): rays count x 8 float32, 16-byte
        aligned; t count float32, ids count x 2 uint32 (int32 tensors work), barycentrics count x 2 float32; None skips an output.
        The library's stream does not wait for the caller's: finish writing the rays first (torch.cuda.synchronize()). Blocks
        until the outputs are written."""
        _ffi.check(self.lib, self.lib.rtcuda_trace_rays_device(self._scene, rays_ptr, count, t_ptr, ids_ptr, barycentrics_ptr),
                   "rtcuda_trace_rays_device")

    def occluded_device(self, rays_ptr: int, count: int, occluded_ptr: int) -> None:
        """occluded() on DEVICE arrays (see trace_device): one uint8 per ray, 1 = occluded."""
        _ffi.check(self.lib, self.lib.rtcuda_occluded_device(self._scene, rays_ptr, count, occluded_ptr), "rtcuda_occluded_device")

    def surfaces(self, rays: np.ndarray) -> RaySurfaces:
        """The surface at the closest hit of every ray of `rays` (float32 [N, 8], make_rays; the rule of trace()): hit point,
        shading normal, uv, material, area light and albedo (rtcuda_trace_surfaces). Host arrays; blocks until the results are
        here. Leaves the render state and stats() alone."""
        rays = _check_rays(rays)
        rec = np.empty(rays.shape[0], SURFACE_DTYPE)
        _ffi.check(self.lib, self.lib.rtcuda_trace_surfaces(self._scene, rays.ctypes.data, rays.shape[0], rec.ctypes.data),
                   "rtcuda_trace_surfaces")
        return RaySurfaces.from_records(rec)

    def surfaces_device(self, rays_ptr: int, count: int, surfaces_ptr: int) -> None:
        """surfaces() on DEVICE arrays of the context's first GPU: rays count x 8 float32 and surfaces count x 16 4-byte words
        (one rtcuda_surface each, e.g. a float32 torch tensor [N, 16] whose integer words 7, 10, 11 and 15 are read through
        .view(torch.int32)), both 16-byte aligned. Finish writing the rays first (torch.cuda.synchronize()). Blocks until
        written."""
        _ffi.check(self.lib, self.lib.rtcuda_trace_surfaces_device(self._scene, rays_ptr, count, surfaces_ptr), "rtcuda_trace_surfaces_device")

    def radiance(self, rays: np.ndarray, settings: RaytracerSettings, stream_base: int = 0) -> np.ndarray:
        """float32 [N, 3]: the path tracer's mean radiance along every ray of `rays` (float32 [N, 8], make_rays) over
        settings.samples_per_pixel samples (rtcuda_radiance). Directions need not be unit length: each ray is normalised and
        its range scaled by the direction's length. Misses return the environment radiance (or 0); invalid rays return 0.
        Sample s of ray i uses the sampler stream of pixel (k & 0xffff, k >> 16), k = stream_base + i, so slicing a ray set
        over calls with stream_base = the slice's offset reproduces one call bit for bit. Host arrays; blocks. stats() keeps
        describing the last render."""
        rays = _check_rays(rays)
        out = np.empty((rays.shape[0], 3), np.float32)
        s = settings.to_c()
        _ffi.check(self.lib, self.lib.rtcuda_radiance(self._scene, C.byref(s), rays.ctypes.data, rays.shape[0], stream_base, out.ctypes.data),
                   "rtcuda_radiance")
        return out

    def radiance_device(self, rays_ptr: int, count: int, settings: RaytracerSettings, radiance_ptr: int, stream_base: int = 0) -> None:
        """radiance() on DEVICE arrays of the context's first GPU (e.g. torch tensors' data_ptr()): rays count x 8 float32, 16-byte
        aligned; radiance count x 3 float32. Finish writing the rays first (torch.cuda.synchronize()). Blocks until written."""
        s = settings.to_c()
        _ffi.check(self.lib, self.lib.rtcuda_radiance_device(self._scene, C.byref(s), rays_ptr, count, stream_base, radiance_ptr),
                   "rtcuda_radiance_device")

    def stats(self) -> dict:
        st = _ffi.Stats()
        _ffi.check(self.lib, self.lib.rtcuda_get_stats(self._scene, C.byref(st)), "rtcuda_get_stats")
        return {name: getattr(st, name) for name, _ in _ffi.Stats._fields_}


def render(scene: Scene, raytracer_settings: RaytracerSettings,
           backend_settings: Optional[CudaBackendSettings] = None) -> RenderOutput:
    """pub fn render(&Scene, &RaytracerSettings, BackendSettings) -> RenderOutput (lib.rs:645-649)."""
    with CudaRenderer(scene, backend_settings) as r:
        return r.render(raytracer_settings)


def render_single_pixel(scene: Scene, raytracer_settings: RaytracerSettings, x: int, y: int,
                        sample_index: Optional[int] = None) -> SinglePixelOutput:
    """pub fn render_single_pixel(.., x, y, sample_index: Option<u32>) (lib.rs:860-866)."""
    i = 0 if sample_index is None else sample_index
    with CudaRenderer(scene, backend_settings=None) as r:
        return r.render_pixel(raytracer_settings, x, y, i, i + 1)[0]
