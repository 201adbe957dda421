"""raytracing-cuda: the B200-native `--backend cuda` render backend (host-side mirror of the
reference's backend interface, crates/raytracing-cpu/src/lib.rs:645-931, over the C ABI in
include/rtcuda.h). The CUDA library is the product; nothing here computes pixels on the CPU."""
from . import _ffi
from .renderer import AovFlags, RaytracerSettings, RenderOutput, Sampler, SinglePixelOutput
from .scene import (Camera, Light, Material, Mesh, Scene, SceneBuilder, Sphere, Texture, scene_from_gltf_file,
                    mesh_from_ply_bytes)
from .pbrt import scene_from_pbrt_file, scene_from_pbrt_string, PbrtParseError
from .backend import CudaBackendSettings, CudaRenderer, RayHits, make_rays, render, render_single_pixel
from . import test_scenes
from . import multi_gpu
from . import exr
from . import imagecmp

__all__ = ["AovFlags", "RaytracerSettings", "RenderOutput", "Sampler", "SinglePixelOutput", "Camera", "Light",
           "Material", "Mesh", "Scene", "SceneBuilder", "Sphere", "Texture", "scene_from_gltf_file", "scene_from_pbrt_file", "scene_from_pbrt_string", "PbrtParseError",
           "mesh_from_ply_bytes", "CudaBackendSettings", "CudaRenderer", "RayHits", "make_rays", "render", "render_single_pixel",
           "test_scenes"]
