//! # CUDA backend for the raytracer (`--backend cuda`)
//!
//! Same shape as `raytracing_cpu` (`crates/raytracing-cpu/src/lib.rs:645-649, 860-866`) and `raytracing_optix`
//! (`crates/raytracing-optix/src/lib.rs:95-99, 172-178`): two free functions over `&Scene` + `&RaytracerSettings`.
//! Everything behind them lives in `libraytracing_cuda.so` (hand-written sm_100a wavefront path tracer, device BVH
//! build); this crate flattens the scene graph into the POD arrays of `rtcuda_scene_desc` and forwards.
//!
//! The flattening rules are the ones `opencl-raytracing_b200/scene.py: SceneDescHolder` implements and the backend's test
//! suite exercises; they are restated here in Rust against the reference's own types.

use std::{ffi::CStr, ops::Range, ptr};

use raytracing::{
    geometry::{Matrix4x4, Shape, Transform, Vec2, Vec3},
    lights::Light,
    materials::{FilterMode, Material, Texture, TextureId, WrapMode},
    renderer::{AovFlags, RaytracerSettings, RenderOutput, SinglePixelOutput},
    sampling::Sampler,
    scene::{primitive::Primitive, camera::CameraType, Scene},
};
use tracing::warn;

#[allow(non_camel_case_types, non_upper_case_globals, non_snake_case, dead_code)]
mod ffi {
    include!(concat!(env!("OUT_DIR"), "/bindings.rs"));
}

/// The analogue of `CpuBackendSettings { num_threads }` (`raytracing-cpu/src/lib.rs:446-457`).
#[derive(Debug, Clone)]
pub struct CudaBackendSettings {
    /// GPUs to render on. One entry: that device. Several: the scene is replicated on all of them, image tiles are dealt
    /// round-robin, and `render` still returns the complete frame (bit-identical to one GPU).
    pub device_ids: Vec<i32>,
    /// Paths in flight per GPU (0 = sized from free HBM).
    pub max_paths_in_flight: u32,
    /// Edge of the tiles dealt to the GPUs (0 = 64, the CPU backend's `RenderTile`; a power of two in 8..=64).
    pub tile_size: u32,
    /// Woop's watertight triangle test instead of the reference's Moller-Trumbore.
    pub watertight: bool,
}

impl Default for CudaBackendSettings {
    fn default() -> Self {
        Self { device_ids: vec![0], max_paths_in_flight: 0, tile_size: 0, watertight: false }
    }
}

impl CudaBackendSettings {
    fn to_c(&self) -> ffi::rtcuda_backend_settings {
        let mut b = ffi::rtcuda_backend_settings::default();
        b.device_id = *self.device_ids.first().unwrap_or(&0);
        b.max_paths_in_flight = self.max_paths_in_flight;
        b.tile_size = self.tile_size;
        b.flags = if self.watertight { ffi::RTCUDA_BACKEND_WATERTIGHT } else { 0 };
        assert!(self.device_ids.len() <= ffi::RTCUDA_MAX_DEVICES as usize, "at most {} GPUs", ffi::RTCUDA_MAX_DEVICES);
        if self.device_ids.len() > 1 {
            b.num_devices = self.device_ids.len() as u32;
            for (slot, id) in b.device_ids.iter_mut().zip(&self.device_ids) {
                *slot = *id;
            }
        }
        b
    }
}

fn check(status: ffi::rtcuda_status, what: &str) {
    if status != ffi::rtcuda_status::RTCUDA_OK {
        // SAFETY: rtcuda_last_error returns a NUL-terminated string owned by the library (thread-local)
        let msg = unsafe { CStr::from_ptr(ffi::rtcuda_last_error()) }.to_string_lossy().into_owned();
        panic!("{what} failed ({status:?}): {msg}");
    }
}

fn mat(m: &Matrix4x4) -> ffi::rtcuda_mat4 {
    let mut out = ffi::rtcuda_mat4::default();
    for r in 0..4 {
        for c in 0..4 {
            out.m[4 * r + c] = m.data[r][c]; // row-major on both sides (matrix4x4.rs:8-13)
        }
    }
    out
}

fn transform(t: &Transform) -> ffi::rtcuda_transform {
    ffi::rtcuda_transform { forward: mat(&t.forward), inverse: mat(&t.inverse) }
}

/// `rtcuda_scene_desc` plus the Vecs its pointers refer to. Mesh arrays are NOT copied: the desc points straight at the
/// scene's `Vec<Vec3>` / `Vec<Vec3u>` / `Vec<Vec2>` (all `repr(C)`, `vec3.rs:7-9, 218-220`, `vec2.rs:8-10`).
struct FlatScene<'a> {
    desc: ffi::rtcuda_scene_desc,
    _shapes: Vec<ffi::rtcuda_shape>,
    _instances: Vec<ffi::rtcuda_instance>,
    _lights: Vec<ffi::rtcuda_light>,
    _materials: Vec<ffi::rtcuda_material>,
    _textures: Vec<ffi::rtcuda_texture>,
    _images: Vec<ffi::rtcuda_image>,
    _image_bytes: Vec<u8>,
    _scene: &'a Scene,
}

const NONE: u32 = ffi::RTCUDA_NONE;

fn tex(t: TextureId) -> u32 {
    t.0
}

fn flatten(scene: &Scene) -> FlatScene<'_> {
    // shapes[i] <- every Primitive::Basic, in `primitives` order; remember raw index -> shape index
    // (DiffuseAreaLight::prim_id and the root's children refer to raw primitive indices)
    let mut shapes = Vec::new();
    let mut shape_of_raw = std::collections::HashMap::new();
    for raw in 0..scene.primitive_count() {   // accessor added by integration/reference.patch (`primitives` is private)
        let idx = scene.primitive_index_from_usize(raw);
        if let Primitive::Basic(basic) = scene.get_primitive(idx) {
            let mut s = ffi::rtcuda_shape::default();
            s.material = basic.material;
            s.area_light = basic.area_light.unwrap_or(NONE);
            s.normal_offset = NONE;
            s.uv_offset = NONE;
            match &basic.shape {
                Shape::TriangleMesh(mesh) => {
                    s.kind = ffi::rtcuda_shape_kind_RTCUDA_SHAPE_TRIANGLE_MESH;
                    s.vertex_count = mesh.vertices.len() as u32;
                    s.tri_count = mesh.tris.len() as u32;
                    s.vertices = mesh.vertices.as_ptr() as *const f32;
                    s.tris = mesh.tris.as_ptr() as *const u32;
                    s.normals = if mesh.normals.is_empty() { ptr::null() } else { mesh.normals.as_ptr() as *const f32 };
                    s.uvs = if mesh.uvs.is_empty() { ptr::null() } else { mesh.uvs.as_ptr() as *const f32 };
                }
                Shape::Sphere { center, radius } => {
                    s.kind = ffi::rtcuda_shape_kind_RTCUDA_SHAPE_SPHERE;
                    s.center = [center.0, center.1, center.2];
                    s.radius = *radius;
                }
            }
            shape_of_raw.insert(raw, shapes.len() as u32);
            shapes.push(s);
        }
    }

    // instances[g] <- child g of the root aggregate after get_descendant flattening (scene.rs:201-224); g is the geom_id
    // the CPU backend stores in PrimPtr (bvh2.rs:278-283)
    let root = scene.root_index();
    let mut instances = Vec::new();
    for g in 0..scene.get_aggregate_primitive(root).children.len() {
        let (leaf, t) = scene.get_descendant(root, g);
        let leaf_raw: usize = leaf.into();
        let shape = *shape_of_raw
            .get(&leaf_raw)
            .expect("nested aggregates are not supported by the cuda backend (no importer creates them)");
        let mut inst = ffi::rtcuda_instance::default();
        inst.shape = shape;
        inst.object_to_world = transform(&t);
        instances.push(inst);
    }

    let lights = scene
        .lights
        .iter()
        .map(|l| {
            let mut c = ffi::rtcuda_light::default();
            match l {
                Light::PointLight { position, intensity } => {
                    c.kind = ffi::rtcuda_light_kind_RTCUDA_LIGHT_POINT;
                    c.position_or_direction = [position.0, position.1, position.2];
                    c.intensity_or_radiance = [intensity.0, intensity.1, intensity.2];
                }
                Light::DirectionLight { direction, radiance } => {
                    c.kind = ffi::rtcuda_light_kind_RTCUDA_LIGHT_DIRECTION;
                    c.position_or_direction = [direction.0, direction.1, direction.2];
                    c.intensity_or_radiance = [radiance.0, radiance.1, radiance.2];
                }
                Light::DiffuseAreaLight { prim_id, radiance, light_to_world } => {
                    c.kind = ffi::rtcuda_light_kind_RTCUDA_LIGHT_DIFFUSE_AREA;
                    c.shape = shape_of_raw[&(prim_id.0 as usize)];
                    c.intensity_or_radiance = [radiance.0, radiance.1, radiance.2];
                    c.light_to_world = mat(light_to_world);
                }
            }
            c
        })
        .collect::<Vec<_>>();

    let materials = scene
        .materials
        .iter()
        .map(|m| {
            let mut c = ffi::rtcuda_material {
                kind: 0, remap_roughness: 0, albedo: NONE, eta: NONE, kappa: NONE, roughness: NONE, thickness: NONE, coat_albedo: NONE,
            };
            match m {
                Material::Diffuse { albedo } => {
                    c.kind = ffi::rtcuda_material_kind_RTCUDA_MATERIAL_DIFFUSE;
                    c.albedo = tex(*albedo);
                }
                Material::SmoothDielectric { eta } => {
                    c.kind = ffi::rtcuda_material_kind_RTCUDA_MATERIAL_SMOOTH_DIELECTRIC;
                    c.eta = tex(*eta);
                }
                Material::SmoothConductor { eta, kappa } => {
                    c.kind = ffi::rtcuda_material_kind_RTCUDA_MATERIAL_SMOOTH_CONDUCTOR;
                    c.eta = tex(*eta);
                    c.kappa = tex(*kappa);
                }
                Material::RoughDielectric { eta, remap_roughness, roughness } => {
                    c.kind = ffi::rtcuda_material_kind_RTCUDA_MATERIAL_ROUGH_DIELECTRIC;
                    c.eta = tex(*eta);
                    c.remap_roughness = *remap_roughness as u32;
                    c.roughness = tex(*roughness);
                }
                Material::RoughConductor { eta, kappa, remap_roughness, roughness } => {
                    c.kind = ffi::rtcuda_material_kind_RTCUDA_MATERIAL_ROUGH_CONDUCTOR;
                    c.eta = tex(*eta);
                    c.kappa = tex(*kappa);
                    c.remap_roughness = *remap_roughness as u32;
                    c.roughness = tex(*roughness);
                }
                Material::CoatedDiffuse { diffuse_albedo, dielectric_eta, dielectric_remap_roughness, dielectric_roughness, thickness, coat_albedo } => {
                    c.kind = ffi::rtcuda_material_kind_RTCUDA_MATERIAL_COATED_DIFFUSE;
                    c.albedo = tex(*diffuse_albedo);
                    c.eta = tex(*dielectric_eta);
                    c.remap_roughness = *dielectric_remap_roughness as u32;
                    c.roughness = dielectric_roughness.map(tex).unwrap_or(NONE);
                    c.thickness = tex(*thickness);
                    c.coat_albedo = tex(*coat_albedo);
                }
            }
            c
        })
        .collect::<Vec<_>>();

    let textures = scene
        .textures
        .iter()
        .map(|t| {
            let mut c = ffi::rtcuda_texture::default();
            c.a = NONE;
            c.b = NONE;
            c.c = NONE;
            match t {
                Texture::ImageTexture { image, sampler } => {
                    c.kind = ffi::rtcuda_texture_kind_RTCUDA_TEXTURE_IMAGE;
                    c.image = image.0;
                    c.filter = match sampler.filter { FilterMode::Nearest => 0, FilterMode::Bilinear => 1, FilterMode::Trilinear => 2 };
                    c.wrap = match sampler.wrap { WrapMode::Repeat => 0, WrapMode::Mirror => 1, WrapMode::Clamp => 2 };
                }
                Texture::ConstantTexture { value } => {
                    c.kind = ffi::rtcuda_texture_kind_RTCUDA_TEXTURE_CONSTANT;
                    c.value = [value.0, value.1, value.2, value.3];
                }
                Texture::CheckerTexture { color1, color2 } => {
                    c.kind = ffi::rtcuda_texture_kind_RTCUDA_TEXTURE_CHECKER;
                    c.value = [color1.0, color1.1, color1.2, color1.3];
                    c.value2 = [color2.0, color2.1, color2.2, color2.3];
                }
                Texture::ScaleTexture { a, b } => {
                    c.kind = ffi::rtcuda_texture_kind_RTCUDA_TEXTURE_SCALE;
                    c.a = a.0;
                    c.b = b.0;
                }
                Texture::MixTexture { a, b, c: amount } => {
                    c.kind = ffi::rtcuda_texture_kind_RTCUDA_TEXTURE_MIX;
                    c.a = a.0;
                    c.b = b.0;
                    c.c = amount.0;
                }
            }
            c
        })
        .collect::<Vec<_>>();

    // images stay in their source encoding (image.rs:56-121: a channel reads as sub / MAX); bytes concatenated, 16-byte aligned
    let mut image_bytes = Vec::new();
    let images = scene
        .images
        .iter()
        .map(|im| {
            use image::ColorType::*;
            let format = match im.buffer.color() {
                L8 | La8 | Rgb8 | Rgba8 => ffi::rtcuda_image_format_RTCUDA_IMAGE_U8,
                L16 | La16 | Rgb16 | Rgba16 => ffi::rtcuda_image_format_RTCUDA_IMAGE_U16,
                Rgb32F | Rgba32F => ffi::rtcuda_image_format_RTCUDA_IMAGE_F32,
                other => unimplemented!("unsupported dynamic image format {other:?}"),
            };
            while image_bytes.len() % 16 != 0 {
                image_bytes.push(0u8);
            }
            let byte_offset = image_bytes.len() as u64;
            image_bytes.extend_from_slice(im.buffer.as_bytes());
            ffi::rtcuda_image { width: im.width(), height: im.height(), channels: im.depth(), format, byte_offset }
        })
        .collect::<Vec<_>>();

    let cam = &scene.camera;
    let mut camera = ffi::rtcuda_camera::default();
    camera.raster_width = cam.raster_width as u32;
    camera.raster_height = cam.raster_height as u32;
    camera.near_clip = cam.near_clip;
    camera.far_clip = cam.far_clip;
    match cam.camera_type {
        CameraType::Orthographic { screen_space_width, screen_space_height } => {
            camera.kind = ffi::rtcuda_camera_kind_RTCUDA_CAMERA_ORTHOGRAPHIC;
            camera.screen_space_width = screen_space_width;
            camera.screen_space_height = screen_space_height;
        }
        CameraType::PinholePerspective { yfov } => {
            camera.kind = ffi::rtcuda_camera_kind_RTCUDA_CAMERA_PINHOLE;
            camera.yfov = yfov;
        }
        CameraType::ThinLensPerspective { yfov, aperture_radius, focal_distance } => {
            camera.kind = ffi::rtcuda_camera_kind_RTCUDA_CAMERA_THIN_LENS;
            camera.yfov = yfov;
            camera.aperture_radius = aperture_radius;
            camera.focal_distance = focal_distance;
        }
    }
    // the three transforms verbatim: the backend never recomputes them (camera.rs:60-203 owns their conventions)
    camera.world_to_raster = transform(&cam.world_to_raster);
    camera.camera_to_world = transform(&cam.camera_to_world);
    camera.raster_to_camera = transform(&cam.raster_to_camera);

    let mut desc = ffi::rtcuda_scene_desc::default();
    desc.abi_version = ffi::RTCUDA_ABI_VERSION;
    desc.camera = camera;
    desc.shapes = shapes.as_ptr();
    desc.shape_count = shapes.len() as u32;
    desc.instances = instances.as_ptr();
    desc.instance_count = instances.len() as u32;
    desc.lights = lights.as_ptr();
    desc.light_count = lights.len() as u32;
    desc.materials = materials.as_ptr();
    desc.material_count = materials.len() as u32;
    desc.textures = textures.as_ptr();
    desc.texture_count = textures.len() as u32;
    desc.images = images.as_ptr();
    desc.image_count = images.len() as u32;
    desc.environment_light_texture = scene.environment_light.as_ref().map(|e| e.radiance.0).unwrap_or(NONE);
    desc.image_bytes = image_bytes.as_ptr();
    desc.image_byte_count = image_bytes.len() as u64;
    // vertices / tris / normals / uvs stay NULL: every mesh carries its own arrays (rtcuda_shape, ABI v2)

    FlatScene { desc, _shapes: shapes, _instances: instances, _lights: lights, _materials: materials, _textures: textures, _images: images,
                _image_bytes: image_bytes, _scene: scene }
}

fn settings_to_c(s: &RaytracerSettings) -> ffi::rtcuda_settings {
    let mut c = ffi::rtcuda_settings::default();
    c.max_ray_depth = s.max_ray_depth;
    c.accumulate_bounces = s.accumulate_bounces as u32;
    c.light_sample_count = s.light_sample_count;
    c.samples_per_pixel = s.samples_per_pixel;
    c.has_seed = s.seed.is_some() as u32;
    c.seed = s.seed.unwrap_or(0);
    match s.sampler {
        Sampler::Independent => c.sampler_kind = 0,
        Sampler::Stratified { jitter, x_strata, y_strata } => {
            c.sampler_kind = 1;
            c.stratified_jitter = jitter as u32;
            c.x_strata = x_strata;
            c.y_strata = y_strata;
        }
    }
    c.outputs = s.outputs.bits(); // same bit values (renderer/mod.rs:13-47)
    c.antialias_primary_rays = s.antialias_primary_rays as u32;
    c.antialias_secondary_rays = s.antialias_secondary_rays as u32;
    c
}

/// A scene uploaded to the device (context + device BVH) that can be rendered repeatedly and moved in place with
/// [`CudaScene::update`]: what a viewer keeps between frames.
pub struct CudaScene {
    ctx: *mut ffi::rtcuda_ctx,
    scene: *mut ffi::rtcuda_scene,
    width: usize,
    height: usize,
}

impl CudaScene {
    pub fn new(scene: &Scene, backend_settings: &CudaBackendSettings) -> Self {
        let flat = flatten(scene);
        let mut ctx = ptr::null_mut();
        let mut sc = ptr::null_mut();
        // SAFETY: the desc points into `flat`, which outlives the call; the library copies everything before it returns
        unsafe {
            check(ffi::rtcuda_init(&backend_settings.to_c(), &mut ctx), "rtcuda_init");
            let st = ffi::rtcuda_scene_upload(ctx, &flat.desc, &mut sc);
            if st != ffi::rtcuda_status::RTCUDA_OK {
                let msg = CStr::from_ptr(ffi::rtcuda_last_error()).to_string_lossy().into_owned();
                ffi::rtcuda_shutdown(ctx);
                panic!("rtcuda_scene_upload failed ({st:?}): {msg}");
            }
        }
        CudaScene { ctx, scene: sc, width: scene.camera.raster_width, height: scene.camera.raster_height }
    }

    /// Moves the camera, the instance transforms and the lights to those of `scene` (`rtcuda_scene_update`): the BVH is
    /// refitted (or rebuilt) on the device and no geometry is copied again. `scene` must have the uploaded scene's topology
    /// (same shapes, instance -> shape map, light kinds, materials, textures, raster size and camera kind); otherwise
    /// RTCUDA_ERR_INVALID_ARGUMENT is returned and the uploaded scene is left as it was.
    pub fn update(&mut self, scene: &Scene) -> Result<(), String> {
        let flat = flatten(scene);   // no mesh data is copied: the shapes point at the scene's own Vecs
        // SAFETY: the desc points into `flat`, which outlives the call; the call blocks until the device scene is updated
        unsafe {
            let st = ffi::rtcuda_scene_update(self.scene, &flat.desc);
            if st != ffi::rtcuda_status::RTCUDA_OK {
                return Err(CStr::from_ptr(ffi::rtcuda_last_error()).to_string_lossy().into_owned());
            }
        }
        Ok(())
    }

    /// The frame `render` returns, from the uploaded (and possibly updated) scene
    pub fn render(&self, raytracer_settings: &RaytracerSettings) -> RenderOutput {
        let (w, h) = (self.width, self.height);
        let n = w * h;
        let o = raytracer_settings.outputs;
        let mut out = RenderOutput::new(w as u32, h as u32);
        // only the requested planes are Some (lib.rs:664-677, 685-811)
        if o.contains(AovFlags::BEAUTY) { out.beauty = Some(vec![Vec3::zero(); n]); }
        if o.contains(AovFlags::NORMALS) { out.normals = Some(vec![Vec3::zero(); n]); }
        if o.contains(AovFlags::ALBEDO) { out.albedo = Some(vec![Vec3::zero(); n]); }
        if o.contains(AovFlags::UV_COORDS) { out.uv = Some(vec![Vec2::zero(); n]); }
        if o.contains(AovFlags::MIP_LEVEL) { out.mip_level = Some(vec![0.0f32; n]); }

        fn plane<T>(p: &mut Option<Vec<T>>) -> *mut f32 {
            p.as_mut().map(|v| v.as_mut_ptr() as *mut f32).unwrap_or(ptr::null_mut())
        }
        let mut planes = ffi::rtcuda_outputs {
            width: w as u32,
            height: h as u32,
            beauty: plane(&mut out.beauty),   // Vec<Vec3> is 3 packed f32 per pixel (vec3.rs:7-9), row-major y*W+x
            normals: plane(&mut out.normals),
            albedo: plane(&mut out.albedo),
            uv: plane(&mut out.uv),
            mip_level: plane(&mut out.mip_level),
            debug_ids: ptr::null_mut(),
            debug_depth: ptr::null_mut(),
        };
        // SAFETY: the planes are alive and sized w*h; the call blocks until they are written
        unsafe {
            check(ffi::rtcuda_render(self.scene, &settings_to_c(raytracer_settings), &mut planes), "rtcuda_render");
            // tail of raytracing_cpu::render (lib.rs:813-854): the device counted the NaN / Inf channels while writing the plane
            let mut st = ffi::rtcuda_stats::default();
            ffi::rtcuda_get_stats(self.scene, &mut st);
            if st.nonfinite_values != 0 {
                warn_nonfinite(out.beauty.as_ref().unwrap(), w, h);
            }
        }
        out
    }
}

/// Closest hit of one query ray (`rtcuda_trace_rays`): `t` is +inf and both ids `RTCUDA_NONE` on a miss; `barycentrics` are
/// the weights of the triangle's v1 and v2 (0 for spheres and misses).
#[derive(Clone, Copy, Debug, PartialEq)]
pub struct RayHit {
    pub t: f32,
    pub geom_id: u32,
    pub prim_id: u32,
    pub barycentrics: [f32; 2],
}

impl CudaScene {
    /// Closest hit of every ray in [t_min, t_max] (`[origin.xyz, t_min, direction.xyz, t_max]`): both bounds inclusive, no
    /// back-face culling, equal-t ties to the larger (geom_id, prim_id). The direction is not normalised (t is in its units).
    pub fn trace_rays(&self, rays: &[[f32; 8]]) -> Vec<RayHit> {
        let n = rays.len();
        let mut t = vec![0.0f32; n];
        let mut ids = vec![0u32; 2 * n];
        let mut uv = vec![0.0f32; 2 * n];
        // SAFETY: [f32; 8] is 8 packed floats; the outputs are sized for n rays; the call blocks until they are written
        unsafe {
            check(ffi::rtcuda_trace_rays(self.scene, rays.as_ptr() as *const f32, n as u64, t.as_mut_ptr(), ids.as_mut_ptr(), uv.as_mut_ptr()),
                  "rtcuda_trace_rays");
        }
        (0..n).map(|i| RayHit { t: t[i], geom_id: ids[2 * i], prim_id: ids[2 * i + 1], barycentrics: [uv[2 * i], uv[2 * i + 1]] }).collect()
    }

    /// Whether anything is hit in [t_min, t_max] along each ray (`rtcuda_occluded`, the any-hit walk of shadow rays).
    pub fn occluded(&self, rays: &[[f32; 8]]) -> Vec<bool> {
        let mut occ = vec![0u8; rays.len()];
        // SAFETY: as in trace_rays
        unsafe {
            check(ffi::rtcuda_occluded(self.scene, rays.as_ptr() as *const f32, rays.len() as u64, occ.as_mut_ptr()), "rtcuda_occluded");
        }
        occ.into_iter().map(|o| o != 0).collect()
    }

    /// The path tracer's mean radiance along every ray (`rtcuda_radiance`) over `settings.samples_per_pixel` samples. Directions
    /// need not be unit length (the library normalises them and scales [t_min, t_max]); misses return the environment radiance
    /// or 0, invalid rays 0. Sample s of ray i uses the sampler stream of pixel (k & 0xffff, k >> 16), k = stream_base + i.
    pub fn radiance(&self, rays: &[[f32; 8]], settings: &RaytracerSettings, stream_base: u32) -> Vec<[f32; 3]> {
        let mut out = vec![[0.0f32; 3]; rays.len()];
        // SAFETY: [f32; 8] / [f32; 3] are packed floats; the output is sized for every ray; the call blocks until it is written
        unsafe {
            check(ffi::rtcuda_radiance(self.scene, &settings_to_c(settings), rays.as_ptr() as *const f32, rays.len() as u64, stream_base,
                                       out.as_mut_ptr() as *mut f32),
                  "rtcuda_radiance");
        }
        out
    }
}

impl Drop for CudaScene {
    fn drop(&mut self) {
        // SAFETY: handles created by rtcuda_init / rtcuda_scene_upload, released exactly once
        unsafe {
            ffi::rtcuda_scene_release(self.scene);
            ffi::rtcuda_shutdown(self.ctx);
        }
    }
}

/// `pub fn render(&Scene, &RaytracerSettings, BackendSettings) -> RenderOutput` (`raytracing-cpu/src/lib.rs:645-649`)
pub fn render(scene: &Scene, raytracer_settings: &RaytracerSettings, backend_settings: CudaBackendSettings) -> RenderOutput {
    CudaScene::new(scene, &backend_settings).render(raytracer_settings)
}

fn warn_nonfinite(beauty: &[Vec3], w: usize, h: usize) {
    let mut count = 0usize;
    for j in 0..h {
        for i in 0..w {
            let Vec3(r, g, b) = beauty[j * w + i];
            for (name, v) in [("R", r), ("G", g), ("B", b)] {
                if v.is_nan() || v.is_infinite() {
                    if count < 10 {
                        warn!("{name} component of ({i}, {j}) is {}", if v.is_nan() { "NaN" } else { "infty" });
                    }
                    count += 1;
                }
            }
        }
    }
    if count > 0 {
        warn!("encountered {count} NaN and infty values in radiance buffer");
    }
}

/// `render_single_pixel` in the `Range<u32>` shape of `raytracing_optix::render_single_pixel`
/// (`raytracing-optix/src/lib.rs:172-178`); `raytracing_cpu`'s `Option<u32>` form is `index..index + 1`.
pub fn render_single_pixel(scene: &Scene, raytracer_settings: &RaytracerSettings, x: u32, y: u32, samples: Range<u32>) -> Vec<SinglePixelOutput> {
    let up = CudaScene::new(scene, &CudaBackendSettings::default());
    let n = samples.end.saturating_sub(samples.start) as usize;
    let mut buf = vec![ffi::rtcuda_pixel_output::default(); n.max(1)];
    // SAFETY: buf holds `n` entries
    unsafe {
        check(
            ffi::rtcuda_render_pixel(up.scene, &settings_to_c(raytracer_settings), x, y, samples.start, samples.end, buf.as_mut_ptr()),
            "rtcuda_render_pixel",
        );
    }
    buf.truncate(n);
    buf.into_iter()
        .map(|p| SinglePixelOutput {
            sample_index: p.sample_index,
            hit: p.hit != 0,
            uv: Vec2(p.uv[0], p.uv[1]),
            normal: Vec3(p.normal[0], p.normal[1], p.normal[2]),
            radiance: Vec3(p.radiance[0], p.radiance[1], p.radiance[2]),
        })
        .collect()
}
