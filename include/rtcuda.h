/*
 * rtcuda.h — C ABI of libraytracing_cuda.so, the B200-native (`--backend cuda`) render backend.
 *
 * This header is the drop-in boundary for the render hot path of buggy213/opencl-raytracing.
 * It is what a `raytracing-cuda` crate would run bindgen over (the way
 * crates/raytracing-optix/build.rs:3-55 runs it over csrc/host/lib_api.h), and it replaces the
 * pair of free functions every backend crate exposes to crates/cli:
 *
 *   raytracing_cpu::render              crates/raytracing-cpu/src/lib.rs:645-858
 *   raytracing_cpu::render_single_pixel crates/raytracing-cpu/src/lib.rs:860-931
 *
 * Conventions (following the OptiX precedent csrc/host/lib_api.h:16-105, with status codes
 * instead of exit()):
 *   - plain C, `extern "C"`, POD structs, pointers + counts; no torch / C++ types;
 *   - all input arrays are HOST memory, copied during rtcuda_scene_upload (caller may free after);
 *   - output planes are caller-allocated HOST memory, row-major idx = y*W + x
 *     (crates/raytracing/src/renderer/mod.rs:49-59), written only when the AOV bit is set;
 *   - opaque handles are created by *_init / *_upload and destroyed by *_release / *_shutdown;
 *   - one caller thread per context; calls block until the result is on the host.
 *
 * Every struct mirrors a type of the backend-independent scene crate (crates/raytracing); the
 * mirrored type is cited on each struct. Matrices are row-major 4x4 f32 exactly like
 * crates/raytracing/src/geometry/matrix4x4.rs:8-13.
 */
#ifndef RTCUDA_H
#define RTCUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define RTCUDA_API __declspec(dllexport)
#else
#define RTCUDA_API __attribute__((visibility("default")))
#endif

#define RTCUDA_ABI_VERSION 4u
#define RTCUDA_MAX_DEVICES 8u
#define RTCUDA_NONE 0xffffffffu

typedef enum rtcuda_status {
    RTCUDA_OK = 0,
    RTCUDA_ERR_INVALID_ARGUMENT = 1,
    RTCUDA_ERR_CUDA = 2,
    RTCUDA_ERR_UNSUPPORTED = 3,
    RTCUDA_ERR_NO_DEVICE = 4,
    RTCUDA_ERR_OUT_OF_MEMORY = 5
} rtcuda_status;

/* crates/raytracing/src/geometry/matrix4x4.rs:8-13 (row-major) */
typedef struct rtcuda_mat4 { float m[16]; } rtcuda_mat4;
/* crates/raytracing/src/geometry/transform.rs:3-8 */
typedef struct rtcuda_transform { rtcuda_mat4 forward; rtcuda_mat4 inverse; } rtcuda_transform;

/* crates/raytracing/src/scene/camera.rs:5-36. The three transforms are uploaded verbatim
 * (never recomputed by the backend, SURVEY §8a "Camera" row). */
typedef enum rtcuda_camera_kind {
    RTCUDA_CAMERA_ORTHOGRAPHIC = 0,
    RTCUDA_CAMERA_PINHOLE = 1,
    RTCUDA_CAMERA_THIN_LENS = 2
} rtcuda_camera_kind;

typedef struct rtcuda_camera {
    uint32_t kind;               /* rtcuda_camera_kind */
    uint32_t raster_width;
    uint32_t raster_height;
    float near_clip;
    float far_clip;
    float yfov;                  /* pinhole / thin lens */
    float aperture_radius;       /* thin lens */
    float focal_distance;        /* thin lens */
    float screen_space_width;    /* orthographic */
    float screen_space_height;   /* orthographic */
    rtcuda_transform world_to_raster;
    rtcuda_transform camera_to_world;
    rtcuda_transform raster_to_camera;
} rtcuda_camera;

/* crates/raytracing/src/geometry/shapes/mod.rs:5-9 + scene/primitive.rs:127-132 (BasicPrimitive).
 * Mesh attributes live in the scene-wide concatenated arrays; *_offset index those arrays in
 * elements (vertices: 3 floats, tris: 3 u32, normals: 3 floats, uvs: 2 floats). A mesh without
 * normals / uvs sets the offset to RTCUDA_NONE (Mesh::normals/uvs empty, mesh.rs:71-76). */
typedef enum rtcuda_shape_kind { RTCUDA_SHAPE_TRIANGLE_MESH = 0, RTCUDA_SHAPE_SPHERE = 1 } rtcuda_shape_kind;

typedef struct rtcuda_shape {
    uint32_t kind;               /* rtcuda_shape_kind */
    uint32_t material;           /* index into materials */
    uint32_t area_light;         /* index into lights or RTCUDA_NONE */
    uint32_t vertex_offset, vertex_count;
    uint32_t tri_offset, tri_count;
    uint32_t normal_offset;      /* RTCUDA_NONE when the mesh has no normals */
    uint32_t uv_offset;          /* RTCUDA_NONE when the mesh has no uvs */
    float center[3];             /* sphere, object space */
    float radius;                /* sphere */
    /* Optional per-shape host arrays (ABI v2): when `vertices` is non-NULL this mesh is read from these pointers
     * (vertex_count x 3 floats, tri_count x 3 indices, normals / uvs per vertex or NULL) instead of the scene-wide
     * arrays, and the four offsets above are ignored (the library assigns them). A binding can then point straight at
     * the caller's `Mesh { vertices, tris, normals, uvs }` Vecs (repr(C), geometry/shapes/mesh.rs:71-76) without
     * concatenating them: for the 16.8 M-triangle mesh that copy was 95 ms of a 445 ms end-to-end frame. Either every
     * mesh of a scene uses its own pointers or none does. */
    const float* vertices;
    const uint32_t* tris;
    const float* normals;
    const float* uvs;
} rtcuda_shape;

/* One child of the root AggregatePrimitive after Scene::get_descendant flattening
 * (crates/raytracing/src/scene/scene.rs:201-224): a BasicPrimitive plus the composed
 * object->aggregate Transform. The index of an instance in this array is the `geom_id`
 * the CPU backend stores in PrimPtr (crates/raytracing/src/accel/bvh2.rs:278-283). */
typedef struct rtcuda_instance {
    uint32_t shape;              /* index into shapes */
    uint32_t _pad[3];
    rtcuda_transform object_to_world;
} rtcuda_instance;

/* crates/raytracing/src/lights/light.rs:7-28 */
typedef enum rtcuda_light_kind {
    RTCUDA_LIGHT_POINT = 0,
    RTCUDA_LIGHT_DIRECTION = 1,
    RTCUDA_LIGHT_DIFFUSE_AREA = 2
} rtcuda_light_kind;

typedef struct rtcuda_light {
    uint32_t kind;               /* rtcuda_light_kind */
    uint32_t shape;              /* DiffuseAreaLight::prim_id -> index into shapes */
    float position_or_direction[3];
    float intensity_or_radiance[3];
    rtcuda_mat4 light_to_world;  /* DiffuseAreaLight only */
} rtcuda_light;

/* crates/raytracing/src/materials/mod.rs:2-56 */
typedef enum rtcuda_material_kind {
    RTCUDA_MATERIAL_DIFFUSE = 0,
    RTCUDA_MATERIAL_SMOOTH_DIELECTRIC = 1,
    RTCUDA_MATERIAL_SMOOTH_CONDUCTOR = 2,
    RTCUDA_MATERIAL_ROUGH_DIELECTRIC = 3,
    RTCUDA_MATERIAL_ROUGH_CONDUCTOR = 4,
    RTCUDA_MATERIAL_COATED_DIFFUSE = 5
} rtcuda_material_kind;

typedef struct rtcuda_material {
    uint32_t kind;               /* rtcuda_material_kind */
    uint32_t remap_roughness;    /* bool */
    /* texture ids; unused slots RTCUDA_NONE.
     * Diffuse:          albedo
     * SmoothDielectric: eta
     * SmoothConductor:  eta, kappa
     * RoughDielectric:  eta, roughness
     * RoughConductor:   eta, kappa, roughness
     * CoatedDiffuse:    albedo=diffuse_albedo, eta=dielectric_eta, roughness=dielectric_roughness
     *                   (RTCUDA_NONE = Option::None), thickness, coat_albedo */
    uint32_t albedo;
    uint32_t eta;
    uint32_t kappa;
    uint32_t roughness;
    uint32_t thickness;
    uint32_t coat_albedo;
} rtcuda_material;

/* crates/raytracing/src/materials/texture.rs:9-112 */
typedef enum rtcuda_texture_kind {
    RTCUDA_TEXTURE_IMAGE = 0,
    RTCUDA_TEXTURE_CONSTANT = 1,
    RTCUDA_TEXTURE_CHECKER = 2,
    RTCUDA_TEXTURE_SCALE = 3,
    RTCUDA_TEXTURE_MIX = 4
} rtcuda_texture_kind;
typedef enum rtcuda_filter_mode { RTCUDA_FILTER_NEAREST = 0, RTCUDA_FILTER_BILINEAR = 1, RTCUDA_FILTER_TRILINEAR = 2 } rtcuda_filter_mode;
typedef enum rtcuda_wrap_mode { RTCUDA_WRAP_REPEAT = 0, RTCUDA_WRAP_MIRROR = 1, RTCUDA_WRAP_CLAMP = 2 } rtcuda_wrap_mode;

typedef struct rtcuda_texture {
    uint32_t kind;               /* rtcuda_texture_kind */
    uint32_t image;              /* IMAGE: index into images */
    uint32_t filter;             /* IMAGE: rtcuda_filter_mode */
    uint32_t wrap;               /* IMAGE: rtcuda_wrap_mode */
    uint32_t a, b, c;            /* SCALE: a,b  MIX: a,b,c (texture ids) */
    uint32_t _pad;
    float value[4];              /* CONSTANT: value; CHECKER: color1 */
    float value2[4];             /* CHECKER: color2 */
} rtcuda_texture;

/* crates/raytracing/src/materials/image.rs:21-121: images stay in their source encoding;
 * a texel channel reads as sub/MAX (u8: /255, u16: /65535, f32: /1.0), missing channels 0. */
typedef enum rtcuda_image_format { RTCUDA_IMAGE_U8 = 0, RTCUDA_IMAGE_U16 = 1, RTCUDA_IMAGE_F32 = 2 } rtcuda_image_format;

typedef struct rtcuda_image {
    uint32_t width, height;
    uint32_t channels;           /* 1..4 */
    uint32_t format;             /* rtcuda_image_format */
    uint64_t byte_offset;        /* into image_bytes; row-major, interleaved channels, tightly packed */
} rtcuda_image;

/* Flat, pointer-to-array mirror of crates/raytracing/src/scene/scene.rs:13-27 (`Scene`). */
typedef struct rtcuda_scene_desc {
    uint32_t abi_version;        /* RTCUDA_ABI_VERSION */
    uint32_t _pad;
    rtcuda_camera camera;

    const rtcuda_shape* shapes;       uint32_t shape_count;
    const rtcuda_instance* instances; uint32_t instance_count;
    const rtcuda_light* lights;       uint32_t light_count;
    const rtcuda_material* materials; uint32_t material_count;
    const rtcuda_texture* textures;   uint32_t texture_count;
    const rtcuda_image* images;       uint32_t image_count;

    uint32_t environment_light_texture; /* EnvironmentLight::radiance or RTCUDA_NONE (light.rs:100-109) */
    uint32_t _pad2;

    const float* vertices;    uint64_t vertex_count;   /* 3 floats each */
    const uint32_t* tris;     uint64_t tri_count;      /* 3 u32 each, mesh-local vertex indices */
    const float* normals;     uint64_t normal_count;   /* 3 floats each */
    const float* uvs;         uint64_t uv_count;       /* 2 floats each */
    const uint8_t* image_bytes; uint64_t image_byte_count;
} rtcuda_scene_desc;

/* crates/raytracing/src/renderer/mod.rs:13-47 */
enum {
    RTCUDA_AOV_BEAUTY = 1u << 0,
    RTCUDA_AOV_NORMALS = 1u << 1,
    RTCUDA_AOV_ALBEDO = 1u << 2,
    RTCUDA_AOV_UV_COORDS = 1u << 3,
    RTCUDA_AOV_MIP_LEVEL = 1u << 4,
    RTCUDA_AOV_FIRST_HIT = (1u << 1) | (1u << 2) | (1u << 3) | (1u << 4),
    /* Debug planes that do not exist in the reference (SURVEY §8b "Outputs"): the closest-hit
     * record of the un-jittered primary ray, used for the primary-hit agreement gate. */
    RTCUDA_AOV_DEBUG_IDS = 1u << 16,   /* geom_id, prim_id (u32 each, RTCUDA_NONE on miss) */
    RTCUDA_AOV_DEBUG_DEPTH = 1u << 17  /* hit t (f32, 0 on miss) */
};

/* crates/raytracing/src/sampling/mod.rs:2-10 */
typedef enum rtcuda_sampler_kind { RTCUDA_SAMPLER_INDEPENDENT = 0, RTCUDA_SAMPLER_STRATIFIED = 1 } rtcuda_sampler_kind;

/* crates/raytracing/src/renderer/mod.rs:84-117 (`RaytracerSettings`) */
typedef struct rtcuda_settings {
    uint32_t max_ray_depth;
    uint32_t accumulate_bounces;      /* bool */
    uint32_t light_sample_count;
    uint32_t samples_per_pixel;
    uint32_t has_seed;                /* Option<u64>: 0 => None => 42 (sample.rs:30) */
    uint32_t sampler_kind;            /* rtcuda_sampler_kind */
    uint64_t seed;
    uint32_t stratified_jitter;       /* bool */
    uint32_t x_strata, y_strata;
    uint32_t outputs;                 /* RTCUDA_AOV_* bits */
    uint32_t antialias_primary_rays;  /* bool */
    uint32_t antialias_secondary_rays;/* bool */
} rtcuda_settings;

enum {
    RTCUDA_STATS_COUNTERS = 1u << 0,      /* count BVH node / primitive fetches (instrumented traversal kernels) */
    RTCUDA_STATS_KERNEL_TIMES = 1u << 1   /* CUDA events around every extend / shade / shadow launch */
};

enum {
    /* Intersect triangles with the watertight test of Woop et al. 2013 instead of the reference's Moller-Trumbore
     * (crates/raytracing-cpu/src/geometry.rs:301-340, not watertight): no leaks along shared edges / silhouettes.
     * Off by default: the parity gates compare against the reference's test (SURVEY appendix A.1). */
    RTCUDA_BACKEND_WATERTIGHT = 1u << 0
};

/* The analogue of CpuBackendSettings (crates/raytracing-cpu/src/lib.rs:446-457) /
 * OptixBackendSettings (crates/raytracing-optix/src/lib.rs:25-28). */
typedef struct rtcuda_backend_settings {
    int32_t device_id;                /* CUDA device ordinal */
    uint32_t max_paths_in_flight;     /* wavefront size; 0 => default */
    /* Image-tile partition for multi-GPU (SURVEY §8e): this context renders the tiles (tx, ty) of the row-major tile
     * grid (crates/raytracing-cpu/src/lib.rs:481-504) with (ty * stride + tx) % tile_world == tile_rank, where stride is
     * the number of tiles per row, plus one when that number is a multiple of tile_world (so that ranks do not own whole
     * tile columns); all other pixels are left 0 so frames can be summed or gathered. */
    uint32_t tile_rank;
    uint32_t tile_world;              /* 0 or 1 => whole image */
    uint32_t collect_stats;           /* RTCUDA_STATS_* bits */
    uint32_t flags;                   /* RTCUDA_BACKEND_* bits */
    /* Edge of the square tiles dealt to the ranks: 0 => 64 (the reference's RenderTile grid); a power of two in
     * [8, 64]. Smaller tiles balance scenes whose cost is concentrated in part of the frame (C3: the box covers a
     * quarter of the 16:9 raster) at no cost in coherence: inside a tile pixels follow a Morton curve either way. */
    uint32_t tile_size;
    /* Multi-GPU inside one context (ABI v3; SURVEY §8b "CudaBackendSettings{device_ids / num_gpus}", the analogue of the CPU
     * backend's in-process worker pool, crates/raytracing-cpu/src/lib.rs:706-805): num_devices > 1 replicates the scene on
     * device_ids[0 .. num_devices) (rtcuda_scene_upload uploads and builds on all of them, one host thread per GPU), deals the
     * image tiles round-robin to them exactly like tile_rank / tile_world (which must then be left 0), and rtcuda_render
     * returns the complete frame: every GPU copies the pixels it owns straight into the caller's host planes. The device
     * variants (rtcuda_render_device, rtcuda_render_samples_device) take planes on device_ids[0]; the other GPUs send their
     * owned pixels there over NVLink (one peer copy of a packed buffer per GPU and frame). 0 or 1: one GPU, device_id.
     * Every pixel is the same as on one GPU, bit for bit. */
    uint32_t num_devices;
    int32_t device_ids[RTCUDA_MAX_DEVICES];
} rtcuda_backend_settings;

/* RenderOutput (crates/raytracing/src/renderer/mod.rs:49-59). NULL planes are skipped. */
typedef struct rtcuda_outputs {
    uint32_t width, height;           /* must equal the camera raster size */
    float* beauty;                    /* 3 floats / pixel */
    float* normals;                   /* 3 floats / pixel */
    float* albedo;                    /* 3 floats / pixel */
    float* uv;                        /* 2 floats / pixel */
    float* mip_level;                 /* 1 float / pixel */
    uint32_t* debug_ids;              /* 2 u32 / pixel: geom_id, prim_id */
    float* debug_depth;               /* 1 float / pixel */
} rtcuda_outputs;

/* SinglePixelOutput (crates/raytracing/src/renderer/mod.rs:75-82) */
typedef struct rtcuda_pixel_output {
    uint32_t sample_index;
    uint32_t hit;                     /* bool */
    float uv[2];
    float normal[3];
    float radiance[3];
} rtcuda_pixel_output;

/* Counters of the last render (SURVEY §8d): rays actually traced per class; BVH fetch counts per
 * traversal kernel (only with RTCUDA_STATS_COUNTERS); device milliseconds of the render window, of the BVH
 * build, and per kernel class (only with RTCUDA_STATS_KERNEL_TIMES: CUDA events around every launch). */
typedef struct rtcuda_stats {
    uint64_t samples;
    uint64_t primary_rays, bounce_rays, shadow_rays, aov_rays;
    uint64_t nodes_fetched, prims_fetched;      /* all traversal kernels */
    uint64_t extend_nodes, extend_prims;        /* closest-hit `extend` kernel */
    uint64_t shadow_nodes, shadow_prims;        /* any-hit `shadow` kernel */
    uint64_t shaded_vertices;                   /* path vertices that reached material evaluation */
    uint64_t kernel_launches;
    uint64_t extend_launches, shade_launches, shadow_launches;
    double render_ms;                 /* CUDA-event time, inputs resident, excludes D2H */
    double bvh_build_ms;              /* last scene upload */
    double upload_ms;
    double extend_ms, shade_ms, shadow_ms, other_ms;   /* RTCUDA_STATS_KERNEL_TIMES (other: raygen; see gather_ms) */
    uint64_t bvh_node_count, bvh_prim_count;
    /* NaN / Inf channels of the beauty plane of the last render: the device side of the reference's scan
     * (lib.rs:813-854); the binding prints its warnings ("R component of (x, y) is NaN", first 10) when non-zero. */
    uint64_t nonfinite_values;
    /* Camera rays (counted in primary_rays) that missed the scene bounds and were dropped before the wavefront: the
     * root-AABB reject of traverse_bvh (accel.rs:95) done in ray generation; only without an environment light. */
    uint64_t primary_rays_culled;
    /* Continuation rays of the last depth that could not add radiance (non-specular sample, no environment light:
     * crates/raytracing-cpu/src/lib.rs:294-298, 318-322) and were not traced; NOT counted in bounce_rays. The reference
     * traces them: bounce_rays + final_rays_skipped is its bounce-ray count. */
    uint64_t final_rays_skipped;
    /* 1 when the PLOC tree of the last upload was deeper than the traversal stack covers and the scene was rebuilt as an
     * LBVH (same pixels, usually more node fetches per ray). */
    uint64_t bvh_fallback_lbvh;
    /* ABI v3 */
    double gather_ms;                 /* RTCUDA_STATS_KERNEL_TIMES: the shadow-gather launches (shadow_ms is the any-hit kernel alone) */
    /* Pixels of this context that the beauty pass did not allocate path slots for: none of their camera rays can reach the
     * scene bounds (raster rectangle of the projected bounds; only without an environment light, pinhole / orthographic
     * cameras). Their samples are counted in primary_rays and primary_rays_culled like the per-sample culls. */
    uint64_t pixels_dropped;
    /* ABI v4 */
    double update_ms;                 /* device time of the last rtcuda_scene_update */
    /* SAH cost of the current wide tree, (A(root) + sum over inner children A(c) + sum over leaf children A(c) * |c|) / A(root)
     * with A the surface area of the child's float box (node and primitive cost 1); 0 until the first update computed it. */
    double bvh_sah_cost;
    uint64_t bvh_last_update;         /* last rtcuda_scene_update: 0 nothing changed, 1 camera / lights only, 2 refit, 3 rebuild */
} rtcuda_stats;

typedef struct rtcuda_ctx rtcuda_ctx;
typedef struct rtcuda_scene rtcuda_scene;

/* Replaces initOptix (csrc/host/lib_api.h:17). */
RTCUDA_API rtcuda_status rtcuda_init(const rtcuda_backend_settings* settings, rtcuda_ctx** out_ctx);
RTCUDA_API void rtcuda_shutdown(rtcuda_ctx* ctx);

/* Replaces prepare_cpu_acceleration_structures + CpuRaytracingContext::new
 * (crates/raytracing-cpu/src/scene.rs:14-73, lib.rs:81-105): copies the scene to the device,
 * builds the mip pyramids for trilinear textures and the 8-wide BVH on the device. */
RTCUDA_API rtcuda_status rtcuda_scene_upload(rtcuda_ctx* ctx, const rtcuda_scene_desc* desc, rtcuda_scene** out_scene);
RTCUDA_API void rtcuda_scene_release(rtcuda_scene* scene);

/* Moves what the caller moved: reads desc->camera (raster size and kind must be unchanged),
 * desc->instances[i].object_to_world (forward + inverse), and desc->lights[i]
 * position_or_direction / intensity_or_radiance / light_to_world.
 * desc must have the topology of the uploaded scene:
 *   - same shape / instance / light / material / texture / image counts;
 *   - same instances[i].shape;
 *   - same lights[i].kind and .shape.
 * Geometry arrays, shapes, materials, textures and images are NOT read (may be NULL).
 * On a mismatch: RTCUDA_ERR_INVALID_ARGUMENT and the scene is left untouched.
 * Blocks until the device scene is updated. Multi-device scenes are updated on every GPU.
 * The library compares desc against what it holds and does only the work the differences need: new kernel constants for
 * the camera and the lights; for moved instances a refit of the wide BVH on the device (primitive slots recomputed in
 * place, node boxes re-fitted level by level), or a rebuild from the resident geometry when the refit's SAH cost grew too
 * far over the built tree's. Frames rendered afterwards equal the frames of a fresh upload of desc, bit for bit. */
RTCUDA_API rtcuda_status rtcuda_scene_update(rtcuda_scene* scene, const rtcuda_scene_desc* desc);

/* The path-state arena of a released scene (multi-GB: batches are sized for HBM) is parked per process and reused by
 * the next scene on the same device, so back-to-back one-shot renders do not pay for mapping device memory again.
 * This call returns the parked memory to the driver. No reference counterpart (the CPU backend allocates per tile). */
RTCUDA_API void rtcuda_release_cached_memory(void);

/* Optional allocator for the HOST planes handed to rtcuda_render: page-locked memory from a per-process cache. A frame rendered
 * into such a plane is written by the GPU's copy engine directly (no staging copy on the host, no first-touch page faults of a
 * freshly allocated frame: ~2.5 ms per 1080p beauty plane). Planes from anywhere else (Vec<f32>, malloc) keep working through a
 * staging buffer. rtcuda_host_free returns the memory to the cache (rtcuda_release_cached_memory gives it back to the OS).
 * Counterpart in the reference: RenderOutput's Vec<Vec3> planes (renderer/mod.rs:53-73), allocated by the backend. */
RTCUDA_API void* rtcuda_host_alloc(size_t bytes);
RTCUDA_API void rtcuda_host_free(void* ptr);

/* Replaces raytracing_cpu::render (lib.rs:645-858). */
RTCUDA_API rtcuda_status rtcuda_render(rtcuda_scene* scene, const rtcuda_settings* settings, rtcuda_outputs* outputs);

/* Same render, but every non-NULL plane of `outputs` is a DEVICE pointer on this context's GPU
 * (used to hand the frame to an NCCL reduce without a host round trip, SURVEY §8e). */
RTCUDA_API rtcuda_status rtcuda_render_device(rtcuda_scene* scene, const rtcuda_settings* settings, rtcuda_outputs* device_outputs);

/* Sample-range render (SURVEY §8e "alternate mode", and the progressive hook a viewer needs): traces samples
 * [sample_lo, sample_hi) of every pixel this context owns, with exactly the streams `rtcuda_render` gives those sample
 * indices at settings->samples_per_pixel, and writes the UN-NORMALISED radiance sum to the device plane `beauty_sum`
 * (3 floats / pixel, row-major; pixels of other ranks 0). Summing the planes of disjoint ranges and multiplying by
 * 1 / samples_per_pixel reproduces `rtcuda_render` up to the association of the float sum over samples (the render
 * itself adds samples in index order, like render_tile, lib.rs:538-548). Beauty only: AOVs are sample-independent. */
RTCUDA_API rtcuda_status rtcuda_render_samples_device(rtcuda_scene* scene, const rtcuda_settings* settings,
                                                      uint32_t sample_lo, uint32_t sample_hi, float* beauty_sum);

/* Progressive form of the call above — the hook a viewer needs (crates/viewer/src/render_output_view.rs:84-98 calls `render`
 * once and shows the result; with this a caller can show a converging image): ADDS the un-normalised radiance sum of
 * samples [sample_lo, sample_hi) to the device plane `beauty_sum` in place (pixels of other ranks untouched). Starting from
 * a zeroed plane and calling it for consecutive ranges, `beauty_sum / sample_hi` after each call is the image a render
 * with sample_hi samples per pixel of the same streams would give (up to the association of the float sum). */
RTCUDA_API rtcuda_status rtcuda_render_samples_accumulate_device(rtcuda_scene* scene, const rtcuda_settings* settings,
                                                                 uint32_t sample_lo, uint32_t sample_hi, float* beauty_sum);

/* Replaces raytracing_cpu::render_single_pixel (lib.rs:860-931) in the Range<u32> shape of
 * raytracing_optix::render_single_pixel (crates/raytracing-optix/src/lib.rs:172-234):
 * out has sample_hi - sample_lo entries. Out-of-bounds x / y are clamped (lib.rs:867-876). */
RTCUDA_API rtcuda_status rtcuda_render_pixel(rtcuda_scene* scene, const rtcuda_settings* settings,
                                             uint32_t x, uint32_t y, uint32_t sample_lo, uint32_t sample_hi,
                                             rtcuda_pixel_output* out);

/* Ray queries: caller-supplied rays against the uploaded scene's BVH (the analogue of Embree's rtcIntersect / rtcOccluded).
 * `rays` is `count` x 8 floats per ray: origin.xyz, t_min, direction.xyz, t_max (32 bytes, the shape of the render's ray queue).
 *   - Closest hit: the hit with the smallest t in [t_min, t_max]. Both bounds are inclusive, there is no back-face culling, and
 *     equal-t ties go to the larger (geom_id, prim_id): the acceptance rule of the render's traversal. Triangles are tested with
 *     the context's test (Moller-Trumbore, or Woop's watertight test under RTCUDA_BACKEND_WATERTIGHT). t is in units of the
 *     direction's length (the direction is not normalised) and there is no implicit epsilon: a ray that starts on a surface
 *     needs its own t_min offset.
 *   - Outputs, each NULL to skip it (at least one must be given): t[i]; ids[2i] = instance index (geom_id), ids[2i+1] = primitive
 *     index within the shape (prim_id; 0 for a sphere); barycentrics[2i], [2i+1] = (u, v), the weights of v1 and v2 (0 for a
 *     sphere). The winning triangle is re-tested in object space like the first-hit AOVs, so t / u / v are the reference's
 *     intersect_shape values to rounding.
 *   - Miss: t = +INFINITY, both ids RTCUDA_NONE, barycentrics 0. A ray with t_min > t_max, a zero direction, a NaN bound or a
 *     non-finite origin or direction component is a miss, not an error.
 *   - Occlusion: occluded[i] = 1 when any primitive is hit in [t_min, t_max], else 0 (the any-hit walk of shadow rays).
 *   - The plain variants take HOST arrays and block until the results are on the host; on a multi-device scene the rays are cut
 *     into contiguous slices, one per GPU. The _device variants take DEVICE pointers on device_ids[0] (the context's GPU), rays
 *     16-byte aligned, and block until the outputs are written. The library's stream does not wait for other streams: the caller
 *     must have finished writing the rays (e.g. torch.cuda.synchronize()) before the call.
 *   - count == 0 is RTCUDA_OK; count >= 2^32, NULL rays with count > 0, no output, or (device variants) a pointer that is not
 *     device memory of that GPU are RTCUDA_ERR_INVALID_ARGUMENT, refused before any device work.
 *   - Queries read the scene only: rtcuda_get_stats keeps reporting the last render, and nothing a render caches is touched.
 * Results are the same bit for bit on one GPU, on several, and from host or device arrays. */
RTCUDA_API rtcuda_status rtcuda_trace_rays(rtcuda_scene* scene, const float* rays, uint64_t count, float* t, uint32_t* ids,
                                           float* barycentrics);
RTCUDA_API rtcuda_status rtcuda_trace_rays_device(rtcuda_scene* scene, const float* rays, uint64_t count, float* t, uint32_t* ids,
                                                  float* barycentrics);
RTCUDA_API rtcuda_status rtcuda_occluded(rtcuda_scene* scene, const float* rays, uint64_t count, uint8_t* occluded);
RTCUDA_API rtcuda_status rtcuda_occluded_device(rtcuda_scene* scene, const float* rays, uint64_t count, uint8_t* occluded);

/* One closest hit with the reference's HitInfo (accel.rs:13-25) plus the material's albedo. 64 bytes (four 16-byte
 * words: the device writes each with one 16-byte store, so device arrays of it must be 16-byte aligned). */
typedef struct rtcuda_surface {
    float point[3];  float t;             /* world-space hit point; t exactly as rtcuda_trace_rays reports it */
    float normal[3]; uint32_t material;   /* HitInfo::normal (world space, unit, NOT flipped toward the ray); instance's material */
    float uv[2];     uint32_t geom_id; uint32_t prim_id;   /* HitInfo::uv; ids exactly as rtcuda_trace_rays */
    float albedo[3]; uint32_t light;      /* get_albedo with a zero texture footprint; instance's area light or RTCUDA_NONE */
} rtcuda_surface;

/* Surface queries: the shading attributes at the closest hit of caller-supplied rays (picking, lightmap and probe set-up, G-buffers
 * and denoiser guides for cameras the scene format lacks).
 *   - Rays are packed and accepted exactly like the ray queries above: 8 floats per ray, the same closest-hit rule, the context's
 *     triangle test, no epsilon, t in units of the direction's length.
 *   - t, geom_id and prim_id are bit-identical to rtcuda_trace_rays on the same ray (the same walk and object-space re-test).
 *   - point: o + d * t for triangles; for spheres the object-space hit point taken through the instance's object-to-world transform.
 *   - normal, uv: the reference's HitInfo::normal / HitInfo::uv, the values of the NORMALS and UV_COORDS first-hit planes. The
 *     normal is the interpolated vertex normal (or the geometric one of a mesh without normals, or (p - c) / r on a sphere) through
 *     the instance's inverse transpose, unit length, and not flipped toward the ray. A mesh without uvs uses (0,0), (1,0), (0,1);
 *     a sphere uses (phi / 2pi, theta / pi).
 *   - material, light: the hit instance's material index and area light (RTCUDA_NONE when it emits nothing).
 *   - albedo: the material's albedo with a zero texture footprint (uv only), as the path tracer evaluates every hit that has no ray
 *     differentials, rtcuda_radiance's first vertex included. A caller's ray has no differentials, so for trilinear (mip-mapped)
 *     image textures it can differ from the render's ALBEDO plane, which filters over the camera's pixel footprint.
 *   - Miss, or an invalid ray (the ray-query rule): t = +INFINITY, point / normal / uv / albedo 0, geom_id / prim_id / material /
 *     light RTCUDA_NONE.
 *   - rtcuda_trace_surfaces takes HOST arrays and blocks until the records are on the host; on a multi-device scene the rays are cut
 *     into contiguous slices, one per GPU. rtcuda_trace_surfaces_device takes DEVICE pointers on device_ids[0], rays and surfaces
 *     16-byte aligned, and blocks until the records are written; the caller must have finished writing the rays.
 *   - count == 0 is RTCUDA_OK; count >= 2^32, NULL rays with count > 0, NULL surfaces, a NULL scene, or (device variant) a pointer
 *     that is not device memory of that GPU or is misaligned are RTCUDA_ERR_INVALID_ARGUMENT, refused before any device work.
 *   - Like the ray queries they read the scene only: rtcuda_get_stats keeps reporting the last render, and nothing a render keeps
 *     (frame graph, pixel lists, path-state memory) is touched.
 * Records are the same bit for bit on one GPU, on several, and from host or device arrays. */
RTCUDA_API rtcuda_status rtcuda_trace_surfaces(rtcuda_scene* scene, const float* rays, uint64_t count, rtcuda_surface* surfaces);
RTCUDA_API rtcuda_status rtcuda_trace_surfaces_device(rtcuda_scene* scene, const float* rays, uint64_t count, rtcuda_surface* surfaces);

/* Radiance along caller-supplied rays: the path tracer's estimate of the radiance arriving at each ray's origin from its direction
 * (light probes, lightmap texels, cameras the scene format lacks, reference radiance along chosen rays).
 *   - `rays` is `count` x 8 floats per ray, packed like the ray queries: origin.xyz, t_min, direction.xyz, t_max. The direction need
 *     not have unit length: each ray is first normalised as len = sqrtf((dx*dx + dy*dy) + dz*dz), d' = d / len (one IEEE division
 *     per component), t_min' = t_min * len, t_max' = t_max * len, and its first segment is traced over [t_min', t_max'].
 *   - radiance[3i .. 3i+2] = the mean over samples [0, settings->samples_per_pixel) of the radiance the integrator carries back
 *     along ray i: the renderer's path (emission, next-event estimation, every BSDF, textures, environment light), summed in
 *     sample order and multiplied by 1 / spp like a pixel. A valid ray that hits nothing returns the environment radiance (0
 *     without an environment light). An invalid ray (the ray-query rule: non-finite origin or direction, zero direction, NaN
 *     bound, t_min > t_max; also a direction whose squared length is outside the float range) returns exactly 0 and is not traced.
 *   - Settings used: max_ray_depth, accumulate_bounces, light_sample_count, samples_per_pixel, the seed and the sampler fields.
 *     `outputs` is ignored, and antialias_primary_rays is treated as 0 (a caller's ray has no differentials).
 *   - Sampler streams: sample s of ray i draws from the stream of the renderer's pixel (k & 0xffff, k >> 16) at sample s, with
 *     k = stream_base + i; no camera numbers are drawn. So key k shares its numbers with that pixel at the same seed (callers who
 *     combine both should use different seeds), and a ray's result depends only on the ray, its key, the settings and the scene:
 *     not on chunking, batch sizes, GPU count or host vs device arrays. Slicing a ray set over calls with stream_base = the
 *     slice's offset gives the bits of one call.
 *   - rtcuda_radiance takes HOST arrays and blocks until the radiance is on the host; on a multi-device scene the rays are cut
 *     into contiguous slices, one per GPU, each keeping its keys. rtcuda_radiance_device takes DEVICE pointers on device_ids[0],
 *     rays 16-byte aligned, and blocks until the radiance is written; the caller must have finished writing the rays.
 *   - count == 0 is RTCUDA_OK. count >= 2^32, stream_base + count > 2^32, NULL rays with count > 0, NULL radiance, NULL settings,
 *     samples_per_pixel == 0, strata < 1 with the stratified sampler, or (device variant) a pointer that is not device memory of
 *     that GPU are RTCUDA_ERR_INVALID_ARGUMENT, refused before any device work.
 *   - rtcuda_get_stats keeps reporting the last render. The call may reuse (and grow) the scene's path-state memory. */
RTCUDA_API rtcuda_status rtcuda_radiance(rtcuda_scene* scene, const rtcuda_settings* settings, const float* rays, uint64_t count,
                                         uint32_t stream_base, float* radiance);
RTCUDA_API rtcuda_status rtcuda_radiance_device(rtcuda_scene* scene, const rtcuda_settings* settings, const float* rays, uint64_t count,
                                                uint32_t stream_base, float* radiance);

RTCUDA_API rtcuda_status rtcuda_get_stats(const rtcuda_scene* scene, rtcuda_stats* out);

/* Message of the last failing call on this thread ("" if none). */
RTCUDA_API const char* rtcuda_last_error(void);
RTCUDA_API uint32_t rtcuda_abi_version(void);

/* Binding self-check: sizeof() of the ABI structs as this library was compiled, in the order
 * camera, shape, instance, light, material, texture, image, scene_desc, settings,
 * backend_settings, outputs, pixel_output, stats. Returns the number of entries written. */
RTCUDA_API uint32_t rtcuda_abi_struct_sizes(uint32_t* out, uint32_t capacity);

#ifdef __cplusplus
}
#endif
#endif /* RTCUDA_H */
