// rays.cpp — TEST INFRASTRUCTURE ONLY. liboracle.so's translation unit: the oracle (oracle.cpp, included unchanged) plus its
// references for the library's caller-supplied rays. oracle.cpp alone is the CPU-baseline build (oracle_py.use_native_build),
// so the renderer it times compiles to the same code whatever entry points are added here. Build: see oracle/Makefile.
#include "oracle.cpp"

namespace {

// The query API's rule for caller-supplied rays it does not trace (include/rtcuda.h), on 8 floats (origin, t_min, direction,
// t_max): non-finite origin / direction, zero direction, NaN bound, t_min > t_max
bool ray_valid(const float* r) {
    for (int k : {0, 1, 2, 4, 5, 6})
        if (!std::isfinite(r[k])) return false;
    return (r[4] != 0.0f || r[5] != 0.0f || r[6] != 0.0f) && r[3] <= r[7];
}

// rt_query.h radiance_prep_ray restated: len = sqrtf((dx*dx + dy*dy) + dz*dz), d' = d / len, t' = t * len (this file is built with
// -ffp-contract=off); invalid rays become (0, 0, 0, 1 | 0, 0, 0, 0)
bool prep_ray(const float* r, float* p) {
    const float len = std::sqrt((r[4] * r[4] + r[5] * r[5]) + r[6] * r[6]);
    const float q[8] = {r[0], r[1], r[2], r[3] * len, r[4] / len, r[5] / len, r[6] / len, r[7] * len};
    const bool valid = ray_valid(r) && ray_valid(q);
    for (int k = 0; k < 8; k++) p[k] = valid ? q[k] : (k == 3 ? 1.0f : 0.0f);
    return valid;
}

}  // namespace

extern "C" {

// ---- the references for the library's caller-supplied rays: each ray walked with traverse_bvh over its own [t_min, t_max] ----

// n rays of 8 floats (origin, t_min, direction, t_max). flags: 1 = brute force. Closest hit into t (+inf on a miss), ids
// (geom_id, prim_id; RTCUDA_NONE on a miss) and barycentrics (u, v of the reference's object-space Moller-Trumbore; 0 for
// spheres); any hit into occluded. Every output may be null.
__attribute__((visibility("default")))
int oracle_trace_rays(const rtcuda_scene_desc* desc, const float* rays, uint64_t n, uint32_t flags, float* t, uint32_t* ids,
                      float* barycentrics, uint8_t* occluded) {
    if (!desc || (!rays && n)) return 1;
    SceneView sv(desc);
    Context ctx;
    build_context(ctx, sv, flags & ORACLE_FLAG_BRUTE_FORCE);
    for (uint64_t i = 0; i < n; i++) {
        const float* r = rays + 8 * i;
        const Ray ray{{r[0], r[1], r[2]}, {r[4], r[5], r[6]}};
        const bool valid = ray_valid(r);
        HitInfo h;
        const bool hit = valid && traverse_bvh(ctx, ray, r[3], r[7], false, h);
        float u = 0.0f, v = 0.0f, th = hit ? h.t : INFINITY;
        if (hit) {
            const uint32_t shape = desc->instances[h.geom_id].shape;
            if (desc->shapes[shape].kind == RTCUDA_SHAPE_TRIANGLE_MESH) {   // the winner's barycentrics (intersect_shape reports uvs)
                const MeshView& m = sv.meshes[shape];
                const Ray o_ray = ray_transform(ray, sv.inst_tf[h.geom_id].invert());
                float tt;
                ray_triangle_intersect(m.v(m.tris[3 * h.prim_id]), m.v(m.tris[3 * h.prim_id + 1]), m.v(m.tris[3 * h.prim_id + 2]), o_ray,
                                       r[3], r[7], tt, u, v);
            }
        }
        if (t) t[i] = th;
        if (ids) { ids[2 * i] = hit ? h.geom_id : RTCUDA_NONE; ids[2 * i + 1] = hit ? h.prim_id : RTCUDA_NONE; }
        if (barycentrics) { barycentrics[2 * i] = u; barycentrics[2 * i + 1] = v; }
        if (occluded) {
            HitInfo a;
            occluded[i] = valid && traverse_bvh(ctx, ray, r[3], r[7], true, a) ? 1 : 0;
        }
    }
    return 0;
}

// n rays of 8 floats. flags: 1 = brute force. n records of 16 words laid out like rtcuda_surface: the winner's HitInfo and
// get_albedo with a zero texture footprint, (point.xyz, t), (normal.xyz, material), (uv, geom_id, prim_id), (albedo.xyz, light).
// A miss is (0, inf), (0, NONE), (0, 0, NONE, NONE), (0, NONE).
__attribute__((visibility("default")))
int oracle_trace_surfaces(const rtcuda_scene_desc* desc, const float* rays, uint64_t n, uint32_t flags, float* surfaces) {
    if (!desc || (!rays && n) || !surfaces) return 1;
    SceneView sv(desc);
    Context ctx;
    build_context(ctx, sv, flags & ORACLE_FLAG_BRUTE_FORCE);
    for (uint64_t i = 0; i < n; i++) {
        const float* r = rays + 8 * i;
        const Ray ray{{r[0], r[1], r[2]}, {r[4], r[5], r[6]}};
        float* o = surfaces + 16 * i;
        HitInfo h;
        if (!ray_valid(r) || !traverse_bvh(ctx, ray, r[3], r[7], false, h)) {
            const uint32_t none = RTCUDA_NONE;
            for (int k = 0; k < 16; k++) o[k] = 0.0f;
            o[3] = INFINITY;
            for (int k : {7, 10, 11, 15}) std::memcpy(o + k, &none, 4);
            continue;
        }
        const Vec3 a = get_albedo(sv, desc->materials[h.material_idx], mec_no_aa(h.uv));
        const float f[16] = {h.point.x, h.point.y, h.point.z, h.t, h.normal.x, h.normal.y, h.normal.z, 0.0f,
                             h.uv.x, h.uv.y, 0.0f, 0.0f, a.x, a.y, a.z, 0.0f};
        std::memcpy(o, f, sizeof f);
        std::memcpy(o + 7, &h.material_idx, 4);
        std::memcpy(o + 10, &h.geom_id, 4);
        std::memcpy(o + 11, &h.prim_id, 4);
        std::memcpy(o + 15, &h.light_idx, 4);
    }
    return 0;
}

// The reference for rtcuda_radiance: ray_radiance (lib.rs:247-393) per ray and sample. n rays of 8 floats; radiance[3i..3i+2] =
// the mean over samples [0, spp) from the sampler stream of pixel (k & 0xffff, k >> 16), k = stream_base + i, summed in sample
// order and multiplied by 1 / spp; antialias_primary_rays is taken as 0. `prepared` (may be null) receives the normalised rays.
// ray_radiance traces the first segment over the camera clip of the scene description, so each thread works on a private copy
// of the description whose near / far clip it sets to the ray's normalised range.
__attribute__((visibility("default")))
int oracle_radiance(const rtcuda_scene_desc* desc, const rtcuda_settings* st, const float* rays, uint64_t n, uint32_t stream_base,
                    uint32_t num_threads, float* radiance, float* prepared) {
    if (!desc || !st || (!rays && n) || !radiance) return 1;
    rtcuda_settings s = *st;
    s.antialias_primary_rays = 0;
    const float inv_spp = 1.0f / (float)s.samples_per_pixel;
    auto worker = [&](uint32_t t, uint32_t nt) {
        rtcuda_scene_desc d = *desc;   // the SceneView (and so ray_radiance) reads the camera clip from here
        SceneView sv(&d);
        Context ctx;
        build_context(ctx, sv, false);
        const Sampler base = Sampler::from_settings(s);
        for (uint64_t i = t; i < n; i += nt) {
            float p[8];
            const bool valid = prep_ray(rays + 8 * i, p);
            if (prepared) std::memcpy(prepared + 8 * i, p, sizeof p);
            Vec3 sum{0, 0, 0};
            if (valid) {
                d.camera.near_clip = p[3];
                d.camera.far_clip = p[7];
                const uint32_t k = stream_base + (uint32_t)i;
                for (uint32_t j = 0; j < s.samples_per_pixel; j++) {
                    Sampler smp = base;
                    smp.start_sample(k & 0xffffu, k >> 16, j);
                    const Ray ray{{p[0], p[1], p[2]}, {p[4], p[5], p[6]}};
                    const RayDifferentials rd{};
                    sum += ray_radiance(ray, rd, ctx, smp, s);
                }
            }
            radiance[3 * i] = sum.x * inv_spp;
            radiance[3 * i + 1] = sum.y * inv_spp;
            radiance[3 * i + 2] = sum.z * inv_spp;
        }
    };
    if (num_threads <= 1) worker(0, 1);
    else {
        std::vector<std::thread> th;
        for (uint32_t t = 0; t < num_threads; t++) th.emplace_back(worker, t, num_threads);
        for (auto& x : th) x.join();
    }
    return 0;
}
}  // extern "C"
