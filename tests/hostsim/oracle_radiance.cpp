// oracle_radiance.cpp — TEST INFRASTRUCTURE ONLY. The reference for rtcuda_radiance: the CPU oracle (oracle/oracle.cpp, compiled
// into this library unchanged) runs its ray_radiance (lib.rs:247-393) per caller-supplied ray and sample. ray_radiance traces the
// first segment over the camera clip of the scene description, so each thread works on a private copy of the description whose
// camera near / far clip it sets to the ray's normalised range. Never loaded by the product.
#include "../../oracle/oracle.cpp"

namespace {
// The query rule for rays that are not traced (include/rtcuda.h): non-finite origin / direction, zero direction, NaN bound,
// t_min > t_max
bool ray_valid(const float* o4, const float* d4) {
    for (int k = 0; k < 3; k++)
        if (!std::isfinite(o4[k]) || !std::isfinite(d4[k])) return false;
    return (d4[0] != 0.0f || d4[1] != 0.0f || d4[2] != 0.0f) && o4[3] <= d4[3];
}

// rt_query.h radiance_prep_ray restated: len = sqrtf((dx*dx + dy*dy) + dz*dz), d' = d / len, t' = t * len (this file is built with
// -ffp-contract=off); invalid rays become (0, 0, 0, 1 | 0, 0, 0, 0)
bool prep_ray(const float* r, float* p) {
    const float len = std::sqrt((r[4] * r[4] + r[5] * r[5]) + r[6] * r[6]);
    const float q[8] = {r[0], r[1], r[2], r[3] * len, r[4] / len, r[5] / len, r[6] / len, r[7] * len};
    const bool valid = ray_valid(r, r + 4) && ray_valid(q, q + 4);
    for (int k = 0; k < 8; k++) p[k] = valid ? q[k] : (k == 3 ? 1.0f : 0.0f);
    return valid;
}
}  // namespace

extern "C" {
// n rays of 8 floats; radiance[3i..3i+2] = the mean of ray_radiance over samples [0, spp) from the sampler stream of pixel
// (k & 0xffff, k >> 16), k = stream_base + i, summed in sample order and multiplied by 1 / spp; antialias_primary_rays is taken
// as 0. `prepared` (may be null) receives the normalised rays.
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
