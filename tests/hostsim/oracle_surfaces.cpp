// oracle_surfaces.cpp — TEST INFRASTRUCTURE ONLY. The reference for the library's surface query: the CPU oracle (oracle/oracle.cpp,
// compiled into this library unchanged) walks each caller-supplied ray with traverse_bvh over the ray's own [t_min, t_max], in
// BVH2 or brute-force mode, and reports the winner's HitInfo (point, normal, uv, material, light) and get_albedo with a zero
// texture footprint. Never loaded by the product.
#include "../../oracle/oracle.cpp"

namespace {
// The query API's rule for rays it does not trace (include/rtcuda.h): non-finite origin / direction, zero direction, NaN bound,
// t_min > t_max
bool ray_valid(const float* r) {
    for (int k : {0, 1, 2, 4, 5, 6})
        if (!std::isfinite(r[k])) return false;
    return (r[4] != 0.0f || r[5] != 0.0f || r[6] != 0.0f) && r[3] <= r[7];
}
}  // namespace

extern "C" {
// n rays of 8 floats (origin, t_min, direction, t_max). flags: 1 = brute force. n records of 16 words laid out like
// rtcuda_surface: (point.xyz, t), (normal.xyz, material), (uv, geom_id, prim_id), (albedo.xyz, light). A miss is (0, inf),
// (0, NONE), (0, 0, NONE, NONE), (0, NONE).
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
}  // extern "C"
