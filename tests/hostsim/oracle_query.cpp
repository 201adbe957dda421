// oracle_query.cpp — TEST INFRASTRUCTURE ONLY. The reference for the library's ray queries: the CPU oracle (oracle/oracle.cpp,
// compiled into this library unchanged) walks each caller-supplied ray with traverse_bvh over the ray's own [t_min, t_max], in
// BVH2 or brute-force mode, and reports the object-space (t, u, v) of the reference's Moller-Trumbore. Never loaded by the product.
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
// n rays of 8 floats (origin, t_min, direction, t_max). flags: 1 = brute force. Closest hit into t (+inf on a miss), ids
// (geom_id, prim_id; RTCUDA_NONE on a miss) and barycentrics (u, v of the object-space test; 0 for spheres); any hit into
// occluded. Every output may be null.
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
}  // extern "C"
