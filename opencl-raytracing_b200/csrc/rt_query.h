// rt_query.h — ray queries on an uploaded scene (rtcuda_trace_rays / rtcuda_occluded): the per-ray logic of k_trace (kernels.cu,
// the traversal) and k_trace_finish (kernels_aov.cu, ids and the object-space re-test), shared with the CPU harness. Also the
// surface record of rtcuda_trace_surfaces (k_surface_finish, kernels_aov.cu), and the per-ray stages of rtcuda_radiance (prep,
// live list, ray generation) that feed the caller's rays into the wavefront integrator.
//
// A query ray is two float4, (origin.xyz, t_min) and (direction.xyz, t_max): the shape of the wavefront's ray queue. Closest hit
// and occlusion follow the acceptance rule of the extend / shadow walks (rt_traverse.h): hits with t in [t_min, t_max], both
// bounds inclusive, no back-face culling, equal-t ties to the larger (geom_id, prim_id).
#pragma once
#include "rt_integrator.h"

namespace rt {

// Rays the traversal cannot take are misses: a non-finite origin or direction component, a zero direction, a NaN bound or
// t_min > t_max. (A NaN or infinite origin would otherwise pass the triangle test's range checks, which NaN compares never fail.)
RT_HD bool query_ray_valid(float4 o4, float4 d4) {
    const float big = 3.402823466e38f;
    const bool finite = fabsf(o4.x) <= big && fabsf(o4.y) <= big && fabsf(o4.z) <= big && fabsf(d4.x) <= big && fabsf(d4.y) <= big &&
                        fabsf(d4.z) <= big;
    return finite && (d4.x != 0.0f || d4.y != 0.0f || d4.z != 0.0f) && o4.w <= d4.w;
}

// The 16-byte scratch entry of a closest-hit query between the two kernels: the traversal's Hit (t, packed primitive slot, u, v)
RT_HD float4 query_miss_entry() { return make_float4(RT_INF, u2f(NONE), 0.0f, 0.0f); }
RT_HD float4 query_hit_entry(const Hit& h) { return make_float4(h.t, u2f(h.prim), h.u, h.v); }

// One ray start to finish with the walk of rt_traverse.h (the CPU harness; k_trace runs the same state machine per warp phase)
RT_HD float4 query_closest_ray(const SceneD& sc, float4 o4, float4 d4) {
    Hit h;
    if (!query_ray_valid(o4, d4) || !traverse<false, false>(sc, xyz(o4), xyz(d4), o4.w, d4.w, h, nullptr)) return query_miss_entry();
    return query_hit_entry(h);
}
RT_HD uint8_t query_occluded_ray(const SceneD& sc, float4 o4, float4 d4) {
    Hit h;
    return query_ray_valid(o4, d4) && traverse<true, false>(sc, xyz(o4), xyz(d4), o4.w, d4.w, h, nullptr) ? 1u : 0u;
}

// Outputs of a closest-hit query, indexed like the rays; null = not requested
struct QueryOut {
    float* t;          // 1 per ray: hit t, +inf on a miss
    uint32_t* ids;     // 2 per ray: geom_id (instance), prim_id (0 for a sphere); NONE on a miss
    float* uv;         // 2 per ray: barycentrics (weights of v1, v2), 0 for spheres and misses
};

// Ray i's scratch entry -> ids through the primitive slot, the winning triangle re-tested in object space over the ray's own
// [t_min, t_max] like the first-hit AOVs (refine_triangle_hit_in_object_space), then the requested outputs.
RT_HD void trace_finish_body(uint32_t i, const SceneD& sc, const float4* rays, const float4* hits, const QueryOut& out) {
    const float4 e = hits[i];
    Hit h;
    h.t = e.x; h.prim = f2u(e.y); h.u = e.z; h.v = e.w;
    uint32_t geom = NONE, pid = NONE;
    if (h.prim != NONE) {
        const Prim* pr = sc.prims + h.prim;
        geom = f2u(ldg(&pr->a).w);
        pid = f2u(ldg(&pr->b).w);
        const float4 o4 = rays[2 * (size_t)i], d4 = rays[2 * (size_t)i + 1];
        Ray ray;
        ray.o = xyz(o4);
        ray.d = xyz(d4);
        refine_triangle_hit_in_object_space(sc, ray, o4.w, d4.w, h);
    } else {
        h.t = RT_INF; h.u = 0.0f; h.v = 0.0f;
    }
    if (out.t) out.t[i] = h.t;
    if (out.ids) { out.ids[2 * (size_t)i] = geom; out.ids[2 * (size_t)i + 1] = pid; }
    if (out.uv) { out.uv[2 * (size_t)i] = h.u; out.uv[2 * (size_t)i + 1] = h.v; }
}

// ---- the surface at caller-supplied rays' closest hits (rtcuda_trace_surfaces) ------------------------------------------------
// Ray i's record is four float4 at out[4i]: the layout of rtcuda_surface (include/rtcuda.h; api.cu static_asserts it):
//   (point.xyz, t), (normal.xyz, material), (uv.xy, geom_id, prim_id), (albedo.xyz, light).
// t and the ids are trace_finish_body's (ids from the primitive slot, the winner re-tested in object space over the ray's own range);
// point / normal / uv / material / light are reconstruct_hit's HitInfo, and the albedo is get_albedo with a zero texture footprint,
// as for every hit without ray differentials. A miss (or an invalid ray, which k_trace misses) is (0, +inf), (0, NONE),
// (0, 0, NONE, NONE), (0, NONE).
RT_HD void surface_finish_body(uint32_t i, const SceneD& sc, const float4* rays, const float4* hits, float4* out) {
    const float4 e = hits[i];
    Hit h;
    h.t = e.x; h.prim = f2u(e.y); h.u = e.z; h.v = e.w;
    float4* o = out + 4 * (size_t)i;
    if (h.prim == NONE) {
        o[0] = make_float4(0.0f, 0.0f, 0.0f, RT_INF);
        o[1] = make_float4(0.0f, 0.0f, 0.0f, u2f(NONE));
        o[2] = make_float4(0.0f, 0.0f, u2f(NONE), u2f(NONE));
        o[3] = make_float4(0.0f, 0.0f, 0.0f, u2f(NONE));
        return;
    }
    const Prim* pr = sc.prims + h.prim;
    const uint32_t geom = f2u(ldg(&pr->a).w), pid = f2u(ldg(&pr->b).w);
    const float4 o4 = rays[2 * (size_t)i], d4 = rays[2 * (size_t)i + 1];
    Ray ray;
    ray.o = xyz(o4);
    ray.d = xyz(d4);
    refine_triangle_hit_in_object_space(sc, ray, o4.w, d4.w, h);
    HitInfo hit;
    reconstruct_hit(sc, ray.o, ray.d, h, false, hit);
    const V3 a = get_albedo(sc, sc.materials[hit.material], matctx_no_aa(hit.uv));
    o[0] = make_float4(hit.point.x, hit.point.y, hit.point.z, h.t);
    o[1] = make_float4(hit.normal.x, hit.normal.y, hit.normal.z, u2f(hit.material));
    o[2] = make_float4(hit.uv.x, hit.uv.y, u2f(geom), u2f(pid));
    o[3] = make_float4(a.x, a.y, a.z, u2f(hit.light));
}

// ---- radiance along caller-supplied rays (rtcuda_radiance) -------------------------------------------------------------------
// The BSDFs need a unit wo, so a caller's ray is normalised first: len = sqrtf((dx*dx + dy*dy) + dz*dz), d' = d / len (one IEEE
// division per component), t' = t * len for both bounds. k_radiance_prep runs this in the IEEE translation unit (kernels_aov.cu) so
// that the CPU reference reproduces it bit for bit. A ray the query rule calls invalid (query_ray_valid), or whose normalised form
// is (|d|^2 outside the float range), becomes the zero-direction ray below: k_trace misses it and it is never live, so its
// radiance is exactly 0. Returns whether the ray is valid.
RT_HD bool radiance_prep_ray(float4 o4, float4 d4, float4& po, float4& pd) {
    const float len = sqrtf((d4.x * d4.x + d4.y * d4.y) + d4.z * d4.z);
    po = make_float4(o4.x, o4.y, o4.z, o4.w * len);
    pd = make_float4(d4.x / len, d4.y / len, d4.z / len, d4.w * len);
    if (query_ray_valid(o4, d4) && query_ray_valid(po, pd)) return true;
    po = make_float4(0.0f, 0.0f, 0.0f, 1.0f);
    pd = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    return false;
}

// A prepared ray takes path slots when it is valid and its first segment either hit something or ends in the environment: the
// per-ray form of the renderer's pixel culling. Every other ray's radiance is 0.
RT_HD bool radiance_ray_live(const SceneD& sc, const float4* rays, const float4* first_hits, uint32_t r) {
    return query_ray_valid(rays[2 * (size_t)r], rays[2 * (size_t)r + 1]) && (f2u(first_hits[r].y) != NONE || sc.env_texture != NONE);
}

// k_raygen_rays: path slot `slot` of a batch over (live rays x samples), laid out like the renderer's (slot = s_local * n_pixels +
// p_local, w.pixel_list = the live rays' indices in the chunk). Sample s of ray r uses the sampler stream of the renderer's pixel
// (k & 0xffff, k >> 16), k = key_base + r, at dimension 0: no camera draws, the first draw is the first bounce's. The slot starts
// like a camera path (radiance 0, weight 1, specular flag set) and is queued at position `slot` with the ray's depth-0 hit, which
// k_trace found once per ray, so the depth-0 extend is skipped.
RT_HD void raygen_rays_body(uint32_t slot, const RenderParams& rp, const Wave& w, const float4* rays, const float4* first_hits, uint32_t key_base) {
    const uint32_t r = w.pixel_list[w.pixel_base + slot % w.n_pixels];
    const uint32_t sidx = w.sample_base + slot / w.n_pixels, k = key_base + r;
    Sampler s;
    s.init(rp.sampler);
    s.start_sample(k & 0xffffu, k >> 16, sidx);
    w.radiance[slot] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    RngState rs;
    rs.state = s.rng.state; rs.inc = s.rng.inc;
    w.state[slot].rng = rs;
    w.state[slot].weight = make_float4(1.0f, 1.0f, 1.0f, u2f(1u | (s.dimension << 8)));
    const float4 o4 = rays[2 * (size_t)r], d4 = rays[2 * (size_t)r + 1];
    w.ray_o_out[slot] = make_float4(o4.x, o4.y, o4.z, d4.w);
    w.ray_d_out[slot] = make_float4(d4.x, d4.y, d4.z, u2f(slot));
    w.hits[slot] = first_hits[r];
}

}  // namespace rt
