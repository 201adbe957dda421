// rt_integrator.h — per-thread bodies of the wavefront kernels: raygen, shade (material + NEE + BSDF
// sampling), shadow, resolve, and the first-hit AOV pass.
//
// Replaces camera_ray / generate_ray / ray_radiance / first_hit_aovs / render_aovs / render_tile
// (crates/raytracing-cpu/src/lib.rs:145-625), intersect_shape / ray_mesh_intersect hit-record construction
// (geometry.rs:92-136, 229-298), sample_light / light_radiance / environment_light_radiance / occluded
// (lights.rs:14-168) and MaterialEvalContext (materials.rs:702-809).
//
// The reference walks one path to completion per loop iteration; here a path is a slot of SoA state that
// moves through raygen -> [extend -> shade -> shadow]* one bounce per launch. All paths of a batch are
// at the same depth, so t_min / t_max and the "add emitted / add direct" predicates are launch constants.
#pragma once
#include "rt_bsdf.h"
#include "rt_traverse.h"

namespace rt {

struct RenderParams {  // RaytracerSettings (renderer/mod.rs:84-98)
    uint32_t max_ray_depth, accumulate_bounces, light_sample_count, samples_per_pixel;
    uint32_t antialias_primary_rays;
    SamplerParams sampler;
};

struct alignas(16) RngState { uint64_t state, inc; };
// Per-slot path state that shade reads and writes back together, interleaved (32 B = one DRAM sector): at depth >= 1 only a
// fraction of the slots is alive, so slot-indexed accesses are scattered and two separate 16-byte arrays cost two half-used
// sectors each way. The accumulated radiance stays a dense array of its own (resolve streams it; shadow_gather updates it).
struct alignas(32) PathState {
    float4 weight;     // xyz path weight | w: bit0 specular_bounce, bits 8.. stratified dimension
    RngState rng;      // PCG32 state + inc (inc is a pure function of (x, y, sample); carried so that shade needs no pixel lookup)
};

// Wavefront state of one batch (all pointers device memory; DESIGN.md "Path state").
struct Wave {
    // batch shape: slot = s_local * n_pixels + p_local
    const uint32_t* pixel_list;  // packed (y << 16 | x) of the pixels this context renders, coherent order
    uint32_t pixel_base, n_pixels, sample_base, n_samples;
    uint32_t capacity;           // slots allocated (>= n_pixels * n_samples)
    uint32_t depth;              // bounce index of the rays in the current queue
    PathState* state;            // weight + rng, by slot
    float4* radiance;            // xyz accumulated radiance of this sample, by slot
    // ray queue (compacted), by queue position
    const float4* ray_o_in;      // origin.xyz | t_max
    const float4* ray_d_in;      // direction.xyz | slot
    float4* ray_o_out;
    float4* ray_d_out;
    float4* hits;                // t | prim | u | v
    const uint32_t* n_in;        // rays in the current queue (device counter of this depth)
    uint32_t* n_out;             // rays pushed for the next bounce
    unsigned long long* n_shadow;  // this depth's NEE counter: low 32 bits = vertices with shadow rays, high 32 = shadow rays
    unsigned long long* stats;   // STAT_* counters (rays per class, BVH fetches)
    // next-event estimation: a compacted queue of shadow rays (one entry per light sample with a non-zero unoccluded
    // contribution; the rays of a vertex are consecutive) and a queue of the vertices they belong to
    uint32_t shadow_k;           // light samples per vertex = sum over lights of their sample counts
    float4* sray_o;              // light-side origin.xyz | t_max (distance - 0.001; negative: never occluded, not traced)
    float4* sray_d;              // unit direction light -> shading point
    float4* scontrib;            // weighted contribution.xyz if unoccluded; zeroed by k_shadow when the ray is blocked
    uint4* svertex;              // slot | first ray | ray count | -
    // material split (scenes that mix Diffuse with other materials): queue positions of the vertices the Diffuse shade kernel
    // met with another material and left for the general kernel, and their count at this depth
    uint32_t* deferred;
    uint32_t* n_deferred;
};

enum { STAT_PRIMARY = 0, STAT_BOUNCE = 1, STAT_SHADOW = 2, STAT_AOV = 3, STAT_EXT_NODES = 4, STAT_EXT_PRIMS = 5, STAT_SH_NODES = 6,
       STAT_SH_PRIMS = 7, STAT_AOV_NODES = 8, STAT_AOV_PRIMS = 9, STAT_SHADED = 10, STAT_NONFINITE = 11, STAT_CULLED = 12, STAT_FINAL_SKIPPED = 13, STAT_TOTAL = 16 };

struct Ray { V3 o, d; };

struct RayDiff { V3 x_origin, y_origin, x_direction, y_direction; };

// lib.rs:145-195
RT_HD_CALL Ray camera_ray(const CameraD& cam, float x, float y, bool has_lens, V2 lens) {
    V3 raster = mk3(x, y, 0.0f);
    Ray r;
    V3 cp = apply_point(cam.raster_to_camera, raster);
    if (cam.kind == 0) {
        r.o = apply_point(cam.camera_to_world, cp);
        r.d = unit(apply_vector(cam.camera_to_world, mk3(0, 0, 1)));
        return r;
    }
    if (cam.kind == 1) {
        r.o = apply_point(cam.camera_to_world, mk3(0, 0, 0));
        r.d = unit(apply_vector(cam.camera_to_world, unit(cp)));
        return r;
    }
    float t = cam.focal_distance / cp.z;
    V3 focus = cp * t;
    V3 co = mk3(0, 0, 0), cd;
    if (has_lens) {
        co = mk3(lens.x * cam.aperture_radius, lens.y * cam.aperture_radius, 0.0f);
        cd = unit(focus - co);
    } else cd = unit(cp);
    r.o = apply_point(cam.camera_to_world, co);
    r.d = unit(apply_vector(cam.camera_to_world, cd));
    return r;
}

// lib.rs:198-245
template <bool WITH_DIFF>
RT_HD void generate_ray(const CameraD& cam, uint32_t px, uint32_t py, Sampler& s, uint32_t spp, bool jitter, Ray& ray, RayDiff& rd) {
    float x, y;
    if (jitter) { V2 d = s.uniform2(); x = (float)px + d.x; y = (float)py + d.y; }
    else { x = (float)px + 0.5f; y = (float)py + 0.5f; }
    bool has_lens = cam.kind == 2;
    V2 lens = mk2(0, 0);
    if (has_lens) lens = sample_unit_disk_concentric(s.uniform2());
    ray = camera_ray(cam, x, y, has_lens, lens);
    if (WITH_DIFF) {
        Ray rx = camera_ray(cam, x + 1.0f, y, has_lens, lens);
        Ray ry = camera_ray(cam, x, y + 1.0f, has_lens, lens);
        float scale = fmaxf(0.125f, sqrtf(1.0f / (float)spp));
        V3 sx = ray.d + (rx.d - ray.d) * scale;
        V3 sy = ray.d + (ry.d - ray.d) * scale;
        rd.x_origin = rx.o - ray.o;
        rd.y_origin = ry.o - ray.o;
        rd.x_direction = unit(sx) - ray.d;
        rd.y_direction = unit(sy) - ray.d;
    }
}

struct HitInfo {  // accel.rs:13-25 (+ ids for the debug planes)
    float t;
    V2 uv;
    V3 point, normal, dpdu, dpdv;
    uint32_t material, light, geom_id, prim_id;
};

// intersect_shape + ray_mesh_intersect / ray_sphere_intersect + the identity local_to_root step of
// traverse_bvh (accel.rs:144-164), from the (t, prim, u, v) record the traversal kernel wrote.
RT_HD void reconstruct_hit(const SceneD& sc, V3 o, V3 d, const Hit& h, bool need_derivs, HitInfo& out) {
    if (!need_derivs && sc.shade_recs) {   // the gathered record (rt_scene.h ShadeRec): same values, two load levels instead of five
        const ShadeRec* r = sc.shade_recs + h.prim;
        const float4 a = ldg(&r->n0_geom), b = ldg(&r->n1_prim), c = ldg(&r->n2_flags);
        const uint32_t flags = f2u(c.w);
        if (!(flags & REC_SPHERE)) {
            const uint32_t geom = f2u(a.w);
            const Instance& inst = sc.instances[geom];
            // the instance's inverse rows and its (shape, kind, material, light) quad as four 128-bit loads
            float4 w0, w1, w2;
            load_rows3(inst.w2o, w0, w1, w2);
            const uint4 ids = load_u4(&inst.shape);
            out.t = h.t;
            out.geom_id = geom;
            out.prim_id = f2u(b.w);
            out.material = ids.z;     // (the record's copies are the instance's values: one scattered load less for
            out.light = ids.w;        //  meshes without uvs, whose fourth and fifth record words are never read)
            const float u = h.u, v = h.v, w = 1.0f - u - v;
            const V3 n_obj = (flags & REC_FLAT) ? xyz(a) : unit(w * xyz(a) + u * xyz(b) + v * xyz(c));
            V2 uv0 = mk2(0, 0), uv1 = mk2(1, 0), uv2 = mk2(0, 1);
            if (flags & REC_UV) {
                const float4 q = ldg(&r->uv01), e = ldg(&r->uv2_mat);
                uv0 = mk2(q.x, q.y); uv1 = mk2(q.z, q.w); uv2 = mk2(e.x, e.y);
            }
            out.uv = w * uv0 + u * uv1 + v * uv2;
            out.point = o + d * h.t;
            out.normal = unit(unit(mk3(w0.x * n_obj.x + w1.x * n_obj.y + w2.x * n_obj.z, w0.y * n_obj.x + w1.y * n_obj.y + w2.y * n_obj.z,
                                       w0.z * n_obj.x + w1.z * n_obj.y + w2.z * n_obj.z)));   // apply_vector_transposed(inst.w2o, n_obj)
            // dpdu / dpdv = o2w * 0: only the anti-aliased primary hit reads them, and that hit takes the long way below
            out.dpdu = mk3(0.0f);
            out.dpdv = mk3(0.0f);
            return;
        }
    }
    const Prim* pr = sc.prims + h.prim;
    const uint32_t geom = f2u(ldg(&pr->a).w), prim_id = f2u(ldg(&pr->b).w), kind = f2u(ldg(&pr->c).w);
    const Instance& inst = sc.instances[geom];
    out.t = h.t;
    out.geom_id = geom;
    out.prim_id = prim_id;
    out.material = inst.material;
    out.light = inst.area_light;
    V3 n_obj, dpdu = mk3(0.0f), dpdv = mk3(0.0f);
    if (kind == 0) {
        const uint32_t* t = sc.tris + 3 * (size_t)(inst.tri_offset + prim_id);
        const uint32_t i0 = ldg(t), i1 = ldg(t + 1), i2 = ldg(t + 2);
        const float u = h.u, v = h.v, w = 1.0f - u - v;
        V3 p0 = mk3(0.0f), p1 = mk3(0.0f), p2 = mk3(0.0f);
        const bool has_n = inst.normal_offset != NONE;
        if (!has_n || need_derivs) {
            p0 = load3(sc.vertices, inst.vertex_offset + i0);
            p1 = load3(sc.vertices, inst.vertex_offset + i1);
            p2 = load3(sc.vertices, inst.vertex_offset + i2);
        }
        if (!has_n) n_obj = unit(cross(p2 - p0, p1 - p0));
        else n_obj = unit(w * load3(sc.normals, inst.normal_offset + i0) + u * load3(sc.normals, inst.normal_offset + i1) +
                          v * load3(sc.normals, inst.normal_offset + i2));
        V2 uv0 = mk2(0, 0), uv1 = mk2(1, 0), uv2 = mk2(0, 1);
        if (inst.uv_offset != NONE) {
            uv0 = load2(sc.uvs, inst.uv_offset + i0);
            uv1 = load2(sc.uvs, inst.uv_offset + i1);
            uv2 = load2(sc.uvs, inst.uv_offset + i2);
        }
        out.uv = w * uv0 + u * uv1 + v * uv2;
        if (need_derivs) {
            V2 duv02 = uv0 - uv2, duv12 = uv1 - uv2;
            V3 dp02 = p0 - p2, dp12 = p1 - p2;
            float det = duv02.x * duv12.y - duv02.y * duv12.x;
            if (!(fabsf(det) < 1.0e-9f)) {
                float inv_det = 1.0f / det;
                dpdu = inv_det * (duv12.y * dp02 - duv02.y * dp12);
                dpdv = inv_det * (duv02.x * dp12 - duv12.x * dp02);
            }
        }
        out.point = o + d * h.t;
    } else {
        V3 center = mk3(inst.center[0], inst.center[1], inst.center[2]);
        float radius = inst.radius;
        V3 oo = apply_point(inst.w2o, o), od = apply_vector(inst.w2o, d);
        V3 point = oo + od * h.t;
        V3 local = point - center;
        float theta = acosf(local.z / radius);
        float sin_theta = sinf(theta);
        float cos_phi = local.x / (radius * sin_theta);
        float sin_phi = local.y / (radius * sin_theta);
        float phi = local.y > 0.0f ? acosf(cos_phi) : 2.0f * PI - acosf(cos_phi);
        out.uv = mk2(phi / (2.0f * PI), theta / PI);
        dpdu = mk3(-2.0f * PI * local.y, 2.0f * PI * local.x, 0.0f);
        dpdv = PI * mk3(local.z * cos_phi, local.z * sin_phi, -radius * sin_theta);
        n_obj = local / radius;
        out.point = apply_point(inst.o2w, point);
    }
    // Transform::apply_normal = inverse^T (transform.rs:68-73); re-unit twice as the reference does
    // (geometry.rs:127 and accel.rs:152)
    out.normal = unit(unit(apply_vector_transposed(inst.w2o, n_obj)));
    out.dpdu = apply_vector(inst.o2w, dpdu);
    out.dpdv = apply_vector(inst.o2w, dpdv);
}

// materials.rs:715-796
RT_HD MatCtx matctx_from_differentials(const HitInfo& hit, const Ray& ray, const RayDiff& rd) {
    V3 n = hit.normal, p = hit.point;
    V3 rx_o = ray.o + rd.x_origin, rx_d = ray.d + rd.x_direction;
    V3 ry_o = ray.o + rd.y_origin, ry_d = ray.d + rd.y_direction;
    float dd = -dot(n, p);
    float tx = -(dot(n, rx_o) + dd) / dot(n, rx_d);
    float ty = -(dot(n, ry_o) + dd) / dot(n, ry_d);
    V3 px = rx_o + tx * rx_d, py = ry_o + ty * ry_d;
    V3 dpdx = px - hit.point, dpdy = py - hit.point;
    V3 dpdu = hit.dpdu, dpdv = hit.dpdv;
    float ata00 = dot(dpdu, dpdu), ata11 = dot(dpdv, dpdv), ata01 = dot(dpdu, dpdv);
    float det = ata00 * ata11 - ata01 * ata01;
    float inv_det = 1.0f / det;
    float atb0x = dot(dpdu, dpdx), atb1x = dot(dpdv, dpdx), atb0y = dot(dpdu, dpdy), atb1y = dot(dpdv, dpdy);
    float dudx = inv_det * (ata11 * atb0x - ata01 * atb1x);
    float dvdx = inv_det * (ata00 * atb1x - ata01 * atb0x);
    float dudy = inv_det * (ata11 * atb0y - ata01 * atb1y);
    float dvdy = inv_det * (ata00 * atb1y - ata01 * atb0y);
    MatCtx c;
    c.uv = hit.uv;
    c.dudx = finite_f(dudx) ? rs_clamp(dudx, -1.0e8f, 1.0e8f) : 0.0f;
    c.dudy = finite_f(dudy) ? rs_clamp(dudy, -1.0e8f, 1.0e8f) : 0.0f;
    c.dvdx = finite_f(dvdx) ? rs_clamp(dvdx, -1.0e8f, 1.0e8f) : 0.0f;
    c.dvdy = finite_f(dvdy) ? rs_clamp(dvdy, -1.0e8f, 1.0e8f) : 0.0f;
    return c;
}

struct LightSample { V3 radiance; V3 origin; V3 dir; float distance, pdf; };

// lights.rs:14-122 (quirks kept: object-space triangle area and normal, un-normalised dir_world in the cosine)
// `em_tri_count` / `em_has_normals`: the two fields of the emitter's shape record an area light needs (callers read them from
// SceneD::shapes, or from the kernel-parameter copy for light 0).
RT_HD LightSample sample_light(const SceneD& sc, const LightD& l, uint32_t em_tri_count, bool em_has_normals, V3 point, Sampler& s) {
    LightSample ls;
    V3 a = mk3(l.a[0], l.a[1], l.a[2]), b = mk3(l.b[0], l.b[1], l.b[2]);
    if (l.kind == 0) {
        V3 dir = point - a;
        float d = length(dir), d2 = d * d;
        ls.radiance = b / d2; ls.origin = a; ls.dir = dir / d; ls.distance = d; ls.pdf = 1.0f;
        return ls;
    }
    if (l.kind == 1) {
        float diam = sc.scene_radius * 2.0f;
        ls.radiance = b; ls.origin = point - a * diam; ls.dir = unit(a); ls.distance = diam; ls.pdf = 1.0f;
        return ls;
    }
    float pdf = 1.0f;
    pdf /= (float)em_tri_count;
    uint32_t tri = s.u32_range(0, em_tri_count);
    V2 smp = s.uniform2();
    V3 bary;
    if (smp.x < smp.y) { float b0 = smp.x / 2.0f, b1 = smp.y - smp.x / 2.0f; bary = mk3(b0, b1, 1.0f - b0 - b1); }
    else { float b0 = smp.x - smp.y / 2.0f, b1 = smp.y / 2.0f; bary = mk3(b0, b1, 1.0f - b0 - b1); }
    const LightTri* lt = sc.light_tris + (l.tri_table + tri);
    const float4 r0 = ldg(&lt->p0_area), r1 = ldg(&lt->p1_nx), r2 = ldg(&lt->p2_ny);
    const V3 p0 = xyz(r0), p1 = xyz(r1), p2 = xyz(r2);
    pdf /= r0.w;  // Mesh::tri_area, mesh.rs:271-278
    V3 p_local = bary.x * p0 + bary.y * p1 + bary.z * p2;
    V3 p_world = apply_point(l.light_to_world, p_local);
    V3 dir_world = point - p_world;
    float d = length(dir_world);
    V3 n;
    if (!em_has_normals) n = mk3(r1.w, r2.w, ldg(&lt->nz).x);
    else n = unit(bary.x * xyz(ldg(&lt->n0)) + bary.y * xyz(ldg(&lt->n1)) + bary.z * xyz(ldg(&lt->n2)));   // the table's copies of the vertex normals
    ls.radiance = dot(dir_world, n) < 0.0f ? mk3(0.0f) : b;
    pdf *= (d * d) / fabsf(dot(dir_world, n));
    ls.origin = p_world; ls.dir = dir_world / d; ls.distance = d; ls.pdf = pdf;
    return ls;
}

RT_HD_CALL V3 environment_radiance(const SceneD& sc, V3 direction) {  // lights.rs:137-157
    direction = unit(direction);
    float t = acosf(direction.z) * FRAC_1_PI;
    float s = (atan2f(direction.x, direction.y) + PI) * FRAC_1_PI * 0.5f;
    return xyz(tex(sc, sc.env_texture, matctx_no_aa(mk2(s, t))));
}

RT_HD void slot_to_sample(const Wave& w, uint32_t slot, uint32_t& px, uint32_t& py, uint32_t& sidx) {
    uint32_t p_local = slot % w.n_pixels;
    uint32_t packed = ldg(w.pixel_list + w.pixel_base + p_local);
    px = packed & 0xffffu;
    py = packed >> 16;
    sidx = w.sample_base + slot / w.n_pixels;
}

// ---- raygen: CpuSampler::start_sample + generate_ray(jitter = true) (lib.rs:527-536) -----------------
// Slab test of a camera ray against the scene bounds (SceneD::bounds_lo/hi, already grown by a margin far above the rounding
// of this test): the reference rejects such rays at the BVH root (accel.rs:95) and, without an environment light, their
// sample is black. t >= 0 only (near_clip >= 0): a box behind the camera cannot be hit either.
RT_HD bool ray_misses_scene(const SceneD& sc, V3 o, V3 d) {
    float t0 = 0.0f, t1 = RT_INF;
    const float oo[3] = {o.x, o.y, o.z}, dd[3] = {d.x, d.y, d.z};
    for (int k = 0; k < 3; k++) {
        const float a = fabsf(dd[k]) > 1.0e-20f ? dd[k] : copysignf(1.0e-20f, dd[k]);
        const float inv = 1.0f / a;
        const float ta = (sc.bounds_lo[k] - oo[k]) * inv, tb = (sc.bounds_hi[k] - oo[k]) * inv;
        t0 = fmaxf(t0, fminf(ta, tb));
        t1 = fminf(t1, fmaxf(ta, tb));
    }
    return !(t0 <= t1);
}

// Initialises the slot's path state and returns the camera ray; false when no ray needs to be traced for this sample
// (it misses the scene bounds and there is no environment light: its radiance stays 0, the slot is never read again).
RT_HD bool raygen_body(uint32_t slot, const SceneD& sc, const RenderParams& rp, const Wave& w, float4& ray_o, float4& ray_d) {
    uint32_t px, py, sidx;
    slot_to_sample(w, slot, px, py, sidx);
    Sampler s;
    s.init(rp.sampler);
    s.start_sample(px, py, sidx);
    Ray ray;
    RayDiff rd;
    generate_ray<false>(sc.camera, px, py, s, rp.samples_per_pixel, true, ray, rd);
    w.radiance[slot] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (sc.env_texture == NONE && ray_misses_scene(sc, ray.o, ray.d)) return false;
    RngState rs;
    rs.state = s.rng.state; rs.inc = s.rng.inc;
    w.state[slot].rng = rs;
    w.state[slot].weight = make_float4(1.0f, 1.0f, 1.0f, u2f(1u | (s.dimension << 8)));
    ray_o = make_float4(ray.o.x, ray.o.y, ray.o.z, sc.camera.far_clip);
    ray_d = make_float4(ray.d.x, ray.d.y, ray.d.z, u2f(slot));
    return true;
}

// ---- shade: one iteration of the ray_radiance loop after traverse_bvh (lib.rs:284-391) ------------------
// A vertex can emit three kinds of output: a continuation ray, up to K shadow rays, and one NEE vertex record.
// Their queue positions come from `alloc`, which every thread of the launch calls exactly once per queue chunk
// (on the device it is a warp scan + two global atomics per warp, kernels.cu; the CPU harness hands out running
// counters). The shadow-ray count has to be known before the positions: with up to NEE_STAGE light samples per vertex
// the entries are evaluated once and staged in thread-local memory until `alloc` returns (nee_pass<1>); with more, a
// counting pass and a writing pass draw the same numbers from the same sampler state (nee_pass<0>, nee_pass<2>).
template <typename Surf>
struct ShadeState {
    uint32_t slot, flags, sidx;
    Ray ray;
    V3 emitted, path_weight;   // emitted: radiance of the emitter hit after a specular bounce / at depth 0 (added when `dirty`)
    Sampler s;
    HitInfo hit;
    Surf surf;
    Frame fr;
    V3 wo;
    bool dirty;
};

// radiance += path_weight * emitted (lib.rs:289, 296): the only read-modify-write of the slot's radiance in shade
template <typename Surf>
RT_HD void add_emitted(const Wave& w, const ShadeState<Surf>& S) {
    V3 r = xyz(w.radiance[S.slot]);
    r += S.path_weight * S.emitted;
    w.radiance[S.slot] = make_float4(r.x, r.y, r.z, 0.0f);
}

// lib.rs:284-322: miss / emission / material setup. False when the path ends here (state already written back).
// DEFER_OTHERS (the Diffuse kernel of a scene with mixed materials): a vertex whose material is not Diffuse is left untouched for
// the general kernel (`deferred` set, nothing read-modified-written yet).
template <typename Surf, bool DEFER_OTHERS = false>
RT_HD bool shade_begin(uint32_t q, const SceneD& sc, const RenderParams& rp, const Wave& w, ShadeState<Surf>& S, bool& deferred) {
    const float4 ro4 = ld_stream(&w.ray_o_in[q]), rd4 = ld_stream(&w.ray_d_in[q]), h4 = ld_stream(&w.hits[q]);
    const uint32_t slot = f2u(rd4.w);
    S.slot = slot;
    S.ray.o = xyz(ro4);
    S.ray.d = xyz(rd4);
    Hit h;
    h.t = h4.x; h.prim = f2u(h4.y); h.u = h4.z; h.v = h4.w;
    const uint32_t depth = w.depth;
    const bool has_hit = h.prim != NONE;
    if (!has_hit && sc.env_texture == NONE) return false;

    // The slot's accumulated radiance is only touched by the few vertices that add to it here (an emitter seen directly or
    // through specular bounces, the environment on a miss): reading it for every vertex cost a scattered 32-byte sector each.
    const float4 wt4 = w.state[slot].weight;
    S.path_weight = xyz(wt4);
    S.flags = f2u(wt4.w);
    S.dirty = false;
    S.emitted = mk3(0.0f);
    if (!has_hit) {
        S.emitted = environment_radiance(sc, S.ray.d);
        add_emitted(w, S);
        return false;
    }
    const bool specular_bounce = (S.flags & 1u) != 0;
    const RngState rs = w.state[slot].rng;
    S.sidx = w.sample_base + slot / w.n_pixels;
    S.s.init(rp.sampler);
    S.s.rng.state = rs.state;
    S.s.rng.inc = rs.inc;
    S.s.dimension = S.flags >> 8;
    S.s.sample_index = S.sidx;

    const bool aa = depth == 0 && rp.antialias_primary_rays && sc.tex_uses_derivs;
    reconstruct_hit(sc, S.ray.o, S.ray.d, h, aa, S.hit);
    if (DEFER_OTHERS && ldg(sc.mat_const + S.hit.material).w == 0.0f) { deferred = true; return false; }

    const bool add_zero_bounce = rp.accumulate_bounces || rp.max_ray_depth == depth;
    if (specular_bounce && add_zero_bounce && S.hit.light != NONE) {
        const LightD& l = sc.lights[S.hit.light];
        if (l.kind == 2) { S.emitted = mk3(l.b[0], l.b[1], l.b[2]); S.dirty = true; }
    }

    MatCtx mc;
    if (aa) {
        // the camera-ray differentials are a pure function of (pixel, sample): re-derive them from a fresh
        // stream instead of carrying 48 bytes per path (lib.rs:206-243)
        uint32_t px, py, sidx;
        slot_to_sample(w, slot, px, py, sidx);
        Sampler s0;
        s0.init(rp.sampler);
        s0.start_sample(px, py, sidx);
        Ray cam_ray;
        RayDiff rdiff;
        generate_ray<true>(sc.camera, px, py, s0, rp.samples_per_pixel, true, cam_ray, rdiff);
        mc = matctx_from_differentials(S.hit, S.ray, rdiff);
    } else mc = matctx_no_aa(S.hit.uv);

    get_surface_of(sc, S.hit.material, mc, S.surf);
    S.fr.n = S.hit.normal;
    make_orthonormal_basis(S.hit.normal, S.fr.x, S.fr.y);
    S.wo = S.fr.to_local(-S.ray.d);

    if (depth + 1 > rp.max_ray_depth) {
        if (S.dirty) add_emitted(w, S);
        return false;
    }
    return true;
}

// lib.rs:324-356: every light, every sample; entries with a non-zero unoccluded contribution become shadow rays.
// MODE 0 counts them, MODE 1 stages up to NEE_STAGE of them in thread-local memory (and counts), MODE 2 writes them
// (at most `limit`) to the shadow-ray queue starting at `first`. All modes draw the same numbers from `s`.
#ifndef RT_NEE_STAGE
#define RT_NEE_STAGE 8
#endif
constexpr uint32_t NEE_STAGE = RT_NEE_STAGE;
struct NeeStage { float4 e[3 * NEE_STAGE]; };   // entry k: origin | t_max, direction, contribution at e[3k .. 3k+2]
// Where nee_pass<1> parks the entries: field f of entry k lives at p[(3k + f) * stride]. The kernels hand every thread a
// column of a SHARED-memory array (stride = block size, up to NEE_SMEM entries: the default 4 light samples of one area
// light); thread-local memory (stride 1) serves larger counts and the CPU harness. Staged entries in thread-local memory
// were 40 % of k_shade's local-memory sectors, and local memory was most of what the kernel wrote to DRAM (ncu, round 2:
// 10.1 GB written against 6.5 GB of queue / state stores in the depth-0 launch of a 34 M-vertex batch).
#ifndef RT_NEE_SMEM
#define RT_NEE_SMEM 4
#endif
constexpr uint32_t NEE_SMEM = RT_NEE_SMEM;
struct StagePtr { float4* p; uint32_t stride, capacity; };

template <int MODE, typename Surf>
RT_HD uint32_t nee_pass(const SceneD& sc, const RenderParams& rp, const Wave& w, const ShadeState<Surf>& S, Sampler& s, uint32_t first, uint32_t limit,
                        StagePtr stage) {
    uint32_t k = 0;
    // one light at a time; `first_only` runs the body for light 0 from the kernel-parameter copy (SceneD::light0), whose
    // fields are then constant-bank operands; the remaining lights come from memory
    auto one_light = [&](const LightD& light, uint32_t em_tri_count, bool em_has_normals) {
        const uint32_t n = light.kind == 2 ? rp.light_sample_count : 1u;
        const float inv_n = 1.0f / (float)n;
        for (uint32_t j = 0; j < n; j++) {
            LightSample ls = sample_light(sc, light, em_tri_count, em_has_normals, S.hit.point, s);
            V3 wi = S.fr.to_local(-ls.dir);
            // contribution if unoccluded (lib.rs:337-343); zero contributions never need a shadow ray
            V3 c = mk3(0.0f);
            float cosv = fmaxf(0.0f, wi.z);
            if (!(is_zero(ls.radiance) || cosv == 0.0f) || !(ls.pdf > 0.0f)) {
                V3 bv = surface_eval(S.surf, S.wo, wi);
                c = S.path_weight * ((bv * ls.radiance * cosv / ls.pdf) * inv_n);
            }
            if (!is_zero(c)) {
                if (MODE != 0 && k < limit) {
                    // a non-finite origin (directional light with an infinite scene radius: single-primitive
                    // scenes, bvh2.rs:448-452) can never be occluded in the reference: NaN slab test
                    const bool skip_test = !(finite_f(ls.origin.x) && finite_f(ls.origin.y) && finite_f(ls.origin.z));
                    const float4 eo = make_float4(ls.origin.x, ls.origin.y, ls.origin.z, skip_test ? -1.0f : ls.distance - 0.001f);
                    const float4 ed = make_float4(ls.dir.x, ls.dir.y, ls.dir.z, 0.0f), ec = make_float4(c.x, c.y, c.z, 0.0f);
                    if (MODE == 1) { float4* e = stage.p + (size_t)(3u * k) * stage.stride; e[0] = eo; e[stage.stride] = ed; e[2u * stage.stride] = ec; }
                    else { const size_t e = (size_t)first + k; RT_CHECK(e < (size_t)w.capacity * (w.shadow_k ? w.shadow_k : 1u)); w.sray_o[e] = eo; w.sray_d[e] = ed; w.scontrib[e] = ec; }
                }
                k++;
            }
        }
    };
    uint32_t li = 0;
    if (sc.use_light0 && sc.light_count) { one_light(sc.light0, sc.light0_tri_count, sc.light0_has_normals != 0u); li = 1; }
    for (; li < sc.light_count; li++) {
        const LightD& light = sc.lights[li];
        uint32_t tc = 0; bool hn = false;
        if (light.kind == 2) { const ShapeD& em = sc.shapes[light.shape]; tc = em.tri_count; hn = em.normal_offset != NONE; }
        one_light(light, tc, hn);
    }
    if (MODE == 2)   // the passes are the same arithmetic; should a compiler ever make them disagree, stay in bounds
        for (; k < limit; k++) {
            const size_t e = (size_t)first + k;
            w.sray_o[e] = make_float4(0.0f, 0.0f, 0.0f, -1.0f);
            w.sray_d[e] = make_float4(0.0f, 0.0f, 1.0f, 0.0f);
            w.scontrib[e] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
    return k;
}

// alloc(continue_path, has_nee_vertex, n_shadow_rays, final_ray_skipped, &ray_pos, &vertex_pos, &first_shadow_ray)
// The kernel splits the allocation in three so that the two global atomics of a warp are in flight while it still has work:
//   early(has_nee_vertex, n_shadow_rays)   right after next-event estimation: the shadow-queue atomic is issued here and
//                                          returns during BSDF sampling;
//   alloc(...)                             as above, but it may leave ray_pos unset ...
//   late(&ray_pos)                         ... until after the shadow entries have been copied out.
// All three are warp-collective: every thread of the launch calls each of them exactly once per chunk. The CPU harness passes
// `alloc` only.
// SHARED_STAGE_ONLY: the caller guarantees that every vertex's entries fit the shared-memory column it passes (the kernel is
// instantiated that way for launches with shadow_k <= NEE_SMEM): no thread-local staging array exists in that instantiation, and
// the staging accesses are shared-memory instructions instead of generic ones.
// DEFER_OTHERS: see shade_begin; `defer(q)` receives the queue positions left for the general kernel.
template <typename Surf, bool SHARED_STAGE_ONLY = false, bool DEFER_OTHERS = false, typename Alloc, typename Early, typename Late, typename Defer>
RT_HD void shade_vertex(bool active, uint32_t q, const SceneD& sc, const RenderParams& rp, const Wave& w, Alloc&& alloc, StagePtr shared_stage, Early&& early,
                        Late&& late, Defer&& defer) {
    ShadeState<Surf> S;
    Sampler s2;
    BsdfSample bs;
    typename std::conditional<SHARED_STAGE_ONLY, char, NeeStage>::type local_stage;
    uint32_t k = 0;
    bool alive = false, final_skipped = false;
    V3 nd = mk3(0.0f);
    // few light samples per vertex (the usual case): one evaluation, entries staged (shared memory when the kernel offers a
    // column that holds them, else thread-local memory) until their queue position is known; otherwise count first and
    // evaluate again when writing
    const bool staged = SHARED_STAGE_ONLY || w.shadow_k <= NEE_STAGE;
    StagePtr stage = shared_stage;
    if constexpr (!SHARED_STAGE_ONLY) {
        if (!(shared_stage.p && w.shadow_k <= shared_stage.capacity)) stage = StagePtr{local_stage.e, 1u, NEE_STAGE};
    } else (void)local_stage;
    if (active) {
        bool deferred = false;
        active = shade_begin<Surf, DEFER_OTHERS>(q, sc, rp, w, S, deferred);
        if (DEFER_OTHERS && deferred) defer(q);
    }
    if (active) {
        s2 = S.s;
        const bool add_direct = rp.accumulate_bounces || rp.max_ray_depth == w.depth + 1;
        const bool nee = !surface_is_delta(S.surf) && add_direct;
        if (nee) k = staged ? nee_pass<1>(sc, rp, w, S, s2, 0u, NEE_STAGE, stage) : nee_pass<0>(sc, rp, w, S, s2, 0u, 0u, stage);
    }
    early(k != 0u, k);
    if (active) {
        alive = surface_sample(S.surf, S.wo, s2, bs) == S_VALID;
        if (alive && (is_zero(bs.f) || bs.pdf == 0.0f)) alive = false;
        // The ray of the last depth can only add emitted light after a specular bounce, or the environment on a miss
        // (lib.rs:294-298, 318-322: the loop ends right after that hit's emission): after a non-specular sample in a scene
        // without environment light the reference traces it for nothing, and it is not traced here.
        if (alive && w.depth + 1 == rp.max_ray_depth && sc.env_texture == NONE && !(bs.component & SPECULAR)) {
            alive = false;
            final_skipped = true;
        }
        // Everything that does not need a queue position happens BEFORE the allocation (a warp-wide scan plus two global
        // atomics whose return the warp waits for): the emitted light, the path state of the continuation, and the new
        // direction. What stays live across the wait is the hit point, the direction and three counters — the frame, the
        // BSDF sample, the weights and the sampler state used to be carried across it through thread-local memory, and the
        // reloads behind the wait were 17 % of the kernel's stall samples (ncu, profiles/r4e).
        if (S.dirty) add_emitted(w, S);
        if (alive) {
            const V3 pw = S.path_weight * (bs.f * fabsf(bs.wi.z) / bs.pdf);
            const uint32_t spec = (bs.component & SPECULAR) ? 1u : 0u;
            w.state[S.slot].weight = make_float4(pw.x, pw.y, pw.z, u2f(spec | (s2.dimension << 8)));
            RngState rs;
            rs.state = s2.rng.state; rs.inc = s2.rng.inc;
            w.state[S.slot].rng = rs;
            nd = S.fr.to_world(bs.wi);
        }
    }
    uint32_t rpos = 0, vpos = 0, first = 0;
    alloc(alive, k != 0u, k, final_skipped, rpos, vpos, first);
    if (active && k) {
        if (staged)
            for (uint32_t j = 0; j < k; j++) {
                const size_t e = (size_t)first + j;
                RT_CHECK(e < (size_t)w.capacity * (w.shadow_k ? w.shadow_k : 1u));
                const float4* se = stage.p + (size_t)(3u * j) * stage.stride;
                st_stream(&w.sray_o[e], se[0]); st_stream(&w.sray_d[e], se[stage.stride]); st_stream(&w.scontrib[e], se[2u * stage.stride]);
            }
        else nee_pass<2>(sc, rp, w, S, S.s, first, k, stage);
        RT_CHECK(vpos < w.capacity && S.slot < w.capacity);
        w.svertex[vpos] = make_uint4(S.slot, first, k, 0u);
    }
    late(rpos);
    if (!alive) return;
    RT_CHECK(rpos < w.capacity);
    st_stream(&w.ray_o_out[rpos], make_float4(S.hit.point.x, S.hit.point.y, S.hit.point.z, RT_INF));
    st_stream(&w.ray_d_out[rpos], make_float4(nd.x, nd.y, nd.z, u2f(S.slot)));
}

template <typename Surf, typename Alloc>
RT_HD void shade_vertex(bool active, uint32_t q, const SceneD& sc, const RenderParams& rp, const Wave& w, Alloc&& alloc, StagePtr shared_stage = StagePtr{nullptr, 0u, 0u}) {
    shade_vertex<Surf, false, false>(active, q, sc, rp, w, alloc, shared_stage, [](bool, uint32_t) {}, [](uint32_t&) {}, [](uint32_t) {});
}

// ---- shadow gather: add the unoccluded contributions of one NEE vertex to its path, in light-sample order ----
// (`occluded`, lights.rs:159-168, is the any-hit traversal in k_shadow, which zeroes the entries it finds blocked)
RT_HD void shadow_gather_body(uint32_t v, const Wave& w) {
    const uint4 rec = w.svertex[v];
    RT_CHECK(rec.x < w.capacity && (size_t)rec.y + rec.z <= (size_t)w.capacity * (w.shadow_k ? w.shadow_k : 1u));
    V3 sum = mk3(0.0f);
    for (uint32_t j = 0; j < rec.z; j++) sum += xyz(w.scontrib[(size_t)rec.y + j]);
    const float4 r = w.radiance[rec.x];
    w.radiance[rec.x] = make_float4(r.x + sum.x, r.y + sum.y, r.z + sum.z, 0.0f);
}

// ---- resolve: render_tile's per-pixel sample loop tail (lib.rs:538-548) — sum in sample order -----------
RT_HD void resolve_body(uint32_t p_local, const Wave& w, float4* accum) {
    float4 a = accum[w.pixel_base + p_local];
    for (uint32_t s = 0; s < w.n_samples; s++) {
        float4 r = w.radiance[(size_t)s * w.n_pixels + p_local];
        a.x += r.x; a.y += r.y; a.z += r.z;
    }
    accum[w.pixel_base + p_local] = a;
}

// ---- first-hit AOVs: render_aovs / first_hit_aovs (lib.rs:395-444, 556-625) ------------------------------
struct AovPlanes {  // device planes, row-major y*W+x; null = not requested
    float* normals; float* albedo; float* uv; float* mip_level; uint32_t* ids; float* depth;
};
struct FirstHit { bool hit; V2 uv; V3 normal, albedo; bool has_mip; float mip; uint32_t geom, prim; float t; };

// The traversal intersects world-space triangles (one transform per triangle at build time instead of one per ray and
// instance); the reference intersects in OBJECT space: the ray goes through the instance's inverse transform and
// Moller-Trumbore runs on the mesh's own vertices (intersect_shape, geometry.rs:92-136; t is shared between the spaces).
// Both are the same hit to rounding, but on small triangles the barycentrics differ in the 4th decimal (a 5 mm triangle
// seen from 4 m resolves its hit point to ~1e-6, i.e. ~2e-4 of its edge) — visible in the uv AOV of meshes without uvs, where
// uv IS the barycentrics. The first-hit AOV pass (one ray per pixel) therefore repeats the test of the WINNING triangle the
// reference's way and reports those (t, u, v): same operations in the same order, un-fused in this translation unit.
// [t_min, t_max] is the range the ray was traced over (the camera clip for first hits, the caller's range for ray queries).
RT_HD void refine_triangle_hit_in_object_space(const SceneD& sc, const Ray& ray, float t_min, float t_max, Hit& h) {
    const Prim* pr = sc.prims + h.prim;
    if (f2u(ldg(&pr->c).w) != 0u) return;   // spheres are intersected in object space already
    const uint32_t geom = f2u(ldg(&pr->a).w), prim_id = f2u(ldg(&pr->b).w);
    const Instance& inst = sc.instances[geom];
    const uint32_t* t3 = sc.tris + 3 * (size_t)(inst.tri_offset + prim_id);
    const V3 p0 = load3(sc.vertices, inst.vertex_offset + ldg(t3)), p1 = load3(sc.vertices, inst.vertex_offset + ldg(t3 + 1)),
             p2 = load3(sc.vertices, inst.vertex_offset + ldg(t3 + 2));
    const V3 oo = apply_point(inst.w2o, ray.o), od = apply_vector(inst.w2o, ray.d);
    float t, u, v;
    const bool ok = sc.watertight ? triangle_watertight(p0, p1, p2, oo, od, t_min, t_max, t, u, v)
                                  : triangle_t(p0, p1, p2, oo, od, t_min, t_max, t, u, v);
    if (ok) { h.t = t; h.u = u; h.v = v; }
}

template <bool STATS>
RT_HD FirstHit first_hit(const SceneD& sc, const RenderParams& rp, uint32_t px, uint32_t py, uint32_t sidx, TraverseStats* stats) {
    Sampler s;
    s.init(rp.sampler);
    s.start_sample(px, py, sidx);
    Ray ray;
    RayDiff rd;
    generate_ray<true>(sc.camera, px, py, s, rp.samples_per_pixel, false, ray, rd);
    FirstHit r;
    r.hit = false; r.uv = mk2(0, 0); r.normal = mk3(0.0f); r.albedo = mk3(0.0f); r.has_mip = false; r.mip = 0.0f;
    r.geom = NONE; r.prim = NONE; r.t = 0.0f;
    Hit h;
    if (!traverse<false, STATS>(sc, ray.o, ray.d, sc.camera.near_clip, sc.camera.far_clip, h, stats)) return r;
    refine_triangle_hit_in_object_space(sc, ray, sc.camera.near_clip, sc.camera.far_clip, h);
    HitInfo hit;
    reconstruct_hit(sc, ray.o, ray.d, h, true, hit);
    MatCtx mc = matctx_from_differentials(hit, ray, rd);
    const MaterialD& m = sc.materials[hit.material];
    r.hit = true;
    r.uv = hit.uv;
    r.normal = hit.normal;
    r.albedo = get_albedo(sc, m, mc);
    r.has_mip = get_mip_level(sc, m, mc, r.mip);
    r.geom = hit.geom_id;
    r.prim = hit.prim_id;
    r.t = hit.t;
    return r;
}

template <bool STATS>
RT_HD void aov_body(uint32_t i, const SceneD& sc, const RenderParams& rp, const uint32_t* pixel_list, const AovPlanes& pl, TraverseStats* stats) {
    uint32_t packed = pixel_list[i];
    uint32_t px = packed & 0xffffu, py = packed >> 16;
    FirstHit fh = first_hit<STATS>(sc, rp, px, py, 0u, stats);
    size_t idx = (size_t)py * sc.camera.width + px;
    if (pl.normals) { pl.normals[3 * idx] = fh.normal.x; pl.normals[3 * idx + 1] = fh.normal.y; pl.normals[3 * idx + 2] = fh.normal.z; }
    if (pl.albedo) { pl.albedo[3 * idx] = fh.albedo.x; pl.albedo[3 * idx + 1] = fh.albedo.y; pl.albedo[3 * idx + 2] = fh.albedo.z; }
    if (pl.uv) { pl.uv[2 * idx] = fh.uv.x; pl.uv[2 * idx + 1] = fh.uv.y; }
    if (pl.mip_level) pl.mip_level[idx] = fh.has_mip ? fh.mip : 0.0f;
    if (pl.ids) { pl.ids[2 * idx] = fh.geom; pl.ids[2 * idx + 1] = fh.prim; }
    if (pl.depth) pl.depth[idx] = fh.hit ? fh.t : 0.0f;
}

}  // namespace rt
