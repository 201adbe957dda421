// hostsim.cpp — TEST INFRASTRUCTURE ONLY. Compiles the per-thread kernel bodies of libraytracing_cuda
// (opencl-raytracing_b200/csrc/rt_*.h) with g++ and runs them sequentially on the CPU, so the builder,
// traversal and shading logic can be debugged and checked against the oracle in the build container,
// which has no GPU. It is never linked into or loaded by the product library; the GPU tests call
// libraytracing_cuda.so through the C ABI. Mirrors the launch sequence of api.cu: renders, scene updates, ray queries, surface
// queries and radiance along caller-supplied rays.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <vector>

#include <vector>
#include <cstdint>
// HOSTSIM_STRUCTURAL=1: classify the primitives shadow rays test (profiles/r1_notes.md, "structural" tests)
static thread_local std::vector<uint32_t>* g_prim_trace = nullptr;
#define RT_TRACE_PRIM_HOOK(pi) do { if (g_prim_trace) g_prim_trace->push_back(pi); } while (0)
#include "../../include/rtcuda.h"
#include "../../opencl-raytracing_b200/csrc/rt_build.h"
#include "../../opencl-raytracing_b200/csrc/rt_integrator.h"
#include "../../opencl-raytracing_b200/csrc/rt_cull.h"
#include "../../opencl-raytracing_b200/csrc/rt_query.h"

using namespace rt;

namespace {

M4 to_m4(const rtcuda_mat4& m) { M4 r; std::memcpy(r.m, m.m, sizeof r.m); return r; }
uint32_t next_pow2(uint32_t v) { uint32_t p = 1; while (p < v) p <<= 1; return p; }
bool is_pow2(uint32_t v) { return v && !(v & (v - 1)); }
uint32_t bps(uint32_t fmt) { return fmt == 0 ? 1 : (fmt == 1 ? 2 : 4); }

struct HostScene {
    SceneD sc{};
    std::vector<Instance> instances;
    std::vector<ShapeD> shapes;
    std::vector<LightD> lights;
    std::vector<LightTri> light_tris;
    std::vector<float4> mat_const;
    std::vector<MaterialD> materials;
    std::vector<TextureD> textures;
    std::vector<ImageD> images;
    std::vector<MipChain> mips;
    std::vector<uint8_t> image_bytes;
    std::vector<Node8> nodes;
    std::vector<Prim> prims;
    std::vector<ShadeRec> shade_recs;
    uint32_t n_levels = 0;
};

void build(HostScene& hs, const rtcuda_scene_desc* d) {
    SceneD& sc = hs.sc;
    sc.camera.kind = d->camera.kind; sc.camera.width = d->camera.raster_width; sc.camera.height = d->camera.raster_height;
    sc.camera.near_clip = d->camera.near_clip; sc.camera.far_clip = d->camera.far_clip;
    sc.camera.aperture_radius = d->camera.aperture_radius; sc.camera.focal_distance = d->camera.focal_distance;
    sc.camera.raster_to_camera = to_m4(d->camera.raster_to_camera.forward);
    sc.camera.camera_to_world = to_m4(d->camera.camera_to_world.forward);
    hs.shapes.resize(d->shape_count);
    for (uint32_t i = 0; i < d->shape_count; i++) {
        const rtcuda_shape& a = d->shapes[i];
        ShapeD& b = hs.shapes[i];
        b.kind = a.kind; b.material = a.material; b.area_light = a.area_light; b.vertex_offset = a.vertex_offset; b.vertex_count = a.vertex_count;
        b.tri_offset = a.tri_offset; b.tri_count = a.tri_count; b.normal_offset = a.normal_offset; b.uv_offset = a.uv_offset;
        std::memcpy(b.center, a.center, sizeof b.center); b.radius = a.radius;
    }
    hs.instances.resize(d->instance_count);
    uint32_t n_prims = 0;
    for (uint32_t i = 0; i < d->instance_count; i++) {
        const rtcuda_instance& a = d->instances[i];
        const rtcuda_shape& sh = d->shapes[a.shape];
        Instance& b = hs.instances[i];
        std::memset(&b, 0, sizeof b);
        b.o2w = to_m4(a.object_to_world.forward); b.w2o = to_m4(a.object_to_world.inverse);
        b.shape = a.shape; b.kind = sh.kind; b.material = sh.material; b.area_light = sh.area_light;
        b.vertex_offset = sh.vertex_offset; b.tri_offset = sh.tri_offset; b.normal_offset = sh.normal_offset; b.uv_offset = sh.uv_offset;
        b.tri_count = sh.tri_count; b.prim_base = n_prims;
        std::memcpy(b.center, sh.center, sizeof b.center); b.radius = sh.radius;
        n_prims += sh.kind == 0 ? sh.tri_count : 1;
    }
    hs.lights.resize(d->light_count);
    for (uint32_t i = 0; i < d->light_count; i++) {
        const rtcuda_light& a = d->lights[i];
        LightD& b = hs.lights[i];
        b.kind = a.kind; b.shape = a.shape;
        std::memcpy(b.a, a.position_or_direction, sizeof b.a); std::memcpy(b.b, a.intensity_or_radiance, sizeof b.b);
        b.light_to_world = to_m4(a.light_to_world);
        b.tri_table = 0;
        if (a.kind == 2) {
            b.tri_table = (uint32_t)hs.light_tris.size();
            hs.light_tris.resize(hs.light_tris.size() + hs.shapes[a.shape].tri_count);
            for (uint32_t t = 0; t < hs.shapes[a.shape].tri_count; t++)
                light_tri_body(t, hs.shapes[a.shape], d->vertices, d->tris, d->normals, hs.light_tris.data() + b.tri_table);
        }
    }
    hs.materials.resize(d->material_count);
    for (uint32_t i = 0; i < d->material_count; i++) {
        const rtcuda_material& a = d->materials[i];
        hs.materials[i] = MaterialD{a.kind, a.remap_roughness, a.albedo, a.eta, a.kappa, a.roughness, a.thickness, a.coat_albedo};
    }
    hs.textures.resize(d->texture_count);
    for (uint32_t i = 0; i < d->texture_count; i++) {
        const rtcuda_texture& a = d->textures[i];
        TextureD& b = hs.textures[i];
        b.kind = a.kind; b.image = a.image; b.filter = a.filter; b.wrap = a.wrap; b.a = a.a; b.b = a.b; b.c = a.c; b.mip_base = NONE;
        std::memcpy(b.value, a.value, sizeof b.value); std::memcpy(b.value2, a.value2, sizeof b.value2);
    }
    hs.images.resize(d->image_count);
    for (uint32_t i = 0; i < d->image_count; i++) hs.images[i] = ImageD{d->images[i].width, d->images[i].height, d->images[i].channels, d->images[i].format, d->images[i].byte_offset};
    hs.image_bytes.assign(d->image_bytes, d->image_bytes + d->image_byte_count);

    // mip pyramids (api.cu build_mips)
    std::vector<int> chain_of(d->image_count, -1);
    for (uint32_t t = 0; t < d->texture_count; t++) {
        const rtcuda_texture& tx = d->textures[t];
        if (tx.kind != 0 || tx.filter != 2) continue;
        if (chain_of[tx.image] < 0) {
            const rtcuda_image im = d->images[tx.image];
            const uint32_t ch = im.channels, fmt = im.format;
            uint32_t w = im.width, h = im.height;
            std::vector<float> cur((size_t)w * h * ch);
            for (uint32_t i = 0; i < cur.size(); i++) to_f32_body(i, hs.image_bytes.data() + im.byte_offset, fmt, cur.data());
            uint32_t size = w;
            if (!(is_pow2(w) && is_pow2(h)) || w != h) size = std::max(next_pow2(w), next_pow2(h));
            auto resize = [&](uint32_t nw, uint32_t nh) {
                std::vector<float> tmp((size_t)w * nh * ch), out((size_t)nw * nh * ch);
                for (uint32_t i = 0; i < tmp.size(); i++) resize_body(i, cur.data(), tmp.data(), w, h, ch, nh, 0);
                for (uint32_t i = 0; i < out.size(); i++) resize_body(i, tmp.data(), out.data(), w, nh, ch, nw, 1);
                cur.swap(out); w = nw; h = nh;
            };
            if (w != size || h != size) resize(size, size);
            MipChain mc; mc.first_image = (uint32_t)hs.images.size(); mc.level_count = 0;
            for (;;) {
                size_t off = (hs.image_bytes.size() + 15) & ~(size_t)15;
                hs.image_bytes.resize(off + (size_t)w * h * ch * bps(fmt));
                for (uint32_t i = 0; i < w * h * ch; i++) cast_body(i, cur.data(), fmt, hs.image_bytes.data() + off);
                hs.images.push_back(ImageD{w, h, ch, fmt, off});
                mc.level_count++;
                if (!(w > 1 && h > 1)) break;
                resize(w / 2, h / 2);
            }
            chain_of[tx.image] = (int)hs.mips.size();
            hs.mips.push_back(mc);
        }
        hs.textures[t].mip_base = (uint32_t)chain_of[tx.image];
    }

    sc.instances = hs.instances.data(); sc.shapes = hs.shapes.data(); sc.lights = hs.lights.data(); sc.light_tris = hs.light_tris.data(); sc.materials = hs.materials.data();
    sc.textures = hs.textures.data(); sc.images = hs.images.data(); sc.mips = hs.mips.data(); sc.image_bytes = hs.image_bytes.data();
    sc.vertices = d->vertices; sc.tris = d->tris; sc.normals = d->normals; sc.uvs = d->uvs;
    sc.instance_count = d->instance_count; sc.light_count = d->light_count; sc.material_count = d->material_count;
    sc.texture_count = d->texture_count; sc.env_texture = d->environment_light_texture;
    // the kernel-parameter copies (SceneD::light0, mat_const) exactly as api.cu fills them
    hs.mat_const.assign(d->material_count, make_float4(0.0f, 0.0f, 0.0f, 0.0f));
    for (uint32_t i = 0; i < d->material_count; i++) {
        if (d->materials[i].kind != 0) continue;
        const uint32_t t = d->materials[i].albedo;
        hs.mat_const[i].w = 2.0f;
        if (t != RTCUDA_NONE && t < d->texture_count && d->textures[t].kind == RTCUDA_TEXTURE_CONSTANT)
            hs.mat_const[i] = make_float4(d->textures[t].value[0], d->textures[t].value[1], d->textures[t].value[2], 1.0f);
    }
    sc.mat_const = d->material_count ? hs.mat_const.data() : nullptr;
    sc.use_light0 = 0;
    if (d->light_count) {
        sc.light0 = hs.lights[0];
        sc.light0_tri_count = hs.lights[0].kind == 2 ? hs.shapes[hs.lights[0].shape].tri_count : 0u;
        sc.light0_has_normals = hs.lights[0].kind == 2 && hs.shapes[hs.lights[0].shape].normal_offset != NONE ? 1u : 0u;
        sc.use_light0 = std::getenv("HOSTSIM_NO_LIGHT0") ? 0u : 1u;
    }
    sc.watertight = std::getenv("HOSTSIM_WATERTIGHT") ? 1u : 0u;   // test switch for RTCUDA_BACKEND_WATERTIGHT
    sc.all_diffuse = 1;
    sc.any_diffuse = 0;
    for (uint32_t m = 0; m < d->material_count; m++) { if (d->materials[m].kind != 0) sc.all_diffuse = 0; else sc.any_diffuse = 1; }
    sc.tex_uses_derivs = 0;
    for (uint32_t t = 0; t < d->texture_count; t++)
        if (d->textures[t].kind == RTCUDA_TEXTURE_IMAGE || d->textures[t].kind == RTCUDA_TEXTURE_CHECKER) sc.tex_uses_derivs = 1;
    sc.prim_count = n_prims; sc.node_count = 0;
    const uint32_t prim_slots = RT_FIXED_SLOTS ? 3u * n_prims : n_prims;   // api.cu build_bvh
    Prim hole;
    std::memset(&hole, 0xff, sizeof hole);
    hs.nodes.resize(std::max(1u, n_prims)); hs.prims.assign(std::max(1u, prim_slots), hole);
    sc.nodes = hs.nodes.data(); sc.prims = hs.prims.data();
    if (!n_prims) return;

    // BVH (api.cu build_bvh)
    const uint32_t n = n_prims;
    std::vector<Prim> prims_unsorted(n);
    std::vector<float4> aabb_lo(n), aabb_hi(n), node_lo(2 * (size_t)n), node_hi(2 * (size_t)n);
    std::vector<uint32_t> vals(n), vals_sorted(n), left(n), right(n), parent(2 * (size_t)n), count(2 * (size_t)n), visit(n, 0);
    std::vector<uint64_t> keys(n), keys_sorted(n);
    std::vector<WorkItem> qa(n), qb(n);
    uint32_t bounds_keys[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0, 0, 0};
    uint32_t counters[4] = {0, 1, 0, 0};
    BuildCtx b{};
    b.instances = hs.instances.data(); b.instance_count = d->instance_count; b.vertices = d->vertices; b.tris = d->tris; b.n = n;
    b.prims_unsorted = prims_unsorted.data(); b.aabb_lo = aabb_lo.data(); b.aabb_hi = aabb_hi.data(); b.bounds_keys = bounds_keys;
    b.keys = keys.data(); b.vals = vals.data(); b.keys_sorted = keys_sorted.data(); b.vals_sorted = vals_sorted.data();
    b.left = left.data(); b.right = right.data(); b.parent = parent.data(); b.count = count.data();
    b.node_lo = node_lo.data(); b.node_hi = node_hi.data(); b.visit = visit.data();
    b.nodes = hs.nodes.data(); b.prims = hs.prims.data(); b.counters = counters; b.prim_capacity = prim_slots;
    for (uint32_t i = 0; i < n; i++) prim_setup_body(i, b);
    for (uint32_t i = 0; i < n; i++) morton_body(i, b);
    std::vector<uint32_t> order(n);
    std::iota(order.begin(), order.end(), 0u);
    std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return keys[x] < keys[y]; });
    for (uint32_t i = 0; i < n; i++) { keys_sorted[i] = keys[order[i]]; vals_sorted[i] = vals[order[i]]; }
    const char* builder = std::getenv("RTCUDA_BUILDER");
    if (builder && std::strcmp(builder, "lbvh") == 0) {
        for (uint32_t i = 0; i + 1 < n; i++) karras_body(i, b);
        for (uint32_t i = 0; i < n; i++) refit_body(i, b);
    } else {  // PLOC (api.cu build_bvh): rounds of nearest-neighbour search, flag scan, merge + compaction
        std::vector<uint32_t> cl_a(n), cl_b(n), nn(n);
        std::vector<uint64_t> scan(n);
        uint32_t ploc_out[2] = {0, 0};
        b.nn = nn.data(); b.scan = scan.data(); b.ploc_out = ploc_out;
        b.cl_out = cl_a.data();
        for (uint32_t k = 0; k < n; k++) ploc_init_body(k, b);
        uint32_t* cin = cl_a.data();
        uint32_t* cout = cl_b.data();
        b.m = n; b.next_node = n - 1;
        while (b.m > 1) {
            b.cl_in = cin; b.cl_out = cout;
            for (uint32_t i = 0; i < b.m; i++) ploc_nn_body(i, b);
            for (uint32_t i = 0; i < b.m; i++) ploc_flag_body(i, b);
            uint64_t run = 0;
            for (uint32_t i = 0; i < b.m; i++) { const uint64_t f = scan[i]; scan[i] = run; run += f; }
            for (uint32_t i = 0; i < b.m; i++) ploc_merge_body(i, b);
            b.m = ploc_out[0]; b.next_node -= ploc_out[1];
            std::swap(cin, cout);
        }
    }
    qa[0] = WorkItem{0, 0};
    uint32_t n_items = 1;
    WorkItem* qin = qa.data();
    WorkItem* qout = qb.data();
    while (n_items) {
        b.queue_in = qin; b.queue_out = qout;
        for (uint32_t i = 0; i < n_items; i++) collapse_body(i, b);
        n_items = counters[0];
        counters[0] = 0;
        std::swap(qin, qout);
        hs.n_levels++;
    }
    sc.node_count = counters[1];
    if (!RT_FIXED_SLOTS && std::getenv("HOSTSIM_NODESTATS") != nullptr) {
        uint32_t hist[9] = {0}, inner = 0, leafc = 0, prims = 0, hi_empty = 0;
        for (uint32_t i = 0; i < counters[1]; i++) {
            const Node8& nd = hs.nodes[i];
            uint32_t m[2] = {f2u(nd.n1.z), f2u(nd.n1.w)}, c = 0;
            for (int k = 0; k < 8; k++) {
                uint32_t meta = (m[k >> 2] >> (8 * (k & 3))) & 0xff;
                if (!meta) continue;
                c++;
                if ((meta & 0x18) == 0x18) inner++; else { leafc++; prims += __builtin_popcount(meta >> 5); }
            }
            hist[c]++;
            if (!m[1]) hi_empty++;
        }
        std::fprintf(stderr, "wide nodes %u: children histogram", counters[1]);
        for (int k = 0; k <= 8; k++) std::fprintf(stderr, " %d:%u", k, hist[k]);
        std::fprintf(stderr, " | inner children %u leaf children %u prims %u | upper half empty %u\n", inner, leafc, prims, hi_empty);
    }
    V3 mn = mk3(key_float(bounds_keys[0]), key_float(bounds_keys[1]), key_float(bounds_keys[2]));
    V3 mx = mk3(key_float(bounds_keys[3]), key_float(bounds_keys[4]), key_float(bounds_keys[5]));
    V3 c = (mx + mn) / 2.0f;
    sc.scene_center[0] = c.x; sc.scene_center[1] = c.y; sc.scene_center[2] = c.z;
    sc.scene_radius = n == 1 ? INFINITY : length(mx - c);
    set_scene_bounds(sc, mn, mx, true);
    sc.prim_count = counters[2];   // primitive slots (holes included with RT_FIXED_SLOTS)
    if (std::getenv("HOSTSIM_NODESTATS")) std::fprintf(stderr, "wide nodes %u, primitives %u in %u slots (%.3f slots per primitive)\n", counters[1], counters[3], counters[2], (double)counters[2] / counters[3]);
    if (counters[3] != n || counters[2] > prim_slots) sc.node_count = 0xdeadbeef;  // lost primitives: surfaced through the stats
    else if (!std::getenv("HOSTSIM_NO_SHADE_RECS")) {
        hs.shade_recs.resize(sc.prim_count);
        for (uint32_t i = 0; i < sc.prim_count; i++) shade_rec_body(i, sc, hs.shade_recs.data());
        sc.shade_recs = hs.shade_recs.data();
    }
}

RenderParams make_params(const rtcuda_settings* st) {
    RenderParams rp{};
    rp.max_ray_depth = st->max_ray_depth; rp.accumulate_bounces = st->accumulate_bounces; rp.light_sample_count = st->light_sample_count;
    rp.samples_per_pixel = st->samples_per_pixel; rp.antialias_primary_rays = st->antialias_primary_rays;
    rp.sampler.seed_hashed = hash_seed(st->has_seed ? st->seed : 42ull);
    rp.sampler.stratified = st->sampler_kind == RTCUDA_SAMPLER_STRATIFIED; rp.sampler.jitter = st->stratified_jitter;
    rp.sampler.x_strata = st->x_strata; rp.sampler.y_strata = st->y_strata;
    return rp;
}

}  // namespace


// ---- warp-phase simulator (tuning aid for the persistent traversal kernels, kernels.cu) ---------------------
// Runs the rays of one queue through 32-lane "warps" with the same refill / vote loop as k_extend / k_shadow and
// charges each iteration the instruction cost of the phase it executed, so policies can be compared without a GPU.
// HOSTSIM_WARPSIM="policy,tri_min,refill_min": policy 0 = node + all its primitives per iteration (the r1b kernels),
// 1 = vote, lanes with pending primitives idle during node phases, 2 = vote, pending primitives are stashed.
struct SimRay { V3 o, d; float t_min, t_max; };
template <bool ANY_HIT>
static void warp_sim(const SceneD& sc, const std::vector<SimRay>& rays, const char* label) {
    const char* cfg = std::getenv("HOSTSIM_WARPSIM");
    if (!cfg || rays.empty()) return;
    int policy = 2, tri_min = 12, refill_min = 8, rays_per_warp = 0;  // rays_per_warp 0: one warp drains the whole queue (no tail)
    std::sscanf(cfg, "%d,%d,%d,%d", &policy, &tri_min, &refill_min, &rays_per_warp);
    const double C_NODE = 230, C_TRI = 85, C_INIT = 45, C_LOOP = 14, C_FIN = 8;
    struct Lane { Traversal<ANY_HIT, true> tr; uint2 stack[TRAVERSE_STACK]; bool have = false; };
    struct Warp { std::vector<Lane> lanes; bool done = false; };
    const size_t n_warps = rays_per_warp > 0 ? std::max<size_t>(1, rays.size() / rays_per_warp) : 1;
    std::vector<Warp> warps(n_warps);
    for (auto& w : warps) { w.lanes.resize(32); for (auto& l : w.lanes) l.tr.stack = l.stack; }
    TraverseStats ts{0, 0};
    size_t cursor = 0, live = n_warps;
    double cost = 0, useful = 0;
    uint64_t iters = 0, node_phases = 0, tri_phases = 0, node_lanes = 0, tri_lanes = 0, idle_lanes = 0;
    while (live) {
        for (auto& wp : warps) {   // round robin: one loop iteration per live warp
            if (wp.done) continue;
            auto& lanes = wp.lanes;
            int need = 0;
            for (auto& l : lanes) need += !l.have;
            const bool exhausted = cursor >= rays.size();
            if (need == 32 && exhausted) { wp.done = true; live--; continue; }
            cost += C_LOOP; iters++; idle_lanes += need;
            if (!exhausted && need >= refill_min) {
                cost += C_INIT;
                for (auto& l : lanes)
                    if (!l.have && cursor < rays.size()) {
                        const SimRay& r = rays[cursor++];
                        l.have = l.tr.init(sc, r.o, r.d, r.t_min, r.t_max);
                        useful += C_INIT / 32;
                    }
            }
            if (policy == 0) {
                int max_tris = 0, n_act = 0, tri_work = 0;
                for (auto& l : lanes) {
                    if (!l.have) continue;
                    n_act++;
                    l.tr.node_step(sc, &ts);
                    int k = 0;
                    while (l.tr.has_tris()) { l.tr.tri_step(sc, &ts); k++; }
                    tri_work += k;
                    max_tris = std::max(max_tris, k);
                }
                cost += C_NODE + max_tris * C_TRI;
                useful += (n_act * C_NODE + tri_work * C_TRI) / 32;
                node_phases++; node_lanes += n_act;
            } else {
                int nt = 0, nn = 0;
                for (auto& l : lanes) {
                    if (!l.have) continue;
                    const bool wt = l.tr.has_tris(), wn = l.tr.has_nodes() && (policy == 2 ? (!wt || l.tr.can_stash()) : !wt);
                    nt += wt; nn += wn;
                }
                const bool tri_phase = nt > 0 && (nn == 0 || nt >= tri_min || (policy == 1 && nt >= nn) || (policy == 3 && nt * 2 >= nn));
                if (tri_phase) {
                    for (auto& l : lanes) if (l.have && l.tr.has_tris()) l.tr.tri_step(sc, &ts);
                    cost += C_TRI; useful += nt * C_TRI / 32; tri_phases++; tri_lanes += nt;
                } else {
                    for (auto& l : lanes) {
                        if (!l.have) continue;
                        const bool wt = l.tr.has_tris();
                        if (l.tr.has_nodes() && (policy == 2 ? (!wt || l.tr.can_stash()) : !wt)) l.tr.node_step(sc, &ts);
                    }
                    cost += C_NODE; useful += nn * C_NODE / 32; node_phases++; node_lanes += nn;
                }
            }
            int fin = 0;
            for (auto& l : lanes) if (l.have && !l.tr.next()) { l.have = false; fin++; }
            if (fin) { cost += C_FIN; useful += fin * C_FIN / 32; }
        }
    }
    std::fprintf(stderr, "  warpsim %-9s policy %d tri_min %d refill %d warps %zu: rays %zu cost/ray %.1f util %.3f nodes/ray %.2f prims/ray %.2f "
                 "node-phases %llu (%.1f lanes) tri-phases %llu (%.1f lanes) idle %.1f\n", label, policy, tri_min, refill_min, n_warps, rays.size(),
                 cost / rays.size(), useful / cost, (double)ts.nodes / rays.size(), (double)ts.prims / rays.size(),
                 (unsigned long long)node_phases, (double)node_lanes / std::max<uint64_t>(1, node_phases), (unsigned long long)tri_phases,
                 (double)tri_lanes / std::max<uint64_t>(1, tri_phases), (double)idle_lanes / iters);
}

namespace {

// The caller's rays of a radiance batch (api.cu CallerRays): the prepared rays, the depth-0 hit k_trace found for each, and the
// stream key of ray 0
struct CallerRays {
    const float4* rays;
    const float4* first_hits;
    uint32_t key_base;
};

// One batch of the wavefront, shaped like api.cu run_batch: raygen, then per depth extend -> shade -> shadow -> gather. `ro` / `rd`
// are the two ray-queue buffers the depths alternate between. Without `caller` the paths start at the camera (k_raygen: only the
// rays that reach the scene bounds are queued); with it they start from the caller's rays at their known depth-0 hits
// (k_raygen_rays) and the depth-0 extend is skipped. rays[0..2] += primary, bounce and shadow rays; ts counts the BVH fetches.
// The debug hooks HOSTSIM_WARPSIM, HOSTSIM_STRUCTURAL, HOSTSIM_TRACE and HOSTSIM_NO_MATERIAL_SPLIT apply to every wavefront
// (renders, scene updates, radiance); with none of them set, every caller's wavefront runs only the kernels' bodies, in api.cu's
// order, and the counters change no result.
void run_batch(const SceneD& sc, const RenderParams& rp, Wave& w, float4* const ro[2], float4* const rd[2], uint32_t n_paths,
               TraverseStats* ts, uint64_t* rays, const CallerRays* caller) {
    uint32_t n_rays = 0;
    w.depth = 0; w.ray_o_out = ro[0]; w.ray_d_out = rd[0];
    if (caller) {
        n_rays = n_paths;
        for (uint32_t slot = 0; slot < n_paths; slot++) raygen_rays_body(slot, rp, w, caller->rays, caller->first_hits, caller->key_base);
    } else {
        for (uint32_t i = 0; i < n_paths; i++) {   // k_raygen: rays that miss the scene bounds are not queued
            float4 o4, d4;
            if (raygen_body(i, sc, rp, w, o4, d4)) { ro[0][n_rays] = o4; rd[0][n_rays] = d4; n_rays++; }
        }
        rays[0] += n_paths;
    }
    for (uint32_t depth = 0; depth <= rp.max_ray_depth && n_rays; depth++) {
        const int in = depth & 1, ot = in ^ 1;
        w.depth = depth;
        w.ray_o_in = ro[in]; w.ray_d_in = rd[in]; w.ray_o_out = ro[ot]; w.ray_d_out = rd[ot];
        const float t_min = depth == 0 ? sc.camera.near_clip : 0.0001f;
        const TraverseStats ts_before = *ts;
        if (depth || !caller) {   // k_extend
            if (std::getenv("HOSTSIM_WARPSIM")) {
                std::vector<SimRay> sim(n_rays);
                for (uint32_t q = 0; q < n_rays; q++) sim[q] = SimRay{xyz(w.ray_o_in[q]), xyz(w.ray_d_in[q]), t_min, w.ray_o_in[q].w};
                char label[32];
                std::snprintf(label, sizeof label, "ext d%u", depth);
                warp_sim<false>(sc, sim, label);
            }
            for (uint32_t q = 0; q < n_rays; q++) {
                Hit h;
                traverse<false, true>(sc, xyz(w.ray_o_in[q]), xyz(w.ray_d_in[q]), t_min, w.ray_o_in[q].w, h, ts);
                w.hits[q] = make_float4(h.t, u2f(h.prim), h.u, h.v);
            }
        }
        if (depth) rays[1] += n_rays;
        const TraverseStats ts_mid = *ts;
        uint32_t n_out = 0, n_shadow = 0, n_sray = 0, cur_q = 0;
        static const bool structural = std::getenv("HOSTSIM_STRUCTURAL") != nullptr;
        std::vector<uint32_t> vertex_prim;
        auto alloc = [&](bool cont, bool has_vertex, uint32_t k, bool final_skipped, uint32_t& rpos, uint32_t& vpos, uint32_t& first) {
            rpos = n_out; vpos = n_shadow; first = n_sray;
            if (structural && has_vertex) vertex_prim.push_back(f2u(w.hits[cur_q].y));
            n_out += cont; n_shadow += has_vertex; n_sray += k;
            rays[1] += final_skipped;   // reported with the bounce rays: the oracle (like the reference) traces them
        };
        // like launch_shade (kernels.cu): scenes that mix Diffuse with other materials take the Diffuse body first, which
        // leaves the other materials on a list for the general body (HOSTSIM_NO_MATERIAL_SPLIT: everything through the general one)
        const bool no_split = std::getenv("HOSTSIM_NO_MATERIAL_SPLIT") != nullptr;
        const bool split = !sc.all_diffuse && sc.any_diffuse && !no_split;
        std::vector<uint32_t> deferred;
        const StagePtr no_stage{nullptr, 0u, 0u};
        for (uint32_t q = 0; q < n_rays; q++) {
            cur_q = q;
            if (sc.all_diffuse) shade_vertex<DiffuseSurface>(true, q, sc, rp, w, alloc);
            else if (split) shade_vertex<DiffuseSurface, false, true>(true, q, sc, rp, w, alloc, no_stage, [](bool, uint32_t) {}, [](uint32_t&) {},
                                                                      [&](uint32_t dq) { deferred.push_back(dq); });
            else shade_vertex<Surface>(true, q, sc, rp, w, alloc);
        }
        for (uint32_t q : deferred) {
            cur_q = q;
            shade_vertex<Surface>(true, q, sc, rp, w, alloc);
        }
        uint32_t shadow_rays = 0;
        std::vector<SimRay> sim;
        std::vector<uint32_t> ray_vertex;
        if (structural) {
            ray_vertex.assign(n_sray, 0u);
            for (uint32_t v = 0; v < n_shadow; v++) for (uint32_t j = 0; j < w.svertex[v].z; j++) ray_vertex[w.svertex[v].y + j] = v;
        }
        std::vector<uint32_t> trace;
        for (uint32_t r = 0; r < n_sray; r++) {   // k_shadow
            if (!(w.sray_o[r].w >= 0.0f)) continue;
            shadow_rays++;
            if (structural) {   // one extra walk that records the primitives tested, classified against the ray's two end points
                static uint64_t c_rays = 0, c_total = 0, c_emitter = 0, c_exact = 0, c_same_geom = 0, c_other = 0, c_occluded = 0;
                trace.clear();
                g_prim_trace = &trace;
                Hit hh;
                TraverseStats dummy{0, 0};
                const bool occ = traverse<true, true>(sc, xyz(w.sray_o[r]), xyz(w.sray_d[r]), 0.001f, w.sray_o[r].w, hh, &dummy);
                g_prim_trace = nullptr;
                const uint32_t vp = vertex_prim[ray_vertex[r]];
                const uint32_t vgeom = f2u(sc.prims[vp].a.w);
                for (uint32_t pi : trace) {
                    const uint32_t geom = f2u(sc.prims[pi].a.w);
                    c_total++;
                    if (pi == vp) c_exact++;
                    else if (geom == vgeom) c_same_geom++;
                    else if (sc.instances[geom].area_light != NONE) c_emitter++;
                    else c_other++;
                }
                c_rays++; c_occluded += occ;
                if (r + 1 == n_sray)
                    std::fprintf(stderr, "structural (cumulative): shadow rays %llu occluded %llu | prim tests %llu = end-point triangle %llu + same instance as the end point %llu + emitter instance %llu + other %llu\n",
                                 (unsigned long long)c_rays, (unsigned long long)c_occluded, (unsigned long long)c_total, (unsigned long long)c_exact,
                                 (unsigned long long)c_same_geom, (unsigned long long)c_emitter, (unsigned long long)c_other);
            }
            if (std::getenv("HOSTSIM_WARPSIM")) sim.push_back(SimRay{xyz(w.sray_o[r]), xyz(w.sray_d[r]), 0.001f, w.sray_o[r].w});
            Hit h;
            if (traverse<true, true>(sc, xyz(w.sray_o[r]), xyz(w.sray_d[r]), 0.001f, w.sray_o[r].w, h, ts)) w.scontrib[r] = make_float4(0, 0, 0, 0);
        }
        if (!sim.empty()) {
            char label[32];
            std::snprintf(label, sizeof label, "shadow d%u", depth);
            warp_sim<true>(sc, sim, label);
        }
        for (uint32_t v = 0; v < n_shadow; v++) shadow_gather_body(v, w);
        rays[2] += shadow_rays;
        if (std::getenv("HOSTSIM_TRACE"))  // per-depth work profile (DESIGN.md "Measurement": ray-class table)
            std::fprintf(stderr, "depth %u: extend rays %u nodes %u prims %u | vertices %u shadow rays %u nodes %u prims %u | next %u\n", depth,
                         n_rays, ts_mid.nodes - ts_before.nodes, ts_mid.prims - ts_before.prims, n_shadow, shadow_rays,
                         ts->nodes - ts_mid.nodes, ts->prims - ts_mid.prims, n_out);
        n_rays = n_out;
    }
}

// The wavefront over `n_items` path sources (`items`: a frame's pixels, or the live rays of a radiance call) x samples
// [sample_lo, sample_hi), in batches of at most `capacity` path slots (0: 2^20); accum[n_items] receives each item's sum over its
// samples (k_resolve). The batch shape follows api.cu batch_shape, except that the samples per batch are not evened out.
void run_wavefront(const SceneD& sc, const RenderParams& rp, const uint32_t* items, uint32_t n_items, uint32_t sample_lo, uint32_t sample_hi,
                   uint32_t capacity, TraverseStats* ts, uint64_t* rays, float4* accum, const CallerRays* caller = nullptr) {
    if (!capacity) capacity = 1u << 20;
    uint32_t shadow_k = 0;
    for (uint32_t i = 0; i < sc.light_count; i++) shadow_k += sc.lights[i].kind == 2 ? rp.light_sample_count : 1;
    const uint32_t np_batch = std::min(n_items, capacity);
    const uint32_t ns_batch = std::max(1u, std::min(sample_hi - sample_lo, capacity / np_batch));
    const uint32_t cap = np_batch * ns_batch;
    const size_t kk = std::max(1u, shadow_k);
    std::vector<PathState> state(cap);
    std::vector<float4> radiance(cap), ro[2], rd[2], hits(cap), sray_o(cap * kk), sray_d(cap * kk), scontrib(cap * kk);
    for (int i = 0; i < 2; i++) { ro[i].resize(cap); rd[i].resize(cap); }
    std::vector<uint4> svertex(cap);
    unsigned long long kernel_stats[STAT_TOTAL] = {0};   // the kernels' STAT_* block: the harness counts rays itself
    Wave w{};
    w.pixel_list = items; w.capacity = cap;
    w.state = state.data(); w.radiance = radiance.data(); w.hits = hits.data(); w.stats = kernel_stats;
    w.shadow_k = shadow_k; w.svertex = svertex.data(); w.sray_o = sray_o.data(); w.sray_d = sray_d.data(); w.scontrib = scontrib.data();
    float4* const qo[2] = {ro[0].data(), ro[1].data()};
    float4* const qd[2] = {rd[0].data(), rd[1].data()};
    for (uint32_t p0 = 0; p0 < n_items; p0 += np_batch) {
        const uint32_t np = std::min(np_batch, n_items - p0);
        for (uint32_t s0 = sample_lo; s0 < sample_hi; s0 += ns_batch) {
            const uint32_t ns = std::min(ns_batch, sample_hi - s0);
            w.pixel_base = p0; w.n_pixels = np; w.sample_base = s0; w.n_samples = ns;
            run_batch(sc, rp, w, qo, qd, np * ns, ts, rays, caller);
            for (uint32_t i = 0; i < np; i++) resolve_body(i, w, accum);
        }
    }
}

// The frame of a built scene (api.cu render_device). sample_hi == 0: the whole frame (mean over all samples). Otherwise samples
// [sample_lo, sample_hi) only and the beauty plane holds their un-normalised sum — the harness's rtcuda_render_samples_device
// (sample-range partition across ranks). stats_out[8]: primary, bounce, shadow, aov rays, nodes fetched, prims fetched, wide node
// count, collapse levels.
int render_scene(const HostScene& hs, const rtcuda_settings* st, rtcuda_outputs* out, uint32_t tile_rank, uint32_t tile_world,
                 uint32_t capacity, uint64_t* stats_out, uint32_t sample_lo, uint32_t sample_hi) {
    const bool sum_mode = sample_hi != 0;
    if (!sum_mode) sample_hi = st->samples_per_pixel;
    if (sample_lo >= sample_hi || sample_hi > st->samples_per_pixel) return 1;
    const SceneD& sc = hs.sc;
    const RenderParams rp = make_params(st);
    const uint32_t W = sc.camera.width, H = sc.camera.height, TS = 64;
    if (out->width != W || out->height != H) return 1;
    if (tile_world == 0) tile_world = 1;
    std::vector<uint32_t> pixels;
    const uint32_t tiles_x = (W + TS - 1) / TS, tiles_y = (H + TS - 1) / TS;
    for (uint32_t ty = 0; ty < tiles_y; ty++)
        for (uint32_t tx = 0; tx < tiles_x; tx++) {
            if ((ty * (tiles_x + (tile_world > 1 && tiles_x % tile_world == 0 ? 1u : 0u)) + tx) % tile_world != tile_rank) continue;
            for (uint32_t m = 0; m < TS * TS; m++) {
                uint32_t x = 0, y = 0;
                for (uint32_t bit = 0; bit < 6; bit++) { x |= ((m >> (2 * bit)) & 1u) << bit; y |= ((m >> (2 * bit + 1)) & 1u) << bit; }
                x += tx * TS; y += ty * TS;
                if (x < W && y < H) pixels.push_back((y << 16) | x);
            }
        }
    const uint32_t np_all = (uint32_t)pixels.size();
    const size_t npix = (size_t)W * H;
    uint64_t stats[8] = {0};
    TraverseStats ts{0, 0};
    const uint32_t o = st->outputs;
    AovPlanes pl{};
    pl.normals = (o & RTCUDA_AOV_NORMALS) ? out->normals : nullptr; pl.albedo = (o & RTCUDA_AOV_ALBEDO) ? out->albedo : nullptr;
    pl.uv = (o & RTCUDA_AOV_UV_COORDS) ? out->uv : nullptr; pl.mip_level = (o & RTCUDA_AOV_MIP_LEVEL) ? out->mip_level : nullptr;
    pl.ids = (o & RTCUDA_AOV_DEBUG_IDS) ? out->debug_ids : nullptr; pl.depth = (o & RTCUDA_AOV_DEBUG_DEPTH) ? out->debug_depth : nullptr;
    if (pl.normals || pl.albedo || pl.uv || pl.mip_level || pl.ids || pl.depth) {
        if (pl.normals) std::memset(pl.normals, 0, npix * 12);
        if (pl.albedo) std::memset(pl.albedo, 0, npix * 12);
        if (pl.uv) std::memset(pl.uv, 0, npix * 8);
        if (pl.mip_level) std::memset(pl.mip_level, 0, npix * 4);
        if (pl.ids) std::memset(pl.ids, 0, npix * 8);
        if (pl.depth) std::memset(pl.depth, 0, npix * 4);
        for (uint32_t i = 0; i < np_all; i++) aov_body<true>(i, sc, rp, pixels.data(), pl, &ts);
        stats[3] += np_all;
    }
    if ((o & RTCUDA_AOV_BEAUTY) && out->beauty && np_all) {
        std::memset(out->beauty, 0, npix * 12);
        // api.cu build_pixel_list: the beauty pass only takes the pixels whose camera rays can reach the scene bounds (rt_cull.h)
        int rect[4];
        if (!std::getenv("HOSTSIM_NO_PIXEL_CULL") && scene_raster_rect(sc, rect)) {
            std::vector<uint32_t> kept;
            for (uint32_t packed : pixels) {
                const int x = (int)(packed & 0xffffu), y = (int)(packed >> 16);
                if (x >= rect[0] && x <= rect[2] && y >= rect[1] && y <= rect[3]) kept.push_back(packed);
            }
            stats[0] += (uint64_t)(pixels.size() - kept.size()) * (sample_hi - sample_lo);   // still primary rays, dropped like raygen's culled ones
            pixels.swap(kept);
        }
        const uint32_t nb = (uint32_t)pixels.size();
        if (nb) {
            std::vector<float4> accum(nb, make_float4(0, 0, 0, 0));
            run_wavefront(sc, rp, pixels.data(), nb, sample_lo, sample_hi, capacity, &ts, stats, accum.data());
            const float inv_spp = sum_mode ? 1.0f : 1.0f / (float)st->samples_per_pixel;
            for (uint32_t i = 0; i < nb; i++) {
                size_t idx = (size_t)(pixels[i] >> 16) * W + (pixels[i] & 0xffffu);
                out->beauty[3 * idx] = accum[i].x * inv_spp; out->beauty[3 * idx + 1] = accum[i].y * inv_spp; out->beauty[3 * idx + 2] = accum[i].z * inv_spp;
            }
        }
    }
    stats[4] = ts.nodes; stats[5] = ts.prims; stats[6] = sc.node_count; stats[7] = hs.n_levels;
    if (stats_out) std::memcpy(stats_out, stats, sizeof stats);
    return 0;
}

// ---- scene updates (api.cu update_scene): rt_build.h refit_prims_body / refit_nodes_body, the SAH cost and the refit-or-rebuild rule

// Wide nodes per level, root first: level L + 1 is the contiguous run of the inner children of level L (api.cu keeps these
// counts from the collapse; here they are read back from the tree)
std::vector<uint32_t> wide_levels(const HostScene& hs) {
    std::vector<uint32_t> levels;
    if (!hs.sc.node_count) return levels;
    uint32_t first = 0, count = 1;
    while (count) {
        levels.push_back(count);
        uint32_t next = 0;
        for (uint32_t i = first; i < first + count; i++) next += (uint32_t)__builtin_popcount(f2u(hs.nodes[i].n1.z) >> 24);
        first += count;
        count = next;
    }
    return levels;
}

RefitCtx refit_ctx(HostScene& hs, std::vector<float4>& node_box, uint32_t* bounds_keys) {
    RefitCtx r{};
    r.instances = hs.instances.data(); r.vertices = hs.sc.vertices; r.tris = hs.sc.tris;
    r.prims = hs.prims.data(); r.prim_slots = hs.sc.prim_count; r.nodes = hs.nodes.data();
    node_box.assign(2 * (size_t)std::max(1u, hs.sc.node_count), make_float4(0, 0, 0, 0));
    r.node_box = node_box.data();
    r.bounds_keys = bounds_keys;
    return r;
}

// api.cu refit_nodes: every level, deepest first, then the SAH cost
double refit_nodes(HostScene& hs, RefitCtx& r, bool write) {
    r.write_nodes = write ? 1u : 0u;
    const std::vector<uint32_t> levels = wide_levels(hs);
    std::vector<uint32_t> first(levels.size());
    uint32_t n = 0;
    for (size_t L = 0; L < levels.size(); L++) { first[L] = n; n += levels[L]; }
    for (size_t L = levels.size(); L-- > 0;)
        for (uint32_t i = 0; i < levels[L]; i++) refit_nodes_body(first[L] + i, r);
    double children = 0.0;
    for (uint32_t i = 0; i < n; i++) children += (double)r.node_box[2 * (size_t)i].w;
    return sah_cost(r.node_box, children);
}

void refit_prims(RefitCtx& r) {
    for (uint32_t i = 0; i < r.prim_slots; i++) {
        V3 lo, hi;
        if (!refit_prims_body(i, r, lo, hi)) continue;
        atomic_min_u32(&r.bounds_keys[0], float_key(lo.x)); atomic_min_u32(&r.bounds_keys[1], float_key(lo.y)); atomic_min_u32(&r.bounds_keys[2], float_key(lo.z));
        atomic_max_u32(&r.bounds_keys[3], float_key(hi.x)); atomic_max_u32(&r.bounds_keys[4], float_key(hi.y)); atomic_max_u32(&r.bounds_keys[5], float_key(hi.z));
    }
}

// api.cu update_scene on the harness's scene; `d` has the topology of the scene hs was built from. Returns bvh_last_update
// (2 refit, 3 rebuild); *sah: the cost of the tree after the update.
uint32_t update(HostScene& hs, const rtcuda_scene_desc* d, double max_growth, double* sah) {
    SceneD& sc = hs.sc;
    std::vector<float4> node_box;
    uint32_t keys[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
    RefitCtx r = refit_ctx(hs, node_box, keys);
    const double built = refit_nodes(hs, r, false);
    for (uint32_t i = 0; i < d->instance_count; i++) {
        hs.instances[i].o2w = to_m4(d->instances[i].object_to_world.forward);
        hs.instances[i].w2o = to_m4(d->instances[i].object_to_world.inverse);
    }
    for (uint32_t i = 0; i < d->light_count; i++) {
        LightD& b = hs.lights[i];
        std::memcpy(b.a, d->lights[i].position_or_direction, sizeof b.a);
        std::memcpy(b.b, d->lights[i].intensity_or_radiance, sizeof b.b);
        b.light_to_world = to_m4(d->lights[i].light_to_world);
    }
    if (d->light_count) sc.light0 = hs.lights[0];
    sc.camera.near_clip = d->camera.near_clip; sc.camera.far_clip = d->camera.far_clip;
    sc.camera.aperture_radius = d->camera.aperture_radius; sc.camera.focal_distance = d->camera.focal_distance;
    sc.camera.raster_to_camera = to_m4(d->camera.raster_to_camera.forward);
    sc.camera.camera_to_world = to_m4(d->camera.camera_to_world.forward);
    if (!sc.prim_count) { *sah = 0.0; return 1; }
    refit_prims(r);
    const double refit = refit_nodes(hs, r, true);
    if (refit_needs_rebuild(refit, built, max_growth)) {
        // api.cu rebuilds from the resident geometry and the updated instance table: the build of d
        hs = HostScene();
        build(hs, d);
        RefitCtx r2 = refit_ctx(hs, node_box, keys);
        *sah = refit_nodes(hs, r2, false);
        return 3;
    }
    uint32_t n_prims = 0;
    for (const Instance& inst : hs.instances) n_prims += inst.kind == 0 ? inst.tri_count : 1;
    const V3 mn = mk3(key_float(keys[0]), key_float(keys[1]), key_float(keys[2])), mx = mk3(key_float(keys[3]), key_float(keys[4]), key_float(keys[5]));
    const V3 c = (mx + mn) / 2.0f;
    sc.scene_center[0] = c.x; sc.scene_center[1] = c.y; sc.scene_center[2] = c.z;
    sc.scene_radius = n_prims == 1 ? INFINITY : length(mx - c);
    set_scene_bounds(sc, mn, mx, true);
    *sah = refit;
    return 2;
}

}  // namespace

extern "C" {

// mode 0: triangle_t (the reference's Moller-Trumbore), mode 1: triangle_watertight. out = t, u, v
__attribute__((visibility("default")))
int hostsim_ray_triangle(int mode, const float* p0, const float* p1, const float* p2, const float* o, const float* d, float t_min, float t_max,
                         float* out) {
    float t = 0, u = 0, v = 0;
    const V3 a = mk3(p0[0], p0[1], p0[2]), b = mk3(p1[0], p1[1], p1[2]), c = mk3(p2[0], p2[1], p2[2]);
    const V3 oo = mk3(o[0], o[1], o[2]), dd = mk3(d[0], d[1], d[2]);
    const bool h = mode ? triangle_watertight(a, b, c, oo, dd, t_min, t_max, t, u, v) : triangle_t(a, b, c, oo, dd, t_min, t_max, t, u, v);
    out[0] = t; out[1] = u; out[2] = v;
    return h ? 1 : 0;
}

// rt_cull.h scene_raster_rect for a scene description: 1 and rect = [x0, y0, x1, y1] when pixels outside it can be dropped
__attribute__((visibility("default")))
int hostsim_raster_rect(const rtcuda_scene_desc* d, int* rect) {
    HostScene hs;
    build(hs, d);
    return scene_raster_rect(hs.sc, rect) ? 1 : 0;
}

// Build d, then render_scene
__attribute__((visibility("default")))
int hostsim_render_samples(const rtcuda_scene_desc* d, const rtcuda_settings* st, rtcuda_outputs* out, uint32_t tile_rank, uint32_t tile_world,
                           uint32_t capacity, uint64_t* stats_out, uint32_t sample_lo, uint32_t sample_hi) {
    HostScene hs;
    build(hs, d);
    return render_scene(hs, st, out, tile_rank, tile_world, capacity, stats_out, sample_lo, sample_hi);
}

__attribute__((visibility("default")))
int hostsim_render(const rtcuda_scene_desc* d, const rtcuda_settings* st, rtcuda_outputs* out, uint32_t tile_rank, uint32_t tile_world,
                   uint32_t capacity, uint64_t* stats_out) {
    return hostsim_render_samples(d, st, out, tile_rank, tile_world, capacity, stats_out, 0, 0);
}

// Build d, then refit the tree with d's own (unchanged) transforms. counts = {wide nodes, primitive slots}; the node / slot arrays
// of the build and of the refit are copied out when the pointers are non-null (sized from a first call with null pointers).
// sah = {cost of the built tree, cost after the refit}.
__attribute__((visibility("default")))
int hostsim_refit_identity(const rtcuda_scene_desc* d, uint32_t* counts, Node8* nodes_built, Node8* nodes_refit, Prim* prims_built,
                           Prim* prims_refit, double* sah) {
    HostScene hs;
    build(hs, d);
    counts[0] = hs.sc.node_count; counts[1] = hs.sc.prim_count;
    if (nodes_built) std::memcpy(nodes_built, hs.nodes.data(), hs.sc.node_count * sizeof(Node8));
    if (prims_built) std::memcpy(prims_built, hs.prims.data(), hs.sc.prim_count * sizeof(Prim));
    std::vector<float4> node_box;
    uint32_t keys[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
    RefitCtx r = refit_ctx(hs, node_box, keys);
    sah[0] = refit_nodes(hs, r, false);
    refit_prims(r);
    sah[1] = refit_nodes(hs, r, true);
    if (nodes_refit) std::memcpy(nodes_refit, hs.nodes.data(), hs.sc.node_count * sizeof(Node8));
    if (prims_refit) std::memcpy(prims_refit, hs.prims.data(), hs.sc.prim_count * sizeof(Prim));
    return 0;
}

// Build a, update it to b (camera, instance transforms, lights; the rebuild rule at `max_growth`, 0 forces the rebuild), then
// render_scene the whole frame. stats_out[8] as for render_scene; info = {bvh_last_update, SAH cost after the update}.
__attribute__((visibility("default")))
int hostsim_update_render(const rtcuda_scene_desc* a, const rtcuda_scene_desc* b, const rtcuda_settings* st, rtcuda_outputs* out,
                          double max_growth, uint64_t* stats_out, double* info) {
    HostScene hs;
    build(hs, a);
    double sah = 0.0;
    info[0] = (double)update(hs, b, max_growth, &sah);
    info[1] = sah;
    return render_scene(hs, st, out, 0, 1, 0, stats_out, 0, 0);
}

// Ray queries (rt_query.h: the traversal of k_trace one ray at a time, then the k_trace_finish body) over the build of d: n packed
// rays (8 floats each). Closest hit into t / ids / barycentrics (each may be null), any hit into occluded (may be null).
__attribute__((visibility("default")))
int hostsim_trace_rays(const rtcuda_scene_desc* d, const float* rays, uint64_t n, float* t, uint32_t* ids, float* barycentrics,
                       uint8_t* occluded) {
    HostScene hs;
    build(hs, d);
    const float4* r = (const float4*)rays;
    std::vector<float4> hits(n);
    for (uint64_t i = 0; i < n; i++) hits[i] = query_closest_ray(hs.sc, r[2 * i], r[2 * i + 1]);
    const QueryOut out{t, ids, barycentrics};
    for (uint64_t i = 0; i < n; i++) trace_finish_body((uint32_t)i, hs.sc, r, hits.data(), out);
    if (occluded)
        for (uint64_t i = 0; i < n; i++) occluded[i] = query_occluded_ray(hs.sc, r[2 * i], r[2 * i + 1]);
    return 0;
}

// Surface queries over the build of d: query_closest_ray, then surface_finish_body (k_surface_finish), 16 words per packed ray laid
// out like rtcuda_surface.
__attribute__((visibility("default")))
int hostsim_trace_surfaces(const rtcuda_scene_desc* d, const float* rays, uint64_t n, float* surfaces) {
    HostScene hs;
    build(hs, d);
    const float4* r = (const float4*)rays;
    std::vector<float4> hits(n);
    for (uint64_t i = 0; i < n; i++) hits[i] = query_closest_ray(hs.sc, r[2 * i], r[2 * i + 1]);
    for (uint64_t i = 0; i < n; i++) surface_finish_body((uint32_t)i, hs.sc, r, hits.data(), (float4*)surfaces);
    return 0;
}

// rtcuda_radiance in the launch order of api.cu radiance_chunk: build d, then n packed rays (8 floats each) through the wavefront
// in batches of at most `capacity` path slots (0: 2^20), keys stream_base + i. radiance: n x 3 floats; prepared (may be null): the
// normalised rays, n x 8 floats.
__attribute__((visibility("default")))
int hostsim_radiance(const rtcuda_scene_desc* d, const rtcuda_settings* st, const float* rays, uint64_t n, uint32_t stream_base,
                     uint32_t capacity, float* radiance, float* prepared) {
    if (!st->samples_per_pixel) return 1;
    HostScene hs;
    build(hs, d);
    const SceneD& sc = hs.sc;
    RenderParams rp = make_params(st);
    rp.antialias_primary_rays = 0;
    const float4* in = (const float4*)rays;
    std::vector<float4> prep(2 * n), first(n);
    for (uint64_t i = 0; i < n; i++) radiance_prep_ray(in[2 * i], in[2 * i + 1], prep[2 * i], prep[2 * i + 1]);   // k_radiance_prep
    if (prepared) std::memcpy(prepared, prep.data(), n * 32);
    for (uint64_t i = 0; i < n; i++) first[i] = query_closest_ray(sc, prep[2 * i], prep[2 * i + 1]);                // k_trace
    std::vector<uint32_t> live;                                                                                       // k_radiance_live
    for (uint64_t i = 0; i < n; i++)
        if (radiance_ray_live(sc, prep.data(), first.data(), (uint32_t)i)) live.push_back((uint32_t)i);
    std::memset(radiance, 0, n * 12);
    const uint32_t n_live = (uint32_t)live.size(), spp = st->samples_per_pixel;
    if (!n_live) return 0;
    std::vector<float4> accum(n_live, make_float4(0, 0, 0, 0));
    const CallerRays caller{prep.data(), first.data(), stream_base};
    TraverseStats ts{0, 0};   // the call reports no statistics; counting fetches leaves the walks' hits unchanged
    uint64_t counts[3] = {0, 0, 0};
    run_wavefront(sc, rp, live.data(), n_live, 0, spp, capacity, &ts, counts, accum.data(), &caller);
    const float inv_spp = 1.0f / (float)spp;   // k_finalize
    for (uint32_t i = 0; i < n_live; i++) {
        const uint32_t r = live[i];
        radiance[3 * r] = accum[i].x * inv_spp; radiance[3 * r + 1] = accum[i].y * inv_spp; radiance[3 * r + 2] = accum[i].z * inv_spp;
    }
    return 0;
}
}  // extern "C"
