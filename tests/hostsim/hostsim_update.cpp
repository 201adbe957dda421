// hostsim_update.cpp — TEST INFRASTRUCTURE ONLY. The scene-update refit of libraytracing_cuda (rt_build.h refit_prims_body /
// refit_nodes_body, the SAH cost and the refit-or-rebuild rule, driven like api.cu update_scene) run on the CPU over the
// harness's scene build (hostsim.cpp, compiled into this library unchanged), plus a render of an already built scene that
// follows hostsim_render's launch sequence, so that build(A) -> update to B -> render can be compared with build(B) -> render.
#include "hostsim.cpp"

namespace {

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

// The frame of a built scene, following hostsim_render_samples (whole image, all samples, batches of up to 2^20 paths, beauty
// pixels culled to the scene's raster rectangle); stats = {nodes fetched, primitives fetched}.
void render_scene(const HostScene& hs, const rtcuda_scene_desc* d, const rtcuda_settings* st, rtcuda_outputs* out, uint64_t* stats) {
    const SceneD& sc = hs.sc;
    const RenderParams rp = make_params(st);
    const uint32_t W = sc.camera.width, H = sc.camera.height, TS = 64;
    std::vector<uint32_t> pixels;
    for (uint32_t ty = 0; ty < (H + TS - 1) / TS; ty++)
        for (uint32_t tx = 0; tx < (W + TS - 1) / TS; tx++)
            for (uint32_t m = 0; m < TS * TS; m++) {
                uint32_t x = 0, y = 0;
                for (uint32_t bit = 0; bit < 6; bit++) { x |= ((m >> (2 * bit)) & 1u) << bit; y |= ((m >> (2 * bit + 1)) & 1u) << bit; }
                x += tx * TS; y += ty * TS;
                if (x < W && y < H) pixels.push_back((y << 16) | x);
            }
    const size_t npix = (size_t)W * H;
    TraverseStats ts{0, 0};
    const uint32_t o = st->outputs;
    AovPlanes pl{};
    pl.normals = (o & RTCUDA_AOV_NORMALS) ? out->normals : nullptr; pl.albedo = (o & RTCUDA_AOV_ALBEDO) ? out->albedo : nullptr;
    pl.uv = (o & RTCUDA_AOV_UV_COORDS) ? out->uv : nullptr; pl.mip_level = (o & RTCUDA_AOV_MIP_LEVEL) ? out->mip_level : nullptr;
    pl.ids = (o & RTCUDA_AOV_DEBUG_IDS) ? out->debug_ids : nullptr; pl.depth = (o & RTCUDA_AOV_DEBUG_DEPTH) ? out->debug_depth : nullptr;
    if (pl.normals) std::memset(pl.normals, 0, npix * 12);
    if (pl.albedo) std::memset(pl.albedo, 0, npix * 12);
    if (pl.uv) std::memset(pl.uv, 0, npix * 8);
    if (pl.mip_level) std::memset(pl.mip_level, 0, npix * 4);
    if (pl.ids) std::memset(pl.ids, 0, npix * 8);
    if (pl.depth) std::memset(pl.depth, 0, npix * 4);
    if (pl.normals || pl.albedo || pl.uv || pl.mip_level || pl.ids || pl.depth)
        for (uint32_t i = 0; i < (uint32_t)pixels.size(); i++) aov_body<true>(i, sc, rp, pixels.data(), pl, &ts);
    if ((o & RTCUDA_AOV_BEAUTY) && out->beauty) {
        std::memset(out->beauty, 0, npix * 12);
        int rect[4];
        if (scene_raster_rect(sc, rect)) {
            std::vector<uint32_t> kept;
            for (uint32_t packed : pixels) {
                const int x = (int)(packed & 0xffffu), y = (int)(packed >> 16);
                if (x >= rect[0] && x <= rect[2] && y >= rect[1] && y <= rect[3]) kept.push_back(packed);
            }
            pixels.swap(kept);
        }
        const uint32_t np_all = (uint32_t)pixels.size(), spp = st->samples_per_pixel;
        if (np_all) {
            const uint32_t capacity = 1u << 20;
            uint32_t shadow_k = 0;
            for (uint32_t i = 0; i < d->light_count; i++) shadow_k += d->lights[i].kind == 2 ? rp.light_sample_count : 1;
            const uint32_t np_batch = std::min(np_all, capacity);
            const uint32_t ns_batch = std::max(1u, std::min(spp, capacity / np_batch));
            const uint32_t cap = np_batch * ns_batch;
            const size_t kk = std::max(1u, shadow_k);
            std::vector<PathState> state(cap);
            std::vector<float4> radiance(cap), ro[2], rd[2], hits(cap), sray_o(cap * kk), sray_d(cap * kk), scontrib(cap * kk);
            for (int i = 0; i < 2; i++) { ro[i].resize(cap); rd[i].resize(cap); }
            std::vector<uint4> svertex(cap);
            std::vector<float4> accum(np_all, make_float4(0, 0, 0, 0));
            unsigned long long dummy_stats[STAT_TOTAL] = {0};
            Wave w{};
            w.pixel_list = pixels.data(); w.capacity = cap;
            w.state = state.data(); w.radiance = radiance.data(); w.hits = hits.data(); w.stats = dummy_stats;
            w.shadow_k = shadow_k; w.svertex = svertex.data(); w.sray_o = sray_o.data(); w.sray_d = sray_d.data(); w.scontrib = scontrib.data();
            const bool split = !sc.all_diffuse && sc.any_diffuse;
            for (uint32_t p0 = 0; p0 < np_all; p0 += np_batch) {
                const uint32_t np = std::min(np_batch, np_all - p0);
                for (uint32_t s0 = 0; s0 < spp; s0 += ns_batch) {
                    const uint32_t ns = std::min(ns_batch, spp - s0);
                    w.pixel_base = p0; w.n_pixels = np; w.sample_base = s0; w.n_samples = ns;
                    uint32_t n_rays = 0;
                    w.depth = 0; w.ray_o_out = ro[0].data(); w.ray_d_out = rd[0].data();
                    for (uint32_t i = 0; i < np * ns; i++) {
                        float4 o4, d4;
                        if (raygen_body(i, sc, rp, w, o4, d4)) { ro[0][n_rays] = o4; rd[0][n_rays] = d4; n_rays++; }
                    }
                    for (uint32_t depth = 0; depth <= rp.max_ray_depth && n_rays; depth++) {
                        const int in = depth & 1, ot = in ^ 1;
                        w.depth = depth;
                        w.ray_o_in = ro[in].data(); w.ray_d_in = rd[in].data(); w.ray_o_out = ro[ot].data(); w.ray_d_out = rd[ot].data();
                        const float t_min = depth == 0 ? sc.camera.near_clip : 0.0001f;
                        for (uint32_t q = 0; q < n_rays; q++) {
                            Hit h;
                            traverse<false, true>(sc, xyz(w.ray_o_in[q]), xyz(w.ray_d_in[q]), t_min, w.ray_o_in[q].w, h, &ts);
                            hits[q] = make_float4(h.t, u2f(h.prim), h.u, h.v);
                        }
                        uint32_t n_out = 0, n_shadow = 0, n_sray = 0;
                        auto alloc = [&](bool cont, bool has_vertex, uint32_t k, bool, uint32_t& rpos, uint32_t& vpos, uint32_t& first) {
                            rpos = n_out; vpos = n_shadow; first = n_sray;
                            n_out += cont; n_shadow += has_vertex; n_sray += k;
                        };
                        std::vector<uint32_t> deferred;
                        const StagePtr no_stage{nullptr, 0u, 0u};
                        for (uint32_t q = 0; q < n_rays; q++) {
                            if (sc.all_diffuse) shade_vertex<DiffuseSurface>(true, q, sc, rp, w, alloc);
                            else if (split) shade_vertex<DiffuseSurface, false, true>(true, q, sc, rp, w, alloc, no_stage, [](bool, uint32_t) {}, [](uint32_t&) {},
                                                                                      [&](uint32_t dq) { deferred.push_back(dq); });
                            else shade_vertex<Surface>(true, q, sc, rp, w, alloc);
                        }
                        for (uint32_t q : deferred) shade_vertex<Surface>(true, q, sc, rp, w, alloc);
                        for (uint32_t r = 0; r < n_sray; r++) {
                            if (!(sray_o[r].w >= 0.0f)) continue;
                            Hit h;
                            if (traverse<true, true>(sc, xyz(sray_o[r]), xyz(sray_d[r]), 0.001f, sray_o[r].w, h, &ts)) scontrib[r] = make_float4(0, 0, 0, 0);
                        }
                        for (uint32_t v = 0; v < n_shadow; v++) shadow_gather_body(v, w);
                        n_rays = n_out;
                    }
                    for (uint32_t i = 0; i < np; i++) resolve_body(i, w, accum.data());
                }
            }
            const float inv_spp = 1.0f / (float)spp;
            for (uint32_t i = 0; i < np_all; i++) {
                const size_t idx = (size_t)(pixels[i] >> 16) * W + (pixels[i] & 0xffffu);
                out->beauty[3 * idx] = accum[i].x * inv_spp; out->beauty[3 * idx + 1] = accum[i].y * inv_spp; out->beauty[3 * idx + 2] = accum[i].z * inv_spp;
            }
        }
    }
    stats[0] = ts.nodes; stats[1] = ts.prims;
}

}  // namespace

extern "C" {
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

// mode 0: build b and render it; mode 1: build a, update it to b (camera, instance transforms, lights; the rebuild rule at
// `max_growth`, 0 forces the rebuild) and render. stats = {nodes fetched, primitives fetched}; info = {bvh_last_update, SAH cost}.
__attribute__((visibility("default")))
int hostsim_update_render(int mode, const rtcuda_scene_desc* a, const rtcuda_scene_desc* b, const rtcuda_settings* st, rtcuda_outputs* out,
                          double max_growth, uint64_t* stats, double* info) {
    if (st->samples_per_pixel == 0 || out->width != b->camera.raster_width || out->height != b->camera.raster_height) return 1;
    HostScene hs;
    info[0] = 0.0; info[1] = 0.0;
    if (mode == 0) build(hs, b);
    else {
        build(hs, a);
        double sah = 0.0;
        info[0] = (double)update(hs, b, max_growth, &sah);
        info[1] = sah;
    }
    render_scene(hs, b, st, out, stats);
    return 0;
}
}  // extern "C"
