// hostsim_radiance.cpp — TEST INFRASTRUCTURE ONLY. rtcuda_radiance on the CPU: the new per-ray bodies (rt_query.h: prep, live
// list, raygen_rays) and the wavefront's extend / shade / shadow / gather / resolve bodies run sequentially over the harness's scene
// build (hostsim.cpp, compiled into this library unchanged), in the launch order of api.cu radiance_chunk, so that the
// library's radiance can be checked against the oracle without a GPU.
#include "hostsim.cpp"
#include "../../opencl-raytracing_b200/csrc/rt_query.h"

extern "C" {
// Build d, then n packed rays (8 floats each) through the wavefront in batches of at most `capacity` path slots (0: 2^20), keys
// stream_base + i. radiance: n x 3 floats; prepared (may be null): the normalised rays, n x 8 floats.
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
    if (!capacity) capacity = 1u << 20;
    uint32_t shadow_k = 0;
    for (uint32_t i = 0; i < d->light_count; i++) shadow_k += d->lights[i].kind == 2 ? rp.light_sample_count : 1;
    const uint32_t np_batch = std::min(n_live, capacity);
    const uint32_t ns_batch = std::max(1u, std::min(spp, capacity / np_batch));
    const uint32_t cap = np_batch * ns_batch;
    const size_t kk = std::max(1u, shadow_k);
    std::vector<PathState> state(cap);
    std::vector<float4> rad(cap), ro[2], rd[2], hits(cap), sray_o(cap * kk), sray_d(cap * kk), scontrib(cap * kk), accum(n_live, make_float4(0, 0, 0, 0));
    for (int i = 0; i < 2; i++) { ro[i].resize(cap); rd[i].resize(cap); }
    std::vector<uint4> svertex(cap);
    unsigned long long stats[STAT_TOTAL] = {0};
    Wave w{};
    w.pixel_list = live.data(); w.capacity = cap;
    w.state = state.data(); w.radiance = rad.data(); w.hits = hits.data(); w.stats = stats;
    w.shadow_k = shadow_k; w.svertex = svertex.data(); w.sray_o = sray_o.data(); w.sray_d = sray_d.data(); w.scontrib = scontrib.data();
    const bool split = !sc.all_diffuse && sc.any_diffuse;   // launch_shade's material split
    for (uint32_t p0 = 0; p0 < n_live; p0 += np_batch) {
        const uint32_t np = std::min(np_batch, n_live - p0);
        for (uint32_t s0 = 0; s0 < spp; s0 += ns_batch) {
            const uint32_t ns = std::min(ns_batch, spp - s0);
            w.pixel_base = p0; w.n_pixels = np; w.sample_base = s0; w.n_samples = ns;
            w.depth = 0; w.ray_o_out = ro[0].data(); w.ray_d_out = rd[0].data();
            uint32_t n_rays = np * ns;
            for (uint32_t slot = 0; slot < n_rays; slot++) raygen_rays_body(slot, rp, w, prep.data(), first.data(), stream_base);   // k_raygen_rays
            for (uint32_t depth = 0; depth <= rp.max_ray_depth && n_rays; depth++) {
                const int i0 = depth & 1, i1 = i0 ^ 1;
                w.depth = depth;
                w.ray_o_in = ro[i0].data(); w.ray_d_in = rd[i0].data(); w.ray_o_out = ro[i1].data(); w.ray_d_out = rd[i1].data();
                if (depth)   // k_extend (depth 0: the hits k_trace found, queued by raygen_rays)
                    for (uint32_t q = 0; q < n_rays; q++) {
                        Hit h;
                        traverse<false, false>(sc, xyz(w.ray_o_in[q]), xyz(w.ray_d_in[q]), 0.0001f, w.ray_o_in[q].w, h, nullptr);
                        hits[q] = make_float4(h.t, u2f(h.prim), h.u, h.v);
                    }
                uint32_t n_out = 0, n_shadow = 0, n_sray = 0;
                auto alloc = [&](bool cont, bool has_vertex, uint32_t k, bool, uint32_t& rpos, uint32_t& vpos, uint32_t& first_ray) {
                    rpos = n_out; vpos = n_shadow; first_ray = n_sray;
                    n_out += cont; n_shadow += has_vertex; n_sray += k;
                };
                std::vector<uint32_t> deferred;
                const StagePtr no_stage{nullptr, 0u, 0u};
                for (uint32_t q = 0; q < n_rays; q++) {   // k_shade
                    if (sc.all_diffuse) shade_vertex<DiffuseSurface>(true, q, sc, rp, w, alloc);
                    else if (split) shade_vertex<DiffuseSurface, false, true>(true, q, sc, rp, w, alloc, no_stage, [](bool, uint32_t) {}, [](uint32_t&) {},
                                                                              [&](uint32_t dq) { deferred.push_back(dq); });
                    else shade_vertex<Surface>(true, q, sc, rp, w, alloc);
                }
                for (uint32_t q : deferred) shade_vertex<Surface>(true, q, sc, rp, w, alloc);
                for (uint32_t r = 0; r < n_sray; r++) {   // k_shadow
                    if (!(sray_o[r].w >= 0.0f)) continue;
                    Hit h;
                    if (traverse<true, false>(sc, xyz(sray_o[r]), xyz(sray_d[r]), 0.001f, sray_o[r].w, h, nullptr)) scontrib[r] = make_float4(0, 0, 0, 0);
                }
                for (uint32_t v = 0; v < n_shadow; v++) shadow_gather_body(v, w);   // k_shadow_gather
                n_rays = n_out;
            }
            for (uint32_t i = 0; i < np; i++) resolve_body(i, w, accum.data());   // k_resolve
        }
    }
    const float inv_spp = 1.0f / (float)spp;   // k_finalize
    for (uint32_t i = 0; i < n_live; i++) {
        const uint32_t r = live[i];
        radiance[3 * r] = accum[i].x * inv_spp; radiance[3 * r + 1] = accum[i].y * inv_spp; radiance[3 * r + 2] = accum[i].z * inv_spp;
    }
    return 0;
}
}  // extern "C"
