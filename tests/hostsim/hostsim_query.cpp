// hostsim_query.cpp — TEST INFRASTRUCTURE ONLY. The ray queries of libraytracing_cuda (rt_query.h: the traversal of k_trace,
// one ray at a time, and the k_trace_finish body) run on the CPU over the harness's scene build (hostsim.cpp, compiled into this
// library unchanged), so that rtcuda_trace_rays / rtcuda_occluded can be checked against the oracle without a GPU.
#include "hostsim.cpp"
#include "../../opencl-raytracing_b200/csrc/rt_query.h"

extern "C" {
// Build d (RTCUDA_BUILDER / HOSTSIM_WATERTIGHT as for hostsim_render), then query n packed rays (8 floats each). Closest hit into
// t / ids / barycentrics (each may be null), any hit into occluded (may be null).
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
}  // extern "C"
