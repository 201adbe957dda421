// hostsim_surfaces.cpp — TEST INFRASTRUCTURE ONLY. The surface query of libraytracing_cuda (rt_query.h: the traversal of k_trace,
// one ray at a time, and the k_surface_finish body) runs on the CPU over the harness's scene build (hostsim.cpp, compiled into this
// library unchanged), so that rtcuda_trace_surfaces can be checked against the oracle without a GPU.
#include "hostsim.cpp"
#include "../../opencl-raytracing_b200/csrc/rt_query.h"

extern "C" {
// Build d (RTCUDA_BUILDER / HOSTSIM_WATERTIGHT as for hostsim_render), then the surface records of n packed rays (8 floats each):
// query_closest_ray, then surface_finish_body, 16 words per ray laid out like rtcuda_surface.
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
}  // extern "C"
