// kernels_aov.cu — the first-hit AOV pass and the single-pixel diagnostics kernels.
//
// Compiled with -fmad=false (Makefile): the AOV planes carry the strict 1e-4 parity gate against the CPU
// reference, which never contracts a*b+c (Rust has no implicit fma). One primary ray per pixel, so the cost of
// unfused multiply-adds is irrelevant here; the wavefront kernels (kernels.cu) keep FMA contraction.
#include "kernels.cuh"

namespace rt {

constexpr int BLOCK = 256;
static inline uint32_t grid_for(uint32_t n, int block = BLOCK) { return n ? (n + block - 1) / block : 1; }

__device__ __forceinline__ void warp_add_stat(unsigned long long* dst, uint32_t v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31u) == 0 && v) atomicAdd(dst, (unsigned long long)v);
}

template <bool STATS>
__global__ void __launch_bounds__(BLOCK) k_aov(const __grid_constant__ SceneD sc, const __grid_constant__ RenderParams rp, const uint32_t* pixel_list, uint32_t n, AovPlanes pl,
                                                unsigned long long* stats) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    TraverseStats ts;
    ts.nodes = ts.prims = 0;
    if (i < n) aov_body<STATS>(i, sc, rp, pixel_list, pl, &ts);
    if (i == 0) atomicAdd(&stats[STAT_AOV], (unsigned long long)n);
    if (STATS) {
        warp_add_stat(&stats[STAT_AOV_NODES], ts.nodes);
        warp_add_stat(&stats[STAT_AOV_PRIMS], ts.prims);
    }
}

__global__ void k_pixel_aov(const __grid_constant__ SceneD sc, const __grid_constant__ RenderParams rp, uint32_t x, uint32_t y, uint32_t lo, uint32_t n, PixelOut* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    TraverseStats ts;
    FirstHit fh = first_hit<false>(sc, rp, x, y, lo + i, &ts);
    PixelOut& o = out[i];
    o.sample_index = lo + i;
    o.hit = fh.hit ? 1u : 0u;
    o.uv[0] = fh.uv.x; o.uv[1] = fh.uv.y;
    o.normal[0] = fh.normal.x; o.normal[1] = fh.normal.y; o.normal[2] = fh.normal.z;
}
__global__ void k_pixel_radiance(const float4* radiance, uint32_t n, PixelOut* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i].radiance[0] = radiance[i].x; out[i].radiance[1] = radiance[i].y; out[i].radiance[2] = radiance[i].z;
}

// Ray queries, after k_trace (kernels.cu): here, in the IEEE translation unit, so that the re-test of the winning triangle reports
// the reference's object-space t / u / v to rounding like the first-hit AOVs
__global__ void __launch_bounds__(BLOCK) k_trace_finish(const __grid_constant__ SceneD sc, const float4* rays, const float4* hits, uint32_t n,
                                                         const QueryOut out) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    if (i < n) trace_finish_body(i, sc, rays, hits, out);
}

void launch_trace_finish(cudaStream_t st, const SceneD& sc, const float4* rays, const float4* hits, uint32_t n, const QueryOut& out,
                         LaunchCounter& lc) {
    k_trace_finish<<<grid_for(n), BLOCK, 0, st>>>(sc, rays, hits, n, out);
    lc.launches++;
}

// rtcuda_radiance: the caller's rays normalised (rt_query.h radiance_prep_ray) here, in the IEEE translation unit, so that the CPU
// reference reproduces the prepared rays bit for bit
__global__ void __launch_bounds__(BLOCK) k_radiance_prep(const float4* rays, uint32_t n, float4* prepared) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    if (i >= n) return;
    float4 o, d;
    radiance_prep_ray(rays[2 * (size_t)i], rays[2 * (size_t)i + 1], o, d);
    prepared[2 * (size_t)i] = o;
    prepared[2 * (size_t)i + 1] = d;
}

void launch_radiance_prep(cudaStream_t st, const float4* rays, uint32_t n, float4* prepared, LaunchCounter& lc) {
    k_radiance_prep<<<grid_for(n), BLOCK, 0, st>>>(rays, n, prepared);
    lc.launches++;
}

void launch_aov(cudaStream_t st, const SceneD& sc, const RenderParams& rp, const uint32_t* pixel_list, uint32_t n_pixels,
                const AovPlanes& planes, unsigned long long* stats, bool collect, LaunchCounter& lc) {
    if (collect) k_aov<true><<<grid_for(n_pixels), BLOCK, 0, st>>>(sc, rp, pixel_list, n_pixels, planes, stats);
    else k_aov<false><<<grid_for(n_pixels), BLOCK, 0, st>>>(sc, rp, pixel_list, n_pixels, planes, stats);
    lc.launches++;
}
void launch_pixel_aov(cudaStream_t st, const SceneD& sc, const RenderParams& rp, uint32_t x, uint32_t y, uint32_t sample_lo, uint32_t n,
                      PixelOut* out, LaunchCounter& lc) {
    k_pixel_aov<<<grid_for(n, 64), 64, 0, st>>>(sc, rp, x, y, sample_lo, n, out);
    lc.launches++;
}
void launch_pixel_radiance(cudaStream_t st, const float4* radiance, uint32_t n, PixelOut* out, LaunchCounter& lc) {
    k_pixel_radiance<<<grid_for(n, 64), 64, 0, st>>>(radiance, n, out);
    lc.launches++;
}

}  // namespace rt
