// kernels.cuh — launch interface of the sm_100a kernels (implemented in kernels.cu, driven by api.cu).
#pragma once
#include "rt_build.h"
#include "rt_integrator.h"
#include "rt_query.h"

namespace rt {

struct LaunchCounter { unsigned long long launches = 0; };

// One tile a context owns (api.cu build_pixel_list): its rectangle clipped to the image, the offset of its pixels in the context's
// pixel list (= in the packed runs of the multi-device exchange), and the part of it inside the scene's raster rectangle
// (tile-relative; cw * ch pixels at `coff` of the culled list).
struct TileRec { uint32_t x0, y0, w, h, off, cx, cy, cw, ch, coff; };

// wavefront
void launch_raygen(cudaStream_t st, const SceneD& sc, const RenderParams& rp, const Wave& w, uint32_t n, LaunchCounter& lc);
void launch_extend(cudaStream_t st, const SceneD& sc, const Wave& w, uint32_t n_max, float t_min, uint32_t* fetch_counter, bool stats,
                   LaunchCounter& lc);
void launch_shade(cudaStream_t st, const SceneD& sc, const RenderParams& rp, const Wave& w, uint32_t n_max, LaunchCounter& lc);
void launch_shadow(cudaStream_t st, const SceneD& sc, const Wave& w, uint32_t n_max, uint32_t* fetch_counter, bool stats, LaunchCounter& lc);
void launch_shadow_gather(cudaStream_t st, const Wave& w, uint32_t n_max, LaunchCounter& lc);
void launch_resolve(cudaStream_t st, const Wave& w, float4* accum, LaunchCounter& lc);
void launch_finalize(cudaStream_t st, const uint32_t* pixel_list, uint32_t n_pixels, uint32_t width, const float4* accum,
                     float inv_spp, float* beauty, unsigned long long* stats, bool accumulate, LaunchCounter& lc);
// multi-device exchange: mode 0 pack plane -> packed, 1 unpack packed -> plane, 2 unpack adding floats (planes of `ch` 32-bit channels)
void launch_pixel_lists(cudaStream_t st, const TileRec* tiles, uint32_t n_tiles, uint32_t tile_size, uint32_t* list, uint32_t* culled, LaunchCounter& lc);
void launch_pack_tiles(cudaStream_t st, int mode, const TileRec* tiles, uint32_t n_tiles, uint32_t width, uint32_t ch, uint32_t* plane, uint32_t* packed,
                       LaunchCounter& lc);
void launch_aov(cudaStream_t st, const SceneD& sc, const RenderParams& rp, const uint32_t* pixel_list, uint32_t n_pixels,
                const AovPlanes& planes, unsigned long long* stats, bool collect, LaunchCounter& lc);
// single-pixel diagnostics (render_single_pixel): one thread per sample index
struct PixelOut { uint32_t sample_index, hit; float uv[2]; float normal[3]; float radiance[3]; };
void launch_pixel_aov(cudaStream_t st, const SceneD& sc, const RenderParams& rp, uint32_t x, uint32_t y, uint32_t sample_lo,
                      uint32_t n, PixelOut* out, LaunchCounter& lc);
void launch_pixel_radiance(cudaStream_t st, const float4* radiance, uint32_t n, PixelOut* out, LaunchCounter& lc);

// ray queries (rtcuda_trace_rays / rtcuda_occluded): persistent traversal of n packed rays (rt_query.h), then, for closest hits,
// one thread per ray for the ids and the object-space re-test. `fetch_counter` must be zero.
void launch_trace(cudaStream_t st, const SceneD& sc, const float4* rays, uint32_t n, float4* hits, uint32_t* fetch_counter, LaunchCounter& lc);
void launch_occluded(cudaStream_t st, const SceneD& sc, const float4* rays, uint32_t n, uint8_t* occluded, uint32_t* fetch_counter,
                     LaunchCounter& lc);
void launch_trace_finish(cudaStream_t st, const SceneD& sc, const float4* rays, const float4* hits, uint32_t n, const QueryOut& out,
                         LaunchCounter& lc);
// rtcuda_trace_surfaces: after launch_trace, one thread per ray writes its 64-byte surface record (four float4 at surfaces[4i])
void launch_surface_finish(cudaStream_t st, const SceneD& sc, const float4* rays, const float4* hits, uint32_t n, float4* surfaces,
                           LaunchCounter& lc);

// radiance along caller-supplied rays (rtcuda_radiance, rt_query.h): normalisation (kernels_aov.cu), the live-ray list (`n_live` must
// be zero), and the depth-0 path slots of a batch, queued with the hits k_trace found
void launch_radiance_prep(cudaStream_t st, const float4* rays, uint32_t n, float4* prepared, LaunchCounter& lc);
void launch_radiance_live(cudaStream_t st, const SceneD& sc, const float4* rays, const float4* first_hits, uint32_t n, uint32_t* live,
                          uint32_t* n_live, LaunchCounter& lc);
void launch_raygen_rays(cudaStream_t st, const RenderParams& rp, const Wave& w, const float4* rays, const float4* first_hits, uint32_t key_base,
                        uint32_t n, LaunchCounter& lc);

// BVH build
void launch_prim_setup(cudaStream_t st, const BuildCtx& b, LaunchCounter& lc);
void launch_morton(cudaStream_t st, const BuildCtx& b, LaunchCounter& lc);
size_t sort_temp_bytes(uint32_t n);
void launch_sort(cudaStream_t st, void* temp, size_t temp_bytes, const uint64_t* keys_in, uint64_t* keys_out, const uint32_t* vals_in,
                 uint32_t* vals_out, uint32_t n, LaunchCounter& lc);
void launch_karras(cudaStream_t st, const BuildCtx& b, LaunchCounter& lc);
void launch_refit(cudaStream_t st, const BuildCtx& b, LaunchCounter& lc);
void launch_collapse(cudaStream_t st, const BuildCtx& b, uint32_t bound, uint32_t* level, LaunchCounter& lc);
void launch_ploc_init(cudaStream_t st, const BuildCtx& b, LaunchCounter& lc);
size_t ploc_scan_temp_bytes(uint32_t n);
constexpr uint32_t PLOC_TAIL_MAX = 8192;   // clusters at or below which one block finishes PLOC in a single launch (kernels.cu k_ploc_tail)
void launch_ploc_tail(cudaStream_t st, const BuildCtx& b, const uint32_t* state, uint32_t* state_out, uint32_t* cl_a, uint32_t* cl_b, bool in_is_a, LaunchCounter& lc);
// one PLOC round: nearest neighbours, merge flags, exclusive scan (CUB), merged nodes + compacted cluster list
void launch_ploc_round(cudaStream_t st, const BuildCtx& b, uint32_t bound, const uint32_t* state, uint32_t* state_next, void* scan_temp,
                       size_t scan_temp_bytes, LaunchCounter& lc);

// refit of the wide BVH (rtcuda_scene_update): primitive slots, then one launch per wide level (deepest first), then the SAH terms
void launch_refit_prims(cudaStream_t st, const RefitCtx& r, LaunchCounter& lc);
void launch_refit_nodes(cudaStream_t st, const RefitCtx& r, uint32_t first, uint32_t count, LaunchCounter& lc);
constexpr uint32_t SAH_BLOCKS = 256;   // partial sums launch_sah_partial writes (doubles)
void launch_sah_partial(cudaStream_t st, const float4* node_box, uint32_t n, double* partial, LaunchCounter& lc);

// emitter triangle table (rt_scene.h LightTri)
void launch_check_indices(cudaStream_t st, const uint32_t* idx, size_t n, uint32_t vertex_count, uint32_t* bad, LaunchCounter& lc);
void launch_light_tris(cudaStream_t st, const ShapeD* shapes, uint32_t shape, uint32_t tri_count, const float* vertices, const uint32_t* tris,
                       const float* normals, LightTri* out, LaunchCounter& lc);

// shading records (rt_scene.h ShadeRec), one per packed primitive
void launch_shade_recs(cudaStream_t st, const SceneD& sc, ShadeRec* out, LaunchCounter& lc);

// mip pyramids
void launch_to_f32(cudaStream_t st, const uint8_t* src, uint32_t format, float* dst, uint32_t n, LaunchCounter& lc);
void launch_resize(cudaStream_t st, const float* src, float* dst, uint32_t w, uint32_t h, uint32_t ch, uint32_t n_out, int axis, LaunchCounter& lc);
void launch_cast(cudaStream_t st, const float* src, uint32_t format, uint8_t* dst, uint32_t n, LaunchCounter& lc);

}  // namespace rt
