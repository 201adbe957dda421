// kernels.cu — the sm_100a kernels of the wavefront path tracer and of the device BVH / mip builders.
//
// Each __global__ function is a thin wrapper around a per-thread body from rt_*.h; what lives here is the
// data-parallel plumbing: grid-stride-free one-thread-per-item launches sized from device counters,
// warp-ballot + block-aggregated queue compaction, and warp-reduced statistics.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <type_traits>

#include "kernels.cuh"

namespace rt {

constexpr int BLOCK = 256;
// Block shape of k_shade: 128 threads, 7 resident blocks per SM asked of the Diffuse-only instantiation = 72 registers per thread and
// 28 warps per SM. The kernel waits on dependent loads (queue entry -> path state / primitive record -> instance), so warps in
// flight count for more than registers: on C3 (256 threads x 3 blocks = 80 registers, 24 warps) 76.1 ms -> 72.5 ms; 64 registers /
// 32 warps spills too much (79.1 ms), 96 registers / 20 warps 81.2 ms (profiles/r4f_ab.log, r4g_ab.log). The general
// instantiation (every non-Diffuse material) keeps 128 registers.
// k_shade prefetches the queue entry (ray origin, direction, hit: three coalesced streams) of a thread's next iteration into L2 at
// the top of the current one: the first of the three dependent round trips at the head of a vertex becomes an L2 hit. C3 shade
// 71.9 -> 69.3 ms, rough-metal box 23.6 -> 22.4, C4 unchanged (profiles/r6a_ab.log). The value is the distance in iterations.
#ifndef RT_SHADE_QUEUE_PREFETCH
#define RT_SHADE_QUEUE_PREFETCH 1
#endif
#ifndef SHADE_BLOCKS
#define SHADE_BLOCKS 7
#endif
#ifndef SHADE_THREADS
#define SHADE_THREADS 128
#endif
// (queue positions are handed out per warp — two atomics per warp with output — instead of per block with one scan and two
// barriers per chunk: shade 114 -> 110 ms on C3, 10.9 -> 10.0 ms on C5s, profiles/r1o_ab.log)

static inline uint32_t grid_for(uint32_t n, int block = BLOCK) { return n ? (n + block - 1) / block : 1; }

// L2 prefetch of a line a later iteration reads (no register, no scoreboard entry)
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// Queue entries the persistent traversal kernels prefetch ahead of their fetch counter, in units of the rays the grid holds
// in flight (0 = off)
#ifndef RT_REFILL_PREFETCH
#define RT_REFILL_PREFETCH 1
#endif
// (k_shade: an L2 prefetch of the next chunk's slot-indexed state and primitive record, one iteration ahead, cost 3 ms of 87 on C3
// instead of hiding the two dependent round trips at the head of a vertex — profiles/r4b_ab.log, variant spf)

// ---------------------------------------------------------------------------------------------------
// queue compaction: one global atomic per block per queue
// ---------------------------------------------------------------------------------------------------
// Returns the queue position of this thread's item (valid only when `push`). All threads of the block must call.
__device__ __forceinline__ uint32_t block_push(bool push, uint32_t* global_counter, uint32_t* s_count, uint32_t* s_base) {
    const unsigned mask = __ballot_sync(0xffffffffu, push);
    const unsigned lane = threadIdx.x & 31u;
    uint32_t warp_off = 0;
    if (lane == 0 && mask) warp_off = atomicAdd(s_count, (uint32_t)__popc(mask));
    warp_off = __shfl_sync(0xffffffffu, warp_off, 0);
    __syncthreads();
    if (threadIdx.x == 0) *s_base = *s_count ? atomicAdd(global_counter, *s_count) : 0u;
    __syncthreads();
    return *s_base + warp_off + (uint32_t)__popc(mask & ((1u << lane) - 1u));
}

__device__ __forceinline__ void warp_add_stat(unsigned long long* dst, uint32_t v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31u) == 0 && v) atomicAdd(dst, (unsigned long long)v);
}

// ---------------------------------------------------------------------------------------------------
// wavefront kernels
// ---------------------------------------------------------------------------------------------------
// One thread per path slot; the camera rays that can hit something are compacted into the depth-0 queue (one atomic per block).
// Every generated sample counts as a primary ray, like the reference's per-sample traverse_bvh call that stops at the root box.
__global__ void __launch_bounds__(BLOCK) k_raygen(const __grid_constant__ SceneD sc, const __grid_constant__ RenderParams rp,
                                                   const __grid_constant__ Wave w, uint32_t n) {
    __shared__ uint32_t s_count, s_base;
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    if (threadIdx.x == 0) s_count = 0;
    if (i == 0) atomicAdd(&w.stats[STAT_PRIMARY], (unsigned long long)n);
    __syncthreads();
    float4 ro, rd;
    const bool keep = i < n && raygen_body(i, sc, rp, w, ro, rd);
    const uint32_t pos = block_push(keep, w.n_out, &s_count, &s_base);
    if (keep) {
        w.ray_o_out[pos] = ro;
        w.ray_d_out[pos] = rd;
    }
    if (threadIdx.x == 0) {   // after block_push's barriers: s_count = rays this block queued
        const uint32_t in_block = min(n - blockIdx.x * BLOCK, (uint32_t)BLOCK);
        if (in_block != s_count) atomicAdd(&w.stats[STAT_CULLED], (unsigned long long)(in_block - s_count));
    }
}

// rtcuda_radiance: k_raygen for caller-supplied rays (rt_query.h raygen_rays_body). Every slot is queued at its own position, so
// the depth-0 queue length is the batch size.
__global__ void __launch_bounds__(BLOCK) k_raygen_rays(const __grid_constant__ RenderParams rp, const __grid_constant__ Wave w, const float4* rays,
                                                        const float4* first_hits, uint32_t key_base, uint32_t n) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    if (i == 0) *w.n_out = n;
    if (i < n) raygen_rays_body(i, rp, w, rays, first_hits, key_base);
}

// rtcuda_radiance: the indices of a chunk's live rays (rt_query.h radiance_ray_live), one atomic per block like k_raygen
__global__ void __launch_bounds__(BLOCK) k_radiance_live(const __grid_constant__ SceneD sc, const float4* rays, const float4* first_hits, uint32_t n,
                                                          uint32_t* live, uint32_t* n_live) {
    __shared__ uint32_t s_count, s_base;
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    if (threadIdx.x == 0) s_count = 0;
    __syncthreads();
    const bool keep = i < n && radiance_ray_live(sc, rays, first_hits, i);
    const uint32_t pos = block_push(keep, n_live, &s_count, &s_base);
    if (keep) live[pos] = i;
}

// Persistent traversal kernels. A warp keeps pulling work from the launch's queue: whenever at least
// REFILL_MIN lanes are out of work they fetch new rays together (one global atomic per refill), so the walk
// runs with nearly full warps although the rays of a bounce have wildly different traversal lengths
// (profiles/r1_notes.md: 7.3 of 32 lanes active with one ray per thread). Within the loop the warp votes, every
// iteration, between a NODE phase (each lane with a pending wide node tests its 8 child boxes; lanes that still
// hold untested leaf primitives stash them on their stack) and a PRIMITIVE phase (each lane with pending leaf
// primitives intersects one): in a given step only a few lanes have leaf hits, and looping over them right after
// the box test ran the Moller-Trumbore code at ~8 of 32 lanes. The policy and its constants were tuned with the
// warp simulator in tests/hostsim (HOSTSIM_WARPSIM). Every lane stays in the loop until the whole warp is out
// of work, which keeps the full-mask ballots / shuffles legal.
#ifndef RT_REFILL_MIN
#define RT_REFILL_MIN 10
#endif
#ifndef RT_TRI_MIN
#define RT_TRI_MIN 12
#endif
constexpr int REFILL_MIN = RT_REFILL_MIN;
constexpr int TRI_MIN = RT_TRI_MIN;
// (policy constants re-swept on the B200 after TRI_PER_PHASE = 2: refill threshold 4 / 6 / 10 / 14 / 18 / 24 -> k_extend + k_shadow
// 261 / 248 / 242 / 244-252 / 270 / 340 ms on C3, primitive-phase threshold 8 / 12 / 16 / 20 -> 258 / 248 / 244 / 249 ms; profiles/r1q_ab.log, r1r_ab.log)
// Primitives a lane may intersect per primitive phase: with 2, a lane holding several leaf primitives (a leaf has up to 3, a
// node step can hit several leaves) does not pay the vote / refill bookkeeping of the loop for each of them: k_extend
// 100.7 -> 93.1 ms, k_shadow 169.3 -> 154.0 ms on C3; 3 gains nothing more and spills in k_shadow (profiles/r1p_ab.log).
#ifndef TRI_PER_PHASE
#define TRI_PER_PHASE 2
#endif
// (refills served from per-warp reservations of 32 / 64 / 128 queue positions — one atomic per reservation instead of one per
// refill — with both halves of a ray loaded before either is looked at and a bare MUFU.RCP for 1 / direction: k_extend 61.3 ->
// 60.6 ms, k_shadow 112.8 -> 113.2-115.9 ms on C3; the extra loop-carried state spills in the 48-register kernel — not kept,
// profiles/r4j_ab.log)
// (a second node step per node phase for lanes that found inner children only: extend 92 -> 98 ms, shadow 149 -> 165 ms — not kept)
// Resident blocks per SM asked of the any-hit kernel: 5 (48 registers, ~76 B of spills) hides more of its load latency than the 4
// that 64 registers allow — k_shadow 174 -> 168 ms on C3; the closest-hit kernel carries more state and lost 1 % (A/B in
// profiles/r1_notes.md), so it keeps the register count it wants.
#ifndef RT_SHADOW_PARALLEL_LOADS
#define RT_SHADOW_PARALLEL_LOADS 0
#endif
#ifndef SHADOW_BLOCKS
#define SHADOW_BLOCKS 5
#endif

template <bool ANY_HIT, bool STATS>
__device__ __forceinline__ void warp_phase(Traversal<ANY_HIT, STATS>& tr, uint32_t have, const SceneD& sc, TraverseStats* ts) {
    const unsigned FULL = 0xffffffffu;
    const bool wt = have && tr.has_tris();
    const bool wn = have && tr.has_nodes() && (!wt || tr.can_stash());
    const unsigned mt = __ballot_sync(FULL, wt), mn = __ballot_sync(FULL, wn);
    if (mt != 0u && (mn == 0u || __popc(mt) >= TRI_MIN)) {
        if (wt) {
            tr.tri_step(sc, ts);
#if TRI_PER_PHASE > 1
#pragma unroll 1
            for (int r = 1; r < TRI_PER_PHASE && tr.has_tris(); r++) tr.tri_step(sc, ts);
#endif
        }
    } else if (wn) tr.node_step(sc, ts);
}

template <bool STATS>
__global__ void __launch_bounds__(BLOCK, 4) k_extend(const __grid_constant__ SceneD sc, const __grid_constant__ Wave w, float t_min,
                                                   uint32_t* fetch_counter) {
    const uint32_t n = *w.n_in;
    const unsigned FULL = 0xffffffffu;
    const unsigned lane = threadIdx.x & 31u, lt = (1u << lane) - 1u;
    if (blockIdx.x == 0 && threadIdx.x == 0 && w.depth != 0) atomicAdd(&w.stats[STAT_BOUNCE], (unsigned long long)n);   // primary rays: counted by k_raygen
    uint2 stack_mem[TRAVERSE_STACK];
    Traversal<false, STATS> tr;
    tr.stack = stack_mem;
    TraverseStats ts;
    ts.nodes = ts.prims = 0;
    uint32_t have = 0u, exhausted = n == 0 ? 1u : 0u;   // 32-bit flags: bools get packed into half registers (PRMT traffic in the loop)
    uint32_t q = 0;
    for (;;) {
        const unsigned need = __ballot_sync(FULL, !have);
        if (need == FULL && exhausted) break;
        if (!exhausted && __popc(need) >= REFILL_MIN) {
            const int cnt = __popc(need), leader = __ffs(need) - 1;
            uint32_t base = 0;
            if ((int)lane == leader) base = atomicAdd(fetch_counter, (uint32_t)cnt);
            base = __shfl_sync(FULL, base, leader);
            if (!have) {
                const uint32_t mine = base + (uint32_t)__popc(need & lt);
#if RT_REFILL_PREFETCH
                {
                    const uint32_t ahead = mine + (uint32_t)RT_REFILL_PREFETCH * gridDim.x * BLOCK;
                    if (ahead < n) { prefetch_l2(w.ray_o_in + ahead); prefetch_l2(w.ray_d_in + ahead); }
                }
#endif
                if (mine < n) {
                    q = mine;
                    const float4 o4 = ld_stream(&w.ray_o_in[q]), d4 = ld_stream(&w.ray_d_in[q]);
                    have = tr.init(sc, xyz(o4), xyz(d4), t_min, o4.w) ? 1u : 0u;
                    if (!have) st_stream(&w.hits[q], make_float4(o4.w, u2f(NONE), 0.0f, 0.0f));
                }
            }
            if (base + (uint32_t)cnt >= n) exhausted = 1u;
        }
        warp_phase(tr, have, sc, &ts);
        if (have && !tr.next()) {
            st_stream(&w.hits[q], make_float4(tr.hit.t, u2f(tr.hit.prim), tr.hit.u, tr.hit.v));
            have = 0u;
        }
    }
    if (STATS) {
        warp_add_stat(&w.stats[STAT_EXT_NODES], ts.nodes);
        warp_add_stat(&w.stats[STAT_EXT_PRIMS], ts.prims);
    }
}

// Shading: persistent blocks walk the ray queue in block-sized chunks (the live queue length is only known on the
// device; a grid sized for the whole batch spent a third of its warp time in blocks that found nothing to do,
// profiles/r1_notes.md). Per chunk ONE warp scan hands out the positions of all three outputs — continuation
// rays, NEE vertices, shadow rays (a variable number per thread, consecutive per vertex) — and the last lane issues
// the warp's two global atomics (one per queue counter; the 64-bit one carries vertices | shadow rays << 32).
// Scenes that mix Diffuse with other materials are shaded in two launches per depth (SPLIT): the Diffuse instantiation walks the
// whole queue and leaves the vertices with another material on a list (SPLIT = 1: one atomic per such vertex); the general
// instantiation then walks that list only (SPLIT = 2). Run over everything, the general kernel executed at 11.5 of 32 lanes (a
// warp's Diffuse and conductor lanes take turns), a quarter of its stall samples were instruction-cache misses of its 26 k
// instructions, and the Diffuse majority paid for its 128 registers (rough-metal box CM: ncu, profiles/r5b).
template <typename Surf, bool SHARED_STAGE_ONLY, int SPLIT>
__global__ void __launch_bounds__(SHADE_THREADS, std::is_same<Surf, DiffuseSurface>::value ? SHADE_BLOCKS : 512 / SHADE_THREADS) k_shade(const __grid_constant__ SceneD sc, const __grid_constant__ RenderParams rp,
                                                  const __grid_constant__ Wave w) {
    const uint32_t n = SPLIT == 2 ? *w.n_deferred : *w.n_in;
    const unsigned FULL = 0xffffffffu;
    const unsigned lane = threadIdx.x & 31u, lt = (1u << lane) - 1u;
#if RT_NEE_SMEM > 0
    // staging columns of the next-event entries (rt_integrator.h StagePtr): NEE_SMEM entries x 3 fields per thread, 48 KB per block
    __shared__ float4 s_stage[3 * NEE_SMEM * SHADE_THREADS];
    const StagePtr stage_col{s_stage + threadIdx.x, (uint32_t)SHADE_THREADS, NEE_SMEM};
#else
    const StagePtr stage_col{nullptr, 0u, 0u};
#endif
    if (SPLIT != 2 && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&w.stats[STAT_SHADED], (unsigned long long)n);
    for (uint32_t base = blockIdx.x * SHADE_THREADS; base < n; base += gridDim.x * SHADE_THREADS) {
        const uint32_t qi = base + threadIdx.x;
        const uint32_t q = SPLIT == 2 ? (qi < n ? w.deferred[qi] : 0u) : qi;
#if RT_SHADE_QUEUE_PREFETCH
        if (SPLIT != 2) {   // the queue entry of this thread's next iteration, into L2 (three streams, one line each per 8 threads)
            const uint32_t qn = qi + (uint32_t)RT_SHADE_QUEUE_PREFETCH * gridDim.x * SHADE_THREADS;
            if (qn < n) { prefetch_l2(w.ray_o_in + qn); prefetch_l2(w.ray_d_in + qn); prefetch_l2(w.hits + qn); }
        }
#endif
        // Per-warp allocation (two atomics per warp that has output, no block barrier: the warps of a block drift apart on
        // their dependent loads, and a barrier per chunk made all of them wait for the slowest), issued as early as their
        // counts are known and consumed as late as possible: the shadow-queue atomic right after next-event estimation (it
        // returns during BSDF sampling), the ray-queue atomic before the shadow entries are copied out. Waiting for the two
        // returns back to back was 6 % of the kernel's stall samples (ncu, profiles/r4e).
        unsigned long long base1 = 0;   // lane 31: vertices | shadow rays << 32 before this warp's
        uint32_t base0 = 0, incl = 0;    // lane 31: rays before this warp's; inclusive scan of the shadow-ray counts
        unsigned mc = 0, mv = 0;
        shade_vertex<Surf, SHARED_STAGE_ONLY, SPLIT == 1>(qi < n, q, sc, rp, w,
            [&](bool cont, bool has_vertex, uint32_t k, bool final_skipped, uint32_t& rpos, uint32_t& vpos, uint32_t& first) {
                (void)has_vertex; (void)rpos;
                mc = __ballot_sync(FULL, cont);
                if (w.depth + 1 == rp.max_ray_depth) {   // launch-uniform: only the shade launch before the last depth can skip rays
                    const unsigned mf = __ballot_sync(FULL, final_skipped);
                    if (mf && lane == 0) atomicAdd(&w.stats[STAT_FINAL_SKIPPED], (unsigned long long)__popc(mf));
                }
                if (lane == 31 && mc) base0 = atomicAdd(w.n_out, (uint32_t)__popc(mc));
                const unsigned long long b1 = __shfl_sync(FULL, base1, 31);
                vpos = (uint32_t)b1 + (uint32_t)__popc(mv & lt);
                first = (uint32_t)(b1 >> 32) + (incl - k);
            },
            stage_col,
            [&](bool has_vertex, uint32_t k) {
                mv = __ballot_sync(FULL, has_vertex);
                incl = k;   // inclusive warp scan of the shadow-ray counts
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t up = __shfl_up_sync(FULL, incl, o);
                    if ((int)lane >= o) incl += up;
                }
                if (lane == 31) {
                    const unsigned long long n1 = (unsigned long long)__popc(mv) | ((unsigned long long)incl << 32);
                    if (n1) base1 = atomicAdd(w.n_shadow, n1);
                }
            },
            [&](uint32_t& rpos) { rpos = __shfl_sync(FULL, base0, 31) + (uint32_t)__popc(mc & lt); },
            [&](uint32_t deferred_q) { w.deferred[atomicAdd(w.n_deferred, 1u)] = deferred_q; });
    }
}

// `occluded` (lights.rs:159-168): any-hit traversal of the compacted shadow-ray queue, same persistent refill / phase
// vote loop as k_extend. A blocked ray zeroes its contribution entry; k_shadow_gather then adds each vertex's
// entries to the path in light-sample order (deterministic: one thread per vertex, no float atomics).
template <bool STATS>
__global__ void __launch_bounds__(BLOCK, SHADOW_BLOCKS) k_shadow(const __grid_constant__ SceneD sc, const __grid_constant__ Wave w, uint32_t* fetch_counter) {
    const uint32_t n = (uint32_t)(*w.n_shadow >> 32);
    const unsigned FULL = 0xffffffffu;
    const unsigned lane = threadIdx.x & 31u, lt = (1u << lane) - 1u;
    uint2 stack_mem[TRAVERSE_STACK];
    Traversal<true, STATS> tr;
    tr.stack = stack_mem;
    TraverseStats ts;
    ts.nodes = ts.prims = 0;
    uint32_t have = 0u, exhausted = n == 0 ? 1u : 0u;
    uint32_t q = 0, n_rays = 0;
    for (;;) {
        const unsigned need = __ballot_sync(FULL, !have);
        if (need == FULL && exhausted) break;
        if (!exhausted && __popc(need) >= REFILL_MIN) {
            const int cnt = __popc(need), leader = __ffs(need) - 1;
            uint32_t base = 0;
            if ((int)lane == leader) base = atomicAdd(fetch_counter, (uint32_t)cnt);
            base = __shfl_sync(FULL, base, leader);
            if (!have) {
                const uint32_t mine = base + (uint32_t)__popc(need & lt);
#if RT_REFILL_PREFETCH
                {
                    const uint32_t ahead = mine + (uint32_t)RT_REFILL_PREFETCH * gridDim.x * BLOCK;
                    if (ahead < n) { prefetch_l2(w.sray_o + ahead); prefetch_l2(w.sray_d + ahead); }
                }
#endif
                if (mine < n) {
                    q = mine;
                    const float4 o4 = ld_stream(&w.sray_o[q]), d4 = ld_stream(&w.sray_d[q]);
#if RT_SHADOW_PARALLEL_LOADS
                    // both halves of the entry are loaded before either is looked at (testing t_max first makes the direction a
                    // second, dependent round trip)
                    const uint32_t traced = o4.w >= 0.0f ? 1u : 0u;
                    n_rays += traced;
                    have = tr.init(sc, xyz(o4), xyz(d4), 0.001f, o4.w) ? traced : 0u;
#else
                    if (o4.w >= 0.0f) {   // negative: never occluded (non-finite origin quirk), not traced
                        n_rays++;
                        have = tr.init(sc, xyz(o4), xyz(d4), 0.001f, o4.w) ? 1u : 0u;
                    }
#endif
                }
            }
            if (base + (uint32_t)cnt >= n) exhausted = 1u;
        }
        warp_phase(tr, have, sc, &ts);
        if (have && !tr.next()) {
            if (tr.found) w.scontrib[q] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            have = 0u;
        }
    }
    warp_add_stat(&w.stats[STAT_SHADOW], n_rays);
    if (STATS) {
        warp_add_stat(&w.stats[STAT_SH_NODES], ts.nodes);
        warp_add_stat(&w.stats[STAT_SH_PRIMS], ts.prims);
    }
}

// Ray queries (rtcuda_trace_rays / rtcuda_occluded): caller-supplied rays (rt_query.h), closest hit or any hit, with the
// refill / phase-vote loop of k_extend and k_shadow. The loop is duplicated here on purpose: folding the three kernels onto one
// loop would make the renderer's hottest kernels branch on their caller and change their SASS. Launch bounds follow the
// kernel each variant mirrors. Closest hit writes the traversal's Hit per ray (k_trace_finish turns it into ids and the
// object-space t / u / v); any hit writes the occlusion byte.
template <bool ANY_HIT>
__global__ void __launch_bounds__(BLOCK, ANY_HIT ? SHADOW_BLOCKS : 4) k_trace(const __grid_constant__ SceneD sc, const float4* __restrict__ rays,
                                                                            uint32_t n, float4* hits, uint8_t* occluded, uint32_t* fetch_counter) {
    const unsigned FULL = 0xffffffffu;
    const unsigned lane = threadIdx.x & 31u, lt = (1u << lane) - 1u;
    uint2 stack_mem[TRAVERSE_STACK];
    Traversal<ANY_HIT, false> tr;
    tr.stack = stack_mem;
    uint32_t have = 0u, exhausted = n == 0 ? 1u : 0u;
    uint32_t q = 0;
    for (;;) {
        const unsigned need = __ballot_sync(FULL, !have);
        if (need == FULL && exhausted) break;
        if (!exhausted && __popc(need) >= REFILL_MIN) {
            const int cnt = __popc(need), leader = __ffs(need) - 1;
            uint32_t base = 0;
            if ((int)lane == leader) base = atomicAdd(fetch_counter, (uint32_t)cnt);
            base = __shfl_sync(FULL, base, leader);
            if (!have) {
                const uint32_t mine = base + (uint32_t)__popc(need & lt);
#if RT_REFILL_PREFETCH
                {
                    const uint32_t ahead = mine + (uint32_t)RT_REFILL_PREFETCH * gridDim.x * BLOCK;
                    if (ahead < n) prefetch_l2(rays + 2 * (size_t)ahead);   // both halves of a ray share a 32-byte sector
                }
#endif
                if (mine < n) {
                    q = mine;
                    const float4 o4 = ld_stream(&rays[2 * (size_t)q]), d4 = ld_stream(&rays[2 * (size_t)q + 1]);
                    have = query_ray_valid(o4, d4) && tr.init(sc, xyz(o4), xyz(d4), o4.w, d4.w) ? 1u : 0u;
                    if (!have) {
                        if (ANY_HIT) occluded[q] = 0u;
                        else st_stream(&hits[q], query_miss_entry());
                    }
                }
            }
            if (base + (uint32_t)cnt >= n) exhausted = 1u;
        }
        warp_phase(tr, have, sc, (TraverseStats*)nullptr);
        if (have && !tr.next()) {
            if (ANY_HIT) occluded[q] = tr.found ? 1u : 0u;
            else st_stream(&hits[q], tr.found ? query_hit_entry(tr.hit) : query_miss_entry());
            have = 0u;
        }
    }
}

__global__ void __launch_bounds__(BLOCK) k_shadow_gather(const __grid_constant__ Wave w) {
    const uint32_t n = (uint32_t)(*w.n_shadow & 0xffffffffull);
    for (uint32_t v = blockIdx.x * BLOCK + threadIdx.x; v < n; v += gridDim.x * BLOCK) shadow_gather_body(v, w);
}

__global__ void __launch_bounds__(BLOCK) k_resolve(const __grid_constant__ Wave w, float4* accum) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    if (i < w.n_pixels) resolve_body(i, w, accum);
}

// Pixel mean + the NaN / Inf scan of the beauty plane (lib.rs:813-854: every channel is classified): the count of
// non-finite channels goes to the stats block; the caller side prints the reference's warnings from it.
template <bool ACCUMULATE>
__global__ void __launch_bounds__(BLOCK) k_finalize(const uint32_t* pixel_list, uint32_t n, uint32_t width, const float4* accum,
                                                     float inv_spp, float* beauty, unsigned long long* stats) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    uint32_t bad = 0;
    if (i < n) {
        const uint32_t packed = pixel_list[i];
        const size_t idx = (size_t)(packed >> 16) * width + (packed & 0xffffu);
        const float4 a = accum[i];
        float r = a.x * inv_spp, g = a.y * inv_spp, b = a.z * inv_spp;  // `radiance /= spp` is a multiply by the reciprocal (vec3.rs:122-126)
        if (ACCUMULATE) { r += beauty[3 * idx]; g += beauty[3 * idx + 1]; b += beauty[3 * idx + 2]; }   // progressive: add this range's sum to the plane
        beauty[3 * idx] = r;
        beauty[3 * idx + 1] = g;
        beauty[3 * idx + 2] = b;
        bad = (isfinite(r) ? 0u : 1u) + (isfinite(g) ? 0u : 1u) + (isfinite(b) ? 0u : 1u);
    }
    if (__any_sync(0xffffffffu, bad != 0u)) warp_add_stat(&stats[STAT_NONFINITE], bad);
}

void launch_raygen(cudaStream_t st, const SceneD& sc, const RenderParams& rp, const Wave& w, uint32_t n, LaunchCounter& lc) {
    k_raygen<<<grid_for(n), BLOCK, 0, st>>>(sc, rp, w, n);
    lc.launches++;
}
void launch_raygen_rays(cudaStream_t st, const RenderParams& rp, const Wave& w, const float4* rays, const float4* first_hits, uint32_t key_base,
                        uint32_t n, LaunchCounter& lc) {
    k_raygen_rays<<<grid_for(n), BLOCK, 0, st>>>(rp, w, rays, first_hits, key_base, n);
    lc.launches++;
}
void launch_radiance_live(cudaStream_t st, const SceneD& sc, const float4* rays, const float4* first_hits, uint32_t n, uint32_t* live,
                          uint32_t* n_live, LaunchCounter& lc) {
    k_radiance_live<<<grid_for(n), BLOCK, 0, st>>>(sc, rays, first_hits, n, live, n_live);
    lc.launches++;
}
static uint32_t persistent_grid(const void* kernel, uint32_t n_max, int block = BLOCK) {
    static int sm_counts[64] = {0};   // per device: a process may drive several GPUs (multi-device contexts)
    int dev = 0;
    cudaGetDevice(&dev);
    int& sm_count = sm_counts[dev & 63];
    if (!sm_count) cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, 0);
    const uint32_t resident = (uint32_t)sm_count * (uint32_t)(per_sm > 0 ? per_sm : 1);
    return std::max(1u, std::min(resident, grid_for(n_max, block)));
}
void launch_extend(cudaStream_t st, const SceneD& sc, const Wave& w, uint32_t n_max, float t_min, uint32_t* fetch_counter, bool stats,
                   LaunchCounter& lc) {
    if (stats) k_extend<true><<<persistent_grid((const void*)k_extend<true>, n_max), BLOCK, 0, st>>>(sc, w, t_min, fetch_counter);
    else k_extend<false><<<persistent_grid((const void*)k_extend<false>, n_max), BLOCK, 0, st>>>(sc, w, t_min, fetch_counter);
    lc.launches++;
}
void launch_shade(cudaStream_t st, const SceneD& sc, const RenderParams& rp, const Wave& w, uint32_t n_max, LaunchCounter& lc) {
    // launches whose light samples per vertex fit the shared-memory staging column take the instantiation without the thread-local one
    const bool smem_only = RT_NEE_SMEM > 0 && w.shadow_k <= NEE_SMEM;
    auto go = [&](auto kernel) { kernel<<<persistent_grid((const void*)kernel, n_max, SHADE_THREADS), SHADE_THREADS, 0, st>>>(sc, rp, w); };
    // (Diffuse-only scenes: C4's shade 60.3 -> 55.6 ms; the general instantiation lost 2.5 ms of 38.5 on CM with it and keeps both
    // stages — profiles/r4p_ab.log)
    if (sc.all_diffuse) { if (smem_only) go(k_shade<DiffuseSurface, true, 0>); else go(k_shade<DiffuseSurface, false, 0>); }
    else if (sc.any_diffuse) {   // mixed materials: the Diffuse kernel first, then the general kernel over what it left
        if (smem_only) go(k_shade<DiffuseSurface, true, 1>); else go(k_shade<DiffuseSurface, false, 1>);
        go(k_shade<Surface, false, 2>);
        lc.launches++;
    } else go(k_shade<Surface, false, 0>);
    lc.launches++;
}
void launch_shadow(cudaStream_t st, const SceneD& sc, const Wave& w, uint32_t n_max, uint32_t* fetch_counter, bool stats, LaunchCounter& lc) {
    if (stats) k_shadow<true><<<persistent_grid((const void*)k_shadow<true>, n_max), BLOCK, 0, st>>>(sc, w, fetch_counter);
    else k_shadow<false><<<persistent_grid((const void*)k_shadow<false>, n_max), BLOCK, 0, st>>>(sc, w, fetch_counter);
    lc.launches++;
}
void launch_trace(cudaStream_t st, const SceneD& sc, const float4* rays, uint32_t n, float4* hits, uint32_t* fetch_counter, LaunchCounter& lc) {
    k_trace<false><<<persistent_grid((const void*)k_trace<false>, n), BLOCK, 0, st>>>(sc, rays, n, hits, nullptr, fetch_counter);
    lc.launches++;
}
void launch_occluded(cudaStream_t st, const SceneD& sc, const float4* rays, uint32_t n, uint8_t* occluded, uint32_t* fetch_counter,
                     LaunchCounter& lc) {
    k_trace<true><<<persistent_grid((const void*)k_trace<true>, n), BLOCK, 0, st>>>(sc, rays, n, nullptr, occluded, fetch_counter);
    lc.launches++;
}
void launch_shadow_gather(cudaStream_t st, const Wave& w, uint32_t n_max, LaunchCounter& lc) {
    k_shadow_gather<<<persistent_grid((const void*)k_shadow_gather, n_max), BLOCK, 0, st>>>(w);
    lc.launches++;
}
void launch_resolve(cudaStream_t st, const Wave& w, float4* accum, LaunchCounter& lc) {
    k_resolve<<<grid_for(w.n_pixels), BLOCK, 0, st>>>(w, accum);
    lc.launches++;
}
void launch_finalize(cudaStream_t st, const uint32_t* pixel_list, uint32_t n_pixels, uint32_t width, const float4* accum, float inv_spp,
                     float* beauty, unsigned long long* stats, bool accumulate, LaunchCounter& lc) {
    if (accumulate) k_finalize<true><<<grid_for(n_pixels), BLOCK, 0, st>>>(pixel_list, n_pixels, width, accum, inv_spp, beauty, stats);
    else k_finalize<false><<<grid_for(n_pixels), BLOCK, 0, st>>>(pixel_list, n_pixels, width, accum, inv_spp, beauty, stats);
    lc.launches++;
}

// Pixel lists of a context (api.cu build_pixel_list): one block per owned tile writes the tile's pixels in Morton order
// (a warp then covers an 8x4 block of the image) at the tile's offset — the pixels inside the image for `list`, and those that
// also lie inside the scene's raster rectangle for `culled` (the beauty pass; null = nothing is culled). The host only walks the
// tiles (offsets are areas of clipped rectangles); enumerating 8 M pixels of a 4K frame on one core took 23 ms per call.
__device__ __forceinline__ uint32_t compact_even_bits(uint32_t v) {   // bits 0, 2, 4, ... of v packed together
    v &= 0x55555555u;
    v = (v | (v >> 1)) & 0x33333333u;
    v = (v | (v >> 2)) & 0x0f0f0f0fu;
    v = (v | (v >> 4)) & 0x00ff00ffu;
    v = (v | (v >> 8)) & 0x0000ffffu;
    return v;
}
__global__ void __launch_bounds__(BLOCK) k_pixel_lists(const TileRec* tiles, uint32_t tile_area, uint32_t* list, uint32_t* culled) {
    __shared__ uint32_t s_warp[BLOCK / 32][2];
    __shared__ uint32_t s_run[2];
    const TileRec t = tiles[blockIdx.x];
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, lt = (1u << lane) - 1u;
    if (threadIdx.x == 0) s_run[0] = s_run[1] = 0u;
    __syncthreads();
    for (uint32_t base = 0; base < tile_area; base += BLOCK) {
        const uint32_t m = base + threadIdx.x;
        const uint32_t x = compact_even_bits(m), y = compact_even_bits(m >> 1);
        const bool in = m < tile_area && x < t.w && y < t.h;
        const bool keep = in && culled && x >= t.cx && x < t.cx + t.cw && y >= t.cy && y < t.cy + t.ch;
        const unsigned b0 = __ballot_sync(0xffffffffu, in), b1 = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) { s_warp[warp][0] = (uint32_t)__popc(b0); s_warp[warp][1] = (uint32_t)__popc(b1); }
        __syncthreads();
        uint32_t before0 = s_run[0], before1 = s_run[1], total0 = 0, total1 = 0;
#pragma unroll
        for (int i = 0; i < BLOCK / 32; i++) {
            if (i < (int)warp) { before0 += s_warp[i][0]; before1 += s_warp[i][1]; }
            total0 += s_warp[i][0]; total1 += s_warp[i][1];
        }
        const uint32_t packed = ((t.y0 + y) << 16) | (t.x0 + x);
        if (in) list[t.off + before0 + (uint32_t)__popc(b0 & lt)] = packed;
        if (keep) culled[t.coff + before1 + (uint32_t)__popc(b1 & lt)] = packed;
        __syncthreads();
        if (threadIdx.x == 0) { s_run[0] += total0; s_run[1] += total1; }
        __syncthreads();
    }
}
void launch_pixel_lists(cudaStream_t st, const TileRec* tiles, uint32_t n_tiles, uint32_t tile_size, uint32_t* list, uint32_t* culled, LaunchCounter& lc) {
    if (!n_tiles) return;
    k_pixel_lists<<<n_tiles, BLOCK, 0, st>>>(tiles, tile_size * tile_size, list, culled);
    lc.launches++;
}

// Multi-device exchange of owned pixels (api.cu multi_*): a plane of `ch` 32-bit channels per pixel <-> the packed run of one
// rank's tiles, tile after tile, ROW-MAJOR inside a tile (the host side then moves whole tile rows). One block per tile.
// PACK reads the plane; UNPACK writes (or, for progressive sums, adds floats to) it.
template <int MODE>   // 0 pack, 1 unpack, 2 unpack-add (float)
__global__ void __launch_bounds__(BLOCK) k_pack_tiles(const TileRec* tiles, uint32_t width, uint32_t ch, uint32_t* plane, uint32_t* packed) {
    const TileRec t = tiles[blockIdx.x];
    const uint32_t row_words = t.w * ch, words = row_words * t.h;
    uint32_t* run = packed + (size_t)t.off * ch;
    for (uint32_t i = threadIdx.x; i < words; i += BLOCK) {
        const uint32_t row = i / row_words, rem = i - row * row_words;
        const size_t at = ((size_t)(t.y0 + row) * width + t.x0) * ch + rem;
        if (MODE == 0) run[i] = plane[at];
        else if (MODE == 1) plane[at] = run[i];
        else plane[at] = __float_as_uint(__uint_as_float(plane[at]) + __uint_as_float(run[i]));
    }
}
void launch_pack_tiles(cudaStream_t st, int mode, const TileRec* tiles, uint32_t n_tiles, uint32_t width, uint32_t ch, uint32_t* plane, uint32_t* packed,
                       LaunchCounter& lc) {
    if (!n_tiles) return;
    if (mode == 0) k_pack_tiles<0><<<n_tiles, BLOCK, 0, st>>>(tiles, width, ch, plane, packed);
    else if (mode == 1) k_pack_tiles<1><<<n_tiles, BLOCK, 0, st>>>(tiles, width, ch, plane, packed);
    else k_pack_tiles<2><<<n_tiles, BLOCK, 0, st>>>(tiles, width, ch, plane, packed);
    lc.launches++;
}

// ---------------------------------------------------------------------------------------------------
// BVH build kernels
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BLOCK) k_prim_setup(BuildCtx b) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    if (i < b.n) prim_setup_body(i, b);
}
__global__ void __launch_bounds__(BLOCK) k_morton(BuildCtx b) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    if (i < b.n) morton_body(i, b);
}
__global__ void __launch_bounds__(BLOCK) k_karras(BuildCtx b) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    if (i + 1 < b.n) karras_body(i, b);
}
__global__ void __launch_bounds__(BLOCK) k_refit(BuildCtx b) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    if (i < b.n) refit_body(i, b);
}
__global__ void __launch_bounds__(BLOCK) k_ploc_init(BuildCtx b) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    if (i < b.n) ploc_init_body(i, b);
}
// PLOC rounds read the cluster count and the next free node id of their round from DEVICE memory (`st`: {m, next_node}, written
// by the previous round's merge kernel into the other half of a ping-pong pair), so the host can queue several rounds behind
// each other and read the state back once per batch: a scene of 20 k triangles needs ~30 rounds, and one host round trip per
// round was most of its 2.5 ms build. The launches of a batch are sized for the batch's first round (`bound`); threads past
// the round's own count do nothing, and a round that finds a single cluster left only carries the state forward.
__global__ void __launch_bounds__(BLOCK) k_ploc_nn(BuildCtx b, const uint32_t* st) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    b.m = st[0]; b.next_node = st[1];
    if (b.m > 1 && i < b.m) ploc_nn_body(i, b);
}
__global__ void __launch_bounds__(BLOCK) k_ploc_flag(BuildCtx b, const uint32_t* st, uint32_t bound) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    b.m = st[0]; b.next_node = st[1];
    if (b.m > 1 && i < b.m) ploc_flag_body(i, b);
    else if (i < bound) b.scan[i] = 0ull;   // the scan runs over `bound` items
}
__global__ void __launch_bounds__(BLOCK) k_ploc_merge(BuildCtx b, const uint32_t* st, uint32_t* st_next) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    b.m = st[0]; b.next_node = st[1];
    if (b.m <= 1) {
        if (i == 0) { st_next[0] = b.m; st_next[1] = b.next_node; }
        return;
    }
    if (i >= b.m) return;
    ploc_merge_body(i, b);
    if (i == b.m - 1) { st_next[0] = b.ploc_out[0]; st_next[1] = b.next_node - b.ploc_out[1]; }   // (ploc_out: written by this thread just now)
}
// One wide level per launch. The level's item count is read from the device (`level[0]`), the launch is sized for an upper
// bound; a one-thread kernel then moves the next level's count (counters[0], summed by the bodies) into `level[1]`: the host
// queues several levels before it reads a count back (one round trip per level was a quarter of a small scene's build time).
__global__ void __launch_bounds__(128) k_collapse(BuildCtx b, const uint32_t* level) {
    const uint32_t i = blockIdx.x * 128 + threadIdx.x;
    if (i < level[0]) collapse_body(i, b);
}
__global__ void k_collapse_next(uint32_t* counters, uint32_t* level) {
    level[1] = counters[0];
    counters[0] = 0u;
}
void launch_prim_setup(cudaStream_t st, const BuildCtx& b, LaunchCounter& lc) { k_prim_setup<<<grid_for(b.n), BLOCK, 0, st>>>(b); lc.launches++; }
void launch_morton(cudaStream_t st, const BuildCtx& b, LaunchCounter& lc) { k_morton<<<grid_for(b.n), BLOCK, 0, st>>>(b); lc.launches++; }
void launch_karras(cudaStream_t st, const BuildCtx& b, LaunchCounter& lc) { if (b.n > 1) { k_karras<<<grid_for(b.n - 1), BLOCK, 0, st>>>(b); lc.launches++; } }
void launch_refit(cudaStream_t st, const BuildCtx& b, LaunchCounter& lc) { k_refit<<<grid_for(b.n), BLOCK, 0, st>>>(b); lc.launches++; }
void launch_collapse(cudaStream_t st, const BuildCtx& b, uint32_t bound, uint32_t* level, LaunchCounter& lc) {
    k_collapse<<<grid_for(bound, 128), 128, 0, st>>>(b, level);
    k_collapse_next<<<1, 1, 0, st>>>(b.counters, level);
    lc.launches += 2;
}

// Refit (rtcuda_scene_update). One thread per primitive slot; the bounds are min / max of order-preserving keys, exact in any
// order, so a warp reduces its keys before one lane does the six atomics (one atomic per slot on six addresses serialises).
__global__ void __launch_bounds__(BLOCK) k_refit_prims(RefitCtx r) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    V3 lo, hi;
    const bool filled = i < r.prim_slots && refit_prims_body(i, r, lo, hi);
    uint32_t k[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
    if (filled) {
        k[0] = float_key(lo.x); k[1] = float_key(lo.y); k[2] = float_key(lo.z);
        k[3] = float_key(hi.x); k[4] = float_key(hi.y); k[5] = float_key(hi.z);
    }
    if (!__any_sync(0xffffffffu, filled)) return;
#pragma unroll
    for (int a = 0; a < 3; a++) {
        k[a] = __reduce_min_sync(0xffffffffu, k[a]);
        k[3 + a] = __reduce_max_sync(0xffffffffu, k[3 + a]);
    }
    if ((threadIdx.x & 31u) == 0) {
#pragma unroll
        for (int a = 0; a < 3; a++) { atomicMin(&r.bounds_keys[a], k[a]); atomicMax(&r.bounds_keys[3 + a], k[3 + a]); }
    }
}
__global__ void __launch_bounds__(128) k_refit_nodes(RefitCtx r, uint32_t first, uint32_t count) {
    const uint32_t i = blockIdx.x * 128 + threadIdx.x;
    if (i < count) refit_nodes_body(first + i, r);
}
// per-block sums of the nodes' SAH terms (node_box[2i].w), each block over a fixed strided subset in a fixed order (the host adds
// the SAH_BLOCKS partials in block order): the same figure on every run and every GPU
__global__ void __launch_bounds__(256) k_sah_partial(const float4* node_box, uint32_t n, double* partial) {
    __shared__ double s[256];
    double v = 0.0;
    for (uint32_t i = blockIdx.x * 256 + threadIdx.x; i < n; i += SAH_BLOCKS * 256) v += (double)node_box[2 * (size_t)i].w;
    s[threadIdx.x] = v;
    __syncthreads();
    for (uint32_t o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[blockIdx.x] = s[0];
}
void launch_refit_prims(cudaStream_t st, const RefitCtx& r, LaunchCounter& lc) {
    k_refit_prims<<<grid_for(r.prim_slots), BLOCK, 0, st>>>(r);
    lc.launches++;
}
void launch_refit_nodes(cudaStream_t st, const RefitCtx& r, uint32_t first, uint32_t count, LaunchCounter& lc) {
    k_refit_nodes<<<grid_for(count, 128), 128, 0, st>>>(r, first, count);
    lc.launches++;
}
void launch_sah_partial(cudaStream_t st, const float4* node_box, uint32_t n, double* partial, LaunchCounter& lc) {
    k_sah_partial<<<SAH_BLOCKS, 256, 0, st>>>(node_box, n, partial);
    lc.launches++;
}

void launch_ploc_init(cudaStream_t st, const BuildCtx& b, LaunchCounter& lc) { k_ploc_init<<<grid_for(b.n), BLOCK, 0, st>>>(b); lc.launches++; }
size_t ploc_scan_temp_bytes(uint32_t n) {
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, bytes, (uint64_t*)nullptr, (uint64_t*)nullptr, (int)n);
    return bytes;
}
// The tail of PLOC in ONE launch: once few clusters are left (PLOC_TAIL_MAX), a single block of 1024 threads runs all remaining
// rounds itself — nearest neighbours, flags, a block-wide exclusive scan and the merge, separated by block barriers — instead
// of seven tiny dependent kernels per round. A 20 k-triangle scene needs ~30 rounds, and that chain of ~200 launches (each a few
// microseconds of latency, not of work) was half of its build time. Same per-item bodies, same order, same tree.
constexpr uint32_t PLOC_TAIL_THREADS = 1024;
__global__ void __launch_bounds__(PLOC_TAIL_THREADS) k_ploc_tail(BuildCtx b, const uint32_t* st, uint32_t* st_out, uint32_t* cl_a, uint32_t* cl_b, uint32_t in_is_a) {
    __shared__ unsigned long long s_warp[PLOC_TAIL_THREADS / 32];
    __shared__ uint32_t s_m, s_next;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (tid == 0) { s_m = st[0]; s_next = st[1]; }
    __syncthreads();
    uint32_t flip = in_is_a ? 0u : 1u;
    for (;;) {
        const uint32_t m = s_m;
        if (m <= 1u) break;
        b.m = m; b.next_node = s_next;
        b.cl_in = flip ? cl_b : cl_a;
        b.cl_out = flip ? cl_a : cl_b;
        for (uint32_t i = tid; i < m; i += PLOC_TAIL_THREADS) ploc_nn_body(i, b);
        __syncthreads();
        for (uint32_t i = tid; i < m; i += PLOC_TAIL_THREADS) ploc_flag_body(i, b);
        __syncthreads();
        // exclusive scan of b.scan[0 .. m) in place: a contiguous chunk per thread, the chunk totals scanned across the block
        const uint32_t chunk = (m + PLOC_TAIL_THREADS - 1) / PLOC_TAIL_THREADS;
        const uint32_t lo = min(m, tid * chunk), hi = min(m, lo + chunk);
        unsigned long long sum = 0;
        for (uint32_t i = lo; i < hi; i++) sum += b.scan[i];
        unsigned long long incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long up = __shfl_up_sync(0xffffffffu, incl, o);
            if ((int)lane >= o) incl += up;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            unsigned long long w = s_warp[lane];   // 32 warps
            unsigned long long wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long up = __shfl_up_sync(0xffffffffu, wi, o);
                if ((int)lane >= o) wi += up;
            }
            s_warp[lane] = wi - w;   // exclusive
        }
        __syncthreads();
        unsigned long long run = s_warp[warp] + (incl - sum);
        for (uint32_t i = lo; i < hi; i++) { const unsigned long long f = b.scan[i]; b.scan[i] = run; run += f; }
        __syncthreads();
        for (uint32_t i = tid; i < m; i += PLOC_TAIL_THREADS) ploc_merge_body(i, b);
        __syncthreads();
        if (tid == 0) { s_m = b.ploc_out[0]; s_next = b.next_node - b.ploc_out[1]; }   // (written by the thread of item m - 1, before the barrier)
        flip ^= 1u;
        __syncthreads();
        if (s_m >= m) break;   // no progress (cannot happen: the best pair is always mutual): the host sees m != 1 and reports it
    }
    if (tid == 0) { st_out[0] = s_m; st_out[1] = s_next; }
}
void launch_ploc_tail(cudaStream_t st, const BuildCtx& b, const uint32_t* state, uint32_t* state_out, uint32_t* cl_a, uint32_t* cl_b, bool in_is_a, LaunchCounter& lc) {
    k_ploc_tail<<<1, PLOC_TAIL_THREADS, 0, st>>>(b, state, state_out, cl_a, cl_b, in_is_a ? 1u : 0u);
    lc.launches++;
}

// one round; `bound` >= the round's cluster count (the count at the start of the batch), state = {m, next_node} ping-pong pair
void launch_ploc_round(cudaStream_t st, const BuildCtx& b, uint32_t bound, const uint32_t* state, uint32_t* state_next, void* scan_temp,
                       size_t scan_temp_bytes, LaunchCounter& lc) {
    k_ploc_nn<<<grid_for(bound), BLOCK, 0, st>>>(b, state);
    k_ploc_flag<<<grid_for(bound), BLOCK, 0, st>>>(b, state, bound);
    cub::DeviceScan::ExclusiveSum(scan_temp, scan_temp_bytes, b.scan, b.scan, (int)bound, st);  // library prefix sum, like the sort
    k_ploc_merge<<<grid_for(bound), BLOCK, 0, st>>>(b, state, state_next);
    lc.launches += 5;
}

// The Morton keys are sorted with the toolkit's radix sort (a library call, like cuBLAS for a GEMM);
// everything else in the build is hand-written.
size_t sort_temp_bytes(uint32_t n) {
    size_t bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const uint32_t*)nullptr,
                                    (uint32_t*)nullptr, (int)n, 0, 63);
    return bytes;
}
void launch_sort(cudaStream_t st, void* temp, size_t temp_bytes, const uint64_t* keys_in, uint64_t* keys_out, const uint32_t* vals_in,
                 uint32_t* vals_out, uint32_t n, LaunchCounter& lc) {
    cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys_in, keys_out, vals_in, vals_out, (int)n, 0, 63, st);
    lc.launches += 4;
}

__global__ void __launch_bounds__(BLOCK) k_light_tris(const ShapeD* shapes, uint32_t shape, uint32_t tri_count, const float* vertices,
                                                       const uint32_t* tris, const float* normals, LightTri* out) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    if (i < tri_count) light_tri_body(i, shapes[shape], vertices, tris, normals, out);
}
void launch_light_tris(cudaStream_t st, const ShapeD* shapes, uint32_t shape, uint32_t tri_count, const float* vertices, const uint32_t* tris,
                       const float* normals, LightTri* out, LaunchCounter& lc) {
    if (!tri_count) return;
    k_light_tris<<<grid_for(tri_count), BLOCK, 0, st>>>(shapes, shape, tri_count, vertices, tris, normals, out);
    lc.launches++;
}

// upload-time validation of a mesh's triangle indices (api.cu: validate_desc leaves this to the device)
__global__ void __launch_bounds__(BLOCK) k_check_indices(const uint32_t* idx, size_t n, uint32_t vertex_count, uint32_t* bad) {
    bool any = false;
    for (size_t i = (size_t)blockIdx.x * BLOCK + threadIdx.x; i < n; i += (size_t)gridDim.x * BLOCK) any |= idx[i] >= vertex_count;
    if (__any_sync(0xffffffffu, any) && (threadIdx.x & 31u) == 0) atomicOr(bad, 1u);
}
void launch_check_indices(cudaStream_t st, const uint32_t* idx, size_t n, uint32_t vertex_count, uint32_t* bad, LaunchCounter& lc) {
    const uint32_t grid = (uint32_t)std::min<size_t>((n + BLOCK - 1) / BLOCK, 148 * 16);
    k_check_indices<<<std::max(grid, 1u), BLOCK, 0, st>>>(idx, n, vertex_count, bad);
    lc.launches++;
}

__global__ void __launch_bounds__(BLOCK) k_shade_recs(const __grid_constant__ SceneD sc, ShadeRec* out) {
    const uint32_t i = blockIdx.x * BLOCK + threadIdx.x;
    if (i < sc.prim_count) shade_rec_body(i, sc, out);
}
void launch_shade_recs(cudaStream_t st, const SceneD& sc, ShadeRec* out, LaunchCounter& lc) {
    if (!sc.prim_count) return;
    k_shade_recs<<<grid_for(sc.prim_count), BLOCK, 0, st>>>(sc, out);
    lc.launches++;
}

// ---------------------------------------------------------------------------------------------------
// mip pyramid kernels
// ---------------------------------------------------------------------------------------------------
__global__ void k_to_f32(const uint8_t* src, uint32_t format, float* dst, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) to_f32_body(i, src, format, dst);
}
__global__ void k_resize(const float* src, float* dst, uint32_t w, uint32_t h, uint32_t ch, uint32_t n_out, int axis, uint32_t total) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < total) resize_body(i, src, dst, w, h, ch, n_out, axis);
}
__global__ void k_cast(const float* src, uint32_t format, uint8_t* dst, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) cast_body(i, src, format, dst);
}
void launch_to_f32(cudaStream_t st, const uint8_t* src, uint32_t format, float* dst, uint32_t n, LaunchCounter& lc) {
    k_to_f32<<<grid_for(n), BLOCK, 0, st>>>(src, format, dst, n);
    lc.launches++;
}
void launch_resize(cudaStream_t st, const float* src, float* dst, uint32_t w, uint32_t h, uint32_t ch, uint32_t n_out, int axis, LaunchCounter& lc) {
    const uint32_t total = axis == 0 ? n_out * w * ch : h * n_out * ch;
    k_resize<<<grid_for(total), BLOCK, 0, st>>>(src, dst, w, h, ch, n_out, axis, total);
    lc.launches++;
}
void launch_cast(cudaStream_t st, const float* src, uint32_t format, uint8_t* dst, uint32_t n, LaunchCounter& lc) {
    k_cast<<<grid_for(n), BLOCK, 0, st>>>(src, format, dst, n);
    lc.launches++;
}

}  // namespace rt
