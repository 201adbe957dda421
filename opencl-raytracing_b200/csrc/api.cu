// api.cu — the C ABI of libraytracing_cuda.so (include/rtcuda.h): context, scene upload (device BVH +
// mip pyramids), the wavefront render loop, single-pixel diagnostics, statistics.
//
// Replaces raytracing_cpu::render / render_single_pixel (crates/raytracing-cpu/src/lib.rs:645-931),
// prepare_cpu_acceleration_structures (scene.rs:14-73) and CpuRaytracingContext::new (lib.rs:81-105).
// Error handling: status codes + rtcuda_last_error() instead of the exit() of the OptiX precedent
// (crates/raytracing-optix/csrc/host/util.hpp:7-27).
#include <algorithm>
#include <chrono>
#include <cstddef>
#include <cstdlib>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/rtcuda.h"
#include "kernels.cuh"
#include "rt_cull.h"

using namespace rt;

namespace {

thread_local std::string g_last_error;

struct RtError {
    rtcuda_status status;
    std::string msg;
};

// what the device had left when an allocation failed (appended to the error text)
inline std::string oom_note(cudaError_t e) {
    if (e != cudaErrorMemoryAllocation) return "";
    cudaGetLastError();
    int dev = -1;
    size_t free_b = 0, total_b = 0;
    cudaGetDevice(&dev);
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); return ""; }
    return " (device " + std::to_string(dev) + ": " + std::to_string(free_b >> 20) + " MiB free of " + std::to_string(total_b >> 20) + ")";
}

#define CK(call)                                                                                            \
    do {                                                                                                    \
        cudaError_t e_ = (call);                                                                            \
        if (e_ != cudaSuccess) {                                                                            \
            rtcuda_status st_ = e_ == cudaErrorMemoryAllocation ? RTCUDA_ERR_OUT_OF_MEMORY : RTCUDA_ERR_CUDA; \
            throw RtError{st_, std::string(#call) + ": " + cudaGetErrorString(e_) + oom_note(e_)};            \
        }                                                                                                   \
    } while (0)

#define REQUIRE(cond, msg)                                            \
    do {                                                              \
        if (!(cond)) throw RtError{RTCUDA_ERR_INVALID_ARGUMENT, msg}; \
    } while (0)

// Device buffers come from the device's stream-ordered memory pool (cudaMallocAsync on the calling context's stream;
// the pool keeps freed blocks, rtcuda_init raises its release threshold): a one-shot render creates ~40 buffers for the
// scene and the BVH build and frees them again, and cudaMalloc / cudaFree serialise on the driver and get slow once tens
// of GB are mapped in the process.
static thread_local cudaStream_t tls_stream = nullptr;

// RTCUDA_TRACE=1: host-side wall-clock marks of the phases of a call, per thread, on stderr (diagnostic of the end-to-end path)
struct Trace {
    static bool on() { static const bool v = std::getenv("RTCUDA_TRACE") != nullptr; return v; }
    std::chrono::steady_clock::time_point t0;
    const char* what; int rank;
    Trace(const char* w, int r = 0) : t0(std::chrono::steady_clock::now()), what(w), rank(r) {}
    void mark(const char* phase) {
        if (!on()) return;
        const auto t1 = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[rtcuda trace] %s r%d %-18s %8.3f ms\n", what, rank, phase, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

// Plain (peer-mapped) device allocations released by a scene, parked per process like the path-state arenas: with peer
// access enabled between 8 GPUs a cudaMalloc / cudaFree pair of a 200 MB array costs ~10 ms (every allocation is mapped into
// seven other address spaces), which a one-shot render of a large mesh paid four times per GPU (C5 at 8 GPUs: upload + build
// 40 -> 69 ms, release 1 -> 22 ms, profiles/r4o). At most PLAIN_KEEP buffers per device stay parked.
struct PlainCache {
    struct Slot { int device; void* p; size_t bytes; };
    static constexpr size_t PLAIN_KEEP = 8;
    std::mutex mu;
    std::vector<Slot> parked;
    void* take(int device, size_t need, size_t& got) {   // best fit that wastes at most half of the block
        std::lock_guard<std::mutex> g(mu);
        int best = -1;
        for (int i = 0; i < (int)parked.size(); i++)
            if (parked[i].device == device && parked[i].bytes >= need && parked[i].bytes <= 2 * need + (1u << 20) &&
                (best < 0 || parked[i].bytes < parked[best].bytes)) best = i;
        if (best < 0) return nullptr;
        Slot sl = parked[best];
        parked.erase(parked.begin() + best);
        got = sl.bytes;
        return sl.p;
    }
    void park(int device, void* p, size_t bytes) {
        void* evict = nullptr;
        {
            std::lock_guard<std::mutex> g(mu);
            parked.push_back({device, p, bytes});
            size_t mine = 0;
            int oldest = -1;
            for (int i = 0; i < (int)parked.size(); i++) if (parked[i].device == device) { if (oldest < 0) oldest = i; mine++; }
            if (mine > PLAIN_KEEP) { evict = parked[oldest].p; parked.erase(parked.begin() + oldest); }
        }
        if (evict) cudaFree(evict);   // (the calling thread has `device` current)
    }
    void release_all() {
        std::lock_guard<std::mutex> g(mu);
        int cur = 0;
        cudaGetDevice(&cur);
        for (const Slot& sl : parked) { cudaSetDevice(sl.device); cudaFree(sl.p); }
        cudaSetDevice(cur);
        parked.clear();
    }
};
static PlainCache g_plain_cache;

// Streams of released contexts, parked per process and device: creating and destroying a stream costs ~50-100 us each, which a
// one-shot render on 8 GPUs paid 16 times per call (init 0.4 ms, shutdown 0.8 ms of a 40 ms call).
struct StreamCache {
    std::mutex mu;
    std::vector<std::pair<int, cudaStream_t>> parked;
    cudaStream_t take(int device) {
        std::lock_guard<std::mutex> g(mu);
        for (size_t i = 0; i < parked.size(); i++)
            if (parked[i].first == device) { cudaStream_t st = parked[i].second; parked.erase(parked.begin() + i); return st; }
        return nullptr;
    }
    void park(int device, cudaStream_t st) { std::lock_guard<std::mutex> g(mu); parked.push_back({device, st}); }
    void release_all() {
        std::lock_guard<std::mutex> g(mu);
        int cur = 0;
        cudaGetDevice(&cur);
        for (auto& e : parked) { cudaSetDevice(e.first); cudaStreamDestroy(e.second); }
        cudaSetDevice(cur);
        parked.clear();
    }
};
static StreamCache g_stream_cache;

template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    // `peer_visible`: a plain cudaMalloc, which other GPUs of a multi-device context can read and write once peer access is
    // enabled (cudaDeviceEnablePeerAccess maps every plain allocation). The stream-ordered pools stay private to their device:
    // with peer access granted on the pools (cudaMemPoolSetAccess) cudaMallocAsync failed with "out of memory" on boxes with
    // 150 GB free when several host threads grew peer-mapped pools at once (2-GPU test box, 8-GPU bench box, round 2).
    bool peer_visible = false, is_plain = false;
    size_t plain_bytes = 0;
    int plain_device = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    void release() {
        if (p) {
            if (is_plain) { cudaStreamSynchronize(tls_stream); g_plain_cache.park(plain_device, p, plain_bytes); }   // (no work of this stream may still touch it)
            else cudaFreeAsync(p, tls_stream);
        }
        p = nullptr;
        n = 0;
    }
    void alloc(size_t count) {
        release();
        n = count;
        is_plain = peer_visible;
        const size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
        if (is_plain) {
            cudaGetDevice(&plain_device);
            void* q = g_plain_cache.take(plain_device, bytes, plain_bytes);
            if (!q) { CK(cudaMalloc(&q, bytes)); plain_bytes = bytes; }
            p = (T*)q;
        } else CK(cudaMallocAsync((void**)&p, bytes, tls_stream));
    }
    void ensure(size_t count) {
        if (count > n || !p) alloc(count);
    }
    void upload(const T* src, size_t count, cudaStream_t st) {
        alloc(count);
        if (count) CK(cudaMemcpyAsync(p, src, count * sizeof(T), cudaMemcpyHostToDevice, st));
    }
};

M4 to_m4(const rtcuda_mat4& m) {
    M4 r;
    std::memcpy(r.m, m.m, sizeof r.m);
    return r;
}

uint32_t next_pow2(uint32_t v) {
    uint32_t p = 1;
    while (p < v) p <<= 1;
    return p;
}
bool is_pow2(uint32_t v) { return v && !(v & (v - 1)); }
uint32_t bytes_per_sample(uint32_t fmt) { return fmt == RTCUDA_IMAGE_U8 ? 1 : (fmt == RTCUDA_IMAGE_U16 ? 2 : 4); }

}  // namespace

// Path-state arena: one allocation holding every wavefront buffer of a scene. Arenas are multi-GB (the batch is
// sized for HBM, render_device) and mapping that much fresh device memory costs far more than a 1080p frame's worth
// of kernels, so a released arena is parked in a per-process cache and handed to the next scene on the same device
// (a one-shot `render(scene, settings)` call creates and destroys its context every time). rtcuda_release_cached_memory
// returns the parked memory to the driver.
struct ArenaCache {
    struct Slot { int device; void* p; size_t bytes; };
    std::mutex mu;
    std::vector<Slot> parked;
    void* take(int device, size_t need, size_t& got) {  // best fit, or null; smaller parked slots of this device are freed
        std::lock_guard<std::mutex> g(mu);
        int best = -1;
        for (int i = 0; i < (int)parked.size(); i++)
            if (parked[i].device == device && parked[i].bytes >= need && (best < 0 || parked[i].bytes < parked[best].bytes)) best = i;
        if (best >= 0) {
            Slot sl = parked[best];
            parked.erase(parked.begin() + best);
            got = sl.bytes;
            return sl.p;
        }
        for (int i = (int)parked.size() - 1; i >= 0; i--)
            if (parked[i].device == device) { cudaFree(parked[i].p); parked.erase(parked.begin() + i); }
        return nullptr;
    }
    void park(int device, void* p, size_t bytes) {
        std::lock_guard<std::mutex> g(mu);
        parked.push_back({device, p, bytes});
    }
    size_t largest(int device) {
        std::lock_guard<std::mutex> g(mu);
        size_t b = 0;
        for (const Slot& sl : parked) if (sl.device == device) b = std::max(b, sl.bytes);
        return b;
    }
    size_t parked_bytes(int device) {
        std::lock_guard<std::mutex> g(mu);
        size_t b = 0;
        for (const Slot& sl : parked) if (sl.device == device) b += sl.bytes;
        return b;
    }
    void release_all() {
        std::lock_guard<std::mutex> g(mu);
        int cur = 0;
        cudaGetDevice(&cur);
        for (const Slot& sl : parked) { cudaSetDevice(sl.device); cudaFree(sl.p); }
        cudaSetDevice(cur);
        parked.clear();
    }
};
static ArenaCache g_arena_cache;

// Pinned host staging for device -> host frames, parked per process like the arenas (a one-shot `render` creates and
// destroys its context; pinning 25 MB anew costs more than copying it). D2H into pageable memory ran at ~3 GB/s (the driver
// stages it through small bounce buffers): 8-15 ms for a 1080p beauty plane against 0.5 ms over PCIe 5 from pinned memory.
struct PinnedCache {
    struct Slot { void* p; size_t bytes; };
    std::mutex mu;
    std::vector<Slot> parked;
    void* take(size_t need, size_t& got) {
        {
            std::lock_guard<std::mutex> g(mu);
            int best = -1;
            for (int i = 0; i < (int)parked.size(); i++)
                if (parked[i].bytes >= need && (best < 0 || parked[i].bytes < parked[best].bytes)) best = i;
            if (best >= 0) {
                Slot sl = parked[best];
                parked.erase(parked.begin() + best);
                got = sl.bytes;
                return sl.p;
            }
        }
        void* p = nullptr;
        if (cudaMallocHost(&p, need) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        got = need;
        return p;
    }
    void park(void* p, size_t bytes) {
        std::lock_guard<std::mutex> g(mu);
        parked.push_back({p, bytes});
    }
    void release_all() {
        std::lock_guard<std::mutex> g(mu);
        for (const Slot& sl : parked) cudaFreeHost(sl.p);
        parked.clear();
    }
};
static PinnedCache g_pinned_cache;

// Host planes handed out by rtcuda_host_alloc (page-locked, from the cache above): a frame rendered into one of them is written
// by the GPU's copy engine directly — no staging buffer, no host memcpy, and no first-touch page faults in a freshly
// allocated frame (a new 25 MB pageable plane costs ~2.5 ms of faults and zeroing per 1080p call).
struct HostAllocs {
    std::mutex mu;
    std::map<uintptr_t, size_t> live;   // base -> bytes
    void add(void* p, size_t bytes) { std::lock_guard<std::mutex> g(mu); live[(uintptr_t)p] = bytes; }
    size_t take(void* p) {
        std::lock_guard<std::mutex> g(mu);
        auto it = live.find((uintptr_t)p);
        if (it == live.end()) return 0;
        const size_t b = it->second;
        live.erase(it);
        return b;
    }
    bool covers(const void* p, size_t bytes) {
        std::lock_guard<std::mutex> g(mu);
        auto it = live.upper_bound((uintptr_t)p);
        if (it == live.begin()) return false;
        --it;
        return (uintptr_t)p + bytes <= it->first + it->second;
    }
};
static HostAllocs g_host_allocs;

// dst <- src on up to `max_threads` host threads (a 25 MB frame: ~2.5 ms on one core)
static void parallel_memcpy(void* dst, const void* src, size_t bytes, unsigned max_threads = 4) {
    const size_t chunk = 4u << 20;
    if (bytes <= chunk || max_threads <= 1) { std::memcpy(dst, src, bytes); return; }
    const unsigned n = (unsigned)std::min<size_t>(max_threads, (bytes + chunk - 1) / chunk);
    const size_t per = ((bytes + n - 1) / n + 63) & ~(size_t)63;
    std::vector<std::thread> th;
    for (unsigned i = 1; i < n; i++) {
        const size_t lo = std::min(bytes, per * i), hi = std::min(bytes, lo + per);
        if (hi > lo) th.emplace_back([=] { std::memcpy((uint8_t*)dst + lo, (const uint8_t*)src + lo, hi - lo); });
    }
    std::memcpy(dst, src, std::min(bytes, per));
    for (std::thread& t : th) t.join();
}

struct WaveArena {
    int device = 0;
    uint8_t* base = nullptr;
    size_t bytes = 0, used = 0;
    WaveArena() = default;
    WaveArena(const WaveArena&) = delete;
    WaveArena& operator=(const WaveArena&) = delete;
    ~WaveArena() { if (base) g_arena_cache.park(device, base, bytes); }
    void reserve(int dev, size_t need) {
        used = 0;
        if (base && bytes >= need) return;
        if (base) { cudaFree(base); base = nullptr; bytes = 0; }
        device = dev;
        size_t got = 0;
        if (void* p = g_arena_cache.take(dev, need, got)) { base = (uint8_t*)p; bytes = got; return; }
        CK(cudaMalloc((void**)&base, need));
        bytes = need;
    }
    template <typename T>
    T* carve(size_t count) {
        const size_t off = (used + 255) & ~(size_t)255;
        used = off + count * sizeof(T);
        if (used > bytes) throw RtError{RTCUDA_ERR_CUDA, "path-state arena overflow"};
        return (T*)(base + off);
    }
};
template <typename T>
struct View { T* p = nullptr; size_t n = 0; };

struct rtcuda_ctx {
    int device = 0;
    rtcuda_backend_settings bs{};
    cudaStream_t stream = nullptr;
    // Multi-device context (backend_settings.num_devices > 1): one single-device context per GPU, subs[r] on device_ids[r]
    // rendering the tiles of rank r of num_devices. The parent owns no stream of its own; `device` is device_ids[0].
    std::vector<rtcuda_ctx*> subs;
};

struct rtcuda_scene {
    rtcuda_ctx* ctx = nullptr;
    SceneD sc{};
    uint32_t width = 0, height = 0;
    // scene data
    DevBuf<float> vertices, normals, uvs;
    DevBuf<uint32_t> tris;
    DevBuf<uint8_t> image_bytes;
    DevBuf<Instance> instances;
    DevBuf<ShapeD> shapes;
    DevBuf<LightD> lights;
    DevBuf<LightTri> light_tris;
    DevBuf<MaterialD> materials;
    DevBuf<float4> mat_const;
    DevBuf<TextureD> textures;
    DevBuf<ImageD> images;
    DevBuf<MipChain> mips;
    DevBuf<Node8> nodes;
    DevBuf<Prim> prims;
    DevBuf<ShadeRec> shade_recs;
    std::vector<rtcuda_light> host_lights;
    // What rtcuda_scene_update compares a new description against: the camera and the instance rows as uploaded
    rtcuda_camera host_camera{};
    std::vector<Instance> host_instances;
    std::vector<LightD> light_rows;
    uint32_t shape_count = 0, material_count = 0, texture_count = 0, image_count = 0;
    // Wide BVH levels (nodes per level, root first; level L + 1 is the contiguous node range the collapse of level L
    // allocated) and, from the first update on, every node's float box and SAH term (RefitCtx::node_box)
    std::vector<uint32_t> level_counts;
    DevBuf<float4> node_box;
    double sah_built = 0.0;   // SAH cost of the tree as last built (0: not computed yet)
    // Multi-device scene: the per-GPU scenes (subs[r] belongs to ctx->subs[r]); the parent holds nothing else of the above.
    std::vector<rtcuda_scene*> subs;
    // ... and, in each sub-scene, what the exchange of owned pixels needs (multi_* functions below): the packed planes of this
    // rank's tiles on its GPU, their pinned host mirror, the tile table (host_tiles / tiles below); on rank 0 also the other ranks'
    // tile tables and a receive buffer per rank (plain cudaMalloc: peer-accessible once peer access is enabled).
    uint32_t* packed = nullptr; size_t packed_words = 0; bool packed_plain = false;
    uint32_t* h_packed = nullptr; size_t h_packed_words = 0;
    std::vector<TileRec> host_tiles;   // the tiles this context owns (build_pixel_list), also on the device:
    DevBuf<TileRec> tiles;
    std::vector<TileRec*> peer_list; std::vector<uint32_t*> peer_recv; std::vector<size_t> peer_recv_words;
    cudaEvent_t sent = nullptr;
    // render state
    DevBuf<uint32_t> pixel_list;
    uint32_t n_my_pixels = 0;
    // The pixels of `pixel_list` whose camera rays can reach the scene bounds at all (build_pixel_list): the beauty pass
    // allocates path slots for these only. Same buffer as pixel_list when nothing is dropped.
    DevBuf<uint32_t> beauty_list_buf;
    const uint32_t* beauty_list = nullptr;
    uint32_t n_beauty_pixels = 0;
    DevBuf<float4> accum;
    WaveArena arena;
    size_t arena_capacity = 0, arena_shadow_k = 0, arena_depth = 0;
    View<PathState> state;
    View<float4> radiance, ray_o[2], ray_d[2], hits, sray_o, sray_d, scontrib;
    View<uint4> svertex;
    View<uint32_t> deferred;
    View<uint32_t> counters;
    View<unsigned long long> counters64;
    DevBuf<unsigned long long> stats_dev;
    size_t wave_bytes() const { return arena.bytes + g_arena_cache.parked_bytes(ctx->device); }  // reusable by the next render
    DevBuf<PixelOut> pixel_out;
    // host-API staging planes
    DevBuf<float> d_beauty, d_normals, d_albedo, d_uv, d_mip, d_depth;
    DevBuf<uint32_t> d_ids;
    rtcuda_stats stats{};
    LaunchCounter lc;
    // RTCUDA_STATS_KERNEL_TIMES: CUDA events around every extend / shade / shadow launch
    std::vector<cudaEvent_t> ev_pool;
    struct Span { int cls; size_t e0, e1; };
    std::vector<Span> spans;
    size_t ev_used = 0;
    // The beauty pass of a frame (every batch: raygen, extend / shade / shadow per depth, resolve; then finalize) captured as a
    // CUDA graph and replayed while the frame's key (settings, buffers, partition) stays the same: the ~330 launches of a C3
    // frame then reach the GPU in one submission, so a host thread that loses its core for tens of ms (shared box) no longer
    // leaves the GPU idle between kernels (5-40 ms gaps per 360 ms frame, profiles/r1s_gap.log).
    cudaGraphExec_t frame_exec = nullptr;
    std::vector<uint64_t> frame_key, seen_key;   // key of the instantiated graph; key of the last frame launched directly
    unsigned long long frame_launches = 0;
    bool capturing = false;
    ~rtcuda_scene() {
        if (frame_exec) cudaGraphExecDestroy(frame_exec);
        for (cudaEvent_t e : ev_pool) cudaEventDestroy(e);
        if (packed) { if (packed_plain) cudaFree(packed); else cudaFreeAsync(packed, tls_stream); }   // (the releasing thread has entered this scene's context)
        if (h_packed) g_pinned_cache.park(h_packed, h_packed_words * 4);
        for (TileRec* q : peer_list) if (q) cudaFree(q);
        for (uint32_t* q : peer_recv) if (q) cudaFree(q);
        if (sent) cudaEventDestroy(sent);
    }
};

namespace {

// Rendezvous of the per-GPU host threads of a multi-device call. A thread that fails calls fail(): every waiter (now or
// later) then returns false and unwinds, so one GPU's error cannot leave the others parked.
struct Rendezvous {
    std::mutex mu;
    std::condition_variable cv;
    int n = 1, waiting = 0;
    uint64_t phase = 0;
    bool failed = false;
    bool wait() {
        std::unique_lock<std::mutex> g(mu);
        if (failed) return false;
        const uint64_t my = phase;
        if (++waiting == n) { waiting = 0; phase++; cv.notify_all(); return true; }
        cv.wait(g, [&] { return phase != my || failed; });
        return !failed;
    }
    void fail() {
        std::lock_guard<std::mutex> g(mu);
        failed = true;
        cv.notify_all();
    }
};

// How the big geometry arrays reach N GPUs (multi-device upload): the host arrays are cut into N slices, GPU r copies slice r
// over ITS PCIe link, then forwards it to the other GPUs over NVLink (peer copies) — the host side of the transfer is paid
// once in total instead of once per GPU (16.8 M triangles: 400 MB of pageable host memory per replica).
struct GeoShare {
    int rank = 0, world = 1;
    std::vector<rtcuda_scene*>* subs = nullptr;
    Rendezvous* meet = nullptr;
};

// ---------------------------------------------------------------------------------------------------
// scene upload
// ---------------------------------------------------------------------------------------------------
void validate_desc(const rtcuda_scene_desc* d) {
    REQUIRE(d->abi_version == RTCUDA_ABI_VERSION, "scene_desc.abi_version mismatch");
    REQUIRE(d->camera.raster_width > 0 && d->camera.raster_height > 0, "empty raster");
    REQUIRE(d->camera.raster_width < 65536 && d->camera.raster_height < 65536, "raster larger than 65535");
    REQUIRE(d->camera.kind <= RTCUDA_CAMERA_THIN_LENS, "unknown camera kind");
    int mesh_mode = -1;   // 0: scene-wide arrays + offsets, 1: per-shape host arrays
    for (uint32_t i = 0; i < d->shape_count; i++) {
        const rtcuda_shape& s = d->shapes[i];
        REQUIRE(s.kind <= RTCUDA_SHAPE_SPHERE, "unknown shape kind");
        REQUIRE(s.material < d->material_count, "shape.material out of range");
        REQUIRE(s.area_light == RTCUDA_NONE || s.area_light < d->light_count, "shape.area_light out of range");
        if (s.kind == RTCUDA_SHAPE_TRIANGLE_MESH) {
            const bool own = s.vertices != nullptr;
            if (mesh_mode < 0) mesh_mode = own ? 1 : 0;
            REQUIRE(mesh_mode == (own ? 1 : 0), "either every mesh carries its own host arrays or none does");
            if (own) {
                REQUIRE(s.tris != nullptr || s.tri_count == 0, "shape.tris is NULL");
            } else {
                REQUIRE((uint64_t)s.vertex_offset + s.vertex_count <= d->vertex_count, "shape vertices out of range");
                REQUIRE((uint64_t)s.tri_offset + s.tri_count <= d->tri_count, "shape tris out of range");
                REQUIRE(s.normal_offset == RTCUDA_NONE || (uint64_t)s.normal_offset + s.vertex_count <= d->normal_count, "shape normals out of range");
                REQUIRE(s.uv_offset == RTCUDA_NONE || (uint64_t)s.uv_offset + s.vertex_count <= d->uv_count, "shape uvs out of range");
            }
            // the triangle indices themselves are checked on the device after the upload (upload_scene): 50 M host-side
            // comparisons were a tenth of the end-to-end time of the 16.8 M-triangle mesh
        }
    }
    for (uint32_t i = 0; i < d->instance_count; i++) REQUIRE(d->instances[i].shape < d->shape_count, "instance.shape out of range");
    for (uint32_t i = 0; i < d->light_count; i++) {
        const rtcuda_light& l = d->lights[i];
        REQUIRE(l.kind <= RTCUDA_LIGHT_DIFFUSE_AREA, "unknown light kind");
        if (l.kind == RTCUDA_LIGHT_DIFFUSE_AREA) {
            REQUIRE(l.shape < d->shape_count, "area light shape out of range");
            // lights.rs:59: sampling a sphere emitter is todo!() in the reference
            if (d->shapes[l.shape].kind != RTCUDA_SHAPE_TRIANGLE_MESH)
                throw RtError{RTCUDA_ERR_UNSUPPORTED, "DiffuseAreaLight over a sphere is not supported (todo!() in the reference, lights.rs:59)"};
            REQUIRE(d->shapes[l.shape].tri_count > 0, "area light mesh has no triangles");
        }
    }
    auto tex_ok = [&](uint32_t t) { return t < d->texture_count; };
    for (uint32_t i = 0; i < d->material_count; i++) {
        const rtcuda_material& m = d->materials[i];
        REQUIRE(m.kind <= RTCUDA_MATERIAL_COATED_DIFFUSE, "unknown material kind");
        switch (m.kind) {
            case RTCUDA_MATERIAL_DIFFUSE: REQUIRE(tex_ok(m.albedo), "material texture out of range"); break;
            case RTCUDA_MATERIAL_SMOOTH_DIELECTRIC: REQUIRE(tex_ok(m.eta), "material texture out of range"); break;
            case RTCUDA_MATERIAL_SMOOTH_CONDUCTOR: REQUIRE(tex_ok(m.eta) && tex_ok(m.kappa), "material texture out of range"); break;
            case RTCUDA_MATERIAL_ROUGH_DIELECTRIC: REQUIRE(tex_ok(m.eta) && tex_ok(m.roughness), "material texture out of range"); break;
            case RTCUDA_MATERIAL_ROUGH_CONDUCTOR: REQUIRE(tex_ok(m.eta) && tex_ok(m.kappa) && tex_ok(m.roughness), "material texture out of range"); break;
            default:
                REQUIRE(tex_ok(m.albedo) && tex_ok(m.eta) && tex_ok(m.thickness) && tex_ok(m.coat_albedo) &&
                            (m.roughness == RTCUDA_NONE || tex_ok(m.roughness)), "material texture out of range");
        }
    }
    for (uint32_t i = 0; i < d->texture_count; i++) {
        const rtcuda_texture& t = d->textures[i];
        REQUIRE(t.kind <= RTCUDA_TEXTURE_MIX, "unknown texture kind");
        if (t.kind == RTCUDA_TEXTURE_IMAGE) REQUIRE(t.image < d->image_count && t.filter <= 2 && t.wrap <= 2, "image texture out of range");
        // Scale / Mix operands: any texture of the scene; cycles and nesting beyond what the device evaluator unrolls
        // (TEXTURE_NEST) are refused by texture_depth at upload
        if (t.kind == RTCUDA_TEXTURE_SCALE) REQUIRE(tex_ok(t.a) && tex_ok(t.b), "scale texture operand out of range");
        if (t.kind == RTCUDA_TEXTURE_MIX) REQUIRE(tex_ok(t.a) && tex_ok(t.b) && tex_ok(t.c), "mix texture operand out of range");
    }
    for (uint32_t i = 0; i < d->image_count; i++) {
        const rtcuda_image& im = d->images[i];
        REQUIRE(im.channels >= 1 && im.channels <= 4 && im.format <= RTCUDA_IMAGE_F32 && im.width && im.height, "bad image header");
        REQUIRE(im.byte_offset + (uint64_t)im.width * im.height * im.channels * bytes_per_sample(im.format) <= d->image_byte_count, "image bytes out of range");
        REQUIRE(im.byte_offset % bytes_per_sample(im.format) == 0, "image byte_offset must be aligned to the sample size (u16: 2, f32: 4)");
    }
    REQUIRE(d->environment_light_texture == RTCUDA_NONE || tex_ok(d->environment_light_texture), "environment texture out of range");
}

// texture nesting depth (Scale / Mix): the device evaluator is bounded at TEXTURE_NEST
uint32_t texture_depth(const rtcuda_scene_desc* d, uint32_t t, uint32_t guard) {
    if (guard > 16) throw RtError{RTCUDA_ERR_UNSUPPORTED, "texture graph too deep or cyclic"};
    const rtcuda_texture& tx = d->textures[t];
    if (tx.kind == RTCUDA_TEXTURE_SCALE) return 1 + std::max(texture_depth(d, tx.a, guard + 1), texture_depth(d, tx.b, guard + 1));
    if (tx.kind == RTCUDA_TEXTURE_MIX)
        return 1 + std::max({texture_depth(d, tx.a, guard + 1), texture_depth(d, tx.b, guard + 1), texture_depth(d, tx.c, guard + 1)});
    return 0;
}

void build_mips(rtcuda_scene* s, const rtcuda_scene_desc* d, std::vector<ImageD>& images, std::vector<TextureD>& textures,
                std::vector<MipChain>& chains) {
    cudaStream_t st = s->ctx->stream;
    // which images need a pyramid (CpuTextures::new, texture.rs:214-233)
    std::vector<int> chain_of(d->image_count, -1);
    uint64_t total_bytes = d->image_byte_count;
    struct Plan { uint32_t image; uint32_t size; uint64_t offset; };
    std::vector<Plan> plans;
    for (uint32_t t = 0; t < d->texture_count; t++) {
        const rtcuda_texture& tx = d->textures[t];
        if (tx.kind != RTCUDA_TEXTURE_IMAGE || tx.filter != RTCUDA_FILTER_TRILINEAR) continue;
        if (chain_of[tx.image] < 0) {
            const rtcuda_image& im = d->images[tx.image];
            uint32_t size = im.width;
            if (!(is_pow2(im.width) && is_pow2(im.height)) || im.width != im.height) size = std::max(next_pow2(im.width), next_pow2(im.height));
            total_bytes = (total_bytes + 15) & ~15ull;
            chain_of[tx.image] = (int)plans.size();
            plans.push_back({tx.image, size, total_bytes});
            for (uint32_t lv = size; lv >= 1; lv /= 2) {
                total_bytes += ((uint64_t)lv * lv * im.channels * bytes_per_sample(im.format) + 15) & ~15ull;
                if (lv == 1) break;
            }
        }
        textures[t].mip_base = (uint32_t)chain_of[tx.image];
    }
    s->image_bytes.alloc(total_bytes);
    if (d->image_byte_count) CK(cudaMemcpyAsync(s->image_bytes.p, d->image_bytes, d->image_byte_count, cudaMemcpyHostToDevice, st));
    for (const Plan& pl : plans) {
        const rtcuda_image& im = d->images[pl.image];
        const uint32_t ch = im.channels, fmt = im.format, bps = bytes_per_sample(fmt);
        DevBuf<float> cur, tmp, nxt;
        uint32_t w = im.width, h = im.height;
        cur.alloc((size_t)w * h * ch);
        launch_to_f32(st, s->image_bytes.p + im.byte_offset, fmt, cur.p, w * h * ch, s->lc);
        if (w != pl.size || h != pl.size) {  // resize to the square power of two (vertical pass, then horizontal)
            tmp.alloc((size_t)w * pl.size * ch);
            nxt.alloc((size_t)pl.size * pl.size * ch);
            launch_resize(st, cur.p, tmp.p, w, h, ch, pl.size, 0, s->lc);
            launch_resize(st, tmp.p, nxt.p, w, pl.size, ch, pl.size, 1, s->lc);
            CK(cudaStreamSynchronize(st));
            std::swap(cur.p, nxt.p);
            std::swap(cur.n, nxt.n);
            w = h = pl.size;
        }
        MipChain mc;
        mc.first_image = (uint32_t)images.size();
        mc.level_count = 0;
        uint64_t off = pl.offset;
        for (;;) {
            ImageD lv;
            lv.width = w; lv.height = h; lv.channels = ch; lv.format = fmt; lv.byte_offset = off;
            launch_cast(st, cur.p, fmt, s->image_bytes.p + off, w * h * ch, s->lc);
            images.push_back(lv);
            mc.level_count++;
            off += ((uint64_t)w * h * ch * bps + 15) & ~15ull;
            if (!(w > 1 && h > 1)) break;
            const uint32_t nw = w / 2, nh = h / 2;
            tmp.alloc((size_t)w * nh * ch);
            nxt.alloc((size_t)nw * nh * ch);
            launch_resize(st, cur.p, tmp.p, w, h, ch, nh, 0, s->lc);
            launch_resize(st, tmp.p, nxt.p, w, nh, ch, nw, 1, s->lc);
            CK(cudaStreamSynchronize(st));
            std::swap(cur.p, nxt.p);
            std::swap(cur.n, nxt.n);
            w = nw;
            h = nh;
        }
        chains.push_back(mc);
    }
    CK(cudaStreamSynchronize(st));
}

void build_bvh(rtcuda_scene* s, const std::vector<Instance>& instances, uint32_t n_prims) {
    cudaStream_t st = s->ctx->stream;
    s->sc.prim_count = n_prims;
    s->sc.node_count = 0;
    if (n_prims == 0) {
        s->level_counts.clear();
        s->nodes.alloc(1);
        s->prims.alloc(1);
        s->sc.scene_center[0] = s->sc.scene_center[1] = s->sc.scene_center[2] = 0.0f;
        s->sc.scene_radius = 0.0f;
        set_scene_bounds(s->sc, mk3(0.0f), mk3(0.0f), false);
        return;
    }
    const uint32_t n = n_prims;
    DevBuf<Prim> prims_unsorted;
    DevBuf<float4> aabb_lo, aabb_hi, node_lo, node_hi;
    DevBuf<uint32_t> bounds_keys, vals, vals_sorted, left, right, parent, count, visit, counters, cl_a, cl_b, nn, ploc_out, ploc_state, level_count;
    DevBuf<uint64_t> keys, keys_sorted, scan;
    DevBuf<WorkItem> queue_a, queue_b;
    DevBuf<uint8_t> sort_temp, scan_temp;
    prims_unsorted.alloc(n); aabb_lo.alloc(n); aabb_hi.alloc(n);
    node_lo.alloc(2 * (size_t)n); node_hi.alloc(2 * (size_t)n);
    bounds_keys.alloc(6); vals.alloc(n); vals_sorted.alloc(n); keys.alloc(n); keys_sorted.alloc(n);
    left.alloc(n); right.alloc(n); parent.alloc(2 * (size_t)n); count.alloc(2 * (size_t)n); visit.alloc(n);
    counters.alloc(4);
    queue_a.alloc(n); queue_b.alloc(n);
    s->nodes.alloc(n);   // every wide node consumes at least one binary internal node
    // primitive slots: 3 per leaf child of the wide tree (rt_scene.h Node8), at most 3 per primitive; unfilled slots keep the
    // 0xff pattern (PRIM_HOLE)
    const size_t prim_slots = RT_FIXED_SLOTS ? 3 * (size_t)n : (size_t)n;
    REQUIRE(prim_slots < 0xffffffffull, "too many primitives");
    s->prims.alloc(prim_slots);
    const size_t temp_bytes = sort_temp_bytes(n);
    sort_temp.alloc(temp_bytes);

    const uint32_t init_keys[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
    CK(cudaMemcpyAsync(bounds_keys.p, init_keys, sizeof init_keys, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(visit.p, 0, (size_t)n * 4, st));

    BuildCtx b{};
    b.instances = s->instances.p; b.instance_count = (uint32_t)instances.size();
    b.vertices = s->vertices.p; b.tris = s->tris.p; b.n = n;
    b.prims_unsorted = prims_unsorted.p; b.aabb_lo = aabb_lo.p; b.aabb_hi = aabb_hi.p; b.bounds_keys = bounds_keys.p;
    b.keys = keys.p; b.vals = vals.p; b.keys_sorted = keys_sorted.p; b.vals_sorted = vals_sorted.p;
    b.left = left.p; b.right = right.p; b.parent = parent.p; b.count = count.p;
    b.node_lo = node_lo.p; b.node_hi = node_hi.p; b.visit = visit.p;
    b.nodes = s->nodes.p; b.prims = s->prims.p; b.counters = counters.p; b.prim_capacity = (uint32_t)prim_slots;

    launch_prim_setup(st, b, s->lc);
    launch_morton(st, b, s->lc);
    launch_sort(st, sort_temp.p, temp_bytes, keys.p, keys_sorted.p, vals.p, vals_sorted.p, n, s->lc);
    const char* builder = std::getenv("RTCUDA_BUILDER");   // A/B aid: "lbvh" selects the Karras tree + refit
    bool use_lbvh = builder && std::strcmp(builder, "lbvh") == 0;
    uint32_t h_counters[4];
  for (;;) {   // PLOC first; a tree deeper than the traversal stack covers is rebuilt as an LBVH (depth bounded by the key length)
    if (use_lbvh) {
        CK(cudaMemsetAsync(visit.p, 0, (size_t)n * 4, st));
        launch_karras(st, b, s->lc);
        launch_refit(st, b, s->lc);
    } else {
        // PLOC: one round = nearest neighbours, flags, scan, merge + compaction; the host reads back the new cluster count
        cl_a.alloc(n); cl_b.alloc(n); nn.alloc(n); scan.alloc(n); ploc_out.alloc(2);
        const size_t scan_bytes = ploc_scan_temp_bytes(n);
        scan_temp.alloc(scan_bytes);
        b.nn = nn.p; b.scan = scan.p; b.ploc_out = ploc_out.p;
        b.cl_out = cl_a.p;
        launch_ploc_init(st, b, s->lc);
        uint32_t* cin = cl_a.p;
        uint32_t* cout = cl_b.p;
        b.m = n; b.next_node = n - 1;
        // rounds are queued in batches with the round state on the device (kernels.cu k_ploc_*): one read-back per batch.
        // Large inputs go round by round (their launches are sized for the batch's first round, and every round halves the count).
        ploc_state.alloc(4);
        uint32_t h_state[2] = {b.m, b.next_node};
        CK(cudaMemcpyAsync(ploc_state.p, h_state, sizeof h_state, cudaMemcpyHostToDevice, st));
        uint32_t flip = 0;
        while (b.m > 1) {
            if (b.m <= PLOC_TAIL_MAX && !std::getenv("RTCUDA_NO_PLOC_TAIL")) {   // (the variable is an A/B aid)
                // few clusters left: one block runs all remaining rounds in a single launch
                launch_ploc_tail(st, b, ploc_state.p + 2 * flip, ploc_state.p + 2 * (flip ^ 1u), cl_a.p, cl_b.p, cin == cl_a.p, s->lc);
                flip ^= 1u;
                CK(cudaMemcpyAsync(h_state, ploc_state.p + 2 * flip, sizeof h_state, cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st));
                if (h_state[0] != 1u) throw RtError{RTCUDA_ERR_CUDA, "PLOC tail did not finish"};
                b.m = h_state[0]; b.next_node = h_state[1];
                break;
            }
            const uint32_t batch = b.m > (1u << 20) ? 1u : (b.m > (1u << 16) ? 4u : 8u), bound = b.m;
            for (uint32_t r = 0; r < batch; r++) {
                b.cl_in = cin; b.cl_out = cout;
                launch_ploc_round(st, b, bound, ploc_state.p + 2 * flip, ploc_state.p + 2 * (flip ^ 1u), scan_temp.p, scan_bytes, s->lc);
                flip ^= 1u;
                std::swap(cin, cout);
            }
            CK(cudaMemcpyAsync(h_state, ploc_state.p + 2 * flip, sizeof h_state, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (h_state[0] >= b.m) throw RtError{RTCUDA_ERR_CUDA, "PLOC round made no progress"};
            b.m = h_state[0]; b.next_node = h_state[1];
        }
    }

    // collapse, one launch per wide level
    CK(cudaMemsetAsync(s->prims.p, 0xff, prim_slots * sizeof(Prim), st));
    WorkItem root{0u, 0u};
    CK(cudaMemcpyAsync(queue_a.p, &root, sizeof root, cudaMemcpyHostToDevice, st));
    h_counters[0] = 0u; h_counters[1] = 1u; h_counters[2] = 0u; h_counters[3] = 0u;  // next-level size, wide nodes (root allocated), packed prims
    CK(cudaMemcpyAsync(counters.p, h_counters, sizeof h_counters, cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));   // h_counters is reused as the read-back target below
    uint32_t n_items = 1, n_levels = 0;
    bool too_deep = false;
    WorkItem* qin = queue_a.p;
    WorkItem* qout = queue_b.p;
    // item counts per level live on the device (level_count[L]); the host queues up to 4 levels per read-back, each launch sized
    // for an upper bound of its level (8^L items, never more than n)
    constexpr uint32_t MAX_LEVELS = (uint32_t)(TRAVERSE_STACK / 2 - 1);
    level_count.alloc(MAX_LEVELS + 8);
    CK(cudaMemsetAsync(level_count.p, 0, (MAX_LEVELS + 8) * 4, st));
    const uint32_t one = 1;
    CK(cudaMemcpyAsync(level_count.p, &one, 4, cudaMemcpyHostToDevice, st));
    uint64_t bound = 1;
    while (n_items) {
        uint32_t queued = 0;
        for (; queued < 4; queued++) {
            // a ray holds at most two stack entries per level of the wide tree (the rest of a node group and a postponed
            // primitive group, rt_traverse.h): deeper trees than the traversal stack covers are refused, not overrun
            if (n_levels + queued + 1 > MAX_LEVELS) break;
            b.queue_in = qin;
            b.queue_out = qout;
            launch_collapse(st, b, (uint32_t)std::min<uint64_t>(bound, n), level_count.p + n_levels + queued, s->lc);
            bound = std::min<uint64_t>(bound * 8, n);
            std::swap(qin, qout);
        }
        if (!queued) { too_deep = true; break; }
        uint32_t h_levels[5] = {0, 0, 0, 0, 0};   // counts of the levels just run ([0]) .. of the level after them ([queued])
        CK(cudaMemcpyAsync(h_levels, level_count.p + n_levels, (queued + 1) * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        n_items = h_levels[queued];
        for (uint32_t k = 1; k <= queued; k++) if (h_levels[k] == 0) { n_items = 0; queued = k; break; }   // levels past the last one ran empty
        n_levels += queued;
    }
    CK(cudaMemcpyAsync(h_counters, counters.p, sizeof h_counters, cudaMemcpyDeviceToHost, st));
    s->level_counts.resize(n_levels);
    CK(cudaMemcpyAsync(s->level_counts.data(), level_count.p, n_levels * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (!use_lbvh && std::getenv("RTCUDA_TEST_PLOC_TOO_DEEP")) too_deep = true;   // test hook for the fallback below
    if (!too_deep) break;
    if (use_lbvh) throw RtError{RTCUDA_ERR_UNSUPPORTED, "wide BVH deeper than the traversal stack allows (degenerate primitive distribution)"};
    use_lbvh = true;
    s->stats.bvh_fallback_lbvh = 1;
  }
    if (h_counters[3] != n || h_counters[2] > prim_slots) throw RtError{RTCUDA_ERR_CUDA, "BVH build lost primitives"};
    s->sc.prim_count = h_counters[2];   // primitive SLOTS (holes included): what shade records and bounds checks range over
    s->sc.node_count = h_counters[1];
    s->stats.bvh_node_count = h_counters[1];
    s->stats.bvh_prim_count = n;

    // CpuRaytracingContext::new (lib.rs:81-105): centre / radius of the root bounds (aabb.rs:27-33); a
    // single-primitive scene has a leaf root with infinite bounds in the reference (bvh2.rs:448-452)
    uint32_t hk[6];
    CK(cudaMemcpyAsync(hk, bounds_keys.p, sizeof hk, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    V3 mn = mk3(key_float(hk[0]), key_float(hk[1]), key_float(hk[2])), mx = mk3(key_float(hk[3]), key_float(hk[4]), key_float(hk[5]));
    V3 c = (mx + mn) / 2.0f;
    s->sc.scene_center[0] = c.x; s->sc.scene_center[1] = c.y; s->sc.scene_center[2] = c.z;
    s->sc.scene_radius = n == 1 ? INFINITY : length(mx - c);
    set_scene_bounds(s->sc, mn, mx, true);
}

void upload_scene(rtcuda_scene* s, const rtcuda_scene_desc* d, const GeoShare* share = nullptr) {
    cudaStream_t st = s->ctx->stream;
    Trace tr("upload", share ? share->rank : 0);
    validate_desc(d);
    for (uint32_t m = 0; m < d->material_count; m++) {
        const rtcuda_material& mm = d->materials[m];
        const uint32_t ids[6] = {mm.albedo, mm.eta, mm.kappa, mm.roughness, mm.thickness, mm.coat_albedo};
        for (uint32_t t : ids)
            if (t != RTCUDA_NONE && t < d->texture_count && texture_depth(d, t, 0) > (uint32_t)TEXTURE_NEST)
                throw RtError{RTCUDA_ERR_UNSUPPORTED, "texture nesting deeper than the device evaluator supports"};
    }
    if (d->environment_light_texture != RTCUDA_NONE && texture_depth(d, d->environment_light_texture, 0) > (uint32_t)TEXTURE_NEST)
        throw RtError{RTCUDA_ERR_UNSUPPORTED, "environment texture nesting deeper than the device evaluator supports"};
    cudaEvent_t e0, e1, e2;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1)); CK(cudaEventCreate(&e2));
    CK(cudaEventRecord(e0, st));

    s->width = d->camera.raster_width;
    s->height = d->camera.raster_height;
    CameraD& cam = s->sc.camera;
    cam.kind = d->camera.kind; cam.width = s->width; cam.height = s->height;
    cam.near_clip = d->camera.near_clip; cam.far_clip = d->camera.far_clip;
    cam.aperture_radius = d->camera.aperture_radius; cam.focal_distance = d->camera.focal_distance;
    cam.raster_to_camera = to_m4(d->camera.raster_to_camera.forward);
    cam.camera_to_world = to_m4(d->camera.camera_to_world.forward);

    // Geometry: either the scene-wide arrays as given, or every mesh's own arrays packed behind each other on the device
    // (offsets assigned here). `rs` is the shape table with resolved offsets.
    std::vector<rtcuda_shape> rs(d->shapes, d->shapes + d->shape_count);
    bool own_arrays = false;
    for (const rtcuda_shape& a : rs) own_arrays |= a.kind == RTCUDA_SHAPE_TRIANGLE_MESH && a.vertices != nullptr;
    struct Piece { int which; size_t dst_off; const void* src; size_t bytes; };   // which: 0 vertices, 1 tris, 2 normals, 3 uvs (byte offsets)
    std::vector<Piece> pieces;
    constexpr size_t SHARE_MIN = 4u << 20;   // smaller arrays: every GPU reads the host copy itself
    const bool sharing = share && share->world > 1;
    // arrays that hold a piece the GPUs pass between them live in plain (peer-mapped) allocations
    auto geo_alloc = [&](auto& buf, size_t count, size_t elem_bytes, size_t largest_piece_bytes) {
        (void)elem_bytes;
        buf.peer_visible = sharing && largest_piece_bytes >= SHARE_MIN;
        buf.alloc(count);
    };
    if (!own_arrays) {
        geo_alloc(s->vertices, d->vertex_count * 3, 4, d->vertex_count * 12); geo_alloc(s->tris, d->tri_count * 3, 4, d->tri_count * 12);
        geo_alloc(s->normals, d->normal_count * 3, 4, d->normal_count * 12); geo_alloc(s->uvs, d->uv_count * 2, 4, d->uv_count * 8);
        pieces.push_back({0, 0, d->vertices, d->vertex_count * 12});
        pieces.push_back({1, 0, d->tris, d->tri_count * 12});
        pieces.push_back({2, 0, d->normals, d->normal_count * 12});
        pieces.push_back({3, 0, d->uvs, d->uv_count * 8});
    } else {
        uint64_t nv = 0, nt = 0, nn = 0, nuv = 0;
        for (rtcuda_shape& a : rs) {
            if (a.kind != RTCUDA_SHAPE_TRIANGLE_MESH) continue;
            a.vertex_offset = (uint32_t)nv; a.tri_offset = (uint32_t)nt;
            a.normal_offset = a.normals ? (uint32_t)nn : RTCUDA_NONE;
            a.uv_offset = a.uvs ? (uint32_t)nuv : RTCUDA_NONE;
            nv += a.vertex_count; nt += a.tri_count;
            if (a.normals) nn += a.vertex_count;
            if (a.uvs) nuv += a.vertex_count;
            REQUIRE(nv < 0xffffffffull && nt < 0xffffffffull, "too many vertices / triangles");
        }
        size_t big_v = 0, big_t = 0, big_n = 0, big_uv = 0;   // the largest piece of each array
        for (const rtcuda_shape& a : rs) {
            if (a.kind != RTCUDA_SHAPE_TRIANGLE_MESH) continue;
            big_v = std::max<size_t>(big_v, (size_t)a.vertex_count * 12); big_t = std::max<size_t>(big_t, (size_t)a.tri_count * 12);
            if (a.normals) big_n = std::max<size_t>(big_n, (size_t)a.vertex_count * 12);
            if (a.uvs) big_uv = std::max<size_t>(big_uv, (size_t)a.vertex_count * 8);
        }
        geo_alloc(s->vertices, nv * 3, 4, big_v); geo_alloc(s->tris, nt * 3, 4, big_t); geo_alloc(s->normals, nn * 3, 4, big_n); geo_alloc(s->uvs, nuv * 2, 4, big_uv);
        for (const rtcuda_shape& a : rs) {
            if (a.kind != RTCUDA_SHAPE_TRIANGLE_MESH) continue;
            pieces.push_back({0, (size_t)a.vertex_offset * 12, a.vertices, (size_t)a.vertex_count * 12});
            pieces.push_back({1, (size_t)a.tri_offset * 12, a.tris, (size_t)a.tri_count * 12});
            if (a.normals) pieces.push_back({2, (size_t)a.normal_offset * 12, a.normals, (size_t)a.vertex_count * 12});
            if (a.uvs) pieces.push_back({3, (size_t)a.uv_offset * 8, a.uvs, (size_t)a.vertex_count * 8});
        }
    }
    {
        auto base_of = [](rtcuda_scene* q, int which) -> uint8_t* {
            return which == 0 ? (uint8_t*)q->vertices.p : which == 1 ? (uint8_t*)q->tris.p : which == 2 ? (uint8_t*)q->normals.p : (uint8_t*)q->uvs.p;
        };
        const bool shared = sharing;
        if (shared) {   // every GPU's arrays must exist before anybody writes into them
            CK(cudaStreamSynchronize(st));
            if (!share->meet->wait()) throw RtError{RTCUDA_ERR_CUDA, "another device failed during the upload"};
        }
        for (const Piece& pc : pieces) {
            if (!pc.bytes) continue;
            if (!shared || pc.bytes < SHARE_MIN) {
                CK(cudaMemcpyAsync(base_of(s, pc.which) + pc.dst_off, pc.src, pc.bytes, cudaMemcpyHostToDevice, st));
                continue;
            }
            const size_t world = (size_t)share->world, slice = ((pc.bytes + world - 1) / world + 255) & ~(size_t)255;
            const size_t lo = std::min(pc.bytes, slice * (size_t)share->rank), hi = std::min(pc.bytes, lo + slice);
            if (hi == lo) continue;
            uint8_t* mine = base_of(s, pc.which) + pc.dst_off + lo;
            CK(cudaMemcpyAsync(mine, (const uint8_t*)pc.src + lo, hi - lo, cudaMemcpyHostToDevice, st));
            for (int q = 0; q < share->world; q++) {
                if (q == share->rank) continue;
                rtcuda_scene* other = (*share->subs)[q];
                CK(cudaMemcpyPeerAsync(base_of(other, pc.which) + pc.dst_off + lo, other->ctx->device, mine, s->ctx->device, hi - lo, st));
            }
        }
        if (shared) {   // all slices have arrived everywhere
            CK(cudaStreamSynchronize(st));
            if (!share->meet->wait()) throw RtError{RTCUDA_ERR_CUDA, "another device failed during the upload"};
        }
    }
    tr.mark("geometry");
    {   // triangle indices must stay inside their mesh: checked on the device, one flag read back
        DevBuf<uint32_t> bad;
        bad.alloc(1);
        CK(cudaMemsetAsync(bad.p, 0, 4, st));
        for (const rtcuda_shape& a : rs)
            if (a.kind == RTCUDA_SHAPE_TRIANGLE_MESH && a.tri_count)
                launch_check_indices(st, s->tris.p + (size_t)a.tri_offset * 3, (size_t)a.tri_count * 3, a.vertex_count, bad.p, s->lc);
        uint32_t h_bad = 0;
        CK(cudaMemcpyAsync(&h_bad, bad.p, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        REQUIRE(h_bad == 0, "triangle index out of range");
    }

    std::vector<ShapeD> shapes(d->shape_count);
    for (uint32_t i = 0; i < d->shape_count; i++) {
        const rtcuda_shape& a = rs[i];
        ShapeD& b = shapes[i];
        b.kind = a.kind; b.material = a.material; b.area_light = a.area_light;
        b.vertex_offset = a.vertex_offset; b.vertex_count = a.vertex_count; b.tri_offset = a.tri_offset; b.tri_count = a.tri_count;
        b.normal_offset = a.normal_offset; b.uv_offset = a.uv_offset;
        std::memcpy(b.center, a.center, sizeof b.center);
        b.radius = a.radius;
    }
    std::vector<Instance> instances(d->instance_count);
    uint64_t n_prims = 0;
    for (uint32_t i = 0; i < d->instance_count; i++) {
        const rtcuda_instance& a = d->instances[i];
        const rtcuda_shape& sh = rs[a.shape];
        Instance& b = instances[i];
        std::memset(&b, 0, sizeof b);
        b.o2w = to_m4(a.object_to_world.forward);
        b.w2o = to_m4(a.object_to_world.inverse);
        b.shape = a.shape; b.kind = sh.kind; b.material = sh.material; b.area_light = sh.area_light;
        b.vertex_offset = sh.vertex_offset; b.tri_offset = sh.tri_offset; b.normal_offset = sh.normal_offset; b.uv_offset = sh.uv_offset;
        b.tri_count = sh.tri_count;
        b.prim_base = (uint32_t)n_prims;
        std::memcpy(b.center, sh.center, sizeof b.center);
        b.radius = sh.radius;
        n_prims += sh.kind == RTCUDA_SHAPE_TRIANGLE_MESH ? sh.tri_count : 1;
        REQUIRE(n_prims < 0x7fffffffull, "too many primitives");
    }
    // instances without primitives (empty meshes) would break the prim -> instance search: give them an
    // empty range that the search skips (prim_base is non-decreasing; the LAST instance with base <= i wins)
    std::vector<LightD> lights(d->light_count);
    uint64_t n_light_tris = 0;
    for (uint32_t i = 0; i < d->light_count; i++) {
        const rtcuda_light& a = d->lights[i];
        LightD& b = lights[i];
        b.kind = a.kind; b.shape = a.shape;
        std::memcpy(b.a, a.position_or_direction, sizeof b.a);
        std::memcpy(b.b, a.intensity_or_radiance, sizeof b.b);
        b.light_to_world = to_m4(a.light_to_world);
        b.tri_table = 0;
        if (a.kind == RTCUDA_LIGHT_DIFFUSE_AREA) {
            b.tri_table = (uint32_t)n_light_tris;
            n_light_tris += d->shapes[a.shape].tri_count;
        }
    }
    s->host_lights.assign(d->lights, d->lights + d->light_count);
    s->host_camera = d->camera;
    s->host_instances = instances;
    s->light_rows = lights;
    s->shape_count = d->shape_count; s->material_count = d->material_count; s->texture_count = d->texture_count; s->image_count = d->image_count;
    std::vector<MaterialD> materials(d->material_count);
    for (uint32_t i = 0; i < d->material_count; i++) {
        const rtcuda_material& a = d->materials[i];
        materials[i] = MaterialD{a.kind, a.remap_roughness, a.albedo, a.eta, a.kappa, a.roughness, a.thickness, a.coat_albedo};
    }
    std::vector<TextureD> textures(d->texture_count);
    for (uint32_t i = 0; i < d->texture_count; i++) {
        const rtcuda_texture& a = d->textures[i];
        TextureD& b = textures[i];
        b.kind = a.kind; b.image = a.image; b.filter = a.filter; b.wrap = a.wrap; b.a = a.a; b.b = a.b; b.c = a.c; b.mip_base = NONE;
        std::memcpy(b.value, a.value, sizeof b.value);
        std::memcpy(b.value2, a.value2, sizeof b.value2);
    }
    std::vector<ImageD> images(d->image_count);
    for (uint32_t i = 0; i < d->image_count; i++) {
        const rtcuda_image& a = d->images[i];
        images[i] = ImageD{a.width, a.height, a.channels, a.format, a.byte_offset};
    }
    std::vector<MipChain> chains;
    build_mips(s, d, images, textures, chains);

    s->shapes.upload(shapes.data(), shapes.size(), st);
    s->instances.upload(instances.data(), instances.size(), st);
    s->lights.upload(lights.data(), lights.size(), st);
    s->materials.upload(materials.data(), materials.size(), st);
    s->textures.upload(textures.data(), textures.size(), st);
    s->images.upload(images.data(), images.size(), st);
    s->mips.upload(chains.data(), chains.size(), st);
    s->light_tris.alloc(n_light_tris);
    for (uint32_t i = 0; i < d->light_count; i++)
        if (lights[i].kind == RTCUDA_LIGHT_DIFFUSE_AREA)
            launch_light_tris(st, s->shapes.p, lights[i].shape, shapes[lights[i].shape].tri_count, s->vertices.p, s->tris.p, s->normals.p,
                              s->light_tris.p + lights[i].tri_table, s->lc);
    // constant albedo per material (SceneD::mat_const)
    std::vector<float4> mat_const(d->material_count, make_float4(0.0f, 0.0f, 0.0f, 0.0f));
    for (uint32_t i = 0; i < d->material_count; i++) {
        if (d->materials[i].kind != RTCUDA_MATERIAL_DIFFUSE) continue;   // w = 0
        const uint32_t t = d->materials[i].albedo;
        mat_const[i].w = 2.0f;
        if (t != RTCUDA_NONE && t < d->texture_count && d->textures[t].kind == RTCUDA_TEXTURE_CONSTANT)
            mat_const[i] = make_float4(d->textures[t].value[0], d->textures[t].value[1], d->textures[t].value[2], 1.0f);
    }
    s->mat_const.upload(mat_const.data(), mat_const.size(), st);
    CK(cudaStreamSynchronize(st));  // host vectors die at scope end
    CK(cudaEventRecord(e1, st));
    tr.mark("tables+mips");

    SceneD& sc = s->sc;
    sc.instances = s->instances.p; sc.shapes = s->shapes.p; sc.lights = s->lights.p; sc.light_tris = s->light_tris.p; sc.materials = s->materials.p;
    sc.textures = s->textures.p; sc.images = s->images.p; sc.mips = s->mips.p; sc.image_bytes = s->image_bytes.p;
    sc.vertices = s->vertices.p; sc.tris = s->tris.p; sc.normals = s->normals.p; sc.uvs = s->uvs.p;
    sc.instance_count = d->instance_count; sc.light_count = d->light_count; sc.material_count = d->material_count;
    sc.texture_count = d->texture_count; sc.env_texture = d->environment_light_texture;
    sc.mat_const = d->material_count ? s->mat_const.p : nullptr;
    sc.use_light0 = 0;
    if (d->light_count) {   // light 0 rides in the kernel parameter block (SceneD::light0)
        sc.light0 = lights[0];
        sc.light0_tri_count = lights[0].kind == RTCUDA_LIGHT_DIFFUSE_AREA ? shapes[lights[0].shape].tri_count : 0u;
        sc.light0_has_normals = lights[0].kind == RTCUDA_LIGHT_DIFFUSE_AREA && shapes[lights[0].shape].normal_offset != NONE ? 1u : 0u;
        sc.use_light0 = std::getenv("RTCUDA_NO_LIGHT0") ? 0u : 1u;   // (the variable is an A/B aid)
    }
    sc.watertight = (s->ctx->bs.flags & RTCUDA_BACKEND_WATERTIGHT) ? 1u : 0u;
    sc.all_diffuse = 1;
    sc.any_diffuse = 0;
    for (uint32_t m = 0; m < d->material_count; m++) {
        if (d->materials[m].kind != RTCUDA_MATERIAL_DIFFUSE) sc.all_diffuse = 0;
        else sc.any_diffuse = 1;
    }
    if (std::getenv("RTCUDA_NO_MATERIAL_SPLIT")) sc.any_diffuse = sc.all_diffuse;   // (A/B aid: mixed scenes through the general kernel only)
    sc.tex_uses_derivs = 0;
    for (uint32_t t = 0; t < d->texture_count; t++)
        if (d->textures[t].kind == RTCUDA_TEXTURE_IMAGE || d->textures[t].kind == RTCUDA_TEXTURE_CHECKER) sc.tex_uses_derivs = 1;

    build_bvh(s, instances, (uint32_t)n_prims);
    sc.nodes = s->nodes.p;
    sc.prims = s->prims.p;
    sc.shade_recs = nullptr;
    if (n_prims) {
        s->shade_recs.alloc(sc.prim_count);
        launch_shade_recs(st, sc, s->shade_recs.p, s->lc);
        sc.shade_recs = s->shade_recs.p;
    }
    CK(cudaEventRecord(e2, st));
    CK(cudaStreamSynchronize(st));
    tr.mark("bvh");
    float ms_up = 0, ms_build = 0;
    CK(cudaEventElapsedTime(&ms_up, e0, e1));
    CK(cudaEventElapsedTime(&ms_build, e1, e2));
    s->stats.upload_ms = ms_up;
    s->stats.bvh_build_ms = ms_build;
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(e2);
}

// ---------------------------------------------------------------------------------------------------
// pixel list: the pixels this context renders, in a ray-coherent order
// ---------------------------------------------------------------------------------------------------
// Square tiles (64x64 unless backend_settings.tile_size says otherwise) in row-major tile order (create_render_jobs,
// lib.rs:481-504), tile i belongs to this context iff i % tile_world == tile_rank; inside a tile pixels follow a
// Morton curve so that a warp covers an 8x4 block of the image.
void build_pixel_list(rtcuda_scene* s) {
    cudaStream_t st = s->ctx->stream;
    const uint32_t W = s->width, H = s->height, TS = s->ctx->bs.tile_size ? s->ctx->bs.tile_size : 64u;
    const uint32_t tiles_x = (W + TS - 1) / TS, tiles_y = (H + TS - 1) / TS;
    const uint32_t world = std::max(1u, s->ctx->bs.tile_world), rank = s->ctx->bs.tile_rank;
    // Round-robin over the row-major tile index — with one idle slot per tile row when the row length is a multiple of the
    // world size: otherwise every rank would own whole tile COLUMNS and a scene that covers 7.5 periods of them gives half
    // the ranks 8 heavy columns and the other half 7 (C3 at 8 ranks: 37.8 vs 41.5 ms per frame, profiles/r2m_bench_c3_n8.json).
    const uint32_t stride = tiles_x + (world > 1 && tiles_x % world == 0 ? 1u : 0u);
    int rect[4] = {0, 0, (int)W - 1, (int)H - 1};
    const bool cull = !std::getenv("RTCUDA_NO_PIXEL_CULL") && scene_raster_rect(s->sc, rect);   // (the variable is an A/B aid)
    // The host walks the tiles only (offsets are areas of clipped rectangles); the pixels themselves are enumerated on the
    // device, one block per tile (k_pixel_lists).
    std::vector<TileRec>& tiles = s->host_tiles;
    tiles.clear();
    uint64_t n_all = 0, n_kept = 0;
    for (uint32_t ty = 0; ty < tiles_y; ty++)
        for (uint32_t tx = 0; tx < tiles_x; tx++) {
            if ((ty * stride + tx) % world != rank) continue;
            TileRec t{};
            t.x0 = tx * TS; t.y0 = ty * TS;
            t.w = std::min(TS, W - t.x0); t.h = std::min(TS, H - t.y0);
            t.off = (uint32_t)n_all;
            const int lo_x = std::max(rect[0], (int)t.x0), hi_x = std::min(rect[2] + 1, (int)(t.x0 + t.w));
            const int lo_y = std::max(rect[1], (int)t.y0), hi_y = std::min(rect[3] + 1, (int)(t.y0 + t.h));
            if (hi_x > lo_x && hi_y > lo_y) { t.cx = (uint32_t)lo_x - t.x0; t.cy = (uint32_t)lo_y - t.y0; t.cw = (uint32_t)(hi_x - lo_x); t.ch = (uint32_t)(hi_y - lo_y); }
            t.coff = (uint32_t)n_kept;
            n_all += (uint64_t)t.w * t.h;
            n_kept += (uint64_t)t.cw * t.ch;
            tiles.push_back(t);
        }
    s->n_my_pixels = (uint32_t)n_all;
    s->tiles.upload(tiles.data(), tiles.size(), st);
    s->pixel_list.alloc(n_all);
    const bool drop = cull && n_kept != n_all;
    if (drop) s->beauty_list_buf.alloc(n_kept);
    launch_pixel_lists(st, s->tiles.p, (uint32_t)tiles.size(), TS, s->pixel_list.p, drop ? s->beauty_list_buf.p : nullptr, s->lc);
    s->beauty_list = drop ? s->beauty_list_buf.p : s->pixel_list.p;
    s->n_beauty_pixels = drop ? (uint32_t)n_kept : s->n_my_pixels;
    CK(cudaStreamSynchronize(st));   // (the tile table was uploaded from a vector that may be rebuilt)
}

RenderParams make_params(const rtcuda_settings* st) {
    RenderParams rp{};
    rp.max_ray_depth = st->max_ray_depth;
    rp.accumulate_bounces = st->accumulate_bounces;
    rp.light_sample_count = st->light_sample_count;
    rp.samples_per_pixel = st->samples_per_pixel;
    rp.antialias_primary_rays = st->antialias_primary_rays;
    rp.sampler.seed_hashed = hash_seed(st->has_seed ? st->seed : 42ull);  // sample.rs:30-35
    rp.sampler.stratified = st->sampler_kind == RTCUDA_SAMPLER_STRATIFIED;
    rp.sampler.jitter = st->stratified_jitter;
    rp.sampler.x_strata = st->x_strata;
    rp.sampler.y_strata = st->y_strata;
    return rp;
}

uint32_t shadow_entries_per_vertex(const rtcuda_scene* s, const RenderParams& rp) {
    uint64_t k = 0;
    for (const rtcuda_light& l : s->host_lights) k += l.kind == RTCUDA_LIGHT_DIFFUSE_AREA ? rp.light_sample_count : 1;
    REQUIRE(k < (1u << 20), "too many light samples per path vertex");
    return (uint32_t)k;
}

// Bytes of path state for `cap` slots (every buffer ensure_wave carves, plus alignment slack).
size_t arena_bytes(size_t cap, uint32_t shadow_k, uint32_t max_depth) {
    const size_t k = std::max(1u, shadow_k), n_counters = 4 * ((size_t)max_depth + 3);
    return cap * (16 + 16 * 7 + 16 + 4) + cap * k * 48 + n_counters * 4 + ((size_t)max_depth + 3) * 8 + 16 * 256;
}

// Allocate the wavefront state for `capacity` path slots. Returns whether the buffers were carved anew (their addresses may have
// changed even when the arena's base did not).
bool ensure_wave(rtcuda_scene* s, uint32_t capacity, uint32_t shadow_k, uint32_t max_depth) {
    s->stats_dev.ensure(STAT_TOTAL);
    const size_t k = std::max(1u, shadow_k), n_counters = 4 * ((size_t)max_depth + 3);
    if (s->arena.base && capacity <= s->arena_capacity && k <= s->arena_shadow_k && max_depth <= s->arena_depth) return false;
    const size_t cap = capacity;
    REQUIRE((uint64_t)cap * k < (1ull << 32), "paths in flight x light samples per vertex must stay below 2^32");
    const size_t need = arena_bytes(cap, shadow_k, max_depth);
    s->arena.reserve(s->ctx->device, need);
    auto view = [&](auto& v, size_t count) { v.p = s->arena.carve<std::remove_pointer_t<decltype(v.p)>>(count); v.n = count; };
    view(s->state, cap);
    view(s->radiance, cap);
    for (int i = 0; i < 2; i++) { view(s->ray_o[i], cap); view(s->ray_d[i], cap); }
    view(s->hits, cap);
    view(s->svertex, cap);
    view(s->deferred, cap);
    view(s->sray_o, cap * k);
    view(s->sray_d, cap * k);
    view(s->scontrib, cap * k);
    view(s->counters, n_counters);
    view(s->counters64, (size_t)max_depth + 3);
    s->arena_capacity = capacity; s->arena_shadow_k = k; s->arena_depth = max_depth;
    return true;
}

constexpr size_t MAX_BATCH = (size_t)1 << 28;   // path slots per wavefront batch (see batch_shape)

// Batch shape of a wavefront over `n_items` path sources (a frame's pixels, or the live rays of rtcuda_radiance) x `n_samples`
// samples: items and samples per batch.
void batch_shape(rtcuda_scene* s, uint32_t n_items, uint32_t n_samples, uint32_t shadow_k, uint32_t max_depth, uint32_t& np_batch,
                 uint32_t& ns_batch) {
    // Wavefront size. Deep bounces keep only a fraction of a batch alive (C3: 15 % fewer per bounce, 30 % left at
    // depth 8) and every launch of a persistent kernel ends with a drain tail, so batches are sized for the 180 GB
    // of HBM3e, not for L2: up to 256 Mi paths (336 B of path state each with 4 light samples per vertex), capped
    // to 40 % of the free device memory. C3's 143 M live paths are ONE batch of 111 launches (48 GB); with 64 Mi-path
    // batches the same frame took 327 launches and 3.4 % longer (profiles/r3a_ab.log).
    uint32_t capacity = s->ctx->bs.max_paths_in_flight;
    if (!capacity)
        if (const char* env = std::getenv("RTCUDA_MAX_PATHS")) capacity = (uint32_t)std::strtoul(env, nullptr, 0);  // tuning aid
    if (!capacity) {
        // Memory already held for path state (this scene's arena, or one parked by a released scene) that fits the
        // wavefront this job wants settles the size without asking the driver: cudaMemGetInfo is a trip into the
        // kernel driver (it queues behind NVML queries of a monitoring thread and other processes' calls) and sat
        // inside the render window with the GPU idle — 5-35 ms per frame on a busy box (profiles/r1s_gap.log).
        const size_t want = std::min<size_t>(MAX_BATCH, std::max<size_t>(1024, (size_t)n_items * n_samples));
        const size_t held = std::max(s->arena.base ? s->arena.bytes : 0, g_arena_cache.largest(s->ctx->device));
        if (held >= arena_bytes(want, shadow_k, max_depth)) capacity = (uint32_t)want;
        else if (held >= ((size_t)8 << 30)) {
            // a large arena that is smaller than this job's wish was itself cut to the 40 % rule when it was made:
            // run in batches of what it holds rather than ask the driver again (28 ms in one C5 call, profiles/r4k)
            const size_t per_slot = arena_bytes(1u << 20, shadow_k, max_depth) >> 20;
            capacity = (uint32_t)std::min<size_t>(want, (held - (1u << 20)) / std::max<size_t>(1, per_slot));
        }
    }
    if (!capacity) {
        const size_t bytes_per_slot = 16 + 16 * 7 + 16 + 4 + 48 * (size_t)std::max(1u, shadow_k);
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        const size_t have_b = free_b + s->wave_bytes();
        capacity = (uint32_t)std::min<size_t>(std::min<size_t>(MAX_BATCH, std::max<size_t>(1024, (size_t)n_items * n_samples)), (size_t)(0.4 * (double)have_b) / bytes_per_slot);
    }
    capacity = std::min(capacity, (uint32_t)(0xffffffffull / std::max(1u, shadow_k)));   // shadow-ray queue positions are 32-bit
    capacity = std::max(capacity, 1024u);
    np_batch = std::min(n_items, capacity);
    // samples per batch: as many as fit, then evened out over the batches (256 spp in batches of 124 would end with a
    // batch of 8 samples, whose launches are all drain tail)
    ns_batch = std::max(1u, std::min(n_samples, capacity / np_batch));
    const uint32_t n_sample_batches = (n_samples + ns_batch - 1) / ns_batch;
    ns_batch = (n_samples + n_sample_batches - 1) / n_sample_batches;
}
enum { CLS_EXTEND = 0, CLS_SHADE = 1, CLS_SHADOW = 2, CLS_OTHER = 3, CLS_GATHER = 4, CLS_COUNT = 5 };

// The event pool and the span list are shared by direct launches and by the captured frame (whose event-record nodes keep
// pointing at the pool's events): starting a new span list outside a capture drops the cached frame graph.
void reset_spans(rtcuda_scene* s, bool drop_frame_graph = true) {
    s->spans.clear();
    s->ev_used = 0;
    if (drop_frame_graph && s->frame_exec) { cudaGraphExecDestroy(s->frame_exec); s->frame_exec = nullptr; }
}

size_t record_event(rtcuda_scene* s) {
    if (s->ev_used == s->ev_pool.size()) {
        cudaEvent_t e;
        CK(cudaEventCreate(&e));
        s->ev_pool.push_back(e);
    }
    // inside a capture the record becomes an event-record node of the frame graph (external event: it can be timed after a replay)
    CK(cudaEventRecordWithFlags(s->ev_pool[s->ev_used], s->ctx->stream, s->capturing ? cudaEventRecordExternal : cudaEventRecordDefault));
    return s->ev_used++;
}
struct SpanGuard {  // times one launch when kernel timing is on
    rtcuda_scene* s;
    int cls;
    size_t e0 = 0;
    bool on;
    SpanGuard(rtcuda_scene* s_, int cls_, bool on_) : s(s_), cls(cls_), on(on_) { if (on) e0 = record_event(s); }
    ~SpanGuard() noexcept(false) { if (on) s->spans.push_back({cls, e0, record_event(s)}); }
};

// The caller's rays of an rtcuda_radiance batch: the chunk's prepared rays, the depth-0 hit k_trace found for each, the stream key
// of the chunk's first ray, and the call's own launch counter (the scene's counts describe the last render)
struct CallerRays {
    const float4* rays;
    const float4* first_hits;
    uint32_t key_base;
    LaunchCounter* lc;
};

// One batch of the wavefront: raygen, then per bounce extend -> shade -> shadow. All launches are sized by
// the batch (an upper bound); kernels read the live queue length from device counters, so the host never
// synchronises inside a batch. With `caller` the paths start from the caller's rays (k_raygen_rays) at their known depth-0 hits:
// the depth-0 extend is skipped, and no kernel time is recorded.
void run_batch(rtcuda_scene* s, const RenderParams& rp, Wave w, uint32_t n_paths, bool collect, const CallerRays* caller = nullptr) {
    cudaStream_t st = s->ctx->stream;
    const bool timing = !caller && (s->ctx->bs.collect_stats & RTCUDA_STATS_KERNEL_TIMES) != 0;
    LaunchCounter& lc = caller ? *caller->lc : s->lc;
    const uint32_t max_depth = rp.max_ray_depth;
    uint32_t* rays = s->counters.p;                       // rays[d]: queue length at depth d
    uint32_t* fetch_ext = s->counters.p + (max_depth + 3);      // work-fetch cursors of the persistent kernels
    uint32_t* fetch_sh = s->counters.p + 2 * (max_depth + 3);
    uint32_t* deferred_n = s->counters.p + 3 * (max_depth + 3);   // vertices the Diffuse shade kernel left for the general one, per depth
    unsigned long long* shadows = s->counters64.p;              // shadows[d]: NEE vertices | shadow rays << 32
    CK(cudaMemsetAsync(s->counters.p, 0, 4 * ((size_t)max_depth + 3) * 4, st));
    CK(cudaMemsetAsync(s->counters64.p, 0, ((size_t)max_depth + 3) * 8, st));
    w.depth = 0;
    w.ray_o_out = s->ray_o[0].p;
    w.ray_d_out = s->ray_d[0].p;
    w.n_out = rays;
    {
        SpanGuard g(s, CLS_OTHER, timing);
        if (caller) launch_raygen_rays(st, rp, w, caller->rays, caller->first_hits, caller->key_base, n_paths, lc);
        else launch_raygen(st, s->sc, rp, w, n_paths, lc);
    }
    for (uint32_t depth = 0; depth <= max_depth; depth++) {
        const int in = depth & 1, out = in ^ 1;
        w.depth = depth;
        w.ray_o_in = s->ray_o[in].p; w.ray_d_in = s->ray_d[in].p;
        w.ray_o_out = s->ray_o[out].p; w.ray_d_out = s->ray_d[out].p;
        w.n_in = rays + depth; w.n_out = rays + depth + 1; w.n_shadow = shadows + depth;
        w.deferred = s->deferred.p; w.n_deferred = deferred_n + depth;
        if (depth || !caller) { SpanGuard g(s, CLS_EXTEND, timing); launch_extend(st, s->sc, w, n_paths, depth == 0 ? s->sc.camera.near_clip : 0.0001f, fetch_ext + depth, collect, lc); }
        { SpanGuard g(s, CLS_SHADE, timing); launch_shade(st, s->sc, rp, w, n_paths, lc); }
        if (depth < max_depth && w.shadow_k) {
            { SpanGuard g(s, CLS_SHADOW, timing); launch_shadow(st, s->sc, w, (uint32_t)std::min<uint64_t>(0xffffffffull, (uint64_t)n_paths * std::max(1u, w.shadow_k)), fetch_sh + depth, collect, lc); }
            { SpanGuard g(s, CLS_GATHER, timing); launch_shadow_gather(st, w, n_paths, lc); }
        }
    }
}

// sample_hi == 0: the whole frame (all samples, mean). Otherwise samples [sample_lo, sample_hi) only and the beauty plane
// receives their un-normalised sum (rtcuda_render_samples_device).
void render_device(rtcuda_scene* s, const rtcuda_settings* settings, const rtcuda_outputs* out, uint32_t sample_lo = 0, uint32_t sample_hi = 0,
                   bool accumulate = false) {
    cudaStream_t st = s->ctx->stream;
    REQUIRE(out->width == s->width && out->height == s->height, "output size must equal the camera raster size");
    REQUIRE(settings->samples_per_pixel >= 1, "samples_per_pixel must be >= 1");
    if (settings->sampler_kind == RTCUDA_SAMPLER_STRATIFIED) REQUIRE(settings->x_strata >= 1 && settings->y_strata >= 1, "strata must be >= 1");
    const bool sum_mode = sample_hi != 0;
    if (sum_mode) REQUIRE(sample_lo < sample_hi && sample_hi <= settings->samples_per_pixel, "sample range must satisfy lo < hi <= samples_per_pixel");
    else sample_hi = settings->samples_per_pixel;
    const uint32_t n_samples_total = sample_hi - sample_lo;
    const RenderParams rp = make_params(settings);
    const bool collect = (s->ctx->bs.collect_stats & RTCUDA_STATS_COUNTERS) != 0;
    Trace tr("render_device", (int)s->ctx->bs.tile_rank);
    if (!s->pixel_list.p) build_pixel_list(s);
    tr.mark("pixel list");
    const uint32_t np_all = s->n_my_pixels;
    const size_t npix_img = (size_t)s->width * s->height;
    s->stats_dev.ensure(STAT_TOTAL);
    CK(cudaMemsetAsync(s->stats_dev.p, 0, STAT_TOTAL * sizeof(unsigned long long), st));
    const unsigned long long launches0 = s->lc.launches;

    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    CK(cudaEventRecord(e0, st));

    const uint32_t o = settings->outputs;
    if (!((o & RTCUDA_AOV_BEAUTY) && out->beauty && s->n_beauty_pixels)) reset_spans(s);   // no beauty pass: no kernel spans
    AovPlanes pl{};
    pl.normals = (o & RTCUDA_AOV_NORMALS) ? out->normals : nullptr;
    pl.albedo = (o & RTCUDA_AOV_ALBEDO) ? out->albedo : nullptr;
    pl.uv = (o & RTCUDA_AOV_UV_COORDS) ? out->uv : nullptr;
    pl.mip_level = (o & RTCUDA_AOV_MIP_LEVEL) ? out->mip_level : nullptr;
    pl.ids = (o & RTCUDA_AOV_DEBUG_IDS) ? out->debug_ids : nullptr;
    pl.depth = (o & RTCUDA_AOV_DEBUG_DEPTH) ? out->debug_depth : nullptr;
    const bool partial = np_all != npix_img;
    if (pl.normals || pl.albedo || pl.uv || pl.mip_level || pl.ids || pl.depth) {
        if (partial) {  // pixels of other ranks stay 0 (ids: 0 too) so frames can be summed
            if (pl.normals) CK(cudaMemsetAsync(pl.normals, 0, npix_img * 12, st));
            if (pl.albedo) CK(cudaMemsetAsync(pl.albedo, 0, npix_img * 12, st));
            if (pl.uv) CK(cudaMemsetAsync(pl.uv, 0, npix_img * 8, st));
            if (pl.mip_level) CK(cudaMemsetAsync(pl.mip_level, 0, npix_img * 4, st));
            if (pl.ids) CK(cudaMemsetAsync(pl.ids, 0, npix_img * 8, st));
            if (pl.depth) CK(cudaMemsetAsync(pl.depth, 0, npix_img * 4, st));
        }
        if (np_all) launch_aov(st, s->sc, rp, s->pixel_list.p, np_all, pl, s->stats_dev.p, collect, s->lc);
    }

    uint64_t samples = 0, dropped_samples = 0;
    if ((o & RTCUDA_AOV_BEAUTY) && out->beauty) {
        samples = (uint64_t)np_all * n_samples_total;
        dropped_samples = (uint64_t)(np_all - s->n_beauty_pixels) * n_samples_total;   // every one a camera ray that misses the scene bounds
        const uint32_t nb = s->n_beauty_pixels;   // owned pixels whose rays can reach the scene bounds (build_pixel_list)
        if (nb != npix_img && !accumulate) CK(cudaMemsetAsync(out->beauty, 0, npix_img * 12, st));   // (accumulate: the plane holds the running sum)
        if (nb) {
            const uint32_t shadow_k = shadow_entries_per_vertex(s, rp);
            uint32_t np_batch = 0, ns_batch = 0;
            batch_shape(s, nb, n_samples_total, shadow_k, rp.max_ray_depth, np_batch, ns_batch);
            tr.mark("sizing");
            ensure_wave(s, np_batch * ns_batch, shadow_k, rp.max_ray_depth);
            s->accum.ensure(nb);
            tr.mark("arena");
            Wave w{};
            w.pixel_list = s->beauty_list;
            w.capacity = np_batch * ns_batch;
            w.state = s->state.p; w.radiance = s->radiance.p; w.hits = s->hits.p;
            w.stats = s->stats_dev.p;
            w.shadow_k = shadow_k; w.svertex = s->svertex.p;
            w.sray_o = s->sray_o.p; w.sray_d = s->sray_d.p; w.scontrib = s->scontrib.p;
            auto enqueue_frame = [&] {
                CK(cudaMemsetAsync(s->accum.p, 0, (size_t)nb * sizeof(float4), st));
                for (uint32_t p0 = 0; p0 < nb; p0 += np_batch) {
                    const uint32_t np = std::min(np_batch, nb - p0);
                    for (uint32_t s0 = sample_lo; s0 < sample_hi; s0 += ns_batch) {
                        const uint32_t ns = std::min(ns_batch, sample_hi - s0);
                        w.pixel_base = p0; w.n_pixels = np; w.sample_base = s0; w.n_samples = ns;
                        run_batch(s, rp, w, np * ns, collect);
                        launch_resolve(st, w, s->accum.p, s->lc);
                    }
                }
                launch_finalize(st, s->beauty_list, nb, s->width, s->accum.p, sum_mode ? 1.0f : 1.0f / (float)settings->samples_per_pixel, out->beauty, s->stats_dev.p, accumulate, s->lc);
            };
            // frames of at least 4 Mi paths go through the graph (below that instantiating ~40 nodes per batch costs more
            // than the launches it saves); RTCUDA_NO_GRAPH=1 keeps direct launches (A/B, debugging)
            static const bool no_graph = std::getenv("RTCUDA_NO_GRAPH") != nullptr;
            if (no_graph || (uint64_t)nb * n_samples_total < (1ull << 22)) {
                reset_spans(s);
                enqueue_frame();
            } else {
                std::vector<uint64_t> key = {settings->max_ray_depth, settings->accumulate_bounces, settings->light_sample_count, settings->samples_per_pixel,
                                             settings->has_seed, settings->seed, settings->sampler_kind, settings->stratified_jitter, settings->x_strata,
                                             settings->y_strata, settings->antialias_primary_rays, settings->antialias_secondary_rays,
                                             (uint64_t)(uintptr_t)out->beauty, (uint64_t)(uintptr_t)s->arena.base, (uint64_t)(uintptr_t)s->accum.p,
                                             (uint64_t)(uintptr_t)s->stats_dev.p, (uint64_t)(uintptr_t)s->beauty_list, nb, np_batch, ns_batch, sample_lo,
                                             sample_hi, shadow_k, (uint64_t)s->ctx->bs.collect_stats, (uint64_t)sum_mode, (uint64_t)accumulate};
                // The first frame of a key is launched directly: capture + instantiation cost 2-3 ms, which a one-shot
                // `render(scene, settings)` would pay for a graph it never replays. The second frame with the same key is
                // captured, later ones replay it.
                const bool have_graph = s->frame_exec && key == s->frame_key;
                if (!have_graph && key != s->seen_key) {   // first frame of this key: direct launches
                    if (s->frame_exec) { cudaGraphExecDestroy(s->frame_exec); s->frame_exec = nullptr; }
                    s->frame_key.clear();
                    s->seen_key = key;
                    reset_spans(s);
                    enqueue_frame();
                } else {
                    if (!have_graph) {                     // second frame of this key: capture and instantiate
                        reset_spans(s);
                        const unsigned long long l0 = s->lc.launches;
                        cudaGraph_t graph = nullptr;
                        CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
                        s->capturing = true;
                        try {
                            enqueue_frame();
                        } catch (...) {
                            s->capturing = false;
                            cudaStreamEndCapture(st, &graph);
                            if (graph) cudaGraphDestroy(graph);
                            throw;
                        }
                        s->capturing = false;
                        CK(cudaStreamEndCapture(st, &graph));
                        const cudaError_t ie = cudaGraphInstantiate(&s->frame_exec, graph, 0);
                        cudaGraphDestroy(graph);
                        CK(ie);
                        s->frame_launches = s->lc.launches - l0;
                        s->lc.launches = l0;
                        s->frame_key = key;
                    }
                    CK(cudaGraphLaunch(s->frame_exec, st));
                    s->lc.launches += s->frame_launches;
                }
            }
        }
    }
    CK(cudaEventRecord(e1, st));
    tr.mark("enqueue");
    unsigned long long h_stats[STAT_TOTAL];
    CK(cudaMemcpyAsync(h_stats, s->stats_dev.p, sizeof h_stats, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    tr.mark("gpu");
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    s->stats.samples = samples;
    s->stats.primary_rays = h_stats[STAT_PRIMARY] + dropped_samples;
    s->stats.bounce_rays = h_stats[STAT_BOUNCE];
    s->stats.shadow_rays = h_stats[STAT_SHADOW];
    s->stats.aov_rays = h_stats[STAT_AOV];
    s->stats.extend_nodes = h_stats[STAT_EXT_NODES];
    s->stats.extend_prims = h_stats[STAT_EXT_PRIMS];
    s->stats.shadow_nodes = h_stats[STAT_SH_NODES];
    s->stats.shadow_prims = h_stats[STAT_SH_PRIMS];
    s->stats.nodes_fetched = h_stats[STAT_EXT_NODES] + h_stats[STAT_SH_NODES] + h_stats[STAT_AOV_NODES];
    s->stats.prims_fetched = h_stats[STAT_EXT_PRIMS] + h_stats[STAT_SH_PRIMS] + h_stats[STAT_AOV_PRIMS];
    s->stats.shaded_vertices = h_stats[STAT_SHADED];
    s->stats.nonfinite_values = h_stats[STAT_NONFINITE];
    s->stats.primary_rays_culled = h_stats[STAT_CULLED] + dropped_samples;
    s->stats.pixels_dropped = (o & RTCUDA_AOV_BEAUTY) && out->beauty ? np_all - s->n_beauty_pixels : 0;
    s->stats.final_rays_skipped = h_stats[STAT_FINAL_SKIPPED];
    s->stats.kernel_launches = s->lc.launches - launches0;
    s->stats.render_ms = ms;
    double cls_ms[CLS_COUNT] = {0, 0, 0, 0, 0};
    uint64_t cls_n[CLS_COUNT] = {0, 0, 0, 0, 0};
    for (const rtcuda_scene::Span& sp : s->spans) {
        float t = 0;
        CK(cudaEventElapsedTime(&t, s->ev_pool[sp.e0], s->ev_pool[sp.e1]));
        cls_ms[sp.cls] += t;
        cls_n[sp.cls]++;
    }
    s->stats.extend_ms = cls_ms[CLS_EXTEND]; s->stats.shade_ms = cls_ms[CLS_SHADE]; s->stats.shadow_ms = cls_ms[CLS_SHADOW];
    s->stats.other_ms = cls_ms[CLS_OTHER];
    s->stats.gather_ms = cls_ms[CLS_GATHER];
    s->stats.extend_launches = cls_n[CLS_EXTEND]; s->stats.shade_launches = cls_n[CLS_SHADE]; s->stats.shadow_launches = cls_n[CLS_SHADOW];
}

template <typename T>
T* stage_plane(DevBuf<T>& buf, bool wanted, size_t count) {
    if (!wanted) return nullptr;
    buf.ensure(count);
    return buf.p;
}

void render_host(rtcuda_scene* s, const rtcuda_settings* settings, rtcuda_outputs* out) {
    cudaStream_t st = s->ctx->stream;
    REQUIRE(out->width == s->width && out->height == s->height, "output size must equal the camera raster size");
    const size_t n = (size_t)s->width * s->height;
    const uint32_t o = settings->outputs;
    rtcuda_outputs dev{};
    dev.width = out->width; dev.height = out->height;
    dev.beauty = stage_plane(s->d_beauty, (o & RTCUDA_AOV_BEAUTY) && out->beauty, n * 3);
    dev.normals = stage_plane(s->d_normals, (o & RTCUDA_AOV_NORMALS) && out->normals, n * 3);
    dev.albedo = stage_plane(s->d_albedo, (o & RTCUDA_AOV_ALBEDO) && out->albedo, n * 3);
    dev.uv = stage_plane(s->d_uv, (o & RTCUDA_AOV_UV_COORDS) && out->uv, n * 2);
    dev.mip_level = stage_plane(s->d_mip, (o & RTCUDA_AOV_MIP_LEVEL) && out->mip_level, n);
    dev.debug_ids = stage_plane(s->d_ids, (o & RTCUDA_AOV_DEBUG_IDS) && out->debug_ids, n * 2);
    dev.debug_depth = stage_plane(s->d_depth, (o & RTCUDA_AOV_DEBUG_DEPTH) && out->debug_depth, n);
    render_device(s, settings, &dev);
    // device planes -> pinned staging (one async copy per plane) -> the caller's (pageable) planes on a few host threads
    struct Copy { void* host; const void* devp; size_t bytes, off; };
    std::vector<Copy> copies;
    size_t total = 0;
    auto add = [&](void* h, const void* d, size_t bytes) { if (d) { copies.push_back({h, d, bytes, total}); total += (bytes + 255) & ~(size_t)255; } };
    add(out->beauty, dev.beauty, n * 12); add(out->normals, dev.normals, n * 12); add(out->albedo, dev.albedo, n * 12);
    add(out->uv, dev.uv, n * 8); add(out->mip_level, dev.mip_level, n * 4); add(out->debug_ids, dev.debug_ids, n * 8);
    add(out->debug_depth, dev.debug_depth, n * 4);
    if (!total) return;
    size_t got = 0;
    uint8_t* stage = (uint8_t*)g_pinned_cache.take(total, got);
    if (!stage) {   // no pinned memory to be had: straight into the caller's planes
        for (const Copy& c : copies) CK(cudaMemcpyAsync(c.host, c.devp, c.bytes, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        return;
    }
    std::vector<char> direct(copies.size(), 0);   // planes from rtcuda_host_alloc: the copy engine writes them itself
    for (size_t i = 0; i < copies.size(); i++) direct[i] = g_host_allocs.covers(copies[i].host, copies[i].bytes) ? 1 : 0;
    try {
        for (size_t i = 0; i < copies.size(); i++) {
            const Copy& c = copies[i];
            CK(cudaMemcpyAsync(direct[i] ? c.host : (void*)(stage + c.off), c.devp, c.bytes, cudaMemcpyDeviceToHost, st));
        }
        CK(cudaStreamSynchronize(st));
    } catch (...) {
        g_pinned_cache.park(stage, got);
        throw;
    }
    for (size_t i = 0; i < copies.size(); i++) if (!direct[i]) parallel_memcpy(copies[i].host, stage + copies[i].off, copies[i].bytes);
    g_pinned_cache.park(stage, got);
}

void render_pixel(rtcuda_scene* s, const rtcuda_settings* settings, uint32_t x, uint32_t y, uint32_t lo, uint32_t hi, rtcuda_pixel_output* out) {
    cudaStream_t st = s->ctx->stream;
    REQUIRE(hi >= lo, "sample_hi < sample_lo");
    const uint32_t n = hi - lo;
    if (!n) return;
    REQUIRE(n <= (1u << 22), "sample range too large");
    x = std::min(x, s->width - 1);   // lib.rs:867-876
    y = std::min(y, s->height - 1);
    const RenderParams rp = make_params(settings);
    const uint32_t shadow_k = shadow_entries_per_vertex(s, rp);
    ensure_wave(s, n, shadow_k, rp.max_ray_depth);
    s->pixel_out.ensure(n);
    CK(cudaMemsetAsync(s->stats_dev.p, 0, STAT_TOTAL * sizeof(unsigned long long), st));
    DevBuf<uint32_t> one_pixel;
    const uint32_t packed = (y << 16) | x;
    one_pixel.upload(&packed, 1, st);
    launch_pixel_aov(st, s->sc, rp, x, y, lo, n, s->pixel_out.p, s->lc);
    Wave w{};
    w.pixel_list = one_pixel.p;
    w.pixel_base = 0; w.n_pixels = 1; w.sample_base = lo; w.n_samples = n; w.capacity = n;
    w.state = s->state.p; w.radiance = s->radiance.p; w.hits = s->hits.p;
    w.stats = s->stats_dev.p;
    w.shadow_k = shadow_k; w.svertex = s->svertex.p;
    w.sray_o = s->sray_o.p; w.sray_d = s->sray_d.p; w.scontrib = s->scontrib.p;
    reset_spans(s);
    run_batch(s, rp, w, n, false);
    launch_pixel_radiance(st, s->radiance.p, n, s->pixel_out.p, s->lc);
    static_assert(sizeof(PixelOut) == sizeof(rtcuda_pixel_output), "pixel output layout");
    CK(cudaMemcpyAsync(out, s->pixel_out.p, (size_t)n * sizeof(PixelOut), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
}

// ---------------------------------------------------------------------------------------------------
// ray queries (rtcuda_trace_rays / rtcuda_occluded): caller-supplied rays against the scene's BVH
// ---------------------------------------------------------------------------------------------------
// A query reads the scene and nothing else: no stats, no frame graph, no pixel lists, no path-state arena. Its scratch comes from
// the stream-ordered pool, sized for one chunk of rays.
constexpr uint64_t QUERY_CHUNK = 1ull << 24;   // rays per launch: 512 MB of rays and 256 MB of scratch hits

// Query outputs as the C ABI takes them (occluded set: an occlusion query; surfaces set: a surface query; otherwise a closest-hit
// query)
struct QueryPtrs {
    const float* rays;
    float* t;
    uint32_t* ids;
    float* uv;
    uint8_t* occluded;
    rtcuda_surface* surfaces;
};

// k_surface_finish writes rtcuda_surface as four float4 (rt_query.h surface_finish_body)
static_assert(sizeof(rtcuda_surface) == 4 * sizeof(float4), "surface record layout");
static_assert(offsetof(rtcuda_surface, point) == 0 && offsetof(rtcuda_surface, t) == 12, "surface record layout");
static_assert(offsetof(rtcuda_surface, normal) == 16 && offsetof(rtcuda_surface, material) == 28, "surface record layout");
static_assert(offsetof(rtcuda_surface, uv) == 32 && offsetof(rtcuda_surface, geom_id) == 40 && offsetof(rtcuda_surface, prim_id) == 44,
              "surface record layout");
static_assert(offsetof(rtcuda_surface, albedo) == 48 && offsetof(rtcuda_surface, light) == 60, "surface record layout");

// Checks that need no device: done first, so that a refused query does no device work
void validate_query(const rtcuda_scene* s, const QueryPtrs& q, uint64_t count) {
    REQUIRE(count < (1ull << 32), "ray count must be below 2^32");
    REQUIRE(q.rays || count == 0, "rays is NULL");
    REQUIRE(q.t || q.ids || q.uv || q.occluded || q.surfaces, "every output is NULL");
    REQUIRE(s, "scene is NULL");
}

// Pointers of the device variants must be device (or managed) memory of the GPU the scene's first context runs on
void require_device_pointer(const void* p, int device, const char* what) {
    if (!p) return;
    cudaPointerAttributes a{};
    const cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) cudaGetLastError();
    REQUIRE(e == cudaSuccess && (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) && a.device == device,
            std::string(what) + " is not device memory of device " + std::to_string(device));
}

// Kernels of one chunk: rays and outputs are device pointers already offset to the chunk
void query_chunk(rtcuda_scene* s, const float4* rays, uint32_t n, const QueryPtrs& out, float4* hits, uint32_t* counter, LaunchCounter& lc) {
    cudaStream_t st = s->ctx->stream;
    CK(cudaMemsetAsync(counter, 0, sizeof(uint32_t), st));
    if (out.occluded) {
        launch_occluded(st, s->sc, rays, n, out.occluded, counter, lc);
        return;
    }
    launch_trace(st, s->sc, rays, n, hits, counter, lc);
    if (out.surfaces) launch_surface_finish(st, s->sc, rays, hits, n, (float4*)out.surfaces, lc);
    else launch_trace_finish(st, s->sc, rays, hits, n, QueryOut{out.t, out.ids, out.uv}, lc);
}

// Device arrays on this scene's GPU; blocks until the outputs are written
void query_device(rtcuda_scene* s, const QueryPtrs& q, uint64_t count) {
    LaunchCounter lc;   // (not the scene's: the stats keep describing the last render)
    DevBuf<uint32_t> counter;
    DevBuf<float4> hits;
    counter.alloc(1);
    if (!q.occluded) hits.alloc(std::min(count, QUERY_CHUNK));
    for (uint64_t b = 0; b < count; b += QUERY_CHUNK) {
        const uint32_t n = (uint32_t)std::min(QUERY_CHUNK, count - b);
        const QueryPtrs o{nullptr, q.t ? q.t + b : nullptr, q.ids ? q.ids + 2 * b : nullptr, q.uv ? q.uv + 2 * b : nullptr,
                          q.occluded ? q.occluded + b : nullptr, q.surfaces ? q.surfaces + b : nullptr};
        query_chunk(s, (const float4*)q.rays + 2 * b, n, o, hits.p, counter.p, lc);
    }
    CK(cudaStreamSynchronize(s->ctx->stream));
}

// Host arrays: per chunk, rays in, kernels, requested outputs out (cudaMemcpyAsync on the scene's stream); blocks until the
// results are on the host
void query_host(rtcuda_scene* s, const QueryPtrs& q, uint64_t count) {
    cudaStream_t st = s->ctx->stream;
    LaunchCounter lc;
    const uint64_t cap = std::min(count, QUERY_CHUNK);
    DevBuf<uint32_t> counter;
    DevBuf<float4> rays, hits, surf;
    DevBuf<float> t, uv;
    DevBuf<uint32_t> ids;
    DevBuf<uint8_t> occ;
    counter.alloc(1);
    rays.alloc(2 * cap);
    if (q.occluded) occ.alloc(cap);
    else hits.alloc(cap);
    if (q.t) t.alloc(cap);
    if (q.ids) ids.alloc(2 * cap);
    if (q.uv) uv.alloc(2 * cap);
    if (q.surfaces) surf.alloc(4 * cap);
    const QueryPtrs dev{nullptr, q.t ? t.p : nullptr, q.ids ? ids.p : nullptr, q.uv ? uv.p : nullptr, q.occluded ? occ.p : nullptr,
                        q.surfaces ? (rtcuda_surface*)surf.p : nullptr};
    for (uint64_t b = 0; b < count; b += QUERY_CHUNK) {
        const uint32_t n = (uint32_t)std::min(QUERY_CHUNK, count - b);
        CK(cudaMemcpyAsync(rays.p, q.rays + 8 * b, (size_t)n * 32, cudaMemcpyHostToDevice, st));
        query_chunk(s, rays.p, n, dev, hits.p, counter.p, lc);
        if (q.t) CK(cudaMemcpyAsync(q.t + b, t.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
        if (q.ids) CK(cudaMemcpyAsync(q.ids + 2 * b, ids.p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
        if (q.uv) CK(cudaMemcpyAsync(q.uv + 2 * b, uv.p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
        if (q.occluded) CK(cudaMemcpyAsync(q.occluded + b, occ.p, (size_t)n, cudaMemcpyDeviceToHost, st));
        if (q.surfaces) CK(cudaMemcpyAsync(q.surfaces + b, surf.p, (size_t)n * sizeof(rtcuda_surface), cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
}

// ---------------------------------------------------------------------------------------------------
// radiance along caller-supplied rays (rtcuda_radiance): the wavefront integrator started from the caller's rays
// ---------------------------------------------------------------------------------------------------
// Per chunk of rays: k_radiance_prep normalises them, k_trace walks each first segment once, k_radiance_live lists the rays that
// need path slots, then batches over (live rays x samples) run the renderer's wavefront from depth 0 with the depth-0 extend
// skipped, k_resolve sums the samples, and k_finalize writes the means. The call may re-carve the scene's path-state arena; the
// stats, the launch count and the kernel-time spans of the last render are left alone.

// Checks that need no device: done first, so that a refused call does no device work
void validate_radiance(const rtcuda_scene* s, const rtcuda_settings* st, const float* rays, uint64_t count, uint32_t stream_base,
                       const float* radiance) {
    REQUIRE(count < (1ull << 32), "ray count must be below 2^32");
    REQUIRE((uint64_t)stream_base + count <= (1ull << 32), "stream_base + count must not exceed 2^32");
    REQUIRE(rays || count == 0, "rays is NULL");
    REQUIRE(radiance, "radiance is NULL");
    REQUIRE(st, "settings is NULL");
    REQUIRE(st->samples_per_pixel >= 1, "samples_per_pixel must be >= 1");
    if (st->sampler_kind == RTCUDA_SAMPLER_STRATIFIED) REQUIRE(st->x_strata >= 1 && st->y_strata >= 1, "strata must be >= 1");
    REQUIRE(s, "scene is NULL");
}

// Device scratch of one call, sized for its largest chunk
struct RadianceScratch {
    DevBuf<float4> prepared, first_hits, accum;
    DevBuf<uint32_t> live, counters;     // counters: k_trace's fetch cursor, the live-ray count
    DevBuf<unsigned long long> stats;    // STAT_* of the call's wavefront (the scene's block belongs to the render)
    LaunchCounter lc;
    explicit RadianceScratch(uint64_t chunk) {
        prepared.alloc(2 * chunk); first_hits.alloc(chunk); accum.alloc(chunk); live.alloc(chunk);
        counters.alloc(2); stats.alloc(STAT_TOTAL);
    }
};

// One chunk of n rays: `rays` and `out` are device pointers offset to the chunk, key_base the stream key of its first ray
void radiance_chunk(rtcuda_scene* s, const rtcuda_settings* settings, const float4* rays, uint32_t n, uint32_t key_base, float* out,
                    RadianceScratch& x) {
    cudaStream_t st = s->ctx->stream;
    RenderParams rp = make_params(settings);
    rp.antialias_primary_rays = 0;   // a caller's ray has no differentials: its first hit uses matctx_no_aa like every later bounce
    launch_radiance_prep(st, rays, n, x.prepared.p, x.lc);
    CK(cudaMemsetAsync(x.counters.p, 0, 2 * sizeof(uint32_t), st));
    launch_trace(st, s->sc, x.prepared.p, n, x.first_hits.p, x.counters.p, x.lc);
    launch_radiance_live(st, s->sc, x.prepared.p, x.first_hits.p, n, x.live.p, x.counters.p + 1, x.lc);
    CK(cudaMemsetAsync(out, 0, (size_t)n * 3 * sizeof(float), st));
    uint32_t n_live = 0;
    CK(cudaMemcpyAsync(&n_live, x.counters.p + 1, sizeof n_live, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (!n_live) return;
    const uint32_t spp = settings->samples_per_pixel, shadow_k = shadow_entries_per_vertex(s, rp);
    uint32_t np_batch = 0, ns_batch = 0;
    batch_shape(s, n_live, spp, shadow_k, rp.max_ray_depth, np_batch, ns_batch);
    // The captured frame graph's nodes hold buffer pointers carved from the arena, and its key holds the arena's base but not the
    // carve; a re-carve keeps the base when the allocation is big enough (WaveArena::reserve). The graph must not outlive it.
    if (ensure_wave(s, np_batch * ns_batch, shadow_k, rp.max_ray_depth) && s->frame_exec) {
        cudaGraphExecDestroy(s->frame_exec);
        s->frame_exec = nullptr;
    }
    CK(cudaMemsetAsync(x.accum.p, 0, (size_t)n_live * sizeof(float4), st));
    Wave w{};
    w.pixel_list = x.live.p;
    w.capacity = np_batch * ns_batch;
    w.state = s->state.p; w.radiance = s->radiance.p; w.hits = s->hits.p;
    w.stats = x.stats.p;
    w.shadow_k = shadow_k; w.svertex = s->svertex.p;
    w.sray_o = s->sray_o.p; w.sray_d = s->sray_d.p; w.scontrib = s->scontrib.p;
    const CallerRays caller{x.prepared.p, x.first_hits.p, key_base, &x.lc};
    for (uint32_t p0 = 0; p0 < n_live; p0 += np_batch) {
        const uint32_t np = std::min(np_batch, n_live - p0);
        for (uint32_t s0 = 0; s0 < spp; s0 += ns_batch) {
            const uint32_t ns = std::min(ns_batch, spp - s0);
            w.pixel_base = p0; w.n_pixels = np; w.sample_base = s0; w.n_samples = ns;
            run_batch(s, rp, w, np * ns, false, &caller);
            launch_resolve(st, w, x.accum.p, x.lc);
        }
    }
    // k_finalize reused with the live list as its pixel list and a width of 65536: idx = (r >> 16) * 65536 + (r & 0xffff) = r,
    // the ray's index in the chunk (chunks hold at most 2^24 rays)
    launch_finalize(st, x.live.p, n_live, 65536u, x.accum.p, 1.0f / (float)spp, out, x.stats.p, false, x.lc);
}

// Device arrays on this scene's GPU; blocks until the radiance is written
void radiance_device(rtcuda_scene* s, const rtcuda_settings* settings, const float* rays, uint64_t count, uint32_t stream_base, float* radiance) {
    RadianceScratch x(std::min(count, QUERY_CHUNK));
    for (uint64_t b = 0; b < count; b += QUERY_CHUNK) {
        const uint32_t n = (uint32_t)std::min(QUERY_CHUNK, count - b);
        radiance_chunk(s, settings, (const float4*)rays + 2 * b, n, stream_base + (uint32_t)b, radiance + 3 * b, x);
    }
    CK(cudaStreamSynchronize(s->ctx->stream));
}

// Host arrays: per chunk, rays in and radiance out with cudaMemcpyAsync on the scene's stream; blocks until the radiance is here
void radiance_host(rtcuda_scene* s, const rtcuda_settings* settings, const float* rays, uint64_t count, uint32_t stream_base, float* radiance) {
    cudaStream_t st = s->ctx->stream;
    const uint64_t cap = std::min(count, QUERY_CHUNK);
    RadianceScratch x(cap);
    DevBuf<float4> d_rays;
    DevBuf<float> d_out;
    d_rays.alloc(2 * cap);
    d_out.alloc(3 * cap);
    for (uint64_t b = 0; b < count; b += QUERY_CHUNK) {
        const uint32_t n = (uint32_t)std::min(QUERY_CHUNK, count - b);
        CK(cudaMemcpyAsync(d_rays.p, rays + 8 * b, (size_t)n * 32, cudaMemcpyHostToDevice, st));
        radiance_chunk(s, settings, d_rays.p, n, stream_base + (uint32_t)b, d_out.p, x);
        CK(cudaMemcpyAsync(radiance + 3 * b, d_out.p, (size_t)n * 12, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
}


// ---------------------------------------------------------------------------------------------------
// scene update: camera, instance transforms and lights of an uploaded scene, in place
// ---------------------------------------------------------------------------------------------------
// The description must have the uploaded scene's topology; only what update_scene reads is checked, and all of it before any
// device work, so a refused update leaves the scene as it was.
void validate_update(const rtcuda_scene* s, const rtcuda_scene_desc* d) {
    REQUIRE(d->abi_version == RTCUDA_ABI_VERSION, "scene_desc.abi_version mismatch");
    REQUIRE(d->camera.raster_width == s->host_camera.raster_width && d->camera.raster_height == s->host_camera.raster_height,
            "update: the raster size differs from the uploaded scene's");
    REQUIRE(d->camera.kind == s->host_camera.kind, "update: the camera kind differs from the uploaded scene's");
    REQUIRE(d->shape_count == s->shape_count && d->instance_count == s->host_instances.size() && d->light_count == s->host_lights.size() &&
                d->material_count == s->material_count && d->texture_count == s->texture_count && d->image_count == s->image_count,
            "update: the shape / instance / light / material / texture / image counts differ from the uploaded scene's");
    REQUIRE(d->instance_count == 0 || d->instances, "update: instances is NULL");
    REQUIRE(d->light_count == 0 || d->lights, "update: lights is NULL");
    for (uint32_t i = 0; i < d->instance_count; i++)
        REQUIRE(d->instances[i].shape == s->host_instances[i].shape, "update: an instance refers to another shape than the uploaded one");
    for (uint32_t i = 0; i < d->light_count; i++)
        REQUIRE(d->lights[i].kind == s->host_lights[i].kind && d->lights[i].shape == s->host_lights[i].shape,
                "update: a light's kind or shape differs from the uploaded one");
}

// Node pass over every level, deepest first, then the deterministic SAH sum; returns the cost (RefitCtx::node_box)
double refit_nodes(rtcuda_scene* s, RefitCtx& r, bool write_nodes) {
    cudaStream_t st = s->ctx->stream;
    r.write_nodes = write_nodes ? 1u : 0u;
    std::vector<uint32_t> first(s->level_counts.size());
    uint32_t n_nodes = 0;
    for (size_t L = 0; L < s->level_counts.size(); L++) { first[L] = n_nodes; n_nodes += s->level_counts[L]; }
    for (size_t L = s->level_counts.size(); L-- > 0;) launch_refit_nodes(st, r, first[L], s->level_counts[L], s->lc);
    DevBuf<double> partial;
    partial.alloc(SAH_BLOCKS);
    launch_sah_partial(st, r.node_box, n_nodes, partial.p, s->lc);
    double h_partial[SAH_BLOCKS];
    float4 root[2];
    CK(cudaMemcpyAsync(h_partial, partial.p, sizeof h_partial, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(root, r.node_box, sizeof root, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    double children = 0.0;
    for (uint32_t b = 0; b < SAH_BLOCKS; b++) children += h_partial[b];
    return sah_cost(root, children);
}

void update_scene(rtcuda_scene* s, const rtcuda_scene_desc* d) {
    cudaStream_t st = s->ctx->stream;
    Trace tr("update", (int)s->ctx->bs.tile_rank);
    const bool cam_changed = std::memcmp(&d->camera, &s->host_camera, sizeof d->camera) != 0;
    bool lights_changed = false, moved = false;
    for (uint32_t i = 0; i < d->light_count; i++) {
        const rtcuda_light& a = d->lights[i];
        const rtcuda_light& h = s->host_lights[i];
        lights_changed |= std::memcmp(a.position_or_direction, h.position_or_direction, sizeof a.position_or_direction) != 0 ||
                          std::memcmp(a.intensity_or_radiance, h.intensity_or_radiance, sizeof a.intensity_or_radiance) != 0 ||
                          std::memcmp(&a.light_to_world, &h.light_to_world, sizeof a.light_to_world) != 0;
    }
    std::vector<uint8_t> row_moved(d->instance_count, 0);
    for (uint32_t i = 0; i < d->instance_count; i++) {
        const Instance& h = s->host_instances[i];
        const M4 f = to_m4(d->instances[i].object_to_world.forward), v = to_m4(d->instances[i].object_to_world.inverse);
        row_moved[i] = std::memcmp(&f, &h.o2w, sizeof f) != 0 || std::memcmp(&v, &h.w2o, sizeof v) != 0;
        moved |= row_moved[i] != 0;
    }
    const uint32_t n_prims = (uint32_t)s->stats.bvh_prim_count;
    const bool have_tree = n_prims != 0;
    if (have_tree && !RT_FIXED_SLOTS) throw RtError{RTCUDA_ERR_UNSUPPORTED, "scene updates need the fixed-slot primitive layout (RT_FIXED_SLOTS=1)"};
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    CK(cudaEventRecord(e0, st));

    RefitCtx r{};
    r.instances = s->instances.p; r.vertices = s->vertices.p; r.tris = s->tris.p;
    r.prims = s->prims.p; r.prim_slots = s->sc.prim_count; r.nodes = s->nodes.p;
    // the cost of the tree as built, from the unchanged primitives (first update of the scene; after a rebuild, below)
    if (have_tree && s->sah_built == 0.0) {
        s->node_box.alloc(2 * (size_t)s->sc.node_count);
        r.node_box = s->node_box.p;
        s->sah_built = refit_nodes(s, r, false);
        s->stats.bvh_sah_cost = s->sah_built;
    }
    r.node_box = s->node_box.p;
    tr.mark("baseline");

    // instance rows: runs of moved rows, one copy each
    for (uint32_t i = 0; i < d->instance_count;) {
        if (!row_moved[i]) { i++; continue; }
        uint32_t j = i;
        for (; j < d->instance_count && row_moved[j]; j++) {
            s->host_instances[j].o2w = to_m4(d->instances[j].object_to_world.forward);
            s->host_instances[j].w2o = to_m4(d->instances[j].object_to_world.inverse);
        }
        CK(cudaMemcpyAsync(s->instances.p + i, s->host_instances.data() + i, (j - i) * sizeof(Instance), cudaMemcpyHostToDevice, st));
        i = j;
    }
    if (lights_changed) {
        for (uint32_t i = 0; i < d->light_count; i++) {
            const rtcuda_light& a = d->lights[i];
            LightD& b = s->light_rows[i];
            std::memcpy(b.a, a.position_or_direction, sizeof b.a);
            std::memcpy(b.b, a.intensity_or_radiance, sizeof b.b);
            b.light_to_world = to_m4(a.light_to_world);
            s->host_lights[i] = a;
        }
        CK(cudaMemcpyAsync(s->lights.p, s->light_rows.data(), s->light_rows.size() * sizeof(LightD), cudaMemcpyHostToDevice, st));
        s->sc.light0 = s->light_rows[0];
    }
    if (cam_changed) {
        CameraD& cam = s->sc.camera;
        cam.near_clip = d->camera.near_clip; cam.far_clip = d->camera.far_clip;
        cam.aperture_radius = d->camera.aperture_radius; cam.focal_distance = d->camera.focal_distance;
        cam.raster_to_camera = to_m4(d->camera.raster_to_camera.forward);
        cam.camera_to_world = to_m4(d->camera.camera_to_world.forward);
        s->host_camera = d->camera;
    }

    uint32_t last = cam_changed || lights_changed ? 1u : 0u;
    if (moved && have_tree) {
        DevBuf<uint32_t> bounds_keys;
        bounds_keys.alloc(6);
        const uint32_t init_keys[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
        CK(cudaMemcpyAsync(bounds_keys.p, init_keys, sizeof init_keys, cudaMemcpyHostToDevice, st));
        r.bounds_keys = bounds_keys.p;
        launch_refit_prims(st, r, s->lc);
        const double sah_refit = refit_nodes(s, r, true);
        tr.mark("refit");
        // RTCUDA_TEST_REFIT_MAX_GROWTH: test / measurement hook that replaces the rule's factor (scripts/update_bench.py keeps
        // every refit with a huge value, to measure what a refit costs where the rule would rebuild)
        const char* growth = std::getenv("RTCUDA_TEST_REFIT_MAX_GROWTH");
        if (refit_needs_rebuild(sah_refit, s->sah_built, growth ? std::atof(growth) : REFIT_MAX_GROWTH)) {
            // from the resident geometry: the instance table on the device is current
            build_bvh(s, s->host_instances, n_prims);
            s->sc.nodes = s->nodes.p;
            s->sc.prims = s->prims.p;
            s->shade_recs.alloc(s->sc.prim_count);
            launch_shade_recs(st, s->sc, s->shade_recs.p, s->lc);
            s->sc.shade_recs = s->shade_recs.p;
            s->node_box.alloc(2 * (size_t)s->sc.node_count);
            r.prims = s->prims.p; r.prim_slots = s->sc.prim_count; r.nodes = s->nodes.p; r.node_box = s->node_box.p;
            s->sah_built = refit_nodes(s, r, false);
            s->stats.bvh_sah_cost = s->sah_built;
            last = 3;
            tr.mark("rebuild");
        } else {
            // scene centre, radius and culling bounds from the refitted primitives, exactly as build_bvh derives them
            uint32_t hk[6];
            CK(cudaMemcpyAsync(hk, bounds_keys.p, sizeof hk, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            const V3 mn = mk3(key_float(hk[0]), key_float(hk[1]), key_float(hk[2])), mx = mk3(key_float(hk[3]), key_float(hk[4]), key_float(hk[5]));
            const V3 c = (mx + mn) / 2.0f;
            s->sc.scene_center[0] = c.x; s->sc.scene_center[1] = c.y; s->sc.scene_center[2] = c.z;
            s->sc.scene_radius = n_prims == 1 ? INFINITY : length(mx - c);
            set_scene_bounds(s->sc, mn, mx, true);
            s->stats.bvh_sah_cost = sah_refit;
            last = 2;
        }
    } else if (moved) last = 1;   // instances without primitives: nothing in the tree moves
    if (last) {
        // Everything derived from the camera, the lights or the bounds: the captured frame graph (its launches hold the old
        // kernel parameters, and its key sees neither the camera nor the scene constants), the pixel lists and the tile table
        // (the culling rectangle of build_pixel_list is the projected scene bounds).
        reset_spans(s);
        s->frame_key.clear();
        s->seen_key.clear();
        s->pixel_list.release();
        s->beauty_list_buf.release();
        s->beauty_list = nullptr;
        s->n_my_pixels = s->n_beauty_pixels = 0;
        s->host_tiles.clear();
        s->tiles.release();
    }
    CK(cudaEventRecord(e1, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    s->stats.update_ms = ms;
    s->stats.bvh_last_update = last;
}

// ---------------------------------------------------------------------------------------------------
// multi-device contexts (backend_settings.num_devices > 1): the scene replicated on every GPU, tiles dealt round-robin,
// one host thread per GPU per call — the in-process analogue of the CPU backend's worker pool (lib.rs:706-805)
// ---------------------------------------------------------------------------------------------------
void enter(rtcuda_scene* sub) {
    CK(cudaSetDevice(sub->ctx->device));
    tls_stream = sub->ctx->stream;
}

// f(r) on one thread per GPU; the first error (by rank) is rethrown on the caller's thread after all have finished
template <typename F>
void for_each_device(size_t n, F&& f) {
    std::vector<RtError> errs(n, RtError{RTCUDA_OK, ""});
    std::vector<std::thread> threads;
    threads.reserve(n);
    for (size_t r = 0; r < n; r++)
        threads.emplace_back([&, r] {
            try { f(r); }
            catch (const RtError& e) { errs[r] = e; }
            catch (const std::bad_alloc&) { errs[r] = RtError{RTCUDA_ERR_OUT_OF_MEMORY, "host allocation failed"}; }
            catch (const std::exception& e) { errs[r] = RtError{RTCUDA_ERR_CUDA, e.what()}; }
        });
    for (std::thread& t : threads) t.join();
    for (size_t r = 0; r < n; r++)
        if (errs[r].status != RTCUDA_OK) throw RtError{errs[r].status, "device " + std::to_string(r) + ": " + errs[r].msg};
}

void multi_upload(rtcuda_ctx* ctx, const rtcuda_scene_desc* desc, rtcuda_scene* parent) {
    const size_t n = ctx->subs.size();
    parent->width = desc->camera.raster_width;
    parent->height = desc->camera.raster_height;
    parent->subs.assign(n, nullptr);
    for (size_t r = 0; r < n; r++) {
        parent->subs[r] = new rtcuda_scene();
        parent->subs[r]->ctx = ctx->subs[r];
    }
    rtcuda_scene* first = parent->subs[0];
    first->peer_list.assign(n, nullptr);
    first->peer_recv.assign(n, nullptr);
    first->peer_recv_words.assign(n, 0);
    Rendezvous meet;
    meet.n = (int)n;
    for_each_device(n, [&](size_t r) {
        try {
            enter(parent->subs[r]);
            GeoShare share{(int)r, (int)n, &parent->subs, &meet};
            upload_scene(parent->subs[r], desc, &share);
            CK(cudaEventCreateWithFlags(&parent->subs[r]->sent, cudaEventDisableTiming));
        } catch (...) {
            meet.fail();
            throw;
        }
    });
}

// Validated once against rank 0's copies (every rank holds the same), then every GPU updates its replica on its own thread. Rank 0's
// copies of the other ranks' tile tables go with their pixel lists.
void multi_update(rtcuda_scene* parent, const rtcuda_scene_desc* desc) {
    validate_update(parent->subs[0], desc);
    for_each_device(parent->subs.size(), [&](size_t r) {
        enter(parent->subs[r]);
        update_scene(parent->subs[r], desc);
    });
    rtcuda_scene* first = parent->subs[0];
    if (first->stats.bvh_last_update) {
        enter(first);
        for (TileRec*& q : first->peer_list) { if (q) cudaFree(q); q = nullptr; }
    }
}

void multi_release(rtcuda_scene* parent) {
    // one host thread per GPU, like every other multi-device call (the ~40 stream-ordered frees of a sub-scene are host work)
    std::vector<std::thread> threads;
    for (rtcuda_scene* sub : parent->subs) {
        if (!sub) continue;
        threads.emplace_back([sub] {
            cudaSetDevice(sub->ctx->device);
            tls_stream = sub->ctx->stream;
            cudaStreamSynchronize(tls_stream);   // the parked path-state arena may be picked up by another stream next
            delete sub;
        });
    }
    for (std::thread& t : threads) t.join();
    parent->subs.clear();
}

struct PlaneSlot { uint32_t ch; void* ptr; };
constexpr int N_PLANES = 7;
void planes_of(const rtcuda_outputs& o, uint32_t outputs, PlaneSlot out[N_PLANES]) {
    out[0] = {3, (outputs & RTCUDA_AOV_BEAUTY) ? (void*)o.beauty : nullptr};
    out[1] = {3, (outputs & RTCUDA_AOV_NORMALS) ? (void*)o.normals : nullptr};
    out[2] = {3, (outputs & RTCUDA_AOV_ALBEDO) ? (void*)o.albedo : nullptr};
    out[3] = {2, (outputs & RTCUDA_AOV_UV_COORDS) ? (void*)o.uv : nullptr};
    out[4] = {1, (outputs & RTCUDA_AOV_MIP_LEVEL) ? (void*)o.mip_level : nullptr};
    out[5] = {2, (outputs & RTCUDA_AOV_DEBUG_IDS) ? (void*)o.debug_ids : nullptr};
    out[6] = {1, (outputs & RTCUDA_AOV_DEBUG_DEPTH) ? (void*)o.debug_depth : nullptr};
}

// this GPU's staging planes for the requested outputs (the planes render_host uses)
rtcuda_outputs staging_planes(rtcuda_scene* s, uint32_t o, const rtcuda_outputs& like) {
    const size_t n = (size_t)s->width * s->height;
    rtcuda_outputs dev{};
    dev.width = s->width; dev.height = s->height;
    dev.beauty = stage_plane(s->d_beauty, (o & RTCUDA_AOV_BEAUTY) && like.beauty, n * 3);
    dev.normals = stage_plane(s->d_normals, (o & RTCUDA_AOV_NORMALS) && like.normals, n * 3);
    dev.albedo = stage_plane(s->d_albedo, (o & RTCUDA_AOV_ALBEDO) && like.albedo, n * 3);
    dev.uv = stage_plane(s->d_uv, (o & RTCUDA_AOV_UV_COORDS) && like.uv, n * 2);
    dev.mip_level = stage_plane(s->d_mip, (o & RTCUDA_AOV_MIP_LEVEL) && like.mip_level, n);
    dev.debug_ids = stage_plane(s->d_ids, (o & RTCUDA_AOV_DEBUG_IDS) && like.debug_ids, n * 2);
    dev.debug_depth = stage_plane(s->d_depth, (o & RTCUDA_AOV_DEBUG_DEPTH) && like.debug_depth, n);
    return dev;
}

// Gather this GPU's owned pixels of every requested plane into its packed buffer (plane after plane); returns the words used.
size_t pack_owned(rtcuda_scene* sub, const PlaneSlot planes[N_PLANES], bool peer_visible) {
    cudaStream_t st = sub->ctx->stream;
    const uint32_t np = sub->n_my_pixels;
    size_t words = 0;
    for (int i = 0; i < N_PLANES; i++) if (planes[i].ptr) words += (size_t)np * planes[i].ch;
    if (words > sub->packed_words || (peer_visible && !sub->packed_plain)) {
        // host frames: from the stream-ordered pool (a plain cudaMalloc / cudaFree pair costs milliseconds per one-shot render
        // once peer mappings exist); device planes: a plain allocation, which GPU 0 can be sent from (kept across frames)
        if (sub->packed) { if (sub->packed_plain) { CK(cudaStreamSynchronize(st)); cudaFree(sub->packed); } else CK(cudaFreeAsync(sub->packed, st)); }
        sub->packed = nullptr; sub->packed_words = 0;
        if (peer_visible) CK(cudaMalloc((void**)&sub->packed, words * 4));
        else CK(cudaMallocAsync((void**)&sub->packed, words * 4, st));
        sub->packed_plain = peer_visible;
        sub->packed_words = words;
    }
    size_t off = 0;
    for (int i = 0; i < N_PLANES; i++) {
        if (!planes[i].ptr) continue;
        launch_pack_tiles(st, 0, sub->tiles.p, (uint32_t)sub->host_tiles.size(), sub->width, planes[i].ch, (uint32_t*)planes[i].ptr, sub->packed + off, sub->lc);
        off += (size_t)np * planes[i].ch;
    }
    return words;
}

// rtcuda_render on a multi-device scene: every GPU renders its tiles and copies the pixels it owns straight into the caller's
// host planes (its own PCIe link, its own host thread): no GPU-to-GPU hop, no second pass over the frame on the host.
void multi_render_host(rtcuda_scene* parent, const rtcuda_settings* settings, rtcuda_outputs* out) {
    REQUIRE(out->width == parent->width && out->height == parent->height, "output size must equal the camera raster size");
    const uint32_t o = settings->outputs;
    for_each_device(parent->subs.size(), [&](size_t r) {
        rtcuda_scene* sub = parent->subs[r];
        enter(sub);
        cudaStream_t st = sub->ctx->stream;
        Trace tr("render_host", (int)r);
        rtcuda_outputs dev = staging_planes(sub, o, *out);
        tr.mark("staging planes");
        render_device(sub, settings, &dev);
        tr.mark("render_device");
        PlaneSlot dp[N_PLANES], hp[N_PLANES];
        planes_of(dev, o, dp);
        planes_of(*out, o, hp);
        const size_t words = pack_owned(sub, dp, false);
        if (!words) return;
        if (words > sub->h_packed_words) {
            if (sub->h_packed) g_pinned_cache.park(sub->h_packed, sub->h_packed_words * 4);
            sub->h_packed = nullptr; sub->h_packed_words = 0;
            size_t got = 0;
            sub->h_packed = (uint32_t*)g_pinned_cache.take(words * 4, got);
            if (!sub->h_packed) throw RtError{RTCUDA_ERR_OUT_OF_MEMORY, "no pinned host memory for the frame staging"};
            sub->h_packed_words = got / 4;
        }
        CK(cudaMemcpyAsync(sub->h_packed, sub->packed, words * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        tr.mark("pack + d2h");
        const uint32_t np = sub->n_my_pixels, W = sub->width;
        // the packed runs are tile after tile, row-major inside a tile: whole tile rows move into the caller's planes, on a few
        // host threads per GPU (a 1080p beauty plane pixel by pixel on one thread: 13 ms)
        const std::vector<TileRec>& tiles = sub->host_tiles;
        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        const unsigned n_thr = (unsigned)std::max<size_t>(1, std::min<size_t>(std::min<size_t>(8, hw / parent->subs.size()), np / 65536));
        auto scatter = [&](size_t t0, size_t t1) {
            size_t off = 0;
            for (int i = 0; i < N_PLANES; i++) {
                if (!dp[i].ptr) continue;
                const uint32_t ch = dp[i].ch;
                uint32_t* dst = (uint32_t*)hp[i].ptr;
                const uint32_t* src = sub->h_packed + off;
                for (size_t k = t0; k < t1; k++) {
                    const TileRec& t = tiles[k];
                    for (uint32_t row = 0; row < t.h; row++)
                        std::memcpy(dst + ((size_t)(t.y0 + row) * W + t.x0) * ch, src + ((size_t)t.off + (size_t)row * t.w) * ch, (size_t)t.w * ch * 4);
                }
                off += (size_t)np * ch;
            }
        };
        std::vector<std::thread> helpers;
        const size_t per = (tiles.size() + n_thr - 1) / n_thr;
        for (unsigned t = 1; t < n_thr; t++) helpers.emplace_back(scatter, std::min(tiles.size(), per * t), std::min(tiles.size(), per * (t + 1)));
        scatter(0, std::min(tiles.size(), per));
        for (std::thread& h : helpers) h.join();
        tr.mark("host scatter");
    });
}

// Device-plane variants on a multi-device scene: the planes live on device_ids[0]. GPU 0 renders its tiles into them; every
// other GPU packs the pixels it owns and sends them with ONE peer copy (NVLink) into a receive buffer on GPU 0, which
// scatters (or, for progressive sums, adds) them into the planes.
void multi_render_device(rtcuda_scene* parent, const rtcuda_settings* settings, const rtcuda_outputs* out, uint32_t sample_lo, uint32_t sample_hi,
                         bool accumulate) {
    REQUIRE(out->width == parent->width && out->height == parent->height, "output size must equal the camera raster size");
    const uint32_t o = settings->outputs;
    rtcuda_scene* first = parent->subs[0];
    const size_t n = parent->subs.size();
    std::vector<size_t> sent_words(n, 0);
    for_each_device(n, [&](size_t r) {
        rtcuda_scene* sub = parent->subs[r];
        enter(sub);
        cudaStream_t st = sub->ctx->stream;
        if (r == 0) {
            render_device(sub, settings, out, sample_lo, sample_hi, accumulate);
            return;
        }
        rtcuda_outputs dev = staging_planes(sub, o, *out);
        render_device(sub, settings, &dev, sample_lo, sample_hi, false);
        PlaneSlot dp[N_PLANES];
        planes_of(dev, o, dp);
        const size_t words = pack_owned(sub, dp, true);
        sent_words[r] = words;
        if (!words) return;
        if (words > first->peer_recv_words[r]) {   // receive buffer of rank r on GPU 0 (slot r is only ever touched by this thread)
            CK(cudaStreamSynchronize(st));
            CK(cudaSetDevice(first->ctx->device));
            if (first->peer_recv[r]) cudaFree(first->peer_recv[r]);
            first->peer_recv[r] = nullptr; first->peer_recv_words[r] = 0;
            const cudaError_t e = cudaMalloc((void**)&first->peer_recv[r], words * 4);
            cudaSetDevice(sub->ctx->device);
            CK(e);
            first->peer_recv_words[r] = words;
        }
        CK(cudaMemcpyPeerAsync(first->peer_recv[r], first->ctx->device, sub->packed, sub->ctx->device, words * 4, st));
        CK(cudaEventRecord(sub->sent, st));
        CK(cudaStreamSynchronize(st));
    });
    enter(first);
    cudaStream_t st0 = first->ctx->stream;
    PlaneSlot up[N_PLANES];
    planes_of(*out, o, up);
    for (size_t r = 1; r < n; r++) {
        rtcuda_scene* sub = parent->subs[r];
        if (!sent_words[r]) continue;
        if (!first->peer_list[r]) {   // rank r's tile table, once, on GPU 0
            CK(cudaMalloc((void**)&first->peer_list[r], std::max<size_t>(1, sub->host_tiles.size()) * sizeof(TileRec)));
            CK(cudaMemcpyAsync(first->peer_list[r], sub->host_tiles.data(), sub->host_tiles.size() * sizeof(TileRec), cudaMemcpyHostToDevice, st0));
        }
        CK(cudaStreamWaitEvent(st0, sub->sent, 0));
        size_t off = 0;
        for (int i = 0; i < N_PLANES; i++) {
            if (!up[i].ptr) continue;
            launch_pack_tiles(st0, accumulate && i == 0 ? 2 : 1, first->peer_list[r], (uint32_t)sub->host_tiles.size(), first->width, up[i].ch, (uint32_t*)up[i].ptr,
                              first->peer_recv[r] + off, first->lc);
            off += (size_t)sub->n_my_pixels * up[i].ch;
        }
    }
    CK(cudaStreamSynchronize(st0));
}

// Host-array queries on a multi-device scene: contiguous slices of the rays, one per GPU, each on its own host thread. Every ray is
// traced on a replica of the same tree, so the results are those of one GPU.
void multi_query_host(rtcuda_scene* parent, const QueryPtrs& q, uint64_t count) {
    const size_t n = parent->subs.size();
    const uint64_t per = (count + n - 1) / n;
    for_each_device(n, [&](size_t r) {
        const uint64_t lo = std::min<uint64_t>(count, per * r), hi = std::min<uint64_t>(count, lo + per);
        if (hi == lo) return;
        enter(parent->subs[r]);
        const QueryPtrs slice{q.rays + 8 * lo, q.t ? q.t + lo : nullptr, q.ids ? q.ids + 2 * lo : nullptr, q.uv ? q.uv + 2 * lo : nullptr,
                              q.occluded ? q.occluded + lo : nullptr, q.surfaces ? q.surfaces + lo : nullptr};
        query_host(parent->subs[r], slice, hi - lo);
    });
}

// Host-array radiance on a multi-device scene: contiguous slices of the rays, one per GPU, each keeping its rays' stream keys
void multi_radiance_host(rtcuda_scene* parent, const rtcuda_settings* settings, const float* rays, uint64_t count, uint32_t stream_base,
                         float* radiance) {
    const size_t n = parent->subs.size();
    const uint64_t per = (count + n - 1) / n;
    for_each_device(n, [&](size_t r) {
        const uint64_t lo = std::min<uint64_t>(count, per * r), hi = std::min<uint64_t>(count, lo + per);
        if (hi == lo) return;
        enter(parent->subs[r]);
        radiance_host(parent->subs[r], settings, rays + 8 * lo, hi - lo, stream_base + (uint32_t)lo, radiance + 3 * lo);
    });
}

// rtcuda_get_stats of a multi-device scene: ray / fetch / launch counters summed over the GPUs, times = the slowest GPU
rtcuda_stats multi_stats(const rtcuda_scene* parent) {
    rtcuda_stats t{};
    bool first = true;
    for (const rtcuda_scene* sub : parent->subs) {
        const rtcuda_stats& a = sub->stats;
        t.samples += a.samples; t.primary_rays += a.primary_rays; t.bounce_rays += a.bounce_rays; t.shadow_rays += a.shadow_rays; t.aov_rays += a.aov_rays;
        t.nodes_fetched += a.nodes_fetched; t.prims_fetched += a.prims_fetched; t.extend_nodes += a.extend_nodes; t.extend_prims += a.extend_prims;
        t.shadow_nodes += a.shadow_nodes; t.shadow_prims += a.shadow_prims; t.shaded_vertices += a.shaded_vertices;
        t.kernel_launches += a.kernel_launches; t.extend_launches += a.extend_launches; t.shade_launches += a.shade_launches; t.shadow_launches += a.shadow_launches;
        t.nonfinite_values += a.nonfinite_values; t.primary_rays_culled += a.primary_rays_culled; t.final_rays_skipped += a.final_rays_skipped;
        t.bvh_fallback_lbvh = std::max(t.bvh_fallback_lbvh, a.bvh_fallback_lbvh);
        t.render_ms = std::max(t.render_ms, a.render_ms); t.bvh_build_ms = std::max(t.bvh_build_ms, a.bvh_build_ms); t.upload_ms = std::max(t.upload_ms, a.upload_ms);
        t.extend_ms = std::max(t.extend_ms, a.extend_ms); t.shade_ms = std::max(t.shade_ms, a.shade_ms); t.shadow_ms = std::max(t.shadow_ms, a.shadow_ms);
        t.other_ms = std::max(t.other_ms, a.other_ms); t.gather_ms = std::max(t.gather_ms, a.gather_ms);
        t.pixels_dropped += a.pixels_dropped;
        t.update_ms = std::max(t.update_ms, a.update_ms);
        if (first) {
            t.bvh_node_count = a.bvh_node_count; t.bvh_prim_count = a.bvh_prim_count;
            t.bvh_sah_cost = a.bvh_sah_cost; t.bvh_last_update = a.bvh_last_update;   // (the same on every GPU: same data, same decision)
            first = false;
        }
    }
    return t;
}

template <typename F>
rtcuda_status guarded(F&& f) {
    try {
        f();
        g_last_error.clear();
        return RTCUDA_OK;
    } catch (const RtError& e) {
        g_last_error = e.msg;
        return e.status;
    } catch (const std::bad_alloc&) {
        g_last_error = "host allocation failed";
        return RTCUDA_ERR_OUT_OF_MEMORY;
    } catch (const std::exception& e) {
        g_last_error = e.what();
        return RTCUDA_ERR_CUDA;
    }
}

}  // namespace

extern "C" {

namespace {
// One single-device context (the per-GPU part of rtcuda_init).
rtcuda_ctx* make_device_ctx(const rtcuda_backend_settings& bs, int device_count) {
    REQUIRE(bs.device_id >= 0 && bs.device_id < device_count, "device_id out of range");
    REQUIRE(bs.tile_world <= 1 || bs.tile_rank < bs.tile_world, "tile_rank >= tile_world");
    REQUIRE(bs.tile_size == 0 || (bs.tile_size >= 8 && bs.tile_size <= 64 && (bs.tile_size & (bs.tile_size - 1)) == 0),
            "tile_size must be 0 or a power of two in [8, 64]");
    auto ctx = std::make_unique<rtcuda_ctx>();
    ctx->device = bs.device_id;
    ctx->bs = bs;
    CK(cudaSetDevice(ctx->device));
    ctx->stream = g_stream_cache.take(ctx->device);
    if (!ctx->stream) CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    cudaMemPool_t pool;
    CK(cudaDeviceGetDefaultMemPool(&pool, ctx->device));
    uint64_t keep = UINT64_MAX;   // freed blocks stay in the pool until rtcuda_release_cached_memory
    CK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    return ctx.release();
}
void destroy_ctx(rtcuda_ctx* ctx) {
    if (!ctx) return;
    for (rtcuda_ctx* sub : ctx->subs) destroy_ctx(sub);
    if (ctx->stream) g_stream_cache.park(ctx->device, ctx->stream);   // (pending stream-ordered frees stay ordered before whatever the next owner submits)
    delete ctx;
}
}  // namespace

RTCUDA_API rtcuda_status rtcuda_init(const rtcuda_backend_settings* settings, rtcuda_ctx** out_ctx) {
    return guarded([&] {
        REQUIRE(settings && out_ctx, "null argument");
        *out_ctx = nullptr;
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0) throw RtError{RTCUDA_ERR_NO_DEVICE, "no CUDA device: the cuda backend has no CPU fallback"};
        if (settings->num_devices <= 1) {
            rtcuda_backend_settings bs = *settings;
            if (bs.num_devices == 1) bs.device_id = bs.device_ids[0];
            bs.num_devices = 0;
            *out_ctx = make_device_ctx(bs, count);
            return;
        }
        // multi-device: one sub-context per GPU, rank r of num_devices in the tile deal
        const uint32_t n = settings->num_devices;
        REQUIRE(n <= RTCUDA_MAX_DEVICES, "num_devices > RTCUDA_MAX_DEVICES");
        REQUIRE(settings->tile_world <= 1, "tile_rank / tile_world cannot be combined with num_devices > 1");
        for (uint32_t i = 0; i < n; i++) {
            // (entries may repeat: several ranks then share a GPU — no use in production, but it lets a one-GPU box run this path)
            REQUIRE(settings->device_ids[i] >= 0 && settings->device_ids[i] < count, "device_ids entry out of range");
        }
        std::unique_ptr<rtcuda_ctx, void (*)(rtcuda_ctx*)> parent(new rtcuda_ctx(), destroy_ctx);
        parent->device = settings->device_ids[0];
        parent->bs = *settings;
        for (uint32_t i = 0; i < n; i++) {
            rtcuda_backend_settings bs = *settings;
            bs.device_id = settings->device_ids[i];
            bs.num_devices = 0;
            bs.tile_rank = i;
            bs.tile_world = n;
            parent->subs.push_back(make_device_ctx(bs, count));
        }
        // NVLink peer access in both directions between every pair (geometry slices are forwarded all-to-all, owned pixels go to
        // GPU 0): what the GPUs pass between them lives in plain allocations
        static std::mutex peer_mu;
        static uint64_t peer_done[64] = {0};   // per process: pairs already set up (the calls below cost milliseconds each)
        std::lock_guard<std::mutex> peer_lock(peer_mu);
        for (uint32_t i = 0; i < n; i++) {
            CK(cudaSetDevice(settings->device_ids[i]));
            for (uint32_t j = 0; j < n; j++) {
                if (settings->device_ids[i] == settings->device_ids[j]) continue;
                const int di = settings->device_ids[i] & 63, dj = settings->device_ids[j] & 63;
                if (peer_done[di] & (1ull << dj)) continue;
                peer_done[di] |= 1ull << dj;
                int can = 0;
                CK(cudaDeviceCanAccessPeer(&can, settings->device_ids[i], settings->device_ids[j]));
                if (!can) continue;   // copies between the two then go through the host (still correct)
                const cudaError_t pe = cudaDeviceEnablePeerAccess(settings->device_ids[j], 0);
                if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) CK(pe);
                cudaGetLastError();   // (plain allocations only: the pools stay private to their device, see DevBuf::peer_visible)
            }
        }
        *out_ctx = parent.release();
    });
}

RTCUDA_API void rtcuda_shutdown(rtcuda_ctx* ctx) { destroy_ctx(ctx); }

RTCUDA_API rtcuda_status rtcuda_scene_upload(rtcuda_ctx* ctx, const rtcuda_scene_desc* desc, rtcuda_scene** out_scene) {
    return guarded([&] {
        REQUIRE(ctx && desc && out_scene, "null argument");
        *out_scene = nullptr;
        auto s = std::make_unique<rtcuda_scene>();
        s->ctx = ctx;
        if (!ctx->subs.empty()) {
            try {
                multi_upload(ctx, desc, s.get());
            } catch (...) {
                multi_release(s.get());
                throw;
            }
            *out_scene = s.release();
            return;
        }
        CK(cudaSetDevice(ctx->device));
        tls_stream = ctx->stream;
        upload_scene(s.get(), desc);
        *out_scene = s.release();
    });
}

RTCUDA_API rtcuda_status rtcuda_scene_update(rtcuda_scene* scene, const rtcuda_scene_desc* desc) {
    return guarded([&] {
        REQUIRE(scene && desc, "null argument");
        if (!scene->subs.empty()) { multi_update(scene, desc); return; }
        validate_update(scene, desc);
        CK(cudaSetDevice(scene->ctx->device));
        tls_stream = scene->ctx->stream;
        update_scene(scene, desc);
    });
}

RTCUDA_API void rtcuda_release_cached_memory(void) {
    g_arena_cache.release_all();
    g_plain_cache.release_all();
    g_stream_cache.release_all();
    g_pinned_cache.release_all();
    int cur = 0, count = 0;
    if (cudaGetDevice(&cur) != cudaSuccess || cudaGetDeviceCount(&count) != cudaSuccess) return;
    for (int dev = 0; dev < count; dev++) {   // every device this process may have used
        cudaMemPool_t pool;
        if (cudaSetDevice(dev) != cudaSuccess || cudaDeviceGetDefaultMemPool(&pool, dev) != cudaSuccess) continue;
        uint64_t reserved = 0;
        if (cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved) != cudaSuccess || reserved == 0) continue;
        cudaDeviceSynchronize();
        cudaMemPoolTrimTo(pool, 0);
    }
    cudaSetDevice(cur);
    cudaGetLastError();
}

RTCUDA_API void* rtcuda_host_alloc(size_t bytes) {
    if (!bytes) return nullptr;
    size_t got = 0;
    void* p = g_pinned_cache.take(bytes, got);
    if (p) g_host_allocs.add(p, got);
    return p;
}

RTCUDA_API void rtcuda_host_free(void* p) {
    if (!p) return;
    const size_t bytes = g_host_allocs.take(p);
    if (bytes) g_pinned_cache.park(p, bytes);
}

RTCUDA_API void rtcuda_scene_release(rtcuda_scene* scene) {
    if (!scene) return;
    if (!scene->subs.empty()) {
        multi_release(scene);
        delete scene;
        return;
    }
    cudaSetDevice(scene->ctx->device);
    tls_stream = scene->ctx->stream;
    cudaStreamSynchronize(tls_stream);
    delete scene;
    cudaStreamSynchronize(tls_stream);
}

RTCUDA_API rtcuda_status rtcuda_render(rtcuda_scene* scene, const rtcuda_settings* settings, rtcuda_outputs* outputs) {
    return guarded([&] {
        REQUIRE(scene && settings && outputs, "null argument");
        if (!scene->subs.empty()) { multi_render_host(scene, settings, outputs); return; }
        CK(cudaSetDevice(scene->ctx->device));
        tls_stream = scene->ctx->stream;
        render_host(scene, settings, outputs);
    });
}

RTCUDA_API rtcuda_status rtcuda_render_device(rtcuda_scene* scene, const rtcuda_settings* settings, rtcuda_outputs* device_outputs) {
    return guarded([&] {
        REQUIRE(scene && settings && device_outputs, "null argument");
        if (!scene->subs.empty()) { multi_render_device(scene, settings, device_outputs, 0, 0, false); return; }
        CK(cudaSetDevice(scene->ctx->device));
        tls_stream = scene->ctx->stream;
        render_device(scene, settings, device_outputs);
    });
}

namespace {
rtcuda_status render_samples(rtcuda_scene* scene, const rtcuda_settings* settings, uint32_t sample_lo, uint32_t sample_hi, float* beauty_sum, bool accumulate) {
    return guarded([&] {
        REQUIRE(scene && settings && beauty_sum, "null argument");
        REQUIRE(sample_hi != 0, "empty sample range");
        rtcuda_settings st = *settings;
        st.outputs = RTCUDA_AOV_BEAUTY;
        rtcuda_outputs o{};
        o.width = scene->width; o.height = scene->height;
        o.beauty = beauty_sum;
        if (!scene->subs.empty()) { multi_render_device(scene, &st, &o, sample_lo, sample_hi, accumulate); return; }
        CK(cudaSetDevice(scene->ctx->device));
        tls_stream = scene->ctx->stream;
        render_device(scene, &st, &o, sample_lo, sample_hi, accumulate);
    });
}
}  // namespace

RTCUDA_API rtcuda_status rtcuda_render_samples_device(rtcuda_scene* scene, const rtcuda_settings* settings, uint32_t sample_lo,
                                                      uint32_t sample_hi, float* beauty_sum) {
    return render_samples(scene, settings, sample_lo, sample_hi, beauty_sum, false);
}

RTCUDA_API rtcuda_status rtcuda_render_samples_accumulate_device(rtcuda_scene* scene, const rtcuda_settings* settings, uint32_t sample_lo,
                                                                 uint32_t sample_hi, float* beauty_sum) {
    return render_samples(scene, settings, sample_lo, sample_hi, beauty_sum, true);
}

RTCUDA_API rtcuda_status rtcuda_render_pixel(rtcuda_scene* scene, const rtcuda_settings* settings, uint32_t x, uint32_t y,
                                             uint32_t sample_lo, uint32_t sample_hi, rtcuda_pixel_output* out) {
    return guarded([&] {
        REQUIRE(scene && settings && (out || sample_hi == sample_lo), "null argument");
        rtcuda_scene* one = scene->subs.empty() ? scene : scene->subs[0];   // a pixel's samples do not depend on the tile deal
        CK(cudaSetDevice(one->ctx->device));
        tls_stream = one->ctx->stream;
        render_pixel(one, settings, x, y, sample_lo, sample_hi, out);
    });
}

namespace {
rtcuda_status query(rtcuda_scene* scene, const QueryPtrs& q, uint64_t count, bool device_arrays) {
    return guarded([&] {
        validate_query(scene, q, count);
        if (count == 0) return;
        if (!device_arrays && !scene->subs.empty()) { multi_query_host(scene, q, count); return; }
        rtcuda_scene* one = scene->subs.empty() ? scene : scene->subs[0];   // device arrays live on device_ids[0]
        CK(cudaSetDevice(one->ctx->device));
        tls_stream = one->ctx->stream;
        if (!device_arrays) { query_host(one, q, count); return; }
        REQUIRE(((uintptr_t)q.rays & 15u) == 0, "rays must be 16-byte aligned");
        REQUIRE(((uintptr_t)q.surfaces & 15u) == 0, "surfaces must be 16-byte aligned");
        require_device_pointer(q.rays, one->ctx->device, "rays");
        require_device_pointer(q.t, one->ctx->device, "t");
        require_device_pointer(q.ids, one->ctx->device, "ids");
        require_device_pointer(q.uv, one->ctx->device, "barycentrics");
        require_device_pointer(q.occluded, one->ctx->device, "occluded");
        require_device_pointer(q.surfaces, one->ctx->device, "surfaces");
        query_device(one, q, count);
    });
}
}  // namespace

RTCUDA_API rtcuda_status rtcuda_trace_rays(rtcuda_scene* scene, const float* rays, uint64_t count, float* t, uint32_t* ids, float* barycentrics) {
    return query(scene, QueryPtrs{rays, t, ids, barycentrics, nullptr, nullptr}, count, false);
}
RTCUDA_API rtcuda_status rtcuda_trace_rays_device(rtcuda_scene* scene, const float* rays, uint64_t count, float* t, uint32_t* ids,
                                                  float* barycentrics) {
    return query(scene, QueryPtrs{rays, t, ids, barycentrics, nullptr, nullptr}, count, true);
}
RTCUDA_API rtcuda_status rtcuda_occluded(rtcuda_scene* scene, const float* rays, uint64_t count, uint8_t* occluded) {
    return query(scene, QueryPtrs{rays, nullptr, nullptr, nullptr, occluded, nullptr}, count, false);
}
RTCUDA_API rtcuda_status rtcuda_occluded_device(rtcuda_scene* scene, const float* rays, uint64_t count, uint8_t* occluded) {
    return query(scene, QueryPtrs{rays, nullptr, nullptr, nullptr, occluded, nullptr}, count, true);
}
// (a NULL surfaces pointer is refused as "every output is NULL")
RTCUDA_API rtcuda_status rtcuda_trace_surfaces(rtcuda_scene* scene, const float* rays, uint64_t count, rtcuda_surface* surfaces) {
    return query(scene, QueryPtrs{rays, nullptr, nullptr, nullptr, nullptr, surfaces}, count, false);
}
RTCUDA_API rtcuda_status rtcuda_trace_surfaces_device(rtcuda_scene* scene, const float* rays, uint64_t count, rtcuda_surface* surfaces) {
    return query(scene, QueryPtrs{rays, nullptr, nullptr, nullptr, nullptr, surfaces}, count, true);
}

namespace {
rtcuda_status radiance_call(rtcuda_scene* scene, const rtcuda_settings* settings, const float* rays, uint64_t count, uint32_t stream_base,
                            float* radiance, bool device_arrays) {
    return guarded([&] {
        validate_radiance(scene, settings, rays, count, stream_base, radiance);
        if (count == 0) return;
        if (!device_arrays && !scene->subs.empty()) { multi_radiance_host(scene, settings, rays, count, stream_base, radiance); return; }
        rtcuda_scene* one = scene->subs.empty() ? scene : scene->subs[0];   // device arrays live on device_ids[0]
        CK(cudaSetDevice(one->ctx->device));
        tls_stream = one->ctx->stream;
        if (!device_arrays) { radiance_host(one, settings, rays, count, stream_base, radiance); return; }
        REQUIRE(((uintptr_t)rays & 15u) == 0, "rays must be 16-byte aligned");
        require_device_pointer(rays, one->ctx->device, "rays");
        require_device_pointer(radiance, one->ctx->device, "radiance");
        radiance_device(one, settings, rays, count, stream_base, radiance);
    });
}
}  // namespace

RTCUDA_API rtcuda_status rtcuda_radiance(rtcuda_scene* scene, const rtcuda_settings* settings, const float* rays, uint64_t count,
                                         uint32_t stream_base, float* radiance) {
    return radiance_call(scene, settings, rays, count, stream_base, radiance, false);
}
RTCUDA_API rtcuda_status rtcuda_radiance_device(rtcuda_scene* scene, const rtcuda_settings* settings, const float* rays, uint64_t count,
                                                uint32_t stream_base, float* radiance) {
    return radiance_call(scene, settings, rays, count, stream_base, radiance, true);
}

RTCUDA_API rtcuda_status rtcuda_get_stats(const rtcuda_scene* scene, rtcuda_stats* out) {
    return guarded([&] {
        REQUIRE(scene && out, "null argument");
        *out = scene->subs.empty() ? scene->stats : multi_stats(scene);
    });
}

RTCUDA_API const char* rtcuda_last_error(void) { return g_last_error.c_str(); }
RTCUDA_API uint32_t rtcuda_abi_version(void) { return RTCUDA_ABI_VERSION; }

RTCUDA_API uint32_t rtcuda_abi_struct_sizes(uint32_t* out, uint32_t capacity) {
    const uint32_t sizes[] = {sizeof(rtcuda_camera), sizeof(rtcuda_shape), sizeof(rtcuda_instance), sizeof(rtcuda_light),
                              sizeof(rtcuda_material), sizeof(rtcuda_texture), sizeof(rtcuda_image), sizeof(rtcuda_scene_desc),
                              sizeof(rtcuda_settings), sizeof(rtcuda_backend_settings), sizeof(rtcuda_outputs),
                              sizeof(rtcuda_pixel_output), sizeof(rtcuda_stats)};
    const uint32_t n = sizeof(sizes) / sizeof(sizes[0]);
    for (uint32_t i = 0; i < n && i < capacity; i++) out[i] = sizes[i];
    return n;
}

}  // extern "C"
