// ccu_host.h - host-side state behind the C ABI (include/chunkycu.h): the context object, small RAII helpers and the
// error plumbing shared by chunkycu.cu (single-GPU entry points) and ccu_group.cu (multi-GPU entry points).
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/chunkycu.h"
#include "ccu_device.cuh"

namespace ccu_host {

int fail(int code, const char *fmt, ...);          // sets the calling thread's error string, returns code
const char *last_error();

#define CU(call)                                                                                                          \
    do {                                                                                                                  \
        cudaError_t e_ = (call);                                                                                          \
        if (e_ != cudaSuccess)                                                                                            \
            return ccu_host::fail(e_ == cudaErrorMemoryAllocation ? CCU_ENOMEM : CCU_ECUDA, "%s: %s (%s:%d)", #call,      \
                                  cudaGetErrorString(e_), __FILE__, __LINE__);                                            \
    } while (0)

// Owning holders of CUDA resources: move-only, released by their destructor.  Nothing outside them frees a resource.
template <class T>
struct DevBuf {
    // never smaller than one 64-byte record: the straight-line kernels read element 0 of an empty array on lanes that have no
    // work (the value is dropped)
    static constexpr size_t MIN_ELEMS = 64 / sizeof(T) > 4 ? 64 / sizeof(T) : 4;
    T *p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    DevBuf(DevBuf &&o) noexcept : p(std::exchange(o.p, nullptr)), n(std::exchange(o.n, 0)) {}
    DevBuf &operator=(DevBuf &&o) noexcept { std::swap(p, o.p); std::swap(n, o.n); return *this; }
    ~DevBuf() { release(); }
    cudaError_t alloc(size_t count) {
        release();
        n = count;
        const size_t a = std::max<size_t>(count, MIN_ELEMS);   // zero-length arrays become zero words (ClIntBuffer.java:15-18)
        cudaError_t e = cudaMalloc(&p, a * sizeof(T));
        if (e != cudaSuccess) { p = nullptr; n = 0; }
        return e;
    }
    cudaError_t upload(const T *host, size_t count, cudaStream_t st) {
        cudaError_t e = alloc(count);
        if (e != cudaSuccess) return e;
        e = cudaMemsetAsync(p, 0, std::max<size_t>(count, MIN_ELEMS) * sizeof(T), st);
        if (e != cudaSuccess) return e;
        if (count) e = cudaMemcpyAsync(p, host, count * sizeof(T), cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) return e;
        return cudaStreamSynchronize(st);   // host memory is not retained past the call
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
    size_t bytes() const { return p ? std::max<size_t>(n, MIN_ELEMS) * sizeof(T) : 0; }
};

// an event, a stream or pinned host memory; converts to the raw handle / pointer
template <class H, auto Destroy>
struct Handle {
    H h = nullptr;
    Handle() = default;
    Handle(Handle &&o) noexcept : h(std::exchange(o.h, nullptr)) {}
    Handle &operator=(Handle &&o) noexcept { std::swap(h, o.h); return *this; }
    ~Handle() { reset(); }
    operator H() const { return h; }
    void reset() {
        if (h) Destroy(h);
        h = nullptr;
    }
};
struct Event : Handle<cudaEvent_t, cudaEventDestroy> {
    cudaError_t create(unsigned flags) { reset(); return cudaEventCreateWithFlags(&h, flags); }
};
struct Stream : Handle<cudaStream_t, cudaStreamDestroy> {
    cudaError_t create() { reset(); return cudaStreamCreateWithFlags(&h, cudaStreamNonBlocking); }
};
template <class T>
struct HostBuf : Handle<T *, cudaFreeHost> {
    cudaError_t alloc(size_t count) {
        this->reset();
        cudaError_t e = cudaMallocHost(&this->h, count * sizeof(T));
        if (e != cudaSuccess) this->h = nullptr;
        return e;
    }
};

constexpr int SEED_SLOTS = 4, SEED_SLOT_INTS = 32768;   // one launch covers at most 32768 passes (16-bit pass index in the wavefront kernel)
constexpr int MERGE_CHUNKS = 8;                         // read-back chunks of a window merge, one event each

// The seed words of the passes in flight (the only per-pass host->device traffic, OpenClPathTracingRenderer.java:106-109),
// staged in a small ring of pinned slots so that a render call neither retains the caller's array nor waits for the passes
// in flight.  Allocated whole or not at all.
struct SeedRing {
    DevBuf<int> dev;
    HostBuf<int> pinned;
    Event ev[SEED_SLOTS];   // last launch that read each slot
    int slot = 0;
};

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        int cur = -1;
        cudaGetDevice(&cur);
        if (prev >= 0 && cur != prev) cudaSetDevice(prev);
    }
};

// One asynchronous read-back + merge into the host sample buffer (ccu_render_merge_async, ccu_group_render_merge_async).
// The owner's lock guards the fields; the worker writes status / error only, and only before it ends.
struct MergeJob {
    std::thread worker;
    bool active = false;
    int status = CCU_OK;
    std::string error;

    // runs `body` on the worker; body returns a CCU_* code and sets the thread's error text when it fails
    template <class F>
    void start(F body) {
        active = true;
        status = CCU_OK;
        worker = std::thread([this, body] {
            const int rc = body();
            if (rc != CCU_OK) { status = rc; error = last_error(); }
        });
    }
    // waits for the worker with `lk` (the owner's lock) released; returns the worker's status and clears it
    int join(std::unique_lock<std::mutex> &lk) {
        if (!active) return CCU_OK;
        std::thread t = std::move(worker);
        lk.unlock();
        if (t.joinable()) t.join();
        lk.lock();
        active = false;
        if (status == CCU_OK) return CCU_OK;
        const int rc = status;
        status = CCU_OK;
        return fail(rc, "%s", error.c_str());
    }
};

// The scalar state of a committed scene: what commit derived from the uploads, and what the uploads set besides arrays.
struct SceneInfo {
    int depth = 0, sky_res = 0;
    int world_root = 0, actor_root = 0, use_bvh2 = 0, use_air = 0, air_deep = 0;
    int world_bvh_empty = 1, actor_bvh_empty = 1;   // the bvh.h:23-32 probe of the committed BVHs
    int cell_level = 0, top_log2 = 0, use_wide = 0, air_cell_level = 4, air_top_log2 = 0;
    int atlas_w = 0, atlas_h = 0, atlas_layers = 0;
    int has_specular = 0;   // a material word 5 is not 0: CCU_RENDER_SPECULAR launches the specular kernels
    int has_emitters = 0;   // the emitter table is not empty: CCU_RENDER_EMITTER_SAMPLING launches the NEE kernels
    int emit_g0[3] = {0, 0, 0}, emit_dim[3] = {0, 0, 0}, emit_shift = 3;   // emitter grid (EmitView::g0 ...)
    int has_model_emitters = 0;   // the wider table of CCU_RENDER_EMITTER_MODELS exists: a model emitter is in the octree
    int memit_g0[3] = {0, 0, 0}, memit_dim[3] = {0, 0, 0}, memit_shift = 3;   // its grid
    int has_biome = 0;      // biome colours were set: CCU_RENDER_BIOME_TINT launches the biome kernels
    int biome_box[4] = {0, 0, 0, 0};   // the biome grid's chunk box (BiomeView::x0, z0, gx, gz)
    int has_fog = 0;        // ccu_scene_set_fog with sigma > 0: CCU_RENDER_FOG launches the fog kernels
    float fog_sigma = 0, fog_sky = 0, fog_color[3] = {0, 0, 0};   // DScene::fog_*
    int fog_fast = 0;
    int has_clouds = 0;     // a cloud mask with a set cell: CCU_RENDER_CLOUDS launches the cloud kernels
    float cloud_inv = 0, cloud_y0 = 0, cloud_y1 = 0, cloud_u0 = 0, cloud_v0 = 0;   // CloudView::inv ...
    void set_fog(float sigma, float sky, const float *color, int fast) {   // color may be null for sigma = 0 (no fog)
        has_fog = sigma > 0.0f;
        fog_sigma = sigma;
        fog_sky = sky;
        for (int i = 0; i < 3; i++) fog_color[i] = color ? color[i] : 0.0f;
        fog_fast = fast;
    }
    float sky_intensity = 0;
    int sun_host[6] = {0, 0, 0, 0, 0, 0};
    bool have_sun = false, have_atlas = false, have_sky = false;
    float3 su{}, sv{}, sw{};   // sun basis (k_sun_setup)
    float sun_radius_cos = 0;
};

// The reference's packed int arrays, one ccu_scene_set_* call each.
enum SceneArray { OCTREE, BLOCK_PALETTE, QUAD_MODELS, AABB_MODELS, MAT_PALETTE, TRIANGLES, WORLD_BVH, ACTOR_BVH, N_ARRAYS };
struct ArrayDesc {
    const char *setter;   // entry point named in error messages
    bool optional;        // released by ccu_scene_begin; absent at commit, it is one zero word (empty palette / EMPTY_NODE)
};
constexpr ArrayDesc ARRAY_DESC[N_ARRAYS] = {
    {"ccu_scene_set_octree", false},      {"ccu_scene_set_block_palette", false}, {"ccu_scene_set_quad_models", true},
    {"ccu_scene_set_aabb_models", true},  {"ccu_scene_set_material_palette", false}, {"ccu_scene_set_triangles", true},
    {"ccu_scene_set_world_bvh", true},    {"ccu_scene_set_actor_bvh", true},
};
// The device buffer of one packed array and the host copy commit builds its layouts from.  `host` is set exactly while `dev`
// holds the array; it never changes once set, so a replica shares it.
struct PackedArray {
    DevBuf<int> dev;
    std::shared_ptr<const std::vector<int>> host;
};

// The biome colours of ccu_scene_set_biome_colors as given (n chunks); commit lays them out (build_biome_layout).
struct BiomeColors {
    std::vector<int32_t> chunks;   // n x {cx, cz}
    std::vector<float> rgb;        // n x 3 planes x 256 texels x 3
};

// The cloud layer of ccu_scene_set_clouds (DESIGN §15): the mask bit-packed as the kernels read it (CloudView), and the
// parameters; commit uploads the mask.
constexpr int CLOUD_CELLS = 256 * 256, CLOUD_WORDS = CLOUD_CELLS / 32;
struct CloudLayer {
    unsigned bits[CLOUD_WORDS] = {};
    bool any = false;   // a cell is set
    float inv = 0, y0 = 0, y1 = 0, u0 = 0, v0 = 0;
};

// Everything a context knows about its scene: the uploads, the layouts commit builds from them, and the launch view.
struct Scene {
    PackedArray arrays[N_ARRAYS];
    DevBuf<unsigned> top, wide;                       // value-carrying octree layout
    DevBuf<unsigned> air_top, air_wide, air_bricks;   // march layout (ccu_march.cuh)
    DevBuf<int> world_rec, actor_rec, tris2;          // BVH stage layout (ccu_queue.cuh)
    DevBuf<int> block_rec, mat_rec, quad_rec, aabb_rec;   // 16-byte-vectorised palettes (DScene::block_rec ...)
    DevBuf<int> emit, emit_off, emit_list;                // emitter table and cell lists (EmitView)
    DevBuf<int> memit, memit_off, memit_list, memit_head, memit_prim;   // the wider table with model emitters (EmitView)
    DevBuf<int> biome_grid;                               // biome colours (BiomeView), only when set
    DevBuf<float4> biome_tiles;
    std::shared_ptr<const BiomeColors> biome;             // set while the scene has biome colours; shared by a replica
    DevBuf<unsigned> cloud_mask;                          // the cloud mask (CloudView), only when set
    std::shared_ptr<const CloudLayer> clouds;             // set while the scene has a cloud layer; shared by a replica
    DevBuf<uchar4> atlas, sky;
    SceneInfo info;
    ccu::DScene view{};   // every field that depends on the committed scene alone (commit, replicate_scene)
    ccu::EmitView emit_view{};   // the emitter table's launch view (fill_view, with `view`)
    ccu::EmitView memit_view{};  // the wider table's launch view (CCU_RENDER_EMITTER_MODELS)
    ccu::BiomeView biome_view{};  // the biome colours' launch view (CCU_RENDER_BIOME_TINT)
    ccu::CloudView cloud_view{};  // the cloud layer's launch view (CCU_RENDER_CLOUDS)

    // Calls f(a's buffer, b's same buffer) for every device array of a scene (replicate_scene, ccu_scene_device_bytes).
    template <class F>
    static void each_buf(Scene &a, Scene &b, F f) {
        for (int i = 0; i < N_ARRAYS; i++) f(a.arrays[i].dev, b.arrays[i].dev);
        f(a.top, b.top); f(a.wide, b.wide); f(a.air_top, b.air_top); f(a.air_wide, b.air_wide); f(a.air_bricks, b.air_bricks);
        f(a.world_rec, b.world_rec); f(a.actor_rec, b.actor_rec); f(a.tris2, b.tris2); f(a.block_rec, b.block_rec);
        f(a.mat_rec, b.mat_rec); f(a.quad_rec, b.quad_rec); f(a.aabb_rec, b.aabb_rec); f(a.atlas, b.atlas); f(a.sky, b.sky);
        f(a.emit, b.emit); f(a.emit_off, b.emit_off); f(a.emit_list, b.emit_list);
        f(a.memit, b.memit); f(a.memit_off, b.memit_off); f(a.memit_list, b.memit_list); f(a.memit_head, b.memit_head);
        f(a.memit_prim, b.memit_prim); f(a.biome_grid, b.biome_grid); f(a.biome_tiles, b.biome_tiles);
        f(a.cloud_mask, b.cloud_mask);
    }
};

}  // namespace ccu_host

// Members are destroyed in reverse order of declaration: the streams are declared first so that they outlive every buffer and
// event used on them.  ccu_ctx_destroy joins the merge worker and synchronises both streams before the delete.
struct ccu_ctx {
    int device = 0;
    ccu_host::Stream stream;        // render stream
    ccu_host::Stream copy_stream;   // read-back of finished windows, camera-ray uploads
    ccu_host::Event ev0, ev1;
    ccu_host::Event chunk_ev[ccu_host::MERGE_CHUNKS];   // read-back chunks of a merge
    ccu_host::Event window_ev;      // the window being merged is complete on the render stream
    // Locking: `mu` guards every field below and is never held across a wait for rendering work (ccu_render_sync waits on an
    // event outside the lock), so preview / tonemap / camera calls from other threads are not blocked by a long batch;
    // `cam_mu` serialises camera updates.
    std::mutex mu, cam_mu;
    int sm_count = 0;

    ccu_host::Scene scene;
    bool committed = false;   // `scene` is complete: render calls launch on it
    double commit_ms = 0;     // host time of the last ccu_scene_commit
    ccu_host::DevBuf<float> unorm;

    // camera: pre-generated rays are double buffered so that an upload overlaps the passes in flight
    int projector_type = 0;
    float cam[15] = {0};
    ccu_host::DevBuf<float> rays[2];
    ccu_host::Event rays_used[2];   // last launch that read rays[i]
    int rays_active = 0;
    bool have_camera = false;

    // render target: the accumulation window is double buffered so that the read-back / merge of a finished window
    // overlaps the rendering of the next one (OpenClPathTracingRenderer.java:150-151,172-177)
    int width = 0, height = 0;
    ccu_host::DevBuf<float> accum[2];       // running mean float[accum_floats] each
    size_t accum_floats = 0;                // 3*W*H rounded up (ccu_group needs equal reduce-scatter shares)
    size_t accum_align = 256;               // accum_floats is a multiple of this (set by the group before ccu_render_begin)
    int accum_active = 0;
    const float *window_base = nullptr;     // the buffer that holds what the reference's single buffer would hold right now
    ccu_host::HostBuf<float> pinned;        // host staging float[accum_floats]
    ccu_host::SeedRing seeds;
    ccu_host::DevBuf<int> fh_scratch;       // first-hit planes (kept between calls)
    ccu_host::DevBuf<float> feat_scratch;   // feature buffers: albedo and normal, float[3*W*H] each (kept between calls)
    ccu_host::DevBuf<int> feat_seeds;       // feature buffers: the pass seeds (CCU_FEATURES_MAX_PASSES)
    ccu_host::DevBuf<float4> dn_scratch;    // denoiser: working records, 4 per pixel (kept between calls)
    ccu_host::DevBuf<double> dn_io;         // denoiser: the colour in and the result out, double[3*W*H], then albedo and normal float[3*W*H]
    ccu_host::DevBuf<unsigned> work_counter;
    ccu_host::DevBuf<int> bvh_deep;         // wavefront kernel, BVH scenes: traversal-stack entries beyond the shared-memory part
    int yield_below = 20;
    int q_refill_min = 8;
    int q_march_bias = 4;
    int q_shade_min = 0;
    int q_sticky_min = 0;      // 0 = default by kernel (CCU_Q_STICKY)
    int q_march_warps = 18;
    int window_spp = 0;
    int closed_spp = 0;          // passes of the window closed by ccu_render_window_close, read-back in flight, not merged yet
    bool target_live = false;    // between ccu_render_begin and ccu_render_end
    ccu_render_params params = {256, 5, 13.0f, 0, 0};
    ccu_host::MergeJob merge;

    float last_ms = 0;
    bool timing_pending = false;
    int64_t launches = 0;
    int32_t last_render[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};   // the last render launch's instance (ccu_debug_last_render_n)
    int32_t last_features[4] = {0, 0, 0, 0};                // the last feature launch's instance (ccu_debug_last_features)
};

namespace ccu_host {
// internal entry points shared with ccu_group.cu (caller holds no lock)
int start_readback(ccu_ctx *c, const float *src_dev, size_t lo, size_t hi, cudaStream_t stream);
int merge_readback(ccu_ctx *c, size_t lo, size_t hi, double *sample_buffer, double ds, double dp, double sinv, unsigned max_threads);
int replicate_scene(ccu_ctx *src, ccu_ctx *dst);
// multiplies the first n floats of the active accumulation window by `factor` on the render stream and counts the launch
// (caller holds c->mu, c->device is current); the launch error is left for cudaGetLastError
void scale_window(ccu_ctx *c, float factor, size_t n);
}  // namespace ccu_host
