// ccu_host.h - host-side state behind the C ABI (include/chunkycu.h): the context object, small RAII helpers and the
// error plumbing shared by chunkycu.cu (single-GPU entry points) and ccu_group.cu (multi-GPU entry points).
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
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

template <class T>
struct DevBuf {
    // never smaller than one 64-byte record: the straight-line kernels read element 0 of an empty array on lanes that have no
    // work (the value is dropped)
    static constexpr size_t MIN_ELEMS = 64 / sizeof(T) > 4 ? 64 / sizeof(T) : 4;
    T *p = nullptr;
    size_t n = 0;
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

constexpr int SEED_SLOTS = 4, SEED_SLOT_INTS = 32768;   // one launch covers at most 32768 passes (16-bit pass index in the wavefront kernel)

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

// one asynchronous read-back + merge of a finished window into the host sample buffer (ccu_render_merge_async)
struct MergeJob {
    std::thread worker;
    bool active = false;
    int status = CCU_OK;
    std::string error;
};

}  // namespace ccu_host

struct ccu_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;        // render stream
    cudaStream_t copy_stream = nullptr;   // read-back of finished windows, camera-ray uploads
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t chunk_ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // read-back chunks of a merge
    cudaEvent_t window_ev = nullptr;      // the window being merged is complete on the render stream
    // Locking: `mu` guards every field below and is never held across a wait for rendering work (ccu_render_sync waits on an
    // event outside the lock), so preview / tonemap / camera calls from other threads are not blocked by a long batch;
    // `cam_mu` serialises camera updates.
    std::mutex mu, cam_mu;
    int sm_count = 0;

    // scene as uploaded (reference packed layouts)
    ccu_host::DevBuf<int> tree, block_palette, quad_models, aabb_models, mat_palette, trigs, world_bvh, actor_bvh, sun_words;
    std::vector<int> tree_host, world_host, actor_host, trigs_host, block_host, mat_host;   // kept for the commit-time layouts
    // commit-time layouts
    ccu_host::DevBuf<unsigned> top, wide;                       // value-carrying octree layout
    ccu_host::DevBuf<unsigned> air_top, air_wide, air_bricks;   // march layout (ccu_march.cuh)
    ccu_host::DevBuf<int> world_rec, actor_rec, tris2;          // BVH stage layout (ccu_queue.cuh)
    ccu_host::DevBuf<int> block_rec, mat_rec, quad_rec, aabb_rec;   // 16-byte-vectorised palettes (DScene::block_rec ...)
    std::vector<int> quad_host, aabb_host;
    int world_root = 0, actor_root = 0, use_bvh2 = 0, use_air = 0, air_deep = 0;
    int cell_level = 0, top_log2 = 0, use_wide = 0, air_cell_level = 4, air_top_log2 = 0;
    double commit_ms = 0;                                       // host time of the last ccu_scene_commit
    ccu_host::DevBuf<uchar4> atlas, sky;
    int atlas_w = 0, atlas_h = 0, atlas_layers = 0;
    int depth = 0, sky_res = 0;
    float sky_intensity = 0;
    int sun_host[6] = {0, 0, 0, 0, 0, 0};
    bool have_sun = false, have_octree = false, have_blocks = false, have_mats = false, have_atlas = false, have_sky = false;
    bool committed = false;
    ccu_host::DevBuf<float> sun_basis;
    float *unorm = nullptr;

    // camera: pre-generated rays are double buffered so that an upload overlaps the passes in flight
    int projector_type = 0;
    float cam[15] = {0};
    ccu_host::DevBuf<float> rays[2];
    cudaEvent_t rays_used[2] = {nullptr, nullptr};   // last launch that read rays[i]
    int rays_active = 0;
    bool have_camera = false;

    // render target: the accumulation window is double buffered so that the read-back / merge of a finished window
    // overlaps the rendering of the next one (OpenClPathTracingRenderer.java:150-151,172-177)
    int width = 0, height = 0;
    float *accum[2] = {nullptr, nullptr};   // running mean float[accum_floats] each
    size_t accum_floats = 0;                // 3*W*H rounded up (ccu_group needs equal reduce-scatter shares)
    size_t accum_align = 256;               // accum_floats is a multiple of this (set by the group before ccu_render_begin)
    int accum_active = 0;
    const float *window_base = nullptr;     // the buffer that holds what the reference's single buffer would hold right now
    float *pinned = nullptr;                // host staging float[accum_floats]
    int *seeds_dev = nullptr, *seeds_pinned = nullptr;   // ring of seed slots (device / pinned host)
    cudaEvent_t seeds_ev[4] = {nullptr, nullptr, nullptr, nullptr};
    int seeds_slot = 0;
    int *fh_scratch = nullptr;              // first-hit planes (kept between calls)
    size_t fh_scratch_pixels = 0;
    unsigned int *work_counter = nullptr;
    int *bvh_deep = nullptr;                // wavefront kernel, BVH scenes: traversal-stack entries beyond the shared-memory part
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

    ccu::DScene scene{};
};

namespace ccu_host {
// internal entry points shared with ccu_group.cu (caller holds no lock)
int start_readback(ccu_ctx *c, const float *src_dev, size_t lo, size_t hi, cudaStream_t stream);
int merge_readback(ccu_ctx *c, size_t lo, size_t hi, double *sample_buffer, double ds, double dp, double sinv, unsigned max_threads);
int merge_window_range(ccu_ctx *c, const float *src_dev, size_t lo, size_t hi, double *sample_buffer, double ds, double dp, double sinv,
                       cudaStream_t stream, unsigned max_threads);
int replicate_scene(ccu_ctx *src, ccu_ctx *dst);
}  // namespace ccu_host
