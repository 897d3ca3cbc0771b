// chunkycu.cu - kernels and the C ABI (include/chunkycu.h) of libchunkycu.so.  sm_100a only.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <climits>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include <chrono>

#include "ccu_host.h"
#include "ccu_march.cuh"
#include "ccu_queue.cuh"
#include "ccu_render.cuh"
#include "ccu_tonemap.cuh"
#include "ccu_layout.h"

using namespace ccu;

// ======================================================================================================
// kernels
// ======================================================================================================

// Sun_new (sky.h:19-40) once per scene, on the device so it uses the device's arithmetic.
__global__ void k_sun_setup(const int *sun_words, float *out /* su sv sw radius_cos : 10 floats */) {
    float phi = i2f(sun_words[4]), theta = i2f(sun_words[5]);
    float r = fabsf(dm_cos(phi));
    float3 sw = f3(dm_cos(theta) * r, dm_sin(phi), dm_sin(theta) * r);
    float3 su = (fabsf(sw.x) > 0.1f) ? f3(0, 1, 0) : f3(1, 0, 0);
    float3 sv = normalize3(cross3(sw, su));
    su = cross3(sv, sw);
    out[0] = su.x; out[1] = su.y; out[2] = su.z;
    out[3] = sv.x; out[4] = sv.y; out[5] = sv.z;
    out[6] = sw.x; out[7] = sw.y; out[8] = sw.z;
    out[9] = dm_cos(0.03f);
}

__device__ __forceinline__ int face_of(float3 n) {
    if (n.x == -1 && n.y == 0 && n.z == 0) return 0;
    if (n.x == 1 && n.y == 0 && n.z == 0) return 1;
    if (n.x == 0 && n.y == -1 && n.z == 0) return 2;
    if (n.x == 0 && n.y == 1 && n.z == 0) return 3;
    if (n.x == 0 && n.y == 0 && n.z == -1) return 4;
    if (n.x == 0 && n.y == 0 && n.z == 1) return 5;
    return 6;
}

// First-hit pass (BASELINE config 2): closestIntersect (kernel.h:14-24) for the camera ray of every pixel.
// Pixels are taken in 32x32 screen tiles, 8x4 patches per warp (tile_order_pixel<true>: the lanes of a warp walk neighbouring
// rays, which keeps their step counts and brick loads together).  With the commit-time layouts (MODE 1 / 2) the warp marches on
// the air layout until every lane sits at a non-air leaf or has left the octree, THEN runs the block tests of all those lanes
// together (the block test is ~3x the instructions of a march step; run per lane as each ray arrives it executed at 6 of 32
// lanes), and repeats for the lanes whose block test missed.  The treeData index of the hit leaf (reference numbering,
// ClSceneLoader.java:56-59) is found by one root descent for the hit voxel only.  HAS_BVH = false compiles the entity BVHs out.
// threads per block of the first-hit kernel and resident blocks per SM (the warps of a block do not depend on each other, so
// the block size only decides how many warps wait for the slowest one before their registers are handed on)
#ifndef CCU_FH_THREADS
#define CCU_FH_THREADS 128
#endif
#ifndef CCU_FH_MIN_BLOCKS
#define CCU_FH_MIN_BLOCKS (1024 / CCU_FH_THREADS)
#endif
struct FirstHitOut { int *block, *face, *node, *kind; float *t, *normal, *color; };
__device__ __forceinline__ void first_hit_store(const FirstHitOut &out, int gid, bool hit, int material, float3 n, int node, int kind, float t, float4 color) {
    if (out.block) out.block[gid] = hit ? material : 0;
    if (out.face) out.face[gid] = hit ? face_of(n) : 6;
    if (out.node) out.node[gid] = hit ? node : -1;
    if (out.kind) out.kind[gid] = hit ? kind : 0;
    if (out.t) out.t[gid] = hit ? t : inff_();
    if (out.normal) {
        out.normal[gid * 3 + 0] = hit ? n.x : 0.0f;
        out.normal[gid * 3 + 1] = hit ? n.y : 0.0f;
        out.normal[gid * 3 + 2] = hit ? n.z : 0.0f;
    }
    if (out.color) reinterpret_cast<float4 *>(out.color)[gid] = hit ? color : make_float4(0, 0, 0, 0);
}

// The warp-synchronous march loop of the thread-per-ray kernels: every lane steps its ray until no lane of the warp is marching
// any more.  Kept out of line so that the loop is register-allocated by itself - inlined into the 64-register kernel, next to the
// block test, the ray was spilled and re-loaded inside the loop.  The ray travels through local memory once per call.
// st: 0 marching, anything else: not marching (returned unchanged).
template <bool DEEP>
static __device__ __noinline__ int first_hit_march(const DScene &s, LeanRay *ray, int st) {
    LeanRay r = *ray;
    while (__any_sync(0xffffffffu, st == 0)) {
        if (!DEEP) st = lean_step_flat<false>(s, s.air_top, r, st == 0, st, s.draw_depth, ~0u << s.depth);
        else if (st == 0) st = lean_probe<DEEP, false>(s, s.air_top, r, s.draw_depth);
    }
    ray->t = r.t;
    ray->steps = r.steps;
    return st;
}

template <int MODE, bool HAS_BVH>
__global__ void __launch_bounds__(CCU_FH_THREADS, CCU_FH_MIN_BLOCKS) k_first_hit(const __grid_constant__ DScene s, int seed, int n_pixels, const __grid_constant__ FirstHitOut out) {
    stage_tables_per_warp(s);
    const unsigned full = 0xffffffffu;
    const unsigned k = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = k < (unsigned)n_pixels;
    unsigned px = 0, py = 0;
    if (valid) tile_order_xy<true>(k, s.width, s.height, px, py);
    const int gid = (int)(py * (unsigned)s.width + px);
    uint32_t rng = (uint32_t)seed + (uint32_t)gid;
    rng_next(rng);
    float3 o, d;
    camera_ray_xy<false>(s, gid, (int)px, (int)py, rng, o, d);
    if (MODE == 0) {
        Record rec;
        rec.distance = inff_(); rec.material = 0; rec.surf.normal = f3(0, 0, 0); rec.point = f3(0, 0, 0);
        rec.surf.color = make_float4(0, 0, 0, 0); rec.surf.emittance = 0;
        HitInfo hi = {-1, 0, 0, 0, 0};
        bool hit = false;
        if (valid) hit = HAS_BVH ? closest_intersect_ref<PlainShade>(s, o, d, rec, hi) : octree_intersect_ref<PlainShade>(s, o, d, rec, hi);
        if (valid) first_hit_store(out, gid, hit, rec.material, rec.surf.normal, hi.node, hi.kind, rec.distance, rec.surf.color);
        return;
    }
    March m;
    const bool entered = march_begin(s, m, o, d, inff_());
    LeanRay r;
    r.o = m.o; r.d = m.d; r.inv = m.inv; r.t = m.t; r.limit = m.limit; r.steps = m.steps;
    lean_prepare(r);
    int st = (valid && entered) ? 0 : 2;      // 0 marching, 1 at a non-air leaf, 2 left the octree without a hit, 3 hit
    // what an octree hit leaves behind; without BVHs it is written out at once, so that nothing of it stays in registers while
    // the other lanes of the warp keep marching
    Surf surf;
    surf.normal = f3(0, 0, 0); surf.color = make_float4(0, 0, 0, 0); surf.emittance = 0;
    float distance = inff_();
    int material = 0, hbx = 0, hby = 0, hbz = 0;
    for (;;) {
        st = first_hit_march<MODE == 2>(s, &r, st);
        if (st == 1) {
            m.t = r.t; m.steps = r.steps;
            const Cell c = march_cell(m);
            int level;
            const int data = find_leaf_wide(s, c.bx, c.by, c.bz, level);
            float th;
            Surf hs;
            if (march_block<PlainShade>(s, m, data, level, hs, th)) {
                st = 3;
                if (!HAS_BVH) {
                    int hnode = -1;
                    if (out.node) { int lv; find_leaf(s, c.bx, c.by, c.bz, lv, hnode); }
                    first_hit_store(out, gid, true, data, hs.normal, hnode, 1, th, hs.color);
                } else {
                    surf = hs; distance = th; material = data;
                    hbx = c.bx; hby = c.by; hbz = c.bz;
                }
            } else {
                r.t = m.t; r.steps = m.steps;
                st = 0;
            }
        }
        if (!__any_sync(full, st == 0)) break;
    }
    if (!valid) return;
    if (!HAS_BVH) {
        if (st != 3) first_hit_store(out, gid, false, 0, f3(0, 0, 0), -1, 0, inff_(), make_float4(0, 0, 0, 0));
        return;
    }
    bool hit = st == 3;
    int kind = hit ? 1 : 0, bk = 0;
    if (bvh_pair(s, o, d, distance, surf, bk)) { hit = true; kind = bk; }
    int hnode = -1;
    if (out.node && hit && kind == 1) { int lv; find_leaf(s, hbx, hby, hbz, lv, hnode); }
    first_hit_store(out, gid, hit, material, surf.normal, hnode, kind, distance, surf.color);
}

// rayTracer.cl:141-216
template <int MODE>
__global__ void __launch_bounds__(256) k_preview(const __grid_constant__ DScene s, int n_pixels, int *res) {
    stage_tables(s, nullptr);
    const unsigned k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= (unsigned)n_pixels) return;
    const int gid = tile_order_pixel<true>(k, s.width, s.height);
    int W = s.width, H = s.height;
    int px = gid % W, py = gid / W;
    if ((px == W / 2 && (py >= H / 2 - 5 && py <= H / 2 + 5)) || (py == H / 2 && (px >= W / 2 - 5 && px <= W / 2 + 5))) {
        res[gid] = (int)0xFFFFFFFFu;
        return;
    }
    uint32_t rng = 0;
    rng_next(rng);
    float3 o, d;
    camera_ray<true>(s, gid, rng, o, d);
    Record rec;
    rec.distance = inff_(); rec.material = 0; rec.surf.normal = f3(0, 0, 0); rec.point = f3(0, 0, 0);
    rec.surf.color = make_float4(0, 0, 0, 0); rec.surf.emittance = 0;
    HitInfo hi = {-1, 0, 0, 0, 0};
    float3 c;
    if (closest_intersect_mode<MODE, PlainShade>(s, o, d, rec, hi)) {
        float shading = dot3(rec.surf.normal, f3(0.25f, 0.866f, 0.433f));
        shading = fmaxf(0.3f, shading);
        c = f3(rec.surf.color.x * shading, rec.surf.color.y * shading, rec.surf.color.z * shading);
    } else {
        c = sky_radiance(s, d);
    }
    float v[3] = {c.x, c.y, c.z};
    int rgb[3];
    for (int i = 0; i < 3; i++) {
        float q = sqrtf(v[i]) * 255.0f;
        q = fminf(fmaxf(q, 0.0f), 255.0f);
        rgb[i] = f2i(floorf(q));
    }
    res[gid] = (int)(0xFF000000u | ((uint32_t)rgb[0] << 16) | ((uint32_t)rgb[1] << 8) | (uint32_t)rgb[2]);
}

// post_processing_filter.cl:5-51: one work-item per pixel
__global__ void __launch_bounds__(256) k_tonemap(int n_pixels, float exposure, const double *__restrict__ input, int type, uint32_t *__restrict__ res) {
    for (int gid = blockIdx.x * blockDim.x + threadIdx.x; gid < n_pixels; gid += gridDim.x * blockDim.x)
        res[gid] = tonemap_pixel(input + (size_t)gid * 3, exposure, type);
}

__global__ void k_unorm_table(float *t) { t[threadIdx.x] = (float)threadIdx.x / 255.0f; }

__global__ void k_scale(float *buf, float factor, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) buf[i] *= factor;
}

// Re-tile a row-major RGBA8 rectangle into the tile-linear atlas (16x16 texel tiles contiguous = 1 KiB each).
__global__ void k_atlas_write(uchar4 *atlas, int tiles_x, int tiles_y, int x0, int y0, int layer, int w, int h, const uchar4 *src) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= w * h) return;
    int x = x0 + i % w, y = y0 + i / w;
    size_t tile = ((size_t)layer * tiles_y + (y >> 4)) * tiles_x + (x >> 4);
    atlas[tile * 256 + ((y & 15) << 4) + (x & 15)] = src[i];
}

// Roofline denominators this path needs (SURVEY 8d): random 32-byte-sector gathers.  Every thread issues `loads`
// independent 16-byte L2 loads (ld.global.cg) at hashed sector addresses of an array of `sectors` sectors
// (dependent = 0), or walks a dependent chain (dependent = 1: the next address comes from the loaded word).
__global__ void k_gather_fill(uint4 *a, size_t sectors, uint32_t seed) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < sectors * 2; i += (size_t)gridDim.x * blockDim.x) {
        uint32_t h = (uint32_t)i * 2654435761u + seed;
        h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
        a[i] = make_uint4(h, h * 3u + 1u, h ^ 0x9e3779b9u, (uint32_t)i);
    }
}
__global__ void __launch_bounds__(256) k_gather(const uint4 *__restrict__ a, uint32_t sector_mask, int loads, int dependent, uint32_t salt, uint32_t *sink) {
    // salt: every timed launch walks different sectors, so that a repeat does not find its own footprint in L2
    uint32_t st = (blockIdx.x * blockDim.x + threadIdx.x + salt * 0x9e3779b9u) * 747796405u + 2891336453u;
    uint32_t acc = 0;
    if (dependent) {
        // one thread per SM walks the chain: the time per load is the latency of one dependent gather
        if (threadIdx.x != 0) return;
        uint32_t at = st & sector_mask;
        for (int i = 0; i < loads; i++) {
            uint4 v = __ldcg(a + (size_t)at * 2);
            acc ^= v.y;
            at = (v.x ^ (uint32_t)i * 0x9e3779b9u) & sector_mask;
        }
    } else {
#pragma unroll 8
        for (int i = 0; i < loads; i++) {
            st = st * 747796405u + 2891336453u;
            uint32_t at = ((st >> 9) ^ st) & sector_mask;
            uint4 v = __ldcg(a + (size_t)at * 2);
            acc ^= v.x ^ v.w;
        }
    }
    if (acc == 0x12345678u) *sink = acc;
}

// ======================================================================================================
// host side
// ======================================================================================================
namespace ccu_host {
static thread_local std::string g_err;

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
const char *last_error() { return g_err.c_str(); }
}  // namespace ccu_host

using ccu_host::DevBuf;
using ccu_host::DeviceGuard;
using ccu_host::Event;
using ccu_host::fail;
using ccu_host::SEED_SLOTS;
using ccu_host::SEED_SLOT_INTS;

namespace {

int air_layout_id(const ccu_ctx *c) {   // template parameter LAY of k_render_queue
    if (c->scene.info.air_deep) return 2;
    return (c->scene.air_top.n <= (size_t)Q_TOP_WORDS && getenv("CCU_NO_TOPS") == nullptr) ? 0 : 1;
}

// The fields of the launch view that depend on the committed scene alone: its buffers, layouts, atlas, sky and sun.
void fill_view(ccu_host::Scene &sc) {
    DScene &s = sc.view;
    const ccu_host::SceneInfo &in = sc.info;
    const auto arr = [&](ccu_host::SceneArray a) { return (const int *)sc.arrays[a].dev.p; };
    const auto rec = [](const DevBuf<int> &b) { return reinterpret_cast<const int4 *>(b.p); };
    s.tree = arr(ccu_host::OCTREE); s.depth = in.depth;
    s.top = sc.top.p; s.wide = sc.wide.p; s.cell_level = in.cell_level; s.top_log2 = in.top_log2; s.use_wide = in.use_wide;
    s.air_top = sc.air_top.p; s.air_wide = sc.air_wide.p; s.air_bricks = sc.air_bricks.p;
    s.air_cell_level = in.air_cell_level; s.air_top_log2 = in.air_top_log2;
    s.world_rec = rec(sc.world_rec); s.actor_rec = rec(sc.actor_rec); s.tris2 = sc.tris2.p;
    s.world_root = in.world_root; s.actor_root = in.actor_root;
    s.block_palette = arr(ccu_host::BLOCK_PALETTE); s.block_palette_len = (int)sc.arrays[ccu_host::BLOCK_PALETTE].dev.n;
    s.quad_models = arr(ccu_host::QUAD_MODELS); s.aabb_models = arr(ccu_host::AABB_MODELS); s.mat_palette = arr(ccu_host::MAT_PALETTE);
    s.block_rec = rec(sc.block_rec); s.mat_rec = rec(sc.mat_rec); s.quad_rec = rec(sc.quad_rec); s.aabb_rec = rec(sc.aabb_rec);
    s.world_bvh = arr(ccu_host::WORLD_BVH); s.actor_bvh = arr(ccu_host::ACTOR_BVH); s.trigs = arr(ccu_host::TRIANGLES);
    s.world_bvh_empty = in.world_bvh_empty; s.actor_bvh_empty = in.actor_bvh_empty;
    s.atlas = sc.atlas.p;
    s.atlas_w = in.atlas_w; s.atlas_h = in.atlas_h; s.atlas_layers = in.atlas_layers;
    s.atlas_tiles_x = (in.atlas_w + 15) / 16; s.atlas_tiles_y = (in.atlas_h + 15) / 16;
    s.sky = sc.sky.p; s.sky_res = in.sky_res; s.sky_intensity = in.sky_intensity;
    s.su = in.su; s.sv = in.sv; s.sw = in.sw; s.sun_radius_cos = in.sun_radius_cos;
    s.sun_flags = in.sun_host[0]; s.sun_tex_size = in.sun_host[1]; s.sun_tex = in.sun_host[2];
    memcpy(&s.sun_intensity, &in.sun_host[3], 4);
    s.fog_sigma = in.fog_sigma; s.fog_sky = in.fog_sky; s.fog_fast = in.fog_fast;
    s.fog_color = make_float3(in.fog_color[0], in.fog_color[1], in.fog_color[2]);
    EmitView &g = sc.emit_view;
    g.emit = reinterpret_cast<const int4 *>(sc.emit.p); g.off = sc.emit_off.p; g.list = sc.emit_list.p;
    g.g0 = make_int3(in.emit_g0[0], in.emit_g0[1], in.emit_g0[2]);
    g.dim = make_int3(in.emit_dim[0], in.emit_dim[1], in.emit_dim[2]);
    g.shift = in.emit_shift;
    EmitView &mg = sc.memit_view;
    mg.emit = reinterpret_cast<const int4 *>(sc.memit.p); mg.off = sc.memit_off.p; mg.list = sc.memit_list.p;
    mg.g0 = make_int3(in.memit_g0[0], in.memit_g0[1], in.memit_g0[2]);
    mg.dim = make_int3(in.memit_dim[0], in.memit_dim[1], in.memit_dim[2]);
    mg.shift = in.memit_shift;
    mg.mhead = sc.memit_head.p; mg.mprim = reinterpret_cast<const int4 *>(sc.memit_prim.p);
    BiomeView &bv = sc.biome_view;
    bv.grid = sc.biome_grid.p; bv.tiles = sc.biome_tiles.p;
    bv.x0 = in.biome_box[0]; bv.z0 = in.biome_box[1]; bv.gx = in.biome_box[2]; bv.gz = in.biome_box[3];
    CloudView &cv = sc.cloud_view;
    cv.mask = sc.cloud_mask.p;
    cv.inv = in.cloud_inv; cv.y0 = in.cloud_y0; cv.y1 = in.cloud_y1; cv.u0 = in.cloud_u0; cv.v0 = in.cloud_v0;
}

// build_biome_layout with its failures as CCU_* codes; `what` names the entry point
int biome_layout(const int32_t *chunks, const float *rgb, int64_t n, int depth, BiomeLayout &bl, const char *what) {
    try {
        bl = build_biome_layout(chunks, rgb, n, depth);
    } catch (const std::bad_alloc &) {
        return fail(CCU_ENOMEM, "%s: no host memory for the biome layout of %lld chunks", what, (long long)n);
    }
    if (bl.status == 1)
        return fail(CCU_EINVAL, "%s: biome chunk %lld (%d, %d) lies outside the octree's %lld x %lld chunks", what, (long long)bl.bad,
                    chunks[2 * bl.bad], chunks[2 * bl.bad + 1], (long long)bl.extent, (long long)bl.extent);
    if (bl.status == 2)
        return fail(CCU_EINVAL, "%s: the biome chunks span more than %lld chunks (bounding box); the grid holds at most that many", what,
                    (long long)CCU_BIOME_GRID_MAX);
    return CCU_OK;
}

// The checks of ccu_scene_set_biome_colors (also applied by ccu_debug_biome_layout); `what` names the entry point.
int check_biome_colors(const int32_t *chunks, const float *rgb, int64_t n, const char *what) {
    if (n < 0 || (n > 0 && (!chunks || !rgb))) return fail(CCU_EINVAL, "%s: bad arrays (n=%lld)", what, (long long)n);
    std::vector<std::pair<int, int>> seen;
    seen.reserve((size_t)n);
    for (int64_t i = 0; i < n; i++) {
        if (chunks[2 * i] < 0 || chunks[2 * i + 1] < 0)
            return fail(CCU_EINVAL, "%s: chunk %lld (%d, %d) has a negative coordinate", what, (long long)i, chunks[2 * i], chunks[2 * i + 1]);
        seen.emplace_back(chunks[2 * i], chunks[2 * i + 1]);
    }
    std::sort(seen.begin(), seen.end());
    for (size_t i = 1; i < seen.size(); i++)
        if (seen[i] == seen[i - 1]) return fail(CCU_EINVAL, "%s: chunk (%d, %d) is given twice", what, seen[i].first, seen[i].second);
    for (int64_t i = 0; i < n * 3 * 256 * 3; i++)
        if (!std::isfinite(rgb[i]) || rgb[i] < 0.0f)
            return fail(CCU_EINVAL, "%s: colour component %lld of chunk %lld is negative or not finite", what, (long long)i,
                        (long long)(i / (3 * 256 * 3)));
    return CCU_OK;
}

// The launch view with this launch's camera, rays, canvas and render params (caller holds c->mu, the scene is committed).
DScene launch_view(const ccu_ctx *c) {
    DScene s = c->scene.view;
    if (c->params.flags & CCU_RENDER_NO_ENTITIES) s.world_bvh_empty = s.actor_bvh_empty = 1;
    if (c->params.flags & CCU_RENDER_NO_SUN) s.sun_flags &= ~1;
    s.unorm = c->unorm.p;
    s.projector_type = c->projector_type;
    memcpy(s.cam, c->cam, sizeof s.cam);
    s.rays = c->rays[c->rays_active].p;
    s.width = c->width; s.height = c->height;
    s.half_width = (float)(c->width / (2.0 * c->height));   // rayTracer.cl:66
    s.inv_height = (float)(1.0 / c->height);                // rayTracer.cl:67
    s.draw_depth = c->params.draw_depth; s.max_depth = c->params.max_depth; s.emitter_scale = c->params.emitter_scale;
    return s;
}

// Upload one of the reference's packed int arrays and keep its host copy for commit; `depth` is recorded for the octree.
int set_array(ccu_ctx *c, ccu_host::SceneArray a, const int32_t *words, int64_t n, int32_t depth = 0) {
    const char *what = ccu_host::ARRAY_DESC[a].setter;
    if (!c) return fail(CCU_EINVAL, "%s: null context", what);
    if (n < 0 || (n > 0 && !words)) return fail(CCU_EINVAL, "%s: bad array (n=%lld)", what, (long long)n);
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    c->committed = false;
    ccu_host::PackedArray &arr = c->scene.arrays[a];
    arr.host.reset();
    CU(arr.dev.upload(words, (size_t)n, c->stream));
    arr.host = std::make_shared<const std::vector<int>>(words, words + n);
    if (a == ccu_host::OCTREE) c->scene.info.depth = depth;
    return CCU_OK;
}

// device time of the last render / first-hit / preview / tonemap launch(es); waits for them (caller holds c->mu)
void stop_timer(ccu_ctx *c) {
    if (c->timing_pending) {
        cudaEventSynchronize(c->ev1);
        cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
        c->timing_pending = false;
    }
}

// waits for everything queued on the render stream WITHOUT holding the context lock
int wait_render_stream(ccu_ctx *c) {
    Event ev;
    {
        std::lock_guard<std::mutex> lk(c->mu);
        DeviceGuard g(c->device);
        CU(ev.create(cudaEventDisableTiming));
        cudaError_t e = cudaEventRecord(ev, c->stream);
        if (e != cudaSuccess) return fail(CCU_ECUDA, "cudaEventRecord: %s", cudaGetErrorString(e));
    }
    cudaError_t e = cudaEventSynchronize(ev);
    if (e != cudaSuccess) return fail(CCU_ECUDA, "render stream: %s", cudaGetErrorString(e));
    return CCU_OK;
}

void free_target(ccu_ctx *c) {
    c->accum[0].release();
    c->accum[1].release();
    c->pinned.reset();
    c->accum_floats = 0;
}

// The Shade of a render launch (DESIGN §5).  Each flag picks its kernels only on a scene where they compute something the
// others do not:
// - CCU_RENDER_SPECULAR: the specular kernels, on a scene with a specular word;
// - CCU_RENDER_EMITTER_SAMPLING: the NEE kernels, on a scene with emitters; CCU_RENDER_EMITTER_NEAR_FIELD picks the near-field
//   sampler (NEE_NEAR) among them.  CCU_RENDER_EMITTER_MODELS picks the samplers of the wider table (NEE_*_MODELS, EmitView
//   memit_view) when the scene has one; without a model emitter it changes nothing;
// - CCU_RENDER_BIOME_TINT: the biome kernels, on a scene with biome colours;
// - CCU_RENDER_FOG: the fog kernels, on a scene with fog (SceneInfo::has_fog);
// - CCU_RENDER_CLOUDS: the cloud kernels, on a scene with a cloud mask that has a set cell (SceneInfo::has_clouds).
ShadeKey shade_variant(const ccu_ctx *c) {
    const int f = c->params.flags;
    const auto &info = c->scene.info;
    const bool near_field = (f & CCU_RENDER_EMITTER_NEAR_FIELD) != 0;
    int nee = NEE_NONE;
    if (f & CCU_RENDER_EMITTER_SAMPLING) {
        if ((f & CCU_RENDER_EMITTER_MODELS) && info.has_model_emitters) nee = near_field ? NEE_NEAR_MODELS : NEE_AREA_MODELS;
        else if (info.has_emitters) nee = near_field ? NEE_NEAR : NEE_AREA;
    }
    return {(f & CCU_RENDER_SPECULAR) && info.has_specular, nee, (f & CCU_RENDER_BIOME_TINT) && info.has_biome,
            (f & CCU_RENDER_FOG) && info.has_fog, (f & CCU_RENDER_CLOUDS) && info.has_clouds};
}

// the wavefront kernel (ccu_queue.cuh) for the scene's entity BVHs, air layout (queue_layout) and the launch's Shade
QueueFn queue_kernel(bool bvh, int lay, const ShadeKey &v) {
    QueueFn k = nullptr;
    dispatch(bvh, [&](auto B) {
        dispatch<3>(lay, [&](auto L) { k = v.clouds ? queue_kernel_of<B, L, true>(v) : queue_kernel_of<B, L, false>(v); });
    });
    return k;
}

// LAY of a wavefront launch (DESIGN §5): air_layout_id, except that a fog launch whose slot fields do not fit beside the staged
// top table (entity BVHs with the specular or emitter-sampling fields) reads the same table from global memory (LAY 1).
int queue_layout(const ccu_ctx *c, bool bvh, const ShadeKey &v) {
    const int lay = air_layout_id(c);
    if (lay == 0 && v.fog && q_smem_bytes(bvh, true, v.spec, v.nee != NEE_NONE, true) > Q_SMEM_LIMIT) return 1;
    return lay;
}

}  // namespace

namespace ccu_host {

// Read-back of a finished window, in two phases so that the copy overlaps whatever the host does in between:
// start_readback queues the copy of floats [lo, hi) of `src_dev` (indexed by absolute float offset) into the pinned staging
// buffer in chunks on `st`, one event per chunk; merge_readback waits chunk by chunk and folds each into the host sample buffer
// (OpenClPathTracingRenderer.java:164-173):  sample[i] = (sample[i] * ds + mean[i] * dp) * sinv
static size_t merge_chunk_len(size_t n) { return ((n + MERGE_CHUNKS - 1) / MERGE_CHUNKS + 63) & ~(size_t)63; }

int start_readback(ccu_ctx *c, const float *src_dev, size_t lo, size_t hi, cudaStream_t st) {
    const size_t n = hi > lo ? hi - lo : 0;
    const size_t chunk = merge_chunk_len(n);
    for (int k = 0; k < MERGE_CHUNKS; k++) {
        const size_t a = lo + std::min(n, k * chunk), b = lo + std::min(n, (k + 1) * chunk);
        if (b > a) CU(cudaMemcpyAsync(c->pinned + a, src_dev + a, (b - a) * sizeof(float), cudaMemcpyDeviceToHost, st));
        CU(cudaEventRecord(c->chunk_ev[k], st));
    }
    return CCU_OK;
}

int merge_readback(ccu_ctx *c, size_t lo, size_t hi, double *sample_buffer, double ds, double dp, double sinv, unsigned max_threads) {
    if (hi <= lo) return CCU_OK;
    const size_t n = hi - lo;
    const size_t chunk = merge_chunk_len(n);
    unsigned hw = std::thread::hardware_concurrency();
    unsigned nt = std::max(1u, std::min(std::min(16u, max_threads), hw ? hw : 4u));
    if (n < (1u << 20)) nt = 1;
    const float *src = c->pinned;
    const Event *evs = c->chunk_ev;
    const int device = c->device;
    std::vector<cudaError_t> errs(nt, cudaSuccess);
    auto work = [&, device](unsigned t) {
        cudaSetDevice(device);
        for (int k = 0; k < MERGE_CHUNKS; k++) {
            const size_t a = lo + std::min(n, k * chunk), b = lo + std::min(n, (k + 1) * chunk);
            const cudaError_t e = cudaEventSynchronize(evs[k]);
            if (e != cudaSuccess) { errs[t] = e; return; }
            const size_t len = b - a, part = (len + nt - 1) / nt;
            const size_t i0 = a + std::min(len, t * part), i1 = a + std::min(len, (t + 1) * part);
            for (size_t i = i0; i < i1; i++) sample_buffer[i] = (sample_buffer[i] * ds + (double)src[i] * dp) * sinv;
        }
    };
    if (nt == 1) {
        work(0);
    } else {
        std::vector<std::thread> th;
        for (unsigned t = 0; t < nt; t++) th.emplace_back(work, t);
        for (auto &t : th) t.join();
    }
    for (cudaError_t e : errs)
        if (e != cudaSuccess) return fail(CCU_ECUDA, "window read-back: %s", cudaGetErrorString(e));
    return CCU_OK;
}

template <class T>
static int copy_buf(const ccu_ctx *src, ccu_ctx *dst, const DevBuf<T> &a, DevBuf<T> &b) {
    if (!a.p) { b.release(); return CCU_OK; }
    CU(b.alloc(a.n));
    CU(cudaMemcpyPeerAsync(b.p, dst->device, a.p, src->device, a.bytes(), dst->stream));
    return CCU_OK;
}

// Copy the committed scene of `src` to `dst`: device arrays device-to-device, the host copies shared.  A failure leaves `dst`
// uncommitted and with nothing to commit until a scene is loaded again.
int replicate_scene(ccu_ctx *src, ccu_ctx *dst) {
    if (src == dst) return CCU_OK;
    std::lock(src->mu, dst->mu);
    std::lock_guard<std::mutex> l1(src->mu, std::adopt_lock), l2(dst->mu, std::adopt_lock);
    if (!src->committed) return fail(CCU_ESTATE, "replicate: source scene not committed");
    DeviceGuard g(dst->device);
    cudaStreamSynchronize(dst->stream);
    Scene &a = src->scene, &b = dst->scene;
    dst->committed = false;
    b.info = SceneInfo();
    for (PackedArray &p : b.arrays) p.host.reset();
    b.biome.reset();
    b.clouds.reset();
    int rc = CCU_OK;
    Scene::each_buf(a, b, [&](auto &x, auto &y) { if (rc == CCU_OK) rc = copy_buf(src, dst, x, y); });
    if (rc != CCU_OK) return rc;
    CU(cudaStreamSynchronize(dst->stream));
    for (int i = 0; i < N_ARRAYS; i++) b.arrays[i].host = a.arrays[i].host;
    b.biome = a.biome;
    b.clouds = a.clouds;
    b.info = a.info;
    fill_view(b);
    dst->committed = true;
    return CCU_OK;
}

void scale_window(ccu_ctx *c, float factor, size_t n) {
    k_scale<<<c->sm_count * 4, 256, 0, c->stream>>>(c->accum[c->accum_active].p, factor, n);
    c->launches++;
}

}  // namespace ccu_host

extern "C" {

const char *ccu_last_error(void) { return ccu_host::last_error(); }
const char *ccu_version(void) { return "chunkycu 0.2 (sm_100a)"; }

int ccu_device_count(int *count) {
    if (!count) return fail(CCU_EINVAL, "ccu_device_count: null");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        *count = 0;
        return fail(CCU_ENODEVICE, "no CUDA device: %s", cudaGetErrorString(e));
    }
    *count = n;
    return CCU_OK;
}

int ccu_device_info(int index, char *name, int name_len, int *sm_count, int *clock_khz, uint64_t *mem_bytes) {
    int n = 0;
    int rc = ccu_device_count(&n);
    if (rc != CCU_OK) return rc;
    if (index < 0 || index >= n) return fail(CCU_EINVAL, "device index %d out of range [0,%d)", index, n);
    cudaDeviceProp p;
    CU(cudaGetDeviceProperties(&p, index));
    if (name && name_len > 0) snprintf(name, (size_t)name_len, "%s", p.name);
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (clock_khz) {
        int khz = 0;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, index);
        *clock_khz = khz;
    }
    if (mem_bytes) *mem_bytes = (uint64_t)p.totalGlobalMem;
    return CCU_OK;
}

int ccu_ctx_create(int device_index, ccu_ctx **out) {
    if (!out) return fail(CCU_EINVAL, "ccu_ctx_create: null out");
    *out = nullptr;
    int n = 0;
    int rc = ccu_device_count(&n);
    if (rc != CCU_OK) return rc;
    if (n == 0) return fail(CCU_ENODEVICE, "no CUDA device");
    if (device_index < 0 || device_index >= n) return fail(CCU_EINVAL, "device index %d out of range [0,%d)", device_index, n);
    cudaDeviceProp p;
    CU(cudaGetDeviceProperties(&p, device_index));
    if (p.major != 10) return fail(CCU_ENODEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device_index, p.major, p.minor);
    ccu_ctx *c = new ccu_ctx();
    c->device = device_index;
    c->sm_count = p.multiProcessorCount;
    if (const char *e = getenv("CCU_Q_MARCH_WARPS")) c->q_march_warps = std::max(1, std::min(64, atoi(e)));
    if (const char *e = getenv("CCU_Q_MARCH_BIAS")) c->q_march_bias = std::max(-32, std::min(32, atoi(e)));
    if (const char *e = getenv("CCU_Q_REFILL_MIN")) c->q_refill_min = std::max(1, std::min(32, atoi(e)));
    if (const char *e = getenv("CCU_Q_STICKY")) c->q_sticky_min = std::max(1, std::min(33, atoi(e)));
    if (const char *e = getenv("CCU_Q_SHADE_MIN")) c->q_shade_min = std::max(0, std::min(32, atoi(e)));
    if (const char *e = getenv("CCU_YIELD_BELOW")) c->yield_below = std::max(0, std::min(33, atoi(e)));
    DeviceGuard g(device_index);
    cudaError_t e = c->stream.create();
    if (e == cudaSuccess) e = c->copy_stream.create();
    if (e == cudaSuccess) e = c->ev0.create(cudaEventDefault);
    if (e == cudaSuccess) e = c->ev1.create(cudaEventDefault);
    if (e == cudaSuccess) e = c->window_ev.create(cudaEventDisableTiming);
    for (Event &ev : c->chunk_ev) if (e == cudaSuccess) e = ev.create(cudaEventDisableTiming);
    for (Event &ev : c->rays_used) if (e == cudaSuccess) e = ev.create(cudaEventDisableTiming);
    for (bool bvh : {false, true})
        for (int lay = 0; lay < 3; lay++)
            for (int i = 0; i < N_SHADES && e == cudaSuccess; i++)
                e = cudaFuncSetAttribute(queue_kernel(bvh, lay, nth_shade(i)), cudaFuncAttributeMaxDynamicSharedMemorySize, Q_SMEM_LIMIT);
    if (e == cudaSuccess) e = c->unorm.alloc(256);
    if (e == cudaSuccess) {
        k_unorm_table<<<1, 256, 0, c->stream>>>(c->unorm.p);
        c->launches++;
        e = cudaStreamSynchronize(c->stream);
    }
    if (e != cudaSuccess) {
        delete c;   // the holders release whatever was created
        return fail(CCU_ECUDA, "context setup: %s", cudaGetErrorString(e));
    }
    *out = c;
    return CCU_OK;
}

int ccu_ctx_destroy(ccu_ctx *c) {
    if (!c) return CCU_OK;
    DeviceGuard g(c->device);
    {
        std::unique_lock<std::mutex> lk(c->mu);
        c->merge.join(lk);   // the worker reads `pinned` and `chunk_ev`
        cudaStreamSynchronize(c->stream);
        cudaStreamSynchronize(c->copy_stream);
    }
    delete c;   // releases in the order ccu_ctx declares
    return CCU_OK;
}

// A new scene starts from nothing, as the reference's loader does (fresh palettes and EMPTY_NODE BVHs on every load,
// AbstractSceneLoader.java:70-140): arrays of the previous scene do not leak into a scene that does not set them.
int ccu_scene_begin(ccu_ctx *c) {
    if (!c) return fail(CCU_EINVAL, "ccu_scene_begin: null context");
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    cudaStreamSynchronize(c->stream);
    c->committed = false;
    for (int i = 0; i < ccu_host::N_ARRAYS; i++) {
        c->scene.arrays[i].host.reset();
        if (ccu_host::ARRAY_DESC[i].optional) c->scene.arrays[i].dev.release();
    }
    c->scene.info.have_atlas = c->scene.info.have_sky = c->scene.info.have_sun = false;
    c->scene.biome.reset();
    c->scene.biome_grid.release();
    c->scene.biome_tiles.release();
    c->scene.info.set_fog(0.0f, 0.0f, nullptr, 0);
    c->scene.clouds.reset();
    c->scene.cloud_mask.release();
    return CCU_OK;
}

int ccu_scene_set_octree(ccu_ctx *c, const int32_t *tree, int64_t n, int32_t depth) {
    if (depth < 0 || depth > 30) return fail(CCU_EINVAL, "octree depth %d out of range", depth);
    if (n < 1) return fail(CCU_EINVAL, "octree needs at least the root word");
    return set_array(c, ccu_host::OCTREE, tree, n, depth);
}
int ccu_scene_set_block_palette(ccu_ctx *c, const int32_t *w, int64_t n) { return set_array(c, ccu_host::BLOCK_PALETTE, w, n); }
int ccu_scene_set_quad_models(ccu_ctx *c, const int32_t *w, int64_t n) { return set_array(c, ccu_host::QUAD_MODELS, w, n); }
int ccu_scene_set_aabb_models(ccu_ctx *c, const int32_t *w, int64_t n) { return set_array(c, ccu_host::AABB_MODELS, w, n); }
int ccu_scene_set_material_palette(ccu_ctx *c, const int32_t *w, int64_t n) { return set_array(c, ccu_host::MAT_PALETTE, w, n); }
int ccu_scene_set_triangles(ccu_ctx *c, const int32_t *w, int64_t n) { return set_array(c, ccu_host::TRIANGLES, w, n); }
int ccu_scene_set_world_bvh(ccu_ctx *c, const int32_t *w, int64_t n) { return set_array(c, ccu_host::WORLD_BVH, w, n); }
int ccu_scene_set_actor_bvh(ccu_ctx *c, const int32_t *w, int64_t n) { return set_array(c, ccu_host::ACTOR_BVH, w, n); }

// Kept on the host until commit, which lays the colours out for the octree's extent.
int ccu_scene_set_biome_colors(ccu_ctx *c, const int32_t *chunks, const float *rgb, int64_t n) {
    if (!c) return fail(CCU_EINVAL, "ccu_scene_set_biome_colors: null context");
    std::shared_ptr<ccu_host::BiomeColors> b;
    try {
        const int rc = check_biome_colors(chunks, rgb, n, "ccu_scene_set_biome_colors");
        if (rc != CCU_OK) return rc;
        if (n > 0) {
            b = std::make_shared<ccu_host::BiomeColors>();
            b->chunks.assign(chunks, chunks + 2 * n);
            b->rgb.assign(rgb, rgb + n * 3 * 256 * 3);
        }
    } catch (const std::bad_alloc &) {
        return fail(CCU_ENOMEM, "ccu_scene_set_biome_colors: no host memory for %lld chunks", (long long)n);
    }
    std::lock_guard<std::mutex> lk(c->mu);
    c->committed = false;
    c->scene.biome = std::move(b);
    return CCU_OK;
}

int ccu_scene_atlas_create(ccu_ctx *c, int32_t width, int32_t height, int32_t layers) {
    if (!c) return fail(CCU_EINVAL, "ccu_scene_atlas_create: null context");
    if (width <= 0 || height <= 0 || layers <= 0 || width > 16384 || height > 16384) return fail(CCU_EINVAL, "bad atlas extents %dx%dx%d", width, height, layers);
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    c->committed = false;
    c->scene.info.have_atlas = false;
    const size_t tiles = (size_t)((width + 15) / 16) * ((height + 15) / 16) * layers;
    CU(c->scene.atlas.alloc(tiles * 256));
    CU(cudaMemsetAsync(c->scene.atlas.p, 0, c->scene.atlas.n * sizeof(uchar4), c->stream));
    c->scene.info.atlas_w = width; c->scene.info.atlas_h = height; c->scene.info.atlas_layers = layers;
    c->scene.info.have_atlas = true;
    return CCU_OK;
}

int ccu_scene_atlas_write(ccu_ctx *c, int32_t x, int32_t y, int32_t layer, int32_t w, int32_t h, const uint8_t *rgba) {
    if (!c) return fail(CCU_EINVAL, "ccu_scene_atlas_write: null context");
    std::lock_guard<std::mutex> lk(c->mu);
    const ccu_host::SceneInfo &in = c->scene.info;
    if (!c->scene.atlas.p || !in.have_atlas) return fail(CCU_ESTATE, "atlas not created");
    if (!rgba || w <= 0 || h <= 0 || x < 0 || y < 0 || layer < 0 || x + w > in.atlas_w || y + h > in.atlas_h || layer >= in.atlas_layers)
        return fail(CCU_EINVAL, "atlas write %dx%d at (%d,%d,%d) outside %dx%dx%d", w, h, x, y, layer, in.atlas_w, in.atlas_h, in.atlas_layers);
    DeviceGuard g(c->device);
    c->committed = false;
    DevBuf<uchar4> tmp;
    const int n = w * h;
    CU(tmp.alloc(n));
    cudaError_t e = cudaMemcpyAsync(tmp.p, rgba, (size_t)n * 4, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
        k_atlas_write<<<(n + 255) / 256, 256, 0, c->stream>>>(c->scene.atlas.p, (in.atlas_w + 15) / 16, (in.atlas_h + 15) / 16, x, y, layer, w, h, tmp.p);
        c->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return fail(CCU_ECUDA, "atlas write: %s", cudaGetErrorString(e));
    return CCU_OK;
}

int ccu_scene_set_atlas(ccu_ctx *c, const uint8_t *rgba, int32_t width, int32_t height, int32_t layers) {
    int rc = ccu_scene_atlas_create(c, width, height, layers);
    if (rc != CCU_OK) return rc;
    for (int l = 0; l < layers; l++) {
        rc = ccu_scene_atlas_write(c, 0, 0, l, width, height, rgba + (size_t)l * width * height * 4);
        if (rc != CCU_OK) return rc;
    }
    return CCU_OK;
}

int ccu_scene_set_sky(ccu_ctx *c, const uint8_t *rgba, int32_t res, float sky_intensity) {
    if (!c) return fail(CCU_EINVAL, "ccu_scene_set_sky: null context");
    if (!rgba || res <= 0 || res > 16384) return fail(CCU_EINVAL, "bad sky texture (res=%d)", res);
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    c->committed = false;
    CU(c->scene.sky.upload(reinterpret_cast<const uchar4 *>(rgba), (size_t)res * res, c->stream));
    c->scene.info.sky_res = res;
    c->scene.info.sky_intensity = sky_intensity;
    c->scene.info.have_sky = true;
    return CCU_OK;
}

int ccu_scene_set_sun(ccu_ctx *c, const int32_t sun_words[6]) {
    if (!c || !sun_words) return fail(CCU_EINVAL, "ccu_scene_set_sun: null argument");
    std::lock_guard<std::mutex> lk(c->mu);
    c->committed = false;
    memcpy(c->scene.info.sun_host, sun_words, sizeof c->scene.info.sun_host);
    c->scene.info.have_sun = true;
    return CCU_OK;
}

int ccu_scene_set_fog(ccu_ctx *c, float sigma, float sky_density, const float color[3], int32_t fast) {
    if (!c) return fail(CCU_EINVAL, "ccu_scene_set_fog: null context");
    if (!(sigma >= 0.0f) || !std::isfinite(sigma)) return fail(CCU_EINVAL, "ccu_scene_set_fog: sigma %g is negative or not finite", sigma);
    if (!(sky_density >= 0.0f && sky_density <= 1.0f)) return fail(CCU_EINVAL, "ccu_scene_set_fog: sky density %g is not in [0, 1]", sky_density);
    if (!color) return fail(CCU_EINVAL, "ccu_scene_set_fog: null colour");
    for (int i = 0; i < 3; i++)
        if (!(color[i] >= 0.0f) || !std::isfinite(color[i]))
            return fail(CCU_EINVAL, "ccu_scene_set_fog: colour component %d (%g) is negative or not finite", i, color[i]);
    if (fast != 0 && fast != 1) return fail(CCU_EINVAL, "ccu_scene_set_fog: fast must be 0 or 1 (got %d)", fast);
    std::lock_guard<std::mutex> lk(c->mu);
    c->committed = false;
    c->scene.info.set_fog(sigma, sky_density, color, fast);
    return CCU_OK;
}

// Kept on the host, bit-packed, until commit uploads it.
int ccu_scene_set_clouds(ccu_ctx *c, const uint8_t *mask, float size, float y0, float y1, float u0, float v0) {
    if (!c) return fail(CCU_EINVAL, "ccu_scene_set_clouds: null context");
    std::shared_ptr<ccu_host::CloudLayer> cl;
    if (mask) {
        if (!(size > 0.0f) || !std::isfinite(size)) return fail(CCU_EINVAL, "ccu_scene_set_clouds: size %g is not positive and finite", size);
        if (!std::isfinite(y0) || !std::isfinite(y1) || !std::isfinite(u0) || !std::isfinite(v0))
            return fail(CCU_EINVAL, "ccu_scene_set_clouds: y0 %g, y1 %g, u0 %g, v0 %g: each must be finite", y0, y1, u0, v0);
        if (!(y0 < y1)) return fail(CCU_EINVAL, "ccu_scene_set_clouds: y0 %g is not below y1 %g", y0, y1);
        try {
            cl = std::make_shared<ccu_host::CloudLayer>();
        } catch (const std::bad_alloc &) {
            return fail(CCU_ENOMEM, "ccu_scene_set_clouds: no host memory for the mask");
        }
        for (int b = 0; b < ccu_host::CLOUD_CELLS; b++) {
            if (mask[b]) {
                cl->bits[b >> 5] |= 1u << (b & 31);
                cl->any = true;
            }
        }
        cl->inv = 1.0f / size;
        cl->y0 = y0; cl->y1 = y1; cl->u0 = u0; cl->v0 = v0;
    }
    std::lock_guard<std::mutex> lk(c->mu);
    c->committed = false;
    c->scene.clouds = std::move(cl);
    return CCU_OK;
}

// Builds the layouts and the launch view from the uploads.  The context stays uncommitted until every step has succeeded.
int ccu_scene_commit(ccu_ctx *c) {
    if (!c) return fail(CCU_EINVAL, "ccu_scene_commit: null context");
    std::lock_guard<std::mutex> lk(c->mu);
    c->committed = false;
    ccu_host::Scene &sc = c->scene;
    const auto host = [&](ccu_host::SceneArray a) -> const std::vector<int> & { return *sc.arrays[a].host; };
    if (!sc.arrays[ccu_host::OCTREE].host) return fail(CCU_ESTATE, "commit: octree not set");
    if (!sc.arrays[ccu_host::BLOCK_PALETTE].host || !sc.arrays[ccu_host::MAT_PALETTE].host) return fail(CCU_ESTATE, "commit: block/material palette not set");
    if (!sc.info.have_atlas) return fail(CCU_ESTATE, "commit: texture atlas not set");
    if (!sc.info.have_sky) return fail(CCU_ESTATE, "commit: sky not set");
    if (!sc.info.have_sun) return fail(CCU_ESTATE, "commit: sun not set");
    DeviceGuard g(c->device);
    const auto t0 = std::chrono::steady_clock::now();
    // absent optional arrays behave as the reference's single zero word / EMPTY_NODE (only optional ones can be absent here)
    for (ccu_host::PackedArray &a : sc.arrays) {
        if (a.host) continue;
        CU(a.dev.upload(nullptr, 0, c->stream));
        a.host = std::make_shared<const std::vector<int>>();
    }
    ccu_host::SceneInfo in = sc.info;
    // octree layouts: value-carrying (top table + 64-ary nodes) and march layout (top table + bricks); a tree that cannot be
    // encoded (malformed, leaf values beyond 26 bits) leaves the flags at 0 and rendering uses the reference's own array
    {
        const bool enable = getenv("CCU_NO_WIDE") == nullptr;
        const std::vector<int> &tree = host(ccu_host::OCTREE);
        WideLayout wl = build_wide_layout(tree.data(), tree.size(), in.depth);
        in.use_wide = (enable && wl.ok) ? 1 : 0;
        in.cell_level = wl.cell_level;
        in.top_log2 = wl.top_log2;
        CU(sc.top.upload(wl.top.data(), wl.top.size(), c->stream));
        CU(sc.wide.upload(wl.wide.data(), wl.wide.size(), c->stream));
        AirLayout al = build_air_layout(tree.data(), tree.size(), in.depth);
        in.use_air = (enable && al.ok) ? 1 : 0;
        in.air_cell_level = al.cell_level;
        in.air_top_log2 = al.top_log2;
        in.air_deep = al.cell_level > 4 ? 1 : 0;
        CU(sc.air_top.upload(al.top.data(), al.top.size(), c->stream));
        CU(sc.air_wide.upload(al.wide.data(), al.wide.size(), c->stream));
        CU(sc.air_bricks.upload(al.bricks.data(), al.bricks.size(), c->stream));
    }
    // 16-byte-vectorised block / material / model palettes
    {
        PaletteRecs pr = build_palette_recs(host(ccu_host::BLOCK_PALETTE), host(ccu_host::MAT_PALETTE), host(ccu_host::QUAD_MODELS),
                                            host(ccu_host::AABB_MODELS));
        CU(sc.block_rec.upload(pr.block.data(), pr.block.size(), c->stream));
        CU(sc.mat_rec.upload(pr.mat.data(), pr.mat.size(), c->stream));
        CU(sc.quad_rec.upload(pr.quad.data(), pr.quad.size(), c->stream));
        CU(sc.aabb_rec.upload(pr.aabb.data(), pr.aabb.size(), c->stream));
        // word 5 (specular / metalness / roughness) of every material on a record, and of every full cube's material
        in.has_specular = 0;
        for (size_t i = 0; i + 7 < pr.mat.size(); i += 8) in.has_specular |= pr.mat[i + 5] != 0;
        for (size_t i = 0; i + 7 < pr.block.size(); i += 8) in.has_specular |= pr.block[i] == 1 && pr.block[i + 7] != 0;
        // emitter table and cell lists, only when a full cube emits (a scene without one uploads three empty arrays)
        EmitterGrid eg;
        bool any = false;
        for (int b = 0; (size_t)b * 8 < pr.block.size() && !any; b++) any = block_emits(pr.block, b);
        if (any) {
            const std::vector<int> &tree = host(ccu_host::OCTREE);
            eg = build_emitter_grid(tree.data(), tree.size(), in.depth, [&](int b) { return block_emits(pr.block, b); });
        }
        in.has_emitters = eg.emit.empty() ? 0 : 1;
        for (int a = 0; a < 3; a++) { in.emit_g0[a] = eg.g0[a]; in.emit_dim[a] = eg.dim[a]; }
        in.emit_shift = eg.shift;
        CU(sc.emit.upload(eg.emit.data(), eg.emit.size(), c->stream));
        CU(sc.emit_off.upload(eg.off.data(), eg.off.size(), c->stream));
        CU(sc.emit_list.upload(eg.list.data(), eg.list.size(), c->stream));
        // the wider table of CCU_RENDER_EMITTER_MODELS, only when a model emits (otherwise five empty arrays)
        const ModelEmitters me = build_model_emitters(pr, host(ccu_host::MAT_PALETTE));
        const std::vector<int> &mtree = host(ccu_host::OCTREE);
        const EmitterGrid mg = build_model_grid(mtree.data(), mtree.size(), in.depth, pr, me);
        in.has_model_emitters = mg.emit.empty() ? 0 : 1;
        for (int a = 0; a < 3; a++) { in.memit_g0[a] = mg.g0[a]; in.memit_dim[a] = mg.dim[a]; }
        in.memit_shift = mg.shift;
        CU(sc.memit.upload(mg.emit.data(), mg.emit.size(), c->stream));
        CU(sc.memit_off.upload(mg.off.data(), mg.off.size(), c->stream));
        CU(sc.memit_list.upload(mg.list.data(), mg.list.size(), c->stream));
        CU(sc.memit_head.upload(in.has_model_emitters ? me.head.data() : nullptr, in.has_model_emitters ? me.head.size() : 0, c->stream));
        CU(sc.memit_prim.upload(in.has_model_emitters ? me.prim.data() : nullptr, in.has_model_emitters ? me.prim.size() : 0, c->stream));
    }
    // BVH stage layout (pair records + aligned triangle blocks); a scene whose BVHs it cannot hold is rendered by the
    // thread-per-pixel kernel on the reference's own arrays
    {
        const std::vector<int> &world = host(ccu_host::WORLD_BVH), &actor = host(ccu_host::ACTOR_BVH);
        const BvhStage bs = build_bvh_stage(world, actor, host(ccu_host::TRIANGLES));
        in.world_bvh_empty = bvh_is_empty(world);
        in.actor_bvh_empty = bvh_is_empty(actor);
        in.use_bvh2 = bs.ok ? 1 : 0;
        in.world_root = bs.world.root;
        in.actor_root = bs.actor.root;
        CU(sc.world_rec.upload(bs.world.rec.data(), bs.world.rec.size(), c->stream));
        CU(sc.actor_rec.upload(bs.actor.rec.data(), bs.actor.rec.size(), c->stream));
        CU(sc.tris2.upload(bs.tris.data(), bs.tris.size(), c->stream));
    }
    // biome colours (CCU_RENDER_BIOME_TINT), only when set
    in.has_biome = 0;
    for (int &v : in.biome_box) v = 0;
    sc.biome_grid.release();
    sc.biome_tiles.release();
    if (sc.biome) {
        const ccu_host::BiomeColors &bc = *sc.biome;
        BiomeLayout bl;
        const int rc = biome_layout(bc.chunks.data(), bc.rgb.data(), (int64_t)bc.chunks.size() / 2, in.depth, bl, "commit");
        if (rc != CCU_OK) return rc;
        CU(sc.biome_grid.upload(bl.grid.data(), bl.grid.size(), c->stream));
        CU(sc.biome_tiles.upload(reinterpret_cast<const float4 *>(bl.tiles.data()), bl.tiles.size() / 4, c->stream));
        in.has_biome = 1;
        in.biome_box[0] = bl.x0; in.biome_box[1] = bl.z0; in.biome_box[2] = bl.gx; in.biome_box[3] = bl.gz;
    }
    // cloud layer (CCU_RENDER_CLOUDS), only when set
    in.has_clouds = 0;
    in.cloud_inv = in.cloud_y0 = in.cloud_y1 = in.cloud_u0 = in.cloud_v0 = 0.0f;
    sc.cloud_mask.release();
    if (sc.clouds) {
        const ccu_host::CloudLayer &cl = *sc.clouds;
        CU(sc.cloud_mask.upload(cl.bits, ccu_host::CLOUD_WORDS, c->stream));
        in.has_clouds = cl.any ? 1 : 0;
        in.cloud_inv = cl.inv; in.cloud_y0 = cl.y0; in.cloud_y1 = cl.y1; in.cloud_u0 = cl.u0; in.cloud_v0 = cl.v0;
    }
    // sun basis, computed on the device
    {
        DevBuf<int> words;
        DevBuf<float> basis;
        CU(words.upload(in.sun_host, 6, c->stream));
        CU(basis.alloc(10));
        k_sun_setup<<<1, 1, 0, c->stream>>>(words.p, basis.p);
        c->launches++;
        CU(cudaGetLastError());
        float b[10];
        CU(cudaMemcpyAsync(b, basis.p, sizeof b, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        in.su = make_float3(b[0], b[1], b[2]);
        in.sv = make_float3(b[3], b[4], b[5]);
        in.sw = make_float3(b[6], b[7], b[8]);
        in.sun_radius_cos = b[9];
    }
    sc.info = in;
    fill_view(sc);
    c->commit_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    c->committed = true;
    return CCU_OK;
}

// ClCamera.java:33-70 (settings) / :72-105 (pre-generated rays).  Ray uploads go to the buffer no launch is reading, on the
// copy stream, so that they overlap the passes in flight (the reference's cameraGenTask, OpenClPathTracingRenderer.java:146-148);
// the next ccu_render_passes uses the new rays.
int ccu_camera_set(ccu_ctx *c, int32_t projector_type, const float *settings, int64_t n) {
    if (!c || !settings) return fail(CCU_EINVAL, "ccu_camera_set: null argument");
    std::lock_guard<std::mutex> cam(c->cam_mu);
    if (projector_type != -1) {
        if (n < 15) return fail(CCU_EINVAL, "camera settings need 15 floats (got %lld)", (long long)n);
        std::lock_guard<std::mutex> lk(c->mu);
        memcpy(c->cam, settings, sizeof c->cam);
        c->projector_type = projector_type;
        c->have_camera = true;
        return CCU_OK;
    }
    if (n % 6 != 0 || n <= 0) return fail(CCU_EINVAL, "pre-generated rays need 6 floats per pixel (got %lld)", (long long)n);
    int target;
    cudaEvent_t used;
    {
        std::lock_guard<std::mutex> lk(c->mu);
        target = (c->have_camera && c->projector_type == -1) ? 1 - c->rays_active : c->rays_active;
        used = c->rays_used[target];
    }
    DeviceGuard g(c->device);
    CU(cudaEventSynchronize(used));              // launches that read this buffer are done (outside the context lock)
    DevBuf<float> &buf = c->rays[target];        // only camera updates (serialised by cam_mu) touch the inactive buffer
    if (buf.n != (size_t)n) CU(buf.alloc((size_t)n));
    CU(cudaMemcpyAsync(buf.p, settings, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, c->copy_stream));
    CU(cudaStreamSynchronize(c->copy_stream));   // host memory is not retained past the call
    std::lock_guard<std::mutex> lk(c->mu);
    c->rays_active = target;
    c->projector_type = -1;
    c->have_camera = true;
    return CCU_OK;
}

int ccu_render_end(ccu_ctx *c) {
    if (!c) return fail(CCU_EINVAL, "ccu_render_end: null context");
    int rc = wait_render_stream(c);
    std::unique_lock<std::mutex> lk(c->mu);
    const int rc2 = c->merge.join(lk);
    DeviceGuard g(c->device);
    stop_timer(c);
    // the buffers stay cached for the next render of the same size (freed by ccu_ctx_destroy / a size change)
    c->target_live = false;
    c->window_spp = 0;
    c->closed_spp = 0;
    return rc != CCU_OK ? rc : rc2;
}

int ccu_render_begin(ccu_ctx *c, int32_t width, int32_t height) {
    if (!c) return fail(CCU_EINVAL, "ccu_render_begin: null context");
    if (width <= 0 || height <= 0 || (int64_t)width * height > (1ll << 30)) return fail(CCU_EINVAL, "bad canvas %dx%d", width, height);
    std::unique_lock<std::mutex> lk(c->mu);
    int rc = c->merge.join(lk);
    if (rc != CCU_OK) return rc;
    DeviceGuard g(c->device);
    cudaStreamSynchronize(c->stream);
    const size_t align = std::max<size_t>(1, c->accum_align);
    const size_t n = (((size_t)width * height * 3 + align - 1) / align) * align;
    if (c->accum[0].p && c->accum_floats != n) free_target(c);
    if (!c->accum[0].p) {
        cudaError_t e = c->accum[0].alloc(n);
        if (e == cudaSuccess) e = c->accum[1].alloc(n);
        if (e == cudaSuccess) e = c->pinned.alloc(n);
        if (e != cudaSuccess) {
            free_target(c);       // nothing half-allocated survives a failed begin
            return fail(e == cudaErrorMemoryAllocation ? CCU_ENOMEM : CCU_ECUDA, "ccu_render_begin: %s", cudaGetErrorString(e));
        }
        c->accum_floats = n;
        CU(cudaMemsetAsync(c->accum[1].p, 0, n * sizeof(float), c->stream));
    }
    c->accum_active = 0;
    CU(cudaMemsetAsync(c->accum[0].p, 0, n * sizeof(float), c->stream));
    c->window_base = c->accum[0].p;
    c->width = width;
    c->height = height;
    c->window_spp = 0;
    c->closed_spp = 0;
    c->target_live = true;
    return CCU_OK;
}

int ccu_render_set_params(ccu_ctx *c, const ccu_render_params *p) {
    // the parameters are checked before the context, so that a host can validate them without a device
    if (!p) return fail(CCU_EINVAL, "ccu_render_set_params: null argument");
    if (p->draw_depth < 0 || p->draw_depth >= (1 << 24) || p->max_depth < 1 || p->max_depth > 255) return fail(CCU_EINVAL, "bad render params");
    if (p->kernel != 0 && p->kernel != 1 && p->kernel != 4) return fail(CCU_EINVAL, "unknown kernel %d (0 auto, 1 thread-per-pixel, 4 wavefront)", p->kernel);
    if (p->flags & ~(CCU_RENDER_NO_ENTITIES | CCU_RENDER_NO_SUN | CCU_RENDER_SPECULAR | CCU_RENDER_EMITTER_SAMPLING | CCU_RENDER_EMITTER_NEAR_FIELD |
                     CCU_RENDER_EMITTER_MODELS | CCU_RENDER_BIOME_TINT | CCU_RENDER_FOG | CCU_RENDER_CLOUDS))
        return fail(CCU_EINVAL, "unknown render flags 0x%x", p->flags);
    if ((p->flags & CCU_RENDER_EMITTER_NEAR_FIELD) && !(p->flags & CCU_RENDER_EMITTER_SAMPLING))
        return fail(CCU_EINVAL, "CCU_RENDER_EMITTER_NEAR_FIELD needs CCU_RENDER_EMITTER_SAMPLING");
    if ((p->flags & CCU_RENDER_EMITTER_MODELS) && !(p->flags & CCU_RENDER_EMITTER_SAMPLING))
        return fail(CCU_EINVAL, "CCU_RENDER_EMITTER_MODELS needs CCU_RENDER_EMITTER_SAMPLING");
    if (!c) return fail(CCU_EINVAL, "ccu_render_set_params: null argument");
    std::lock_guard<std::mutex> lk(c->mu);
    c->params = *p;
    return CCU_OK;
}

static int render_ready(ccu_ctx *c, const char *what) {
    if (!c->committed) return fail(CCU_ESTATE, "%s: scene not committed", what);
    if (!c->have_camera) return fail(CCU_ESTATE, "%s: camera not set", what);
    if (!c->accum[0].p || !c->target_live) return fail(CCU_ESTATE, "%s: ccu_render_begin not called", what);
    if (c->projector_type == -1 && c->rays[c->rays_active].n != (size_t)c->width * c->height * 6)
        return fail(CCU_ESTATE, "%s: ray buffer holds %zu floats, canvas needs %zu", what, c->rays[c->rays_active].n, (size_t)c->width * c->height * 6);
    return CCU_OK;
}

// which implementation closestIntersect runs on: 0 = the reference's own arrays, 1 / 2 = commit-time layouts (2: deep world)
static int layout_mode(const ccu_ctx *c) { return (c->scene.info.use_wide && c->scene.info.use_air) ? (c->scene.info.air_deep ? 2 : 1) : 0; }

static int render_passes_locked(ccu_ctx *c, const int32_t *seeds, int32_t n_passes, bool first_chunk) {
    ccu_host::SeedRing &ring = c->seeds;
    if (!ring.dev.p) {
        ccu_host::SeedRing r;
        CU(r.dev.alloc((size_t)SEED_SLOTS * SEED_SLOT_INTS));
        CU(r.pinned.alloc((size_t)SEED_SLOTS * SEED_SLOT_INTS));
        for (Event &ev : r.ev) CU(ev.create(cudaEventDisableTiming));
        ring = std::move(r);
    }
    const int slot = ring.slot;
    ring.slot = (slot + 1) % SEED_SLOTS;
    CU(cudaEventSynchronize(ring.ev[slot]));        // blocks only when SEED_SLOTS batches are already queued
    int *seeds_host = ring.pinned + (size_t)slot * SEED_SLOT_INTS, *seeds_dev = ring.dev.p + (size_t)slot * SEED_SLOT_INTS;
    memcpy(seeds_host, seeds, (size_t)n_passes * sizeof(int));
    CU(cudaMemcpyAsync(seeds_dev, seeds_host, (size_t)n_passes * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    const DScene s = launch_view(c);
    const int n_pixels = c->width * c->height;
    if (!c->work_counter.p) CU(c->work_counter.alloc(1));
    if (first_chunk) CU(cudaEventRecord(c->ev0, c->stream));
    const bool bvh = !(s.world_bvh_empty && s.actor_bvh_empty);
    const int mode = layout_mode(c);
    const ShadeKey shade = shade_variant(c);
    const EmitView &emit_view = nee_models(shade.nee) ? c->scene.memit_view : c->scene.emit_view;
    const BiomeView &biome_view = c->scene.biome_view;
    const CloudView &cloud_view = c->scene.cloud_view;
    float *res = c->accum[c->accum_active].p;
    const float *res_prev = c->window_spp == 0 ? c->window_base : res;
    int kernel = c->params.kernel;
    if (kernel == 0) kernel = (mode != 0 && (!bvh || c->scene.info.use_bvh2)) ? 4 : 1;   // layouts refused at commit: the reference's own arrays
    int lay = 0, sky_staged = 0;   // kernel 4: its LAY, and the sky texels it stages in shared memory
    if (kernel == 1) {
        const int threads = 128, blocks = (n_pixels + threads - 1) / threads;
        dispatch<3>(mode, [&](auto M) {
            mega_kernel<M>(shade)<<<blocks, threads, 0, c->stream>>>(s, seeds_dev, n_passes, c->window_spp, res, res_prev, n_pixels,
                                                                     emit_view, biome_view, cloud_view);
        });
    } else {
        // persistent wavefront kernel (ccu_queue.cuh): one CTA per SM, pixels handed out through a counter
        if (mode == 0) return fail(CCU_ESTATE, "ccu_render_passes: kernel 4 needs the commit-time octree layouts (malformed octree?)");
        if (bvh && !c->scene.info.use_bvh2) return fail(CCU_ESTATE, "ccu_render_passes: kernel 4 cannot hold this BVH (malformed, or deeper than the 64 entries of the reference's traversal stack, bvh.h:38); use kernel 0 or 1");
        CU(cudaMemsetAsync(c->work_counter.p, 0, sizeof(unsigned int), c->stream));
        QueueParams qp;
        qp.w.seeds = seeds_dev;
        qp.w.n_passes = n_passes;
        qp.w.start_spp = c->window_spp;
        qp.w.res = res;
        qp.w.res_prev = res_prev;
        qp.w.n_pixels = n_pixels;
        qp.w.next_pixel = c->work_counter.p;
        qp.yield_below = c->yield_below;
        qp.refill_min = c->q_refill_min;
        qp.march_bias = c->q_march_bias;
        qp.shade_min = c->q_shade_min;
        qp.sticky_min = c->q_sticky_min > 0 ? c->q_sticky_min : (bvh ? 16 : 33);   // measured: -3 % with BVH stages, +5 % without
        qp.march_warps = bvh ? 64 : c->q_march_warps;   // the cap applies to the BVH-less kernels; with BVH stages every warp may march
        lay = queue_layout(c, bvh, shade);
        const int grid = c->sm_count, block = Q_WARPS * 32;
        // The sky table is staged in shared memory when it is small: shared memory and L1 are one array on this chip, and a
        // 128 x 128 table (64 KiB) taken from L1 costs more brick / atlas hits than the sky lookups gain (measured: +1.8 % per
        // pass on config 1).  CCU_SKY_SMEM_MAX (bytes, default 16 KiB = 64 x 64 texels) moves the threshold.
        const int sky_texels = c->scene.info.sky_res * c->scene.info.sky_res;
        const int base_smem = q_smem_bytes(bvh, lay == 0, shade.spec, shade.nee != NEE_NONE, shade.fog);
        const char *sky_env = getenv("CCU_SKY_SMEM_MAX");
        const int sky_max = sky_env ? atoi(sky_env) : 16384;
        const bool sky_smem = sky_texels * 4 <= sky_max && base_smem + sky_texels * 4 <= Q_SMEM_LIMIT;
        qp.sky_texels = sky_staged = sky_smem ? sky_texels : 0;
        qp.bvh_deep = nullptr;
        if (bvh) {
            // scratch for traversal-stack entries beyond the shared-memory part (bvh.h:38 allows 64 pending nodes)
            if (!c->bvh_deep.p) CU(c->bvh_deep.alloc((size_t)c->sm_count * Q_SLOTS * Q_DEEP));
            qp.bvh_deep = c->bvh_deep.p;
        }
        const int smem = base_smem + qp.sky_texels * 4;
        queue_kernel(bvh, lay, shade)<<<grid, block, smem, c->stream>>>(s, qp, emit_view, biome_view, cloud_view);
#ifdef CCU_Q_STATS
        {
            cudaStreamSynchronize(c->stream);
            unsigned long long st[32];
            dispatch(bvh, [&](auto B) {
                dispatch<3>(lay, [&](auto L) { dispatch(shade.clouds, [&](auto C) { queue_stats_take<B, L, C>(st); }); });
            });
            const char *names[4] = {"march", "block", "exit", "end"};
            fprintf(stderr, "[qstats] ");
            for (int i = 1; i < 4; i++) fprintf(stderr, "%s: %llu x %.1f lanes  ", names[i], st[2 * i], st[2 * i] ? (double)st[2 * i + 1] / st[2 * i] : 0.0);
            fprintf(stderr, "\n[qstats] march stages %llu, iterations %llu x %.1f lanes in flight, yields %llu, idle rounds %llu, pops %llu retries %llu\n", st[0], st[10],
                    st[10] ? (double)st[11] / st[10] : 0.0, st[13], st[12], st[14], st[15]);
            fprintf(stderr, "[qstats] bvh stages %llu, steps %llu x %.1f walking lanes, leaf turns %llu x %.1f lanes, shade %llu x %.1f lanes\n", st[16], st[18],
                    st[18] ? (double)st[19] / st[18] : 0.0, st[20], st[20] ? (double)st[21] / st[20] : 0.0, st[22], st[22] ? (double)st[23] / st[22] : 0.0);
            fprintf(stderr, "[qstats] march refills %llu, bvh refills %llu\n", st[24], st[25]);
        }
#endif
    }
    c->launches++;
    const int32_t last[9] = {kernel, bvh, kernel == 1 ? mode : lay, shade.spec, shade.nee, shade.biome, sky_staged, shade.fog, shade.clouds};
    std::copy(last, last + 9, c->last_render);
    CU(cudaGetLastError());
    CU(cudaEventRecord(c->ev1, c->stream));
    CU(cudaEventRecord(ring.ev[slot], c->stream));
    if (c->projector_type == -1) CU(cudaEventRecord(c->rays_used[c->rays_active], c->stream));
    c->timing_pending = true;
    c->window_spp += n_passes;
    c->window_base = res;
    return CCU_OK;
}

int ccu_render_passes_async(ccu_ctx *c, const int32_t *seeds, int32_t n_passes) {
    if (!c) return fail(CCU_EINVAL, "ccu_render_passes: null context");
    if (n_passes < 0 || (n_passes > 0 && !seeds)) return fail(CCU_EINVAL, "ccu_render_passes: bad seeds");
    std::lock_guard<std::mutex> lk(c->mu);
    int rc = render_ready(c, "ccu_render_passes");
    if (rc != CCU_OK) return rc;
    if (n_passes == 0) return CCU_OK;
    DeviceGuard g(c->device);
    // one launch covers at most 32768 passes (the wavefront kernel keeps a path's pass index in 16 bits); the reference's
    // windows are at most 1024 passes (OpenClPathTracingRenderer.java:158)
    const int32_t kChunk = SEED_SLOT_INTS;
    for (int32_t off = 0; off < n_passes; off += kChunk) {
        rc = render_passes_locked(c, seeds + off, std::min(kChunk, n_passes - off), off == 0);
        if (rc != CCU_OK) return rc;
    }
    return CCU_OK;
}

int ccu_render_sync(ccu_ctx *c) {
    if (!c) return fail(CCU_EINVAL, "ccu_render_sync: null context");
    int rc = wait_render_stream(c);       // the wait itself runs outside the context lock
    if (rc != CCU_OK) return rc;
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    stop_timer(c);
    return CCU_OK;
}

int ccu_render_passes(ccu_ctx *c, const int32_t *seeds, int32_t n_passes) {
    int rc = ccu_render_passes_async(c, seeds, n_passes);
    if (rc != CCU_OK) return rc;
    return ccu_render_sync(c);
}

int ccu_render_read(ccu_ctx *c, float *mean_rgb, int32_t *window_spp) {
    if (!c || !mean_rgb) return fail(CCU_EINVAL, "ccu_render_read: null argument");
    int rc = wait_render_stream(c);
    if (rc != CCU_OK) return rc;
    std::unique_lock<std::mutex> lk(c->mu);
    if (!c->accum[0].p || !c->target_live) return fail(CCU_ESTATE, "ccu_render_read: no render target");
    rc = c->merge.join(lk);
    if (rc != CCU_OK) return rc;
    if (c->closed_spp > 0) return fail(CCU_ESTATE, "ccu_render_read: a closed window is waiting for ccu_render_window_merge (it owns the staging buffer)");
    DeviceGuard g(c->device);
    const size_t n = (size_t)c->width * c->height * 3;
    CU(cudaMemcpyAsync(c->pinned, c->accum[c->accum_active].p, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    stop_timer(c);
    memcpy(mean_rgb, c->pinned, n * sizeof(float));
    if (window_spp) *window_spp = c->window_spp;
    return CCU_OK;
}

int ccu_render_merge_wait(ccu_ctx *c) {
    if (!c) return fail(CCU_EINVAL, "ccu_render_merge_wait: null context");
    std::unique_lock<std::mutex> lk(c->mu);
    return c->merge.join(lk);
}

// closes the window under the lock: the passes that follow accumulate in the other buffer (the first of them still reads
// what this buffer holds, like the reference's single buffer at bufferSpp = 0, rayTracer.cl:111); the read-back starts
static int window_close_locked(ccu_ctx *c, std::unique_lock<std::mutex> &lk, int32_t *window_spp) {
    if (!c->accum[0].p || !c->target_live) return fail(CCU_ESTATE, "no render target");
    int rc = c->merge.join(lk);       // one merge at a time: they share the staging buffer
    if (rc != CCU_OK) return rc;
    if (c->closed_spp > 0) return fail(CCU_ESTATE, "the previous window was closed but not merged (ccu_render_window_merge)");
    const int pass_spp = c->window_spp;
    if (window_spp) *window_spp = pass_spp;
    if (pass_spp == 0) return CCU_OK;
    DeviceGuard g(c->device);
    CU(cudaEventRecord(c->window_ev, c->stream));
    const float *src = c->accum[c->accum_active].p;
    c->accum_active ^= 1;
    c->window_base = src;
    c->window_spp = 0;   // bufferSppReal = 0 (:170)
    c->closed_spp = pass_spp;
    CU(cudaStreamWaitEvent(c->copy_stream, c->window_ev, 0));
    return ccu_host::start_readback(c, src, 0, (size_t)c->width * c->height * 3, c->copy_stream);
}

int ccu_render_window_close(ccu_ctx *c, int32_t *window_spp) {
    if (!c) return fail(CCU_EINVAL, "ccu_render_window_close: null context");
    std::unique_lock<std::mutex> lk(c->mu);
    return window_close_locked(c, lk, window_spp);
}

int ccu_render_window_merge(ccu_ctx *c, double *sample_buffer, int32_t sample_spp) {
    if (!c || !sample_buffer) return fail(CCU_EINVAL, "ccu_render_window_merge: null argument");
    if (sample_spp < 0) return fail(CCU_EINVAL, "ccu_render_window_merge: negative spp");
    int pass_spp;
    size_t n;
    {
        std::lock_guard<std::mutex> lk(c->mu);
        pass_spp = c->closed_spp;
        n = (size_t)c->width * c->height * 3;
    }
    if (pass_spp == 0) return CCU_OK;
    const double sinv = 1.0 / (double)(sample_spp + pass_spp);
    // the wait for the copies and the merge itself run outside the context lock: the next window renders meanwhile
    int rc = ccu_host::merge_readback(c, 0, n, sample_buffer, (double)sample_spp, (double)pass_spp, sinv, 16);
    std::lock_guard<std::mutex> lk(c->mu);
    c->closed_spp = 0;
    return rc;
}

int ccu_render_merge_async(ccu_ctx *c, double *sample_buffer, int32_t sample_spp, int32_t *merged_spp) {
    if (!c || !sample_buffer) return fail(CCU_EINVAL, "ccu_render_merge: null argument");
    if (sample_spp < 0) return fail(CCU_EINVAL, "ccu_render_merge: negative spp");
    std::unique_lock<std::mutex> lk(c->mu);
    int32_t pass_spp = 0;
    int rc = window_close_locked(c, lk, &pass_spp);
    if (merged_spp) *merged_spp = pass_spp;
    if (rc != CCU_OK || pass_spp == 0) return rc;
    c->merge.start([=] { return ccu_render_window_merge(c, sample_buffer, sample_spp); });
    return CCU_OK;
}

int ccu_render_merge(ccu_ctx *c, double *sample_buffer, int32_t sample_spp, int32_t *merged_spp) {
    if (!c || !sample_buffer) return fail(CCU_EINVAL, "ccu_render_merge: null argument");
    if (sample_spp < 0) return fail(CCU_EINVAL, "ccu_render_merge: negative spp");
    int32_t pass_spp = 0;
    {
        std::unique_lock<std::mutex> lk(c->mu);
        int rc = window_close_locked(c, lk, &pass_spp);
        if (merged_spp) *merged_spp = pass_spp;
        if (rc != CCU_OK) return rc;
    }
    int rc = ccu_render_window_merge(c, sample_buffer, sample_spp);
    if (rc != CCU_OK) return rc;
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    stop_timer(c);
    return CCU_OK;
}

int ccu_render_reset_window(ccu_ctx *c) {
    if (!c) return fail(CCU_EINVAL, "ccu_render_reset_window: null context");
    std::lock_guard<std::mutex> lk(c->mu);
    c->window_spp = 0;
    return CCU_OK;
}

int ccu_render_set_window_spp(ccu_ctx *c, int32_t window_spp) {
    if (!c) return fail(CCU_EINVAL, "ccu_render_set_window_spp: null context");
    if (window_spp < 0) return fail(CCU_EINVAL, "ccu_render_set_window_spp: negative pass count");
    std::lock_guard<std::mutex> lk(c->mu);
    c->window_spp = window_spp;
    return CCU_OK;
}

int ccu_render_device_buffer(ccu_ctx *c, void **device_ptr, int64_t *n_floats) {
    if (!c || !device_ptr) return fail(CCU_EINVAL, "ccu_render_device_buffer: null argument");
    std::lock_guard<std::mutex> lk(c->mu);
    if (!c->accum[0].p || !c->target_live) return fail(CCU_ESTATE, "ccu_render_device_buffer: no render target");
    *device_ptr = c->accum[c->accum_active].p;
    if (n_floats) *n_floats = (int64_t)c->width * c->height * 3;
    return CCU_OK;
}

int ccu_render_scale(ccu_ctx *c, float factor) {
    if (!c) return fail(CCU_EINVAL, "ccu_render_scale: null context");
    std::lock_guard<std::mutex> lk(c->mu);
    if (!c->accum[0].p || !c->target_live) return fail(CCU_ESTATE, "ccu_render_scale: no render target");
    DeviceGuard g(c->device);
    ccu_host::scale_window(c, factor, (size_t)c->width * c->height * 3);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream));
    return CCU_OK;
}

int ccu_stream_handle(ccu_ctx *c, void **cuda_stream) {
    if (!c || !cuda_stream) return fail(CCU_EINVAL, "ccu_stream_handle: null argument");
    std::lock_guard<std::mutex> lk(c->mu);
    *cuda_stream = (void *)c->stream;
    return CCU_OK;
}

int ccu_first_hit(ccu_ctx *c, int32_t seed, int32_t *block, int32_t *face, int32_t *node, int32_t *kind, float *t, float *normal,
                  float *color) {
    if (!c) return fail(CCU_EINVAL, "ccu_first_hit: null context");
    std::lock_guard<std::mutex> lk(c->mu);
    int rc = render_ready(c, "ccu_first_hit");
    if (rc != CCU_OK) return rc;
    DeviceGuard g(c->device);
    size_t n = (size_t)c->width * c->height;
    // one scratch allocation (kept for the next call): 4 int planes, colour(4), t, normal(3) = 12 words per pixel
    if (c->fh_scratch.n < n * 12) {
        cudaStreamSynchronize(c->stream);
        CU(c->fh_scratch.alloc(n * 12));
    }
    int *scratch = c->fh_scratch.p;
    // planes nobody asked for are not written
    int *d_block = block ? scratch : nullptr, *d_face = face ? scratch + n : nullptr, *d_node = node ? scratch + 2 * n : nullptr,
        *d_kind = kind ? scratch + 3 * n : nullptr;
    float *d_color = color ? reinterpret_cast<float *>(scratch + 4 * n) : nullptr;          // 16-byte aligned: n*16 bytes offset
    float *d_t = t ? reinterpret_cast<float *>(scratch + 8 * n) : nullptr;
    float *d_normal = normal ? reinterpret_cast<float *>(scratch + 9 * n) : nullptr;
    const DScene s = launch_view(c);
    const int mode = layout_mode(c);
    const unsigned blocks = (unsigned)((n + CCU_FH_THREADS - 1) / CCU_FH_THREADS);
    cudaEventRecord(c->ev0, c->stream);
    const bool fh_bvh = !(s.world_bvh_empty && s.actor_bvh_empty);
    const FirstHitOut fho = {d_block, d_face, d_node, d_kind, d_t, d_normal, d_color};
    dispatch(fh_bvh, [&](auto B) {
        dispatch<3>(mode, [&](auto M) { k_first_hit<M, B><<<blocks, CCU_FH_THREADS, 0, c->stream>>>(s, seed, (int)n, fho); });
    });
    c->launches++;
    cudaEventRecord(c->ev1, c->stream);
    if (c->projector_type == -1) cudaEventRecord(c->rays_used[c->rays_active], c->stream);
    c->timing_pending = true;
    cudaError_t e = cudaGetLastError();
    auto back = [&](void *dst, const void *src, size_t bytes) {
        if (dst && e == cudaSuccess) e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream);
    };
    back(block, d_block, n * 4); back(face, d_face, n * 4); back(node, d_node, n * 4); back(kind, d_kind, n * 4);
    back(t, d_t, n * 4); back(normal, d_normal, n * 12); back(color, d_color, n * 16);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return fail(CCU_ECUDA, "ccu_first_hit: %s", cudaGetErrorString(e));
    stop_timer(c);
    return CCU_OK;
}

int ccu_preview(ccu_ctx *c, int32_t *argb) {
    if (!c || !argb) return fail(CCU_EINVAL, "ccu_preview: null argument");
    std::lock_guard<std::mutex> lk(c->mu);
    int rc = render_ready(c, "ccu_preview");
    if (rc != CCU_OK) return rc;
    DeviceGuard g(c->device);
    size_t n = (size_t)c->width * c->height;
    DevBuf<int> d;
    CU(d.alloc(n));
    const DScene s = launch_view(c);
    const int mode = layout_mode(c);
    const unsigned blocks = (unsigned)((n + 255) / 256);
    cudaEventRecord(c->ev0, c->stream);
    dispatch<3>(mode, [&](auto M) { k_preview<M><<<blocks, 256, 0, c->stream>>>(s, (int)n, d.p); });
    c->launches++;
    cudaEventRecord(c->ev1, c->stream);
    if (c->projector_type == -1) cudaEventRecord(c->rays_used[c->rays_active], c->stream);
    c->timing_pending = true;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(argb, d.p, n * sizeof(int), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return fail(CCU_ECUDA, "ccu_preview: %s", cudaGetErrorString(e));
    stop_timer(c);
    return CCU_OK;
}

int ccu_last_kernel_ms(ccu_ctx *c, float *ms) {
    if (!c || !ms) return fail(CCU_EINVAL, "ccu_last_kernel_ms: null argument");
    int rc = wait_render_stream(c);
    if (rc != CCU_OK) return rc;
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    stop_timer(c);
    *ms = c->last_ms;
    return CCU_OK;
}

int ccu_launch_count(ccu_ctx *c, int64_t *launches) {
    if (!c || !launches) return fail(CCU_EINVAL, "ccu_launch_count: null argument");
    std::lock_guard<std::mutex> lk(c->mu);
    *launches = c->launches;
    return CCU_OK;
}

int ccu_debug_last_render(ccu_ctx *c, int32_t out[7]) {
    if (!c || !out) return fail(CCU_EINVAL, "ccu_debug_last_render: null argument");
    std::lock_guard<std::mutex> lk(c->mu);
    std::copy(c->last_render, c->last_render + 7, out);
    return CCU_OK;
}

int ccu_debug_last_render_n(ccu_ctx *c, int32_t *out, int32_t n) {
    if (!c || !out || n < 0) return fail(CCU_EINVAL, "ccu_debug_last_render_n: null argument or negative n");
    std::lock_guard<std::mutex> lk(c->mu);
    std::copy(c->last_render, c->last_render + std::min(n, 9), out);
    return CCU_OK;
}

int ccu_scene_device_bytes(ccu_ctx *c, int64_t *bytes) {
    if (!c || !bytes) return fail(CCU_EINVAL, "ccu_scene_device_bytes: null argument");
    std::lock_guard<std::mutex> lk(c->mu);
    size_t sum = 0;
    ccu_host::Scene::each_buf(c->scene, c->scene, [&](auto &b, auto &) { sum += b.bytes(); });
    *bytes = (int64_t)sum;
    return CCU_OK;
}

int ccu_scene_commit_ms(ccu_ctx *c, double *ms) {
    if (!c || !ms) return fail(CCU_EINVAL, "ccu_scene_commit_ms: null argument");
    std::lock_guard<std::mutex> lk(c->mu);
    *ms = c->commit_ms;
    return CCU_OK;
}

int ccu_tonemap(ccu_ctx *c, int32_t width, int32_t height, float exposure, const double *input, int32_t type, int32_t *argb) {
    if (!c || !input || !argb) return fail(CCU_EINVAL, "ccu_tonemap: null argument");
    if (width <= 0 || height <= 0 || (int64_t)width * height > (1ll << 30)) return fail(CCU_EINVAL, "ccu_tonemap: bad canvas %dx%d", width, height);
    if (type < 0 || type > 3) return fail(CCU_EINVAL, "ccu_tonemap: unknown filter %d (0 GAMMA, 1 TONEMAP1, 2 ACES, 3 HABLE)", type);
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    const size_t n = (size_t)width * height;
    DevBuf<double> d_in;
    DevBuf<uint32_t> d_out;
    CU(d_in.alloc(n * 3));
    cudaError_t e = d_out.alloc(n);
    // the reference uploads the whole double buffer and reads the ARGB image back on every call (GpuPostProcessingFilter.java:43-61)
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_in.p, input, n * 3 * sizeof(double), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
        cudaEventRecord(c->ev0, c->stream);
        k_tonemap<<<c->sm_count * 8, 256, 0, c->stream>>>((int)n, exposure, d_in.p, type, d_out.p);
        cudaEventRecord(c->ev1, c->stream);
        c->timing_pending = true;
        c->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(argb, d_out.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return fail(e == cudaErrorMemoryAllocation ? CCU_ENOMEM : CCU_ECUDA, "ccu_tonemap: %s", cudaGetErrorString(e));
    stop_timer(c);
    return CCU_OK;
}

int ccu_bench_gather(ccu_ctx *c, int64_t array_bytes, int32_t dependent, float *gbytes_per_s, float *ns_per_load) {
    if (!c || array_bytes < 4096) return fail(CCU_EINVAL, "ccu_bench_gather: bad argument");
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    size_t sectors = 1;
    while (sectors * 2 * 32 <= (size_t)array_bytes) sectors *= 2;   // power of two number of 32-byte sectors
    DevBuf<uint4> a;
    DevBuf<uint32_t> sink;
    CU(a.alloc(sectors * 2));
    cudaError_t e = sink.alloc(1);
    if (e != cudaSuccess) return fail(CCU_ENOMEM, "ccu_bench_gather: %s", cudaGetErrorString(e));
    k_gather_fill<<<c->sm_count * 8, 256, 0, c->stream>>>(a.p, sectors, 12345u);
    const int loads = dependent ? 2048 : 4096;
    const int blocks = dependent ? c->sm_count : c->sm_count * 8;
    float best = 1e30f;
    for (int it = 0; it < 4; it++) {   // first iteration warms the caches
        cudaEventRecord(c->ev0, c->stream);
        k_gather<<<blocks, dependent ? 32 : 256, 0, c->stream>>>(a.p, (uint32_t)(sectors - 1), loads, dependent, (uint32_t)it, sink.p);
        cudaEventRecord(c->ev1, c->stream);
        e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) break;
        float ms = 0;
        cudaEventElapsedTime(&ms, c->ev0, c->ev1);
        if (it > 0) best = std::min(best, ms);
    }
    c->launches += 5;
    if (e != cudaSuccess) return fail(CCU_ECUDA, "ccu_bench_gather: %s", cudaGetErrorString(e));
    const double n_loads = (double)blocks * (dependent ? 1.0 : 256.0) * loads;
    if (gbytes_per_s) *gbytes_per_s = (float)(n_loads * 32.0 / (best * 1e-3) / 1e9);
    if (ns_per_load) *ns_per_load = (float)(best * 1e6 / loads);   // per thread: meaningful for the dependent chain
    return CCU_OK;
}

// Host-only check of the BVH stage layout (no CUDA call): what ccu_scene_commit uploads for `bvh` as the world BVH of a scene
// without actors, padding included.
int ccu_debug_bvh_layout(const int32_t *bvh, int64_t n_bvh, const int32_t *trigs, int64_t n_trigs, int32_t *rec, int64_t rec_cap,
                         int32_t *tris, int64_t tris_cap, int64_t *rec_words, int64_t *tris_words, int32_t *root, int32_t *ok) {
    if (!bvh || n_bvh < 0 || n_trigs < 0 || (n_trigs > 0 && !trigs) || !rec_words || !tris_words || !root || !ok)
        return fail(CCU_EINVAL, "ccu_debug_bvh_layout: bad argument");
    const BvhStage s = build_bvh_stage(std::vector<int>(bvh, bvh + n_bvh), {}, std::vector<int>(trigs, trigs + n_trigs));
    const std::vector<int> &r = s.world.rec, &t = s.tris;
    *ok = s.ok ? 1 : 0;
    *root = s.world.root;
    *rec_words = (int64_t)r.size();
    *tris_words = (int64_t)t.size();
    if (rec) {
        if (rec_cap < (int64_t)r.size()) return fail(CCU_EINVAL, "ccu_debug_bvh_layout: rec buffer too small");
        std::copy(r.begin(), r.end(), rec);
    }
    if (tris) {
        if (tris_cap < (int64_t)t.size()) return fail(CCU_EINVAL, "ccu_debug_bvh_layout: tris buffer too small");
        std::copy(t.begin(), t.end(), tris);
    }
    return CCU_OK;
}

// Host-only check of the emitter table (no CUDA call): what ccu_scene_commit builds for this octree and these palettes.  info =
// {has_emitters, g0 x y z, dim x y z, shift, emitters, list words}; emit (4 ints per emitter), off (cells + 1) and list are
// filled when given, and must then hold what a call without them reported.
int ccu_debug_emitter_grid(const int32_t *tree, int64_t n_tree, int32_t depth, const int32_t *block_palette, int64_t n_block,
                           const int32_t *mat_palette, int64_t n_mat, int32_t info[10], int32_t *emit, int32_t *off, int32_t *list) {
    if (!tree || n_tree < 1 || depth < 0 || depth > 30 || !block_palette || n_block < 0 || !mat_palette || n_mat < 0 || !info)
        return fail(CCU_EINVAL, "ccu_debug_emitter_grid: bad argument");
    const PaletteRecs pr = build_palette_recs(std::vector<int>(block_palette, block_palette + n_block),
                                              std::vector<int>(mat_palette, mat_palette + n_mat), {}, {});
    const EmitterGrid g = build_emitter_grid(tree, (size_t)n_tree, depth, [&](int b) { return block_emits(pr.block, b); });
    info[0] = g.emit.empty() ? 0 : 1;
    for (int a = 0; a < 3; a++) { info[1 + a] = g.g0[a]; info[4 + a] = g.dim[a]; }
    info[7] = g.shift;
    info[8] = (int)(g.emit.size() / 4);
    info[9] = (int)g.list.size();
    if (emit) std::copy(g.emit.begin(), g.emit.end(), emit);
    if (off) std::copy(g.off.begin(), g.off.end(), off);
    if (list) std::copy(g.list.begin(), g.list.end(), list);
    return CCU_OK;
}

// Host-only check of the wider emitter table of CCU_RENDER_EMITTER_MODELS (no CUDA call): what ccu_scene_commit builds.  info =
// {has_model_emitters, g0 x y z, dim x y z, shift, emitters, list words, head entries, prim words}.
int ccu_debug_emitter_models(const int32_t *tree, int64_t n_tree, int32_t depth, const int32_t *block_palette, int64_t n_block,
                             const int32_t *mat_palette, int64_t n_mat, const int32_t *quad_models, int64_t n_quad,
                             const int32_t *aabb_models, int64_t n_aabb, int32_t info[12], int32_t *emit, int32_t *off,
                             int32_t *list, int32_t *head, int32_t *prim) {
    if (!tree || n_tree < 1 || depth < 0 || depth > 30 || !block_palette || n_block < 0 || !mat_palette || n_mat < 0 || !quad_models ||
        n_quad < 0 || !aabb_models || n_aabb < 0 || !info)
        return fail(CCU_EINVAL, "ccu_debug_emitter_models: bad argument");
    const std::vector<int> mp(mat_palette, mat_palette + n_mat);
    const PaletteRecs pr = build_palette_recs(std::vector<int>(block_palette, block_palette + n_block), mp,
                                              std::vector<int>(quad_models, quad_models + n_quad),
                                              std::vector<int>(aabb_models, aabb_models + n_aabb));
    const ModelEmitters me = build_model_emitters(pr, mp);
    const EmitterGrid g = build_model_grid(tree, (size_t)n_tree, depth, pr, me);
    const bool has = !g.emit.empty();
    info[0] = has ? 1 : 0;
    for (int a = 0; a < 3; a++) { info[1 + a] = g.g0[a]; info[4 + a] = g.dim[a]; }
    info[7] = g.shift;
    info[8] = (int)(g.emit.size() / 4);
    info[9] = (int)g.list.size();
    info[10] = has ? (int)me.head.size() : 0;
    info[11] = has ? (int)me.prim.size() : 0;
    if (emit) std::copy(g.emit.begin(), g.emit.end(), emit);
    if (off) std::copy(g.off.begin(), g.off.end(), off);
    if (list) std::copy(g.list.begin(), g.list.end(), list);
    if (head && has) std::copy(me.head.begin(), me.head.end(), head);
    if (prim && has) std::copy(me.prim.begin(), me.prim.end(), prim);
    return CCU_OK;
}

// Host-only check of the biome layout (no CUDA call): what ccu_scene_commit builds from these colours for an octree of `depth`.
int ccu_debug_biome_layout(const int32_t *chunks, const float *rgb, int64_t n, int32_t depth, int32_t info[5], int32_t *grid, float *tiles) {
    if (depth < 0 || depth > 30 || !info) return fail(CCU_EINVAL, "ccu_debug_biome_layout: bad argument");
    int rc;
    try {
        rc = check_biome_colors(chunks, rgb, n, "ccu_debug_biome_layout");
    } catch (const std::bad_alloc &) {
        return fail(CCU_ENOMEM, "ccu_debug_biome_layout: no host memory for %lld chunks", (long long)n);
    }
    if (rc != CCU_OK) return rc;
    BiomeLayout bl;
    rc = biome_layout(chunks, rgb, n, depth, bl, "ccu_debug_biome_layout");
    if (rc != CCU_OK) return rc;
    info[0] = bl.x0; info[1] = bl.z0; info[2] = bl.gx; info[3] = bl.gz;
    info[4] = (int)n;
    if (grid) std::copy(bl.grid.begin(), bl.grid.end(), grid);
    if (tiles) std::copy(bl.tiles.begin(), bl.tiles.end(), tiles);
    return CCU_OK;
}

// Host-only check of the commit-time traversal layouts (no CUDA call): for every voxel of `xyz` (count x 3 ints) returns what
// the value-carrying layout (find_leaf_wide) and the march layout (lean_probe) answer, so that CPU tests can compare both
// with the reference's root descent (octree.h:81-88).
int ccu_debug_layout_lookup(const int32_t *tree, int64_t n, int32_t depth, const int32_t *xyz, int64_t count, int32_t *wide_value,
                            int32_t *wide_level, int32_t *air_solid, int32_t *air_level) {
    if (!tree || n < 1 || depth < 0 || depth > 30 || (count > 0 && !xyz)) return fail(CCU_EINVAL, "ccu_debug_layout_lookup: bad argument");
    WideLayout wl = build_wide_layout(tree, (size_t)n, depth);
    AirLayout al = build_air_layout(tree, (size_t)n, depth);
    if (!al.ok) return fail(CCU_ESTATE, "air layout could not be built");
    const int cl = wl.cell_level, tl = wl.top_log2;
    for (int64_t i = 0; i < count; i++) {
        const int bx = xyz[3 * i], by = xyz[3 * i + 1], bz = xyz[3 * i + 2];
        if (((bx | by | bz) >> depth) != 0) return fail(CCU_EINVAL, "voxel %lld outside the octree cube", (long long)i);
        if (wl.ok) {
            const size_t cell = ((((size_t)(bx >> cl) << tl) + (size_t)(by >> cl)) << tl) + (size_t)(bz >> cl);
            unsigned e = wl.top[cell];
            int lvl = cl;
            while (!(e & CCU_WIDE_LEAF)) {
                lvl -= 2;
                e = wl.wide[(size_t)e * 64 + ((((bx >> lvl) & 3) << 4) | (((by >> lvl) & 3) << 2) | ((bz >> lvl) & 3))];
            }
            const unsigned v = e & CCU_WIDE_ANY;
            if (wide_value) wide_value[i] = v == CCU_WIDE_ANY ? CCU_ANY_TYPE : (int)v;
            if (wide_level) wide_level[i] = (int)((e >> 26) & 31);
        } else {
            if (wide_value) wide_value[i] = -1;
            if (wide_level) wide_level[i] = -1;
        }
        // the lookup of lean_probe (ccu_march.cuh)
        int lvl = al.cell_level;
        const int atl = al.top_log2;
        unsigned e = al.top[((((size_t)(bx >> lvl) << atl) + (size_t)(by >> lvl)) << atl) + (size_t)(bz >> lvl)];
        while (lvl > 4 && !(e & CCU_WIDE_LEAF)) {
            lvl -= 2;
            e = al.wide[(size_t)e * 64 + ((((bx >> lvl) & 3) << 4) | (((by >> lvl) & 3) << 2) | ((bz >> lvl) & 3))];
        }
        int level;   // -1 = not air
        if (e & CCU_WIDE_LEAF) {        // deep worlds only: shallow top entries are all brick offsets
            level = ((int)(e << 1)) >> 27;
        } else {
            const int code = air_brick_level(al.bricks[(size_t)e + air_brick_word(bx, by, bz)], bz);
            level = code == CCU_AIR_SOLID ? -1 : code;
        }
        if (air_solid) air_solid[i] = level < 0 ? 1 : 0;
        if (air_level) air_level[i] = level;
    }
    return CCU_OK;
}

}  // extern "C"
