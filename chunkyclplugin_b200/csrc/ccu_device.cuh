// ccu_device.cuh - device-side scene description and the traversal / shading functions.
//
// Written from the behaviour of the reference kernels (cited per function, paths under
// /root/reference/src/main/opencl/kernel/include/); structure, data layout and control flow are ours.
#pragma once
#include "ccu_math.cuh"

namespace ccu {

#define CCU_ANY_TYPE 0x7FFFFFFE   // block.h:32

struct DScene {   // what a launch reads: commit fills the scene's fields once (ccu_host::Scene::view), a launch adds the rest
    // octree (reference numbering: ClSceneLoader.java:56-59)
    const int *__restrict__ tree;
    int depth;
    // traversal layout built at commit (result-identical to the root descent of octree.h:81-88):
    //   top[]   dense table over the cells of level `cell_level` (edge 1 << cell_level), index (x*dim + y)*dim + z
    //   wide[]  64-ary nodes, each covering two octree levels: entry ((x&3)<<4 | (y&3)<<2 | (z&3)) at the node's level
    // entry encoding: bit 31 set = leaf {level: bits 30..26, value: bits 25..0 (0x3FFFFFF = ANY_TYPE)};
    //                 bit 31 clear = index of a wide node (in units of 64 words)
    const unsigned *__restrict__ top;
    const unsigned *__restrict__ wide;
    int cell_level, top_log2;
    int use_wide;
    // march-loop ("air") layout, see ccu_march.cuh: top table over cells of level air_cell_level (>= 4), 64-ary nodes
    // down to level 4 (deep worlds only), one 1-KiB brick of 2-bit voxel codes per 16^3 cell that is not a single leaf
    const unsigned *__restrict__ air_top;
    const unsigned *__restrict__ air_wide;
    const unsigned *__restrict__ air_bricks;
    int air_cell_level, air_top_log2;
    // palettes (reference packed layouts, SURVEY 8a)
    const int *__restrict__ block_palette;
    int block_palette_len;
    const int *__restrict__ quad_models;
    const int *__restrict__ aabb_models;
    const int *__restrict__ mat_palette;
    // 16-byte-vectorised palettes built at commit (always present): block_rec[2 * b] = {type, model ref, material flags, tint},
    // block_rec[2 * b + 1] = {texSize, texLocation / ARGB, emittance, spec} for palette position b (a full-cube block is ONE
    // 32-byte record: entry and material fused); mat_rec[2 * (ptr / 6)] the same six material words for everything else;
    // quad_rec / aabb_rec: {count, 0, 0, 0} followed by one 64-byte record per quad (15 words + pad) / box (13 words + pad),
    // referenced from block_rec in units of 16 bytes
    const int4 *__restrict__ block_rec;
    const int4 *__restrict__ mat_rec;
    const int4 *__restrict__ quad_rec;
    const int4 *__restrict__ aabb_rec;
    const int *__restrict__ world_bvh;
    const int *__restrict__ actor_bvh;
    const int *__restrict__ trigs;
    int world_bvh_empty, actor_bvh_empty;   // the bvh.h:23-32 probe, evaluated once at commit; CCU_RENDER_NO_ENTITIES sets both
    // BVH stage layout (built at commit): one 64-byte record per inner node = two 32-byte halves of the same shape, {box (6 floats),
    // ref, 0} of the first child and of the second child (a pair of lanes fetches a record with ONE L1 wavefront, ccu_queue.cuh);
    // 32-byte aligned triangle blocks {count, 0 x 7} + count x 24 words (PackedTriangle's 20 words + pad: three 256-bit loads per
    // triangle); ref >= 0 record, ref < 0: -(1 + block offset / 8 words)
    const int4 *__restrict__ world_rec;
    const int4 *__restrict__ actor_rec;
    const int *__restrict__ tris2;
    int world_root, actor_root;
    // atlas: RGBA8, tile-linear (16x16 texel tiles contiguous), clamp extents = image extents
    const uchar4 *__restrict__ atlas;
    int atlas_w, atlas_h, atlas_layers, atlas_tiles_x, atlas_tiles_y;
    // sky: RGBA8 res x res
    const uchar4 *__restrict__ sky;
    int sky_res;
    float sky_intensity;
    const float *__restrict__ unorm;      // unorm[b] = (float)b / 255.0f
    // sun (Sun_new sky.h:19-40 evaluated once on the device at commit)
    int sun_flags, sun_tex_size, sun_tex;
    float sun_intensity, sun_radius_cos;
    float3 su, sv, sw;
    // camera (per launch, like everything below)
    int projector_type;
    float cam[15];
    const float *__restrict__ rays;
    int width, height;
    float half_width, inv_height;
    // launch parameters
    int draw_depth, max_depth;
    float emitter_scale;
    // the scene's fog (ccu_scene_set_fog, DESIGN §14), read only by the fog kernels; kept last so that no other field moves
    float fog_sigma, fog_sky;
    float3 fog_color;
    int fog_fast;
};

// The emitter table of CCU_RENDER_EMITTER_SAMPLING (DESIGN §10), built at commit and passed to the thread-per-pixel kernel as
// an argument of its own (after the others, so that every kernel keeps the parameter offsets it had without it):
// emit[i] = {x, y, z, block palette position} sorted by (x, y, z); the cell lists in CSR form, L(c) = list[off[c] .. off[c + 1]),
// cells of 1 << shift voxels, index (cx * dim.y + cy) * dim.z + cz over the cell box whose low voxel corner is g0.
// The wider table of CCU_RENDER_EMITTER_MODELS (DESIGN §12) also lists model emitters: mhead[b] is the int4 index in mprim of
// palette position b's emitting primitives, -1 when b is no model emitter; there mprim holds {m, bbox xmin, xmax, ymin},
// {ymax, zmin, zmax, 0} (float bits, block-local) and then m records of four int4 (model_prim_words).  The table of
// CCU_RENDER_EMITTER_SAMPLING alone leaves both null.
struct EmitView {
    const int4 *__restrict__ emit;
    const int *__restrict__ off;
    const int *__restrict__ list;
    int3 g0, dim;
    int shift;
    const int *__restrict__ mhead;
    const int4 *__restrict__ mprim;
};

// The biome colours of CCU_RENDER_BIOME_TINT (DESIGN §13), built at commit and passed to both render kernels as an argument of
// their own after the others: over the chunks' bounding box (gx x gz chunks from chunk (x0, z0)), grid[(cx - x0) * gz + cz - z0]
// is the tile of chunk (cx, cz) or -1; tiles holds per tile three planes of 256 texels {r, g, b, 0} in tint-type order
// (foliage, grass, water), texel (z & 15) * 16 + (x & 15).
struct BiomeView {
    const int *__restrict__ grid;
    const float4 *__restrict__ tiles;
    int x0, z0, gx, gz;
};
// The biome kernels copy their BiomeView here when they start, so that the material evaluation reaches it without one more
// argument on every function between the kernel and the block test.
__device__ __forceinline__ BiomeView &biome_smem() {
    __shared__ BiomeView b;
    return b;
}

// The cloud layer of CCU_RENDER_CLOUDS (DESIGN §15), set by ccu_scene_set_clouds and passed to both render kernels as an argument
// of their own after the others, like the emitter table and the biome colours.  mask: 256 x 256 bits, cell (i, k) at bit
// (k & 255) * 256 + (i & 255) (8 KiB, read through the read-only path); the box of a set cell is i <= x * inv + u0 <= i + 1,
// y0 <= y <= y1, k <= z * inv + v0 <= k + 1.
struct CloudView {
    const unsigned *__restrict__ mask;
    float inv, y0, y1, u0, v0;
};

// What a successful intersection writes into the IntersectionRecord (wavefront.h:37-78).  The specular kernels (SPEC, DESIGN
// "Beyond the reference: specular materials") also carry word 5 of the material the colour came from: specular, metalness and
// roughness bytes.  The other kernels keep the reference's record exactly.
template <bool SPEC = false>
struct SurfT {
    static constexpr bool has_spec = false;
    float3 normal;
    float4 color;
    float emittance;
};
template <>
struct SurfT<true> {
    static constexpr bool has_spec = true;
    float3 normal;
    float4 color;
    float emittance;
    uint32_t spec;
};
using Surf = SurfT<false>;
__device__ __forceinline__ void surf_set_spec(SurfT<false> &, uint32_t) {}
__device__ __forceinline__ void surf_set_spec(SurfT<true> &r, uint32_t w) { r.spec = w; }

template <bool SPEC = false>
struct RecordT {     // IntersectionRecord, wavefront.h:37-78
    float distance;
    int material;
    float3 point;
    SurfT<SPEC> surf;
};
using Record = RecordT<false>;

struct HitInfo {     // first-hit bookkeeping, not part of the reference's record
    int node;        // treeData index of the hit leaf (reference layout), -1 when unknown / BVH hit
    int kind;        // 0 miss, 1 octree, 2 world BVH, 3 actor BVH, 4 cloud (render kernels with CCU_RENDER_CLOUDS only)
    int bx, by, bz;  // voxel of the octree hit
};

// ------------------------------------------------------------------------------------------------------
// images
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 color_from_argb(uint32_t argb) {   // utils.h:6-14
    float4 c;
    c.w = (float)((argb >> 24) & 0xFF) / 256.0f;
    c.x = (float)((argb >> 16) & 0xFF) / 256.0f;
    c.y = (float)((argb >> 8) & 0xFF) / 256.0f;
    c.z = (float)(argb & 0xFF) / 256.0f;
    return c;
}
// Small read-only tables every kernel of this file stages in shared memory when it starts (stage_tables): the UNORM8 -> float
// table, and a pointer to the sky texels - the wavefront kernel copies the sky table itself into its dynamic shared memory
// (res^2 <= 16384 texels, 64 KiB) and points `sky` there, the thread-per-ray kernels leave it pointing at global memory.
struct SmemTables {
    float unorm[256];
    const uchar4 *sky;
};
__device__ __forceinline__ SmemTables &smem_tables() {
    __shared__ SmemTables t;
    return t;
}
// cooperative; ends with a barrier.  sky_smem: where the kernel staged the sky texels (nullptr: read them from global memory)
__device__ __forceinline__ void stage_tables(const DScene &s, const uchar4 *sky_smem) {
    SmemTables &t = smem_tables();
    for (int i = threadIdx.x; i < 256; i += blockDim.x) t.unorm[i] = __ldg(s.unorm + i);
    if (threadIdx.x == 0) t.sky = sky_smem ? sky_smem : s.sky;
    __syncthreads();
}
// The same without a block barrier, for the short thread-per-ray kernels: EVERY warp writes the whole table (all warps write the
// same values, so it does not matter whose store lands last) and only waits for its own lanes.
__device__ __forceinline__ void stage_tables_per_warp(const DScene &s) {
    SmemTables &t = smem_tables();
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int i = 0; i < 8; i++) t.unorm[i * 32 + lane] = __ldg(s.unorm + i * 32 + lane);
    if (lane == 0) t.sky = s.sky;
    __syncwarp();
}
// RGBA8 UNORM -> float: byte / 255.0f, read from a 256-entry table holding exactly those IEEE quotients
// (built once on the device by k_unorm_table), which replaces four divisions per texel by four shared-memory loads.
__device__ __forceinline__ float4 unorm8(const DScene &s, uchar4 t) {
    const float *u = smem_tables().unorm;
    return make_float4(u[t.x], u[t.y], u[t.z], u[t.w]);
}
// textureAtlas.h:10-16: nearest / clamp-to-edge / integer coordinates
__device__ __forceinline__ float4 atlas_read_xy(const DScene &s, int x, int y, int location) {
    x += ((location >> 22) & 0x1FF) * 16;
    y += ((location >> 13) & 0x1FF) * 16;
    int d = location & 0x7FFFF;
    x = min(max(x, 0), s.atlas_w - 1);
    y = min(max(y, 0), s.atlas_h - 1);
    d = min(max(d, 0), s.atlas_layers - 1);
    size_t tile = ((size_t)d * s.atlas_tiles_y + (y >> 4)) * s.atlas_tiles_x + (x >> 4);
    return unorm8(s, __ldg(s.atlas + tile * 256 + ((y & 15) << 4) + (x & 15)));
}
// textureAtlas.h:18-28
__device__ __forceinline__ float4 atlas_read_uv(const DScene &s, float u, float v, int location, int size) {
    int width = (size >> 16) & 0xFFFF;
    int height = size & 0xFFFF;
    v = 1.0f - v;
    int x = min(max(f2i((u - CCU_EPS) * (float)width), 0), width - 1);
    int y = min(max(f2i((v - CCU_EPS) * (float)height), 0), height - 1);
    return atlas_read_xy(s, x, y, location);
}
// sky.h:95 sampler semantics (OpenCL 1.2 s8.2: normalised, mirrored repeat, linear), fp32 weights
__device__ __forceinline__ void sky_axis(float s, int w, int &i0, int &i1, float &a) {
    float sp = 2.0f * rintf(0.5f * s);
    sp = fabsf(s - sp);
    float u = sp * (float)w;
    float um = u - 0.5f;
    float fl = floorf(um);
    int j0 = f2i(fl);
    int j1 = j0 + 1;
    a = um - fl;
    i0 = j0 < 0 ? 0 : j0;
    i1 = j1 > w - 1 ? w - 1 : j1;
}
__device__ __forceinline__ float4 sky_read(const DScene &s, float cs, float ct) {
    int w = s.sky_res, i0, i1, j0, j1;
    float a, b;
    sky_axis(cs, w, i0, i1, a);
    sky_axis(ct, w, j0, j1, b);
    const uchar4 *sky = smem_tables().sky;      // shared memory (wavefront kernel, table staged) or global memory
    float4 t00 = unorm8(s, sky[j0 * w + i0]);
    float4 t10 = unorm8(s, sky[j0 * w + i1]);
    float4 t01 = unorm8(s, sky[j1 * w + i0]);
    float4 t11 = unorm8(s, sky[j1 * w + i1]);
    float w00 = (1.0f - a) * (1.0f - b), w10 = a * (1.0f - b), w01 = (1.0f - a) * b, w11 = a * b;
    float4 r;
    r.x = ((w00 * t00.x + w10 * t10.x) + w01 * t01.x) + w11 * t11.x;
    r.y = ((w00 * t00.y + w10 * t10.y) + w01 * t01.y) + w11 * t11.y;
    r.z = ((w00 * t00.z + w10 * t10.z) + w01 * t01.z) + w11 * t11.z;
    r.w = ((w00 * t00.w + w10 * t10.w) + w01 * t01.w) + w11 * t11.w;
    return r;
}

// ------------------------------------------------------------------------------------------------------
// material.h:31-82
// ------------------------------------------------------------------------------------------------------
// CCU_RENDER_BIOME_TINT: the biome colour of tint type tt (1..3) at voxel column (bx, bz), with w = 255 / 256 (the alpha of the
// fixed tints); false where the chunk has no tile.
__device__ __forceinline__ bool biome_color(uint32_t tt, int bx, int bz, float4 &c) {
    const BiomeView &b = biome_smem();
    const int cx = (bx >> 4) - b.x0, cz = (bz >> 4) - b.z0;
    if (cx < 0 || cz < 0 || cx >= b.gx || cz >= b.gz) return false;
    const int tile = __ldg(b.grid + (size_t)cx * b.gz + cz);
    if (tile < 0) return false;
    c = __ldg(b.tiles + ((size_t)tile * 3 + (tt - 1)) * 256 + ((bz & 15) << 4) + (bx & 15));
    c.w = 255.0f / 256.0f;
    return true;
}

// the material words {flags, tint, texSize, texLocation / ARGB, emittance} evaluated at (u, v).  BIOME: the surface belongs to
// octree voxel column (bx, bz), whose biome colour replaces the fixed tints of tint types 1-3 (DESIGN §13).
struct MatOut { float4 color; float emittance; int ok; };
template <bool BIOME = false>
__device__ __forceinline__ MatOut material_eval_core(const DScene &s, uint32_t flags, uint32_t tint, uint32_t tex_size, uint32_t col, uint32_t normal_emittance,
                                                     float u, float v, int bx = 0, int bz = 0) {
    MatOut out;
    out.emittance = 0.0f;
    out.ok = 0;
    float4 color;
    if (flags & 4u) color = atlas_read_uv(s, u, v, (int)col, (int)tex_size);
    else color = color_from_argb(col);
    out.color = color;
    if (!(color.w > CCU_EPS)) return out;
    uint32_t tt = tint >> 24;
    if (tt == 0xFF || (tt >= 1 && tt <= 3)) {
        if constexpr (BIOME) {
            float4 t;
            if (tt == 0xFF || !biome_color(tt, bx, bz, t))
                t = color_from_argb(tt == 0xFF ? tint : (tt == 1 ? 0xFF71A74Du : (tt == 2 ? 0xFF8EB971u : 0xFF3F76E4u)));
            out.color.x *= t.x; out.color.y *= t.y; out.color.z *= t.z; out.color.w *= t.w;
        } else {   // the code before the flag, unchanged: the other kernels compile to the same instructions (DESIGN §13)
            uint32_t argb = tt == 0xFF ? tint : (tt == 1 ? 0xFF71A74Du : (tt == 2 ? 0xFF8EB971u : 0xFF3F76E4u));
            float4 t = color_from_argb(argb);
            out.color.x *= t.x; out.color.y *= t.y; out.color.z *= t.z; out.color.w *= t.w;
        }
    }
    if (flags & 2u) out.emittance = atlas_read_uv(s, u, v, (int)normal_emittance, (int)tex_size).w;
    // material.h:79 divides by the double literal 255.0: (float)((double)b / 255.0) == (float)b / 255.0f for all 256 byte values
    // (checked exhaustively, tests/test_oracle_kat.py), i.e. the UNORM table entry - no fp64 division on the device
    else out.emittance = smem_tables().unorm[normal_emittance & 0xFF];
    out.ok = 1;
    return out;
}
// rec.color / rec.emittance (and rec.spec) are written only on success (material.h:50-54 rejects before storing)
template <bool BIOME, class Surface>
__device__ __forceinline__ bool material_eval(const DScene &s, uint32_t flags, uint32_t tint, uint32_t tex_size, uint32_t col, uint32_t normal_emittance,
                                              uint32_t spec, Surface &rec, float u, float v, int bx = 0, int bz = 0) {
    const MatOut m = material_eval_core<BIOME>(s, flags, tint, tex_size, col, normal_emittance, u, v, bx, bz);
    if (!m.ok) return false;
    rec.color = m.color;
    rec.emittance = m.emittance;
    surf_set_spec(rec, spec);
    return true;
}
// Material_get + Material_sample for material pointer `material` (an int offset into matPalette, 6 words per material):
// two 16-byte loads from the commit-time records, or the reference's own array for a pointer that is not on a record
template <bool BIOME = false, class Surface>
__device__ __forceinline__ bool material_sample(const DScene &s, int material, Surface &rec, float u, float v, int bx = 0, int bz = 0) {
    const int idx = material / 6;
    if (material >= 0 && idx * 6 == material) {
        const int4 a = __ldg(s.mat_rec + 2 * idx), b = __ldg(s.mat_rec + 2 * idx + 1);
        return material_eval<BIOME>(s, (uint32_t)a.x, (uint32_t)a.y, (uint32_t)a.z, (uint32_t)a.w, (uint32_t)b.x, (uint32_t)b.y, rec, u, v, bx, bz);
    }
    const int *m = s.mat_palette + material;
    return material_eval<BIOME>(s, __ldg(m), __ldg(m + 1), __ldg(m + 2), __ldg(m + 3), __ldg(m + 4), Surface::has_spec ? (uint32_t)__ldg(m + 5) : 0u,
                                rec, u, v, bx, bz);
}

// ------------------------------------------------------------------------------------------------------
// primitives.h
// ------------------------------------------------------------------------------------------------------
struct Box { float xmin, xmax, ymin, ymax, zmin, zmax; };

// primitives.h:30-48
__device__ __forceinline__ float box_entry(const Box &b, float3 o, float3 inv) {
    float t1x = (b.xmin - o.x) * inv.x, t1y = (b.ymin - o.y) * inv.y, t1z = (b.zmin - o.z) * inv.z;
    float t2x = (b.xmax - o.x) * inv.x, t2y = (b.ymax - o.y) * inv.y, t2z = (b.zmax - o.z) * inv.z;
    float tmin = fmaxf(fminf(t1x, t2x), fmaxf(fminf(t1y, t2y), fminf(t1z, t2z)));
    float tmax = fminf(fmaxf(t1x, t2x), fminf(fmaxf(t1y, t2y), fmaxf(t1z, t2z)));
    return (tmax < tmin) ? nanf_() : tmin;
}
// primitives.h:52-61
__device__ __forceinline__ float box_exit(const Box &b, float3 o, float3 inv) {
    float t1x = (b.xmin - o.x) * inv.x, t1y = (b.ymin - o.y) * inv.y, t1z = (b.zmin - o.z) * inv.z;
    float t2x = (b.xmax - o.x) * inv.x, t2y = (b.ymax - o.y) * inv.y, t2z = (b.zmax - o.z) * inv.z;
    return fminf(fmaxf(t1x, t2x), fminf(fmaxf(t1y, t2y), fmaxf(t1z, t2z)));
}
// primitives.h:66-112 (MAP2 = false) / :117-162 (MAP2 = true); later face matches overwrite earlier ones
template <bool MAP2>
__device__ __forceinline__ float box_full(const Box &b, float3 origin, float3 dir, float3 inv, float3 &normal, float &u, float &v) {
    float t1x = (b.xmin - origin.x) * inv.x, t1y = (b.ymin - origin.y) * inv.y, t1z = (b.zmin - origin.z) * inv.z;
    float t2x = (b.xmax - origin.x) * inv.x, t2y = (b.ymax - origin.y) * inv.y, t2z = (b.zmax - origin.z) * inv.z;
    float tmin = fmaxf(fminf(t1x, t2x), fmaxf(fminf(t1y, t2y), fminf(t1z, t2z)));
    float tmax = fminf(fmaxf(t1x, t2x), fminf(fmaxf(t1y, t2y), fmaxf(t1z, t2z)));
    if (tmax < tmin) return nanf_();
    float3 o = origin + dir * tmin;
    if (!MAP2) {
        float dx = 1.0f / (b.xmax - b.xmin), dy = 1.0f / (b.ymax - b.ymin), dz = 1.0f / (b.zmax - b.zmin);
        if (t1x == tmin) { u = 1.0f - (o.z - b.zmin) * dz; v = (o.y - b.ymin) * dy; normal = f3(-1, 0, 0); }
        if (t2x == tmin) { u = (o.z - b.zmin) * dz; v = (o.y - b.ymin) * dy; normal = f3(1, 0, 0); }
        if (t1y == tmin) { u = (o.x - b.xmin) * dx; v = 1.0f - (o.z - b.zmin) * dz; normal = f3(0, -1, 0); }
        if (t2y == tmin) { u = (o.x - b.xmin) * dx; v = (o.z - b.zmin) * dz; normal = f3(0, 1, 0); }
        if (t1z == tmin) { u = (o.x - b.xmin) * dx; v = (o.y - b.ymin) * dy; normal = f3(0, 0, -1); }
        if (t2z == tmin) { u = 1.0f - (o.x - b.xmin) * dx; v = (o.y - b.ymin) * dy; normal = f3(0, 0, 1); }
    } else {
        if (t1x == tmin) { u = o.z; v = o.y; normal = f3(-1, 0, 0); }
        if (t2x == tmin) { u = 1.0f - o.z; v = o.y; normal = f3(1, 0, 0); }
        if (t1y == tmin) { u = o.x; v = o.z; normal = f3(0, -1, 0); }
        if (t2y == tmin) { u = o.x; v = 1.0f - o.z; normal = f3(0, 1, 0); }
        if (t1z == tmin) { u = 1.0f - o.x; v = o.y; normal = f3(0, 0, -1); }
        if (t2z == tmin) { u = o.x; v = o.y; normal = f3(0, 0, 1); }
    }
    return tmin;
}

// primitives.h:200-260.  +z face: the reference reads an uninitialised material (SURVEY Q10); defined as 0 / flags 0.
// w[0..12]: the box's 13 words (PackedAabb.java:75-102)
__device__ __forceinline__ float textured_box(const int *w, float distance, float3 origin, float3 dir, float3 inv,
                                              float3 &normal, float &u, float &v, int &material) {
    Box b = {i2f(w[0]), i2f(w[1]), i2f(w[2]), i2f(w[3]), i2f(w[4]), i2f(w[5])};
    float3 n = f3(0, 0, 0);
    float tu = 0, tv = 0;
    float dist = box_full<true>(b, origin, dir, inv, n, tu, tv);
    if (dist >= distance || dist < -CCU_EPS) return nanf_();
    if (is_nan(dist)) return nanf_();
    int bflags = w[6];
    int slot = -1, flags = 0;
    if (n.z == -1.0f) { slot = 7; flags = bflags; }
    if (n.x == 1.0f) { slot = 8; flags = bflags >> 4; }
    if (n.z == -1.0f) { slot = 9; flags = bflags >> 8; }
    if (n.x == -1.0f) { slot = 10; flags = bflags >> 12; }
    if (n.y == 1.0f) { slot = 11; flags = bflags >> 16; }
    if (n.y == -1.0f) { slot = 12; flags = bflags >> 20; }
    if (flags & 8) return nanf_();
    if (flags & 4) tu = 1.0f - tu;
    if (flags & 2) tv = 1.0f - tv;
    if (flags & 1) { float t = tu; tu = tv; tv = t; }
    material = 0;
#pragma unroll
    for (int k = 7; k < 13; k++) if (slot == k) material = w[k];
    normal = n; u = tu; v = tv;
    return dist;
}

// primitives.h:274-319
// q[0..12]: the quad's first 13 words (PackedQuad.java:41-66)
__device__ __forceinline__ float quad_hit(const int *q, float distance, float3 origin, float3 dir, float3 &normal, float &u, float &v) {
    float3 qo = f3(i2f(q[0]), i2f(q[1]), i2f(q[2]));
    float3 xv = f3(i2f(q[3]), i2f(q[4]), i2f(q[5]));
    float3 yv = f3(i2f(q[6]), i2f(q[7]), i2f(q[8]));
    float3 n = normalize3(cross3(xv, yv));
    float denom = dot3(dir, n);
    if (denom < -CCU_EPS) {
        float t = -(dot3(origin, n) - dot3(n, qo)) / denom;
        if (t > -CCU_EPS && t < distance) {
            float3 pt = (origin + dir * t) - qo;
            float uu = dot3(pt, xv) / dot3(xv, xv);
            float vv = dot3(pt, yv) / dot3(yv, yv);
            if (uu >= 0 && uu <= 1 && vv >= 0 && vv <= 1) {
                u = i2f(q[9]) + (uu * i2f(q[10]));
                v = i2f(q[11]) + (vv * i2f(q[12]));
                normal = n;
                return t;
            }
        }
    }
    return nanf_();
}

// primitives.h:335-409 (Moeller-Trumbore on pre-stored edges)
__device__ __forceinline__ float triangle_hit(const int *t, float distance, float3 origin, float3 dir, float3 &normal,
                                              float &ou, float &ov, int &material) {
    int flags = __ldg(t);
    float3 e1 = f3(i2f(__ldg(t + 1)), i2f(__ldg(t + 2)), i2f(__ldg(t + 3)));
    float3 e2 = f3(i2f(__ldg(t + 4)), i2f(__ldg(t + 5)), i2f(__ldg(t + 6)));
    float3 pvec = cross3(dir, e2);
    float det = dot3(e1, pvec);
    if ((flags >> 8) & 1) {
        if (det > -CCU_EPS && det < CCU_EPS) return nanf_();
    } else if (det > -CCU_EPS) {
        return nanf_();
    }
    float recip = 1.0f / det;
    float3 o = f3(i2f(__ldg(t + 7)), i2f(__ldg(t + 8)), i2f(__ldg(t + 9)));
    float3 tvec = origin - o;
    float u = dot3(tvec, pvec) * recip;
    if (u < 0 || u > 1) return nanf_();
    float3 qvec = cross3(tvec, e1);
    float v = dot3(dir, qvec) * recip;
    if (v < 0 || (u + v) > 1) return nanf_();
    float tt = dot3(e2, qvec) * recip;
    if (tt > CCU_EPS && tt < distance) {
        float w = 1.0f - u - v;
        ou = (i2f(__ldg(t + 13)) * u + i2f(__ldg(t + 15)) * v) + i2f(__ldg(t + 17)) * w;
        ov = (i2f(__ldg(t + 14)) * u + i2f(__ldg(t + 16)) * v) + i2f(__ldg(t + 18)) * w;
        normal = f3(i2f(__ldg(t + 10)), i2f(__ldg(t + 11)), i2f(__ldg(t + 12)));
        material = __ldg(t + 19);
        return tt;
    }
    return nanf_();
}

// ------------------------------------------------------------------------------------------------------
// block.h:30-118
// ------------------------------------------------------------------------------------------------------
template <bool SPEC>
struct ModelHit {    // returned by value so that callers keep their state in registers
    float dist;      // NaN = no hit
    SurfT<SPEC> surf;
};

// block.h:66-116: AABB models (type 2) and quad models (type 3).  Cold path, kept out of line (intersect_model_block).
template <bool BIOME, class Hit>
__device__ __forceinline__ Hit model_block_hit(const DScene &s, int model_type, int model_ptr, float3 norm_origin, float3 direction, float3 inv,
                                               int bx, int bz) {
    Hit out;
    out.surf.normal = f3(0, 0, 0);
    out.surf.color = make_float4(0, 0, 0, 0);
    out.surf.emittance = 0;
    surf_set_spec(out.surf, 0u);
    float3 normal = f3(0, 0, 0);
    float u = 0, v = 0;
    bool hit = false;
    float dist = inff_();
    // model_ptr: offset into the 16-byte record arrays built at commit, in units of 16 bytes
    int w[16];
    if (model_type == 2) {
        const int boxes = __ldg(s.aabb_rec + model_ptr).x;
        for (int i = 0; i < boxes; i++) {
            const int4 *r = s.aabb_rec + model_ptr + 1 + 4 * i;
#pragma unroll
            for (int k = 0; k < 4; k++) { const int4 t = __ldg(r + k); w[4 * k] = t.x; w[4 * k + 1] = t.y; w[4 * k + 2] = t.z; w[4 * k + 3] = t.w; }
            int material = 0;
            float t = textured_box(w, dist, norm_origin, direction, inv, normal, u, v, material);
            if (!is_nan(t) && material_sample<BIOME>(s, material, out.surf, u, v, bx, bz)) { out.surf.normal = normal; dist = t; hit = true; }
        }
    } else {
        const int quads = __ldg(s.quad_rec + model_ptr).x;
        for (int i = 0; i < quads; i++) {
            const int4 *r = s.quad_rec + model_ptr + 1 + 4 * i;
#pragma unroll
            for (int k = 0; k < 4; k++) { const int4 t = __ldg(r + k); w[4 * k] = t.x; w[4 * k + 1] = t.y; w[4 * k + 2] = t.z; w[4 * k + 3] = t.w; }
            float t = quad_hit(w, dist, norm_origin, direction, normal, u, v);
            if (!is_nan(t) && material_sample<BIOME>(s, w[13], out.surf, u, v, bx, bz)) { out.surf.normal = normal; dist = t; hit = true; }
        }
    }
    out.dist = hit ? dist : nanf_();
    return out;
}
template <bool SPEC>
static __device__ __noinline__ ModelHit<SPEC> intersect_model_block(const DScene &s, int model_type, int model_ptr, float3 norm_origin,
                                                       float3 direction, float3 inv) {
    return model_block_hit<false, ModelHit<SPEC>>(s, model_type, model_ptr, norm_origin, direction, inv, 0, 0);
}
// the same for the biome kernels: (bx, bz) is the model's voxel column
template <bool SPEC>
static __device__ __noinline__ ModelHit<SPEC> intersect_model_block_biome(const DScene &s, int model_type, int model_ptr, float3 norm_origin,
                                                             float3 direction, float3 inv, int bx, int bz) {
    return model_block_hit<true, ModelHit<SPEC>>(s, model_type, model_ptr, norm_origin, direction, inv, bx, bz);
}

// Returns the hit distance relative to the marched position (NaN = miss) and fills `surf` on a hit.
// (The reference also overwrites record.normal when a full block fails its alpha test, block.h:59-60; that
// value is never read before the next successful hit overwrites it, so it is not reproduced.)
// BIOME: the biome colours of voxel column (bx, bz) tint the surface (DESIGN §13).
template <bool BIOME, class Surface>
__device__ __forceinline__ float intersect_block(const DScene &s, int block, int bx, int by, int bz, Surface &surf, float3 pos,
                                                 float3 direction, float3 inv) {
    if (block == CCU_ANY_TYPE) return nanf_();
    if (block < 0 || block + 1 >= s.block_palette_len) return nanf_();   // out-of-palette leaf (undefined in the reference)
    const int4 r0 = __ldg(s.block_rec + 2 * block);
    const int model_type = r0.x, model_ptr = r0.y;
    float3 norm_origin = (pos - direction * CCU_OFFSET) - f3((float)bx, (float)by, (float)bz);
    if (model_type == 1) {
        Box unit = {0, 1, 0, 1, 0, 1};
        float3 normal = f3(0, 0, 0);
        float u = 0, v = 0;
        // the marched position stands in for the direction here, as in block.h:52 (SURVEY Q2)
        float dist = box_full<false>(unit, norm_origin, pos, inv, normal, u, v);
        if (is_nan(dist)) return nanf_();
        Surf tmp;
        // the full cube's material travels with its palette entry
        const int4 r1 = __ldg(s.block_rec + 2 * block + 1);
        if (!material_eval<BIOME>(s, (uint32_t)r0.z, (uint32_t)r0.w, (uint32_t)r1.x, (uint32_t)r1.y, (uint32_t)r1.z, 0u, tmp, u, v, bx, bz))
            return nanf_();
        surf.color = tmp.color;
        surf.emittance = tmp.emittance;
        surf_set_spec(surf, (uint32_t)r1.w);
        surf.normal = normal;
        return dist - CCU_OFFSET;
    }
    if (model_type == 2 || model_type == 3) {
        const auto m = BIOME ? intersect_model_block_biome<Surface::has_spec>(s, model_type, model_ptr, norm_origin, direction, inv, bx, bz)
                             : intersect_model_block<Surface::has_spec>(s, model_type, model_ptr, norm_origin, direction, inv);
        if (is_nan(m.dist)) return nanf_();
        surf = m.surf;
        return m.dist;
    }
    return nanf_();
}

// ------------------------------------------------------------------------------------------------------
// octree.h:41-109.  find_leaf returns what the reference's root descent (octree.h:81-88) returns for the
// voxel (bx,by,bz): the leaf word, the leaf level and the leaf's index in treeData.
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int find_leaf(const DScene &s, int bx, int by, int bz, int &level, int &node) {
    int lvl = s.depth;
    int idx = 0;
    int data = __ldg(s.tree);
    while (data > 0) {
        lvl--;
        idx = data + ((((bx >> lvl) & 1) << 2) | (((by >> lvl) & 1) << 1) | ((bz >> lvl) & 1));
        data = __ldg(s.tree + idx);
    }
    level = lvl;
    node = idx;
    return -data;
}

#define CCU_WIDE_LEAF 0x80000000u
#define CCU_WIDE_ANY 0x3FFFFFFu
// Same answer as find_leaf (leaf value and level) from the commit-time layout: one table lookup plus one load per
// two octree levels below the table's cell level.
__device__ __forceinline__ int find_leaf_wide(const DScene &s, int bx, int by, int bz, int &level) {
    const int cl = s.cell_level;
    unsigned e = __ldg(s.top + ((((bx >> cl) << s.top_log2) + (by >> cl)) << s.top_log2) + (bz >> cl));
    int lvl = cl;
    while (!(e & CCU_WIDE_LEAF)) {
        lvl -= 2;
        e = __ldg(s.wide + (size_t)e * 64 + ((((bx >> lvl) & 3) << 4) | (((by >> lvl) & 3) << 2) | ((bz >> lvl) & 3)));
    }
    level = (e >> 26) & 31;
    unsigned v = e & CCU_WIDE_ANY;
    return v == CCU_WIDE_ANY ? CCU_ANY_TYPE : (int)v;
}

// One ray being marched through the octree (the loop state of octree.h:66-107).
struct March {
    float3 o, d, inv;
    float t;        // distMarch
    float limit;    // record->distance on entry: +inf for path segments, the surface hit distance for shadow rays
    int steps;
};

// octree.h:43-64: 1 / d, the distance to the octree cube for a ray that starts outside of it, and whether it enters at all.
// Kept out of line (one copy instead of one per ray kind: measured -4 % on the wavefront kernel, whose shading stages are
// limited by instruction fetch); the result is returned by value, so the copy hands it back in registers.
// inv is NaN on an axis whose origin component is NaN.  Every use of inv multiplies it by a coordinate difference that is
// NaN on that axis anyway (the box tests, AABB_exit, the block test), so no result changes; lean_prepare, which sees inv
// but not the origin, needs it to give that axis the NaN exit operand (ccu_march.cuh, lean_exit_axis).
struct MarchStart { float3 inv; float t; int entered; };
static __device__ __noinline__ MarchStart march_begin_core(int depth, float3 origin, float3 direction) {
    MarchStart ms;
    ms.inv = f3(origin.x == origin.x ? 1.0f / direction.x : nanf_(), origin.y == origin.y ? 1.0f / direction.y : nanf_(),
                origin.z == origin.z ? 1.0f / direction.z : nanf_());
    ms.t = 0;
    ms.entered = 1;
    int lx = f2i(floorf(origin.x)) >> depth, ly = f2i(floorf(origin.y)) >> depth, lz = f2i(floorf(origin.z)) >> depth;
    if ((lx | ly | lz) != 0) {
        float size = (float)(1 << depth);
        Box cube = {0, size, 0, size, 0, size};
        float dist = box_entry(cube, origin, ms.inv);
        if (is_nan(dist) || dist < 0) ms.entered = 0;
        else ms.t += dist + CCU_OFFSET;
    }
    return ms;
}
// returns false when the ray starts outside the octree cube and never enters it
__device__ __forceinline__ bool march_begin(const DScene &s, March &m, float3 origin, float3 direction, float limit) {
    const MarchStart ms = march_begin_core(s.depth, origin, direction);
    m.o = origin;
    m.d = direction;
    m.inv = ms.inv;
    m.t = ms.t;
    m.limit = limit;
    m.steps = 0;
    return ms.entered != 0;
}

// The voxel the ray is in after marching m.t (octree.h:72-78): position, offset position and block coordinates.
struct Cell {
    float3 pos, q;
    int bx, by, bz;
};
__device__ __forceinline__ Cell march_cell(const March &m) {
    Cell c;
    c.pos = m.o + m.d * m.t;
    c.q = c.pos + m.d * CCU_OFFSET;
    c.bx = f2i(floorf(c.q.x)); c.by = f2i(floorf(c.q.y)); c.bz = f2i(floorf(c.q.z));
    return c;
}
// octree.h:102-106: leave the leaf cube (level `level`) that contains the cell
__device__ __forceinline__ void march_exit(March &m, const Cell &c, int level) {
    int lx = c.bx >> level, ly = c.by >> level, lz = c.bz >> level;
    Box leaf = {(float)(lx << level), (float)((lx + 1) << level), (float)(ly << level), (float)((ly + 1) << level),
                (float)(lz << level), (float)((lz + 1) << level)};
    m.t += box_exit(leaf, c.q, m.inv) + CCU_OFFSET;
    m.steps++;
}
// Block test of the non-air leaf under the ray (octree.h:92-106).  Returns true on a hit (surf / hit_t filled);
// otherwise the ray has been advanced past the leaf.
// CUT (kernels built with CCU_RENDER_EMITTER_MODELS) and `cut` (the ray is an emitter sample's shadow ray): the hit counts only
// when it lies before the ray's limit, so that a model's own voxel does not occlude the primitive sampled inside it (DESIGN §12).
template <class V, bool CUT = false>
__device__ __forceinline__ bool march_block(const DScene &s, March &m, int data, int level, SurfT<V::spec> &surf, float &hit_t, bool cut = false) {
    Cell c = march_cell(m);
    float dist = intersect_block<V::biome>(s, data, c.bx, c.by, c.bz, surf, c.pos, m.d, m.inv);
    if (!is_nan(dist) && !(CUT && cut && !(m.t + dist < m.limit))) {
        hit_t = m.t + dist;
        return true;
    }
    march_exit(m, c, level);
    return false;
}

// One whole iteration of octree.h:66-107 on the reference's own node array (root descent per step).
// Returns 0 = keep marching, 1 = hit (hit_t / surf / block / node filled), 2 = ray left.
template <class V, bool CUT = false>
__device__ __forceinline__ int march_step_ref(const DScene &s, March &m, SurfT<V::spec> &surf, float &hit_t, int &hit_block, int &hit_node, Cell &hit_cell) {
    if (m.steps >= s.draw_depth || m.t > m.limit) return 2;
    const int depth = s.depth;
    const Cell c = march_cell(m);
    if (((c.bx >> depth) | (c.by >> depth) | (c.bz >> depth)) != 0) return 2;
    int level, node;
    const int data = find_leaf(s, c.bx, c.by, c.bz, level, node);
    if (data == 0) {           // ray->material is always 0 (wavefront.h:34, SURVEY Q3)
        march_exit(m, c, level);
        return 0;
    }
    if (march_block<V, CUT>(s, m, data, level, surf, hit_t, CUT)) {
        hit_block = data;
        hit_node = node;
        hit_cell = c;
        return 1;
    }
    return 0;
}

template <class V, bool CUT = false>
__device__ __forceinline__ bool octree_intersect_ref(const DScene &s, float3 origin, float3 direction, RecordT<V::spec> &rec, HitInfo &hi) {
    March m;
    if (!march_begin(s, m, origin, direction, rec.distance)) return false;
    for (;;) {
        float t;
        int block, node;
        Cell cell;
        int r = march_step_ref<V, CUT>(s, m, rec.surf, t, block, node, cell);
        if (r == 1) {
            rec.distance = t;
            rec.material = block;
            hi.node = node;
            hi.kind = 1;
            hi.bx = cell.bx; hi.by = cell.by; hi.bz = cell.bz;
            return true;
        }
        if (r == 2) return false;
    }
}

// ------------------------------------------------------------------------------------------------------
// bvh.h:22-113
// ------------------------------------------------------------------------------------------------------
template <bool SPEC>
struct BvhHit {
    float dist;      // NaN = no hit closer than `limit`
    SurfT<SPEC> surf;
};

template <bool SPEC>
static __device__ __noinline__ BvhHit<SPEC> bvh_intersect(const DScene &s, const int *__restrict__ bvh, float3 origin, float3 direction, float limit) {
    BvhHit<SPEC> out;
    out.dist = nanf_();
    out.surf.normal = f3(0, 0, 0);
    out.surf.color = make_float4(0, 0, 0, 0);
    out.surf.emittance = 0;
    surf_set_spec(out.surf, 0u);
    float distance = limit;
    int to_visit = 0, current = 0;
    int stack[64];
    float3 inv = f3(1.0f / direction.x, 1.0f / direction.y, 1.0f / direction.z);
    for (;;) {
        int head = __ldg(bvh + current);
        if (head <= 0) {
            int prim = -head;
            int num = __ldg(s.trigs + prim);
            for (int i = 0; i < num; i++) {
                float3 normal;
                float u, v;
                int material;
                float dist = triangle_hit(s.trigs + prim + 1 + 20 * i, distance, origin, direction, normal, u, v, material);
                if (!is_nan(dist) && material_sample(s, material, out.surf, u, v)) {
                    out.surf.normal = normal;      // record.material keeps its octree value (bvh.h:59-65, SURVEY Q15)
                    distance = dist;
                    out.dist = dist;
                }
            }
            if (to_visit == 0) break;
            current = stack[--to_visit];
        } else {
            int second = head;
            const int *n1 = bvh + current + 7;
            const int *n2 = bvh + second;
            Box b1 = {i2f(__ldg(n1 + 1)), i2f(__ldg(n1 + 2)), i2f(__ldg(n1 + 3)), i2f(__ldg(n1 + 4)), i2f(__ldg(n1 + 5)), i2f(__ldg(n1 + 6))};
            Box b2 = {i2f(__ldg(n2 + 1)), i2f(__ldg(n2 + 2)), i2f(__ldg(n2 + 3)), i2f(__ldg(n2 + 4)), i2f(__ldg(n2 + 5)), i2f(__ldg(n2 + 6))};
            float t1 = box_entry(b1, origin, inv);
            float t2 = box_entry(b2, origin, inv);
            bool miss1 = is_nan(t1) || t1 > distance;
            bool miss2 = is_nan(t2) || t2 > distance;
            if (miss1) {
                if (miss2) {
                    if (to_visit == 0) break;
                    current = stack[--to_visit];
                } else {
                    current = second;
                }
            } else if (miss2) {
                current += 7;
            } else if (t1 < t2) {
                stack[to_visit++] = second;
                current += 7;
            } else {
                stack[to_visit++] = current + 7;
                current = second;
            }
        }
    }
    return out;
}

// The two BVH probes of kernel.h:17-18 applied to a record whose octree part is already resolved.
template <bool SPEC>
__device__ __forceinline__ bool bvh_pair(const DScene &s, float3 origin, float3 direction, float &distance, SurfT<SPEC> &surf, int &kind) {
    bool hit = false;
    if (!s.world_bvh_empty) {
        BvhHit<SPEC> h = bvh_intersect<SPEC>(s, s.world_bvh, origin, direction, distance);
        if (!is_nan(h.dist)) { distance = h.dist; surf = h.surf; hit = true; kind = 2; }
    }
    if (!s.actor_bvh_empty) {
        BvhHit<SPEC> h = bvh_intersect<SPEC>(s, s.actor_bvh, origin, direction, distance);
        if (!is_nan(h.dist)) { distance = h.dist; surf = h.surf; hit = true; kind = 3; }
    }
    return hit;
}

// kernel.h:14-24 on the reference's own node array
template <class V, bool CUT = false>
__device__ __forceinline__ bool closest_intersect_ref(const DScene &s, float3 origin, float3 direction, RecordT<V::spec> &rec, HitInfo &hi) {
    bool hit = octree_intersect_ref<V, CUT>(s, origin, direction, rec, hi);
    int kind = 0;
    if (bvh_pair(s, origin, direction, rec.distance, rec.surf, kind)) {
        hit = true;
        hi.kind = kind;
        hi.node = -1;
    }
    if (hit) rec.point = origin + direction * (rec.distance - CCU_OFFSET);
    return hit;
}

// ------------------------------------------------------------------------------------------------------
// sky.h / kernel.h shading
// ------------------------------------------------------------------------------------------------------
// sky.h:97-106 + sky.h:42-66: radiance seen along a ray that left the scene (sky texel x intensity + sun disc)
__device__ __forceinline__ float3 sky_radiance(const DScene &s, float3 d) {
    float theta = dm_atan2(d.z, d.x);
    theta /= CCU_PI_F * 2;
    // fmod(x, 1) == x - trunc(x) exactly for every float (inf -> NaN, NaN -> NaN): sky.h:100 without the libm loop
    theta = theta - truncf(theta);
    theta = theta + 1.0f;
    theta = theta - truncf(theta);
    float phi = (dm_asin(fminf(fmaxf(d.y, -1.0f), 1.0f)) + CCU_PI_2_F) * CCU_INV_PI_F;
    float4 sky = sky_read(s, theta, phi);
    float3 col = f3(sky.x * s.sky_intensity, sky.y * s.sky_intensity, sky.z * s.sky_intensity);
    if ((s.sun_flags & 1) && !(dot3(d, s.sw) < 0.5f)) {
        const float radius = 0.03f;
        const float width = radius * 4;
        const float width2 = width * 2;
        float a = CCU_PI_2_F - dm_acos(dot3(d, s.su)) + width;
        if (a >= 0 && a < width2) {
            float b = CCU_PI_2_F - dm_acos(dot3(d, s.sv)) + width;
            if (b >= 0 && b < width2) {
                float4 sc = atlas_read_uv(s, a / width2, b / width2, s.sun_tex, s.sun_tex_size);
                col.x += sc.x * s.sun_intensity;
                col.y += sc.y * s.sun_intensity;
                col.z += sc.z * s.sun_intensity;
            }
        }
    }
    return col;
}

// camera.h:8-32 + rayTracer.cl:55-91 (NORMALIZE = preview variant, rayTracer.cl:186)
// (px, py): the pixel's column / row, gid = py * width + px (callers that already know them spare the division)
template <bool NORMALIZE>
__device__ __forceinline__ void camera_ray_xy(const DScene &s, int gid, int px, int py, uint32_t &rng, float3 &origin, float3 &direction) {
    if (s.projector_type != -1) {
        // half_width = (float)(W / (2.0 * H)), inv_height = (float)(1.0 / H): the double expressions of
        // rayTracer.cl:66-67, evaluated once on the host (IEEE doubles, identical on any machine)
        const float half_width = s.half_width, inv_height = s.inv_height;
        float x = -half_width + ((float)px + rng_float(rng)) * inv_height;
        float y = (float)(-0.5 + (double)(((float)py + rng_float(rng)) * inv_height));
        float3 o = f3(0, 0, 0), d = f3(0, 0, 1);
        if (s.projector_type == 0) {
            float aperture = s.cam[12], subject_distance = s.cam[13], fov_tan = s.cam[14];
            d = f3(fov_tan * x, fov_tan * y, 1.0f);
            if (aperture > 0) {
                d = d * (subject_distance / d.z);
                float r = sqrtf(rng_float(rng)) * aperture;
                float theta = rng_float(rng) * CCU_PI_F * 2.0f;
                float sn, cs;
                dm_sincos(theta, sn, cs);
                float rx = cs * r, ry = sn * r;
                d = d - f3(rx, ry, 0);
                o = o + f3(rx, ry, 0);
            }
        }
        if (NORMALIZE) d = normalize3(d);
        float3 m1 = f3(s.cam[3], s.cam[4], s.cam[5]), m2 = f3(s.cam[6], s.cam[7], s.cam[8]), m3 = f3(s.cam[9], s.cam[10], s.cam[11]);
        direction = f3(dot3(m1, d), dot3(m2, d), dot3(m3, d));
        origin = f3(dot3(m1, o), dot3(m2, o), dot3(m3, o)) + f3(s.cam[0], s.cam[1], s.cam[2]);
    } else {
        const float *r = s.rays + (size_t)gid * 6;
        origin = f3(__ldg(r), __ldg(r + 1), __ldg(r + 2));
        direction = f3(__ldg(r + 3), __ldg(r + 4), __ldg(r + 5));
    }
}

template <bool NORMALIZE>
__device__ __forceinline__ void camera_ray(const DScene &s, int gid, uint32_t &rng, float3 &origin, float3 &direction) {
    const int py = gid / s.width;
    camera_ray_xy<NORMALIZE>(s, gid, gid - py * s.width, py, rng, origin, direction);
}

// sky.h:68-93: direction towards the sun disc; x1, x2 are the two RNG draws (component-wise product u*v, SURVEY Q5).
// Both direction samplers turn x2 into the same angle 2 pi x2; the *_sc forms take its sine / cosine so that a caller that needs
// either one (the wavefront kernel's shading step) evaluates dm_sincos once for all its lanes.
__device__ __forceinline__ float3 sun_sample_direction_sc(const DScene &s, float x1, float sn, float cs) {
    float cos_a = 1 - x1 + x1 * s.sun_radius_cos;
    float sin_a = sqrtf(1 - cos_a * cos_a);
    float3 u = s.su * (cs * sin_a);
    float3 v = s.sv * (sn * sin_a);
    float3 w = s.sw * cos_a;
    return normalize3((u * v) + w);
}
__device__ __forceinline__ float3 sun_sample_direction(const DScene &s, float x1, float x2) {
    float phi = 2 * CCU_PI_F * x2;
    float sn, cs;
    dm_sincos(phi, sn, cs);
    return sun_sample_direction_sc(s, x1, sn, cs);
}

// kernel.h:50-92: cosine-weighted diffuse bounce direction around normal n; x1, x2 are the two RNG draws
__device__ __forceinline__ float3 diffuse_direction_sc(float3 n, float x1, float sn, float cs) {
    float r = sqrtf(x1);
    float tx = r * cs, ty = r * sn;
    float tz = sqrtf(1 - x1);
    float xx, xy, xz = 0;
    if ((double)fabsf(n.x) > 0.1) { xx = 0; xy = 1; } else { xx = 1; xy = 0; }
    float ux = xy * n.z - xz * n.y;
    float uy = xz * n.x - xx * n.z;
    float uz = xx * n.y - xy * n.x;
    r = 1 / sqrtf((ux * ux + uy * uy) + uz * uz);
    ux *= r; uy *= r; uz *= r;
    float vx = uy * n.z - uz * n.y;
    float vy = uz * n.x - ux * n.z;
    float vz = ux * n.y - uy * n.x;
    return f3((ux * tx + vx * ty) + n.x * tz, (uy * tx + vy * ty) + n.y * tz, (uz * tx + vz * ty) + n.z * tz);
}
__device__ __forceinline__ float3 diffuse_direction(float3 n, float x1, float x2) {
    float theta = 2 * CCU_PI_F * x2;
    float sn, cs;
    dm_sincos(theta, sn, cs);
    return diffuse_direction_sc(n, x1, sn, cs);
}

// ------------------------------------------------------------------------------------------------------
// beyond the reference: specular materials (CCU_RENDER_SPECULAR, DESIGN "Beyond the reference: specular materials")
// ------------------------------------------------------------------------------------------------------
// The event draws of a path-segment hit on a material whose word 5 is w (specular bits 0-7, metalness 8-15, roughness 16-23,
// PackedMaterial.java:68-71): a metal event with probability me, otherwise a (white) specular one with probability sp.  A
// material whose word 5 is 0 draws nothing.  Returns whether the event is specular; `metal` and the roughness `ro` go with it.
__device__ __forceinline__ bool specular_event(uint32_t w, uint32_t &rng, bool &metal, float &ro) {
    const float *u = smem_tables().unorm;
    const float sp = u[w & 0xFF], me = u[(w >> 8) & 0xFF];
    ro = u[(w >> 16) & 0xFF];
    metal = false;
    bool spec = false;
    if (me > 0) metal = rng_float(rng) < me;
    if (!metal && sp > 0) spec = rng_float(rng) < sp;
    return metal || spec;
}
// The direction after a specular event: d mirrored about n, blended towards the cosine-weighted direction q by the roughness.
__device__ __forceinline__ float3 specular_direction(float3 d, float3 n, float3 q, float ro) {
    const float3 r = normalize3(d - n * (2.0f * dot3(d, n)));
    return ro > 0 ? normalize3(r * (1.0f - ro) + q * ro) : r;
}

// ------------------------------------------------------------------------------------------------------
// beyond the reference: emitter sampling (CCU_RENDER_EMITTER_SAMPLING, DESIGN §10)
// ------------------------------------------------------------------------------------------------------
#define CCU_NEE_DELTA (8.0f * CCU_OFFSET)   // the shadow ray stops this far before the sampled point

// The grid cell of voxel (vx, vy, vz); false when the voxel lies outside the grid (always, on a scene without emitters).
__device__ __forceinline__ bool emitter_voxel_cell(const EmitView &g, int vx, int vy, int vz, int3 &c) {
    const long long dx = (long long)vx - g.g0.x, dy = (long long)vy - g.g0.y, dz = (long long)vz - g.g0.z;
    if (dx < 0 || dy < 0 || dz < 0) return false;
    c = make_int3((int)(dx >> g.shift), (int)(dy >> g.shift), (int)(dz >> g.shift));
    return c.x < g.dim.x && c.y < g.dim.y && c.z < g.dim.z;
}
// The cell of point x: that of voxel floor(x); a NaN component is outside.
__device__ __forceinline__ bool emitter_cell(const EmitView &g, float3 x, int3 &c) {
    if (!(x.x == x.x && x.y == x.y && x.z == x.z)) return false;
    return emitter_voxel_cell(g, f2i(floorf(x.x)), f2i(floorf(x.y)), f2i(floorf(x.z)), c);
}
// The list L(c) of cell c: first index into g.list, and its length N.
__device__ __forceinline__ int emitter_list(const EmitView &g, int3 c, int &N) {
    const int ci = (c.x * g.dim.y + c.y) * g.dim.z + c.z;
    const int b = __ldg(g.off + ci);
    N = __ldg(g.off + ci + 1) - b;
    return b;
}
// The emitter sampler a kernel is built with: none, the area sampler of CCU_RENDER_EMITTER_SAMPLING (DESIGN §10), that
// sampler with the near field of CCU_RENDER_EMITTER_NEAR_FIELD (DESIGN §11), or either of the two over the wider table of
// CCU_RENDER_EMITTER_MODELS, which also samples quad and AABB models (DESIGN §12).
enum NeeKind : int { NEE_NONE = 0, NEE_AREA = 1, NEE_NEAR = 2, NEE_AREA_MODELS = 3, NEE_NEAR_MODELS = 4 };
__host__ __device__ constexpr bool nee_near_field(int kind) { return kind == NEE_NEAR || kind == NEE_NEAR_MODELS; }
__host__ __device__ constexpr bool nee_models(int kind) { return kind == NEE_AREA_MODELS || kind == NEE_NEAR_MODELS; }
// The shading variant a render kernel is built with, picked per launch by shade_variant (chunkycu.cu, DESIGN §5).
template <bool S, NeeKind N, bool B, bool F = false, bool C = false>
struct Shade {
    static constexpr bool spec = S, biome = B;
    static constexpr NeeKind nee = N;
    static constexpr bool models = nee_models(N);   // the wider emitter table of CCU_RENDER_EMITTER_MODELS
    static constexpr bool fog = F;                  // the fog of CCU_RENDER_FOG (DESIGN §14)
    static constexpr bool clouds = C;               // the cloud layer of CCU_RENDER_CLOUDS (DESIGN §15)
};
using PlainShade = Shade<false, NEE_NONE, false>;   // the first-hit and preview kernels

// ------------------------------------------------------------------------------------------------------
// beyond the reference: the cloud layer (CCU_RENDER_CLOUDS, DESIGN §15)
// ------------------------------------------------------------------------------------------------------
#define CCU_CLOUD_CELLS 1024            // §15.2: the walk visits at most this many cells, then reports a miss
#define CCU_CLOUD_COORD_MAX 8388608.0f  // §15.2: 2^23, the walk reports a miss where a cell coordinate reaches it

// The ray's parameter interval in cell c (c <= o + d t <= c + 1) of one cell axis; d = 0: the whole line (the walk only visits
// cells that contain o on such an axis, cloud_start).
__device__ __forceinline__ void cloud_axis(float o, float d, int c, float &lo, float &hi) {
    if (d == 0.0f) { lo = -inff_(); hi = inff_(); return; }
    const float a = ((float)c - o) / d, b = ((float)(c + 1) - o) / d;
    lo = d > 0.0f ? a : b;
    hi = d > 0.0f ? b : a;
}
// The walk's first cell on one axis: the cell whose interval holds ts, or the one before it; false for a miss (d = 0 with o on a
// cell boundary, a coordinate at or beyond 2^23, NaN).  step: +1, -1 or 0 for d = 0.
__device__ __forceinline__ bool cloud_start(float o, float d, float ts, int &c, int &step) {
    if (d == 0.0f) {
        const float f = floorf(o);
        if (!(o > f) || !(fabsf(o) < CCU_CLOUD_COORD_MAX)) return false;
        c = (int)f;
        step = 0;
        return true;
    }
    const float x = o + d * ts;
    if (!(fabsf(x) < CCU_CLOUD_COORD_MAX)) return false;
    c = (int)floorf(x);
    step = d > 0.0f ? 1 : -1;
    float lo, hi;
    cloud_axis(o, d, c, lo, hi);
    if (lo > ts) c -= step;
    return true;
}
// §15.2: the smallest t > 0 below `limit` at which the ray o + d t enters the box of a set cell from outside (the boxes are
// open: a ray inside one or on its boundary leaves it without a hit), found by a 2-D walk over the cells inside the slab
// y0 < y < y1; n = the outward normal of the face entered (ties: y, then x, then z).
__device__ __forceinline__ bool cloud_hit(const CloudView &cv, float3 o, float3 d, float limit, float &t, float3 &n) {
    float ylo, yhi;
    if (d.y == 0.0f) {
        if (!(cv.y0 < o.y && o.y < cv.y1)) return false;
        ylo = -inff_();
        yhi = inff_();
    } else {
        const float a = (cv.y0 - o.y) / d.y, b = (cv.y1 - o.y) / d.y;
        if (!(a == a && b == b)) return false;
        ylo = d.y > 0.0f ? a : b;
        yhi = d.y > 0.0f ? b : a;
    }
    const float tend = yhi < limit ? yhi : limit;
    const float ts = ylo > 0.0f ? ylo : 0.0f;
    if (!(ts < tend)) return false;
    const float ox = o.x * cv.inv + cv.u0, dx = d.x * cv.inv;
    const float oz = o.z * cv.inv + cv.v0, dz = d.z * cv.inv;
    int i, k, si, sk;
    if (!cloud_start(ox, dx, ts, i, si) || !cloud_start(oz, dz, ts, k, sk)) return false;
    for (int step = 0; step < CCU_CLOUD_CELLS; step++) {
        float xlo, xhi, zlo, zhi;
        cloud_axis(ox, dx, i, xlo, xhi);
        cloud_axis(oz, dz, k, zlo, zhi);
        const unsigned bit = ((unsigned)(k & 255) << 8) | (unsigned)(i & 255);
        if ((__ldg(cv.mask + (bit >> 5)) >> (bit & 31u)) & 1u) {
            float tn = ylo;
            int axis = 1;
            if (xlo > tn) { tn = xlo; axis = 0; }
            if (zlo > tn) { tn = zlo; axis = 2; }
            float tf = yhi < xhi ? yhi : xhi;
            tf = tf < zhi ? tf : zhi;
            if (tn > 0.0f && tn < tf && tn < limit) {
                t = tn;
                n = axis == 0 ? f3(dx > 0.0f ? -1.0f : 1.0f, 0, 0) : (axis == 1 ? f3(0, d.y > 0.0f ? -1.0f : 1.0f, 0) : f3(0, 0, dz > 0.0f ? -1.0f : 1.0f));
                return true;
            }
        }
        const float te = xhi < zhi ? xhi : zhi;
        if (!(te < tend)) return false;
        if (xhi == te) i += si;
        if (zhi == te) k += sk;
    }
    return false;
}
#define CCU_NEE_RHO2 0.015625f   // DESIGN §11: an emitter is near when its box distance² is below rho² = (1/8)²

// The emission rule: an octree hit on voxel (bx, by, bz) of block palette position `block` that the previous hit's sample
// covered (an emitter whose cell is within Chebyshev distance 1 of that hit's cell c) delivers no emission.  With the model
// table a model emitter (mhead >= 0) counts as well.
template <int KIND = NEE_AREA>
__device__ __forceinline__ bool emitter_covered(const DScene &s, const EmitView &g, int block, int bx, int by, int bz, int3 c) {
    const int4 r0 = __ldg(s.block_rec + 2 * block), r1 = __ldg(s.block_rec + 2 * block + 1);
    if constexpr (nee_models(KIND)) {
        if (!(r0.x == 1 && ((r0.z & 2) || (r1.z & 0xFF))) && __ldg(g.mhead + block) < 0) return false;
    } else {
        if (r0.x != 1 || !((r0.z & 2) || (r1.z & 0xFF))) return false;
    }
    int3 e;
    if (!emitter_voxel_cell(g, bx, by, bz, e)) return false;
    return abs(e.x - c.x) <= 1 && abs(e.y - c.y) <= 1 && abs(e.z - c.z) <= 1;
}

// DESIGN §11 step 4 at a hit x with normal n for emitter e (palette position e.w) from a list of N, whose box distance² is
// below rho²: a cosine-weighted direction (nextPath's, from u2 and u3), scored when it enters the emitter's box through a face
// x lies outside of.  BIOME: the emitter's biome colour tints its material (DESIGN §13).
template <bool BIOME = false>
__device__ __forceinline__ bool nee_near(const DScene &s, int4 e, int N, float3 x, float3 n, float3 T, float u2, float u3, float3 &c,
                                         float3 &w, float &limit) {
    w = diffuse_direction(n, u2, u3);
    const float3 inv = f3(1.0f / w.x, 1.0f / w.y, 1.0f / w.z);
    const float ex = (float)e.x, ey = (float)e.y, ez = (float)e.z;
    const float ax0 = (ex - x.x) * inv.x, ax1 = ((float)(e.x + 1) - x.x) * inv.x;
    const float ay0 = (ey - x.y) * inv.y, ay1 = ((float)(e.y + 1) - x.y) * inv.y;
    const float az0 = (ez - x.z) * inv.z, az1 = ((float)(e.z + 1) - x.z) * inv.z;
    if (!(ax0 == ax0 && ax1 == ax1 && ay0 == ay0 && ay1 == ay1 && az0 == az0 && az1 == az1)) return false;
    // entry: the largest of the near ends (lowest axis on a tie); exit: the smallest of the far ends
    float tn = ax0 < ax1 ? ax0 : ax1, tf = ax0 < ax1 ? ax1 : ax0;
    int axis = 0;
    const float ly = ay0 < ay1 ? ay0 : ay1, hy = ay0 < ay1 ? ay1 : ay0;
    const float lz = az0 < az1 ? az0 : az1, hz = az0 < az1 ? az1 : az0;
    if (ly > tn) { tn = ly; axis = 1; }
    if (lz > tn) { tn = lz; axis = 2; }
    if (hy < tf) tf = hy;
    if (hz < tf) tf = hz;
    if (!(tn <= tf && tn > 0.0f)) return false;
    // the entry face must be one x lies strictly outside of
    const float xa = axis == 0 ? x.x : (axis == 1 ? x.y : x.z), wa = axis == 0 ? w.x : (axis == 1 ? w.y : w.z);
    const int ea = axis == 0 ? e.x : (axis == 1 ? e.y : e.z);
    const int plus = wa < 0.0f ? 1 : 0;
    if (!(plus ? xa > (float)(ea + 1) : xa < (float)ea)) return false;
    // the entry point's in-face coordinates take the places of (u2, u3) in the uv of aabb_full (DESIGN §10 step 3)
    const float3 p = x + w * tn;
    const float px = fminf(fmaxf(p.x - ex, 0.0f), 1.0f), py = fminf(fmaxf(p.y - ey, 0.0f), 1.0f), pz = fminf(fmaxf(p.z - ez, 0.0f), 1.0f);
    float u, v;
    if (axis == 0) { u = plus ? pz : 1.0f - pz; v = py; }
    else if (axis == 1) { u = px; v = plus ? pz : 1.0f - pz; }
    else { u = plus ? 1.0f - px : px; v = py; }
    const int4 r0 = __ldg(s.block_rec + 2 * e.w), r1 = __ldg(s.block_rec + 2 * e.w + 1);
    const MatOut m = material_eval_core<BIOME>(s, (uint32_t)r0.z, (uint32_t)r0.w, (uint32_t)r1.x, (uint32_t)r1.y, (uint32_t)r1.z, u, v, e.x, e.z);
    if (!m.ok) return false;
    // the cosine and 1/pi of the estimator cancel against the direction's density cx / pi
    const float k = (m.emittance * s.emitter_scale) * (float)N;
    c = f3((T.x * (m.color.x * m.color.x)) * k, (T.y * (m.color.y * m.color.y)) * k, (T.z * (m.color.z * m.color.z)) * k);
    limit = tn - CCU_NEE_DELTA;
    return true;
}

// Material_get + Material_sample of material pointer `material` (material_sample's two paths) as a MatOut
template <bool BIOME = false>
__device__ __forceinline__ MatOut material_at(const DScene &s, int material, float u, float v, int bx = 0, int bz = 0) {
    const int idx = material / 6;
    if (material >= 0 && idx * 6 == material) {
        const int4 a = __ldg(s.mat_rec + 2 * idx), b = __ldg(s.mat_rec + 2 * idx + 1);
        return material_eval_core<BIOME>(s, (uint32_t)a.x, (uint32_t)a.y, (uint32_t)a.z, (uint32_t)a.w, (uint32_t)b.x, u, v, bx, bz);
    }
    const int *m = s.mat_palette + material;
    return material_eval_core<BIOME>(s, __ldg(m), __ldg(m + 1), __ldg(m + 2), __ldg(m + 3), __ldg(m + 4), u, v, bx, bz);
}

// DESIGN §12 step 3 for a model entry e (palette position e.w, primitives at g.mprim + h) from a list of N: the near branch
// (NEAR, x within rho of the primitives' bounding box) runs the voxel's block test along a cosine-weighted direction; the far
// branch samples a point on primitive P[min((int)(u1 m), m - 1)].  A primitive record is {kind, material, face flags, w0},
// {w1..w4}, {w5..w8}, {w9..w12}: kind 6 a quad (w0..w12 its 13 words), kind 0..5 the box face axis * 2 + (1 for +) of the box
// w0..w5 (xmin, xmax, ymin, ymax, zmin, zmax).
template <bool NEAR, bool BIOME = false>
__device__ __forceinline__ bool nee_model(const DScene &s, const EmitView &g, int h, int4 e, int N, float3 x, float3 n, float3 T, float u1,
                                          float u2, float u3, float3 &c, float3 &w, float &limit) {
    const int4 h0 = __ldg(g.mprim + h), h1 = __ldg(g.mprim + h + 1);
    const int m = h0.x;
    const float ex = (float)e.x, ey = (float)e.y, ez = (float)e.z;
    if constexpr (NEAR) {
        const float lx = ex + i2f(h0.y), hx = ex + i2f(h0.z), ly = ey + i2f(h0.w), hy = ey + i2f(h1.x), lz = ez + i2f(h1.y), hz = ez + i2f(h1.z);
        const float ox = x.x < lx ? lx - x.x : (x.x > hx ? x.x - hx : 0.0f);
        const float oy = x.y < ly ? ly - x.y : (x.y > hy ? x.y - hy : 0.0f);
        const float oz = x.z < lz ? lz - x.z : (x.z > hz ? x.z - hz : 0.0f);
        if ((ox * ox + oy * oy) + oz * oz < CCU_NEE_RHO2) {
            w = diffuse_direction(n, u2, u3);
            const float3 inv = f3(1.0f / w.x, 1.0f / w.y, 1.0f / w.z);
            Surf hit;
            hit.emittance = 0.0f;
            const float t = intersect_block<BIOME>(s, e.w, e.x, e.y, e.z, hit, x, w, inv);
            if (is_nan(t) || !(hit.emittance > 0.0f)) return false;
            const float k = (hit.emittance * s.emitter_scale) * (float)N;
            c = f3((T.x * (hit.color.x * hit.color.x)) * k, (T.y * (hit.color.y * hit.color.y)) * k, (T.z * (hit.color.z * hit.color.z)) * k);
            limit = t - CCU_NEE_DELTA;
            return true;
        }
    }
    const int4 *r = g.mprim + h + 2 + 4 * min((int)(u1 * (float)m), m - 1);
    const int4 q0 = __ldg(r), q1 = __ldg(r + 1), q2 = __ldg(r + 2), q3 = __ldg(r + 3);
    const bool quad = q0.x == 6;
    const int axis = q0.x >> 1, plus = q0.x & 1;   // box face
    float3 l, nq;        // the sampled point (block-local); the quad's normal
    float u, v, area;
    if (quad) {
        const float3 qo = f3(i2f(q0.w), i2f(q1.x), i2f(q1.y));
        const float3 xv = f3(i2f(q1.z), i2f(q1.w), i2f(q2.x));
        const float3 yv = f3(i2f(q2.y), i2f(q2.z), i2f(q2.w));
        l = (qo + xv * u2) + yv * u3;
        // Quad_intersect's uv at that point
        u = i2f(q3.x) + u2 * i2f(q3.y);
        v = i2f(q3.z) + u3 * i2f(q3.w);
        const float3 cr = cross3(xv, yv);
        nq = normalize3(cr);
        area = sqrtf(dot3(cr, cr));
    } else {
        const float b[6] = {i2f(q0.w), i2f(q1.x), i2f(q1.y), i2f(q1.z), i2f(q1.w), i2f(q2.x)};
        const int a1 = axis == 0 ? 1 : 0, a2 = axis == 2 ? 1 : 2;   // the in-face axes, in increasing order
        const float s1 = b[2 * a1 + 1] - b[2 * a1], s2 = b[2 * a2 + 1] - b[2 * a2];
        float lv[3];
        lv[axis] = b[2 * axis + plus];
        lv[a1] = b[2 * a1] + u2 * s1;
        lv[a2] = b[2 * a2] + u3 * s2;
        l = f3(lv[0], lv[1], lv[2]);
        nq = f3(0, 0, 0);
        area = s1 * s2;
        // AABB_full_intersect_map_2 at l, then the face's flip and swap bits (textured_box)
        if (axis == 0) { u = plus ? 1.0f - l.z : l.z; v = l.y; }
        else if (axis == 1) { u = l.x; v = plus ? 1.0f - l.z : l.z; }
        else { u = plus ? l.x : 1.0f - l.x; v = l.y; }
        const int fl = q0.z;
        if (fl & 4) u = 1.0f - u;
        if (fl & 2) v = 1.0f - v;
        if (fl & 1) { const float t = u; u = v; v = t; }
    }
    const MatOut mo = material_at<BIOME>(s, q0.y, u, v, e.x, e.z);
    if (!mo.ok) return false;
    const float3 dv = f3(ex + l.x, ey + l.y, ez + l.z) - x;
    const float d2 = dot3(dv, dv);
    const float dist = sqrtf(d2);
    w = dv * (1.0f / dist);
    const float cx = dot3(w, n);
    if (!(cx > 0.0f)) return false;
    // the front side: Quad_intersect's test, or x strictly outside the face's plane
    float ce;
    if (quad) {
        const float dn = dot3(w, nq);
        if (!(dn < -CCU_EPS)) return false;
        ce = -dn;
    } else {
        const float xa = axis == 0 ? x.x : (axis == 1 ? x.y : x.z);
        const float pw = (axis == 0 ? ex : (axis == 1 ? ey : ez)) + (axis == 0 ? l.x : (axis == 1 ? l.y : l.z));
        if (!(plus ? xa > pw : xa < pw)) return false;
        ce = fabsf(axis == 0 ? w.x : (axis == 1 ? w.y : w.z));
    }
    const float k = ((mo.emittance * s.emitter_scale) * ((cx * ce) / d2)) * (((float)(N * m) * area) / CCU_PI_F);
    c = f3((T.x * (mo.color.x * mo.color.x)) * k, (T.y * (mo.color.y * mo.color.y)) * k, (T.z * (mo.color.z * mo.color.z)) * k);
    limit = dist - CCU_NEE_DELTA;
    return true;
}

// DESIGN §10 steps 2-4 at a hit x with normal n and throughput T, for the non-empty list emit_list[b .. b + N): draws u0..u3
// and returns whether a shadow ray is traced; if so it runs from x along w up to `limit` and carries the contribution `c`.
// NEE_NEAR(_MODELS): an emitter nearer than rho is sampled by direction instead (DESIGN §11).  NEE_*_MODELS: a model entry
// is sampled by nee_model (DESIGN §12).  BIOME: the emitter's biome colour tints its material (DESIGN §13).
template <int KIND, bool BIOME = false>
__device__ __forceinline__ bool nee_sample(const DScene &s, const EmitView &g, int b, int N, float3 x, float3 n, float3 T, uint32_t &rng, float3 &c,
                                           float3 &w, float &limit) {
    const float u0 = rng_float(rng);
    const float u1 = rng_float(rng);
    const float u2 = rng_float(rng);
    const float u3 = rng_float(rng);
    const int4 e = __ldg(g.emit + __ldg(g.list + b + min((int)(u0 * (float)N), N - 1)));
    if constexpr (nee_models(KIND)) {
        const int h = __ldg(g.mhead + e.w);
        if (h >= 0) return nee_model<nee_near_field(KIND), BIOME>(s, g, h, e, N, x, n, T, u1, u2, u3, c, w, limit);
    }
    const float ex = (float)e.x, ey = (float)e.y, ez = (float)e.z;
    // the faces x lies strictly outside of, in the order -x, +x, -y, +y, -z, +z; 4 bits each: axis * 2 + (1 for the + face)
    unsigned faces = 0;
    int f = 0;
    if (x.x < ex) faces |= 0u << (4 * f++); else if (x.x > (float)(e.x + 1)) faces |= 1u << (4 * f++);
    if (x.y < ey) faces |= 2u << (4 * f++); else if (x.y > (float)(e.y + 1)) faces |= 3u << (4 * f++);
    if (x.z < ez) faces |= 4u << (4 * f++); else if (x.z > (float)(e.z + 1)) faces |= 5u << (4 * f++);
    if (f == 0) return false;
    if constexpr (nee_near_field(KIND)) {
        // box distance² of x to the emitter: o_a is x's distance to the slab [e_a, e_a + 1] on axis a
        const float ox = x.x < ex ? ex - x.x : (x.x > (float)(e.x + 1) ? x.x - (float)(e.x + 1) : 0.0f);
        const float oy = x.y < ey ? ey - x.y : (x.y > (float)(e.y + 1) ? x.y - (float)(e.y + 1) : 0.0f);
        const float oz = x.z < ez ? ez - x.z : (x.z > (float)(e.z + 1) ? x.z - (float)(e.z + 1) : 0.0f);
        if ((ox * ox + oy * oy) + oz * oz < CCU_NEE_RHO2) return nee_near<BIOME>(s, e, N, x, n, T, u2, u3, c, w, limit);
    }
    const int face = (int)((faces >> (4 * min((int)(u1 * (float)f), f - 1))) & 15u);
    const int axis = face >> 1, plus = face & 1;
    // the point and the uv of aabb_full (primitives.h:66-112) at local point (u2, u3) on the face
    float3 p;
    float u, v;
    if (axis == 0) { p = f3((float)(e.x + plus), ey + u2, ez + u3); u = plus ? u3 : 1.0f - u3; v = u2; }
    else if (axis == 1) { p = f3(ex + u2, (float)(e.y + plus), ez + u3); u = u2; v = plus ? u3 : 1.0f - u3; }
    else { p = f3(ex + u2, ey + u3, (float)(e.z + plus)); u = plus ? 1.0f - u2 : u2; v = u3; }
    const int4 r0 = __ldg(s.block_rec + 2 * e.w), r1 = __ldg(s.block_rec + 2 * e.w + 1);
    const MatOut m = material_eval_core<BIOME>(s, (uint32_t)r0.z, (uint32_t)r0.w, (uint32_t)r1.x, (uint32_t)r1.y, (uint32_t)r1.z, u, v, e.x, e.z);
    if (!m.ok) return false;
    const float3 dv = p - x;
    const float d2 = dot3(dv, dv);
    const float dist = sqrtf(d2);
    w = dv * (1.0f / dist);
    const float cx = dot3(w, n);
    if (!(cx > 0.0f)) return false;
    const float ce = fabsf(axis == 0 ? w.x : (axis == 1 ? w.y : w.z));
    const float k = ((m.emittance * s.emitter_scale) * ((cx * ce) / d2)) * ((float)(N * f) / CCU_PI_F);
    c = f3((T.x * (m.color.x * m.color.x)) * k, (T.y * (m.color.y * m.color.y)) * k, (T.z * (m.color.z * m.color.z)) * k);
    limit = dist - CCU_NEE_DELTA;
    return true;
}

}  // namespace ccu
