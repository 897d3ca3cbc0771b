/*
 * chunky_oracle.c - CPU restatement of the ChunkyCL render path.  TEST INFRASTRUCTURE ONLY.
 *
 * This file is the parity oracle: a plain-C restatement of the algorithm of the reference's
 * OpenCL kernels, function by function, quirks included.  Nothing in the product
 * (chunkyclplugin_b200/, include/) may link, load or call it; only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs do.
 *
 * Parity status: PINNED against the reference's own OpenCL kernel executed by the NVIDIA OpenCL
 * runtime on a B200 (oracle/clref, fixtures in tests/golden/clref_*.npz).  The reference itself
 * ships no tests or golden vectors (SURVEY.md section 4).
 *
 * Reference files restated (paths under /root/reference/src/main/opencl/kernel/include/):
 *   rayTracer.cl:40-112 (render), :141-216 (preview)      kernel.h:14-98
 *   octree.h:41-109   block.h:30-118   primitives.h:30-409   bvh.h:22-113
 *   material.h:31-82  textureAtlas.h:10-28  sky.h:19-106  camera.h:8-32
 *   randomness.h:6-17 utils.h:6-27  wavefront.h:13-78  constants.h:4-5
 * Image sampling follows OpenCL 1.2 section 8.2 (SURVEY.md Appendix B).
 * Tonemap filters (oracle_tonemap): /root/reference/src/main/opencl/tonemap/include/post_processing_filter.cl:5-51,
 *   double.h:17-19, rgba.h:6-16; pinned against that kernel run on a B200 (tests/golden/clref_tonemap.npz).
 *
 * Arithmetic contract (shared with the CUDA build, see DESIGN.md "Arithmetic contract"):
 *   - every fp32 operation the reference writes out is a single IEEE-754 round-to-nearest operation, in
 *     source order, no contraction (build with -ffp-contract=off; the CUDA side uses -fmad=false) - i.e.
 *     the reference kernel under "#pragma OPENCL FP_CONTRACT OFF" + -cl-fp32-correctly-rounded-divide-sqrt;
 *   - the vector builtins dot/cross/normalize expand as the NVIDIA OpenCL runtime expands them (explicit
 *     fmaf, see vdot/vcross/vnormalize), so that this file reproduces that build of the reference bit for
 *     bit wherever no transcendental function is involved;
 *   - the reference's implicit double promotions (unsuffixed literals) are kept as doubles;
 *   - float->int conversion saturates and maps NaN to 0 (what cvt.rzi.s32.f32 does on the GPU the
 *     reference runs on; plain C would be UB);
 *   - sin/cos/atan2/asin/acos are the deterministic polynomial versions below ("detmath"),
 *     identical operation for operation to chunkyclplugin_b200/csrc/ccu_math.cuh, so that the
 *     whole path - not only the integer first-hit buffers - is bit-reproducible across CPU and GPU.
 *     math_mode = 1 switches to the platform libm for sensitivity studies.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define EPS 0.000005f   /* constants.h:4 */
#define OFFSET 0.0001f  /* constants.h:5 */
#define PI_F 3.14159274101257f      /* M_PI_F   */
#define PI_2_F 1.57079637050629f    /* M_PI_2_F */
#define INV_PI_F 0.318309886183791f /* M_1_PI_F */
#define ANY_TYPE 0x7FFFFFFE

typedef struct { float x, y, z; } v3;

typedef struct {
    const int32_t *octree;
    int64_t octree_len;
    int32_t octree_depth;
    const int32_t *block_palette;
    const int32_t *quad_models;
    const int32_t *aabb_models;
    const int32_t *world_bvh;
    const int32_t *actor_bvh;
    const int32_t *bvh_trigs;
    const uint8_t *atlas; /* [layers][h][w][4] */
    int32_t atlas_w, atlas_h, atlas_layers;
    const int32_t *mat_palette;
    const uint8_t *sky; /* [res][res][4] */
    int32_t sky_res;
    float sky_intensity;
    const int32_t *sun;
    int32_t projector_type;
    const float *camera;
    int32_t width, height;
    /* launch parameters; reference constants: 256, 5, 13.0f (rayTracer.cl:94,99,107) */
    int32_t draw_depth;
    int32_t max_depth;
    float emitter_scale;
    int32_t math_mode; /* 0 = detmath, 1 = libm */
} OracleScene;

typedef struct {
    uint64_t samples, rays, march_steps, descent_loads, block_tests, material_samples, texel_reads;
    uint64_t bvh_calls, bvh_inner, bvh_leaf, triangles, sky_lookups, sun_texels, aabb_boxes, quads;
    uint64_t segments;
} OracleCounters;

/* ------------------------------------------------------------------------------------------ */
/* scalar helpers                                                                              */
/* ------------------------------------------------------------------------------------------ */
static inline float as_float(int32_t i) { float f; memcpy(&f, &i, 4); return f; }
static inline int32_t f2i(float f) {                /* saturating, NaN -> 0, toward zero */
    if (f != f) return 0;
    if (f >= 2147483648.0f) return INT32_MAX;
    if (f <= -2147483648.0f) return INT32_MIN;
    return (int32_t)f;
}
static inline float fminf_(float a, float b) { return (a != a) ? b : ((b != b) ? a : (a < b ? a : b)); }
static inline float fmaxf_(float a, float b) { return (a != a) ? b : ((b != b) ? a : (a > b ? a : b)); }
static inline int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
static inline v3 V(float x, float y, float z) { v3 r = {x, y, z}; return r; }
static inline v3 vadd(v3 a, v3 b) { return V(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline v3 vsub(v3 a, v3 b) { return V(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline v3 vmul(v3 a, v3 b) { return V(a.x * b.x, a.y * b.y, a.z * b.z); }
static inline v3 vscale(v3 a, float s) { return V(a.x * s, a.y * s, a.z * s); }
/* The OpenCL vector builtins dot / cross / normalize, expanded exactly as the NVIDIA OpenCL runtime expands
 * them (PTX of oracle/clref probe_vec, kept in profiles/clref_vec_strict.ptx): these are library code and use
 * fused multiply-adds even under "#pragma OPENCL FP_CONTRACT OFF". */
static inline float vdot(v3 a, v3 b) { return fmaf(a.z, b.z, fmaf(a.x, b.x, a.y * b.y)); }
static inline v3 vcross(v3 a, v3 b) {
    return V(fmaf(a.y, b.z, -(a.z * b.y)), fmaf(a.z, b.x, -(a.x * b.z)), fmaf(a.x, b.y, -(a.y * b.x)));
}
static inline v3 vnormalize(v3 v) {
    float ax = fabsf(v.x), ay = fabsf(v.y), az = fabsf(v.z);
    if (ax != ax || ay != ay || az != az) return V(NAN, NAN, NAN);
    float m = (ax < ay) ? ay : ax;
    m = (m < az) ? az : m;
    if (m == 0.0f) return V(0, 0, 0);
    if (m == HUGE_VALF) return V(v.x / HUGE_VALF, v.y / HUGE_VALF, v.z / HUGE_VALF);
    float a = ax / m, b = ay / m, c = az / m;
    float r = sqrtf(fmaf(c, c, fmaf(a, a, b * b)));
    float len = m * r;
    if (fabsf(len) != HUGE_VALF) return V(v.x / len, v.y / len, v.z / len);
    return V((v.x / r) / m, (v.y / r) / m, (v.z / r) / m);
}

/* ------------------------------------------------------------------------------------------ */
/* detmath: deterministic fp32 transcendental functions (same operations as ccu_math.cuh)       */
/* ------------------------------------------------------------------------------------------ */
static void dm_sincos(float x, float *s, float *c) {
    float kf = floorf(x * 0.636619772f + 0.5f);
    float r = x - kf * 1.5703125f;
    r = r - kf * 4.837512969970703125e-4f;
    r = r - kf * 7.54978995489188216e-8f;
    int k = f2i(kf) & 3;
    float z = r * r;
    float sp = ((-1.9515295891e-4f * z + 8.3321608736e-3f) * z - 1.6666654611e-1f) * z * r + r;
    float cp = ((2.443315711809948e-5f * z - 1.388731625493765e-3f) * z + 4.166664568298827e-2f) * z * z - 0.5f * z + 1.0f;
    switch (k) {
    case 0: *s = sp; *c = cp; break;
    case 1: *s = cp; *c = -sp; break;
    case 2: *s = -sp; *c = -cp; break;
    default: *s = -cp; *c = sp; break;
    }
}
static float dm_atan(float t) {
    float sign = 1.0f, y0 = 0.0f;
    if (t < 0.0f) { t = -t; sign = -1.0f; }
    if (t > 2.414213562373095f) { y0 = 1.5707963267948966f; t = -(1.0f / t); }
    else if (t > 0.4142135623730950f) { y0 = 0.7853981633974483f; t = (t - 1.0f) / (t + 1.0f); }
    float z = t * t;
    float p = (((8.05374449538e-2f * z - 1.38776856032e-1f) * z + 1.99777106478e-1f) * z - 3.33329491539e-1f) * z * t + t;
    return sign * (y0 + p);
}
static float dm_atan2(float y, float x) {
    if (x != x || y != y) return NAN;
    if (x > 0.0f) return dm_atan(y / x);
    if (x < 0.0f) return (y >= 0.0f) ? dm_atan(y / x) + 3.14159265358979f : dm_atan(y / x) - 3.14159265358979f;
    if (y > 0.0f) return 1.5707963267948966f;
    if (y < 0.0f) return -1.5707963267948966f;
    return 0.0f;
}
static float dm_asin(float x) {
    float a = fabsf(x);
    if (a > 1.0f) return NAN;
    int big = a > 0.5f;
    float z, t;
    if (big) { z = 0.5f * (1.0f - a); t = sqrtf(z); } else { t = a; z = t * t; }
    float p = ((((4.2163199048e-2f * z + 2.4181311049e-2f) * z + 4.5470025998e-2f) * z + 7.4953002686e-2f) * z + 1.6666752422e-1f) * z * t + t;
    if (big) p = 1.5707963267948966f - (p + p);
    return x < 0.0f ? -p : p;
}
static float dm_acos(float x) {
    if (fabsf(x) > 1.0f) return NAN;
    if (x < -0.5f) return 3.14159265358979f - 2.0f * dm_asin(sqrtf(0.5f * (1.0f + x)));
    if (x > 0.5f) return 2.0f * dm_asin(sqrtf(0.5f * (1.0f - x)));
    return 1.5707963267948966f - dm_asin(x);
}

typedef struct { int libm; } Math;
static inline float m_cos(const Math *m, float x) { if (m->libm) return cosf(x); float s, c; dm_sincos(x, &s, &c); return c; }
static inline float m_sin(const Math *m, float x) { if (m->libm) return sinf(x); float s, c; dm_sincos(x, &s, &c); return s; }
static inline float m_atan2(const Math *m, float y, float x) { return m->libm ? atan2f(y, x) : dm_atan2(y, x); }
static inline float m_asin(const Math *m, float x) { return m->libm ? asinf(x) : dm_asin(x); }
static inline float m_acos(const Math *m, float x) { return m->libm ? acosf(x) : dm_acos(x); }

/* ------------------------------------------------------------------------------------------ */
/* RNG - randomness.h:6-17                                                                      */
/* ------------------------------------------------------------------------------------------ */
static inline uint32_t rng_next(uint32_t *state) {
    uint32_t s = *state * 47796405u + 2891336453u;
    s = ((s >> ((s >> 28u) + 4u)) ^ s) * 277803737u;
    s = (s >> 22u) ^ s;
    *state = s;
    return s;
}
static inline float rng_float(uint32_t *state) { return (float)(rng_next(state) >> 8) / 16777216.0f; }

/* ------------------------------------------------------------------------------------------ */
/* per-path state (wavefront.h:6-78 flattened)                                                  */
/* ------------------------------------------------------------------------------------------ */
typedef struct {
    v3 origin, direction; /* Ray (ray.material is always 0: wavefront.h:34, SURVEY Q3) */
    int ray_depth;
    v3 pix_color, throughput; /* Pixel */
} Path;

typedef struct {
    float distance;
    int material;
    v3 normal, point;
    float color[4];
    float emittance;
    /* bookkeeping for the first-hit buffers; not part of the reference's record */
    int hit_node;
    int hit_kind; /* 0 none, 1 octree, 2 world bvh, 3 actor bvh */
} Record;

typedef struct {
    int flags, texture_size, texture;
    float intensity;
    v3 su, sv, sw;
} Sun;

typedef struct {
    const OracleScene *sc;
    Math math;
    Sun sun;
    OracleCounters *cnt;
} Ctx;

/* ------------------------------------------------------------------------------------------ */
/* images                                                                                       */
/* ------------------------------------------------------------------------------------------ */
/* utils.h:6-14 */
static void color_from_argb(uint32_t argb, float out[4]) {
    out[3] = (float)((argb >> 24) & 0xFF) / 256.0f;
    out[0] = (float)((argb >> 16) & 0xFF) / 256.0f;
    out[1] = (float)((argb >> 8) & 0xFF) / 256.0f;
    out[2] = (float)(argb & 0xFF) / 256.0f;
}

/* textureAtlas.h:10-16 - nearest, clamp-to-edge, unnormalised integer coordinates, RGBA8 UNORM */
static void atlas_read_xy(const Ctx *c, int x, int y, int location, float out[4]) {
    const OracleScene *s = c->sc;
    x += ((location >> 22) & 0x1FF) * 16;
    y += ((location >> 13) & 0x1FF) * 16;
    int d = location & 0x7FFFF; /* SURVEY Q9: overlaps the tile-y field */
    x = clampi(x, 0, s->atlas_w - 1);
    y = clampi(y, 0, s->atlas_h - 1);
    d = clampi(d, 0, s->atlas_layers - 1);
    const uint8_t *t = s->atlas + (((size_t)d * s->atlas_h + y) * s->atlas_w + x) * 4;
    for (int i = 0; i < 4; i++) out[i] = (float)t[i] / 255.0f;
    c->cnt->texel_reads++;
}
/* textureAtlas.h:18-28 */
static void atlas_read_uv(const Ctx *c, float u, float v, int location, int size, float out[4]) {
    int width = (size >> 16) & 0xFFFF;
    int height = size & 0xFFFF;
    v = 1.0f - v;
    int x = clampi(f2i((u - EPS) * (float)width), 0, width - 1);
    int y = clampi(f2i((v - EPS) * (float)height), 0, height - 1);
    atlas_read_xy(c, x, y, location, out);
}

/* sky.h:95,105 sampler: normalised coords, mirrored repeat, linear (OpenCL 1.2 s8.2) */
static inline void sky_axis(float s, int w, int *i0, int *i1, float *a) {
    float sp = 2.0f * rintf(0.5f * s);
    sp = fabsf(s - sp);
    float u = sp * (float)w;
    float um = u - 0.5f;
    float fl = floorf(um);
    int j0 = f2i(fl);
    int j1 = j0 + 1;
    *a = um - fl;
    *i0 = j0 < 0 ? 0 : j0;
    *i1 = j1 > w - 1 ? w - 1 : j1;
}
static void sky_read(const Ctx *c, float s, float t, float out[4]) {
    const OracleScene *sc = c->sc;
    int w = sc->sky_res;
    int i0, i1, j0, j1;
    float a, b;
    sky_axis(s, w, &i0, &i1, &a);
    sky_axis(t, w, &j0, &j1, &b);
    const uint8_t *t00 = sc->sky + ((size_t)j0 * w + i0) * 4;
    const uint8_t *t10 = sc->sky + ((size_t)j0 * w + i1) * 4;
    const uint8_t *t01 = sc->sky + ((size_t)j1 * w + i0) * 4;
    const uint8_t *t11 = sc->sky + ((size_t)j1 * w + i1) * 4;
    float w00 = (1.0f - a) * (1.0f - b), w10 = a * (1.0f - b), w01 = (1.0f - a) * b, w11 = a * b;
    for (int k = 0; k < 4; k++) {
        float v = w00 * ((float)t00[k] / 255.0f);
        v = v + w10 * ((float)t10[k] / 255.0f);
        v = v + w01 * ((float)t01[k] / 255.0f);
        v = v + w11 * ((float)t11[k] / 255.0f);
        out[k] = v;
    }
    c->cnt->sky_lookups++;
}

/* ------------------------------------------------------------------------------------------ */
/* material.h:31-82                                                                             */
/* ------------------------------------------------------------------------------------------ */
static int material_sample(const Ctx *c, int material, Record *rec, float u, float v) {
    const int32_t *m = c->sc->mat_palette + material;
    uint32_t flags = (uint32_t)m[0], tint = (uint32_t)m[1], tex_size = (uint32_t)m[2], col = (uint32_t)m[3];
    uint32_t normal_emittance = (uint32_t)m[4];
    c->cnt->material_samples++;
    float color[4];
    if (flags & 4u) atlas_read_uv(c, u, v, (int)col, (int)tex_size, color);
    else color_from_argb(col, color);
    if (color[3] > EPS) memcpy(rec->color, color, sizeof color);
    else return 0;
    float t[4];
    int has_tint = 1;
    switch (tint >> 24) {
    case 0xFF: color_from_argb(tint, t); break;
    case 1: color_from_argb(0xFF71A74Du, t); break;
    case 2: color_from_argb(0xFF8EB971u, t); break;
    case 3: color_from_argb(0xFF3F76E4u, t); break;
    default: has_tint = 0;
    }
    if (has_tint) for (int i = 0; i < 4; i++) rec->color[i] *= t[i];
    if (flags & 2u) {
        float e[4];
        atlas_read_uv(c, u, v, (int)normal_emittance, (int)tex_size, e);
        rec->emittance = e[3];
    } else {
        rec->emittance = (float)((double)(normal_emittance & 0xFF) / 255.0); /* SURVEY Q12 */
    }
    return 1;
}

/* ------------------------------------------------------------------------------------------ */
/* primitives.h                                                                                 */
/* ------------------------------------------------------------------------------------------ */
typedef struct { float xmin, xmax, ymin, ymax, zmin, zmax; } AABB;

/* primitives.h:30-48 */
static float aabb_quick(const AABB *b, v3 o, v3 inv) {
    float t1x = (b->xmin - o.x) * inv.x, t1y = (b->ymin - o.y) * inv.y, t1z = (b->zmin - o.z) * inv.z;
    float t2x = (b->xmax - o.x) * inv.x, t2y = (b->ymax - o.y) * inv.y, t2z = (b->zmax - o.z) * inv.z;
    float tmin = fmaxf_(fminf_(t1x, t2x), fmaxf_(fminf_(t1y, t2y), fminf_(t1z, t2z)));
    float tmax = fminf_(fmaxf_(t1x, t2x), fminf_(fmaxf_(t1y, t2y), fmaxf_(t1z, t2z)));
    return (tmax < tmin) ? NAN : tmin;
}
/* primitives.h:52-61 */
static float aabb_exit(const AABB *b, v3 o, v3 inv) {
    float t1x = (b->xmin - o.x) * inv.x, t1y = (b->ymin - o.y) * inv.y, t1z = (b->zmin - o.z) * inv.z;
    float t2x = (b->xmax - o.x) * inv.x, t2y = (b->ymax - o.y) * inv.y, t2z = (b->zmax - o.z) * inv.z;
    return fminf_(fmaxf_(t1x, t2x), fminf_(fmaxf_(t1y, t2y), fmaxf_(t1z, t2z)));
}
/* primitives.h:66-112 (map2 = 0) and :117-162 (map2 = 1).  Later matches overwrite earlier ones. */
static float aabb_full(const AABB *b, v3 origin, v3 dir, v3 inv, v3 *normal, float *u, float *v, int map2) {
    float t1x = (b->xmin - origin.x) * inv.x, t1y = (b->ymin - origin.y) * inv.y, t1z = (b->zmin - origin.z) * inv.z;
    float t2x = (b->xmax - origin.x) * inv.x, t2y = (b->ymax - origin.y) * inv.y, t2z = (b->zmax - origin.z) * inv.z;
    float tmin = fmaxf_(fminf_(t1x, t2x), fmaxf_(fminf_(t1y, t2y), fminf_(t1z, t2z)));
    float tmax = fminf_(fmaxf_(t1x, t2x), fminf_(fmaxf_(t1y, t2y), fmaxf_(t1z, t2z)));
    if (tmax < tmin) return NAN;
    v3 o = vadd(origin, vscale(dir, tmin));
    if (!map2) {
        float dx = 1.0f / (b->xmax - b->xmin), dy = 1.0f / (b->ymax - b->ymin), dz = 1.0f / (b->zmax - b->zmin);
        if (t1x == tmin) { *u = 1.0f - (o.z - b->zmin) * dz; *v = (o.y - b->ymin) * dy; *normal = V(-1, 0, 0); }
        if (t2x == tmin) { *u = (o.z - b->zmin) * dz; *v = (o.y - b->ymin) * dy; *normal = V(1, 0, 0); }
        if (t1y == tmin) { *u = (o.x - b->xmin) * dx; *v = 1.0f - (o.z - b->zmin) * dz; *normal = V(0, -1, 0); }
        if (t2y == tmin) { *u = (o.x - b->xmin) * dx; *v = (o.z - b->zmin) * dz; *normal = V(0, 1, 0); }
        if (t1z == tmin) { *u = (o.x - b->xmin) * dx; *v = (o.y - b->ymin) * dy; *normal = V(0, 0, -1); }
        if (t2z == tmin) { *u = 1.0f - (o.x - b->xmin) * dx; *v = (o.y - b->ymin) * dy; *normal = V(0, 0, 1); }
    } else {
        if (t1x == tmin) { *u = o.z; *v = o.y; *normal = V(-1, 0, 0); }
        if (t2x == tmin) { *u = 1.0f - o.z; *v = o.y; *normal = V(1, 0, 0); }
        if (t1y == tmin) { *u = o.x; *v = o.z; *normal = V(0, -1, 0); }
        if (t2y == tmin) { *u = o.x; *v = 1.0f - o.z; *normal = V(0, 1, 0); }
        if (t1z == tmin) { *u = 1.0f - o.x; *v = o.y; *normal = V(0, 0, -1); }
        if (t2z == tmin) { *u = o.x; *v = o.y; *normal = V(0, 0, 1); }
    }
    return tmin;
}

/* primitives.h:200-260.  The +z face never selects a material in the reference (it tests
 * normal.z == -1 twice, SURVEY Q10: uninitialised read).  Defined here as material pointer 0, flags 0. */
static float textured_aabb(const int32_t *model, float distance, v3 origin, v3 dir, v3 inv, v3 *normal, float *u, float *v, int *material) {
    AABB box = {as_float(model[0]), as_float(model[1]), as_float(model[2]), as_float(model[3]), as_float(model[4]), as_float(model[5])};
    int bflags = model[6];
    v3 n = V(0, 0, 0);
    float tu = 0, tv = 0;
    float dist = aabb_full(&box, origin, dir, inv, &n, &tu, &tv, 1);
    if (dist >= distance || dist < -EPS) return NAN;
    if (dist != dist) return NAN; /* NaN fails both tests above in the reference and then reads undefined normals */
    int mat = 0, flags = 0;
    if (n.z == -1.0f) { mat = model[7]; flags = bflags; }
    if (n.x == 1.0f) { mat = model[8]; flags = bflags >> 4; }
    if (n.z == -1.0f) { mat = model[9]; flags = bflags >> 8; }
    if (n.x == -1.0f) { mat = model[10]; flags = bflags >> 12; }
    if (n.y == 1.0f) { mat = model[11]; flags = bflags >> 16; }
    if (n.y == -1.0f) { mat = model[12]; flags = bflags >> 20; }
    if (flags & 8) return NAN;
    if (flags & 4) tu = 1.0f - tu;
    if (flags & 2) tv = 1.0f - tv;
    if (flags & 1) { float t = tu; tu = tv; tv = t; }
    *material = mat; *normal = n; *u = tu; *v = tv;
    return dist;
}

/* primitives.h:274-319 */
static float quad_intersect(const int32_t *q, float distance, v3 origin, v3 dir, v3 *normal, float *u, float *v) {
    v3 qo = V(as_float(q[0]), as_float(q[1]), as_float(q[2]));
    v3 xv = V(as_float(q[3]), as_float(q[4]), as_float(q[5]));
    v3 yv = V(as_float(q[6]), as_float(q[7]), as_float(q[8]));
    float uvx = as_float(q[9]), uvy = as_float(q[10]), uvz = as_float(q[11]), uvw = as_float(q[12]);
    v3 n = vnormalize(vcross(xv, yv));
    float denom = vdot(dir, n);
    if (denom < -EPS) {
        float t = -(vdot(origin, n) - vdot(n, qo)) / denom;
        if (t > -EPS && t < distance) {
            v3 pt = vsub(vadd(origin, vscale(dir, t)), qo);
            float uu = vdot(pt, xv) / vdot(xv, xv);
            float vv = vdot(pt, yv) / vdot(yv, yv);
            if (uu >= 0 && uu <= 1 && vv >= 0 && vv <= 1) {
                *u = uvx + (uu * uvy);
                *v = uvz + (vv * uvw);
                *normal = n;
                return t;
            }
        }
    }
    return NAN;
}

/* primitives.h:335-409 */
static float triangle_intersect(const int32_t *t, float distance, v3 origin, v3 dir, v3 *normal, float *ou, float *ov, int *material) {
    int flags = t[0];
    v3 e1 = V(as_float(t[1]), as_float(t[2]), as_float(t[3]));
    v3 e2 = V(as_float(t[4]), as_float(t[5]), as_float(t[6]));
    v3 o = V(as_float(t[7]), as_float(t[8]), as_float(t[9]));
    v3 pvec = vcross(dir, e2);
    float det = vdot(e1, pvec);
    if ((flags >> 8) & 1) {
        if (det > -EPS && det < EPS) return NAN;
    } else if (det > -EPS) {
        return NAN;
    }
    float recip = 1.0f / det;
    v3 tvec = vsub(origin, o);
    float u = vdot(tvec, pvec) * recip;
    if (u < 0 || u > 1) return NAN;
    v3 qvec = vcross(tvec, e1);
    float v = vdot(dir, qvec) * recip;
    if (v < 0 || (u + v) > 1) return NAN;
    float tt = vdot(e2, qvec) * recip;
    if (tt > EPS && tt < distance) {
        float w = 1.0f - u - v;
        float t1x = as_float(t[13]), t1y = as_float(t[14]), t2x = as_float(t[15]), t2y = as_float(t[16]);
        float t3x = as_float(t[17]), t3y = as_float(t[18]);
        *ou = (t1x * u + t2x * v) + t3x * w;
        *ov = (t1y * u + t2y * v) + t3y * w;
        *normal = V(as_float(t[10]), as_float(t[11]), as_float(t[12]));
        *material = t[19];
        return tt;
    }
    return NAN;
}

/* ------------------------------------------------------------------------------------------ */
/* block.h:30-118                                                                               */
/* ------------------------------------------------------------------------------------------ */
static float intersect_block(const Ctx *c, int block, int bx, int by, int bz, Record *rec, v3 origin, v3 direction, v3 inv) {
    if (block == ANY_TYPE) return NAN;
    const OracleScene *s = c->sc;
    int model_type = s->block_palette[block + 0];
    int model_ptr = s->block_palette[block + 1];
    c->cnt->block_tests++;
    v3 norm_origin = vsub(vsub(origin, vscale(direction, OFFSET)), V((float)bx, (float)by, (float)bz));
    v3 normal = V(0, 0, 0);
    float u = 0, v = 0;
    switch (model_type) {
    default:
    case 0:
        return NAN;
    case 1: {
        AABB box = {0, 1, 0, 1, 0, 1};
        /* SURVEY Q2: the marched position is passed where a direction is expected (block.h:52) */
        float dist = aabb_full(&box, norm_origin, origin, inv, &normal, &u, &v, 0);
        if (dist != dist) return NAN;
        rec->normal = normal; /* written before the alpha test, SURVEY Q11 */
        if (material_sample(c, model_ptr, rec, u, v)) return dist - OFFSET;
        return NAN;
    }
    case 2: {
        int hit = 0;
        float dist = HUGE_VALF;
        int material = 0;
        int boxes = s->aabb_models[model_ptr];
        for (int i = 0; i < boxes; i++) {
            const int32_t *model = s->aabb_models + model_ptr + 1 + i * 13;
            c->cnt->aabb_boxes++;
            float t = textured_aabb(model, dist, norm_origin, direction, inv, &normal, &u, &v, &material);
            if (t == t) {
                if (material_sample(c, material, rec, u, v)) { rec->normal = normal; dist = t; hit = 1; }
            }
        }
        return hit ? dist : NAN;
    }
    case 3: {
        int hit = 0;
        float dist = HUGE_VALF;
        int quads = s->quad_models[model_ptr];
        for (int i = 0; i < quads; i++) {
            const int32_t *q = s->quad_models + model_ptr + 1 + i * 15;
            c->cnt->quads++;
            float t = quad_intersect(q, dist, norm_origin, direction, &normal, &u, &v);
            if (t == t) {
                if (material_sample(c, q[13], rec, u, v)) { rec->normal = normal; dist = t; hit = 1; }
            }
        }
        return hit ? dist : NAN;
    }
    }
}

/* ------------------------------------------------------------------------------------------ */
/* octree.h:41-109                                                                              */
/* ------------------------------------------------------------------------------------------ */
static inline void floor3i(v3 p, int *x, int *y, int *z) { *x = f2i(floorf(p.x)); *y = f2i(floorf(p.y)); *z = f2i(floorf(p.z)); }

static int octree_intersect(const Ctx *c, const Path *ray, Record *rec) {
    const OracleScene *s = c->sc;
    const int32_t *tree = s->octree;
    int depth = s->octree_depth;
    float dist_march = 0;
    v3 inv = V(1.0f / ray->direction.x, 1.0f / ray->direction.y, 1.0f / ray->direction.z);
    v3 offset_d = vscale(ray->direction, OFFSET);
    int lx, ly, lz;
    floor3i(ray->origin, &lx, &ly, &lz);
    if (((lx >> depth) != 0) | ((ly >> depth) != 0) | ((lz >> depth) != 0)) {
        float size = (float)(1 << depth);
        AABB box = {0, size, 0, size, 0, size};
        float dist = aabb_quick(&box, ray->origin, inv);
        if (dist != dist || dist < 0) return 0;
        dist_march += dist + OFFSET;
    }
    for (int i = 0; i < s->draw_depth; i++) {
        if (dist_march > rec->distance) return 0;
        v3 pos = vadd(ray->origin, vscale(ray->direction, dist_march));
        int bx, by, bz;
        floor3i(vadd(pos, offset_d), &bx, &by, &bz);
        if (((bx >> depth) != 0) | ((by >> depth) != 0) | ((bz >> depth) != 0)) return 0;
        c->cnt->march_steps++;
        int level = depth;
        int node = 0;
        int data = tree[0];
        c->cnt->descent_loads++;
        while (data > 0) {
            level--;
            node = data + ((((bx >> level) & 1) << 2) | (((by >> level) & 1) << 1) | ((bz >> level) & 1));
            data = tree[node];
            c->cnt->descent_loads++;
        }
        data = -data;
        lx = bx >> level; ly = by >> level; lz = bz >> level;
        if (data != 0) { /* ray->material == 0 always */
            float dist = intersect_block(c, data, bx, by, bz, rec, pos, ray->direction, inv);
            if (dist == dist) {
                rec->distance = dist_march + dist;
                rec->material = data;
                rec->hit_node = node;
                rec->hit_kind = 1;
                return 1;
            }
        }
        AABB box = {(float)(lx << level), (float)((lx + 1) << level), (float)(ly << level), (float)((ly + 1) << level),
                    (float)(lz << level), (float)((lz + 1) << level)};
        dist_march += aabb_exit(&box, vadd(pos, offset_d), inv) + OFFSET;
    }
    return 0;
}

/* ------------------------------------------------------------------------------------------ */
/* bvh.h:22-113                                                                                 */
/* ------------------------------------------------------------------------------------------ */
static int bvh_intersect(const Ctx *c, const int32_t *bvh, const Path *ray, Record *rec, int kind) {
    const int32_t *trigs = c->sc->bvh_trigs;
    c->cnt->bvh_calls++;
    if (bvh[0] == 0) {
        int all_nan = 1;
        for (int i = 1; i < 7; i++) { float f = as_float(bvh[i]); if (f == f) all_nan = 0; }
        if (all_nan) return 0;
    }
    int hit = 0, to_visit = 0, current = 0;
    int stack[64];
    v3 inv = V(1.0f / ray->direction.x, 1.0f / ray->direction.y, 1.0f / ray->direction.z);
    for (;;) {
        int head = bvh[current];
        if (head <= 0) {
            int prim = -head;
            int num = trigs[prim];
            c->cnt->bvh_leaf++;
            for (int i = 0; i < num; i++) {
                v3 normal; float u, v; int material;
                c->cnt->triangles++;
                float dist = triangle_intersect(trigs + prim + 1 + 20 * i, rec->distance, ray->origin, ray->direction, &normal, &u, &v, &material);
                if (dist == dist) {
                    if (material_sample(c, material, rec, u, v)) {
                        rec->normal = normal; rec->distance = dist; hit = 1; /* record->material untouched: SURVEY Q15 */
                        rec->hit_kind = kind; rec->hit_node = -1;
                    }
                }
            }
            if (to_visit == 0) break;
            current = stack[--to_visit];
        } else {
            int offset = head;
            c->cnt->bvh_inner++;
            const int32_t *n1 = bvh + current + 7;
            AABB b1 = {as_float(n1[1]), as_float(n1[2]), as_float(n1[3]), as_float(n1[4]), as_float(n1[5]), as_float(n1[6])};
            float t1 = aabb_quick(&b1, ray->origin, inv);
            const int32_t *n2 = bvh + offset;
            AABB b2 = {as_float(n2[1]), as_float(n2[2]), as_float(n2[3]), as_float(n2[4]), as_float(n2[5]), as_float(n2[6])};
            float t2 = aabb_quick(&b2, ray->origin, inv);
            int miss1 = (t1 != t1) || t1 > rec->distance;
            int miss2 = (t2 != t2) || t2 > rec->distance;
            if (miss1) {
                if (miss2) {
                    if (to_visit == 0) break;
                    current = stack[--to_visit];
                } else {
                    current = offset;
                }
            } else if (miss2) {
                current += 7;
            } else if (t1 < t2) {
                stack[to_visit++] = offset;
                current += 7;
            } else {
                stack[to_visit++] = current + 7;
                current = offset;
            }
        }
    }
    return hit;
}

/* ------------------------------------------------------------------------------------------ */
/* sky.h, kernel.h                                                                              */
/* ------------------------------------------------------------------------------------------ */
static Sun sun_new(const OracleScene *s, const Math *m) { /* sky.h:19-40 */
    Sun sun;
    const int32_t *d = s->sun;
    sun.flags = d[0]; sun.texture_size = d[1]; sun.texture = d[2]; sun.intensity = as_float(d[3]);
    float phi = as_float(d[4]), theta = as_float(d[5]);
    float r = fabsf(m_cos(m, phi));
    sun.sw = V(m_cos(m, theta) * r, m_sin(m, phi), m_sin(m, theta) * r);
    if (fabsf(sun.sw.x) > 0.1f) sun.su = V(0, 1, 0); else sun.su = V(1, 0, 0);
    sun.sv = vnormalize(vcross(sun.sw, sun.su));
    sun.su = vcross(sun.sv, sun.sw);
    return sun;
}

static int sun_intersect(const Ctx *c, v3 direction, Record *rec) { /* sky.h:42-66 */
    const Sun *sun = &c->sun;
    if (!(sun->flags & 1) || vdot(direction, sun->sw) < 0.5f) return 0;
    float radius = 0.03f;
    float width = radius * 4;
    float width2 = width * 2;
    float a = PI_2_F - m_acos(&c->math, vdot(direction, sun->su)) + width;
    if (a >= 0 && a < width2) {
        float b = PI_2_F - m_acos(&c->math, vdot(direction, sun->sv)) + width;
        if (b >= 0 && b < width2) {
            float col[4];
            atlas_read_uv(c, a / width2, b / width2, sun->texture, sun->texture_size, col);
            c->cnt->sun_texels++;
            for (int i = 0; i < 4; i++) rec->color[i] += col[i] * sun->intensity;
            return 1;
        }
    }
    return 0;
}

static void sky_intersect(const Ctx *c, v3 d, Record *rec) { /* sky.h:97-106 */
    float theta = m_atan2(&c->math, d.z, d.x);
    theta /= PI_F * 2;
    theta = fmodf(fmodf(theta, 1.0f) + 1.0f, 1.0f);
    float cl = fminf_(fmaxf_(d.y, -1.0f), 1.0f);
    float phi = (m_asin(&c->math, cl) + PI_2_F) * INV_PI_F;
    float col[4];
    sky_read(c, theta, phi, col);
    for (int i = 0; i < 4; i++) rec->color[i] = col[i] * c->sc->sky_intensity;
}

/* kernel.h:14-24 */
static int closest_intersect(const Ctx *c, const Path *ray, Record *rec) {
    int hit = 0;
    c->cnt->rays++;
    hit |= octree_intersect(c, ray, rec);
    hit |= bvh_intersect(c, c->sc->world_bvh, ray, rec, 2);
    hit |= bvh_intersect(c, c->sc->actor_bvh, ray, rec, 3);
    if (hit) rec->point = vadd(ray->origin, vscale(ray->direction, rec->distance - OFFSET));
    return hit;
}

/* kernel.h:26-31 */
static void intersect_sky(const Ctx *c, Path *p, Record *rec) {
    sky_intersect(c, p->direction, rec);
    sun_intersect(c, p->direction, rec);
    v3 col = V(rec->color[0], rec->color[1], rec->color[2]);
    p->pix_color = vadd(p->pix_color, vscale(vmul(col, p->throughput), rec->emittance));
}

/* kernel.h:33-44 */
static void apply_ray_color(Path *p, Record *rec, float emitter_scale) {
    p->origin = rec->point;
    v3 col = V(rec->color[0], rec->color[1], rec->color[2]);
    p->throughput = vmul(p->throughput, col);
    v3 em = vscale(col, rec->emittance * emitter_scale);
    p->pix_color = vadd(p->pix_color, vmul(em, p->throughput));
}

/* sky.h:68-93 */
static int sun_sample_direction(const Ctx *c, Path *p, Record *rec, uint32_t *state) {
    const Sun *sun = &c->sun;
    if (!(sun->flags & 1)) return 0;
    float radius_cos = m_cos(&c->math, 0.03f);
    float x1 = rng_float(state);
    float x2 = rng_float(state);
    float cos_a = 1 - x1 + x1 * radius_cos;
    float sin_a = sqrtf(1 - cos_a * cos_a);
    float phi = 2 * PI_F * x2;
    v3 u = vscale(sun->su, m_cos(&c->math, phi) * sin_a);
    v3 v = vscale(sun->sv, m_sin(&c->math, phi) * sin_a);
    v3 w = vscale(sun->sw, cos_a);
    p->direction = vmul(u, v); /* component-wise product, SURVEY Q5 */
    p->direction = vadd(p->direction, w);
    p->direction = vnormalize(p->direction);
    rec->emittance = fabsf(vdot(p->direction, rec->normal));
    return 1;
}

/* kernel.h:46-98 */
static int next_path(const Ctx *c, Path *p, Record *rec, uint32_t *state, int max_depth) {
    p->origin = rec->point;
    float x1 = rng_float(state);
    float x2 = rng_float(state);
    float r = sqrtf(x1);
    float theta = 2 * PI_F * x2;
    float tx = r * m_cos(&c->math, theta);
    float ty = r * m_sin(&c->math, theta);
    float tz = sqrtf(1 - x1);
    float xx, xy, xz;
    if ((double)fabsf(rec->normal.x) > 0.1) { xx = 0; xy = 1; } else { xx = 1; xy = 0; }
    xz = 0;
    v3 n = rec->normal;
    float ux = xy * n.z - xz * n.y;
    float uy = xz * n.x - xx * n.z;
    float uz = xx * n.y - xy * n.x;
    r = 1 / sqrtf((ux * ux + uy * uy) + uz * uz);
    ux *= r; uy *= r; uz *= r;
    float vx = uy * n.z - uz * n.y;
    float vy = uz * n.x - ux * n.z;
    float vz = ux * n.y - uy * n.x;
    p->direction.x = (ux * tx + vx * ty) + n.x * tz;
    p->direction.y = (uy * tx + vy * ty) + n.y * tz;
    p->direction.z = (uz * tx + vz * ty) + n.z * tz;
    p->origin = vadd(p->origin, vscale(p->direction, OFFSET));
    p->ray_depth += 1;
    rec->distance = HUGE_VALF;
    return p->ray_depth < max_depth;
}

/* camera.h:8-32 + rayTracer.cl:55-91.  normalize_dir = 1 is the preview variant (rayTracer.cl:186). */
static void camera_ray(const Ctx *c, int gid, uint32_t *state, Path *p, int normalize_dir) {
    const OracleScene *s = c->sc;
    if (s->projector_type != -1) {
        const float *cs = s->camera;
        v3 cam_pos = V(cs[0], cs[1], cs[2]);
        v3 m1 = V(cs[3], cs[4], cs[5]), m2 = V(cs[6], cs[7], cs[8]), m3 = V(cs[9], cs[10], cs[11]);
        float half_width = (float)(s->width / (2.0 * s->height));
        float inv_height = (float)(1.0 / s->height);
        float x = -half_width + ((float)(gid % s->width) + rng_float(state)) * inv_height;
        float y = (float)(-0.5 + (double)(((float)(gid / s->width) + rng_float(state)) * inv_height));
        v3 o = V(0, 0, 0), d = V(0, 0, 1);
        if (s->projector_type == 0) {
            float aperture = cs[12], subject_distance = cs[13], fov_tan = cs[14];
            d = V(fov_tan * x, fov_tan * y, 1.0f);
            if (aperture > 0) {
                d = vscale(d, subject_distance / d.z);
                float r = sqrtf(rng_float(state)) * aperture;
                float theta = rng_float(state) * PI_F * 2.0f;
                float rx = m_cos(&c->math, theta) * r;
                float ry = m_sin(&c->math, theta) * r;
                d = vsub(d, V(rx, ry, 0));
                o = vadd(o, V(rx, ry, 0));
            }
        }
        if (normalize_dir) d = vnormalize(d);
        p->direction = V(vdot(m1, d), vdot(m2, d), vdot(m3, d));
        p->origin = vadd(V(vdot(m1, o), vdot(m2, o), vdot(m3, o)), cam_pos);
    } else {
        const float *r = s->camera + (size_t)gid * 6;
        p->origin = V(r[0], r[1], r[2]);
        p->direction = V(r[3], r[4], r[5]);
    }
}

static void record_new(Record *rec) {
    memset(rec, 0, sizeof *rec);
    rec->distance = HUGE_VALF;
    rec->material = 0;
    rec->hit_node = -1;
}

/* one path sample: rayTracer.cl:40-107 */
static v3 sample_pixel(const Ctx *c, int gid, int32_t seed) {
    Path p;
    Record rec;
    p.pix_color = V(0, 0, 0);
    p.throughput = V(1, 1, 1);
    p.ray_depth = 0;
    record_new(&rec);
    uint32_t state = (uint32_t)seed + (uint32_t)gid;
    rng_next(&state);
    camera_ray(c, gid, &state, &p, 0);
    c->cnt->samples++;
    do {
        c->cnt->segments++;
        if (!closest_intersect(c, &p, &rec)) {
            rec.emittance = 1;
            intersect_sky(c, &p, &rec);
            break;
        }
        apply_ray_color(&p, &rec, c->sc->emitter_scale);
        if (sun_sample_direction(c, &p, &rec, &state)) {
            Record s = rec; /* IntersectionRecord_copy keeps distance: SURVEY Q4 */
            s.point = rec.normal;
            if (!closest_intersect(c, &p, &s)) intersect_sky(c, &p, &s);
        }
    } while (next_path(c, &p, &rec, &state, c->sc->max_depth));
    return p.pix_color;
}

static void ctx_init(Ctx *c, const OracleScene *s, OracleCounters *cnt) {
    c->sc = s;
    c->math.libm = s->math_mode == 1;
    c->sun = sun_new(s, &c->math);
    c->cnt = cnt;
}

static void counters_add(OracleCounters *a, const OracleCounters *b) {
    uint64_t *x = (uint64_t *)a;
    const uint64_t *y = (const uint64_t *)b;
    for (size_t i = 0; i < sizeof(OracleCounters) / 8; i++) x[i] += y[i];
}

/* ------------------------------------------------------------------------------------------ */
/* exported entry points                                                                        */
/* ------------------------------------------------------------------------------------------ */

/* Running-mean accumulation of n_passes passes over pixels [gid0, gid1) (or an explicit list),
 * rayTracer.cl:109-112 with bufferSpp = start_spp + pass.  res is float[3*W*H]. */
int oracle_render(const OracleScene *s, const int32_t *seeds, int n_passes, int start_spp, float *res,
                  const int32_t *gids, int64_t n_gids, int nthreads, OracleCounters *out_counters) {
    int64_t n = gids ? n_gids : (int64_t)s->width * s->height;
    OracleCounters total;
    memset(&total, 0, sizeof total);
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
#pragma omp parallel
    {
        OracleCounters local;
        memset(&local, 0, sizeof local);
        Ctx c;
        ctx_init(&c, s, &local);
#pragma omp for schedule(dynamic, 64)
        for (int64_t k = 0; k < n; k++) {
            int gid = gids ? gids[k] : (int)k;
            float *px = res + (size_t)gid * 3;
            v3 buf = V(px[0], px[1], px[2]);
            for (int pass = 0; pass < n_passes; pass++) {
                v3 col = sample_pixel(&c, gid, seeds[pass]);
                int spp = start_spp + pass;
                buf.x = (buf.x * (float)spp + col.x) / (float)(spp + 1);
                buf.y = (buf.y * (float)spp + col.y) / (float)(spp + 1);
                buf.z = (buf.z * (float)spp + col.z) / (float)(spp + 1);
            }
            px[0] = buf.x; px[1] = buf.y; px[2] = buf.z;
        }
#pragma omp critical
        counters_add(&total, &local);
    }
    if (out_counters) *out_counters = total;
    return 0;
}

/* First-hit buffers for the camera ray of every pixel (BASELINE config 2).
 * block = record.material, face from the normal, node = treeData index of the hit leaf,
 * kind 0 miss / 1 octree / 2 world bvh / 3 actor bvh, t = record.distance, normal[3], color[4]. */
static int face_of(v3 n) {
    if (n.x == -1 && n.y == 0 && n.z == 0) return 0;
    if (n.x == 1 && n.y == 0 && n.z == 0) return 1;
    if (n.x == 0 && n.y == -1 && n.z == 0) return 2;
    if (n.x == 0 && n.y == 1 && n.z == 0) return 3;
    if (n.x == 0 && n.y == 0 && n.z == -1) return 4;
    if (n.x == 0 && n.y == 0 && n.z == 1) return 5;
    return 6;
}
int oracle_first_hit(const OracleScene *s, int32_t seed, int32_t *block, int32_t *face, int32_t *node, int32_t *kind,
                     float *t, float *normal, float *color, int nthreads, OracleCounters *out_counters) {
    int64_t n = (int64_t)s->width * s->height;
    OracleCounters total;
    memset(&total, 0, sizeof total);
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
#pragma omp parallel
    {
        OracleCounters local;
        memset(&local, 0, sizeof local);
        Ctx c;
        ctx_init(&c, s, &local);
#pragma omp for schedule(dynamic, 256)
        for (int64_t gid = 0; gid < n; gid++) {
            Path p;
            Record rec;
            p.pix_color = V(0, 0, 0); p.throughput = V(1, 1, 1); p.ray_depth = 0;
            record_new(&rec);
            uint32_t state = (uint32_t)seed + (uint32_t)gid;
            rng_next(&state);
            camera_ray(&c, (int)gid, &state, &p, 0);
            int hit = closest_intersect(&c, &p, &rec);
            block[gid] = hit ? rec.material : 0;
            kind[gid] = hit ? rec.hit_kind : 0;
            node[gid] = hit ? rec.hit_node : -1;
            face[gid] = hit ? face_of(rec.normal) : 6;
            t[gid] = hit ? rec.distance : HUGE_VALF;
            for (int i = 0; i < 3; i++) normal[gid * 3 + i] = hit ? (&rec.normal.x)[i] : 0.0f;
            for (int i = 0; i < 4; i++) color[gid * 4 + i] = hit ? rec.color[i] : 0.0f;
        }
#pragma omp critical
        counters_add(&total, &local);
    }
    if (out_counters) *out_counters = total;
    return 0;
}

/* preview: rayTracer.cl:141-216.  res is int32[W*H] ARGB. */
int oracle_preview(const OracleScene *s, int32_t *res, int nthreads) {
    int64_t n = (int64_t)s->width * s->height;
    int W = s->width, H = s->height;
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
#pragma omp parallel
    {
        OracleCounters local;
        memset(&local, 0, sizeof local);
        Ctx c;
        ctx_init(&c, s, &local);
#pragma omp for schedule(dynamic, 256)
        for (int64_t gid = 0; gid < n; gid++) {
            int px = (int)(gid % W), py = (int)(gid / W);
            if ((px == W / 2 && (py >= H / 2 - 5 && py <= H / 2 + 5)) || (py == H / 2 && (px >= W / 2 - 5 && px <= W / 2 + 5))) {
                res[gid] = (int32_t)0xFFFFFFFFu;
                continue;
            }
            Path p;
            Record rec;
            p.pix_color = V(0, 0, 0); p.throughput = V(1, 1, 1); p.ray_depth = 0;
            record_new(&rec);
            uint32_t state = 0;
            rng_next(&state);
            camera_ray(&c, (int)gid, &state, &p, 1);
            if (closest_intersect(&c, &p, &rec)) {
                float shading = vdot(rec.normal, V(0.25f, 0.866f, 0.433f));
                shading = fmaxf_(0.3f, shading);
                for (int i = 0; i < 4; i++) rec.color[i] *= shading;
            } else {
                rec.emittance = 1;
                intersect_sky(&c, &p, &rec);
            }
            int rgb[3];
            for (int i = 0; i < 3; i++) {
                float v = sqrtf(rec.color[i]) * 255.0f;
                v = fminf_(fmaxf_(v, 0.0f), 255.0f);
                rgb[i] = f2i(floorf(v));
            }
            res[gid] = (int32_t)(0xFF000000u | ((uint32_t)rgb[0] << 16) | ((uint32_t)rgb[1] << 8) | (uint32_t)rgb[2]);
        }
    }
    return 0;
}

/* probes for the known-answer tests */
void oracle_rng_chain(uint32_t state, int n, uint32_t *states, float *floats) {
    for (int i = 0; i < n; i++) {
        uint32_t s = state;
        floats[i] = rng_float(&s);
        state = s;
        states[i] = s;
    }
}
/* fn: 0 sin, 1 cos, 2 atan2(x,y), 3 asin, 4 acos */
void oracle_math(int fn, int libm, const float *x, const float *y, float *out, int64_t n) {
    Math m = {libm};
    for (int64_t i = 0; i < n; i++) {
        switch (fn) {
        case 0: out[i] = m_sin(&m, x[i]); break;
        case 1: out[i] = m_cos(&m, x[i]); break;
        case 2: out[i] = m_atan2(&m, x[i], y[i]); break;
        case 3: out[i] = m_asin(&m, x[i]); break;
        default: out[i] = m_acos(&m, x[i]); break;
        }
    }
}
/* Sun_new (sky.h:19-40): out = sw, su, sv of the scene's sun */
void oracle_sun_basis(const OracleScene *s, float *out) {
    Math m = {s->math_mode == 1};
    Sun sun = sun_new(s, &m);
    v3 b[3] = {sun.sw, sun.su, sun.sv};
    for (int i = 0; i < 3; i++) { out[3 * i] = b[i].x; out[3 * i + 1] = b[i].y; out[3 * i + 2] = b[i].z; }
}
void oracle_camera_rays(const OracleScene *s, int32_t seed, float *rays) {
    OracleCounters cn;
    Ctx c;
    ctx_init(&c, s, &cn);
    int64_t n = (int64_t)s->width * s->height;
    for (int64_t gid = 0; gid < n; gid++) {
        Path p;
        uint32_t state = (uint32_t)seed + (uint32_t)gid;
        rng_next(&state);
        camera_ray(&c, (int)gid, &state, &p, 0);
        rays[gid * 6 + 0] = p.origin.x; rays[gid * 6 + 1] = p.origin.y; rays[gid * 6 + 2] = p.origin.z;
        rays[gid * 6 + 3] = p.direction.x; rays[gid * 6 + 4] = p.direction.y; rays[gid * 6 + 5] = p.direction.z;
    }
}
int oracle_num_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
int oracle_scene_struct_size(void) { return (int)sizeof(OracleScene); }

/* ------------------------------------------------------------------------------------------------------
 * tonemap filters: post_processing_filter.cl:5-51
 * ------------------------------------------------------------------------------------------------------ */
/* pow() of the filters as a fixed kernel: log2 / exp2 series in fp64 from + - * / only, rounded once to fp32;
 * operation for operation the same as dm_powf in chunkyclplugin_b200/csrc/ccu_tonemap.cuh */
static float dm_powf(float x, float y) {
    if (x != x || y != y) return NAN;
    if (x == 0.0f) return 0.0f;
    if (x == INFINITY || x == -INFINITY) return INFINITY;   /* pow(-inf, y) = +inf for y > 0 that is not an odd integer */
    if (x < 0.0f) return NAN;
    double dx = (double)x;
    int64_t bits;
    memcpy(&bits, &dx, 8);
    int e = (int)((bits >> 52) & 0x7FF) - 1023;
    int64_t mb = (bits & 0x000FFFFFFFFFFFFFLL) | 0x3FF0000000000000LL;
    double m;
    memcpy(&m, &mb, 8);
    if (m > 1.4142135623730951) { m = m * 0.5; e += 1; }
    const double t = (m - 1.0) / (m + 1.0);
    const double t2 = t * t;
    double sr = 1.0 / 15.0;
    sr = sr * t2 + 1.0 / 13.0;
    sr = sr * t2 + 1.0 / 11.0;
    sr = sr * t2 + 1.0 / 9.0;
    sr = sr * t2 + 1.0 / 7.0;
    sr = sr * t2 + 1.0 / 5.0;
    sr = sr * t2 + 1.0 / 3.0;
    sr = sr * t2 + 1.0;
    const double l2 = (double)e + (t * sr) * 2.8853900817779268;
    const double p = (double)y * l2;
    if (p > 200.0) return INFINITY;
    if (p < -200.0) return 0.0f;
    const double k = floor(p + 0.5);
    const double f = (p - k) * 0.6931471805599453;
    double r = 1.0 / 479001600.0;
    r = r * f + 1.0 / 39916800.0;
    r = r * f + 1.0 / 3628800.0;
    r = r * f + 1.0 / 362880.0;
    r = r * f + 1.0 / 40320.0;
    r = r * f + 1.0 / 5040.0;
    r = r * f + 1.0 / 720.0;
    r = r * f + 1.0 / 120.0;
    r = r * f + 1.0 / 24.0;
    r = r * f + 1.0 / 6.0;
    r = r * f + 0.5;
    r = r * f + 1.0;
    r = r * f + 1.0;
    int64_t sb = (int64_t)((int)k + 1023) << 52;
    double scale;
    memcpy(&scale, &sb, 8);
    return (float)(r * scale);
}

static inline uint32_t f2u(float f) {                /* cvt.rzi.u32.f32: saturating, NaN -> 0, toward zero */
    if (f != f || f <= 0.0f) return 0;
    if (f >= 4294967296.0f) return UINT32_MAX;
    return (uint32_t)f;
}

/* math_mode 1: libm powf instead of the fixed kernel (sensitivity studies) */
int oracle_tonemap(int width, int height, float exposure, const double *input, int type, int32_t *res, int math_mode, int nthreads) {
    if (!input || !res || width <= 0 || height <= 0 || type < 0 || type > 3) return -1;
    const int64_t n = (int64_t)width * height;
    const float inv_gamma = (float)(1.0 / 2.2);
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
#pragma omp parallel for schedule(static)
#endif
    for (int64_t gid = 0; gid < n; gid++) {
        float c[3];
        for (int i = 0; i < 3; i++) c[i] = (float)input[gid * 3 + i] * exposure;        /* double.h:19, filter :22 */
        for (int i = 0; i < 3; i++) {
            float x = c[i];
            switch (type) {
                case 0:
                    x = math_mode ? powf(x, inv_gamma) : dm_powf(x, inv_gamma);
                    break;
                case 1:
                    x = fmaxf_(0.0f, x - 0.004f);
                    x = (x * (6.2f * x + 0.5f)) / (x * (6.2f * x + 1.7f) + 0.06f);
                    break;
                case 2:
                    x = (x * (2.51f * x + 0.03f)) / (x * (2.43f * x + 0.59f) + 0.14f);
                    x = fminf_(fmaxf_(x, 0.0f), 1.0f);
                    x = math_mode ? powf(x, inv_gamma) : dm_powf(x, inv_gamma);
                    break;
                default: {
                    x = x * 16.0f;
                    const float a = 0.10f * 0.50f, b = 0.20f * 0.02f, d = 0.20f * 0.30f, g = 0.02f / 0.30f;
                    x = ((x * (0.15f * x + a) + b) / (x * (0.15f * x + 0.50f) + d)) - g;
                    const float w = ((11.2f * (0.15f * 11.2f + a) + b) / (11.2f * (0.15f * 11.2f + 0.50f) + d)) - g;
                    x = x / w;
                    break;
                }
            }
            c[i] = x;
        }
        uint32_t r = f2u(c[0] * 255.0f + 0.5f), g = f2u(c[1] * 255.0f + 0.5f), b = f2u(c[2] * 255.0f + 0.5f);   /* rgba.h:6-16 */
        if (r > 255u) r = 255u;
        if (g > 255u) g = 255u;
        if (b > 255u) b = 255u;
        res[gid] = (int32_t)((255u << 24) | (r << 16) | (g << 8) | b);
    }
    return 0;
}
