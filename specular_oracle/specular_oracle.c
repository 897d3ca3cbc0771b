/*
 * specular_oracle.c - CPU restatement of CCU_RENDER_SPECULAR (DESIGN.md section 9) and CCU_RENDER_EMITTER_SAMPLING
 * (sections 10-12).  TEST INFRASTRUCTURE ONLY.
 *
 * The reference has no specular path, so there is nothing of it to pin this file against: DESIGN.md section 9 is the contract,
 * this file restates it, and the tests hold this restatement and the CUDA kernels to each other bit for bit (plus analytic and
 * statistical checks of the restatement alone).
 *
 * Everything the reference does is taken unchanged from the parity oracle, whose source is compiled into this library as is
 * (camera, octree march, primitives, materials, BVHs, sky, sun, applyRayColor, nextPath, RNG, the arithmetic contract).
 * Restated here are only the functions whose record must also carry word 5 of the material the surface's colour came from
 * (block test, octree march, BVH walk, closestIntersect: the oracle's IntersectionRecord has no such field) and the path
 * loop with the specular event.  Each is the oracle function of the same name plus that word, operation for operation.
 * The octree march also reports the hit voxel, which the emission rule of emitter sampling needs.  The path loop knows
 * both flags; the emitter table it samples is built by the Python side of this package from the packed arrays.
 * CCU_RENDER_BIOME_TINT (section 13) restates the material evaluation with the biome colours of the hit voxel's column; the
 * block test, the octree march and the emitter samplers pass that voxel on.  CCU_RENDER_FOG (section 14) restates the fog of
 * the path loop.  CCU_RENDER_CLOUDS (section 15) restates the cloud walk and where the path loop, the shadow rays, the emitter
 * sample's ray and the fog's sun sample meet it.  The feature buffers of a denoiser (section 16) take the first segment of the path
 * loop with the biome colours and the clouds.  The guided denoiser (section 17) is restated whole: it reads only the buffers
 * it is given.
 */
#include "../oracle/chunky_oracle.c"

/* ---- biome tints (DESIGN.md section 13) ---- */
typedef struct {
    const int32_t *grid;   /* gx x gz chunks from chunk (x0, z0), index (cx - x0) * gz + (cz - z0): the chunk's tile or -1 */
    const float *tiles;    /* per tile 3 planes (foliage, grass, water) x 256 texels x {r, g, b, 0} */
    int32_t x0, z0, gx, gz;
} BiomeTiles;

/* the oracle's context plus the biome colours of this render (NULL: none); every Ctx of this file is the first member of one */
typedef struct {
    Ctx base;
    const BiomeTiles *biome;
} ExtCtx;

/* Material_sample (material.h:31-82) of a surface of voxel column vox = {x, z} (NULL: a triangle): with biome colours, a tint of
 * type 1-3 whose chunk has a tile multiplies the colour by the tile's texel, and the alpha by 255/256 */
static int material_sample_b(const Ctx *c, int material, Record *rec, float u, float v, const int *vox) {
    const BiomeTiles *b = ((const ExtCtx *)c)->biome;
    const int32_t *m = c->sc->mat_palette + material;
    uint32_t tt = (uint32_t)m[1] >> 24;
    if (!b || !vox || tt < 1 || tt > 3) return material_sample(c, material, rec, u, v);
    int cx = (vox[0] >> 4) - b->x0, cz = (vox[1] >> 4) - b->z0;
    if (cx < 0 || cz < 0 || cx >= b->gx || cz >= b->gz) return material_sample(c, material, rec, u, v);
    int32_t tile = b->grid[(size_t)cx * (size_t)b->gz + (size_t)cz];
    if (tile < 0) return material_sample(c, material, rec, u, v);
    const float *t = b->tiles + (((size_t)tile * 3 + (tt - 1)) * 256 + (size_t)(((vox[1] & 15) << 4) + (vox[0] & 15))) * 4;
    uint32_t flags = (uint32_t)m[0], tex_size = (uint32_t)m[2], col = (uint32_t)m[3];
    uint32_t normal_emittance = (uint32_t)m[4];
    c->cnt->material_samples++;
    float color[4];
    if (flags & 4u) atlas_read_uv(c, u, v, (int)col, (int)tex_size, color);
    else color_from_argb(col, color);
    if (color[3] > EPS) memcpy(rec->color, color, sizeof color);
    else return 0;
    rec->color[0] *= t[0];
    rec->color[1] *= t[1];
    rec->color[2] *= t[2];
    rec->color[3] *= 255.0f / 256.0f;
    if (flags & 2u) {
        float e[4];
        atlas_read_uv(c, u, v, (int)normal_emittance, (int)tex_size, e);
        rec->emittance = e[3];
    } else {
        rec->emittance = (float)((double)(normal_emittance & 0xFF) / 255.0);
    }
    return 1;
}

/* Material_sample (material.h:31-82) through material_sample_b; on success also word 5 of the material */
static int material_sample_w5(const Ctx *c, int material, Record *rec, uint32_t *w5, float u, float v, const int *vox) {
    if (!material_sample_b(c, material, rec, u, v, vox)) return 0;
    *w5 = (uint32_t)c->sc->mat_palette[material + 5];
    return 1;
}

/* intersect_block (block.h:30-118) */
static float intersect_block_w5(const Ctx *c, int block, int bx, int by, int bz, Record *rec, uint32_t *w5, v3 origin, v3 direction,
                                v3 inv) {
    if (block == ANY_TYPE) return NAN;
    const OracleScene *s = c->sc;
    int model_type = s->block_palette[block + 0];
    int model_ptr = s->block_palette[block + 1];
    c->cnt->block_tests++;
    v3 norm_origin = vsub(vsub(origin, vscale(direction, OFFSET)), V((float)bx, (float)by, (float)bz));
    const int vox[2] = {bx, bz};
    v3 normal = V(0, 0, 0);
    float u = 0, v = 0;
    switch (model_type) {
    default:
    case 0:
        return NAN;
    case 1: {
        AABB box = {0, 1, 0, 1, 0, 1};
        float dist = aabb_full(&box, norm_origin, origin, inv, &normal, &u, &v, 0);
        if (dist != dist) return NAN;
        rec->normal = normal;
        if (material_sample_w5(c, model_ptr, rec, w5, u, v, vox)) return dist - OFFSET;
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
                if (material_sample_w5(c, material, rec, w5, u, v, vox)) { rec->normal = normal; dist = t; hit = 1; }
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
                if (material_sample_w5(c, q[13], rec, w5, u, v, vox)) { rec->normal = normal; dist = t; hit = 1; }
            }
        }
        return hit ? dist : NAN;
    }
    }
}

/* octree_intersect (octree.h:41-109) */
static int octree_intersect_w5(const Ctx *c, const Path *ray, Record *rec, uint32_t *w5, int vox[3], int cut) {
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
        if (data != 0) {
            float dist = intersect_block_w5(c, data, bx, by, bz, rec, w5, pos, ray->direction, inv);
            /* cut (section 12): an emitter sample's shadow ray counts a block hit only before its limit */
            if (dist == dist && !(cut && !(dist_march + dist < rec->distance))) {
                rec->distance = dist_march + dist;
                rec->material = data;
                rec->hit_node = node;
                rec->hit_kind = 1;
                vox[0] = bx; vox[1] = by; vox[2] = bz;
                return 1;
            }
        }
        AABB box = {(float)(lx << level), (float)((lx + 1) << level), (float)(ly << level), (float)((ly + 1) << level),
                    (float)(lz << level), (float)((lz + 1) << level)};
        dist_march += aabb_exit(&box, vadd(pos, offset_d), inv) + OFFSET;
    }
    return 0;
}

/* bvh_intersect (bvh.h:22-113) */
static int bvh_intersect_w5(const Ctx *c, const int32_t *bvh, const Path *ray, Record *rec, uint32_t *w5, int kind) {
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
                    if (material_sample_w5(c, material, rec, w5, u, v, NULL)) {
                        rec->normal = normal; rec->distance = dist; hit = 1;
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

/* closest_intersect (kernel.h:14-24) */
static int closest_intersect_w5(const Ctx *c, const Path *ray, Record *rec, uint32_t *w5, int vox[3], int cut) {
    int hit = 0;
    c->cnt->rays++;
    hit |= octree_intersect_w5(c, ray, rec, w5, vox, cut);
    hit |= bvh_intersect_w5(c, c->sc->world_bvh, ray, rec, w5, 2);
    hit |= bvh_intersect_w5(c, c->sc->actor_bvh, ray, rec, w5, 3);
    if (hit) rec->point = vadd(ray->origin, vscale(ray->direction, rec->distance - OFFSET));
    return hit;
}

/* The specular event of a path-segment hit on a material with word 5 = w (DESIGN.md section 9, steps 1 and 3): the event
 * draws; on a specular event the emission of applyRayColor, the throughput tinted only by a metal, no sun sample, and the
 * mirror direction blended towards nextPath's cosine-weighted one by the roughness.  Returns 0 for a diffuse event (nothing
 * done), else 1 with *more = whether the path continues. */
static int specular_event(const Ctx *c, Path *p, Record *rec, uint32_t w, uint32_t *state, int *more, int emits) {
    float sp = (float)(w & 0xFF) / 255.0f, me = (float)((w >> 8) & 0xFF) / 255.0f, ro = (float)((w >> 16) & 0xFF) / 255.0f;
    int metal = 0, spec = 0;
    if (me > 0) metal = rng_float(state) < me;
    if (!metal && sp > 0) spec = rng_float(state) < sp;
    if (!metal && !spec) return 0;
    v3 col = V(rec->color[0], rec->color[1], rec->color[2]);
    v3 tinted = vmul(p->throughput, col);
    if (emits) p->pix_color = vadd(p->pix_color, vmul(vscale(col, rec->emittance * c->sc->emitter_scale), tinted));
    if (metal) p->throughput = tinted;
    v3 d = p->direction, n = rec->normal;
    v3 r = vnormalize(vsub(d, vscale(n, 2.0f * vdot(d, n))));
    Path q = *p;
    next_path(c, &q, rec, state, c->sc->max_depth); /* the two draws and the cosine-weighted direction */
    p->direction = ro > 0 ? vnormalize(vadd(vscale(r, 1.0f - ro), vscale(q.direction, ro))) : r;
    p->origin = vadd(rec->point, vscale(p->direction, OFFSET));
    p->ray_depth += 1;
    rec->distance = HUGE_VALF;
    *more = p->ray_depth < c->sc->max_depth;
    return 1;
}

/* ---- emitter sampling (DESIGN.md section 10) ---- */
#define NEE_DELTA (8.0f * OFFSET)

typedef struct {
    const int32_t *emit;   /* {x, y, z, block} per emitter, sorted by (x, y, z) */
    const int32_t *off;    /* cell lists in CSR form */
    const int32_t *list;
    int32_t g0[3], dim[3], shift;
    const int32_t *mhead;  /* section 12: per block palette position the int4 index of its primitives in mprim, or -1; NULL
                              for the table of section 10 */
    const int32_t *mprim;
} EmitterGrid;

static int voxel_cell(const EmitterGrid *g, int vx, int vy, int vz, int cl[3]) {
    int64_t d[3] = {(int64_t)vx - g->g0[0], (int64_t)vy - g->g0[1], (int64_t)vz - g->g0[2]};
    for (int a = 0; a < 3; a++) {
        if (d[a] < 0) return 0;
        cl[a] = (int)(d[a] >> g->shift);
    }
    return cl[0] < g->dim[0] && cl[1] < g->dim[1] && cl[2] < g->dim[2];
}

static int point_cell(const EmitterGrid *g, v3 x, int cl[3]) {
    if (x.x != x.x || x.y != x.y || x.z != x.z) return 0;
    int vx, vy, vz;
    floor3i(x, &vx, &vy, &vz);
    return voxel_cell(g, vx, vy, vz, cl);
}

/* the emission rule: an octree hit on an emitter voxel whose cell is within Chebyshev distance 1 of the sampled cell */
static int emitter_covered(const Ctx *c, const EmitterGrid *g, int block, const int vox[3], const int cell[3]) {
    const int32_t *bp = c->sc->block_palette, *mp = c->sc->mat_palette;
    int cube = bp[block] == 1 && ((mp[bp[block + 1]] & 2) || (mp[bp[block + 1] + 4] & 0xFF));
    if (!cube && !(g->mhead && g->mhead[block] >= 0)) return 0;
    int e[3];
    if (!voxel_cell(g, vox[0], vox[1], vox[2], e)) return 0;
    return abs(e[0] - cell[0]) <= 1 && abs(e[1] - cell[1]) <= 1 && abs(e[2] - cell[2]) <= 1;
}

/* ---- near-field emitter sampling (DESIGN.md section 11) ---- */
#define NEE_RHO2 0.015625f   /* an emitter is near when its box distance^2 is below rho^2 = (1/8)^2 */

/* next_path's cosine-weighted direction about n for the draws x1, x2 (kernel.h:50-92) */
static v3 diffuse_direction(const Ctx *c, v3 n, float x1, float x2) {
    float r = sqrtf(x1);
    float theta = 2 * PI_F * x2;
    float tx = r * m_cos(&c->math, theta);
    float ty = r * m_sin(&c->math, theta);
    float tz = sqrtf(1 - x1);
    float xx, xy, xz;
    if ((double)fabsf(n.x) > 0.1) { xx = 0; xy = 1; } else { xx = 1; xy = 0; }
    xz = 0;
    float ux = xy * n.z - xz * n.y;
    float uy = xz * n.x - xx * n.z;
    float uz = xx * n.y - xy * n.x;
    r = 1 / sqrtf((ux * ux + uy * uy) + uz * uz);
    ux *= r; uy *= r; uz *= r;
    float vx = uy * n.z - uz * n.y;
    float vy = uz * n.x - ux * n.z;
    float vz = ux * n.y - uy * n.x;
    return V((ux * tx + vx * ty) + n.x * tz, (uy * tx + vy * ty) + n.y * tz, (uz * tx + vz * ty) + n.z * tz);
}

static float vget(v3 a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }
static float clamp01(float a) { return a < 0.0f ? 0.0f : (a > 1.0f ? 1.0f : a); }

/* section 11 step 4: the direction from u2, u3, the slab test against emitter e, the material at the entry point and the
 * contribution; returns 0 when no shadow ray is traced */
static int nee_near(const Ctx *c, const int32_t *e, int n, v3 x, v3 normal, v3 T, float u2, float u3, v3 *out, v3 *w, float *limit) {
    *w = diffuse_direction(c, normal, u2, u3);
    float lo[3], hi[3];
    for (int a = 0; a < 3; a++) {
        float inv = 1.0f / vget(*w, a);
        float t0 = ((float)e[a] - vget(x, a)) * inv, t1 = ((float)(e[a] + 1) - vget(x, a)) * inv;
        if (t0 != t0 || t1 != t1) return 0;
        lo[a] = t0 < t1 ? t0 : t1;
        hi[a] = t0 < t1 ? t1 : t0;
    }
    float tn = lo[0], tf = hi[0];
    int axis = 0;
    for (int a = 1; a < 3; a++) {
        if (lo[a] > tn) { tn = lo[a]; axis = a; }
        if (hi[a] < tf) tf = hi[a];
    }
    if (!(tn <= tf && tn > 0.0f)) return 0;
    int plus = vget(*w, axis) < 0.0f;
    if (!(plus ? vget(x, axis) > (float)(e[axis] + 1) : vget(x, axis) < (float)e[axis])) return 0;
    v3 p = vadd(x, vscale(*w, tn));
    float px = clamp01(p.x - (float)e[0]), py = clamp01(p.y - (float)e[1]), pz = clamp01(p.z - (float)e[2]);
    float u, v;
    if (axis == 0) { u = plus ? pz : 1.0f - pz; v = py; }
    else if (axis == 1) { u = px; v = plus ? pz : 1.0f - pz; }
    else { u = plus ? 1.0f - px : px; v = py; }
    Record m;
    record_new(&m);
    const int vox[2] = {e[0], e[2]};
    if (!material_sample_b(c, c->sc->block_palette[e[3] + 1], &m, u, v, vox)) return 0;
    float kk = (m.emittance * c->sc->emitter_scale) * (float)n;
    *out = V((T.x * (m.color[0] * m.color[0])) * kk, (T.y * (m.color[1] * m.color[1])) * kk, (T.z * (m.color[2] * m.color[2])) * kk);
    *limit = tn - NEE_DELTA;
    return 1;
}

/* ---- model emitters (DESIGN.md section 12) ---- */
/* step 3 for a model entry e whose primitives start at int4 index h of g->mprim: the near branch (the voxel's block test along a
 * cosine-weighted direction) or a point on primitive min((int)(u1 m), m - 1) */
static int nee_model(const Ctx *c, const EmitterGrid *g, int h, const int32_t *e, int n, int near, v3 x, v3 normal, v3 T, float u1,
                     float u2, float u3, v3 *out, v3 *w, float *limit) {
    const int32_t *hd = g->mprim + 4 * (size_t)h;
    int m = hd[0];
    float ex = (float)e[0], ey = (float)e[1], ez = (float)e[2];
    if (near) {
        float lo[3] = {ex + as_float(hd[1]), ey + as_float(hd[3]), ez + as_float(hd[5])};
        float hi[3] = {ex + as_float(hd[2]), ey + as_float(hd[4]), ez + as_float(hd[6])};
        float o[3];
        for (int a = 0; a < 3; a++) {
            float xa = vget(x, a);
            o[a] = xa < lo[a] ? lo[a] - xa : (xa > hi[a] ? xa - hi[a] : 0.0f);
        }
        if ((o[0] * o[0] + o[1] * o[1]) + o[2] * o[2] < NEE_RHO2) {
            *w = diffuse_direction(c, normal, u2, u3);
            v3 inv = V(1.0f / w->x, 1.0f / w->y, 1.0f / w->z);
            Record r;
            record_new(&r);
            r.emittance = 0;
            uint32_t w5;
            float t = intersect_block_w5(c, e[3], e[0], e[1], e[2], &r, &w5, x, *w, inv);
            if (t != t || !(r.emittance > 0.0f)) return 0;
            float kk = (r.emittance * c->sc->emitter_scale) * (float)n;
            *out = V((T.x * (r.color[0] * r.color[0])) * kk, (T.y * (r.color[1] * r.color[1])) * kk, (T.z * (r.color[2] * r.color[2])) * kk);
            *limit = t - NEE_DELTA;
            return 1;
        }
    }
    int j = (int)(u1 * (float)m);
    if (j > m - 1) j = m - 1;
    const int32_t *r = hd + 8 + 16 * (size_t)j;
    const int32_t *q = r + 3;    /* the 13 words */
    int quad = r[0] == 6, axis = r[0] >> 1, plus = r[0] & 1;
    v3 l, nq = V(0, 0, 0);
    float u, v, area;
    if (quad) {
        v3 qo = V(as_float(q[0]), as_float(q[1]), as_float(q[2]));
        v3 xv = V(as_float(q[3]), as_float(q[4]), as_float(q[5]));
        v3 yv = V(as_float(q[6]), as_float(q[7]), as_float(q[8]));
        l = vadd(vadd(qo, vscale(xv, u2)), vscale(yv, u3));
        u = as_float(q[9]) + u2 * as_float(q[10]);
        v = as_float(q[11]) + u3 * as_float(q[12]);
        v3 cr = vcross(xv, yv);
        nq = vnormalize(cr);
        area = sqrtf(vdot(cr, cr));
    } else {
        float b[6];
        for (int k = 0; k < 6; k++) b[k] = as_float(q[k]);
        int a1 = axis == 0 ? 1 : 0, a2 = axis == 2 ? 1 : 2;
        float s1 = b[2 * a1 + 1] - b[2 * a1], s2 = b[2 * a2 + 1] - b[2 * a2];
        float lv[3];
        lv[axis] = b[2 * axis + plus];
        lv[a1] = b[2 * a1] + u2 * s1;
        lv[a2] = b[2 * a2] + u3 * s2;
        l = V(lv[0], lv[1], lv[2]);
        area = s1 * s2;
        if (axis == 0) { u = plus ? 1.0f - l.z : l.z; v = l.y; }
        else if (axis == 1) { u = l.x; v = plus ? 1.0f - l.z : l.z; }
        else { u = plus ? l.x : 1.0f - l.x; v = l.y; }
        int fl = r[2];
        if (fl & 4) u = 1.0f - u;
        if (fl & 2) v = 1.0f - v;
        if (fl & 1) { float t = u; u = v; v = t; }
    }
    Record mr;
    record_new(&mr);
    const int vox[2] = {e[0], e[2]};
    if (!material_sample_b(c, r[1], &mr, u, v, vox)) return 0;
    v3 dv = vsub(V(ex + l.x, ey + l.y, ez + l.z), x);
    float d2 = vdot(dv, dv);
    float dist = sqrtf(d2);
    *w = vscale(dv, 1.0f / dist);
    float cx = vdot(*w, normal);
    if (!(cx > 0.0f)) return 0;
    float ce;
    if (quad) {
        float dn = vdot(*w, nq);
        if (!(dn < -EPS)) return 0;
        ce = -dn;
    } else {
        float pw = vget(V(ex, ey, ez), axis) + vget(l, axis);
        if (!(plus ? vget(x, axis) > pw : vget(x, axis) < pw)) return 0;
        ce = fabsf(vget(*w, axis));
    }
    float kk = ((mr.emittance * c->sc->emitter_scale) * ((cx * ce) / d2)) * (((float)(n * m) * area) / PI_F);
    *out = V((T.x * (mr.color[0] * mr.color[0])) * kk, (T.y * (mr.color[1] * mr.color[1])) * kk, (T.z * (mr.color[2] * mr.color[2])) * kk);
    *limit = dist - NEE_DELTA;
    return 1;
}

/* steps 2-4: the four draws, the emitter, face and point, the material at the point and the contribution; returns 0 when
 * no shadow ray is traced.  near: an emitter whose box distance^2 is below rho^2 is sampled by nee_near (section 11).  With
 * the table of section 12 a model entry is sampled by nee_model. */
static int nee_sample(const Ctx *c, const EmitterGrid *g, int near, int b, int n, v3 x, v3 normal, v3 T, uint32_t *state, v3 *out,
                      v3 *w, float *limit) {
    float u0 = rng_float(state);
    float u1 = rng_float(state);
    float u2 = rng_float(state);
    float u3 = rng_float(state);
    int i = (int)(u0 * (float)n);
    if (i > n - 1) i = n - 1;
    const int32_t *e = g->emit + 4 * (size_t)g->list[b + i];
    if (g->mhead && g->mhead[e[3]] >= 0) return nee_model(c, g, g->mhead[e[3]], e, n, near, x, normal, T, u1, u2, u3, out, w, limit);
    float ex = (float)e[0], ey = (float)e[1], ez = (float)e[2];
    int faces[3], f = 0;
    if (x.x < ex) faces[f++] = 0; else if (x.x > (float)(e[0] + 1)) faces[f++] = 1;
    if (x.y < ey) faces[f++] = 2; else if (x.y > (float)(e[1] + 1)) faces[f++] = 3;
    if (x.z < ez) faces[f++] = 4; else if (x.z > (float)(e[2] + 1)) faces[f++] = 5;
    if (f == 0) return 0;
    if (near) {
        float o[3];
        for (int a = 0; a < 3; a++) {
            float xa = vget(x, a), lo = (float)e[a], hi = (float)(e[a] + 1);
            o[a] = xa < lo ? lo - xa : (xa > hi ? xa - hi : 0.0f);
        }
        if ((o[0] * o[0] + o[1] * o[1]) + o[2] * o[2] < NEE_RHO2) return nee_near(c, e, n, x, normal, T, u2, u3, out, w, limit);
    }
    int k = (int)(u1 * (float)f);
    if (k > f - 1) k = f - 1;
    int axis = faces[k] >> 1, plus = faces[k] & 1;
    v3 p;
    float u, v;
    if (axis == 0) { p = V((float)(e[0] + plus), ey + u2, ez + u3); u = plus ? u3 : 1.0f - u3; v = u2; }
    else if (axis == 1) { p = V(ex + u2, (float)(e[1] + plus), ez + u3); u = u2; v = plus ? u3 : 1.0f - u3; }
    else { p = V(ex + u2, ey + u3, (float)(e[2] + plus)); u = plus ? 1.0f - u2 : u2; v = u3; }
    Record m;
    record_new(&m);
    const int vox[2] = {e[0], e[2]};
    if (!material_sample_b(c, c->sc->block_palette[e[3] + 1], &m, u, v, vox)) return 0;
    v3 dv = vsub(p, x);
    float d2 = vdot(dv, dv);
    float dist = sqrtf(d2);
    *w = vscale(dv, 1.0f / dist);
    float cx = vdot(*w, normal);
    if (!(cx > 0.0f)) return 0;
    float ce = fabsf(axis == 0 ? w->x : (axis == 1 ? w->y : w->z));
    float kk = ((m.emittance * c->sc->emitter_scale) * ((cx * ce) / d2)) * ((float)(n * f) / PI_F);
    *out = V((T.x * (m.color[0] * m.color[0])) * kk, (T.y * (m.color[1] * m.color[1])) * kk, (T.z * (m.color[2] * m.color[2])) * kk);
    *limit = dist - NEE_DELTA;
    return 1;
}

/* ---- clouds (DESIGN.md section 15) ---- */
#define CLOUD_CELLS 1024            /* section 15.2: the walk visits at most this many cells, then reports a miss */
#define CLOUD_COORD_MAX 8388608.0f  /* section 15.2: 2^23, the walk reports a miss where a cell coordinate reaches it */

typedef struct {
    const uint32_t *bits;   /* 256 x 256 bits, cell (i, k) at bit (k & 255) * 256 + (i & 255) */
    float inv, y0, y1, u0, v0;
} CloudLayer;

/* the ray's parameter interval in cell c of one cell axis; d = 0: the whole line */
static void cloud_axis(float o, float d, int c, float *lo, float *hi) {
    if (d == 0.0f) { *lo = -HUGE_VALF; *hi = HUGE_VALF; return; }
    float a = ((float)c - o) / d, b = ((float)(c + 1) - o) / d;
    *lo = d > 0.0f ? a : b;
    *hi = d > 0.0f ? b : a;
}

/* the walk's first cell on one axis: the cell whose interval holds ts, or the one before it; 0 for a miss */
static int cloud_start(float o, float d, float ts, int *c, int *step) {
    if (d == 0.0f) {
        float f = floorf(o);
        if (!(o > f) || !(fabsf(o) < CLOUD_COORD_MAX)) return 0;
        *c = (int)f;
        *step = 0;
        return 1;
    }
    float x = o + d * ts;
    if (!(fabsf(x) < CLOUD_COORD_MAX)) return 0;
    *c = (int)floorf(x);
    *step = d > 0.0f ? 1 : -1;
    float lo, hi;
    cloud_axis(o, d, *c, &lo, &hi);
    if (lo > ts) *c -= *step;
    return 1;
}

/* section 15.2: the smallest t > 0 below limit at which o + d t enters the (open) box of a set cell; n = the outward normal of
 * the face entered (ties: y, then x, then z).  visited (may be NULL): the cells the walk tested. */
static int cloud_hit(const CloudLayer *cl, v3 o, v3 d, float limit, float *t, v3 *n, int *visited) {
    float ylo, yhi;
    if (visited) *visited = 0;
    if (d.y == 0.0f) {
        if (!(cl->y0 < o.y && o.y < cl->y1)) return 0;
        ylo = -HUGE_VALF;
        yhi = HUGE_VALF;
    } else {
        float a = (cl->y0 - o.y) / d.y, b = (cl->y1 - o.y) / d.y;
        if (!(a == a && b == b)) return 0;
        ylo = d.y > 0.0f ? a : b;
        yhi = d.y > 0.0f ? b : a;
    }
    float tend = yhi < limit ? yhi : limit;
    float ts = ylo > 0.0f ? ylo : 0.0f;
    if (!(ts < tend)) return 0;
    float ox = o.x * cl->inv + cl->u0, dx = d.x * cl->inv;
    float oz = o.z * cl->inv + cl->v0, dz = d.z * cl->inv;
    int i, k, si, sk;
    if (!cloud_start(ox, dx, ts, &i, &si) || !cloud_start(oz, dz, ts, &k, &sk)) return 0;
    for (int step = 0; step < CLOUD_CELLS; step++) {
        float xlo, xhi, zlo, zhi;
        if (visited) *visited = step + 1;
        cloud_axis(ox, dx, i, &xlo, &xhi);
        cloud_axis(oz, dz, k, &zlo, &zhi);
        uint32_t bit = ((uint32_t)(k & 255) << 8) | (uint32_t)(i & 255);
        if ((cl->bits[bit >> 5] >> (bit & 31u)) & 1u) {
            float tn = ylo;
            int axis = 1;
            if (xlo > tn) { tn = xlo; axis = 0; }
            if (zlo > tn) { tn = zlo; axis = 2; }
            float tf = yhi < xhi ? yhi : xhi;
            tf = tf < zhi ? tf : zhi;
            if (tn > 0.0f && tn < tf && tn < limit) {
                *t = tn;
                *n = axis == 0 ? V(dx > 0.0f ? -1.0f : 1.0f, 0, 0) : (axis == 1 ? V(0, d.y > 0.0f ? -1.0f : 1.0f, 0) : V(0, 0, dz > 0.0f ? -1.0f : 1.0f));
                return 1;
            }
        }
        float te = xhi < zhi ? xhi : zhi;
        if (!(te < tend)) return 0;
        if (xhi == te) i += si;
        if (zhi == te) k += sk;
    }
    return 0;
}

/* section 15.3: a shadow, emitter-sample or fog ray that got through is blocked by a cloud before extent; 0 without clouds */
static int cloud_blocks(const CloudLayer *cl, v3 o, v3 d, float extent) {
    float t;
    v3 n;
    return cl && cloud_hit(cl, o, d, extent, &t, &n, NULL);
}

/* ---- fog (DESIGN.md section 14) ---- */
typedef struct {
    float sigma, sky, color[3];
    int32_t fast;
} FogParams;

/* dm_expf of ccu_math.cuh, operation for operation: an fp64 series rounded once to fp32 */
static float fog_expf(float x) {
    if (x != x) return NAN;
    if (x > 89.0f) return HUGE_VALF;
    if (x < -104.0f) return 0.0f;
    const double p = (double)x * 1.4426950408889634;
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
    const int64_t bits = (int64_t)((int)k + 1023) << 52;
    double scale;
    memcpy(&scale, &bits, sizeof scale);
    return (float)(r * scale);
}

/* section 14.3: a path segment that misses sees the sky blended towards the fog colour by elevation */
static void fog_intersect_sky(const Ctx *c, const FogParams *fog, Path *p, Record *rec) {
    sky_intersect(c, p->direction, rec);
    sun_intersect(c, p->direction, rec);
    v3 d = p->direction;
    float y = d.y / sqrtf(vdot(d, d));
    float f = fog->sky * (y > 0 ? (1 - y) * (1 - y) : 1.0f);
    v3 col = vadd(vscale(V(rec->color[0], rec->color[1], rec->color[2]), 1 - f), vscale(V(fog->color[0], fog->color[1], fog->color[2]), f));
    p->pix_color = vadd(p->pix_color, vscale(vmul(col, p->throughput), rec->emittance));
}

/* section 14.2 step 3: the sun sample from the scattering point x, traced without a limit; w = the pending weight */
static void fog_sun_sample(const Ctx *c, const CloudLayer *cl, v3 x, v3 w, const Record *rec, uint32_t *state, Path *p) {
    Path q = *p;
    Record r = *rec;
    q.origin = x;
    if (!sun_sample_direction(c, &q, &r, state)) return;
    r.distance = HUGE_VALF;
    if (closest_intersect(c, &q, &r)) return;
    if (cloud_blocks(cl, q.origin, q.direction, HUGE_VALF)) return;
    sky_intersect(c, q.direction, &r);
    sun_intersect(c, q.direction, &r);
    p->pix_color = vadd(p->pix_color, vmul(w, V(r.color[0], r.color[1], r.color[2])));
}

/* one path sample: rayTracer.cl:40-107 with the specular events (spec), emitter sampling (g != NULL; near: section 11), fog
 * (fog != NULL, section 14) and clouds (cl != NULL, section 15) */
static v3 sample_pixel_ext(const Ctx *c, int gid, int32_t seed, int spec, const EmitterGrid *g, int near, const FogParams *fog,
                           const CloudLayer *cl) {
    Path p;
    Record rec;
    uint32_t w5 = 0;
    int vox[3] = {0, 0, 0};
    int nee_prev = 0, nee_cell[3] = {0, 0, 0};
    p.pix_color = V(0, 0, 0);
    p.throughput = V(1, 1, 1);
    p.ray_depth = 0;
    record_new(&rec);
    uint32_t state = (uint32_t)seed + (uint32_t)gid;
    rng_next(&state);
    camera_ray(c, gid, &state, &p, 0);
    c->cnt->samples++;
    v3 fog_p = V(0, 0, 0), fog_w = V(0, 0, 0);
    const int fog_sun = fog && (c->sun.flags & 1);
    for (;;) {
        c->cnt->segments++;
        int hit = closest_intersect_w5(c, &p, &rec, &w5, vox, 0);
        int cloud = 0;   /* section 15.3: the segment hit a cloud */
        if (cl) {
            float t;
            v3 n;
            cloud = cloud_hit(cl, p.origin, p.direction, hit ? rec.distance : HUGE_VALF, &t, &n, NULL);
            if (cloud) {
                rec.distance = t;
                rec.material = 0;
                rec.point = vadd(p.origin, vscale(p.direction, t - OFFSET));
                rec.normal = n;
                rec.color[0] = rec.color[1] = rec.color[2] = rec.color[3] = 1.0f;
                rec.emittance = 0;
                rec.hit_kind = 4;
                rec.hit_node = -1;
                w5 = 0;
                hit = 1;
            }
        }
        if (!hit) {
            rec.emittance = 1;
            if (fog) fog_intersect_sky(c, fog, &p, &rec);
            else intersect_sky(c, &p, &rec);
            break;
        }
        if (fog) {   /* section 14.2 steps 1-2 */
            float a = rec.distance * sqrtf(vdot(p.direction, p.direction));
            float e = fog->sigma * a;
            float tau = fog_expf(-e);
            if (fog_sun) {
                float u = rng_float(&state);
                fog_p = vadd(p.origin, vscale(p.direction, u * rec.distance));
                float k = fog->fast ? 1 - tau : e * fog_expf(-(fog->sigma * (u * a)));
                fog_w = vscale(vmul(p.throughput, V(fog->color[0], fog->color[1], fog->color[2])), k);
            }
            p.throughput = vscale(p.throughput, tau);
        }
        int emits = 1;
        if (g) {
            emits = !(nee_prev && rec.hit_kind == 1 && emitter_covered(c, g, rec.material, vox, nee_cell));
            nee_prev = 0;
        }
        int more;
        if (spec && specular_event(c, &p, &rec, w5, &state, &more, emits)) {
            if (fog_sun) fog_sun_sample(c, cl, fog_p, fog_w, &rec, &state, &p);
            if (!more) break;
            continue;
        }
        if (emits) {
            apply_ray_color(&p, &rec, c->sc->emitter_scale);
        } else {   /* applyRayColor without its emission term */
            p.origin = rec.point;
            p.throughput = vmul(p.throughput, V(rec.color[0], rec.color[1], rec.color[2]));
        }
        if (sun_sample_direction(c, &p, &rec, &state)) {
            Record s = rec; /* IntersectionRecord_copy keeps distance: SURVEY Q4 */
            s.point = rec.normal;
            /* the shadow ray needs no word 5 */
            if (!closest_intersect(c, &p, &s) && !cloud_blocks(cl, p.origin, p.direction, HUGE_VALF)) intersect_sky(c, &p, &s);
        }
        int cell[3];
        if (g && !cloud && p.ray_depth + 1 < c->sc->max_depth && point_cell(g, p.origin, cell)) {
            int ci = (cell[0] * g->dim[1] + cell[1]) * g->dim[2] + cell[2];
            int b = g->off[ci], n = g->off[ci + 1] - b;
            if (n > 0) {
                v3 contrib, w;
                float limit;
                nee_prev = 1;
                memcpy(nee_cell, cell, sizeof cell);
                if (nee_sample(c, g, near, b, n, p.origin, rec.normal, p.throughput, &state, &contrib, &w, &limit)) {
                    Path q = p;
                    q.direction = w;
                    Record s = rec;
                    s.distance = limit;
                    if (g->mhead) {   /* section 12: the shadow ray counts a block hit only before its limit */
                        uint32_t sw5;
                        int svox[3];
                        if (!closest_intersect_w5(c, &q, &s, &sw5, svox, 1) && !cloud_blocks(cl, q.origin, w, limit))
                            p.pix_color = vadd(p.pix_color, contrib);
                    } else if (!closest_intersect(c, &q, &s) && !cloud_blocks(cl, q.origin, w, limit)) {
                        p.pix_color = vadd(p.pix_color, contrib);
                    }
                }
            }
        }
        more = next_path(c, &p, &rec, &state, c->sc->max_depth);
        if (fog_sun) fog_sun_sample(c, cl, fog_p, fog_w, &rec, &state, &p);
        if (!more) break;
    }
    return p.pix_color;
}

static int render_ext(const OracleScene *s, const int32_t *seeds, int n_passes, int start_spp, float *res, const int32_t *gids,
                      int64_t n_gids, int nthreads, OracleCounters *out_counters, int spec, const EmitterGrid *g, int near,
                      const BiomeTiles *biome, const FogParams *fog, const CloudLayer *cl) {
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
        ExtCtx ec;
        ctx_init(&ec.base, s, &local);
        ec.biome = biome;
        const Ctx *c = &ec.base;
#pragma omp for schedule(dynamic, 64)
        for (int64_t k = 0; k < n; k++) {
            int gid = gids ? gids[k] : (int)k;
            float *px = res + (size_t)gid * 3;
            v3 buf = V(px[0], px[1], px[2]);
            for (int pass = 0; pass < n_passes; pass++) {
                v3 col = sample_pixel_ext(c, gid, seeds[pass], spec, g, near, fog, cl);
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

/* oracle_render with the specular events (same arguments, same running mean) */
int specular_render(const OracleScene *s, const int32_t *seeds, int n_passes, int start_spp, float *res, const int32_t *gids,
                    int64_t n_gids, int nthreads, OracleCounters *out_counters) {
    return render_ext(s, seeds, n_passes, start_spp, res, gids, n_gids, nthreads, out_counters, 1, NULL, 0, NULL, NULL, NULL);
}

/* oracle_render with CCU_RENDER_SPECULAR (spec), CCU_RENDER_EMITTER_SAMPLING (g != NULL), CCU_RENDER_EMITTER_NEAR_FIELD
 * (near, with g), CCU_RENDER_BIOME_TINT (biome != NULL), CCU_RENDER_FOG (fog != NULL: the scene has fog) and CCU_RENDER_CLOUDS
 * (cl != NULL: the scene has a cloud mask with a set cell) */
int flags_render(const OracleScene *s, const int32_t *seeds, int n_passes, int start_spp, float *res, const int32_t *gids,
                 int64_t n_gids, int nthreads, OracleCounters *out_counters, int spec, const EmitterGrid *g, int near,
                 const BiomeTiles *biome, const FogParams *fog, const CloudLayer *cl) {
    return render_ext(s, seeds, n_passes, start_spp, res, gids, n_gids, nthreads, out_counters, spec, g, near, biome, fog, cl);
}

/* DESIGN.md section 16: the feature buffers (albedo, normal; float[3 * W * H] each, either may be NULL) of n_passes passes.  Pass p
 * traces the camera ray of sample_pixel_ext's pass with seed seeds[p] as its first path segment: closest_intersect with the biome
 * colours (biome != NULL), then the cloud layer (cl != NULL) before the hit.  An octree / BVH hit gives the record's colour and
 * normal, a cloud (1, 1, 1) and its face normal, a miss the sky and sun disc of intersect_sky clamped to 1 and a zero normal.
 * The passes are folded in the running mean of the render loop, from zero. */
int features_render(const OracleScene *s, const int32_t *seeds, int n_passes, float *albedo, float *normal, const BiomeTiles *biome,
                    const CloudLayer *cl, int nthreads) {
    int64_t n = (int64_t)s->width * s->height;
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
#pragma omp parallel
    {
        OracleCounters local;
        memset(&local, 0, sizeof local);
        ExtCtx ec;
        ctx_init(&ec.base, s, &local);
        ec.biome = biome;
        const Ctx *c = &ec.base;
#pragma omp for schedule(dynamic, 64)
        for (int64_t gid = 0; gid < n; gid++) {
            v3 ab = V(0, 0, 0), nb = V(0, 0, 0);
            for (int pass = 0; pass < n_passes; pass++) {
                Path p;
                Record rec;
                uint32_t w5 = 0;
                int vox[3] = {0, 0, 0};
                p.pix_color = V(0, 0, 0);
                p.throughput = V(1, 1, 1);
                p.ray_depth = 0;
                record_new(&rec);
                uint32_t state = (uint32_t)seeds[pass] + (uint32_t)gid;
                rng_next(&state);
                camera_ray(c, (int)gid, &state, &p, 0);
                int hit = closest_intersect_w5(c, &p, &rec, &w5, vox, 0);
                float t;
                v3 a, nrm, cn;
                if (cl && cloud_hit(cl, p.origin, p.direction, hit ? rec.distance : HUGE_VALF, &t, &cn, NULL)) {
                    a = V(1, 1, 1);
                    nrm = cn;
                } else if (hit) {
                    a = V(rec.color[0], rec.color[1], rec.color[2]);
                    nrm = rec.normal;
                } else {
                    Record sky;
                    record_new(&sky);
                    sky_intersect(c, p.direction, &sky);
                    sun_intersect(c, p.direction, &sky);
                    a = V(fminf(sky.color[0], 1.0f), fminf(sky.color[1], 1.0f), fminf(sky.color[2], 1.0f));
                    nrm = V(0, 0, 0);
                }
                const float fs = (float)pass, fs1 = (float)(pass + 1);
                ab.x = (ab.x * fs + a.x) / fs1;
                ab.y = (ab.y * fs + a.y) / fs1;
                ab.z = (ab.z * fs + a.z) / fs1;
                nb.x = (nb.x * fs + nrm.x) / fs1;
                nb.y = (nb.y * fs + nrm.y) / fs1;
                nb.z = (nb.z * fs + nrm.z) / fs1;
            }
            if (albedo) { albedo[gid * 3] = ab.x; albedo[gid * 3 + 1] = ab.y; albedo[gid * 3 + 2] = ab.z; }
            if (normal) { normal[gid * 3] = nb.x; normal[gid * 3 + 1] = nb.y; normal[gid * 3 + 2] = nb.z; }
        }
    }
    return 0;
}

int cloud_layer_struct_size(void) { return (int)sizeof(CloudLayer); }

/* the cloud walk alone, for tests: ray r = o[3 r .. 3 r + 2] + d[3 r .. 3 r + 2] t below limit[r]; out[4 r] = t (NaN for a miss),
 * out[4 r + 1 .. 3] = the normal; visited[r] = the cells the walk tested (0 when it did not start) */
void cloud_hit_batch(const CloudLayer *cl, int64_t n, const float *o, const float *d, const float *limit, float *out, int32_t *visited) {
    for (int64_t r = 0; r < n; r++) {
        float t;
        v3 nrm = V(0, 0, 0);
        int cells = 0;
        int hit = cloud_hit(cl, V(o[3 * r], o[3 * r + 1], o[3 * r + 2]), V(d[3 * r], d[3 * r + 1], d[3 * r + 2]), limit[r], &t, &nrm, &cells);
        out[4 * r] = hit ? t : NAN;
        out[4 * r + 1] = nrm.x; out[4 * r + 2] = nrm.y; out[4 * r + 3] = nrm.z;
        visited[r] = cells;
    }
}

int fog_params_struct_size(void) { return (int)sizeof(FogParams); }

/* the fog's transmittance kernel alone, for tests */
float fog_expf_test(float x) { return fog_expf(x); }

/* ---- the guided denoiser (DESIGN.md section 17) ---- */

/* dm_expf_weight of ccu_math.cuh: fog_expf, with 0 below -87 */
static float denoise_expf(float x) { return x < -87.0f ? 0.0f : fog_expf(x); }

static float denoise_lum(float x, float y, float z) { return 0.2126f * x + 0.7152f * y + 0.0722f * z; }

/* section 2 rule 2: dot(u, v) = fma(u.z, v.z, fma(u.x, v.x, u.y * v.y)) */
static float denoise_dot(const float *u, const float *v) { return fmaf(u[2], v[2], fmaf(u[0], v[0], u[1] * v[1])); }

/* The edge-avoiding a-trous filter of section 17.1 on W x H pixels: color double[3WH] (Chunky's sample buffer), albedo and
 * normal float[3WH], iterations in [0, 8], sigma_l > 0; out double[3WH] may alias color.  Returns -1 without memory. */
int denoise(int32_t w, int32_t h, const double *color, const float *albedo, const float *normal, int32_t iterations, float sigma_l,
            double *out) {
    static const float K[5] = {1.0f / 16, 1.0f / 4, 3.0f / 8, 1.0f / 4, 1.0f / 16};
    const int64_t n = (int64_t)w * h;
    float *e = malloc((size_t)n * 4 * sizeof(float)), *f = malloc((size_t)n * 4 * sizeof(float));   /* (e.rgb, var) */
    float *lum = malloc((size_t)n * sizeof(float));
    unsigned char *valid = malloc((size_t)n);
    if (!e || !f || !lum || !valid) { free(e); free(f); free(lum); free(valid); return -1; }
    /* 1. per-pixel setup */
    for (int64_t i = 0; i < n; i++) {
        int ok = 1;
        for (int k = 0; k < 3; k++) {
            const float c = (float)color[3 * i + k], d = fmaxf(albedo[3 * i + k], 0x1p-8f);
            ok &= isfinite(c) && isfinite(albedo[3 * i + k]) && isfinite(normal[3 * i + k]);
            e[4 * i + k] = c / d;
        }
        e[4 * i + 3] = 0.0f;
        valid[i] = (unsigned char)ok;
        lum[i] = denoise_lum(e[4 * i], e[4 * i + 1], e[4 * i + 2]);
    }
    /* 2. the initial variance: luminance moments over the valid pixels of the 7x7 window inside the image */
    if (iterations > 0) {
#pragma omp parallel for schedule(static)
        for (int64_t i = 0; i < n; i++) {
            if (!valid[i]) continue;
            const int x = (int)(i % w), y = (int)(i / w);
            float s1 = 0.0f, s2 = 0.0f, m = 0.0f;
            for (int dy = -3; dy <= 3; dy++)
                for (int dx = -3; dx <= 3; dx++) {
                    const int qx = x + dx, qy = y + dy;
                    if (qx < 0 || qx >= w || qy < 0 || qy >= h) continue;
                    const int64_t q = (int64_t)qy * w + qx;
                    if (!valid[q]) continue;
                    s1 = s1 + lum[q];
                    s2 = s2 + lum[q] * lum[q];
                    m = m + 1.0f;
                }
            const float mu = s1 / m;
            e[4 * i + 3] = fmaxf(0.0f, s2 / m - mu * mu);
        }
    }
    /* 3. the iterations, step 2^it */
    for (int it = 0; it < iterations; it++) {
        const int step = 1 << it;
#pragma omp parallel for schedule(static)
        for (int64_t i = 0; i < n; i++) {
            const float *ep = e + 4 * i;
            float *fp = f + 4 * i;
            if (!valid[i]) { memcpy(fp, ep, 4 * sizeof(float)); continue; }
            const int x = (int)(i % w), y = (int)(i / w);
            const float *ap = albedo + 3 * i, *np_ = normal + 3 * i;
            const float lp = denoise_lum(ep[0], ep[1], ep[2]);
            const float dl_den = sigma_l * sqrtf(ep[3]) + 1e-4f;
            const int sky_p = np_[0] == 0.0f && np_[1] == 0.0f && np_[2] == 0.0f;
            float sw = 0.0f, sv = 0.0f, s[3] = {0.0f, 0.0f, 0.0f};
            for (int dy = -2; dy <= 2; dy++)
                for (int dx = -2; dx <= 2; dx++) {
                    const int qx = x + dx * step, qy = y + dy * step;
                    if (qx < 0 || qx >= w || qy < 0 || qy >= h) continue;
                    const int64_t q = (int64_t)qy * w + qx;
                    if (!valid[q]) continue;
                    const float *eq = e + 4 * q;
                    float wt;
                    if (dx == 0 && dy == 0) {
                        wt = 9.0f / 64.0f;
                    } else {
                        const float *aq = albedo + 3 * q, *nq = normal + 3 * q;
                        const float dl = fabsf(lp - denoise_lum(eq[0], eq[1], eq[2])) / dl_den;
                        const float da3[3] = {ap[0] - aq[0], ap[1] - aq[1], ap[2] - aq[2]};
                        const float da = denoise_dot(da3, da3) / 0.01f;
                        float wn = 1.0f;
                        if (!(sky_p && nq[0] == 0.0f && nq[1] == 0.0f && nq[2] == 0.0f)) {
                            wn = fmaxf(0.0f, denoise_dot(np_, nq));
                            for (int r = 0; r < 7; r++) wn = wn * wn;
                        }
                        wt = K[dx + 2] * K[dy + 2] * wn * denoise_expf(-(dl + da));
                    }
                    s[0] = s[0] + wt * eq[0];
                    s[1] = s[1] + wt * eq[1];
                    s[2] = s[2] + wt * eq[2];
                    sv = sv + wt * wt * eq[3];
                    sw = sw + wt;
                }
            fp[0] = s[0] / sw;
            fp[1] = s[1] / sw;
            fp[2] = s[2] / sw;
            fp[3] = sv / (sw * sw);
        }
        float *t = e; e = f; f = t;
    }
    /* 4. remodulation */
    for (int64_t i = 0; i < n; i++)
        for (int k = 0; k < 3; k++) out[3 * i + k] = (double)(e[4 * i + k] * fmaxf(albedo[3 * i + k], 0x1p-8f));
    free(e); free(f); free(lum); free(valid);
    return 0;
}

int biome_tiles_struct_size(void) { return (int)sizeof(BiomeTiles); }

int emitter_grid_struct_size(void) { return (int)sizeof(EmitterGrid); }
