// ccu_march.cuh - the octree march loop (octree.h:66-107) on the commit-time march layout ("air layout").
//
// The march loop only needs to know, for the voxel under the ray, whether its leaf is air and - if so - the level of
// that air leaf (octree.h:89-106: an air leaf is left through its cube, anything else goes to the block test).  The
// layout built at commit (chunkycu.cu, build_air_layout) answers that with at most ONE global load below the top table:
//
//   air_top[]     dense table over the cells of level air_cell_level (>= 4), index (x*dim + y)*dim + z.  Entry:
//                   bit 31 set   leaf  {bits 30..26: level of the air leaf, 31 = not air}
//                   bit 31 clear index of a brick (air_cell_level == 4) or of a 64-ary node (deeper worlds)
//   air_wide[]    64-ary nodes (two octree levels per load), only for worlds whose top table would not fit with 16^3
//                 cells (octree depth > 11); same entry encoding, entries at level 4 refer to bricks
//   air_bricks[]  one 1-KiB brick per 16^3 cell that is not a single leaf: 64 blocks of 4^3 voxels, block index
//                 ((x>>2)&3)<<4 | ((y>>2)&3)<<2 | ((z>>2)&3), 4 words per block (word = x&3), 2 bits per voxel at bit
//                 position 2*(((y&3)<<2) | (z&3)):  0 = not air, 1 = air leaf of level 0, 2 = air leaf of level 1.
//                 A 4^3 block that lies inside ONE leaf of level 2 or 3 has all four words = 0 (not air) or
//                 0xC0000000 | level (air); mixed words never have their top code = 3, so `word >= 0xC0000000` tells.
//
// The arithmetic of a step is exactly the reference's (same operations on the same values in the same order, so the
// marched distance is bit-identical); only loop invariants are hoisted and the leaf lookup is replaced.
#pragma once
#include "ccu_device.cuh"

namespace ccu {

#define CCU_BRICK_UNIFORM 0xC0000000u

struct LeanRay {
    float3 o, d, inv, doff;   // doff = d * OFFSET (octree.h:73, loop invariant)
    float t, limit;
    int steps;
    int fmx, fmy, fmz;        // -1 when the leaf cube is left through its upper plane on that axis, else 0
    float nmx, nmy, nmz;      // second operand of the exit term's fmaxf: -inf or NaN (lean_exit_axis)
};

__device__ __forceinline__ void lean_prepare(LeanRay &r) {
    r.doff = r.d * CCU_OFFSET;
    r.fmx = r.inv.x < 0.0f ? 0 : -1;
    r.fmy = r.inv.y < 0.0f ? 0 : -1;
    r.fmz = r.inv.z < 0.0f ? 0 : -1;
    r.nmx = r.inv.x < 0.0f ? -inff_() : nanf_();
    r.nmy = r.inv.y < 0.0f ? -inff_() : nanf_();
    r.nmz = r.inv.z < 0.0f ? -inff_() : nanf_();
}

// AABB_exit (primitives.h:52-61) along one axis for the offset position q of a voxel b of the leaf cube [lo, hi):
// fmax((lo-q)*inv, (hi-q)*inv).  The far-plane term ((hi-q)*inv for inv >= 0, (lo-q)*inv for inv < 0) is that maximum
// except where it is NaN, and then `nm` (lean_prepare) gives the reference's result:
//  - q finite (lo <= q < hi): NaN only for inv = -inf and q == lo, where the reference's other term is -inf, so
//    nm = -inf for inv < 0.  An infinite q never gets here: f2i saturates and the cube test ends the march.
//  - inv NaN, or q NaN (a NaN origin component, or 0 * inf in o + d * t): both of the reference's terms are NaN, and
//    its fmin drops the axis; nm = NaN keeps the NaN, which fminf drops too.  nm = NaN for inv >= 0 and inv NaN;
//    march_begin_core makes inv NaN on an axis whose origin component is NaN, so that case gets NaN too (and costs
//    nothing per step or per load).  The one case left, q NaN from 0 * inf for d = -0 (t infinite), maps to -inf instead,
//    but once t is infinite every axis with a finite non-zero d leaves the cube at the next step and every other
//    axis's q is NaN, so the march only meets voxel (0,0,0) with a NaN position, whose block test misses, until
//    draw_depth: a miss either way.
// The plane is ((b >> level) + far) << level = (b with its low `level` bits cleared / set) + far.
__device__ __forceinline__ float lean_exit_axis(int b, int low, int fm, float q, float inv, float nm) {
    const int plane = ((b & ~low) | (low & fm)) - fm;
    return fmaxf(((float)plane - q) * inv, nm);
}

// One iteration of octree.h:66-107.  Returns 0 = air leaf left (keep marching), 1 = non-air leaf reached (ray not
// advanced; the block test looks the leaf up), 2 = ray finished without a hit.
// TOPS: `top` is the air top table staged in shared memory, otherwise it is read from global memory.
// DEEP: air_cell_level > 4 (64-ary nodes between the top table and the bricks).
template <bool DEEP, bool TOPS>
__device__ __forceinline__ int lean_probe(const DScene &s, const unsigned *__restrict__ top, LeanRay &r) {
    if (r.steps >= s.draw_depth || r.t > r.limit) return 2;
    const float3 pos = r.o + r.d * r.t;
    const float3 q = pos + r.doff;
    const int bx = f2i(floorf(q.x)), by = f2i(floorf(q.y)), bz = f2i(floorf(q.z));
    if (((bx | by | bz) >> s.depth) != 0) return 2;
    const int tl = s.air_top_log2;
    unsigned e;
    if (!DEEP) {
        const unsigned ti = ((((unsigned)(bx >> 4) << tl) + (unsigned)(by >> 4)) << tl) + (unsigned)(bz >> 4);
        e = TOPS ? top[ti] : __ldg(top + ti);
    } else {
        int lvl = s.air_cell_level;
        const unsigned ti = ((((unsigned)(bx >> lvl) << tl) + (unsigned)(by >> lvl)) << tl) + (unsigned)(bz >> lvl);
        e = __ldg(top + ti);
        while (lvl > 4 && !(e & CCU_WIDE_LEAF)) {
            lvl -= 2;
            e = __ldg(s.air_wide + (e * 64u + (unsigned)((((bx >> lvl) & 3) << 4) | (((by >> lvl) & 3) << 2) | ((bz >> lvl) & 3))));
        }
    }
    int level;   // level of the air leaf, -1 = not air
    if (e & CCU_WIDE_LEAF) {
        level = ((int)(e << 1)) >> 27;       // bits 30..26 as a signed field: 31 = -1 = not air
    } else {
        const unsigned wi = (unsigned)(((bx & 12) << 4) | ((by & 12) << 2) | (bz & 12) | (bx & 3));
        const unsigned w = __ldg(s.air_bricks + (e * 256u + wi));
        const int code = (int)((w >> ((((by & 3) << 2) | (bz & 3)) * 2)) & 3u);
        level = w >= CCU_BRICK_UNIFORM ? (int)(w & 31u) : code - 1;
    }
    if (level < 0) return 1;
    const int low = (1 << level) - 1;
    const float ex = lean_exit_axis(bx, low, r.fmx, q.x, r.inv.x, r.nmx);
    const float ey = lean_exit_axis(by, low, r.fmy, q.y, r.inv.y, r.nmy);
    const float ez = lean_exit_axis(bz, low, r.fmz, q.z, r.inv.z, r.nmz);
    r.t += fminf(ex, fminf(ey, ez)) + CCU_OFFSET;
    r.steps++;
    return 0;
}

// The same iteration as straight-line code for the shallow layouts (top table over 16^3 cells + bricks): every lane of the warp
// executes every instruction, lanes without a ray in flight (`active` false) or whose ray ends compute on harmless values and
// commit nothing.  No branch inside the step means no divergence stacks, no fetch redirects and one load latency per iteration
// for the whole warp; the lanes whose cell is a single leaf read brick word 0 (one broadcast sector) instead of skipping the load.
// `done`: the lane's state before the step (only read when !active); returns the state after it.
template <bool TOPS>
__device__ __forceinline__ int lean_step_flat(const DScene &s, const unsigned *__restrict__ top, LeanRay &r, bool active, int done) {
    const bool fin0 = r.steps >= s.draw_depth || r.t > r.limit;
    const float3 pos = r.o + r.d * r.t;
    const float3 q = pos + r.doff;
    const int bx = f2i(floorf(q.x)), by = f2i(floorf(q.y)), bz = f2i(floorf(q.z));
    const bool fin = fin0 || (((bx | by | bz) >> s.depth) != 0);
    const int tl = s.air_top_log2;
    // out-of-cube coordinates (finished lanes only) are folded into the table
    const unsigned ti = (((((unsigned)(bx >> 4) << tl) + (unsigned)(by >> 4)) << tl) + (unsigned)(bz >> 4)) & ((1u << (3 * tl)) - 1u);
    const unsigned e = TOPS ? top[ti] : __ldg(top + ti);
    const bool leaf = (e & CCU_WIDE_LEAF) != 0;
    const unsigned wi = (unsigned)(((bx & 12) << 4) | ((by & 12) << 2) | (bz & 12) | (bx & 3));
    const unsigned w = __ldg(s.air_bricks + (leaf ? 0u : e * 256u + wi));
    const int code = (int)((w >> ((((by & 3) << 2) | (bz & 3)) * 2)) & 3u);
    const int lvl_brick = w >= CCU_BRICK_UNIFORM ? (int)(w & 31u) : code - 1;
    const int level = leaf ? ((int)(e << 1)) >> 27 : lvl_brick;       // -1 = not air
    const int low = (1 << (level & 31)) - 1;
    const float ex = lean_exit_axis(bx, low, r.fmx, q.x, r.inv.x, r.nmx);
    const float ey = lean_exit_axis(by, low, r.fmy, q.y, r.inv.y, r.nmy);
    const float ez = lean_exit_axis(bz, low, r.fmz, q.z, r.inv.z, r.nmz);
    const float tn = r.t + (fminf(ex, fminf(ey, ez)) + CCU_OFFSET);
    const bool adv = active && !fin && level >= 0;
    r.t = adv ? tn : r.t;
    r.steps += adv ? 1 : 0;
    return active ? (fin ? 2 : (level < 0 ? 1 : 0)) : done;
}

// Octree_octreeIntersect (octree.h:41-109) for the thread-per-ray kernels (first-hit, preview, thread-per-pixel render):
// the air steps run on the march layout, the leaf value / block test of a non-air leaf on the value-carrying layout.
// hi.node is left at -1 (the first-hit kernel finds the treeData index of the hit voxel by one root descent).
template <bool DEEP>
__device__ __forceinline__ bool octree_intersect_lean(const DScene &s, float3 origin, float3 direction, Record &rec, HitInfo &hi) {
    March m;
    if (!march_begin(s, m, origin, direction, rec.distance)) return false;
    LeanRay r;
    r.o = m.o; r.d = m.d; r.inv = m.inv; r.t = m.t; r.limit = m.limit; r.steps = m.steps;
    lean_prepare(r);
    for (;;) {
        const int st = lean_probe<DEEP, false>(s, s.air_top, r);
        if (st == 0) continue;
        if (st == 2) return false;
        m.t = r.t; m.steps = r.steps;
        const Cell c = march_cell(m);
        int level;
        const int data = find_leaf_wide(s, c.bx, c.by, c.bz, level);
        float t;
        if (march_block(s, m, data, level, rec.surf, t)) {
            rec.distance = t;
            rec.material = data;
            hi.node = -1;
            hi.kind = 1;
            hi.bx = c.bx; hi.by = c.by; hi.bz = c.bz;
            return true;
        }
        r.t = m.t; r.steps = m.steps;
    }
}

// kernel.h:14-24 on the commit-time layouts
template <bool DEEP>
__device__ __forceinline__ bool closest_intersect_lean(const DScene &s, float3 origin, float3 direction, Record &rec, HitInfo &hi) {
    bool hit = octree_intersect_lean<DEEP>(s, origin, direction, rec, hi);
    int kind = 0;
    if (bvh_pair(s, origin, direction, rec.distance, rec.surf, kind)) {
        hit = true;
        hi.kind = kind;
        hi.node = -1;
    }
    if (hit) rec.point = origin + direction * (rec.distance - CCU_OFFSET);
    return hit;
}

// MODE 0: the reference's own node array (root descent per step); 1: commit-time layouts; 2: commit-time layouts, deep world
template <int MODE>
__device__ __forceinline__ bool closest_intersect_mode(const DScene &s, float3 origin, float3 direction, Record &rec, HitInfo &hi) {
    if (MODE == 0) return closest_intersect_ref(s, origin, direction, rec, hi);
    return closest_intersect_lean<MODE == 2>(s, origin, direction, rec, hi);
}

// one path sample for pixel gid, thread-sequential: rayTracer.cl:40-107 (+ kernel.h:33-98, sky.h:68-93)
template <int MODE>
__device__ __forceinline__ float3 sample_pixel(const DScene &s, int gid, int seed) {
    float3 color = f3(0, 0, 0), throughput = f3(1, 1, 1);
    int ray_depth = 0;
    uint32_t rng = (uint32_t)seed + (uint32_t)gid;
    rng_next(rng);
    float3 origin, direction;
    camera_ray<false>(s, gid, rng, origin, direction);
    Record rec;
    rec.distance = inff_();
    rec.material = 0;
    rec.point = f3(0, 0, 0);
    rec.surf.normal = f3(0, 0, 0);
    rec.surf.color = make_float4(0, 0, 0, 0);
    rec.surf.emittance = 0;
    HitInfo hi = {-1, 0, 0, 0, 0};
    for (;;) {
        if (!closest_intersect_mode<MODE>(s, origin, direction, rec, hi)) {
            // miss: emittance = 1, sky (+ sun disc) added through the throughput (rayTracer.cl:95-97, kernel.h:26-31)
            float3 sky = sky_radiance(s, direction);
            color = color + (sky * throughput) * 1.0f;
            break;
        }
        // kernel.h:33-44
        origin = rec.point;
        float3 col = f3(rec.surf.color.x, rec.surf.color.y, rec.surf.color.z);
        throughput = throughput * col;
        color = color + (col * (rec.surf.emittance * s.emitter_scale)) * throughput;
        // sun sampling + shadow ray (sky.h:68-93, rayTracer.cl:101-106)
        if (s.sun_flags & 1) {
            float x1 = rng_float(rng);
            float x2 = rng_float(rng);
            float3 d = sun_sample_direction(s, x1, x2);
            float shadow_emittance = fabsf(dot3(d, rec.surf.normal));
            Record sh = rec;                          // keeps the surface hit's distance as the ray limit (SURVEY Q4)
            HitInfo shi;
            if (!closest_intersect_mode<MODE>(s, origin, d, sh, shi)) {
                float3 sky = sky_radiance(s, d);
                color = color + (sky * throughput) * shadow_emittance;
            }
        }
        // kernel.h:46-98 diffuse bounce
        float x1 = rng_float(rng);
        float x2 = rng_float(rng);
        direction = diffuse_direction(rec.surf.normal, x1, x2);
        origin = rec.point + direction * CCU_OFFSET;
        ray_depth += 1;
        rec.distance = inff_();
        if (!(ray_depth < s.max_depth)) break;
    }
    return color;
}

}  // namespace ccu
