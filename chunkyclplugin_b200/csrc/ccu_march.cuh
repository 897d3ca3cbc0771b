// ccu_march.cuh - the octree march loop (octree.h:66-107) on the commit-time march layout ("air layout").
//
// The march loop only needs to know, for the voxel under the ray, whether its leaf is air and - if so - the level of
// that air leaf (octree.h:89-106: an air leaf is left through its cube, anything else goes to the block test).  The
// layout built at commit (chunkycu.cu, build_air_layout) answers that with at most ONE global load below the top table:
//
//   air_top[]     dense table over the cells of level air_cell_level (>= 4), index (x*dim + y)*dim + z.
//                 Shallow worlds (air_cell_level == 4): every entry is the word offset of a brick in air_bricks; a cell that
//                 is a single leaf refers to the constant brick of that leaf (every voxel = its level, or not air).
//                 Deep worlds (air_cell_level > 4), and the entries of air_wide[]:
//                   bit 31 set   leaf  {bits 30..26: level of the air leaf, 31 = not air}
//                   bit 31 clear word offset of a brick (entries at level 4) or index of a 64-ary node (above)
//   air_wide[]    64-ary nodes (two octree levels per load), only for worlds whose top table would not fit with 16^3
//                 cells (octree depth > 11)
//   air_bricks[]  one 2-KiB brick (CCU_BRICK_WORDS words) per 16^3 cell: 4 bits per voxel, the level of the voxel's air
//                 leaf (0..14) or CCU_AIR_SOLID (15) = not air.  Voxel (x, y, z) of the cell is the nibble z & 7 of word
//                 (x << 5) | (y << 1) | (z >> 3) (air_brick_word / air_brick_level): one shift and one mask decode it.
//
// The arithmetic of a step is exactly the reference's (same operations on the same values in the same order, so the
// marched distance is bit-identical); only loop invariants are hoisted and the leaf lookup is replaced.
#pragma once
#include "ccu_device.cuh"

namespace ccu {

#define CCU_BRICK_WORDS 512u   // words of a brick: 16^3 voxels x 4 bits
#define CCU_AIR_SOLID 15        // brick code of a voxel that is not air

// word of a brick that holds voxel (x, y, z) of its cell (only the low 4 bits of each coordinate count)
__host__ __device__ __forceinline__ unsigned air_brick_word(int x, int y, int z) {
    return (((unsigned)x & 15u) << 5) | (((unsigned)y & 15u) << 1) | (((unsigned)z >> 3) & 1u);
}
// code of voxel z of brick word w: the level of its air leaf, CCU_AIR_SOLID = not air (the rotation takes z << 2 mod 32)
__host__ __device__ __forceinline__ int air_brick_level(unsigned w, int z) {
#ifdef __CUDA_ARCH__
    return (int)(__funnelshift_r(w, w, (unsigned)z << 2) & 15u);
#else
    return (int)((w >> ((z & 7) * 4)) & 15u);
#endif
}

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
// DEEP: air_cell_level > 4 (64-ary nodes between the top table and the bricks).  draw_depth: as in lean_step_flat.
template <bool DEEP, bool TOPS>
__device__ __forceinline__ int lean_probe(const DScene &s, const unsigned *__restrict__ top, LeanRay &r, int draw_depth) {
    if (r.steps >= draw_depth || r.t > r.limit) return 2;
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
    int level;   // level of the air leaf
    if (DEEP && (e & CCU_WIDE_LEAF)) {
        level = (int)((e >> 26) & 31u);       // 31 = not air
        if (level == 31) return 1;
    } else {
        level = air_brick_level(__ldg(s.air_bricks + (e + air_brick_word(bx, by, bz))), bz);
        if (level == CCU_AIR_SOLID) return 1;
    }
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
// for the whole warp; the lanes whose cell is a single leaf read the constant brick of that leaf.
// `done`: the lane's state before the step (only read when !active); returns the state after it.
// The loop invariants come in as values so that a caller's loop keeps them in registers: the step ends once
// r.steps >= draw_depth (the queue kernel biases steps by -draw_depth and passes 0), and `outside` = ~(2^depth - 1) holds the
// bits a voxel coordinate inside the octree cube never has.
// TOP16: the top table has 16^3 cells (s.air_top_log2 == 4) and is staged in shared memory; it is indexed with immediate
// shifts.  Otherwise it is read from global memory, with s.air_top_log2 cells per axis.
template <bool TOP16>
__device__ __forceinline__ int lean_step_flat(const DScene &s, const unsigned *__restrict__ top, LeanRay &r, bool active, int done,
                                              int draw_depth, unsigned outside) {
    const bool fin0 = r.steps >= draw_depth || r.t > r.limit;
    const float3 pos = r.o + r.d * r.t;
    const float3 q = pos + r.doff;
    const int bx = f2i(floorf(q.x)), by = f2i(floorf(q.y)), bz = f2i(floorf(q.z));
    const bool fin = fin0 || ((unsigned)(bx | by | bz) & outside) != 0;
    // out-of-cube coordinates (finished lanes only) are folded into the table
    unsigned ti;
    if (TOP16) {
        ti = (((unsigned)bx << 4) & 0xF00u) | ((unsigned)by & 0xF0u) | (((unsigned)bz >> 4) & 0xFu);
    } else {
        const int tl = s.air_top_log2;
        ti = (((((unsigned)(bx >> 4) << tl) + (unsigned)(by >> 4)) << tl) + (unsigned)(bz >> 4)) & ((1u << (3 * tl)) - 1u);
    }
    const unsigned e = TOP16 ? top[ti] : __ldg(top + ti);
    const int level = air_brick_level(__ldg(s.air_bricks + (e + air_brick_word(bx, by, bz))), bz);   // CCU_AIR_SOLID = not air
    const int low = (1 << level) - 1;
    const float ex = lean_exit_axis(bx, low, r.fmx, q.x, r.inv.x, r.nmx);
    const float ey = lean_exit_axis(by, low, r.fmy, q.y, r.inv.y, r.nmy);
    const float ez = lean_exit_axis(bz, low, r.fmz, q.z, r.inv.z, r.nmz);
    const float tn = r.t + (fminf(ex, fminf(ey, ez)) + CCU_OFFSET);
    const bool air = level != CCU_AIR_SOLID;
    const bool adv = active && !fin && air;
    r.t = adv ? tn : r.t;
    r.steps += adv ? 1 : 0;
    return active ? (fin ? 2 : (air ? 0 : 1)) : done;
}

// Octree_octreeIntersect (octree.h:41-109) for the thread-per-ray kernels (first-hit, preview, thread-per-pixel render):
// the air steps run on the march layout, the leaf value / block test of a non-air leaf on the value-carrying layout.
// hi.node is left at -1 (the first-hit kernel finds the treeData index of the hit voxel by one root descent).
template <bool DEEP, class V, bool CUT = false>
__device__ __forceinline__ bool octree_intersect_lean(const DScene &s, float3 origin, float3 direction, RecordT<V::spec> &rec, HitInfo &hi) {
    March m;
    if (!march_begin(s, m, origin, direction, rec.distance)) return false;
    LeanRay r;
    r.o = m.o; r.d = m.d; r.inv = m.inv; r.t = m.t; r.limit = m.limit; r.steps = m.steps;
    lean_prepare(r);
    for (;;) {
        const int st = lean_probe<DEEP, false>(s, s.air_top, r, s.draw_depth);
        if (st == 0) continue;
        if (st == 2) return false;
        m.t = r.t; m.steps = r.steps;
        const Cell c = march_cell(m);
        int level;
        const int data = find_leaf_wide(s, c.bx, c.by, c.bz, level);
        float t;
        if (march_block<V, CUT>(s, m, data, level, rec.surf, t, CUT)) {
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
template <bool DEEP, class V, bool CUT = false>
__device__ __forceinline__ bool closest_intersect_lean(const DScene &s, float3 origin, float3 direction, RecordT<V::spec> &rec, HitInfo &hi) {
    bool hit = octree_intersect_lean<DEEP, V, CUT>(s, origin, direction, rec, hi);
    int kind = 0;
    if (bvh_pair(s, origin, direction, rec.distance, rec.surf, kind)) {
        hit = true;
        hi.kind = kind;
        hi.node = -1;
    }
    if (hit) rec.point = origin + direction * (rec.distance - CCU_OFFSET);
    return hit;
}

// MODE 0: the reference's own node array (root descent per step); 1: commit-time layouts; 2: commit-time layouts, deep world.
// CUT: an octree hit counts only before rec.distance (march_block; emitter-sample shadow rays of CCU_RENDER_EMITTER_MODELS).
template <int MODE, class V, bool CUT = false>
__device__ __forceinline__ bool closest_intersect_mode(const DScene &s, float3 origin, float3 direction, RecordT<V::spec> &rec, HitInfo &hi) {
    if (MODE == 0) return closest_intersect_ref<V, CUT>(s, origin, direction, rec, hi);
    return closest_intersect_lean<MODE == 2, V, CUT>(s, origin, direction, rec, hi);
}

// DESIGN §15: whether a shadow, emitter-sample or fog ray that the octree and the BVHs let through is blocked by a cloud before
// `extent` (unbounded, except for an emitter-sample ray: the distance of its target).  Always false without V::clouds.
template <class V>
__device__ __forceinline__ bool cloud_blocks(const CloudView &cv, float3 o, float3 d, float extent) {
    if constexpr (V::clouds) {
        float t;
        float3 n;
        return cloud_hit(cv, o, d, extent, t, n);
    }
    return false;
}

// closestIntersect of a path segment with the cloud layer (DESIGN §15.3): a cloud hit strictly nearer than the octree / BVH hit
// (any, on a miss) replaces it by a white surface that emits nothing, hi.kind 4.
template <int MODE, class V>
__device__ __forceinline__ bool segment_intersect(const DScene &s, const CloudView &cv, float3 origin, float3 direction, RecordT<V::spec> &rec,
                                                  HitInfo &hi) {
    bool hit = closest_intersect_mode<MODE, V>(s, origin, direction, rec, hi);
    float t;
    float3 n;
    if (cloud_hit(cv, origin, direction, hit ? rec.distance : inff_(), t, n)) {
        rec.distance = t;
        rec.material = 0;
        rec.point = origin + direction * (t - CCU_OFFSET);
        rec.surf.normal = n;
        rec.surf.color = make_float4(1, 1, 1, 1);
        rec.surf.emittance = 0;
        surf_set_spec(rec.surf, 0u);
        hi.node = -1;
        hi.kind = 4;
        hit = true;
    }
    return hit;
}

// The fog's sun sample at the end of a hit (DESIGN §14 step 3): the two draws, the sun direction as the surface sun sample
// draws it, and a ray from the scattering point p without a limit; an escaped ray adds the pending weight w times the sky
// (and sun disc) along it.  `rec` is a copy of the hit's record.
template <int MODE, class V>
__device__ __forceinline__ void fog_sun_sample(const DScene &s, const CloudView &cv, uint32_t &rng, float3 p, float3 w, RecordT<V::spec> rec,
                                               float3 &color) {
    const float x1 = rng_float(rng);
    const float x2 = rng_float(rng);
    const float3 d = sun_sample_direction(s, x1, x2);
    rec.distance = inff_();
    HitInfo hi;
    if (!closest_intersect_mode<MODE, V>(s, p, d, rec, hi) && !cloud_blocks<V>(cv, p, d, inff_())) color = color + w * sky_radiance(s, d);
}

// one path sample for pixel gid, thread-sequential: rayTracer.cl:40-107 (+ kernel.h:33-98, sky.h:68-93), with the specular events,
// emitter sampler, biome colours, fog and clouds the Shade V switches on (DESIGN §5)
template <int MODE, class V>
__device__ __forceinline__ float3 sample_pixel(const DScene &s, const EmitView &g, const CloudView &cv, int gid, int seed) {
    float3 color = f3(0, 0, 0), throughput = f3(1, 1, 1);
    int ray_depth = 0;
    uint32_t rng = (uint32_t)seed + (uint32_t)gid;
    rng_next(rng);
    float3 origin, direction;
    camera_ray<false>(s, gid, rng, origin, direction);
    RecordT<V::spec> rec;
    rec.distance = inff_();
    rec.material = 0;
    rec.point = f3(0, 0, 0);
    rec.surf.normal = f3(0, 0, 0);
    rec.surf.color = make_float4(0, 0, 0, 0);
    rec.surf.emittance = 0;
    surf_set_spec(rec.surf, 0u);
    HitInfo hi = {-1, 0, 0, 0, 0};
    bool nee_prev = false;   // NEE: the hit this segment left sampled the list of cell nee_cell
    int3 nee_cell = make_int3(0, 0, 0);
    float3 fog_p = f3(0, 0, 0), fog_w = f3(0, 0, 0);   // fog: the hit's scattering point and its pending weight (DESIGN §14)
    for (;;) {
        bool hit;
        if constexpr (V::clouds) hit = segment_intersect<MODE, V>(s, cv, origin, direction, rec, hi);
        else hit = closest_intersect_mode<MODE, V>(s, origin, direction, rec, hi);
        if (!hit) {
            // miss: emittance = 1, sky (+ sun disc) added through the throughput (rayTracer.cl:95-97, kernel.h:26-31)
            float3 sky = sky_radiance(s, direction);
            if constexpr (V::fog) {   // the sky blended towards the fog colour by elevation (§14.3)
                const float y = direction.y / sqrtf(dot3(direction, direction));
                const float f = s.fog_sky * (y > 0 ? (1 - y) * (1 - y) : 1.0f);
                sky = sky * (1 - f) + s.fog_color * f;
            }
            color = color + (sky * throughput) * 1.0f;
            break;
        }
        if constexpr (V::fog) {   // §14.2 steps 1-2: the scattering draw, then the segment's transmittance
            const float a = rec.distance * sqrtf(dot3(direction, direction));
            const float e = s.fog_sigma * a;
            const float tau = dm_expf(-e);
            if (s.sun_flags & 1) {
                const float u = rng_float(rng);
                fog_p = origin + direction * (u * rec.distance);
                const float k = s.fog_fast ? 1 - tau : e * dm_expf(-(s.fog_sigma * (u * a)));
                fog_w = (throughput * s.fog_color) * k;
            }
            throughput = throughput * tau;
        }
        bool emits = true;   // NEE: an emitter the previous hit's sample covered delivers no emission here
        if constexpr (V::nee) {
            emits = !(nee_prev && hi.kind == 1 && emitter_covered<V::nee>(s, g, rec.material, hi.bx, hi.by, hi.bz, nee_cell));
            nee_prev = false;
        }
        bool specular = false, metal = false;
        float ro = 0;
        if constexpr (V::spec) specular = specular_event(rec.surf.spec, rng, metal, ro);
        if (V::spec && specular) {
            // specular event: the emission of applyRayColor, the throughput tinted by a metal only, no sun sample
            const float3 col = f3(rec.surf.color.x, rec.surf.color.y, rec.surf.color.z);
            const float3 tinted = throughput * col;
            if (emits) color = color + (col * (rec.surf.emittance * s.emitter_scale)) * tinted;
            if (metal) throughput = tinted;
            const float x1 = rng_float(rng);
            const float x2 = rng_float(rng);
            direction = specular_direction(direction, rec.surf.normal, diffuse_direction(rec.surf.normal, x1, x2), ro);
            if constexpr (V::fog) {
                if (s.sun_flags & 1) fog_sun_sample<MODE, V>(s, cv, rng, fog_p, fog_w, rec, color);
            }
            origin = rec.point + direction * CCU_OFFSET;
            ray_depth += 1;
            rec.distance = inff_();
            if (!(ray_depth < s.max_depth)) break;
            continue;
        }
        // kernel.h:33-44
        origin = rec.point;
        float3 col = f3(rec.surf.color.x, rec.surf.color.y, rec.surf.color.z);
        throughput = throughput * col;
        if (emits) color = color + (col * (rec.surf.emittance * s.emitter_scale)) * throughput;
        // sun sampling + shadow ray (sky.h:68-93, rayTracer.cl:101-106)
        if (s.sun_flags & 1) {
            float x1 = rng_float(rng);
            float x2 = rng_float(rng);
            float3 d = sun_sample_direction(s, x1, x2);
            float shadow_emittance = fabsf(dot3(d, rec.surf.normal));
            RecordT<V::spec> sh = rec;                // keeps the surface hit's distance as the ray limit (SURVEY Q4)
            HitInfo shi;
            if (!closest_intersect_mode<MODE, V>(s, origin, d, sh, shi) && !cloud_blocks<V>(cv, origin, d, inff_())) {
                float3 sky = sky_radiance(s, d);
                color = color + (sky * throughput) * shadow_emittance;
            }
        }
        // emitter sampling (DESIGN §10): only where the bounce below will be traced, and without a draw where L(cell) is empty
        if constexpr (V::nee) {
            int3 cell;
            int n_list = 0, first = 0;
            if (ray_depth + 1 < s.max_depth && emitter_cell(g, origin, cell)) first = emitter_list(g, cell, n_list);
            if constexpr (V::clouds) {
                if (hi.kind == 4) n_list = 0;   // a cloud takes no emitter sample (DESIGN §15.4)
            }
            if (n_list > 0) {
                nee_prev = true;
                nee_cell = cell;
                float3 c, w;
                float limit;
                if (nee_sample<V::nee, V::biome>(s, g, first, n_list, origin, rec.surf.normal, throughput, rng, c, w, limit)) {
                    RecordT<V::spec> sh = rec;
                    sh.distance = limit;
                    HitInfo shi;
                    if (!closest_intersect_mode<MODE, V, V::models>(s, origin, w, sh, shi) && !cloud_blocks<V>(cv, origin, w, limit)) color = color + c;
                }
            }
        }
        // kernel.h:46-98 diffuse bounce
        float x1 = rng_float(rng);
        float x2 = rng_float(rng);
        direction = diffuse_direction(rec.surf.normal, x1, x2);
        if constexpr (V::fog) {
            if (s.sun_flags & 1) fog_sun_sample<MODE, V>(s, cv, rng, fog_p, fog_w, rec, color);
        }
        origin = rec.point + direction * CCU_OFFSET;
        ray_depth += 1;
        rec.distance = inff_();
        if (!(ray_depth < s.max_depth)) break;
    }
    return color;
}

}  // namespace ccu
