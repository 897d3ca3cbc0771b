// ccu_queue.cuh - persistent wavefront path tracer with a CTA-wide path pool and per-stage work masks.
//
// One CTA per SM owns Q_SLOTS path slots in shared memory (structure of arrays, one 32-bit word per field and
// slot).  A slot is a pixel walking through its passes: path colour / throughput, RNG state, the surface it sits on
// and its current ray (the pixel's running mean stays in the accumulation buffer).  Slot (row, column) lives at word
// row*32 + column of every field, and column c is only ever touched by lane c of whichever warp works on it, so the slot
// accesses of a stage are bank-conflict free without any data movement between stages.  (The bank conflicts ncu counts for
// the kernel - about 0.1 G cycles per 16-pass 1080p launch - come from the gathers into the staged tables: the octree top
// table in the march step and the UNORM table in the texel conversions, where the lanes of a warp ask for unrelated words.)
//
// Work is tracked per stage and column as a bit mask over rows (mask[stage][column], bit = row).  A warp picks
// the stage with the most non-empty columns, every lane pops one slot of its column (atomicAnd), the warp runs
// the stage for up to 32 paths *of the same kind*, and every lane pushes its slot to the next stage (atomicOr):
//
//   MARCH   step the ray through air leaves (octree.h:66-107) on the "air" layout - straight-line steps in a tight loop
//           (ccu_march.cuh, lean_step_flat); lanes whose rays ended hand them over and pop their next ray in batches, so
//           the march loop stays busy; when too few lanes are busy and another stage has more work the warp parks its
//           rays (t / steps written back) and switches;
//   BLOCK   block / material test of the non-air leaf the ray reached (block.h:30-118); miss -> MARCH;
//           hit -> surface response + sun sampling (kernel.h:33-44, sky.h:68-93) -> MARCH (shadow ray); when the ray
//           was the shadow ray the diffuse bounce (kernel.h:46-98) follows right away -> MARCH, or END at the depth limit;
//   EXIT    the ray left the octree: sky + sun disc (kernel.h:26-31), then the bounce (shadow ray) -> MARCH, or END;
//   END     fold the sample into the running mean (rayTracer.cl:109-112), next pass or next pixel (global work
//           counter), camera ray (rayTracer.cl:55-91) -> MARCH;
//   BVH, LEAF, SHADE   only in the kernels for scenes with entity BVHs: BLOCK / EXIT hand the ray to the BVH walk
//           (bvh.h:22-113, world then actor BVH; BVH steps inner nodes, LEAF tests a leaf's triangles), SHADE then does the
//           shading BLOCK / EXIT do directly otherwise.
//
// Scheduling does not touch arithmetic: every path performs exactly the operations of the thread-per-pixel
// kernel in the same order (RNG draw order, per-pixel pass order), so the image is bit-identical.
#pragma once
#include "ccu_march.cuh"

#ifndef CCU_Q_WARPS
#define CCU_Q_WARPS 28
#endif
#ifndef CCU_Q_ROWS
#define CCU_Q_ROWS 32
#endif

namespace ccu {

constexpr int Q_WARPS = CCU_Q_WARPS;       // warps per CTA (one CTA per SM)
constexpr int Q_ROWS = CCU_Q_ROWS;         // slots per lane column
constexpr int Q_SLOTS = Q_ROWS * 32;
constexpr int Q_MW = (Q_ROWS + 31) / 32;   // 32-bit words per work mask (one mask per stage and column; 64-bit masks for > 32 rows)
static_assert(Q_ROWS >= 1 && Q_ROWS <= 64, "at most two mask words per stage and column");

// QS_BVH / QS_SHADE exist only in the kernels built for scenes with entity BVHs (HAS_BVH): there the BVH traversal runs as
// a stage of its own between the octree part of closestIntersect (BLOCK / EXIT) and the shading (SHADE); without BVHs
// BLOCK / EXIT shade directly.
// A BVH walk is a slot state like a marching ray - its traversal stack lives in shared memory by slot - so walks can be handed
// from warp to warp: QS_BVH steps inner nodes for 32 walks that are all at inner nodes, QS_LEAF runs the triangle tests for 32
// walks that are all at leaves.
enum QStage : int { QS_MARCH = 0, QS_BLOCK, QS_EXIT, QS_END, QS_BVH, QS_SHADE, QS_LEAF, QS_COUNT_BVH };
constexpr int QS_COUNT = QS_BVH;   // stages of the kernels without BVHs

// Slot fields.  The running mean stays in the accumulation buffer (read-modify-write per sample, L2 only); the
// surface point of the current hit is the origin of the shadow ray and lives in QF_O*.
enum QField : int {
    QF_GID = 0, QF_META, QF_RNG, QF_COLX, QF_COLY, QF_COLZ, QF_THRX, QF_THRY, QF_THRZ,
    QF_SNX, QF_SNY, QF_SNZ, QF_SHW,
    QF_OX, QF_OY, QF_OZ, QF_DX, QF_DY, QF_DZ, QF_IX, QF_IY, QF_IZ, QF_T, QF_LIMIT, QF_STEPS,
    QF_COUNT,
    // HAS_BVH only: the closest hit so far while the ray is in the BVH / SHADE stages.  Its distance, emittance and normal.x
    // re-use the march fields of the (finished) ray: QF_LIMIT, QF_T, QF_STEPS.
    QF_HNY = QF_COUNT, QF_HNZ, QF_HCX, QF_HCY, QF_HCZ,
    QF_BREF, QF_BSP,        // the walk's next node and (stack entries | phase << 8)
    QF_COUNT_BVH,
    QF_HSPEC = QF_COUNT_BVH,   // HAS_BVH + SPEC only: word 5 of the closest hit's material
    QF_COUNT_BVH_SPEC,
    QF_HDIST = QF_LIMIT, QF_HEM = QF_T, QF_HNX = QF_STEPS
};
// NEE kernels only (CCU_RENDER_EMITTER_SAMPLING, DESIGN §10): two fields after all the others, q_fields(bvh, spec) + 0 / 1,
// hold the y / z of the emitter sample's contribution while its shadow ray is in flight (x sits in QF_SHW, free then).  The
// surface normal waits in QF_SN* as for the sun's shadow ray; during the bounce segment that follows a sample, QF_SN* hold
// the sampled cell (ints) for the emission rule.
// QF_META: pass (bits 0..15) | ray depth (bits 16..23) | flags
constexpr uint32_t QM_SHADOW = 1u << 24;     // the ray in flight is the sun-sampling shadow ray of the current surface
constexpr uint32_t QM_NEEDPIX = 1u << 25;    // the slot holds no pixel (initial state)
constexpr uint32_t QM_HIT = 1u << 26;        // BVH / SHADE stages: the ray has a hit (QF_H* valid)
constexpr uint32_t QM_NEE_RAY = 1u << 27;    // NEE: the ray in flight is the emitter sample's shadow ray
constexpr uint32_t QM_NEE_PREV = 1u << 28;   // NEE: the segment in flight left a hit that sampled the list of cell QF_SN*
constexpr uint32_t QM_COVERED = 1u << 29;    // NEE + BVH: the closest hit so far is an emitter voxel that list covered
constexpr uint32_t QM_FOG_RAY = 1u << 30;    // FOG: the ray in flight is the fog's sun sample (DESIGN §14); the bounce waits
constexpr uint32_t QM_CLOUD = 1u << 31;      // CLOUDS: the surface the sun's shadow ray left is a cloud (DESIGN §15): no emitter sample
// FOG kernels only (CCU_RENDER_FOG, DESIGN §14): 8 fields after all the others, q_fields(bvh, spec, nee) + 0 .. 7.  From a
// path-segment hit to its bounce, + 0..2 hold the scattering point p and + 3..5 its weight W; while the fog ray flies, + 0..2
// hold the origin of the bounce that follows it, and QF_SHW, + 6, + 7 its direction.

constexpr int Q_TOP_WORDS = 4096;            // top tables up to 16^3 cells are staged in shared memory
// BVH stage: the first Q_STACK entries of a walk's traversal stack (bvh.h:38 nodesToVisit[64]) live in shared memory, one
// word per entry and slot (entry k at word k * Q_SLOTS + slot); bank = lane column, conflict free.  Deeper entries, which a
// reasonable BVH never needs, go to a global scratch array.
#ifndef CCU_Q_STACK
#define CCU_Q_STACK 12
#endif
constexpr int Q_SMEM_LIMIT = 227 * 1024 - 1280;   // dynamic shared memory a CTA may ask for, less the kernel's static tables (SmemTables, BiomeView)
constexpr int Q_STACK = CCU_Q_STACK;
constexpr int Q_DEEP = 64 - Q_STACK;          // stack entries beyond the shared-memory part
constexpr int Q_STACK_WORDS = Q_STACK * Q_SLOTS;
__host__ __device__ constexpr int q_fields(bool bvh, bool spec) { return bvh ? (spec ? (int)QF_COUNT_BVH_SPEC : (int)QF_COUNT_BVH) : (int)QF_COUNT; }
__host__ __device__ constexpr int q_fields(bool bvh, bool spec, bool nee) { return q_fields(bvh, spec) + (nee ? 2 : 0); }
__host__ __device__ constexpr int q_fields(bool bvh, bool spec, bool nee, bool fog) { return q_fields(bvh, spec, nee) + (fog ? 8 : 0); }
__host__ __device__ constexpr int q_stages(bool bvh) { return bvh ? (int)QS_COUNT_BVH : (int)QS_COUNT; }
__host__ __device__ constexpr int q_mask_words(bool bvh) { return q_stages(bvh) * Q_MW * 32; }
// slot fields + work masks + control words (live, tile lock / base / used) [+ the staged top table]
__host__ __device__ constexpr int q_smem_bytes(bool bvh, bool tops, bool spec, bool nee, bool fog = false) {
    return (q_fields(bvh, spec, nee, fog) * Q_SLOTS + q_mask_words(bvh) + 32 + (tops ? Q_TOP_WORDS : 0) + (bvh ? Q_STACK_WORDS : 0)) * 4;
}
static_assert(q_smem_bytes(true, true, true, true) + 64 * 64 * 4 <= Q_SMEM_LIMIT, "the largest kernel still stages a 64 x 64 sky table");

#ifdef CCU_Q_STATS
// debug counters (build with -DCCU_Q_STATS): [2*st] = executions of stage st, [2*st+1] = lanes that had a slot;
// [10] march iterations, [11] lanes in flight summed over iterations, [12] scheduler rounds that found no work,
// [13] march yields, [14] pop attempts, [15] pop retries, [24] march refills, [25] BVH refills
// one copy per translation unit, read through queue_stats_take (ccu_render.cuh)
static __device__ unsigned long long g_qstats[32];   // [16] BVH stage entries, [18] BVH steps, [19] walking lanes, [20] leaf turns, [21] leaf lanes, [22] SHADE runs, [23] lanes
#define QSTAT(i, v) do { const unsigned long long v_ = (unsigned long long)(v); if ((threadIdx.x & 31) == 0) atomicAdd(&g_qstats[i], v_); } while (0)
#define QSTAT_LANE(i, v) atomicAdd(&g_qstats[i], (unsigned long long)(v))
#else
#define QSTAT(i, v) do { } while (0)
#define QSTAT_LANE(i, v) do { } while (0)
#endif

struct PassParams {
    const int *seeds;           // one seed per pass of this launch (rayTracer.cl:55)
    int n_passes;
    int start_spp;              // passes already in the accumulation window (bufferSpp, rayTracer.cl:109-112)
    float *res;                 // running mean float[3*W*H]
    const float *res_prev;      // buffer that holds the previous window's mean (what the reference's single buffer would hold at bufferSpp = 0)
    int n_pixels;
    unsigned int *next_pixel;   // global work counter (zeroed before the launch)
};

struct QueueParams {
    PassParams w;
    int yield_below;   // MARCH: consider switching stage once fewer lanes than this are busy
    int refill_min;    // MARCH: hand over / refill once this many lanes hold a finished ray
    int march_warps;   // scheduler: only warps 0 .. march_warps-1 run the MARCH stage
    int march_bias;    // scheduler: warps of sub-partitions 0..2 count MARCH columns +bias, warps of sub-partition 3 -bias
    int sticky_min;    // scheduler: a warp repeats the one-shot stage it has just run while at least this many columns have work for it (33 = never)
    int shade_min;     // one-shot stages: a warp that got fewer slots than this puts them back and retries (q_pop_batch)
    int sky_texels;    // > 0: the launch reserved this many texels (4 bytes each) behind the other shared arrays for the sky table
    int *bvh_deep;     // BVH kernels: global scratch for traversal-stack entries beyond Q_STACK, Q_DEEP words per slot and CTA
};

// ------------------------------------------------------------------------------------------------------
// work masks: per stage and column a bit per row
// ------------------------------------------------------------------------------------------------------
// Lowest set bit first: warps that pop the same stage at the same time contend for the same rows, and the winner
// takes (most of) a row across all columns.  Rows therefore tend to stay together from stage to stage, which keeps
// the batches full; spreading the warps over different rows (measured) fragments the batches and is slower.
// Masks are 32-bit words (shared-memory atomics are native on 32 bits): Q_MW words per stage and column, word w holds rows
// 32 w .. 32 w + 31, at index (stage * Q_MW + w) * 32 + column.
// Ordering between a slot's fields and its mask bit (both in shared memory, CTA scope): the push releases, a successful pop
// acquires.  The atomics themselves carry the semantics (red.release.cta / atom.acquire.cta: on shared memory the acquire side
// needs no fence instruction at all, the release side is MEMBAR.ALL.CTA + ATOMS).
__device__ __forceinline__ unsigned q_mask_and(unsigned *word, unsigned v) {
    unsigned old;
    asm volatile("atom.acquire.cta.shared.and.b32 %0, [%1], %2;" : "=r"(old) : "r"((unsigned)__cvta_generic_to_shared(word)), "r"(v) : "memory");
    return old;
}
__device__ __forceinline__ void q_mask_or(unsigned *word, unsigned v) {
    asm volatile("red.release.cta.shared.or.b32 [%0], %1;" :: "r"((unsigned)__cvta_generic_to_shared(word)), "r"(v) : "memory");
}
__device__ __forceinline__ int q_pop(unsigned *mask, int stage, int lane) {
#pragma unroll
    for (int w = 0; w < Q_MW; w++) {
        unsigned *word = mask + (stage * Q_MW + w) * 32 + lane;
        unsigned m = *reinterpret_cast<volatile unsigned *>(word);
        while (m) {
            const unsigned bit = m & (0u - m);
            const unsigned old = q_mask_and(word, ~bit);
            QSTAT_LANE(14, 1);
            if (old & bit) return w * 32 + __ffs((int)bit) - 1;
            QSTAT_LANE(15, 1);
            m = old & ~bit;
        }
    }
    return -1;
}
__device__ __forceinline__ void q_push(unsigned *mask, int stage, int lane, int row) {
    q_mask_or(mask + (stage * Q_MW + (Q_MW > 1 ? row >> 5 : 0)) * 32 + lane, 1u << (row & 31));
}
__device__ __forceinline__ bool q_has_work(const unsigned *mask, int stage, int lane) {
    unsigned any = 0;
#pragma unroll
    for (int w = 0; w < Q_MW; w++) any |= *(reinterpret_cast<const volatile unsigned *>(mask) + (stage * Q_MW + w) * 32 + lane);
    return any != 0;
}

// One slot per lane for a one-shot stage.  Several warps often decide for the same stage at the same moment (they all saw the
// same masks); the late ones find most columns already taken and would run the stage's whole code for a handful of paths.
// With min_lanes > 1 such a warp puts its slots back and returns -2 on every lane (the scheduler retries a moment later,
// with min_lanes = 1 after two such rounds, so that the last paths of a launch are never held up).
__device__ __forceinline__ int q_pop_batch(unsigned *mask, int stage, int lane, int min_lanes) {
    const int row = q_pop(mask, stage, lane);
    if (min_lanes > 1) {
        const int got = __popc(__ballot_sync(0xffffffffu, row >= 0));
        if (got < min_lanes) {
            if (row >= 0) q_push(mask, stage, lane, row);
            return -2;
        }
    }
    return row;
}

// start of kernel.h:17-18 / what follows a finished BVH: phase 0 = world BVH, 1 = actor BVH, 2 = both done
__device__ __forceinline__ void bvh_first_ref(const DScene &s, int &ref, int &phase) {
    ref = 0;
    if (!s.world_bvh_empty) { phase = 0; ref = s.world_root; }
    else if (!s.actor_bvh_empty) { phase = 1; ref = s.actor_root; }
    else phase = 2;
}
__device__ __forceinline__ void bvh_phase_done(const DScene &s, int &ref, int &phase) {
    if (phase == 0 && !s.actor_bvh_empty) { phase = 1; ref = s.actor_root; }
    else { phase = 2; ref = 0; }
}

#define QI(f) (*reinterpret_cast<int *>(&F[(f) * Q_SLOTS + slot]))
#define QU(f) (F[(f) * Q_SLOTS + slot])
#define QFL(f) (*reinterpret_cast<float *>(&F[(f) * Q_SLOTS + slot]))

// store the ray a stage has just started (march_begin done) and queue it
__device__ __forceinline__ void q_store_ray(uint32_t *F, unsigned *mask, int lane, int row, const March &m, bool entered) {
    const int slot = row * 32 + lane;
    QFL(QF_OX) = m.o.x; QFL(QF_OY) = m.o.y; QFL(QF_OZ) = m.o.z;
    QFL(QF_DX) = m.d.x; QFL(QF_DY) = m.d.y; QFL(QF_DZ) = m.d.z;
    QFL(QF_IX) = m.inv.x; QFL(QF_IY) = m.inv.y; QFL(QF_IZ) = m.inv.z;
    QFL(QF_T) = m.t; QFL(QF_LIMIT) = m.limit; QI(QF_STEPS) = m.steps;
    // a ray that starts outside the octree cube and never enters it is finished already (octree.h:53-64)
    q_push(mask, entered ? QS_MARCH : QS_EXIT, lane, row);
}

// ------------------------------------------------------------------------------------------------------
// stages
// ------------------------------------------------------------------------------------------------------
// r.steps is loaded as steps - draw_depth (the march loop then ends a ray at r.steps >= 0); q_store_lean_t undoes that.
__device__ __forceinline__ void q_load_lean(const uint32_t *F, int slot, LeanRay &r, int draw_depth) {
    r.o = f3(__uint_as_float(F[QF_OX * Q_SLOTS + slot]), __uint_as_float(F[QF_OY * Q_SLOTS + slot]), __uint_as_float(F[QF_OZ * Q_SLOTS + slot]));
    r.d = f3(__uint_as_float(F[QF_DX * Q_SLOTS + slot]), __uint_as_float(F[QF_DY * Q_SLOTS + slot]), __uint_as_float(F[QF_DZ * Q_SLOTS + slot]));
    r.inv = f3(__uint_as_float(F[QF_IX * Q_SLOTS + slot]), __uint_as_float(F[QF_IY * Q_SLOTS + slot]), __uint_as_float(F[QF_IZ * Q_SLOTS + slot]));
    r.t = __uint_as_float(F[QF_T * Q_SLOTS + slot]);
    r.limit = __uint_as_float(F[QF_LIMIT * Q_SLOTS + slot]);
    r.steps = (int)F[QF_STEPS * Q_SLOTS + slot] - draw_depth;
    lean_prepare(r);
}
__device__ __forceinline__ void q_store_lean_t(uint32_t *F, int slot, const LeanRay &r, int draw_depth) {
    F[QF_T * Q_SLOTS + slot] = __float_as_uint(r.t);
    F[QF_STEPS * Q_SLOTS + slot] = (uint32_t)(r.steps + draw_depth);
}

// MARCH (NST = number of stages of this kernel; LAY: 0 = top table in shared memory, 1 = in global memory, 2 = deep world)
template <int NST, int LAY>
__device__ __forceinline__ void q_stage_march(const DScene &s, const unsigned *__restrict__ top, uint32_t *F, unsigned *mask, int lane,
                                              int yield_below, int refill_min) {
    const unsigned full = 0xffffffffu;
    const int draw_depth = s.draw_depth;
    const unsigned outside = ~0u << s.depth;
    int cur = -1;   // slot of the ray this lane is marching (row * 32 + column), -1 = none
    LeanRay r;
    r.o = r.d = r.inv = r.doff = f3(0, 0, 0);
    r.t = 0; r.limit = 0; r.steps = 0; r.fmx = r.fmy = r.fmz = 0; r.nmx = r.nmy = r.nmz = 0;
    int done = 2;   // 0 = ray in flight, 1 = reached a non-air leaf, 2 = finished or no ray (cur < 0)
    int recheck = 0;
    int busy = 0;   // lanes that hold a ray, in flight or finished (warp-uniform, changes only at a refill)
    int n_fly = 0;  // lanes whose ray is in flight (warp-uniform)
    for (;;) {
        // Finished rays are handed over and idle lanes re-filled in batches: once refill_min lanes hold a finished
        // ray, or nothing is in flight.
        {
            if (done != 0) {
                if (cur >= 0) {
                    q_store_lean_t(F, cur, r, draw_depth);
                    q_push(mask, done == 1 ? QS_BLOCK : QS_EXIT, cur & 31, cur >> 5);
                }
                const int row = q_pop(mask, QS_MARCH, lane);
                cur = row < 0 ? -1 : row * 32 + lane;
                done = cur < 0 ? 2 : 0;
                if (cur >= 0) q_load_lean(F, cur, r, draw_depth);
                else r.steps = 0;   // an idle lane's march step finds its (biased) step budget spent

            }
            busy = __popc(__ballot_sync(full, cur >= 0));
            QSTAT(24, 1);
            if (busy == 0) return;
            if (busy < yield_below) {
                // few busy lanes: switch when another stage has more lanes' worth of work than this warp is using
                if (recheck == 0) {
                    int best = 0;
#pragma unroll
                    for (int st = QS_BLOCK; st < NST; st++) best = max(best, __popc(__ballot_sync(full, q_has_work(mask, st, lane))));
                    if (best > busy) { QSTAT(13, 1); break; }
                    recheck = 4;
                }
                recheck--;
            }
        }
        // march until enough lanes hold a finished ray (busy - n_fly >= refill_min) or nothing is in flight: a tight inner loop
        // with one backward branch
        // The flat step needs no per-lane state besides the ray: a lane whose ray reached a non-air leaf or finished keeps its
        // t and steps, so every further step looks up the same voxel, finds the same answer and commits nothing, and an idle
        // lane has r.steps = 0.
        const int fly_min = max(busy - refill_min, 0);
        do {
            if (LAY != 2) done = lean_step_flat<LAY == 0>(s, top, r, true, 0, 0, outside);
            else if (done == 0) done = lean_probe<LAY == 2, LAY == 0>(s, top, r, 0);
            n_fly = __popc(__ballot_sync(full, done == 0));
            QSTAT(10, 1); QSTAT(11, n_fly);
        } while (n_fly > fly_min);
    }
    // park the rays still in flight, hand over the finished ones
    if (cur >= 0) {
        q_store_lean_t(F, cur, r, draw_depth);
        q_push(mask, done == 0 ? QS_MARCH : (done == 1 ? QS_BLOCK : QS_EXIT), cur & 31, cur >> 5);
    }
}

// What follows closestIntersect in rayTracer.cl:93-107 for a ray whose closest hit is known: sky for a miss
// (kernel.h:26-31), otherwise the surface response (kernel.h:33-44) and the sun sampling ray (sky.h:68-93); when the ray
// was the shadow ray (or sun sampling is off) the diffuse bounce (nextPath, kernel.h:46-98) follows right away.
// V::spec: a specular event at the hit (DESIGN "Beyond the reference: specular materials") bounces right away, without a sun sample.
// V::nee: after the sun sample (or in its place) and before the bounce, the emitter sample of DESIGN §10 (§11 for NEE_NEAR) with its
// own shadow ray (NFI: index of the two NEE fields); `covered`: the hit is an emitter the previous hit's sample covered, whose
// emission is left out.  V::biome: the emitter sample reads the biome colours of CCU_RENDER_BIOME_TINT (DESIGN §13).
// FOG: §14.2 steps 1-2 at a path-segment hit from o along d at record distance `distance`: with the sun on the scattering draw,
// p and W into the fog fields (FFI = the first), then the segment's transmittance on the slot's throughput.
template <int FFI>
__device__ __forceinline__ void q_fog_hit(const DScene &s, uint32_t *F, int slot, float3 o, float3 d, float distance) {
    float3 throughput = f3(QFL(QF_THRX), QFL(QF_THRY), QFL(QF_THRZ));
    const float a = distance * sqrtf(dot3(d, d));
    const float e = s.fog_sigma * a;
    const float tau = dm_expf(-e);
    if (s.sun_flags & 1) {
        uint32_t rng = QU(QF_RNG);
        const float u = rng_float(rng);
        QU(QF_RNG) = rng;
        const float3 p = o + d * (u * distance);
        const float k = s.fog_fast ? 1 - tau : e * dm_expf(-(s.fog_sigma * (u * a)));
        const float3 w = (throughput * s.fog_color) * k;
        QFL(FFI) = p.x; QFL(FFI + 1) = p.y; QFL(FFI + 2) = p.z;
        QFL(FFI + 3) = w.x; QFL(FFI + 4) = w.y; QFL(FFI + 5) = w.z;
    }
    throughput = throughput * tau;
    QFL(QF_THRX) = throughput.x; QFL(QF_THRY) = throughput.y; QFL(QF_THRZ) = throughput.z;
}

// CLOUDS (DESIGN §15): `cloud`: the path segment hit a cloud (q_resolve_clouds), which takes no emitter sample.
template <bool HAS_BVH, class V>
__device__ __forceinline__ void q_shade(const DScene &s, const EmitView &g, uint32_t *F, unsigned *mask, int lane, int row, float3 o,
                                        float3 d, float distance, bool ray_hit, const SurfT<V::spec> &hit, bool covered, bool cloud) {
    constexpr int NFI = q_fields(HAS_BVH, V::spec);
    constexpr int FFI = q_fields(HAS_BVH, V::spec, V::nee);   // FOG: the first fog field
    const int slot = row * 32 + lane;
    uint32_t meta = QU(QF_META) & ~(V::nee ? (QM_HIT | QM_COVERED) : QM_HIT);
    if constexpr (V::fog) {
        if (meta & QM_FOG_RAY) {
            // §14.2 step 3: an escaped fog ray adds W times the sky (and sun disc) along it; then the waiting bounce, or END
            if (!ray_hit) {
                float3 color = f3(QFL(QF_COLX), QFL(QF_COLY), QFL(QF_COLZ));
                color = color + f3(QFL(FFI + 3), QFL(FFI + 4), QFL(FFI + 5)) * sky_radiance(s, d);
                QFL(QF_COLX) = color.x; QFL(QF_COLY) = color.y; QFL(QF_COLZ) = color.z;
            }
            meta &= ~QM_FOG_RAY;
            QU(QF_META) = meta;
            if ((int)((meta >> 16) & 0xFF) < s.max_depth) {
                March m;
                const bool entered = march_begin(s, m, f3(QFL(FFI), QFL(FFI + 1), QFL(FFI + 2)), f3(QFL(QF_SHW), QFL(FFI + 6), QFL(FFI + 7)), inff_());
                q_store_ray(F, mask, lane, row, m, entered);
            } else {
                q_push(mask, QS_END, lane, row);
            }
            return;
        }
    }
    const bool shadow = (meta & QM_SHADOW) != 0;
    const bool nee_ray = V::nee && (meta & QM_NEE_RAY) != 0;
    // What the path continues with: the sun-sampling shadow ray (sky.h:68-93), the diffuse bounce (nextPath, kernel.h:46-98), or
    // nothing (END).  Both continuations draw two random numbers, take the sine / cosine of 2 pi x2 and start a ray: that part is
    // written ONCE below the case analysis, so a batch that mixes the cases runs it once.
    bool sun = false, bounce = false;
    bool nee_step = false;           // NEE: the emitter sample comes first, then the bounce
    bool nee_ran = false;            // NEE: this surface sampled an emitter list (the bounce carries its cell)
    float3 from = o;                 // the shadow ray starts at the surface point, so that is where its bounce starts
    float3 normal = f3(0, 0, 0);     // surface normal for either continuation
    bool specular = false;           // SPEC: the bounce is a specular event's (mirror direction blended by the roughness ro)
    float ro = 0;
    if (!ray_hit) {
        if (V::nee && nee_ray) {
            // the emitter sample's shadow ray reached its limit: its contribution counts
            float3 color = f3(QFL(QF_COLX), QFL(QF_COLY), QFL(QF_COLZ));
            color = color + f3(QFL(QF_SHW), QFL(NFI), QFL(NFI + 1));
            QFL(QF_COLX) = color.x; QFL(QF_COLY) = color.y; QFL(QF_COLZ) = color.z;
            bounce = true;
            nee_ran = true;
        } else {
            // kernel.h:26-31 with emittance 1 (path segment) or |d.n| (shadow ray)
            float3 throughput = f3(QFL(QF_THRX), QFL(QF_THRY), QFL(QF_THRZ));
            float3 color = f3(QFL(QF_COLX), QFL(QF_COLY), QFL(QF_COLZ));
            float3 sky = sky_radiance(s, d);
            if constexpr (V::fog) {   // §14.3: a path segment's sky blended towards the fog colour by elevation
                if (!shadow) {
                    const float y = d.y / sqrtf(dot3(d, d));
                    const float f = s.fog_sky * (y > 0 ? (1 - y) * (1 - y) : 1.0f);
                    sky = sky * (1 - f) + s.fog_color * f;
                }
            }
            color = color + (sky * throughput) * (shadow ? QFL(QF_SHW) : 1.0f);
            QFL(QF_COLX) = color.x; QFL(QF_COLY) = color.y; QFL(QF_COLZ) = color.z;
            if (shadow) { if (V::nee) nee_step = true; else bounce = true; }
            else q_push(mask, QS_END, lane, row);
        }
    } else if (shadow) {
        if (V::nee) nee_step = true; else bounce = true;
    } else if (V::nee && nee_ray) {
        bounce = true;               // the emitter sample is occluded
        nee_ran = true;
    } else if (!V::spec) {
        // kernel.h:20-22 + applyRayColor kernel.h:33-44
        if constexpr (V::fog) q_fog_hit<FFI>(s, F, slot, o, d, distance);
        float3 throughput = f3(QFL(QF_THRX), QFL(QF_THRY), QFL(QF_THRZ));
        float3 color = f3(QFL(QF_COLX), QFL(QF_COLY), QFL(QF_COLZ));
        from = o + d * (distance - CCU_OFFSET);
        float3 col = f3(hit.color.x, hit.color.y, hit.color.z);
        throughput = throughput * col;
        if (!(V::nee && covered)) color = color + (col * (hit.emittance * s.emitter_scale)) * throughput;
        QFL(QF_THRX) = throughput.x; QFL(QF_THRY) = throughput.y; QFL(QF_THRZ) = throughput.z;
        QFL(QF_COLX) = color.x; QFL(QF_COLY) = color.y; QFL(QF_COLZ) = color.z;
        normal = hit.normal;
        if (s.sun_flags & 1) sun = true;
        else if (V::nee) nee_step = true;
        else bounce = true;
    } else {
        // the event draws come first; then applyRayColor (diffuse event) or its emission with the throughput tinted by a
        // metal only (specular event)
        bool metal = false;
        if constexpr (V::fog) q_fog_hit<FFI>(s, F, slot, o, d, distance);   // its draw comes before the event draws
        if constexpr (V::spec) {
            uint32_t rng = QU(QF_RNG);
            specular = specular_event(hit.spec, rng, metal, ro);
            QU(QF_RNG) = rng;
        }
        float3 throughput = f3(QFL(QF_THRX), QFL(QF_THRY), QFL(QF_THRZ));
        float3 color = f3(QFL(QF_COLX), QFL(QF_COLY), QFL(QF_COLZ));
        from = o + d * (distance - CCU_OFFSET);
        float3 col = f3(hit.color.x, hit.color.y, hit.color.z);
        const float3 tinted = throughput * col;
        if (!(V::nee && covered)) color = color + (col * (hit.emittance * s.emitter_scale)) * tinted;
        if (!specular || metal) throughput = tinted;
        QFL(QF_THRX) = throughput.x; QFL(QF_THRY) = throughput.y; QFL(QF_THRZ) = throughput.z;
        QFL(QF_COLX) = color.x; QFL(QF_COLY) = color.y; QFL(QF_COLZ) = color.z;
        normal = hit.normal;
        if ((s.sun_flags & 1) && !specular) sun = true;
        else if (V::nee && !specular) nee_step = true;
        else bounce = true;
    }
    if constexpr (V::clouds) {
        // a cloud takes no emitter sample (DESIGN §15.4): at the hit, nor when the sun's shadow ray it sent returns
        if (nee_step && (cloud || (shadow && (meta & QM_CLOUD)))) { nee_step = false; bounce = true; }
    }
    if constexpr (V::nee) {
        if (nee_step) {
            // DESIGN §10: only where the bounce will be traced, and without a draw where L(cell) is empty
            if (shadow) normal = f3(QFL(QF_SNX), QFL(QF_SNY), QFL(QF_SNZ));
            int3 cell;
            int n_list = 0, first = 0;
            if ((int)((meta >> 16) & 0xFF) + 1 < s.max_depth && emitter_cell(g, from, cell)) first = emitter_list(g, cell, n_list);
            if (n_list > 0) {
                nee_ran = true;
                uint32_t rng = QU(QF_RNG);
                float3 c, w;
                float limit;
                const bool ray = nee_sample<V::nee, V::biome>(s, g, first, n_list, from, normal, f3(QFL(QF_THRX), QFL(QF_THRY), QFL(QF_THRZ)), rng, c, w, limit);
                QU(QF_RNG) = rng;
                if (ray) {
                    QFL(QF_SNX) = normal.x; QFL(QF_SNY) = normal.y; QFL(QF_SNZ) = normal.z;
                    QFL(QF_SHW) = c.x; QFL(NFI) = c.y; QFL(NFI + 1) = c.z;
                    QU(QF_META) = (meta & ~QM_SHADOW) | QM_NEE_RAY;
                    March m;
                    const bool entered = march_begin(s, m, from, w, limit);
                    q_store_ray(F, mask, lane, row, m, entered);
                    return;
                }
            }
            bounce = true;
        }
    }
    if (!(sun || bounce)) return;
    if (shadow || nee_ray) normal = f3(QFL(QF_SNX), QFL(QF_SNY), QFL(QF_SNZ));
    uint32_t rng = QU(QF_RNG);
    const float x1 = rng_float(rng);
    const float x2 = rng_float(rng);
    QU(QF_RNG) = rng;
    float sn, cs;
    dm_sincos(2 * CCU_PI_F * x2, sn, cs);
    float3 next_o, next_d;
    float next_limit;
    bool next_ray = true;
    if (sun) {
        QFL(QF_SNX) = normal.x; QFL(QF_SNY) = normal.y; QFL(QF_SNZ) = normal.z;
        next_d = sun_sample_direction_sc(s, x1, sn, cs);
        QFL(QF_SHW) = fabsf(dot3(next_d, normal));
        QU(QF_META) = meta | QM_SHADOW;
        if constexpr (V::clouds) {
            if (cloud) QU(QF_META) = meta | QM_SHADOW | QM_CLOUD;
        }
        // the shadow ray starts at the surface point and inherits the surface hit's distance as its limit (SURVEY Q4)
        next_o = from;
        next_limit = distance;
    } else {
        next_d = diffuse_direction_sc(normal, x1, sn, cs);
        if (V::spec && specular) next_d = specular_direction(d, normal, next_d, ro);
        next_o = from + next_d * CCU_OFFSET;
        next_limit = inff_();
        const int ray_depth = (int)((meta >> 16) & 0xFF) + 1;
        meta = (meta & ~(0xFFu << 16) & ~QM_SHADOW) | ((uint32_t)ray_depth << 16);
        if constexpr (V::clouds) meta &= ~QM_CLOUD;
        if constexpr (V::nee) {
            // the bounce segment carries the sampled cell for the emission rule at its hit
            meta &= ~(QM_NEE_RAY | QM_NEE_PREV);
            int3 cell;
            if (nee_ran && emitter_cell(g, from, cell)) {
                meta |= QM_NEE_PREV;
                QI(QF_SNX) = cell.x; QI(QF_SNY) = cell.y; QI(QF_SNZ) = cell.z;
            }
        }
        QU(QF_META) = meta;
        bool fog = false;
        if constexpr (V::fog) {
            if (s.sun_flags & 1) {
                // §14.2 step 3: after the bounce's draws, the fog's sun sample from p; the bounce waits in the fog fields
                uint32_t frng = QU(QF_RNG);
                const float y1 = rng_float(frng);
                const float y2 = rng_float(frng);
                QU(QF_RNG) = frng;
                const float3 p = f3(QFL(FFI), QFL(FFI + 1), QFL(FFI + 2));
                QFL(FFI) = next_o.x; QFL(FFI + 1) = next_o.y; QFL(FFI + 2) = next_o.z;
                QFL(QF_SHW) = next_d.x; QFL(FFI + 6) = next_d.y; QFL(FFI + 7) = next_d.z;
                QU(QF_META) = meta | QM_FOG_RAY;
                next_o = p;
                next_d = sun_sample_direction(s, y1, y2);
                fog = true;
            }
        }
        if (!fog && !(ray_depth < s.max_depth)) {
            next_ray = false;
            q_push(mask, QS_END, lane, row);
        }
    }
    if (next_ray) {
        March m;
        const bool entered = march_begin(s, m, next_o, next_d, next_limit);
        q_store_ray(F, mask, lane, row, m, entered);
    }
}

// CLOUDS (DESIGN §15.3): the cloud layer on a ray whose octree / BVH result is known, then q_shade.  A path segment that meets a
// cloud strictly before its octree / BVH hit (anywhere, on a miss) hits the cloud: a white surface that emits nothing.  A shadow
// or fog ray that got through is blocked by a cloud anywhere along it, an emitter sample's ray by one before its limit.
template <bool HAS_BVH, class V>
__device__ __forceinline__ void q_resolve_clouds(const DScene &s, const EmitView &g, const CloudView &cv, uint32_t *F, unsigned *mask, int lane,
                                                 int row, float3 o, float3 d, float distance, bool ray_hit, const SurfT<V::spec> &hit,
                                                 bool covered) {
    if constexpr (V::clouds) {
        const int slot = row * 32 + lane;
        const uint32_t meta = QU(QF_META);
        SurfT<V::spec> h = hit;
        bool cloud = false;
        float t;
        float3 n;
        if (!(meta & (QM_SHADOW | QM_NEE_RAY | QM_FOG_RAY))) {
            cloud = cloud_hit(cv, o, d, ray_hit ? distance : inff_(), t, n);
            if (cloud) {
                h.normal = n; h.color = make_float4(1, 1, 1, 1); h.emittance = 0;
                surf_set_spec(h, 0u);
                distance = t;
                ray_hit = true;
                covered = false;
            }
        } else if (!ray_hit) {
            ray_hit = cloud_hit(cv, o, d, (meta & QM_NEE_RAY) ? distance : inff_(), t, n);
        }
        q_shade<HAS_BVH, V>(s, g, F, mask, lane, row, o, d, distance, ray_hit, h, covered, cloud);
    } else {
        q_shade<HAS_BVH, V>(s, g, F, mask, lane, row, o, d, distance, ray_hit, hit, covered, false);
    }
}

// NEE: whether an octree hit on voxel c of block `data` is an emitter the sample of the previous hit covered (a path-segment
// ray whose meta carries QM_NEE_PREV; the cell waits in QF_SN*)
template <int NEE>
__device__ __forceinline__ bool q_covered(const DScene &s, const EmitView &g, const uint32_t *F, int slot, uint32_t meta, int data, const Cell &c) {
    if (!NEE || (meta & (QM_SHADOW | QM_NEE_RAY)) || !(meta & QM_NEE_PREV)) return false;
    const int3 cell = make_int3((int)F[QF_SNX * Q_SLOTS + slot], (int)F[QF_SNY * Q_SLOTS + slot], (int)F[QF_SNZ * Q_SLOTS + slot]);
    return emitter_covered<NEE>(s, g, data, c.bx, c.by, c.bz, cell);
}

// BLOCK (kind_block = true) and EXIT (false): the octree part of closestIntersect (kernel.h:14-16) is finished here;
// without BVHs the ray is shaded right away, with BVHs it goes to the BVH stage.  kind_block is warp-uniform.
template <bool HAS_BVH, class V>
__device__ __forceinline__ bool q_stage_resolve(const DScene &s, const EmitView &g, const CloudView &cv, uint32_t *F, unsigned *mask, int lane, const bool kind_block,
                                                int min_lanes) {
    const int row = q_pop_batch(mask, kind_block ? QS_BLOCK : QS_EXIT, lane, min_lanes);
    if (row == -2) return false;
    QSTAT(2 * (kind_block ? QS_BLOCK : QS_EXIT), 1); QSTAT(2 * (kind_block ? QS_BLOCK : QS_EXIT) + 1, __popc(__ballot_sync(0xffffffffu, row >= 0)));
    if (row < 0) return true;
    const int slot = row * 32 + lane;
    March m;
    m.o = f3(QFL(QF_OX), QFL(QF_OY), QFL(QF_OZ));
    m.d = f3(QFL(QF_DX), QFL(QF_DY), QFL(QF_DZ));
    m.inv = f3(QFL(QF_IX), QFL(QF_IY), QFL(QF_IZ));
    m.t = QFL(QF_T); m.limit = QFL(QF_LIMIT);
    m.steps = QI(QF_STEPS);
    bool ray_hit = false;
    float hit_t = 0;
    SurfT<V::spec> hit;
    hit.normal = f3(0, 0, 0); hit.color = make_float4(0, 0, 0, 0); hit.emittance = 0;
    surf_set_spec(hit, 0u);
    bool covered = false;   // NEE: the hit is an emitter the previous hit's sample covered
    if (kind_block) {
        // the leaf under the ray (octree.h:81-88): value and level
        const Cell c = march_cell(m);
        int level;
        const int data = find_leaf_wide(s, c.bx, c.by, c.bz, level);   // the kernel is only launched on the commit-time layouts
        // NEE_*_MODELS: an emitter sample's shadow ray counts a block hit only before its limit (march_block)
        const bool cut = V::models ? (QU(QF_META) & QM_NEE_RAY) != 0 : false;
        if (!march_block<V, V::models>(s, m, data, level, hit, hit_t, cut)) {
            QFL(QF_T) = m.t; QI(QF_STEPS) = m.steps;
            q_push(mask, QS_MARCH, lane, row);
            return true;
        }
        ray_hit = true;
        if constexpr (V::nee) covered = !(V::fog && (QU(QF_META) & QM_FOG_RAY)) && q_covered<V::nee>(s, g, F, slot, QU(QF_META), data, c);
    }
    const float distance = ray_hit ? hit_t : m.limit;
    if (HAS_BVH) {
        // the march fields of the finished ray now carry the closest hit so far
        QFL(QF_HDIST) = distance;
        if (ray_hit) {
            QFL(QF_HEM) = hit.emittance;
            QFL(QF_HNX) = hit.normal.x; QFL(QF_HNY) = hit.normal.y; QFL(QF_HNZ) = hit.normal.z;
            QFL(QF_HCX) = hit.color.x; QFL(QF_HCY) = hit.color.y; QFL(QF_HCZ) = hit.color.z;
            if constexpr (V::spec) QU(QF_HSPEC) = hit.spec;
        }
        uint32_t meta = QU(QF_META);
        if constexpr (V::nee) meta = covered ? (meta | QM_COVERED) : (meta & ~QM_COVERED);
        QU(QF_META) = ray_hit ? (meta | QM_HIT) : (meta & ~QM_HIT);
        // A shadow ray only asks WHETHER something lies between the surface and the sun (rayTracer.cl:101-106 uses nothing else
        // of its record): once the octree has answered yes, the BVHs - which can only find a closer hit - cannot change that.
        // The same holds for the emitter sample's shadow ray (NEE).
        // So does the fog's sun sample (FOG).
        if (ray_hit && (meta & ((V::nee ? (QM_SHADOW | QM_NEE_RAY) : QM_SHADOW) | (V::fog ? QM_FOG_RAY : 0u)))) {
            q_push(mask, QS_SHADE, lane, row);
            return true;
        }
        // kernel.h:17-18: the world BVH first, then the actor BVH (the kernel is only launched when at least one is not empty)
        int ref, phase;
        bvh_first_ref(s, ref, phase);
        QI(QF_BREF) = ref;
        QI(QF_BSP) = phase << 8;
        q_push(mask, ref < 0 ? QS_LEAF : QS_BVH, lane, row);
    } else {
        q_resolve_clouds<HAS_BVH, V>(s, g, cv, F, mask, lane, row, m.o, m.d, distance, ray_hit, hit, covered);
    }
    return true;
}

// SHADE (HAS_BVH kernels): closestIntersect is complete (kernel.h:17-22)
template <class V>
__device__ __forceinline__ bool q_stage_shade(const DScene &s, const EmitView &g, const CloudView &cv, uint32_t *F, unsigned *mask, int lane, int min_lanes) {
    const int row = q_pop_batch(mask, QS_SHADE, lane, min_lanes);
    if (row == -2) return false;
    QSTAT(22, 1); QSTAT(23, __popc(__ballot_sync(0xffffffffu, row >= 0)));
    if (row < 0) return true;
    const int slot = row * 32 + lane;
    const float3 o = f3(QFL(QF_OX), QFL(QF_OY), QFL(QF_OZ));
    const float3 d = f3(QFL(QF_DX), QFL(QF_DY), QFL(QF_DZ));
    const bool ray_hit = (QU(QF_META) & QM_HIT) != 0;
    SurfT<V::spec> hit;
    hit.normal = f3(QFL(QF_HNX), QFL(QF_HNY), QFL(QF_HNZ));
    hit.color = make_float4(QFL(QF_HCX), QFL(QF_HCY), QFL(QF_HCZ), 0.0f);
    hit.emittance = QFL(QF_HEM);
    if constexpr (V::spec) hit.spec = QU(QF_HSPEC);
    q_resolve_clouds<true, V>(s, g, cv, F, mask, lane, row, o, d, QFL(QF_HDIST), ray_hit, hit, V::nee && (QU(QF_META) & QM_COVERED) != 0);
    return true;
}

// ------------------------------------------------------------------------------------------------------
// BVH stage: bvh.h:22-113 for the world BVH, then the actor BVH (kernel.h:17-18), on the commit-time layout
// ------------------------------------------------------------------------------------------------------
// Triangle_intersect (primitives.h:335-409) on a 32-byte aligned 24-word record (20 words + pad), three 256-bit loads
// q0: the record's first 32 bytes, loaded by the caller (one triangle ahead, so that the load is in flight during the previous test)
__device__ __forceinline__ float triangle_hit_aligned(const Int8 &q0, const int *__restrict__ t, float distance, float3 origin, float3 dir, float3 &normal,
                                                      float &ou, float &ov, int &material) {
    const int flags = q0.v[0];
    const float3 e1 = f3(i2f(q0.v[1]), i2f(q0.v[2]), i2f(q0.v[3]));
    const float3 e2 = f3(i2f(q0.v[4]), i2f(q0.v[5]), i2f(q0.v[6]));
    float3 pvec = cross3(dir, e2);
    float det = dot3(e1, pvec);
    if ((flags >> 8) & 1) {
        if (det > -CCU_EPS && det < CCU_EPS) return nanf_();
    } else if (det > -CCU_EPS) {
        return nanf_();
    }
    float recip = 1.0f / det;
    const Int8 q1 = ldg256(t + 8);
    float3 o = f3(i2f(q0.v[7]), i2f(q1.v[0]), i2f(q1.v[1]));
    float3 tvec = origin - o;
    float u = dot3(tvec, pvec) * recip;
    if (u < 0 || u > 1) return nanf_();
    float3 qvec = cross3(tvec, e1);
    float v = dot3(dir, qvec) * recip;
    if (v < 0 || (u + v) > 1) return nanf_();
    float tt = dot3(e2, qvec) * recip;
    if (tt > CCU_EPS && tt < distance) {
        const Int8 q2 = ldg256(t + 16);
        float w = 1.0f - u - v;
        // words 13..18: t1.uv, t2.uv, t3.uv; 19: material
        ou = (i2f(q1.v[5]) * u + i2f(q1.v[7]) * v) + i2f(q2.v[1]) * w;
        ov = (i2f(q1.v[6]) * u + i2f(q2.v[0]) * v) + i2f(q2.v[2]) * w;
        normal = f3(i2f(q1.v[2]), i2f(q1.v[3]), i2f(q1.v[4]));
        material = q2.v[3];
        return tt;
    }
    return nanf_();
}

// traversal stack of the walk in `slot` (bvh.h:38): entry k < Q_STACK in shared memory, the rest (which a reasonable BVH never
// needs) in a global scratch array, out of line so that the common path is a compare and one shared-memory access
static __device__ __noinline__ void bvh_deep_store(int *deep, int slot, int k, int value) {
    deep[((size_t)blockIdx.x * Q_SLOTS + slot) * Q_DEEP + (k - Q_STACK)] = value;
}
static __device__ __noinline__ int bvh_deep_load(const int *deep, int slot, int k) {
    return deep[((size_t)blockIdx.x * Q_SLOTS + slot) * Q_DEEP + (k - Q_STACK)];
}
// `on`: this lane pushes / pops (the others pass through without a branch: the shared-memory access is a predicated instruction,
// the out-of-line deep path a branch no lane of a reasonable BVH ever takes)
__device__ __forceinline__ void bvh_stack_push(int *stk, int *deep, int slot, int k, int value, bool on) {
    if (on && k < Q_STACK) stk[k * Q_SLOTS + slot] = value;
    if (on && k >= Q_STACK) bvh_deep_store(deep, slot, k, value);
}
__device__ __forceinline__ int bvh_stack_pop(int *stk, int *deep, int slot, int k, bool on, int otherwise) {
    int v = otherwise;
    if (on && k < Q_STACK) v = stk[k * Q_SLOTS + slot];
    if (on && k >= Q_STACK) v = bvh_deep_load(deep, slot, k);
    return v;
}

// QS_BVH: inner-node steps (bvh.h:73-108) for walks that sit at inner nodes.  Organised like MARCH: a lane keeps its walk in
// registers while it steps from inner node to inner node; a walk that reaches a leaf or finishes is handed over (QS_LEAF /
// QS_SHADE) and the lane takes the next waiting walk, in batches; a warp with too few walks parks them and switches stage.
template <int NST>
__device__ __forceinline__ void q_stage_bvh(const DScene &s, uint32_t *F, unsigned *mask, int *stk, int *deep, int lane, int yield_below, int refill_min) {
    const unsigned full = 0xffffffffu;
    int cur = -1;
    float3 o = f3(0, 0, 0), inv = f3(0, 0, 0);
    float dist = 0;
    int ref = 0, sp = 0, phase = 2;
    int busy = 0, n_fly = 0, recheck = 0;
    for (;;) {
        // hand-over / refill (see q_stage_march)
        if (cur < 0 || phase >= 2 || ref < 0) {
            if (cur >= 0) {
                F[QF_BREF * Q_SLOTS + cur] = (uint32_t)ref;
                F[QF_BSP * Q_SLOTS + cur] = (uint32_t)(sp | (phase << 8));
                q_push(mask, phase >= 2 ? QS_SHADE : QS_LEAF, cur & 31, cur >> 5);
            }
            const int row = q_pop(mask, QS_BVH, lane);
            cur = row < 0 ? -1 : row * 32 + lane;
            phase = 2; ref = 0;
            if (cur >= 0) {
                const int slot = cur;
                o = f3(QFL(QF_OX), QFL(QF_OY), QFL(QF_OZ));
                inv = f3(QFL(QF_IX), QFL(QF_IY), QFL(QF_IZ));      // 1 / d, the same quotients bvh.h:40 computes
                dist = QFL(QF_HDIST);
                ref = QI(QF_BREF);
                const int bsp = QI(QF_BSP);
                sp = bsp & 0xFF;
                phase = bsp >> 8;
            }
        }
        busy = __popc(__ballot_sync(full, cur >= 0));
        QSTAT(25, 1);
        if (busy == 0) return;
        if (busy < yield_below) {
            if (recheck == 0) {
                int best = 0;
#pragma unroll
                for (int st = 0; st < NST; st++)
                    if (st != QS_BVH) best = max(best, __popc(__ballot_sync(full, q_has_work(mask, st, lane))));
                if (best > busy) break;
                recheck = 4;
            }
            recheck--;
        }
        // inner-node steps until enough lanes wait at a leaf / have finished (or none is walking): a tight loop with one backward
        // branch; lanes that are not at an inner node pass through on dummy values (record 0 of the world BVH) and commit nothing
        do {
            const bool on = cur >= 0 && phase < 2 && ref >= 0;
            // inner node: both children's boxes (bvh.h:73-108)
            const int4 *rbase = (on && phase != 0) ? s.actor_rec : s.world_rec;
            const int4 *r = rbase + (size_t)(on ? ref : 0) * 4;
            const Int8 lo = ldg256(r), hi = ldg256(r + 2);
            const Box b1 = {i2f(lo.v[0]), i2f(lo.v[1]), i2f(lo.v[2]), i2f(lo.v[3]), i2f(lo.v[4]), i2f(lo.v[5])};
            const Box b2 = {i2f(hi.v[0]), i2f(hi.v[1]), i2f(hi.v[2]), i2f(hi.v[3]), i2f(hi.v[4]), i2f(hi.v[5])};
            const float t1 = box_entry(b1, o, inv);
            const float t2 = box_entry(b2, o, inv);
            const int left = lo.v[6], right = hi.v[6];
            const bool miss1 = is_nan(t1) || t1 > dist;
            const bool miss2 = is_nan(t2) || t2 > dist;
            // bvh.h:93-108: both missed -> next pending node; one hit -> that child; both hit -> the nearer one, the other is
            // left pending.  Written with selects so that only the stack accesses themselves are divergent.
            const bool both = on && !miss1 && !miss2, none = on && miss1 && miss2;
            const bool go_left = both ? t1 < t2 : !miss1;
            const int far = go_left ? right : left;
            bvh_stack_push(stk, deep, cur, sp, far, both);
            sp += both ? 1 : 0;
            int nref = go_left ? left : right;
            const bool pop = none && sp > 0;
            sp -= pop ? 1 : 0;
            nref = bvh_stack_pop(stk, deep, cur, sp, pop, nref);
            int nphase = phase;
            if (none && !pop) bvh_phase_done(s, nref, nphase);
            ref = on ? nref : ref;
            phase = on ? nphase : phase;
            n_fly = __popc(__ballot_sync(full, cur >= 0 && phase < 2 && ref >= 0));
            QSTAT(18, 1); QSTAT(19, n_fly);
        } while (busy - n_fly < refill_min && n_fly != 0);
    }
    // park the walks still at inner nodes, hand over the others
    if (cur >= 0) {
        F[QF_BREF * Q_SLOTS + cur] = (uint32_t)ref;
        F[QF_BSP * Q_SLOTS + cur] = (uint32_t)(sp | (phase << 8));
        q_push(mask, phase >= 2 ? QS_SHADE : (ref < 0 ? QS_LEAF : QS_BVH), cur & 31, cur >> 5);
    }
}

// QS_LEAF: the triangles of one leaf (bvh.h:52-67) for walks that sit at a leaf, then the walk's next node from its stack
template <class V>
__device__ __forceinline__ bool q_stage_leaf(const DScene &s, uint32_t *F, unsigned *mask, int *stk, int *deep, int lane, int min_lanes) {
    const int row = q_pop_batch(mask, QS_LEAF, lane, min_lanes);
    if (row == -2) return false;
    QSTAT(20, 1); QSTAT(21, __popc(__ballot_sync(0xffffffffu, row >= 0)));
    if (row < 0) return true;
    const int slot = row * 32 + lane;
    const float3 o = f3(QFL(QF_OX), QFL(QF_OY), QFL(QF_OZ));
    const float3 d = f3(QFL(QF_DX), QFL(QF_DY), QFL(QF_DZ));
    float dist = QFL(QF_HDIST);
    int ref = QI(QF_BREF);
    const int bsp = QI(QF_BSP);
    int sp = bsp & 0xFF, phase = bsp >> 8;
    SurfT<V::spec> hit;
    hit.normal = f3(0, 0, 0); hit.color = make_float4(0, 0, 0, 0); hit.emittance = 0;
    surf_set_spec(hit, 0u);
    bool any = false;
    const int *blk = s.tris2 + (size_t)(-(ref + 1)) * 8;
    const int num = __ldg(blk);
    const uint32_t meta = QU(QF_META);
    // a shadow ray (the sun's or, NEE, the emitter sample's) is answered by its first accepted triangle (see q_stage_resolve):
    // the rest of the walk could only find a closer one
    const bool first_hit_ends = (meta & ((V::nee ? (QM_SHADOW | QM_NEE_RAY) : QM_SHADOW) | (V::fog ? QM_FOG_RAY : 0u))) != 0;
    // the head of the first triangle is requested together with the count word (a leaf block holds at least one triangle; the
    // array is padded so that the read is in bounds even for an empty one), the head of triangle i + 1 while triangle i is tested
    Int8 q0 = ldg256(blk + 8);
    for (int i = 0; i < num; i++) {
        float3 normal;
        float u, v;
        int material;
        const Int8 q0_this = q0;
        if (i + 1 < num) q0 = ldg256(blk + 8 + 24 * (i + 1));
        const float t = triangle_hit_aligned(q0_this, blk + 8 + 24 * i, dist, o, d, normal, u, v, material);
        if (!is_nan(t) && material_sample(s, material, hit, u, v)) {
            hit.normal = normal;
            dist = t;
            any = true;
            if (first_hit_ends) break;
        }
    }
    if (any) {
        // record->material keeps its octree value (bvh.h:59-65, SURVEY Q15); nothing downstream reads it
        QFL(QF_HDIST) = dist;
        QFL(QF_HEM) = hit.emittance;
        QFL(QF_HNX) = hit.normal.x; QFL(QF_HNY) = hit.normal.y; QFL(QF_HNZ) = hit.normal.z;
        QFL(QF_HCX) = hit.color.x; QFL(QF_HCY) = hit.color.y; QFL(QF_HCZ) = hit.color.z;
        if constexpr (V::spec) QU(QF_HSPEC) = hit.spec;
        QU(QF_META) = (V::nee ? (meta & ~QM_COVERED) : meta) | QM_HIT;   // NEE: a triangle is no covered emitter
    }
    if (any && first_hit_ends) { phase = 2; ref = 0; }
    else if (sp == 0) bvh_phase_done(s, ref, phase);
    else { sp--; ref = bvh_stack_pop(stk, deep, slot, sp, true, ref); }
    QI(QF_BREF) = ref;
    QI(QF_BSP) = sp | (phase << 8);
    q_push(mask, phase >= 2 ? QS_SHADE : (ref < 0 ? QS_LEAF : QS_BVH), lane, row);
    return true;
}

constexpr int Q_TILE_W = 32, Q_TILE_H = 32;
constexpr unsigned Q_CHUNK = Q_TILE_W * Q_TILE_H;
// k-th pixel in tile order (bands of Q_TILE_H rows, each cut into tiles Q_TILE_W wide, row-major inside a tile;
// the last band / last tile of a band may be smaller): a bijection of [0, W*H) that keeps consecutive k close on screen.
// PATCH: inside full 32x32 tiles, 32 consecutive k cover an 8x4 pixel patch instead of a 32x1 strip (thread-per-ray kernels:
// a warp's rays then form a compact bundle).
template <bool PATCH = false>
__device__ __forceinline__ void tile_order_xy(unsigned k, int W, int H, unsigned &px, unsigned &py) {
    const unsigned band_px = (unsigned)W * Q_TILE_H;
    const unsigned band = k / band_px;
    const unsigned kb = k - band * band_px;
    const unsigned bh = min((unsigned)Q_TILE_H, (unsigned)H - band * Q_TILE_H);     // rows in this band
    const unsigned full_tiles = (unsigned)W / Q_TILE_W;
    unsigned tile, tw = Q_TILE_W, in, iy, ix;
    if (bh == Q_TILE_H && kb < full_tiles * Q_CHUNK) {
        // a full 32x32 tile (all but the last band / last column of tiles): shifts only
        tile = kb / Q_CHUNK;
        in = kb % Q_CHUNK;
        iy = in / Q_TILE_W; ix = in % Q_TILE_W;
    } else {
        const unsigned tile_px = Q_TILE_W * bh;
        tile = kb / tile_px;
        in = kb - tile * tile_px;
        if (tile >= full_tiles) {            // the narrower remainder tile at the right edge
            tile = full_tiles;
            tw = (unsigned)W - full_tiles * Q_TILE_W;
            in = kb - full_tiles * tile_px;
        }
        iy = in / tw; ix = in % tw;
    }
    if (PATCH && tw == Q_TILE_W && bh == Q_TILE_H) {
        // in = [y4 y3 y2 | x4 x3 | y1 y0 | x2 x1 x0]
        ix = (in & 7u) | (((in >> 5) & 3u) << 3);
        iy = ((in >> 3) & 3u) | ((in >> 7) << 2);
    }
    py = band * Q_TILE_H + iy;
    px = tile * Q_TILE_W + ix;
}
template <bool PATCH = false>
__device__ __forceinline__ int tile_order_pixel(unsigned k, int W, int H) {
    unsigned px, py;
    tile_order_xy<PATCH>(k, W, H, px, py);
    return (int)(py * (unsigned)W + px);
}

// rayTracer.cl:109-112, then the next pass / pixel: rayTracer.cl:55-91
// LAST_FIRST: the tile-order indices are handed out from the end.  A launch ends with the pixels drawn last still walking through
// their passes one sample after the other (measured: 0.57 ms of a 16-pass 1080p launch, against 0.10 ms for a 1-pass one), so the
// last pixels should be quick ones.  Without entity BVHs the quick pixels are the sky at the top of the frame (one ray), which
// tile order starts with: config 1 -2.4 % per pass with the order reversed.  With BVHs every ray walks them and the sky is not
// cheap any more (entity scene: +13 % reversed), so those kernels keep the forward order.  Orders derived from a measured per-chunk
// cost (time between draws, or sample latency by chunk) were tried and cost more in the END stage than they gained.
template <bool LAST_FIRST>
__device__ __forceinline__ bool q_stage_end(const DScene &s, const PassParams &w, uint32_t *F, unsigned *mask, int *live, int lane, int min_lanes) {
    const unsigned full = 0xffffffffu;
    const int row = q_pop_batch(mask, QS_END, lane, min_lanes);
    if (row == -2) return false;
    QSTAT(2 * QS_END, 1); QSTAT(2 * QS_END + 1, __popc(__ballot_sync(full, row >= 0)));
    const int slot = row < 0 ? lane : row * 32 + lane;
    uint32_t meta = row >= 0 ? QU(QF_META) : 0u;
    int gid = row >= 0 ? QI(QF_GID) : 0;
    int pass = (int)(meta & 0xFFFFu);
    bool need_pixel = row >= 0 && (meta & QM_NEEDPIX) != 0;
    if (row >= 0 && !need_pixel) {
        // the running mean of this pixel is only ever touched by the slot that owns the pixel; L2 accesses keep it
        // coherent between the warps that run the slot's END stages
        float *px = w.res + (size_t)gid * 3;
        int spp = w.start_spp + pass;
        // at the start of a window the reference's buffer still holds the previous window's mean (it is multiplied by
        // spp = 0, rayTracer.cl:111); with two window buffers that value lives in the other one
        const float *pr = spp == 0 ? w.res_prev + (size_t)gid * 3 : px;
        float3 mean = f3(__ldcg(pr), __ldcg(pr + 1), __ldcg(pr + 2));
        float3 color = f3(QFL(QF_COLX), QFL(QF_COLY), QFL(QF_COLZ));
        float fs = (float)spp, fs1 = (float)(spp + 1);
        mean.x = (mean.x * fs + color.x) / fs1;
        mean.y = (mean.y * fs + color.y) / fs1;
        mean.z = (mean.z * fs + color.z) / fs1;
        __stcg(px, mean.x); __stcg(px + 1, mean.y); __stcg(px + 2, mean.z);
        pass++;
        if (pass >= w.n_passes) need_pixel = true;
    }
    // Pixels are handed out in screen tiles: the CTA draws chunks of Q_TILE_W * Q_TILE_H tile-order indices from the
    // global counter and its warps take their pixels from the CTA's current chunk, so the paths resident on one SM
    // stay in a compact screen region (L1 hit rate of the octree walk).  The order pixels are rendered in does not
    // change any pixel's samples.
    const unsigned want = __ballot_sync(full, need_pixel);
    bool alive = row >= 0;
    if (want) {
        const int n = __popc(want);
        const int leader = __ffs((int)want) - 1;
        unsigned base1 = 0, base2 = 0;
        int n1 = 0;
        if (lane == leader) {
            volatile unsigned *ctl = reinterpret_cast<volatile unsigned *>(live);
            while (atomicCAS(reinterpret_cast<unsigned *>(live) + 1, 0u, 1u) != 0u) __nanosleep(20);
            __threadfence_block();
            const unsigned used = ctl[3];
            n1 = min(n, (int)(Q_CHUNK - used));
            base1 = ctl[2] + used;
            if (n1 < n) {
                base2 = atomicAdd(w.next_pixel, (unsigned)Q_CHUNK);
                ctl[2] = base2;
                ctl[3] = (unsigned)(n - n1);
            } else {
                ctl[3] = used + (unsigned)n;
            }
            __threadfence_block();
            atomicExch(reinterpret_cast<unsigned *>(live) + 1, 0u);
        }
        base1 = __shfl_sync(full, base1, leader);
        base2 = __shfl_sync(full, base2, leader);
        n1 = __shfl_sync(full, n1, leader);
        if (need_pixel) {
            const int rank = __popc(want & ((1u << lane) - 1u));
            const unsigned k = rank < n1 ? base1 + (unsigned)rank : base2 + (unsigned)(rank - n1);
            if (k < (unsigned)w.n_pixels) {
                gid = tile_order_pixel(LAST_FIRST ? (unsigned)w.n_pixels - 1u - k : k, s.width, s.height);
                pass = 0;
            } else {
                alive = false;
            }
        }
    }
    const unsigned died = __ballot_sync(full, row >= 0 && !alive);
    if (died && lane == (__ffs((int)died) - 1)) atomicSub(live, __popc(died));
    if (!alive) return true;
    // new sample
    QI(QF_GID) = gid;
    QU(QF_META) = (uint32_t)pass;   // ray depth 0, no flags
    QFL(QF_COLX) = 0.0f; QFL(QF_COLY) = 0.0f; QFL(QF_COLZ) = 0.0f;
    QFL(QF_THRX) = 1.0f; QFL(QF_THRY) = 1.0f; QFL(QF_THRZ) = 1.0f;
    uint32_t rng = (uint32_t)__ldg(w.seeds + pass) + (uint32_t)gid;
    rng_next(rng);
    float3 o, d;
    camera_ray<false>(s, gid, rng, o, d);
    QU(QF_RNG) = rng;
    March m;
    const bool entered = march_begin(s, m, o, d, inff_());
    q_store_ray(F, mask, lane, row, m, entered);
    return true;
}

// LAY 0: the top table of the air layout fits Q_TOP_WORDS and is staged in shared memory; 1: it is read from global memory;
// 2: deep world (64-ary nodes between the top table and the bricks).  V: the launch's Shade.  The emitter table `g`, the biome
// colours `bv` and the cloud layer `cv` come after the other arguments, so that the kernels without them keep their parameter
// offsets.
template <bool HAS_BVH, int LAY, class V>
__global__ void __launch_bounds__(Q_WARPS * 32, 1) k_render_queue(const __grid_constant__ DScene s, const __grid_constant__ QueueParams qp,
                                                                 const __grid_constant__ EmitView g, const __grid_constant__ BiomeView bv,
                                                                 const __grid_constant__ CloudView cv) {
    constexpr int NST = q_stages(HAS_BVH);
    constexpr int MASK_WORDS = q_mask_words(HAS_BVH);
    extern __shared__ uint32_t q_mem[];
    uint32_t *F = q_mem;
    unsigned *mask = q_mem + q_fields(HAS_BVH, V::spec, V::nee, V::fog) * Q_SLOTS;
    int *live = reinterpret_cast<int *>(mask + MASK_WORDS);
    unsigned *top_s = mask + MASK_WORDS + 32;
    int *stk = reinterpret_cast<int *>(top_s + (LAY == 0 ? Q_TOP_WORDS : 0));   // HAS_BVH only: stacks by slot
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;

    for (int i = threadIdx.x; i < Q_SLOTS; i += blockDim.x) F[QF_META * Q_SLOTS + i] = QM_NEEDPIX;
    for (int i = threadIdx.x; i < NST * Q_MW * 32; i += blockDim.x) {
        // every slot starts in the END stage (QM_NEEDPIX: it fetches its first pixel there)
        const int st = i / (Q_MW * 32), w = (i / 32) % Q_MW;
        const int rows_here = min(32, Q_ROWS - 32 * w);
        mask[i] = st == QS_END ? (rows_here >= 32 ? 0xffffffffu : ((1u << rows_here) - 1u)) : 0u;
    }
    // LAY 0: the top table of a shallow world always has 16^3 cells (build_air_layout pads smaller worlds)
    if (LAY == 0) for (int i = threadIdx.x; i < Q_TOP_WORDS; i += blockDim.x) top_s[i] = __ldg(s.air_top + i);
    // sky / UNORM tables (sky.h:95-106 reads four texels per lookup)
    uchar4 *sky_s = nullptr;
    if (qp.sky_texels > 0) {
        sky_s = reinterpret_cast<uchar4 *>(top_s + (LAY == 0 ? Q_TOP_WORDS : 0) + (HAS_BVH ? Q_STACK_WORDS : 0));
        for (int i = threadIdx.x; i < qp.sky_texels; i += blockDim.x) sky_s[i] = __ldg(s.sky + i);
    }
    if constexpr (V::biome) {
        if (threadIdx.x == 0) biome_smem() = bv;   // read after the barrier of stage_tables
    }
    stage_tables(s, sky_s);
    if (threadIdx.x == 0) {
        live[0] = Q_SLOTS;
        live[1] = 0;                 // tile lock
        live[2] = 0;                 // base of the CTA's current chunk of tile-order indices
        live[3] = (int)Q_CHUNK;      // indices of the chunk handed out so far (exhausted: the first request draws a chunk)
    }
    __syncthreads();
    const unsigned *top = LAY == 0 ? top_s : s.air_top;

    int held = 0;
    int sticky = -1;   // the one-shot stage this warp has just run
    for (;;) {
        // the stage with the most columns that have work
        int best = -1, best_n = 0;
        // A warp that has just run a one-shot stage runs it again while enough columns have work for it: the stage's code
        // (several KB, far more than the L0 instruction cache) is then fetched once for several batches, and the scan over
        // all stages is skipped.  BLOCK and EXIT are one piece of code (q_stage_resolve).
        if (sticky >= 0) {
            int n = __popc(__ballot_sync(full, q_has_work(mask, sticky, lane)));
            int st2 = sticky;
            if (sticky == QS_BLOCK || sticky == QS_EXIT) {
                const int other = sticky == QS_BLOCK ? QS_EXIT : QS_BLOCK;
                const int n2 = __popc(__ballot_sync(full, q_has_work(mask, other, lane)));
                if (n2 > n) { n = n2; st2 = other; }
            }
            if (n >= qp.sticky_min) { best = st2; best_n = n; }
        }
        if (best < 0) {
#pragma unroll
        for (int st = 0; st < NST; st++) {
            int n = __popc(__ballot_sync(full, q_has_work(mask, st, lane)));
            // Warps of one SM sub-partition share an instruction cache: three sub-partitions lean towards the (small)
            // march loop, the fourth towards the (large) shading stages.
            if (st == QS_MARCH && n > 0) n = max(1, n + ((threadIdx.x >> 5 & 3) == 3 ? -qp.march_bias : qp.march_bias));
            if (st == QS_MARCH && (int)(threadIdx.x >> 5) >= qp.march_warps) n = 0;
            if (n > best_n) { best_n = n; best = st; }
        }
        }
        if (best < 0) {
            if (*reinterpret_cast<volatile int *>(live) == 0) break;
            QSTAT(12, 1);
            __nanosleep(100);
            continue;
        }
        const int min_lanes = held < 2 ? qp.shade_min : 1;      // see q_pop_batch
        bool ran = true;
        switch (best) {
            case QS_MARCH: QSTAT(0, 1); q_stage_march<NST, LAY>(s, top, F, mask, lane, qp.yield_below, qp.refill_min); break;
            case QS_BLOCK:
            case QS_EXIT: ran = q_stage_resolve<HAS_BVH, V>(s, g, cv, F, mask, lane, best == QS_BLOCK, min_lanes); break;
            case QS_END: ran = q_stage_end<!HAS_BVH>(s, qp.w, F, mask, live, lane, min_lanes); break;
            case QS_BVH: QSTAT(16, 1); if (HAS_BVH) q_stage_bvh<NST>(s, F, mask, stk, qp.bvh_deep, lane, qp.yield_below, qp.refill_min); break;
            case QS_LEAF: if (HAS_BVH) ran = q_stage_leaf<V>(s, F, mask, stk, qp.bvh_deep, lane, min_lanes); break;
            default: if (HAS_BVH) ran = q_stage_shade<V>(s, g, cv, F, mask, lane, min_lanes); break;
        }
        sticky = (ran && best != QS_MARCH && best != QS_BVH) ? best : -1;
        if (ran) {
            held = 0;
        } else {
            held++;
            __nanosleep(40);
        }
        __syncwarp();
    }
}

#undef QI
#undef QU
#undef QFL

}  // namespace ccu
