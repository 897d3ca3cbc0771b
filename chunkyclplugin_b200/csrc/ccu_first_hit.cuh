// ccu_first_hit.cuh - the march loop of the first-hit kernel (chunkycu.cu), shared with the feature-buffer kernel
// (ccu_features.cuh).  Included by chunkycu.cu where the loop has always stood, at global scope, so that the first-hit kernel
// compiles as it did.
#pragma once
#include "ccu_march.cuh"

// The warp-synchronous march loop of the thread-per-ray kernels (first-hit, feature buffers): every lane steps its ray until no
// lane of the warp is marching any more.  Kept out of line so that the loop is register-allocated by itself - inlined into the
// 64-register first-hit kernel, next to the block test, the ray was spilled and re-loaded inside the loop.  The ray travels
// through local memory once per call.
// st: 0 marching, anything else: not marching (returned unchanged).
template <bool DEEP>
static __device__ __noinline__ int first_hit_march(const ccu::DScene &s, ccu::LeanRay *ray, int st) {
    ccu::LeanRay r = *ray;
    while (__any_sync(0xffffffffu, st == 0)) {
        if (!DEEP) st = ccu::lean_step_flat<false>(s, s.air_top, r, st == 0, st, s.draw_depth, ~0u << s.depth);
        else if (st == 0) st = ccu::lean_probe<DEEP, false>(s, s.air_top, r, s.draw_depth);
    }
    ray->t = r.t;
    ray->steps = r.steps;
    return st;
}
