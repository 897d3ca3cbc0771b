// ccu_features.cuh - the feature-buffer kernel (DESIGN §16); included only by its instance units (render_features_<MODE>.cu).
#pragma once
#include "ccu_first_hit.cuh"
#include "ccu_render.cuh"

namespace ccu {

// The first hit of camera ray (o, d) as a path segment of the render kernels (closestIntersect, then the cloud layer of §15.3
// under V::clouds), on the march of the first-hit kernel: albedo = the material colour shading multiplies into the throughput
// (biome-tinted under V::biome), normal = the surface normal; a cloud is white with the normal of the face entered; a miss is
// the sky clamped to 1 with a zero normal.  Every lane of the warp calls it (the march is warp-synchronous); `valid` false:
// the lane marches nothing.
template <int MODE, bool HAS_BVH, class V>
__device__ __forceinline__ void feature_sample(const DScene &s, const CloudView &cv, bool valid, float3 o, float3 d, float3 &albedo,
                                               float3 &normal) {
    Surf surf;
    surf.normal = f3(0, 0, 0); surf.color = make_float4(0, 0, 0, 0); surf.emittance = 0;
    float distance = inff_();
    bool hit = false;
    if (MODE == 0) {
        Record rec;
        rec.distance = inff_(); rec.material = 0; rec.surf = surf; rec.point = f3(0, 0, 0);
        HitInfo hi = {-1, 0, 0, 0, 0};
        if (valid) hit = HAS_BVH ? closest_intersect_ref<V>(s, o, d, rec, hi) : octree_intersect_ref<V>(s, o, d, rec, hi);
        surf = rec.surf;
        distance = rec.distance;
    } else {
        // k_first_hit's march: the warp marches on the air layout until no lane is marching, then runs the block tests together
        March m;
        const bool entered = march_begin(s, m, o, d, inff_());
        LeanRay r;
        r.o = m.o; r.d = m.d; r.inv = m.inv; r.t = m.t; r.limit = m.limit; r.steps = m.steps;
        lean_prepare(r);
        int st = (valid && entered) ? 0 : 2;      // 0 marching, 1 at a non-air leaf, 2 left the octree without a hit, 3 hit
        for (;;) {
            st = first_hit_march<MODE == 2>(s, &r, st);
            if (st == 1) {
                m.t = r.t; m.steps = r.steps;
                const Cell c = march_cell(m);
                int level;
                const int data = find_leaf_wide(s, c.bx, c.by, c.bz, level);
                float th;
                Surf hs;
                if (march_block<V>(s, m, data, level, hs, th)) {
                    st = 3;
                    surf = hs;
                    distance = th;
                } else {
                    r.t = m.t; r.steps = m.steps;
                    st = 0;
                }
            }
            if (!__any_sync(0xffffffffu, st == 0)) break;
        }
        hit = st == 3;
        if (HAS_BVH && valid) {
            int kind = 0;
            if (bvh_pair(s, o, d, distance, surf, kind)) hit = true;
        }
    }
    if constexpr (V::clouds) {
        float t;
        float3 n;
        if (valid && cloud_hit(cv, o, d, hit ? distance : inff_(), t, n)) {
            albedo = f3(1, 1, 1);
            normal = n;
            return;
        }
    }
    if (hit) {
        albedo = f3(surf.color.x, surf.color.y, surf.color.z);
        normal = surf.normal;
    } else {
        const float3 sky = valid ? sky_radiance(s, d) : f3(0, 0, 0);
        albedo = f3(fminf(sky.x, 1.0f), fminf(sky.y, 1.0f), fminf(sky.z, 1.0f));
        normal = f3(0, 0, 0);
    }
}

// The albedo and normal buffers of n_passes passes (DESIGN §16): pass p traces the camera ray of the render kernels' pass with
// seed seeds[p] and folds its feature_sample into the running mean of the render kernels (rayTracer.cl:109-112), held in
// registers; each output (either may be nullptr) is written once, float[3] per pixel.  Pixels are taken in the first-hit
// kernel's screen tiles.  The biome colours `bv` and the cloud layer `cv` come as the render kernels take them.
template <int MODE, bool HAS_BVH, class V>
__global__ void __launch_bounds__(CCU_FEAT_THREADS) k_features(const __grid_constant__ DScene s, const int *__restrict__ seeds, int n_passes,
                                                               int n_pixels, float *albedo, float *normal,
                                                               const __grid_constant__ BiomeView bv, const __grid_constant__ CloudView cv) {
    if constexpr (V::biome) {
        if (threadIdx.x == 0) biome_smem() = bv;   // read after the barrier of stage_tables
    }
    stage_tables(s, nullptr);
    const unsigned k = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = k < (unsigned)n_pixels;
    unsigned px = 0, py = 0;
    if (valid) tile_order_xy<true>(k, s.width, s.height, px, py);
    const int gid = (int)(py * (unsigned)s.width + px);
    float3 ab = f3(0, 0, 0), nb = f3(0, 0, 0);
    for (int pass = 0; pass < n_passes; pass++) {
        uint32_t rng = (uint32_t)__ldg(seeds + pass) + (uint32_t)gid;
        rng_next(rng);
        float3 o, d;
        camera_ray_xy<false>(s, gid, (int)px, (int)py, rng, o, d);
        float3 a, n;
        feature_sample<MODE, HAS_BVH, V>(s, cv, valid, o, d, a, n);
        const float fs = (float)pass, fs1 = (float)(pass + 1);
        ab.x = (ab.x * fs + a.x) / fs1;
        ab.y = (ab.y * fs + a.y) / fs1;
        ab.z = (ab.z * fs + a.z) / fs1;
        nb.x = (nb.x * fs + n.x) / fs1;
        nb.y = (nb.y * fs + n.y) / fs1;
        nb.z = (nb.z * fs + n.z) / fs1;
    }
    if (!valid) return;
    const size_t at = (size_t)gid * 3;
    if (albedo) { albedo[at] = ab.x; albedo[at + 1] = ab.y; albedo[at + 2] = ab.z; }
    if (normal) { normal[at] = nb.x; normal[at + 1] = nb.y; normal[at + 2] = nb.z; }
}

template <int MODE>
FeaturesFn features_kernel_of(bool bvh, bool biome, bool clouds) {
    FeaturesFn k = nullptr;
    dispatch(bvh, [&](auto B) {
        dispatch(biome, [&](auto T) {
            dispatch(clouds, [&](auto C) { k = k_features<MODE, B, Shade<false, NEE_NONE, T, false, C>>; });
        });
    });
    return k;
}

}  // namespace ccu
