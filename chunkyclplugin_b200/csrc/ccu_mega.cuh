// ccu_mega.cuh - the thread-per-pixel render kernel; included only by its instance units (render_mega_<MODE>.cu).
#pragma once
#include "ccu_march.cuh"
#include "ccu_render.cuh"

namespace ccu {

// Thread-per-pixel path tracer: all passes of the batch in one launch, the running mean of
// rayTracer.cl:109-112 carried in registers between passes (identical arithmetic, no memory round trip).
// MODE: 0 = the reference's own node array, 1 = commit-time layouts, 2 = commit-time layouts of a deep world.
// V: the Shade of the launch (sample_pixel, DESIGN §5).  The emitter table `g`, the biome colours `bv` and the cloud layer `cv`
// come after the other arguments, so that the kernels without them keep their parameter offsets.
template <int MODE, class V>
__global__ void __launch_bounds__(128) k_render_mega(const __grid_constant__ DScene s, const int *__restrict__ seeds, int n_passes,
                                                     int start_spp, float *res, const float *res_prev, int n_pixels,
                                                     const __grid_constant__ EmitView g, const __grid_constant__ BiomeView bv,
                                                     const __grid_constant__ CloudView cv) {
    if constexpr (V::biome) {
        if (threadIdx.x == 0) biome_smem() = bv;   // read after the barrier of stage_tables
    }
    stage_tables(s, nullptr);
    for (int gid = blockIdx.x * blockDim.x + threadIdx.x; gid < n_pixels; gid += gridDim.x * blockDim.x) {
        float *px = res + (size_t)gid * 3;
        const float *pp = res_prev + (size_t)gid * 3;    // what the reference's single buffer holds when the window starts
        float3 buf = f3(pp[0], pp[1], pp[2]);
        for (int pass = 0; pass < n_passes; pass++) {
            float3 col = sample_pixel<MODE, V>(s, g, cv, gid, __ldg(seeds + pass));
            int spp = start_spp + pass;
            float fs = (float)spp, fs1 = (float)(spp + 1);
            buf.x = (buf.x * fs + col.x) / fs1;
            buf.y = (buf.y * fs + col.y) / fs1;
            buf.z = (buf.z * fs + col.z) / fs1;
        }
        px[0] = buf.x; px[1] = buf.y; px[2] = buf.z;
    }
}

template <int MODE, bool CLOUDS>
MegaFn mega_kernel_of(const ShadeKey &v) {
    MegaFn k = nullptr;
    dispatch_clouds<CLOUDS>(v, [&](auto V) { k = k_render_mega<MODE, decltype(V)>; });
    return k;
}

}  // namespace ccu
