// ccu_render.cuh - the render kernels' shading variants as runtime values, and where their instances are.
//
// The instances of k_render_mega and k_render_queue are compiled in translation units of their own, one per MODE or
// (HAS_BVH, LAY) and value of the clouds switch (render_mega_<MODE>.cu, render_queue_<HAS_BVH><LAY>.cu, and the same names with
// _c for the cloud kernels), which the build compiles in parallel with chunkycu.cu and links into the same library; each unit
// returns its kernels through mega_kernel_of<MODE, CLOUDS> / queue_kernel_of<HAS_BVH, LAY, CLOUDS>.  The feature-buffer kernel
// (DESIGN §16) has one unit per MODE (render_features_<MODE>.cu, features_kernel_of<MODE>).  chunkycu.cu sees only the
// declarations.
#pragma once
#include <type_traits>

#include "ccu_queue.cuh"

namespace ccu {

// Calls f(std::integral_constant<int, v>{}) for v in [0, N) (N - 1 for anything larger), or f(std::bool_constant<v>{}):
// picks the template instance of a kernel from a runtime value.
template <int N, int I = 0, class F>
void dispatch(int v, F &&f) {
    if constexpr (I + 1 < N) {
        if (v != I) return dispatch<N, I + 1>(v, f);
    }
    f(std::integral_constant<int, I>{});
}
template <class F>
void dispatch(bool v, F &&f) {
    if (v) f(std::true_type{});
    else f(std::false_type{});
}

// A launch's Shade (ccu_device.cuh) as runtime values
struct ShadeKey {
    bool spec;
    int nee;   // a NeeKind
    bool biome;
    bool fog;
    bool clouds;
};
constexpr int N_SHADES = 2 * 5 * 2 * 2 * 2;
inline ShadeKey nth_shade(int i) { return {i % 2 != 0, i / 2 % 5, i / 10 % 2 != 0, i / 20 % 2 != 0, i / 40 != 0}; }   // i in [0, N_SHADES)

// Calls f(Shade<spec, nee, biome, fog, CLOUDS>{}) for the values of v whose clouds switch is CLOUDS: a unit instantiates the
// kernels of one value of the switch (render_*_c<CLOUDS>.cu) and returns nullptr for the other.
template <bool CLOUDS, class F>
void dispatch_clouds(const ShadeKey &v, F &&f) {
    if (v.clouds != CLOUDS) return;
    dispatch(v.spec, [&](auto S) {
        dispatch<5>(v.nee, [&](auto N) {
            dispatch(v.biome, [&](auto B) { dispatch(v.fog, [&](auto G) { f(Shade<S, NeeKind(N.value), B, G, CLOUDS>{}); }); });
        });
    });
}

using MegaFn = void (*)(DScene, const int *, int, int, float *, const float *, int, EmitView, BiomeView, CloudView);
// k_render_mega<MODE, Shade of v> for the Shades whose clouds switch is CLOUDS, else nullptr (render_mega_<MODE>[_c].cu)
template <int MODE, bool CLOUDS>
MegaFn mega_kernel_of(const ShadeKey &v);
template <int MODE>
MegaFn mega_kernel(const ShadeKey &v) { return v.clouds ? mega_kernel_of<MODE, true>(v) : mega_kernel_of<MODE, false>(v); }

using QueueFn = void (*)(DScene, QueueParams, EmitView, BiomeView, CloudView);
// k_render_queue<HAS_BVH, LAY, Shade of v> for the Shades whose clouds switch is CLOUDS, else nullptr
// (render_queue_<HAS_BVH><LAY>[_c].cu)
template <bool HAS_BVH, int LAY, bool CLOUDS>
QueueFn queue_kernel_of(const ShadeKey &v);
using FeaturesFn = void (*)(DScene, const int *, int, int, float *, float *, BiomeView, CloudView);
// k_features<MODE, bvh, Shade with the biome and clouds switches> of the feature buffers (DESIGN §16, render_features_<MODE>.cu)
template <int MODE>
FeaturesFn features_kernel_of(bool bvh, bool biome, bool clouds);
#define CCU_FEAT_THREADS 128   // threads per block of k_features

#ifdef CCU_Q_STATS
// the debug counters of the unit render_queue_<HAS_BVH><LAY>[_c].cu (_c: CLOUDS): copied to st[32], then cleared
template <bool HAS_BVH, int LAY, bool CLOUDS>
void queue_stats_take(unsigned long long *st);
#endif

}  // namespace ccu
