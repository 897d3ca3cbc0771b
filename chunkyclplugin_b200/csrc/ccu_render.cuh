// ccu_render.cuh - the render kernels' shading variants as runtime values, and where their instances are.
//
// The instances of k_render_mega and k_render_queue are compiled in translation units of their own (render_mega_<MODE>.cu,
// render_queue_<HAS_BVH><LAY>.cu), which the build compiles in parallel with chunkycu.cu and links into the same library; each
// unit returns its kernels through mega_kernel<MODE> / queue_kernel_of<HAS_BVH, LAY>.  chunkycu.cu sees only the declarations.
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
};
constexpr int N_SHADES = 2 * 5 * 2 * 2;
inline ShadeKey nth_shade(int i) { return {i % 2 != 0, i / 2 % 5, i / 10 % 2 != 0, i / 20 != 0}; }   // i in [0, N_SHADES)

// Calls f(Shade<spec, nee, biome, fog>{}) for the values of v.
template <class F>
void dispatch(const ShadeKey &v, F &&f) {
    dispatch(v.spec, [&](auto S) {
        dispatch<5>(v.nee, [&](auto N) {
            dispatch(v.biome, [&](auto B) { dispatch(v.fog, [&](auto G) { f(Shade<S, NeeKind(N.value), B, G>{}); }); });
        });
    });
}

using MegaFn = void (*)(DScene, const int *, int, int, float *, const float *, int, EmitView, BiomeView);
// k_render_mega<MODE, Shade of v> (render_mega_<MODE>.cu)
template <int MODE>
MegaFn mega_kernel(const ShadeKey &v);

using QueueFn = void (*)(DScene, QueueParams, EmitView, BiomeView);
// k_render_queue<HAS_BVH, LAY, Shade of v> (render_queue_<HAS_BVH><LAY>.cu)
template <bool HAS_BVH, int LAY>
QueueFn queue_kernel_of(const ShadeKey &v);
#ifdef CCU_Q_STATS
// the debug counters of the unit render_queue_<HAS_BVH><LAY>.cu: copied to st[32], then cleared
template <bool HAS_BVH, int LAY>
void queue_stats_take(unsigned long long *st);
#endif

}  // namespace ccu
