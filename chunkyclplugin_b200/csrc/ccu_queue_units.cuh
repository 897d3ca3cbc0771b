// ccu_queue_units.cuh - the wavefront kernel's instances; included only by its units (render_queue_<HAS_BVH><LAY>[_c].cu).
#pragma once
#include "ccu_render.cuh"

namespace ccu {

template <bool HAS_BVH, int LAY, bool CLOUDS>
QueueFn queue_kernel_of(const ShadeKey &v) {
    QueueFn k = nullptr;
    dispatch_clouds<CLOUDS>(v, [&](auto V) { k = k_render_queue<HAS_BVH, LAY, decltype(V)>; });
    return k;
}

#ifdef CCU_Q_STATS
template <bool HAS_BVH, int LAY, bool CLOUDS>
void queue_stats_take(unsigned long long *st) {
    cudaMemcpyFromSymbol(st, g_qstats, sizeof(unsigned long long) * 32);
    unsigned long long z[32] = {0};
    cudaMemcpyToSymbol(g_qstats, z, sizeof z);
}
#endif

}  // namespace ccu
