// render_queue_01.cu - the k_render_queue<false, 1, V> instances (ccu_queue_units.cuh), compiled in parallel with the rest of the library.
#include "ccu_queue_units.cuh"

template ccu::QueueFn ccu::queue_kernel_of<false, 1, false>(const ccu::ShadeKey &);
#ifdef CCU_Q_STATS
template void ccu::queue_stats_take<false, 1, false>(unsigned long long *);
#endif
