// render_queue_00_c.cu - the cloud k_render_queue<false, 0, V> instances (ccu_queue_units.cuh), compiled in parallel with the rest of the library.
#include "ccu_queue_units.cuh"

template ccu::QueueFn ccu::queue_kernel_of<false, 0, true>(const ccu::ShadeKey &);
#ifdef CCU_Q_STATS
template void ccu::queue_stats_take<false, 0, true>(unsigned long long *);
#endif
