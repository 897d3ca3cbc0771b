// render_mega_2.cu - the k_render_mega<2, V> instances (ccu_mega.cuh), compiled in parallel with the rest of the library.
#include "ccu_mega.cuh"

template ccu::MegaFn ccu::mega_kernel_of<2, false>(const ccu::ShadeKey &);
