// render_mega_0.cu - the k_render_mega<0, V> instances (ccu_mega.cuh), compiled in parallel with the rest of the library.
#include "ccu_mega.cuh"

template ccu::MegaFn ccu::mega_kernel_of<0, false>(const ccu::ShadeKey &);
