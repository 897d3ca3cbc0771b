// render_mega_2_c.cu - the cloud k_render_mega<2, V> instances (ccu_mega.cuh), compiled in parallel with the rest of the library.
#include "ccu_mega.cuh"

template ccu::MegaFn ccu::mega_kernel_of<2, true>(const ccu::ShadeKey &);
