// denoise.cu - the guided denoiser's kernels (ccu_denoise.cuh, DESIGN §17), compiled in a unit of their own.
#include "ccu_denoise.cuh"
