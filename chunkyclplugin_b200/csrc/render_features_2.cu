// render_features_2.cu - the k_features<2, HAS_BVH, V> instances (ccu_features.cuh), compiled in parallel with the rest of the library.
#include "ccu_features.cuh"

template ccu::FeaturesFn ccu::features_kernel_of<2>(bool, bool, bool);
