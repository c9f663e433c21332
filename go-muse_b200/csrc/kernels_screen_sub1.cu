// kernels_screen_sub1.cu -- instantiations of score_screen_sub_kernel<1, NZ> (muse_screen_sub.cuh), n = 128.
#include "muse_launch.h"

namespace muse {

template cudaError_t launch_screen_sub<1>(const ScreenParams &, int, cudaStream_t);

}  // namespace muse
