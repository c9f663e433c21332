// kernels_screen_sub3.cu -- instantiations of score_screen_sub_kernel<3, NZ> (muse_screen_sub.cuh), n = 512.
#include "muse_launch.h"

namespace muse {

template cudaError_t launch_screen_sub<3>(const ScreenParams &, int, cudaStream_t);

}  // namespace muse
