// kernels_screen_sub4.cu -- instantiations of score_screen_sub_kernel<4, NZ> (muse_screen_sub.cuh), n = 1024.
#include "muse_launch.h"

namespace muse {

template cudaError_t launch_screen_sub<4>(const ScreenParams &, int, cudaStream_t);

}  // namespace muse
