// kernels_screen_sub2.cu -- instantiations of score_screen_sub_kernel<2, NZ> (muse_screen_sub.cuh), n = 256.
#include "muse_launch.h"

namespace muse {

template cudaError_t launch_screen_sub<2>(const ScreenParams &, int, cudaStream_t);

}  // namespace muse
